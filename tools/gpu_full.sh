#!/bin/bash
# Full validation of the current tree on one B200: all GPU tests, smoke, the default bench line,
# the reference arm, a launch list and one full ncu capture of the bench's launch shape.
mkdir -p out
echo "== pytest -m gpu"; timeout 2400 python -m pytest tests -x -q -m gpu 2>&1 | tail -5 | tee out/pytest_gpu.log
echo "== smoke"; timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee out/smoke.log
echo "== bench (default: 125k x 500k resident)"; timeout 1200 python bench.py 2>&1 | tail -1 > out/bench_full.json; cut -c1-600 out/bench_full.json
echo "== bench --impl reference"; timeout 600 python bench.py --impl reference --steps 3 --warmup 1 2>&1 | tail -1 > out/bench_reference.json; cut -c1-400 out/bench_reference.json
echo "== ncu launch list (same command, small step count)"
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -c 60 --csv --log-file out/launches.csv \
    python bench.py --steps 1 --warmup 1 --no-e2e --no-cpu-baseline > out/ncu_launch.log 2>&1; tail -1 out/ncu_launch.log | cut -c1-200
echo "== ncu full of the bench launch shape (32768 rows x 500k)"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'k_fused_pair' -s 1 -c 1 -o out/prof_bench_shape -f \
    python bench.py --variants 32768 --steps 1 --warmup 1 --no-e2e --no-cpu-baseline > out/ncu_full.log 2>&1; tail -1 out/ncu_full.log | cut -c1-200
