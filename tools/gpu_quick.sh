#!/bin/bash
# quick check: parity subset + one bench line (+ optional ncu) for kernel iterations
mkdir -p out
timeout 900 python -m pytest tests/test_gpu_parity.py -x -q -m gpu -k "kernel_paths or full_sample or slow_path or sample_count or empty" 2>&1 | tail -3
B="python bench.py --variants 32768 --steps 3 --warmup 3 --no-cpu-baseline --no-e2e --brief"
timeout 200 $B 2>&1 | tail -1
if [ -n "$NCU" ]; then
timeout 400 ncu --set full --clock-control none --import-source on -k regex:'k_fused_pair' -s 2 -c 1 -o out/prof_quick -f \
    python bench.py --variants 8192 --steps 1 --warmup 2 --no-e2e --no-cpu-baseline > out/ncu_fused.log 2>&1
fi
