#!/bin/bash
# compute-sanitizer over a small parity run of every kernel path (pair kernel with row groups, exact order, int16,
# two-kernel, generic widths, dosage rows, npc_reduce).  Output: out/sanitizer_*.log
mkdir -p out
cat > /tmp/san.py <<'PY'
import os, sys
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import numpy as np, nimpress_b200 as nb, orc
from util_cohort import random_cohort, random_rows, assert_parity
rng = np.random.default_rng(1)
for (n, V, width, ploidy, exact, env) in [(20011, 150, 1, 2, False, {}), (20011, 150, 1, 2, True, {}), (3001, 40, 2, 2, True, {}),
                                           (9001, 60, 2, 2, False, {}), (3001, 40, 1, 3, True, {}), (20011, 90, 1, 2, True, {"NPC_FUSED": "0"}),
                                           # two chunk sets per thread (a raw stage each, idle lanes predicated), 4-tile decider passes
                                           (20011, 90, 1, 2, False, {"NPC_TILE_K": "2", "NPC_TILE_GD": "4"}), (20011, 90, 1, 2, True, {"NPC_TILE_K": "2"}),
                                           # 18 consumer warps: the 72-register instance of the K = 1 kernel
                                           (40003, 70, 1, 2, False, {"NPC_TILE_GR": "16"})]:
    for k, v in env.items(): os.environ[k] = v
    gt = random_cohort(rng, n, V, width=width, ploidy=ploidy, miss_rate=0.03, n_alt=5, sentinel_rate=0.01)
    rows = random_rows(rng, V, n_rows=V + 20, n_alt=5)
    eng = nb.Engine(n, ploidy=ploidy, gt_width=width, max_rows_per_block=256, n_slots=2)
    eng.set_policy(); eng.set_exact_order(exact); eng.reset()
    for r0 in range(0, len(rows), 97): eng.score_host(gt, rows[r0:r0 + 97])
    got = eng.finish(offset=0.5); shape = eng.kernel_shape; eng.close()
    assert_parity(got, orc.score_matrix(gt, n, ploidy, rows, offset=0.5), exact=exact or shape["fused"] != 2)
    print("ok", n, V, width, ploidy, exact, env, shape["fused"], shape["consumer_warps"], shape["chunks_per_thread"], shape["decider_tiles"], flush=True)
    for k in env: os.environ.pop(k)
# FORMAT/DS rows and the multi-context combine
n, V = 5003, 30
ds = np.round(rng.uniform(0, 2, size=(V, -(-n // 32) * 32)), 3).astype(np.float32)
ds.view(np.uint32)[rng.random(ds.shape) < 0.03] = 0x7F800001
rows = random_rows(rng, V, n_rows=40); rows["eaidx"] = np.where(rows["ref_is_ea"] == 1, 0, 1)
eng = nb.Engine(n, ploidy=1, gt_width=4, max_rows_per_block=64, n_slots=2); eng.set_dosage_rows(True); eng.set_policy(); eng.reset()
eng.score_host(ds, rows); got = eng.finish(offset=0.1); eng.close()
assert_parity(got, orc.score_matrix(ds, n, 1, rows.astype(orc.ROW_DTYPE), offset=0.1), exact=True)
print("ok dosage rows", flush=True)
gt = random_cohort(rng, n, V, miss_rate=0.03); rows = random_rows(rng, V, n_rows=50)
es = []
for k in range(3):
    e = nb.Engine(n, max_rows_per_block=64, n_slots=2); e.set_policy(); e.reset(); e.score_host(gt, rows[k * 17:(k + 1) * 17 if k < 2 else 50]); es.append(e)
sc, nl = nb.reduce_contexts(es, offset=0.0)
want = orc.score_matrix(gt, n, 2, rows.astype(orc.ROW_DTYPE))
assert nl == want["nloci"] and np.nanmax(np.abs(sc - want["scores"])) < 1e-12
print("ok npc_reduce over 3 contexts", flush=True)
PY
for tool in memcheck racecheck synccheck; do
  echo "== $tool"; timeout 1200 compute-sanitizer --tool $tool --print-limit 20 python /tmp/san.py > out/sanitizer_$tool.log 2>&1
  grep -E "^ok|ERROR SUMMARY|RACECHECK SUMMARY|Error|hazard" out/sanitizer_$tool.log | head -12
done
