"""What --observed costs (DESIGN.md 4.13): the same scoring passes with and without the per-sample observed counts, in one
process, alternating.

Setup: bench.py's synthetic cohort (npc_synth_fill_device) and score rows, default 125,000 variants x 500,000 samples.
  int8      npc_score_block_device in launches of at most 32,768 rows over the resident int8 slab (bench.py's pass), with
            and without npc_set_observed.
  bed       the same rows packed to PLINK .bed rows (2 bits per sample).
  dose255   the same rows as BGEN 2-byte fixed-point rows (255 x ALT dosage, 0xFFFF missing), --dose-rows of them (the
            2-byte slab of every row does not fit beside the others).
  multi     18 score definitions (each a random 70 % of the rows, bench.py's betas reshuffled) over --multi-rows x
            --multi-samples int8 rows, npc_score_resident_multi against npc_score_resident_multi_observed.
A step is npc_reset + the launches + a synchronise, timed with CUDA events; the report is the median over --steps
alternating rounds.  "added" is the time with counts minus the time without; the observed pass's bytes are one read
of every OK row (what the kernel must load), and its rate is bytes / added, against the 6547 GB/s copy peak.  The
device name and power limit are read in the same run.  Counts are checked against the OK records' ngt sums."""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

LAUNCH = 32768
COPY_PEAK_GBS = 6547.0


def gpu_info(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:                      # noqa: BLE001 -- a report field, not a measurement
        return {"error": str(e)}


def ok_ngt(loci):
    ok = (loci["klass"] == 0) & (loci["used"] != 0)
    return int(loci["ngt"][ok].sum()), int(ok.sum())


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=125_000)
    ap.add_argument("--samples", type=int, default=500_000)
    ap.add_argument("--dose-rows", type=int, default=20_000)
    ap.add_argument("--multi-rows", type=int, default=20_000)
    ap.add_argument("--multi-samples", type=int, default=200_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    args = ap.parse_args()
    import torch
    import nimpress_b200 as nb
    from bench import SEED, cohort_params, make_rows
    from bench_bed import pack_to_bed

    if not torch.cuda.is_available():
        raise SystemExit("bench_observed.py measures on a GPU: no CUDA device")
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    n, V = args.samples, args.rows
    result = {"device": gpu_info(args.device), "samples": n, "rows": V, "launch_rows": LAUNCH, "steps": args.steps,
              "warmup": args.warmup, "copy_peak_gbs": COPY_PEAK_GBS, "runs": {}}

    def synth(n_, V_, v0=0):
        af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(v0, V_)
        stride = -(-2 * n_ // 128) * 128
        gt = torch.empty((V_, stride), dtype=torch.uint8, device=dev)
        e = nb.Engine(n_, gt_width=1, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
        e.set_stream(stream.cuda_stream)
        t = [torch.from_numpy(x.view(np.int32)).to(dev) for x in (af_thr, miss_thr)] + [torch.from_numpy(alt).to(dev)]
        e.synth_fill_device(gt, stride, v0, V_, SEED, *t)
        torch.cuda.synchronize()
        e.close()
        return gt, stride, make_rows(nb.ROW_DTYPE, V_, af, beta, ref_is_ea)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b) * 1e-3

    def bench_layout(name, slab, stride, width, rows, row_bytes):
        engs = {}
        for obs in (False, True):
            e = nb.Engine(n, gt_width=width, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
            e.set_stream(stream.cuda_stream)
            e.set_policy()
            e.set_observed(obs)
            engs[obs] = e
        rel = rows.copy()
        rel["gt_row"] = np.arange(len(rows)) % LAUNCH

        def step(obs):
            e = engs[obs]
            e.reset()

            def go():
                for r0 in range(0, len(rows), LAUNCH):
                    nr = min(LAUNCH, len(rows) - r0)
                    e.score_block_device(slab.data_ptr() + r0 * stride, stride, nr, rel[r0:r0 + nr])
            return timed(go)
        for _ in range(args.warmup):
            step(False); step(True)
        ts = {False: [], True: []}
        for i in range(args.steps):                      # alternating, the order flipped every round
            for obs in ((False, True) if i % 2 == 0 else (True, False)):
                ts[obs].append(step(obs))
        outs = {obs: engs[obs].finish() for obs in engs}
        counts = engs[True].observed()
        ngt, n_ok = ok_ngt(outs[True]["loci"])
        assert int(counts.sum()) == ngt, (name, int(counts.sum()), ngt)
        assert np.array_equal(outs[True]["scores"].view(np.uint64), outs[False]["scores"].view(np.uint64))
        t_off, t_on = float(np.median(ts[False])), float(np.median(ts[True]))
        added = t_on - t_off
        obs_bytes = n_ok * row_bytes
        result["runs"][name] = {"s_without": t_off, "s_with": t_on, "s_added": added, "added_frac": added / t_off,
                                "s_without_range": [float(min(ts[False])), float(max(ts[False]))],
                                "s_with_range": [float(min(ts[True])), float(max(ts[True]))],
                                "observed_pass_bytes": obs_bytes, "observed_pass_gbs": obs_bytes / added / 1e9 if added > 0 else None,
                                "observed_pass_copy_peak_frac": obs_bytes / added / 1e9 / COPY_PEAK_GBS if added > 0 else None,
                                "ok_rows": n_ok}
        for e in engs.values():
            e.close()
        print(json.dumps({name: result["runs"][name]}), flush=True)

    gt, stride, rows = synth(n, V)
    bench_layout("int8", gt, stride, 1, rows, 2 * n)
    bstride = -(-((n + 3) // 4) // 128) * 128
    bed = torch.zeros((V, bstride), dtype=torch.uint8, device=dev)
    pack_to_bed(torch, gt.view(torch.int8), n, bed)
    torch.cuda.synchronize()
    Vd = min(args.dose_rows, V)
    dose_src = gt[:Vd].clone()
    del gt
    torch.cuda.empty_cache()
    bench_layout("bed", bed, bstride, nb.GT_BED, rows, (n + 3) // 4)
    del bed
    torch.cuda.empty_cache()
    dstride = -(-2 * n // 128) * 128
    dose = torch.zeros((Vd, dstride // 2), dtype=torch.int32, device=dev)
    for r0 in range(0, Vd, 1024):
        g = dose_src[r0:r0 + 1024, :2 * n].view(-1, n, 2).to(torch.int32)
        a = (g >> 1) - 1
        k = torch.where((a < 0).any(-1), 0xFFFF, 255 * (a == 1).sum(-1))
        dose[r0:r0 + 1024, :n] = k
    dose16 = dose.to(torch.int16)                      # 0xFFFF wraps to -1: the same two bytes
    del dose, dose_src
    bench_layout("dose255", dose16.view(torch.uint8), dstride, nb.GT_DOSE255, rows[:Vd], 2 * n)
    del dose16
    torch.cuda.empty_cache()

    # 18 definitions through the multi-score sibling
    m_n, m_V = args.multi_samples, args.multi_rows
    mgt, mstride, mrows = synth(m_n, m_V)
    rng = np.random.default_rng(SEED)
    lists = []
    for k in range(18):
        r = mrows[np.sort(rng.choice(m_V, size=int(0.7 * m_V), replace=False))].copy()
        r["beta"] = rng.permutation(r["beta"])
        lists.append(r)
    e = nb.Engine(m_n, gt_width=1, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
    e.set_stream(stream.cuda_stream)
    e.set_policy()
    e.resident_adopt(mgt, mstride, m_V)
    offs = [0.0] * 18
    for _ in range(args.warmup):
        e.score_resident_multi(lists, offs); e.score_resident_multi(lists, offs, observed=True)
    ts = {False: [], True: []}
    for i in range(args.steps):
        for obs in ((False, True) if i % 2 == 0 else (True, False)):
            ts[obs].append(timed(lambda: e.score_resident_multi(lists, offs, observed=obs)))
    got = e.score_resident_multi(lists, offs, observed=True)
    for sc, nloci, loci, counts in got:
        assert int(counts.sum()) == ok_ngt(loci)[0]
    t_off, t_on = float(np.median(ts[False])), float(np.median(ts[True]))
    groups = -(-18 // 8)
    obs_bytes = groups * m_V * 2 * m_n                   # every slab row is an entry of every group
    result["runs"]["multi18"] = {"samples": m_n, "rows": m_V, "s_without": t_off, "s_with": t_on, "s_added": t_on - t_off,
                                 "added_frac": (t_on - t_off) / t_off, "contractions": e.multi_contractions, "groups": groups,
                                 "observed_pass_bytes": obs_bytes,
                                 "observed_pass_gbs": obs_bytes / (t_on - t_off) / 1e9 if t_on > t_off else None}
    e.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
