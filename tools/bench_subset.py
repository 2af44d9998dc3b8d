"""Subset contexts (npc_create_subset, --samples; DESIGN.md 4.11) on one GPU, in three parts, one process.

1. npc_gather_rows_device alone on device-resident rows of 500,000 samples: int8 diploid GT (2 B per sample), .bed
   (2 bits) and 4-byte rows (FORMAT/DS, FORMAT/PL, 32-bit BGEN rows), keep fractions 0.1, 0.5, 0.9 and 0.999, random and
   contiguous.  --gather-rows random-byte rows (default 4,000: 4 GB of int8 rows, far beyond the 126 MB L2), CUDA events
   around --steps launches after --warmup.  Bytes per launch = rows x (32 x the sectors of a full row holding a kept
   sample + the compact row); the keep list itself is read from L2 and not counted.  Reported as us per row and as a
   fraction of the HBM rate (MEASURED_PEAKS.json hbm_gbs, else 6547.2 GB/s); next to it, the H2D copy of the same full
   rows from pinned memory, measured in the same run.
2. Scoring, alternating: bench.py's synthetic cohort (npc_synth_fill_device) of --score-rows variants x 500,000 samples,
   compacted on the device to 250,000 kept samples; a subset context and a plain 250,000-sample context score the same
   compact rows (npc_score_block_device, default order, launches of 32,768 rows).  The kernels are the same, so the times
   should match and the scores must be bit-equal.  Then 1,000,000 kept of 2,000,000: the subset context (one-read tile
   kernel) on the compact rows, with and without the gather, against the plain 2,000,000-sample context (two-read wide
   mode) on the full rows.
3. `nimpress` from disk: a BGZF BCF of --cli-variants x --cli-samples (default 10,000 x 100,000) and the same file with
   a random half of the samples, then `nimpress --samples=<half>` on the full file and `nimpress` on the half file,
   alternating, under NIMPRESS_TIMING=1.  Their WARN lines and scores must be identical (the half file names its samples
   anew, so names are left out of the comparison).

The device name and power limit are read in the same run.  Prints the result JSON, and also writes it to --out when given.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

from bench_bed import gpu_info  # noqa: E402

LAUNCH = 32768
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")


def keep_list(rng, n, frac, contiguous):
    k = max(1, int(round(n * frac)))
    if contiguous:
        s = (n - k) // 2
        return np.arange(s, s + k)
    return np.sort(rng.choice(n, k, replace=False))


def timed(torch, stream, fn, steps, warmup):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(steps):
        fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) * 1e-3 / steps


def part_gather(torch, nb, dev, stream, args, peak):
    n, R = 500_000, args.gather_rows
    rng = np.random.default_rng(1)
    out = []
    layouts = (("int8 diploid GT", 2, 1), (".bed", 2, nb.GT_BED), ("4-byte rows (DS / PL / DOSE32)", 2, nb.GT_PL))
    for name, ploidy, width in layouts:
        sb = nb.gt_row_bytes(n, ploidy, width)
        ss = -(-sb // 128) * 128
        src = torch.randint(0, 256, (R, ss), dtype=torch.uint8, device=dev)
        # H2D of the same full rows from pinned memory (what npc_stage_upload copies before it gathers)
        h = torch.empty((min(R, 512), ss), dtype=torch.uint8, pin_memory=True)
        d = torch.empty_like(h, device=dev)
        t_h2d = timed(torch, stream, lambda: d.copy_(h, non_blocking=True), max(2, args.steps // 2), 1) / h.shape[0]
        for frac in (0.1, 0.5, 0.9, 0.999):
            for contiguous in (False, True):
                keep = keep_list(rng, n, frac, contiguous)
                eng = nb.Engine(0, ploidy=ploidy, gt_width=width, max_rows_per_block=64, device=args.device, keep=keep, n_row_samples=n)
                eng.set_stream(stream.cuda_stream)
                db = nb.gt_row_bytes(len(keep), ploidy, width)
                ds = -(-db // 128) * 128
                dst = torch.empty((R, ds), dtype=torch.uint8, device=dev)
                t = timed(torch, stream, lambda: eng.gather_rows_device(src, ss, R, dst, ds), args.steps, args.warmup)
                # the 32-byte sectors of a full row that hold a kept sample, and the compact row
                sectors = np.unique(keep // 128 if width == nb.GT_BED else keep * (2 if width == 1 else 4) // 32).size
                nbytes = R * (32 * sectors + db)
                out.append({"layout": name, "n_row_samples": n, "keep_fraction": frac, "keep": "contiguous" if contiguous else "random",
                            "rows": R, "us_per_row": t / R * 1e6, "bytes_per_s": nbytes / t, "fraction_of_hbm": nbytes / t / (peak * 1e9),
                            "h2d_us_per_row_same_full_rows": t_h2d * 1e6, "gather_over_h2d": (t / R) / t_h2d})
                print(json.dumps(out[-1]), flush=True)
                eng.close()
                del dst
        del src, h, d
        torch.cuda.empty_cache()
    return out


def part_score(torch, nb, dev, stream, args):
    from bench import SEED, cohort_params, make_rows
    res = []
    for n_row, n_keep, V in ((500_000, 250_000, args.score_rows), (2_000_000, 1_000_000, max(1, args.score_rows // 4))):
        rng = np.random.default_rng(2)
        keep = np.sort(rng.choice(n_row, n_keep, replace=False))
        af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(0, V)
        rows = make_rows(nb.ROW_DTYPE, V, af, beta, ref_is_ea)
        rows["gt_row"] = np.arange(V) % LAUNCH
        t_af, t_ms, t_alt = (torch.from_numpy(x.view(np.int32)).to(dev) for x in (af_thr, miss_thr, alt))
        ss, cs = -(-2 * n_row // 128) * 128, -(-2 * n_keep // 128) * 128
        full = torch.empty((V, ss), dtype=torch.uint8, device=dev)
        whole = nb.Engine(n_row, max_rows_per_block=LAUNCH, device=args.device)
        whole.set_stream(stream.cuda_stream)
        whole.set_policy()
        whole.synth_fill_device(full, ss, 0, V, SEED, t_af, t_ms, t_alt)
        sub = nb.Engine(0, max_rows_per_block=LAUNCH, device=args.device, keep=keep, n_row_samples=n_row)
        plain = nb.Engine(n_keep, max_rows_per_block=LAUNCH, device=args.device)
        for e in (sub, plain):
            e.set_stream(stream.cuda_stream)
            e.set_policy()
        compact = torch.empty((V, cs), dtype=torch.uint8, device=dev)
        t_gather = timed(torch, stream, lambda: sub.gather_rows_device(full, ss, V, compact, cs), 3, 1)

        def score(e, slab, st):
            e.reset()
            for r0 in range(0, V, LAUNCH):
                nr = min(LAUNCH, V - r0)
                e.score_block_device(slab.data_ptr() + r0 * st, st, nr, rows[r0:r0 + nr])

        times = {"subset": [], "plain": []} if n_row == 500_000 else {"subset": [], "whole": []}
        for _ in range(args.warmup):
            for k in times:
                score(sub if k == "subset" else plain if k == "plain" else whole, compact if k != "whole" else full, cs if k != "whole" else ss)
        for _ in range(args.steps):
            for k in times:
                times[k].append(timed(torch, stream, lambda: score(sub if k == "subset" else plain if k == "plain" else whole,
                                                                    compact if k != "whole" else full, cs if k != "whole" else ss), 1, 0))
        r = {"n_row_samples": n_row, "n_keep": n_keep, "variants": V, "gather_s": t_gather,
             "shape_subset": sub.kernel_shape["fused"], "s_per_pass": {k: float(np.median(v)) for k, v in times.items()},
             "spread": {k: [float(min(v)), float(max(v))] for k, v in times.items()}}
        r["kept_genotypes_per_s_subset"] = V * n_keep / r["s_per_pass"]["subset"]
        r["kept_genotypes_per_s_subset_with_gather"] = V * n_keep / (r["s_per_pass"]["subset"] + t_gather)
        a = sub.finish(offset=0.0, want_loci=False)["scores"]
        if "plain" in times:
            r["shape_plain"] = plain.kernel_shape["fused"]
            b = plain.finish(offset=0.0, want_loci=False)["scores"]
            r["scores_bit_equal"] = bool(np.array_equal(a.view(np.uint64), b.view(np.uint64)))
        else:
            r["shape_whole"] = whole.kernel_shape["fused"]
            r["genotypes_per_s_whole"] = V * n_row / r["s_per_pass"]["whole"]
        print(json.dumps(r), flush=True)
        res.append(r)
        for e in (sub, plain, whole):
            e.close()
        del full, compact
        torch.cuda.empty_cache()
    return res


def part_cli(args):
    import orc
    from bench import SEED, cohort_params
    from bench_cli_config3 import write_bcf_streaming
    n, V = args.cli_samples, args.cli_variants
    af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(0, V)
    positions = 10_000 + 137 * np.arange(V)
    keep = np.sort(np.random.default_rng(3).choice(n, n // 2, replace=False))
    tmp = tempfile.mkdtemp(prefix="npsub_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    full, half, score, lst = (os.path.join(tmp, f) for f in ("full.bcf", "half.bcf", "s.score", "keep.txt"))
    with open(score, "w") as f:
        f.write("subset\nsynthetic\ncitation\nhs37d5\n0.125\n")
        for v in range(V):
            f.write(f"1\t{positions[v]}\tA\t{'A' if ref_is_ea[v] else 'C'}\t{float(beta[v])!r}\t{round(float(af[v]), 4)!r}\n")
    batch = max(1, (256 << 20) // (2 * n))

    def rows(sel):
        for v0 in range(0, V, batch):
            gt = np.zeros((min(batch, V - v0), 2 * n), np.int8)
            nv = gt.shape[0]
            orc.synth_fill(gt, n, v0, SEED, af_thr[v0:v0 + nv], miss_thr[v0:v0 + nv], alt[v0:v0 + nv])
            yield gt if sel is None else np.ascontiguousarray(gt.reshape(gt.shape[0], n, 2)[:, sel].reshape(gt.shape[0], -1))
    pool = ThreadPoolExecutor(os.cpu_count() or 4)
    write_bcf_streaming(full, n, V, "1", positions, rows(None), pool)
    write_bcf_streaming(half, len(keep), V, "1", positions, rows(keep), pool)      # names S000000.. again: compared without names
    with open(lst, "w") as f:
        f.write("\n".join(f"S{i:06d}" for i in keep) + "\n")
    out = {"variants": V, "samples": n, "kept": len(keep), "runs": []}
    outs = {}
    for rep in range(args.cli_reps):
        for mode in ("samples", "half_file", "full_file"):
            cmd = [EXE, f"--samples={lst}", score, full] if mode == "samples" else [EXE, score, half if mode == "half_file" else full]
            t0 = time.perf_counter()
            p = subprocess.run(cmd, capture_output=True, text=True, env=dict(os.environ, NIMPRESS_TIMING="1"))
            dt = time.perf_counter() - t0
            assert p.returncode == 0, p.stderr[-2000:]
            outs.setdefault(mode, [ln if ln.startswith("WARN") else ln.split("\t", 1)[1] for ln in p.stdout.splitlines()])
            phases = {ln.split("]")[1].rsplit(None, 2)[0].strip(): float(ln.rsplit(None, 2)[1]) for ln in p.stderr.splitlines()
                      if ln.startswith("[nimpress timing]") and ln.rstrip().endswith("ms")}
            out["runs"].append({"mode": mode, "rep": rep, "wall_s": dt, "phases_ms": phases})
            print(json.dumps(out["runs"][-1]), flush=True)
    out["samples_output_equals_half_file"] = outs["samples"] == outs["half_file"]       # WARN lines and scores, names aside
    for f in (full, half, score, lst):
        os.remove(f)
    os.rmdir(tmp)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--gather-rows", type=int, default=4000)
    ap.add_argument("--score-rows", type=int, default=20_000)
    ap.add_argument("--cli-variants", type=int, default=10_000)
    ap.add_argument("--cli-samples", type=int, default=100_000)
    ap.add_argument("--cli-reps", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--parts", default="gather,score,cli")
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    args = ap.parse_args()
    import torch
    import nimpress_b200 as nb
    if not torch.cuda.is_available():
        raise SystemExit("bench_subset.py measures on a GPU: no CUDA device")
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6547.2
    res = {"gpu": gpu_info(args.device), "hbm_gbs": peak}
    parts = args.parts.split(",")
    if "gather" in parts:
        res["gather"] = part_gather(torch, nb, dev, stream, args, peak)
    if "score" in parts:
        res["score"] = part_score(torch, nb, dev, stream, args)
    if "cli" in parts:
        res["cli"] = part_cli(args)
    res["gpu_after"] = gpu_info(args.device)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(res, open(args.out, "w"), indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
