"""PLINK 1 .bed rows against int8 BCF GT rows on one GPU: the same cohort and score rows, scored in one process,
alternating, in the default and the exact summation order (DESIGN.md 4.7).

Setup: bench.py's synthetic cohort (npc_synth_fill_device: REF / one ALT / missing per allele, so packing it to 2-bit
codes is lossless -- a half call is missing either way) and score rows, default 125,000 variants x 500,000 samples.  The
int8 rows are packed to .bed rows on the GPU with torch, in chunks.  A step is npc_reset + the rows in launches of at
most 32,768 (npc_score_block_device, as bench.py) + a synchronise, timed with CUDA events.

Report, per layout and mode: genotypes/s, algorithmic bytes/s and the fraction of the HBM bound.  Bytes per launch of R
rows over n samples: int8 = 2 n R + 32 R + 16 n (bench.py's definition: one read of the slab); bed = 2 ceil(n/4) R + 32 R
+ 16 n (two reads of the 2-bit rows: tally pass and accumulate pass).  The peak is MEASURED_PEAKS.json hbm_gbs as in
bench.py.  The device name and power limit are read in the same run.

Check: exact-order scores of the two layouts equal bit for bit, records and nloci equal; default order within 1e-12
relative plus 8 eps sum|beta| / nloci (the int8 tile kernel associates its row groups differently).

--rows 1000000: the genome-wide config, resident on one GPU as .bed rows (125 GB at 500,000 samples); the int8 slab
(1 TB) does not fit, so only the bed path is timed, per pass."""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

LAUNCH = 32768


def gpu_info(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:                      # noqa: BLE001 -- a report field, not a measurement
        return {"error": str(e)}


def pack_to_bed(torch, gt, n, bed, chunk=512):
    """int8 diploid rows gt[V, stride] -> .bed rows bed[V, bstride] (00 hom ALT, 01 missing, 10 het, 11 hom REF)."""
    nb4 = (n + 3) // 4
    for r0 in range(0, gt.shape[0], chunk):
        g = gt[r0:r0 + chunk, :2 * n].view(-1, n, 2).to(torch.int16)
        a = (g >> 1) - 1
        miss = (a < 0).any(-1)
        nalt = (a == 1).sum(-1)
        code = torch.where(miss, 1, torch.where(nalt == 2, 0, torch.where(nalt == 1, 2, 3))).to(torch.uint8)
        if nb4 * 4 > n:
            code = torch.cat([code, torch.zeros((code.shape[0], nb4 * 4 - n), dtype=torch.uint8, device=code.device)], 1)
        q = code.view(code.shape[0], nb4, 4)
        bed[r0:r0 + chunk, :nb4] = q[..., 0] | (q[..., 1] << 2) | (q[..., 2] << 4) | (q[..., 3] << 6)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=125_000)
    ap.add_argument("--samples", type=int, default=500_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    args = ap.parse_args()
    import torch
    import nimpress_b200 as nb
    import orc
    from bench import SEED, cohort_params, make_rows

    if not torch.cuda.is_available():
        raise SystemExit("bench_bed.py measures on a GPU: no CUDA device")
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    n, V = args.samples, args.rows
    stride = -(-2 * n // 128) * 128
    bstride = -(-((n + 3) // 4) // 128) * 128
    af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(0, V)
    rows = make_rows(nb.ROW_DTYPE, V, af, beta, ref_is_ea)
    rows_rel = rows.copy()
    rows_rel["gt_row"] = np.arange(V) % LAUNCH
    free = torch.cuda.mem_get_info(dev)[0]
    with_int8 = V * stride + V * bstride + (8 << 30) < free
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    engines = {}
    for layout in (("int8", "bed") if with_int8 else ("bed",)):
        e = nb.Engine(n, gt_width=1 if layout == "int8" else nb.GT_BED, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
        e.set_stream(stream.cuda_stream)
        e.set_policy()
        engines[layout] = e
    # the synthetic int8 cohort, packed to .bed rows (in chunks through a scratch slab when the int8 slab does not fit)
    bed = torch.empty((V, bstride), dtype=torch.uint8, device=dev)
    bed.zero_()
    t_af = torch.from_numpy(af_thr.view(np.int32)).to(dev)
    t_ms = torch.from_numpy(miss_thr.view(np.int32)).to(dev)
    t_alt = torch.from_numpy(alt).to(dev)
    filler = engines.get("int8") or nb.Engine(n, gt_width=1, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
    filler.set_stream(stream.cuda_stream)
    if with_int8:
        gt = torch.empty((V, stride), dtype=torch.uint8, device=dev)
        filler.synth_fill_device(gt, stride, 0, V, SEED, t_af, t_ms, t_alt)
        pack_to_bed(torch, gt.view(torch.int8), n, bed)
    else:
        gt = None
        chunk = 4096
        scratch = torch.empty((chunk, stride), dtype=torch.uint8, device=dev)
        for r0 in range(0, V, chunk):
            nr = min(chunk, V - r0)
            filler.synth_fill_device(scratch, stride, r0, nr, SEED, t_af[r0:], t_ms[r0:], t_alt[r0:])
            pack_to_bed(torch, scratch[:nr].view(torch.int8), n, bed[r0:r0 + nr])
        del scratch
        filler.close()
    torch.cuda.synchronize()

    slabs = {"int8": (gt, stride), "bed": (bed, bstride)}

    def step(layout, exact):
        e = engines[layout]
        slab, st = slabs[layout]
        e.set_exact_order(exact)
        e.reset()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for r0 in range(0, V, LAUNCH):
            nr = min(LAUNCH, V - r0)
            e.score_block_device(slab.data_ptr() + r0 * st, st, nr, rows_rel[r0:r0 + nr])
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b) * 1e-3

    def launch_bytes(layout):
        per_row = 2 * n if layout == "int8" else 2 * ((n + 3) // 4)
        return sum(per_row * min(LAUNCH, V - r0) + 32 * min(LAUNCH, V - r0) + 16 * n for r0 in range(0, V, LAUNCH))

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (no MEASURED_PEAKS.json)"
    combos = [(lay, ex) for ex in (False, True) for lay in engines]
    for _ in range(args.warmup):
        for lay, ex in combos:
            step(lay, ex)
    times = {c: [] for c in combos}
    for _ in range(args.steps):                      # alternating: every combination once per round
        for c in combos:
            times[c].append(step(*c))
    result = {"device": gpu_info(args.device), "samples": n, "rows": V, "launch_rows": LAUNCH, "steps": args.steps, "warmup": args.warmup,
              "peak_gbs": peak, "peak_source": peak_src, "runs": {}}
    for (lay, ex), ts in times.items():
        t = float(np.median(ts))
        gbs = launch_bytes(lay) / t / 1e9
        result["runs"][f"{lay}_{'exact' if ex else 'default'}"] = {
            "s_per_pass": t, "s_min": float(np.min(ts)), "s_max": float(np.max(ts)), "genotypes_per_s": n * V / t,
            "algorithmic_gbs": gbs, "hbm_frac": gbs / peak, "bytes_per_pass": launch_bytes(lay),
            "kernel_shape": engines[lay].kernel_shape}

    # cross-check of the two layouts' outputs on the last configuration scored in each mode
    if with_int8:
        check = {}
        for ex in (True, False):
            outs = {}
            for lay in engines:
                step(lay, ex)
                outs[lay] = engines[lay].finish(offset=0.0)
            a, b = outs["bed"], outs["int8"]
            assert a["nloci"] == b["nloci"]
            for f in ("klass", "used", "eaidx", "ngt", "nmiss", "neff"):
                assert np.array_equal(a["loci"][f], b["loci"][f]), f
            sa, sb = a["scores"], b["scores"]
            assert np.array_equal(np.isnan(sa), np.isnan(sb))
            ok = np.isfinite(sb)
            if ex:
                same = np.array_equal(sa[ok].view(np.uint64), sb[ok].view(np.uint64))
                assert same, "exact order: .bed and int8 scores differ in bits"
                check["exact"] = "bit-equal"
            else:
                floor = orc.abs_floor(rows["beta"], b["nloci"])
                ex_ = float((np.abs(sa[ok] - sb[ok]) / (1e-12 * np.abs(sb[ok]) + floor + 1e-300)).max())
                assert ex_ <= 1.0, ex_
                check["default"] = {"max_error_over_tolerance": ex_, "bit_equal_fraction": float(np.mean(sa[ok].view(np.uint64) == sb[ok].view(np.uint64)))}
        result["check"] = check
        for ex in ("default", "exact"):
            result[f"bed_over_int8_{ex}"] = result["runs"][f"bed_{ex}"]["genotypes_per_s"] / result["runs"][f"int8_{ex}"]["genotypes_per_s"]
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    for e in engines.values():
        e.close()


if __name__ == "__main__":
    main()
