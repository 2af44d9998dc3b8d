"""BGEN fixed-point dosage rows against int8 GT rows in exact order and FORMAT/DS rows on one GPU: the same cohort and
score rows, scored in one process, alternating (DESIGN.md 4.8).

Setup: bench.py's synthetic cohort (npc_synth_fill_device) and score rows, default 20,000 variants x 500,000 samples.
The int8 rows are converted on the GPU with torch: to dosage rows (k = 255 x ALT alleles, 0xFFFF missing; 2 B per
genotype), to DS rows (fp32 ALT allele count, NaN missing; 4 B per genotype), and to a fractional copy of the dosage
rows (every called k moved by a random -40..40 inside 0..510, so that the table lookups of the accumulate pass spread
over the table as imputed data does).  A step is npc_reset + the rows in launches of at most 32,768
(npc_score_block_device) + a synchronise, timed with CUDA events.

Report, per layout: seconds per pass, genotypes/s, algorithmic bytes/s and the fraction of the HBM bound.  Bytes of a
launch of R rows over n samples: int8 = 2 n R + 32 R + 16 n (bench.py's definition: one read of the slab); dose255 =
2 (2 n R) + 32 R + 16 n and ds = 2 (4 n R) + 32 R + 16 n (each row read twice: tally pass and accumulate pass).  The peak
is MEASURED_PEAKS.json hbm_gbs, with bench.py's fallback.  The device name and power limit are read in the same run.

Check: the hard-call dosage rows and the DS rows score bit for bit as the int8 rows in exact order (fl(k/255) and the
DS values are the exact allele counts); records are equal except neff (255 x for dosage rows, the fp64 bits for DS).

Then, with the other slabs freed, one pass over the --shard-rows x samples cohort as dosage rows alone (125,000 x
500,000 = 125 GB by default)."""
import argparse
import json
import os
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from bench_bed import gpu_info  # noqa: E402

LAUNCH = 32768


def to_dose255(torch, g8, n, out):
    """int8 diploid rows g8[R, >= 2n] -> uint16 numerators out[R, >= n] (viewed as int16)."""
    a = (g8[:, :2 * n].view(-1, n, 2).to(torch.int32) >> 1) - 1
    k = torch.where((a < 0).any(-1), 0xFFFF, 255 * (a == 1).sum(-1))
    out[:, :n] = k.to(torch.int32).to(torch.int16)          # 0xFFFF wraps to -1: the same 16 bits


def to_ds(torch, g8, n, out):
    a = (g8[:, :2 * n].view(-1, n, 2).to(torch.int32) >> 1) - 1
    out[:, :n] = torch.where((a < 0).any(-1), float("nan"), (a == 1).sum(-1).to(torch.float32))


def fractional(torch, k16, n, gen):
    """Called numerators moved by a random -40..40 inside 0..510 (in place)."""
    k = k16[:, :n].to(torch.int32) & 0xFFFF
    j = torch.randint(-40, 41, k.shape, device=k.device, generator=gen, dtype=torch.int32)
    k16[:, :n] = torch.where(k > 510, k, (k + j).clamp(0, 510)).to(torch.int16)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=20_000)
    ap.add_argument("--samples", type=int, default=500_000)
    ap.add_argument("--shard-rows", type=int, default=125_000, help="0: skip the dosage-only shard pass")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    args = ap.parse_args()
    import torch
    import nimpress_b200 as nb
    from bench import SEED, cohort_params, make_rows

    if not torch.cuda.is_available():
        raise SystemExit("bench_bgen.py measures on a GPU: no CUDA device")
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    n, V = args.samples, args.rows
    chunk = 1024
    strides = {"int8": -(-2 * n // 128) * 128, "dose255": -(-2 * n // 128) * 128, "dose255_frac": -(-2 * n // 128) * 128,
               "ds": -(-4 * n // 128) * 128}
    per_row = {"int8": 2 * n, "dose255": 4 * n, "dose255_frac": 4 * n, "ds": 8 * n}
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED)

    def params(v0, nv):
        af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(v0, nv)
        rows = make_rows(nb.ROW_DTYPE, nv, af, beta, ref_is_ea)
        return rows, (torch.from_numpy(af_thr.view(np.int32)).to(dev), torch.from_numpy(miss_thr.view(np.int32)).to(dev),
                      torch.from_numpy(alt).to(dev))

    def engine(layout):
        if layout == "ds":
            e = nb.Engine(n, ploidy=1, gt_width=4, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
            e.set_dosage_rows(True)
        else:
            e = nb.Engine(n, gt_width=1 if layout == "int8" else nb.GT_DOSE255, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
        e.set_stream(stream.cuda_stream)
        e.set_policy()
        e.set_exact_order(True)
        return e

    def step(e, slab, st, rows_rel, nv):
        e.reset()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for r0 in range(0, nv, LAUNCH):
            nr = min(LAUNCH, nv - r0)
            e.score_block_device(slab.data_ptr() + r0 * st, st, nr, rows_rel[r0:r0 + nr])
        b.record(stream)
        b.synchronize()
        return a.elapsed_time(b) * 1e-3

    def launch_bytes(layout, nv):
        return sum(per_row[layout] * min(LAUNCH, nv - r0) + 32 * min(LAUNCH, nv - r0) + 16 * n for r0 in range(0, nv, LAUNCH))

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    # ---- the alternating comparison -------------------------------------------------------------------------------
    rows, (t_af, t_ms, t_alt) = params(0, V)
    rows_rel = rows.copy()
    rows_rel["gt_row"] = np.arange(V) % LAUNCH
    engines = {lay: engine(lay) for lay in ("dose255", "dose255_frac", "int8", "ds")}
    slabs = {lay: torch.zeros((V, strides[lay]), dtype=torch.uint8, device=dev) for lay in engines}
    engines["int8"].synth_fill_device(slabs["int8"], strides["int8"], 0, V, SEED, t_af, t_ms, t_alt)
    g8 = slabs["int8"].view(torch.int8)
    for r0 in range(0, V, chunk):
        to_dose255(torch, g8[r0:r0 + chunk], n, slabs["dose255"][r0:r0 + chunk].view(torch.int16))
        to_ds(torch, g8[r0:r0 + chunk], n, slabs["ds"][r0:r0 + chunk].view(torch.float32))
    slabs["dose255_frac"].copy_(slabs["dose255"])
    for r0 in range(0, V, chunk):
        fractional(torch, slabs["dose255_frac"][r0:r0 + chunk].view(torch.int16), n, gen)
    torch.cuda.synchronize()
    for _ in range(args.warmup):
        for lay, e in engines.items():
            step(e, slabs[lay], strides[lay], rows_rel, V)
    times = {lay: [] for lay in engines}
    for _ in range(args.steps):                          # alternating: every layout once per round
        for lay, e in engines.items():
            times[lay].append(step(e, slabs[lay], strides[lay], rows_rel, V))
    result = {"device": gpu_info(args.device), "samples": n, "rows": V, "launch_rows": LAUNCH, "steps": args.steps,
              "warmup": args.warmup, "peak_gbs": peak, "peak_source": peak_src, "order": "exact", "runs": {}}
    for lay, ts in times.items():
        t = float(np.median(ts))
        gbs = launch_bytes(lay, V) / t / 1e9
        result["runs"][lay] = {"s_per_pass": t, "s_min": float(np.min(ts)), "s_max": float(np.max(ts)), "genotypes_per_s": n * V / t,
                               "algorithmic_gbs": gbs, "hbm_frac": gbs / peak, "bytes_per_pass": launch_bytes(lay, V),
                               "kernel_shape": engines[lay].kernel_shape}
    result["dose255_over_ds"] = result["runs"]["dose255"]["genotypes_per_s"] / result["runs"]["ds"]["genotypes_per_s"]
    result["dose255_frac_over_ds"] = result["runs"]["dose255_frac"]["genotypes_per_s"] / result["runs"]["ds"]["genotypes_per_s"]
    # check: hard-call dosage rows and DS rows against the int8 rows, exact order
    outs = {}
    for lay in ("int8", "dose255", "ds"):
        step(engines[lay], slabs[lay], strides[lay], rows_rel, V)
        outs[lay] = engines[lay].finish(offset=0.0)
    ref = outs["int8"]
    for lay in ("dose255", "ds"):
        o = outs[lay]
        assert o["nloci"] == ref["nloci"]
        for f in ("klass", "used", "eaidx", "ngt", "nmiss"):
            assert np.array_equal(o["loci"][f], ref["loci"][f]), (lay, f)
        if lay == "dose255":
            assert np.array_equal(o["loci"]["neff"], np.where(ref["loci"]["neff"] >= 0, 255 * ref["loci"]["neff"], ref["loci"]["neff"]))
        assert np.array_equal(o["scores"].view(np.uint64), ref["scores"].view(np.uint64)), f"{lay}: scores differ from int8 in bits"
    result["check"] = "dose255 and ds scores bit-equal to int8 exact order; records equal (neff scaled)"
    for e in engines.values():
        e.close()
    del slabs, g8
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    # ---- the shard as dosage rows alone --------------------------------------------------------------------------
    if args.shard_rows:
        VS = args.shard_rows
        rows, (t_af, t_ms, t_alt) = params(0, VS)
        rows_rel = rows.copy()
        rows_rel["gt_row"] = np.arange(VS) % LAUNCH
        e, filler = engine("dose255"), engine("int8")                # the synthetic cohort is made as int8 rows
        slab = torch.empty((VS, strides["dose255"]), dtype=torch.uint8, device=dev)
        scratch = torch.empty((chunk, strides["int8"]), dtype=torch.uint8, device=dev)
        for r0 in range(0, VS, chunk):
            nr = min(chunk, VS - r0)
            filler.synth_fill_device(scratch, strides["int8"], r0, nr, SEED, t_af[r0:], t_ms[r0:], t_alt[r0:])
            to_dose255(torch, scratch[:nr].view(torch.int8), n, slab[r0:r0 + nr].view(torch.int16))
        del scratch
        torch.cuda.synchronize()
        filler.close()
        step(e, slab, strides["dose255"], rows_rel, VS)                  # warm-up
        ts = [step(e, slab, strides["dose255"], rows_rel, VS) for _ in range(max(1, min(args.steps, 3)))]
        t = float(np.median(ts))
        gbs = launch_bytes("dose255", VS) / t / 1e9
        result["shard"] = {"rows": VS, "slab_gb": VS * strides["dose255"] / 1e9, "s_per_pass": t, "s_all": ts,
                           "genotypes_per_s": n * VS / t, "algorithmic_gbs": gbs, "hbm_frac": gbs / peak}
        e.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
