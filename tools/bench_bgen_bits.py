"""32-bit BGEN dosage rows against 2-byte dosage rows and FORMAT/DS rows on one GPU, same cohort and score rows, one
process, alternating; then `nimpress` from disk on a zlib 16-bit BGEN file (DESIGN.md 4.9).

Setup: bench.py's synthetic cohort (npc_synth_fill_device) and score rows, default 20,000 variants x 500,000 samples,
converted on the GPU with torch into four slabs: NPC_GT_DOSE255 rows (k = 255 x ALT alleles; 2 B per genotype),
NPC_GT_DOSE32 rows at D = 255 (the same numerators; 4 B per genotype), NPC_GT_DOSE32 rows at D = 65,535 with every called
k moved by a random -5,000..5,000 inside 0..131,070 (fractional 16-bit data), and FORMAT/DS rows (fp32; 4 B per
genotype).  A step is npc_reset + the rows in launches of at most 32,768 (npc_score_block_device) + a synchronise, timed
with CUDA events; exact order for every layout.  Each slab is read twice per pass (tally, accumulate): bytes of a launch
of R rows = 2 R row_bytes + 32 R + 16 n.  Report, per layout: seconds per pass, genotypes/s, those bytes/s, and the
fraction of the 8 B/genotype bound of 32-bit rows and DS rows (two reads of 4 B) at the HBM peak (MEASURED_PEAKS.json
hbm_gbs, or bench.py's fallback).  Check: D = 255 rows score bit for bit as the 2-byte rows.

Ingest: a zlib-compressed 16-bit file of --ingest-variants x --ingest-samples (default 10,000 x 100,000; half the
variants phased, mostly near-certain calls, 10 % uncertain, 1 % missing) and a score file naming every variant, in a
temporary directory; `nimpress --exact-order` with NIMPRESS_THREADS=1 and with the default thread count, alternating,
under NIMPRESS_TIMING=1 ("stream + match + upload" of the pass that completes is the ingest; the pass restarted on 32-bit
rows is counted in the wall time).  The outputs must be byte-identical.  The device name and power limit are read in
the same run."""
import argparse
import json
import multiprocessing as mp
import os
import re
import shutil
import struct
import subprocess
import sys
import tempfile
import time
import zlib

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from bench_bed import gpu_info  # noqa: E402
from bench_bgen import to_dose255, to_ds  # noqa: E402

LAUNCH = 32768
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")


def to_dose32(torch, g8, n, out32, D, gen=None, jitter=0):
    """int8 diploid rows g8[R, >= 2n] -> 32-bit dosage rows, viewed as int32 out32[R, >= 4 + n]: header D, then
    k | 2 << 24 with k = D x ALT alleles (+ a random -jitter..jitter inside 0..2D), -1 (0xFFFFFFFF) missing."""
    a = (g8[:, :2 * n].view(-1, n, 2).to(torch.int32) >> 1) - 1
    miss = (a < 0).any(-1)
    k = D * (a == 1).sum(-1).to(torch.int32)
    if jitter:
        k = (k + torch.randint(-jitter, jitter + 1, k.shape, device=k.device, generator=gen, dtype=torch.int32)).clamp(0, 2 * D)
    out32[:, :4] = 0
    out32[:, 0] = D
    out32[:, 4:4 + n] = torch.where(miss, -1, k | (2 << 24))


def block16(args):
    """One compressed 16-bit variant block (header + genotype block) of variant j."""
    j, n = args
    rng = np.random.default_rng([16, j])
    D = 65535
    phased = j % 2 == 1
    af = rng.uniform(0.01, 0.5)
    if phased:
        vals = np.where(rng.random((n, 2)) < af, 0, D)
        unsure = rng.random((n, 2)) < 0.1
        vals[unsure] = rng.integers(0, D + 1, size=int(unsure.sum()))
    else:
        nalt = (rng.random((n, 2)) < af).sum(1)
        vals = np.stack([np.where(nalt == 0, D, 0), np.where(nalt == 1, D, 0)], 1)
        unsure = rng.random(n) < 0.1
        b0 = rng.integers(0, D + 1, size=int(unsure.sum()))
        vals[unsure] = np.stack([b0, (rng.random(b0.size) * (D + 1 - b0)).astype(np.int64)], 1)
    miss = rng.random(n) < 0.01
    vals[miss] = 0
    ploidy = np.where(miss, 0x82, 2).astype(np.uint8)
    raw = struct.pack("<IHBB", n, 2, 2, 2) + ploidy.tobytes() + struct.pack("<BB", int(phased), 16) + vals.astype("<u2").tobytes()
    z = zlib.compress(raw, 1)
    vid = f"v{j}".encode()
    head = (struct.pack("<H", len(vid)) + vid + struct.pack("<H", len(vid)) + vid + struct.pack("<H", 1) + b"1" +
            struct.pack("<IH", 1000 + 10 * j, 2) + struct.pack("<I", 1) + b"A" + struct.pack("<I", 1) + b"G")
    return head + struct.pack("<II", len(z) + 4, len(raw)) + z


def ingest(n, V, repeats):
    work = tempfile.mkdtemp(prefix="bench_bgen_bits_")
    try:
        path, score = os.path.join(work, "cohort.bgen"), os.path.join(work, "cohort.score")
        ids = b"".join(struct.pack("<H", len(s)) + s for s in (f"S{i}".encode() for i in range(n)))
        sblock = struct.pack("<II", 8 + len(ids), n) + ids
        with open(path, "wb") as fh:
            fh.write(struct.pack("<IIII", 20 + len(sblock), 20, V, n) + b"bgen" + struct.pack("<I", 1 | (2 << 2) | 0x80000000) + sblock)
            with mp.Pool(max(1, (os.cpu_count() or 2) - 1)) as pool:
                for b in pool.imap(block16, ((j, n) for j in range(V)), chunksize=16):
                    fh.write(b)
        rng = np.random.default_rng(3)
        with open(score, "w") as fh:
            fh.write("S\nd\nc\nhs37d5\n0.0\n")
            fh.write("".join(f"1\t{1000 + 10 * j}\tA\t{'G' if rng.random() < 0.7 else 'A'}\t{rng.normal(0, 0.05):.4f}\t{rng.uniform(0.01, 0.5):.4f}\n"
                             for j in range(V)))
        runs, stdout = {"1": [], "all": []}, {}
        for _ in range(repeats):
            for label in ("1", "all"):
                env = dict(os.environ, NIMPRESS_TIMING="1")
                if label == "1":
                    env["NIMPRESS_THREADS"] = "1"
                else:
                    env.pop("NIMPRESS_THREADS", None)
                t = time.time()
                r = subprocess.run([EXE, "--exact-order", score, path], capture_output=True, text=True, env=env)
                wall = time.time() - t
                assert r.returncode == 0, r.stderr
                phases = {m.group(1).strip(): float(m.group(2)) for m in re.finditer(r"\[nimpress timing\] (.+?)\s+([0-9.]+) ms", r.stderr)}
                runs[label].append({"wall_s": wall, "phases_ms": phases, "restarts": r.stderr.count("restart with 32-bit dosage rows")})
                stdout.setdefault(label, r.stdout)
        assert stdout["1"] == stdout["all"], "thread counts gave different outputs"
        return {"variants": V, "samples": n, "bits": 16, "file_gb": os.path.getsize(path) / 1e9, "cpu_count": os.cpu_count(),
                "runs": runs, "wall_s": {k: float(np.median([x["wall_s"] for x in v])) for k, v in runs.items()},
                "ingest_ms": {k: float(np.median([x["phases_ms"].get("stream + match + upload", np.nan) for x in v])) for k, v in runs.items()}}
    finally:
        shutil.rmtree(work, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=20_000)
    ap.add_argument("--samples", type=int, default=500_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--ingest-variants", type=int, default=10_000, help="0: skip the from-disk ingest")
    ap.add_argument("--ingest-samples", type=int, default=100_000)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    args = ap.parse_args()
    import torch
    import nimpress_b200 as nb
    from bench import SEED, cohort_params, make_rows

    if not torch.cuda.is_available():
        raise SystemExit("bench_bgen_bits.py measures on a GPU: no CUDA device")
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    n, V = args.samples, args.rows
    chunk = 1024
    s2, s4, s32 = -(-2 * n // 128) * 128, -(-4 * n // 128) * 128, -(-(16 + 4 * n) // 128) * 128
    strides = {"dose255": s2, "dose32_d255": s32, "dose32_d65535": s32, "ds": s4}
    row_bytes = {"dose255": 2 * n, "dose32_d255": 16 + 4 * n, "dose32_d65535": 16 + 4 * n, "ds": 4 * n}
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED)

    def engine(layout):
        if layout == "ds":
            e = nb.Engine(n, ploidy=1, gt_width=4, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
            e.set_dosage_rows(True)
        else:
            w = {"int8": 1, "dose255": nb.GT_DOSE255}.get(layout, nb.GT_DOSE32)
            e = nb.Engine(n, gt_width=w, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
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
        return sum(2 * row_bytes[layout] * min(LAUNCH, nv - r0) + 32 * min(LAUNCH, nv - r0) + 16 * n for r0 in range(0, nv, LAUNCH))

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    af, beta, ref_is_ea, af_thr, miss_thr, alt = cohort_params(0, V)
    rows = make_rows(nb.ROW_DTYPE, V, af, beta, ref_is_ea)
    t_af, t_ms, t_alt = (torch.from_numpy(af_thr.view(np.int32)).to(dev), torch.from_numpy(miss_thr.view(np.int32)).to(dev),
                         torch.from_numpy(alt).to(dev))
    rows_rel = rows.copy()
    rows_rel["gt_row"] = np.arange(V) % LAUNCH
    engines = {lay: engine(lay) for lay in strides}
    slabs = {lay: torch.zeros((V, strides[lay]), dtype=torch.uint8, device=dev) for lay in engines}
    filler = engine("int8")
    scratch = torch.empty((chunk, s2), dtype=torch.uint8, device=dev)
    for r0 in range(0, V, chunk):
        nr = min(chunk, V - r0)
        filler.synth_fill_device(scratch, s2, r0, nr, SEED, t_af[r0:], t_ms[r0:], t_alt[r0:])
        g8 = scratch[:nr].view(torch.int8)
        to_dose255(torch, g8, n, slabs["dose255"][r0:r0 + nr].view(torch.int16))
        to_ds(torch, g8, n, slabs["ds"][r0:r0 + nr].view(torch.float32))
        to_dose32(torch, g8, n, slabs["dose32_d255"][r0:r0 + nr].view(torch.int32), 255)
        to_dose32(torch, g8, n, slabs["dose32_d65535"][r0:r0 + nr].view(torch.int32), 65535, gen, 5000)
    del scratch
    filler.close()
    torch.cuda.synchronize()
    for _ in range(args.warmup):
        for lay, e in engines.items():
            step(e, slabs[lay], strides[lay], rows_rel, V)
    times = {lay: [] for lay in engines}
    for _ in range(args.steps):                          # alternating: every layout once per round
        for lay, e in engines.items():
            times[lay].append(step(e, slabs[lay], strides[lay], rows_rel, V))
    bound = 8 * n * V / (peak * 1e9)                     # two reads of 4 B per genotype at the HBM peak
    result = {"device": gpu_info(args.device), "samples": n, "rows": V, "launch_rows": LAUNCH, "steps": args.steps,
              "warmup": args.warmup, "peak_gbs": peak, "peak_source": peak_src, "order": "exact", "runs": {}}
    for lay, ts in times.items():
        t = float(np.median(ts))
        gbs = launch_bytes(lay, V) / t / 1e9
        result["runs"][lay] = {"ms_per_pass": 1e3 * t, "ms_min": 1e3 * float(np.min(ts)), "ms_max": 1e3 * float(np.max(ts)),
                               "genotypes_per_s": n * V / t, "algorithmic_gbs": gbs, "hbm_frac": gbs / peak,
                               "frac_of_8B_bound": bound / t, "kernel_shape": engines[lay].kernel_shape}
    g = {lay: r["genotypes_per_s"] for lay, r in result["runs"].items()}
    result["dose32_d65535_over_ds"] = g["dose32_d65535"] / g["ds"]
    result["dose255_over_dose32_d255"] = g["dose255"] / g["dose32_d255"]
    outs = {}
    for lay in ("dose255", "dose32_d255"):
        step(engines[lay], slabs[lay], strides[lay], rows_rel, V)
        outs[lay] = engines[lay].finish(offset=0.0)
    a, b = outs["dose255"], outs["dose32_d255"]
    assert a["nloci"] == b["nloci"] and np.array_equal(a["scores"].view(np.uint64), b["scores"].view(np.uint64))
    for f in ("klass", "used", "eaidx", "ngt", "nmiss", "neff"):
        assert np.array_equal(a["loci"][f], b["loci"][f]), f
    result["check"] = "dose32 rows at D = 255 bit-equal to dose255 rows: scores and records"
    for e in engines.values():
        e.close()
    del slabs
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    if args.ingest_variants:
        result["ingest"] = ingest(args.ingest_samples, args.ingest_variants, 2)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
