"""FORMAT/PL rows against FORMAT/DS rows and 32-bit BGEN dosage rows on one GPU, same cohort and score rows, one process,
alternating; then `nimpress --pl` from disk on a BCF with PL (DESIGN.md 4.10).

Setup: bench.py's synthetic cohort (npc_synth_fill_device) and score rows, default 20,000 variants x 500,000 samples,
converted on the GPU with torch into three slabs of 4 B per genotype: NPC_GT_PL rows (the called genotype's PL is 0,
the other two random in 10..99, so every sample goes through the full posterior; missing calls 0xFFFFFFFF), FORMAT/DS
rows (fp32 ALT count) and NPC_GT_DOSE32 rows at D = 65,535.  A step is npc_reset + the rows in launches of at most
32,768 (npc_score_block_device) + a synchronise, timed with CUDA events; exact order for every layout.  Each slab is read
twice per pass (tally, accumulate).  Report, per layout: ms per pass, genotypes/s, and the fraction of the 8 B/genotype
bound (two reads of 4 B) at the HBM peak (MEASURED_PEAKS.json hbm_gbs, or the 7.7 TB/s of the data sheet).

Ingest: a BGZF BCF of --ingest-variants x --ingest-samples (default 10,000 x 100,000) with GT and int16 PL (1 % missing,
10 % haploid samples) and a score file naming every variant, in a temporary directory; `nimpress --pl` with
NIMPRESS_THREADS=1 and with the default thread count, alternating, under NIMPRESS_TIMING=1 ("stream + match + upload" is
the ingest).  The outputs must be byte-identical.  The device name and power limit are read in the same run."""
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
from bench_bgen import to_ds  # noqa: E402
from bench_bgen_bits import to_dose32  # noqa: E402

LAUNCH = 32768
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
N_ING = 0


def to_pl(torch, g8, n, out32, gen):
    """int8 diploid rows g8[R, >= 2n] -> PL words out32[R, >= n]: j = the ALT count, a and b random in 10..99."""
    a = (g8[:, :2 * n].view(-1, n, 2).to(torch.int32) >> 1) - 1
    miss = (a < 0).any(-1)
    j = (a == 1).sum(-1).to(torch.int32)
    ab = torch.randint(10, 100, (2,) + j.shape, device=j.device, generator=gen, dtype=torch.int32)
    out32[:, :n] = torch.where(miss, -1, ab[0] | (ab[1] << 12) | (j << 24) | (2 << 26))


def _bgzf(data, level=1):
    out = bytearray()
    for i in range(0, len(data), 0xFF00):
        chunk = data[i:i + 0xFF00]
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        comp = co.compress(chunk) + co.flush()
        out += struct.pack("<4BI2BH2BHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, len(comp) + 25) + comp
        out += struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk))
    return bytes(out)


def bcf_group(j0):
    """BGZF bytes of 16 BCF records from variant j0: GT (int8) then PL (int16, 3 per sample)."""
    n = N_ING
    out = bytearray()
    for j in range(j0, j0 + 16):
        rng = np.random.default_rng([7, j])
        af = rng.uniform(0.01, 0.5)
        g = (rng.random((n, 2)) < af).astype(np.int16)
        gt = (((g + 1) << 1)).astype(np.int8)
        hap = rng.random(n) < 0.1
        gt[hap, 1] = -127
        pl = rng.integers(10, 400, size=(n, 3)).astype(np.int16)
        k = np.where(hap, g[:, 0], g.sum(1))
        pl[np.arange(n), k] = 0
        pl[hap, 2] = -32767
        miss = rng.random(n) < 0.01
        pl[miss, 0] = -32768
        pl[miss, 1:] = -32767
        gt[miss] = 0
        shared = struct.pack("<iiif", 0, 1000 + 10 * j - 1, 1, float("nan")) + struct.pack("<II", 2 << 16, (2 << 24) | n)
        shared += bytes([0x07]) + bytes([0x17]) + b"A" + bytes([0x17]) + b"G" + bytes([0x00])
        indiv = bytes([0x11, 1, 0x21]) + gt.tobytes() + bytes([0x11, 2, 0x32]) + pl.tobytes()    # dictionary: PASS, GT, PL
        out += struct.pack("<II", len(shared), len(indiv)) + shared + indiv
    return _bgzf(bytes(out))


def _init(n):
    global N_ING
    N_ING = n


def ingest(n, V, repeats):
    work = tempfile.mkdtemp(prefix="bench_pl_")
    try:
        path, score = os.path.join(work, "cohort.bcf"), os.path.join(work, "cohort.score")
        hdr = ["##fileformat=VCFv4.2", '##FILTER=<ID=PASS,Description="All filters passed">', "##contig=<ID=1>",
               '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
               '##FORMAT=<ID=PL,Number=G,Type=Integer,Description="Phred-scaled genotype likelihoods">',
               "\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + [f"S{i}" for i in range(n)])]
        text = ("\n".join(hdr) + "\n").encode() + b"\0"
        V = -(-V // 16) * 16
        with open(path, "wb") as fh:
            fh.write(_bgzf(b"BCF\2\2" + struct.pack("<I", len(text)) + text))
            with mp.Pool(max(1, (os.cpu_count() or 2) - 1), initializer=_init, initargs=(n,)) as pool:
                for b in pool.imap(bcf_group, range(0, V, 16)):
                    fh.write(b)
            fh.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
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
                r = subprocess.run([EXE, "--pl", score, path], capture_output=True, text=True, env=env)
                wall = time.time() - t
                assert r.returncode == 0, r.stderr
                phases = {m.group(1).strip(): float(m.group(2)) for m in re.finditer(r"\[nimpress timing\] (.+?)\s+([0-9.]+) ms", r.stderr)}
                runs[label].append({"wall_s": wall, "phases_ms": phases})
                stdout.setdefault(label, r.stdout)
        assert stdout["1"] == stdout["all"], "thread counts gave different outputs"
        return {"variants": V, "samples": n, "pl_width": 2, "file_gb": os.path.getsize(path) / 1e9, "cpu_count": os.cpu_count(),
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
        raise SystemExit("bench_pl.py measures on a GPU: no CUDA device")
    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    n, V = args.samples, args.rows
    chunk = 1024
    s2, s4, s32 = -(-2 * n // 128) * 128, -(-4 * n // 128) * 128, -(-(16 + 4 * n) // 128) * 128
    strides = {"pl": s4, "ds": s4, "dose32": s32}
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED)

    def engine(layout):
        if layout == "ds":
            e = nb.Engine(n, ploidy=1, gt_width=4, max_rows_per_block=LAUNCH, n_slots=0, device=args.device)
            e.set_dosage_rows(True)
        else:
            w = {"int8": 1, "pl": nb.GT_PL, "dose32": nb.GT_DOSE32}[layout]
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

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 7700.0, "data sheet (HGX B200, one GPU)"

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
        to_pl(torch, g8, n, slabs["pl"][r0:r0 + nr].view(torch.int32), gen)
        to_ds(torch, g8, n, slabs["ds"][r0:r0 + nr].view(torch.float32))
        to_dose32(torch, g8, n, slabs["dose32"][r0:r0 + nr].view(torch.int32), 65535, gen, 5000)
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
        result["runs"][lay] = {"ms_per_pass": 1e3 * t, "ms_min": 1e3 * float(np.min(ts)), "ms_max": 1e3 * float(np.max(ts)),
                               "genotypes_per_s": n * V / t, "frac_of_8B_bound": bound / t,
                               "kernel_shape": engines[lay].kernel_shape}
    g = {lay: r["genotypes_per_s"] for lay, r in result["runs"].items()}
    result["pl_over_ds"] = g["pl"] / g["ds"]
    result["pl_over_dose32"] = g["pl"] / g["dose32"]
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
