"""`nimpress` from disk on a generated BGEN file: ingest time with one worker thread and with all of them (DESIGN.md 4.8).

Writes a zlib-compressed layout-2 file of --variants x --samples (default 10,000 x 100,000; half the variants phased;
imputation-like probabilities: mostly near-certain calls, some uncertain, 1 % missing) and a score file naming every
variant, into --dir (a temporary directory by default, removed at the end).  Then runs `nimpress --exact-order` on it
with NIMPRESS_THREADS=1 and with the default thread count, alternating, and reports the wall time of each run and the
phase times the driver prints under NIMPRESS_TIMING=1 ("stream + match + upload" is the ingest: walking the variant
headers, reading, inflating and converting the matched blocks, and the uploads).  The two runs' outputs must be
byte-identical.  The device name and power limit are read in the same run."""
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from bench_bed import gpu_info  # noqa: E402

EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")


def block(args):
    """One compressed variant block (header + genotype block) of variant j."""
    j, n = args
    rng = np.random.default_rng([7, j])
    phased = j % 2 == 1
    af = rng.uniform(0.01, 0.5)
    if phased:
        alt = rng.random((n, 2)) < af
        h = np.where(alt, 0, 255)
        unsure = rng.random((n, 2)) < 0.1
        h[unsure] = rng.integers(0, 256, size=int(unsure.sum()))
        probs = h
    else:
        nalt = (rng.random((n, 2)) < af).sum(1)
        probs = np.stack([np.where(nalt == 0, 255, 0), np.where(nalt == 1, 255, 0)], 1)
        unsure = rng.random(n) < 0.1
        b0 = rng.integers(0, 256, size=int(unsure.sum()))
        probs[unsure] = np.stack([b0, (rng.random(b0.size) * (256 - b0)).astype(np.int64)], 1)
    miss = rng.random(n) < 0.01
    probs[miss] = 0
    ploidy = np.where(miss, 0x82, 2).astype(np.uint8)
    raw = struct.pack("<IHBB", n, 2, 2, 2) + ploidy.tobytes() + struct.pack("<BB", int(phased), 8) + probs.astype(np.uint8).tobytes()
    z = zlib.compress(raw, 1)
    vid = f"v{j}".encode()
    head = (struct.pack("<H", len(vid)) + vid + struct.pack("<H", len(vid)) + vid + struct.pack("<H", 1) + b"1" +
            struct.pack("<IH", 1000 + 10 * j, 2) + struct.pack("<I", 1) + b"A" + struct.pack("<I", 1) + b"G")
    return head + struct.pack("<II", len(z) + 4, len(raw)) + z


def write_file(path, n, V, procs):
    ids = b"".join(struct.pack("<H", len(s)) + s for s in (f"S{i}".encode() for i in range(n)))
    sblock = struct.pack("<II", 8 + len(ids), n) + ids
    with open(path, "wb") as fh:
        fh.write(struct.pack("<IIII", 20 + len(sblock), 20, V, n) + b"bgen" + struct.pack("<I", 1 | (2 << 2) | 0x80000000) + sblock)
        with mp.Pool(procs) as pool:
            for b in pool.imap(block, ((j, n) for j in range(V)), chunksize=16):
                fh.write(b)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--variants", type=int, default=10_000)
    ap.add_argument("--samples", type=int, default=100_000)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--dir", default=None)
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    args = ap.parse_args()
    work = args.dir or tempfile.mkdtemp(prefix="bench_bgen_")
    os.makedirs(work, exist_ok=True)
    try:
        n, V = args.samples, args.variants
        path, score = os.path.join(work, "cohort.bgen"), os.path.join(work, "cohort.score")
        t0 = time.time()
        write_file(path, n, V, max(1, (os.cpu_count() or 2) - 1))
        rng = np.random.default_rng(3)
        with open(score, "w") as fh:
            fh.write("S\nd\nc\nhs37d5\n0.0\n")
            fh.write("".join(f"1\t{1000 + 10 * j}\tA\t{'G' if rng.random() < 0.7 else 'A'}\t{rng.normal(0, 0.05):.4f}\t{rng.uniform(0.01, 0.5):.4f}\n"
                             for j in range(V)))
        write_s = time.time() - t0
        runs, stdout = {"1": [], "all": []}, {}
        for _ in range(args.repeats):
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
                runs[label].append({"wall_s": wall, "phases_ms": phases})
                stdout.setdefault(label, r.stdout)
        assert stdout["1"] == stdout["all"], "thread counts gave different outputs"
        result = {"device": gpu_info(0), "variants": V, "samples": n, "file_gb": os.path.getsize(path) / 1e9,
                  "uncompressed_gb": V * (10 + 3 * n) / 1e9, "write_s": write_s, "cpu_count": os.cpu_count(), "runs": runs,
                  "ingest_ms": {k: float(np.median([x["phases_ms"].get("stream + match + upload", np.nan) for x in v])) for k, v in runs.items()}}
        line = json.dumps(result)
        print(line)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                fh.write(line + "\n")
    finally:
        if not args.dir:
            shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
