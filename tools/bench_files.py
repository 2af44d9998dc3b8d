"""`nimpress` from disk on the same records as one genotype file and as 22 per-contig files (DESIGN.md 4.12).

Writes a cohort of --samples samples and --variants biallelic hard-call variants spread over contigs 1-22, and a score
file naming every variant, as one BGEN file and 22 per-contig BGEN files (zlib, 8 bits), and as one BGZF BCF and 22
per-contig BGZF BCFs, into --dir (a temporary directory by default, removed at the end).  Then runs
`nimpress --exact-order` on each layout, alternating one file / 22 files within each kind, and reports the wall time of
every run and the phase times the driver prints under NIMPRESS_TIMING=1.  The outputs over one file and over 22 files
must be byte-identical.  The device name and power limit are read in the same run.  Prints the result JSON, and also
writes it to --out when given."""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

from bench_bed import gpu_info  # noqa: E402
from util_bcf import write_bcf  # noqa: E402
from util_bgen import records_to_variants, write_bgen  # noqa: E402

EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
CONTIGS = [str(c) for c in range(1, 23)]


def cohort(n, V, seed=5):
    """V biallelic diploid records (BCF GT encoding, 30 % phased hets, 1 % missing), V / 22 per contig."""
    rng = np.random.default_rng(seed)
    recs = []
    for j in range(V):
        c = CONTIGS[j * len(CONTIGS) // V]
        af = rng.uniform(0.01, 0.5)
        al = (rng.random((n, 2)) < af).astype(np.int64)
        g = ((al + 1) << 1) | (rng.random((n, 2)) < 0.3)
        g[:, 0] &= ~1
        g[rng.random(n) < 0.01] = 0
        recs.append(dict(contig=c, pos=1000 + 10 * j, ref="A", alts=["G"], filter="PASS", gt=g.astype(np.int8)))
    return recs


def timed(args):
    t = time.time()
    r = subprocess.run([EXE, "--exact-order", *args], capture_output=True, text=True, env=dict(os.environ, NIMPRESS_TIMING="1"))
    wall = time.time() - t
    assert r.returncode == 0, r.stderr
    phases = {}
    for m in re.finditer(r"\[nimpress timing\] (.+?)\s+([0-9.]+) ms", r.stderr):
        phases[m.group(1).strip()] = phases.get(m.group(1).strip(), 0.0) + float(m.group(2))
    return {"wall_s": wall, "phases_ms": phases}, r.stdout


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--variants", type=int, default=4400)
    ap.add_argument("--samples", type=int, default=50_000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--dir", default=None)
    ap.add_argument("--out", default=None, help="also write the result JSON here")
    args = ap.parse_args()
    work = args.dir or tempfile.mkdtemp(prefix="bench_files_")
    os.makedirs(work, exist_ok=True)
    try:
        n, V = args.samples, args.variants
        t0 = time.time()
        recs = cohort(n, V)
        samples = [f"S{i}" for i in range(n)]
        rng = np.random.default_rng(3)
        score = os.path.join(work, "cohort.score")
        with open(score, "w") as fh:
            fh.write("S\nd\nc\nhs37d5\n0.0\n")
            fh.write("".join(f"{r['contig']}\t{r['pos']}\tA\t{'G' if rng.random() < 0.7 else 'A'}\t{rng.normal(0, 0.05):.4f}\t"
                             f"{rng.uniform(0.01, 0.5):.4f}\n" for r in recs))
        variants = records_to_variants(recs, n, np.random.default_rng(1))
        files = {}
        for kind in ("bgen", "bcf"):
            one = os.path.join(work, f"all.{kind}")
            split = [os.path.join(work, f"chr{c}.{kind}") for c in CONTIGS]
            if kind == "bgen":
                write_bgen(one, samples, variants)
                for c, path in zip(CONTIGS, split):
                    write_bgen(path, samples, [v for v in variants if v["contig"] == c])
            else:
                write_bcf(one, samples, recs, contigs=CONTIGS)
                for c, path in zip(CONTIGS, split):
                    write_bcf(path, samples, [r for r in recs if r["contig"] == c], contigs=CONTIGS)
            files[kind] = {"1": [one], "22": split}
        write_s = time.time() - t0
        runs = {k: {"1": [], "22": []} for k in files}
        for kind in files:
            out = {}
            for _ in range(args.repeats):
                for label in ("1", "22"):
                    res, stdout = timed([score, *files[kind][label]])
                    runs[kind][label].append(res)
                    out.setdefault(label, stdout)
            assert out["1"] == out["22"], f"{kind}: one file and 22 files gave different outputs"
        med = {k: {lab: {"wall_s": float(np.median([x["wall_s"] for x in v])),
                         "stream_ms": float(np.median([x["phases_ms"].get("stream + match + upload", np.nan) for x in v]))}
                   for lab, v in r.items()} for k, r in runs.items()}
        result = {"device": gpu_info(0), "variants": V, "samples": n, "write_s": write_s, "cpu_count": os.cpu_count(),
                  "bytes": {k: {lab: sum(os.path.getsize(p) for p in ps) for lab, ps in f.items()} for k, f in files.items()},
                  "median": med, "runs": runs}
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
