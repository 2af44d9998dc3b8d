"""GPU tests of 32-bit fixed-point dosage rows (DESIGN.md 4.9): BGEN blocks at 1 to 16 bits per probability, haploid
and diploid samples.  The quotient fl(k'/D) against numpy for every k' and every bit depth, the C ABI bit for bit against
the restatement of tests/util_bgen_bits.py (pinned to the C oracle on hard calls by tests/test_bgen_bits_cpu.py), D = 255
rows against 2-byte rows, hard calls against int8 GT rows, and the host and CLI on .bgen files against the equivalent VCF
and BCF."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import orc
from util_bgen import write_bgen
from util_bgen_bits import (MISSING32, dose32_rows, genotype_block_bits, hard_cohort, hard_values, numerators,
                            random_values, records_to_variants_bits, reference_scores_dose32 as oracle, refusal_blocks,
                            split_records_keep_haploid)
from util_cohort import assert_loci_equal, bits, random_rows

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
LOC = ("ps", "homref", "fail", "ignore"); MIS = ("homref", "ignore"); SAM = ("ps", "homref", "fail", "int_ps", "int_fail")
POLICIES = [dict(imp_locus=l, imp_missing=m, imp_sample=s) for l in LOC for m in MIS for s in SAM]
AF_LINE = re.compile(r"^WARN Variant \S+ cohort EAF is (?!0 in ).*\n", re.M)      # the AF-mismatch test of a tallied locus
RESTART = "restart with 32-bit dosage rows"


@pytest.fixture(scope="module")
def nb():
    import __graft_entry__ as g
    g.build()
    import nimpress_b200
    return nimpress_b200


def engine(nb, n, max_rows=4096, n_slots=2, exact=False, pol=None, width=None):
    eng = nb.Engine(n, ploidy=2, gt_width=width or nb.GT_DOSE32, max_rows_per_block=max_rows, n_slots=n_slots)
    eng.set_policy(**(pol or {}))
    eng.set_exact_order(exact)
    eng.reset()
    return eng


def check(got, want):
    assert got["nloci"] == want["nloci"]
    assert_loci_equal(got["loci"], want["loci"])
    assert np.array_equal(bits(got["scores"]), bits(want["scores"]))     # NaN included: the same bits


def random_words(rng, n, V, pad=5):
    """V rows of n samples (+ pad garbage words never read): per row its own bit depth, phasing, haploid / ploidy-0 /
    missing rates; some words that are missing without being 0xFFFFFFFF (bit 31 with other bits, ploidy 0 or 3,
    k > p*D) -> (words uint32[V, n + pad], D[V])."""
    words = np.zeros((V, n + pad), np.uint32)
    D = np.zeros(V, np.int64)
    for v in range(V):
        B = int(rng.integers(1, 17))
        D[v] = (1 << B) - 1
        phased = bool(rng.random() < 0.5)
        vals, ploidy, miss = random_values(rng, n, B, phased, haploid_rate=float(rng.choice([0, 0.3, 1])),
                                           ploidy0_rate=0.01, miss_rate=0.04 * float(rng.uniform(0, 2)))
        w = numerators(vals, ploidy, miss, phased, B).astype(np.int64)
        odd = rng.random(n) < 0.01
        p = rng.integers(1, 3, size=n)
        junk = np.stack([rng.integers(1 << 31, 1 << 32, size=n), rng.integers(0, 1 << 24, size=n),
                         (3 << 24) | rng.integers(0, 1 << 24, size=n),
                         (p << 24) | (p * D[v] + 1 + rng.integers(0, 1 << 23, size=n) % ((1 << 24) - p * D[v] - 1))])
        w = np.where(odd, junk[rng.integers(0, 4, size=n), np.arange(n)], w)
        words[v, :n] = w
        words[v, n:] = rng.integers(0, 1 << 32, size=pad)
    return words, D


def test_exhaustive_quotient(nb):
    """For every bit depth B and every k' in 0..2D (diploid) and 0..D (haploid), with effect allele ALT and REF: a row
    scored alone with beta = 1 leaves fl(k'/D) in the raw sums, bit for bit numpy's correctly rounded division."""
    for B in range(1, 17):
        D = (1 << B) - 1
        n = 2 * D + 1
        s = np.arange(n, dtype=np.int64)
        for p, k in ((2, s), (1, s % (D + 1))):
            words = (k | p << 24).astype(np.uint32)[None, :]
            for eaidx in (0, 1):
                rows = np.zeros(1, dtype=orc.ROW_DTYPE)
                rows[0] = (0, eaidx, 1.0, 0.3, 0, 0)
                eng = engine(nb, n, max_rows=4)
                eng.score_host(dose32_rows(words, [D]), rows)
                got = eng.partial()["sums"]
                eng.close()
                kk = p * D - k if eaidx == 0 else k
                want = kk.astype(np.float64) / float(D)
                bad = np.nonzero(bits(got) != bits(want))[0]
                assert bad.size == 0, (B, p, eaidx, kk[bad[:5]], got[bad[:5]], want[bad[:5]])


@pytest.mark.parametrize("n", [1, 7, 8, 9, 130, 1001, 2050])
def test_abi_parity_every_policy(nb, n):
    """Scores, records and nloci equal the restatement bit for bit under every policy, exact order on and off alike, with
    bit depth, phasing and ploidy mixed across rows; kernel_shape reports mode 6."""
    rng = np.random.default_rng(n)
    words, D = random_words(rng, n, 61)
    g = dose32_rows(words, D, rng=rng)
    rows = random_rows(rng, 61, n_rows=83, n_alt=1)
    for pol in POLICIES:
        pol = dict(pol, mincs=min(100, max(n - 2, 0)), maxmis=0.05 if n > 100 else 0.5)
        want = oracle(words, D, n, rows, offset=0.125, **pol)
        for exact in (False, True):
            eng = engine(nb, n, max_rows=128, exact=exact, pol=pol)
            shape = eng.kernel_shape
            assert (shape["fused"], shape["consumer_warps"], shape["chunks_per_thread"]) == (6, 4, 4)
            eng.score_host(g, rows)
            check(eng.finish(offset=0.125), want)
            eng.close()


def test_d255_rows_equal_dose255_context(nb):
    """D = 255 rows of diploid samples score bit for bit as the same numerators in 2-byte rows, records included."""
    rng = np.random.default_rng(255)
    n, V = 3001, 70
    k = rng.integers(0, 511, size=(V, n))
    k[rng.random((V, n)) < 0.3] = 255 * rng.integers(0, 3, size=1)
    miss = rng.random((V, n)) < 0.03
    k16 = np.where(miss, 0xFFFF, k).astype(np.uint16)
    words = np.where(miss, MISSING32, k | 2 << 24).astype(np.uint32)
    rows = random_rows(rng, V, n_rows=120, n_alt=1)
    for pol in (POLICIES[3], POLICIES[17], POLICIES[38]):
        a = engine(nb, n, max_rows=256, pol=pol)
        a.score_host(dose32_rows(words, np.full(V, 255)), rows)
        b = engine(nb, n, max_rows=256, pol=pol, width=nb.GT_DOSE255)
        b.score_host(k16, rows)
        check(a.finish(offset=0.5), b.finish(offset=0.5))
        a.close(); b.close()


@pytest.mark.parametrize("B", [1, 3, 16])
def test_hard_calls_equal_int8_gt(nb, B):
    """Hard calls with haploid samples (int8 GT: allele then vector_end) at B bits score bit for bit as the int8 GT rows in
    exact order; the records are equal except that neff is D x the GT neff."""
    rng = np.random.default_rng(B)
    n, V, D = 1001, 50, (1 << B) - 1
    gt, alleles, ploidy = hard_cohort(rng, n, V, haploid_rate=0.3)
    words = np.stack([numerators(*hard_values(alleles[v], ploidy[v], bool(v % 2), B), bool(v % 2), B) for v in range(V)])
    rows = random_rows(rng, V, n_rows=90, n_alt=1)
    for pol in (POLICIES[3], POLICIES[17], POLICIES[38]):
        pol = dict(pol, mincs=100, maxmis=0.05)
        a = engine(nb, n, max_rows=256, exact=True, pol=pol)
        a.score_host(dose32_rows(words, np.full(V, D)), rows)
        got = a.finish(offset=0.5)
        b = engine(nb, n, max_rows=256, exact=True, pol=pol, width=1)
        b.score_host(gt, rows)
        ref = b.finish(offset=0.5)
        a.close(); b.close()
        assert got["nloci"] == ref["nloci"]
        want = ref["loci"].copy()
        want["neff"] = np.where(want["neff"] >= 0, want["neff"] * D, want["neff"])
        assert_loci_equal(got["loci"], want)
        assert np.array_equal(bits(got["scores"]), bits(ref["scores"]))


def test_launch_cuts_ring_device_slabs_and_wide_cohort(nb):
    """npc_score_resident cut at max_rows_per_block (37), blocks of 17 rows through the staging ring,
    npc_score_block_device on a torch slab, and 1,300,000 samples: the sums carry across launches, the bits equal the
    restatement's; the split calls are NPC_EUNSUPPORTED."""
    import torch
    rng = np.random.default_rng(9)
    n, V = 3001, 90
    words, D = random_words(rng, n, V, pad=0)
    g = dose32_rows(words, D)
    rows = random_rows(rng, V, n_rows=201, n_alt=1)
    want = oracle(words, D, n, rows, offset=-0.5)
    eng = engine(nb, n, max_rows=37)
    assert eng.resident_reserve(V) >= V
    for r0 in range(0, V, 37):
        slot, view = eng.stage_acquire()
        nr = min(37, V - r0)
        view[:nr, :g.shape[1]] = g[r0:r0 + nr]
        eng.stage_upload(slot, nr, r0)
    eng.score_resident(rows)
    check(eng.finish(offset=-0.5), want)
    eng.close()
    want = oracle(words, D, n, rows)
    eng = engine(nb, n, max_rows=128, n_slots=3)
    for r0 in range(0, len(rows), 17):
        eng.score_host(g, rows[r0:r0 + 17])
    check(eng.finish(), want)
    eng.close()
    stride = 16384
    dev = torch.zeros((V, stride), dtype=torch.uint8, device="cuda")
    dev[:, :g.shape[1]] = torch.from_numpy(g).cuda()
    torch.cuda.synchronize()
    eng = engine(nb, n, max_rows=256)
    eng.score_block_device(dev, stride, V, rows)
    check(eng.finish(), want)
    counts = torch.zeros((len(rows), 2), dtype=torch.int64, device="cuda")
    with pytest.raises(nb.NpcError, match="rc=-5"):
        eng.count_block_device(dev, stride, V, rows, counts)
    eng.close()
    n = 1_300_000
    words, D = random_words(rng, n, 24)
    rows = random_rows(rng, 24, n_rows=41, n_alt=1)
    eng = engine(nb, n, max_rows=64)
    eng.score_host(dose32_rows(words, D), rows)
    check(eng.finish(), oracle(words, D, n, rows))
    eng.close()


# ---- host and CLI -------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def api(nb):
    from nimpress_b200 import api
    return api


def dataset(tmp, rng, B, haploid_rate, n=803, V=240):
    """make_dataset's cohort with haploid calls, split biallelic and all-PASS, as VCF, BCF and a hard-call .bgen at B
    bits."""
    from util_bcf import write_bcf, write_vcf
    from util_files import make_dataset
    d = make_dataset(tmp, rng, n=n, V=V, haploid_rate=haploid_rate)
    recs = split_records_keep_haploid(d["records"])
    contigs = list(dict.fromkeys(r["contig"] for r in d["records"]))
    d["vcf"] = os.path.join(tmp, "split.vcf.gz")
    write_vcf(d["vcf"], d["samples"], recs, contigs=contigs, compress="bgzf")
    d["bcf"] = os.path.join(tmp, "split.bcf")
    write_bcf(d["bcf"], d["samples"], recs, contigs=contigs, compress="bgzf")
    d["bgen"] = write_bgen(os.path.join(tmp, "split.bgen"), d["samples"], records_to_variants_bits(recs, n, B, rng))
    return d


def same(b, v, D):
    """b on the .bgen, v on the equivalent VCF / BCF in exact order: the same samples, nloci, score bits, records with
    neff scaled by D, and WARN lines once the AF-mismatch lines of tallied loci are removed."""
    assert b.samples == v.samples and b.nloci == v.nloci
    assert b.warnings == AF_LINE.sub("", v.warnings)
    want = v.loci.copy()
    want["neff"] = np.where(want["neff"] >= 0, want["neff"] * D, want["neff"])
    assert_loci_equal(b.loci, want)
    assert np.array_equal(bits(b.scores), bits(v.scores))


@pytest.mark.parametrize("B, haploid_rate", [(16, 0.0), (8, 0.5), (16, 0.5)])
def test_host_bgen_equals_vcf_and_bcf(api, tmp_path, B, haploid_rate):
    """A hard-call .bgen at 16 bits, and chrX-like files whose "males" are haploid at 8 and 16 bits, score through
    nph_compute_polygenic_scores and the CLI as the equivalent VCF and BCF in exact order, with and without --cov."""
    rng = np.random.default_rng(B + int(10 * haploid_rate))
    d = dataset(str(tmp_path), rng, B, haploid_rate)
    D = (1 << B) - 1
    for cov in (None, d["bed"]):
        b = api.run(d["score"], d["bgen"], cov, exact_order=True)
        for geno in (d["vcf"], d["bcf"]):
            same(b, api.run(d["score"], geno, cov, exact_order=True), D)
        same(api.run(d["score"], d["bgen"], cov), api.run(d["score"], d["vcf"], cov, exact_order=True), D)
    outs = [subprocess.run([EXE, "--exact-order", d["score"], g], capture_output=True, text=True) for g in (d["bgen"], d["vcf"])]
    assert all(o.returncode == 0 for o in outs), [o.stderr for o in outs]
    assert outs[0].stdout == AF_LINE.sub("", outs[1].stdout)


def read_dose32(api, path, n, V, monkeypatch):
    monkeypatch.setenv("NIMPRESS_READ_DOSE32", "1")
    L = api.load_host_library()
    out = np.zeros((V, 16 + 4 * n), np.uint8)
    nrec, ns, w, pl = C.c_int64(), C.c_int64(), C.c_int32(), C.c_int32()
    assert L.nph_read_gt(os.fsencode(path), out.ctypes.data, out.shape[1], V, C.byref(nrec), C.byref(ns), C.byref(w), C.byref(pl)) == 0
    monkeypatch.delenv("NIMPRESS_READ_DOSE32")
    return out[:, 16:].copy().view("<u4"), out[:, :4].copy().view("<u4")[:, 0]


def fractional_file(tmp, rng, n, V, depth):
    """A fractional .bgen (mixed phasing and ploidy, missing samples); depth(j): bit depth of variant j; and its score
    file (REF or ALT effect alleles, two absent loci) -> (path, score, entries)."""
    samples = [f"s{i}" for i in range(n)]
    variants, entries = [], []
    for j in range(V):
        B = depth(j)
        phased = bool(rng.random() < 0.5)
        vals, ploidy, miss = random_values(rng, n, B, phased, haploid_rate=0.3 if B != 8 else 0.0)
        variants.append(dict(contig="X", pos=1000 + 10 * j, alleles=["A", "C"], block=genotype_block_bits(n, vals, ploidy, miss, phased, B)))
        ea = "A" if rng.random() < 0.3 else "C"
        entries.append(("X", 1000 + 10 * j, "A", ea, round(float(rng.normal(0, 0.05)), 4), round(float(rng.uniform(0.01, 0.5)), 4)))
    entries += [("X", 5, "A", "C", 0.1, 0.2), ("X", 1000, "A", "G", 0.1, 0.2)]                      # absent
    path = write_bgen(os.path.join(tmp, "f.bgen"), samples, variants)
    score = os.path.join(tmp, "f.score")
    with open(score, "w") as fh:
        fh.write("S\nd\nc\nhs37d5\n0.125\n" + "\n".join("\t".join(str(x) for x in e) for e in entries) + "\n")
    return path, score, entries


def score_rows(entries, V):
    rows = np.zeros(len(entries), dtype=orc.ROW_DTYPE)
    for i, e in enumerate(entries):
        hit = i < V
        rows[i] = (i if hit else -1, (0 if e[3] == "A" else 1) if hit else -1, e[4], e[5], int(e[2] == e[3]), 0 if hit else 2)
    return rows


@pytest.mark.parametrize("mixed", [False, True])
def test_fractional_host_equals_restatement(api, tmp_path, monkeypatch, mixed):
    """A fractional 16-bit .bgen, and one whose first matched blocks are 8-bit diploid and later ones 16-bit with haploid
    samples, through the host equal the restatement on the rows nph_read_gt returns, bit for bit, with the blocks
    converted on eight worker threads; no AF-mismatch line is written.  Under NIMPRESS_TIMING=1 the CLI reports one
    restart to 32-bit rows for the mixed file."""
    monkeypatch.setenv("NIMPRESS_THREADS", "8")
    rng = np.random.default_rng(5 + mixed)
    n, V = 2003, 120
    path, score, entries = fractional_file(str(tmp_path), rng, n, V, (lambda j: 8 if j < 60 else 16) if mixed else (lambda j: 16))
    words, D = read_dose32(api, path, n, V, monkeypatch)
    rows = score_rows(entries, V)
    for pol in (dict(), dict(imp_sample="int_fail", maxmis=0.03), dict(imp_locus="homref", imp_sample="ps", maxmis=0.02)):
        kw = dict(maxmis=pol.get("maxmis", 0.05), imp_locus=api.ImputeMethodLocus[pol.get("imp_locus", "ps")],
                  imp_sample=api.ImputeMethodSample[pol.get("imp_sample", "int_ps")])
        b = api.run(score, path, exact_order=bool(pol), **kw)
        want = oracle(words, D, n, rows, offset=0.125, **pol)
        assert b.nloci == want["nloci"]
        assert_loci_equal(b.loci, want["loci"])
        assert np.array_equal(bits(b.scores), bits(want["scores"]))
        assert AF_LINE.search(b.warnings) is None
    r = subprocess.run([EXE, score, path], capture_output=True, text=True, env=dict(os.environ, NIMPRESS_TIMING="1"))
    assert r.returncode == 0 and r.stderr.count(RESTART) == 1, r.stderr


def test_8bit_diploid_file_does_not_restart(tmp_path):
    """An 8-bit diploid file stays on 2-byte rows: no restart line."""
    rng = np.random.default_rng(8)
    path, score, _ = fractional_file(str(tmp_path), rng, 301, 40, lambda j: 8)
    r = subprocess.run([EXE, score, path], capture_output=True, text=True, env=dict(os.environ, NIMPRESS_TIMING="1"))
    assert r.returncode == 0 and RESTART not in r.stderr and "[nimpress timing]" in r.stderr, r.stderr


def test_split_contexts_on_16bit_file(api, tmp_path, monkeypatch):
    """NIMPRESS_SPLIT=2 (two contexts, combined by npc_reduce) and NIMPRESS_SLAB_ROWS=7 (scoring in rounds) on a 16-bit
    file with haploid samples score as the equivalent BCF does under the same settings."""
    rng = np.random.default_rng(16)
    d = dataset(str(tmp_path), rng, 16, 0.3, n=1203, V=300)
    monkeypatch.setenv("NIMPRESS_SPLIT", "2")
    b = api.run(d["score"], d["bgen"], d["bed"], exact_order=True)
    assert b.devices == 2
    same(b, api.run(d["score"], d["bcf"], d["bed"], exact_order=True), 65535)
    monkeypatch.delenv("NIMPRESS_SPLIT")
    monkeypatch.setenv("NIMPRESS_SLAB_ROWS", "7")
    b = api.run(d["score"], d["bgen"], d["bed"], exact_order=True)
    v = api.run(d["score"], d["bcf"], d["bed"], exact_order=True)
    assert b.rounds > 2 and b.rounds == v.rounds
    same(b, v, 65535)


def test_cli_refusals_of_streamed_blocks(tmp_path):
    """A matched block that no dosage row holds exits 1 from the CLI, naming the variant; unmatched, the file scores."""
    n = 9
    samples = [f"s{i}" for i in range(n)]
    path = str(tmp_path / "f.bgen")
    score = str(tmp_path / "f.score")
    with open(score, "w") as fh:
        fh.write("S\nd\nc\nhs37d5\n0.0\n1\t100\tA\tG\t0.1\t0.2\n")
    good, cases = refusal_blocks(n, np.random.default_rng(4))
    rest = [dict(contig="1", pos=110 + 10 * j, alleles=["A", "G"], block=good) for j in range(3)]
    write_bgen(path, samples, [dict(contig="1", pos=100, alleles=["A", "G"], block=good)] + rest)
    assert subprocess.run([EXE, score, path], capture_output=True, text=True).returncode == 0
    for blk, msg in cases:
        write_bgen(path, samples, [dict(contig="1", pos=100, alleles=["A", "G"], block=blk)] + rest)
        r = subprocess.run([EXE, score, path], capture_output=True, text=True)
        assert r.returncode == 1 and msg in r.stderr and "1:100 (v0)" in r.stderr, (msg, r.returncode, r.stderr)
        write_bgen(path, samples, [dict(contig="1", pos=105, alleles=["A", "G"], block=blk)] + rest)
        r = subprocess.run([EXE, score, path], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
