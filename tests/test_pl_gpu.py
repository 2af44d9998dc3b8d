"""GPU tests of FORMAT/PL rows (DESIGN.md 4.10): the C ABI bit for bit against the restatement of tests/util_pl.py
(pinned to the C oracle on decisive likelihoods by tests/test_pl_cpu.py) under every policy, at edge allele
frequencies, across launch cuts, the staging ring, device slabs and a wide cohort; decisive PLs against int8 GT rows; and
the host and CLI on VCF and BCF."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import orc
from util_bgen_bits import hard_cohort
from util_cohort import assert_loci_equal, bits, random_rows
from util_pl import decisive_pl, pack_words, random_pl, reference_scores_pl as oracle, with_pl, write_bcf_pl, write_vcf_pl

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
LOC = ("ps", "homref", "fail", "ignore"); MIS = ("homref", "ignore"); SAM = ("ps", "homref", "fail", "int_ps", "int_fail")
POLICIES = [dict(imp_locus=l, imp_missing=m, imp_sample=s) for l in LOC for m in MIS for s in SAM]
AF_LINE = re.compile(r"^WARN Variant \S+ cohort EAF is (?!0 in ).*\n", re.M)      # the AF-mismatch test of a tallied locus


@pytest.fixture(scope="module")
def nb():
    import __graft_entry__ as g
    g.build()
    import nimpress_b200
    return nimpress_b200


def engine(nb, n, max_rows=4096, n_slots=2, exact=False, pol=None, width=None):
    eng = nb.Engine(n, ploidy=2, gt_width=nb.GT_PL if width is None else width, max_rows_per_block=max_rows, n_slots=n_slots)
    eng.set_policy(**(pol or {}))
    eng.set_exact_order(exact)
    eng.reset()
    return eng


def check(got, want):
    assert got["nloci"] == want["nloci"]
    assert_loci_equal(got["loci"], want["loci"])
    assert np.array_equal(bits(got["scores"]), bits(want["scores"]))     # NaN included: the same bits


def random_words(rng, n, V, pad=5):
    """V rows of n samples (+ pad garbage words never read), per row its own haploid and missing rates, and some words
    that are missing without being 0xFFFFFFFF (bit 31 with other bits, ploidy 0 or 3, j > ploidy)."""
    words = np.zeros((V, n + pad), np.uint32)
    for v in range(V):
        pl, cnt, miss = random_pl(rng, n, haploid_rate=float(rng.choice([0, 0.3, 1])), miss_rate=0.04 * float(rng.uniform(0, 2)))
        w = pack_words(pl, cnt, miss).astype(np.int64)
        odd = rng.random(n) < 0.01
        junk = np.stack([rng.integers(1 << 31, 1 << 32, size=n), rng.integers(0, 1 << 24, size=n),
                         (3 << 26) | rng.integers(0, 1 << 26, size=n), (1 << 26) | (2 << 24) | rng.integers(0, 1 << 24, size=n),
                         (2 << 26) | (3 << 24) | rng.integers(0, 1 << 24, size=n)])
        w = np.where(odd, junk[rng.integers(0, 5, size=n), np.arange(n)], w)
        words[v, :n] = w
        words[v, n:] = rng.integers(0, 1 << 32, size=pad)
    return words


@pytest.mark.parametrize("n", [1, 7, 8, 9, 130, 1001, 2050])
def test_abi_parity_every_policy(nb, n):
    """Scores, records and nloci equal the restatement bit for bit under every policy, exact order on and off alike, with
    ploidy and missing rates mixed across rows; kernel_shape reports mode 7."""
    rng = np.random.default_rng(n)
    words = random_words(rng, n, 61)
    rows = random_rows(rng, 61, n_rows=83, n_alt=1)
    for pol in POLICIES:
        pol = dict(pol, mincs=min(100, max(n - 2, 0)), maxmis=0.05 if n > 100 else 0.5)
        want = oracle(words, n, rows, offset=0.125, **pol)
        for exact in (False, True):
            eng = engine(nb, n, max_rows=128, exact=exact, pol=pol)
            shape = eng.kernel_shape
            assert (shape["fused"], shape["consumer_warps"], shape["chunks_per_thread"]) == (7, 4, 4)
            eng.score_host(words, rows)
            check(eng.finish(offset=0.125), want)
            eng.close()


def test_edge_allele_frequencies(nb):
    """eaf 0, 1, NaN, 1.5 and 1e-300 (every sample missing for NaN and 1.5; p*p underflows at 1e-300) on decisive,
    uninformative and random PLs with mixed ploidy, both effect alleles, maxmis 1 so that the rows are decoded."""
    rng = np.random.default_rng(17)
    n = 1500
    gt, alleles, ploidy = hard_cohort(rng, n, 3, haploid_rate=0.4)
    dec = pack_words(*decisive_pl(alleles[0], ploidy[0], rng))
    uni = pack_words(np.full((n, 3), 9), np.where(ploidy[1] == 1, 2, 3), rng.random(n) < 0.02)
    words = np.stack([dec, uni, random_words(rng, n, 1, pad=0)[0]])
    eafs = [0.0, 1.0, np.nan, 1.5, 1e-300, 0.3]
    rows = np.zeros(len(eafs) * 3 * 2, dtype=orc.ROW_DTYPE)
    i = 0
    for e in eafs:
        for g in range(3):
            for ea in (0, 1):
                rows[i] = (g, ea, 0.01 * (i + 1), e, int(ea == 0), 0)
                i += 1
    for pol in (dict(maxmis=1.0), dict(maxmis=1.0, imp_sample="ps"), dict(maxmis=0.5, imp_locus="homref")):
        want = oracle(words, n, rows, offset=0.5, **pol)
        eng = engine(nb, n, max_rows=64, pol=pol)
        eng.score_host(words, rows)
        check(eng.finish(offset=0.5), want)
        eng.close()
    d = want["loci"]
    assert (d["nmiss"][12:24] == n).all()                  # NaN and 1.5: every sample missing


def test_launch_cuts_ring_device_slabs_and_wide_cohort(nb):
    """npc_score_resident cut at max_rows_per_block (37), blocks of 17 rows through the staging ring,
    npc_score_block_device on a torch slab, and 1,300,000 samples: the sums carry across launches, the bits equal the
    restatement's; the split calls are NPC_EUNSUPPORTED."""
    import torch
    rng = np.random.default_rng(9)
    n, V = 3001, 90
    words = random_words(rng, n, V, pad=3)
    rows = random_rows(rng, V, n_rows=201, n_alt=1)
    want = oracle(words, n, rows, offset=-0.5)
    eng = engine(nb, n, max_rows=37)
    assert eng.resident_reserve(V) >= V
    g8 = words.view(np.uint8)
    for r0 in range(0, V, 37):
        slot, view = eng.stage_acquire()
        nr = min(37, V - r0)
        view[:nr, :g8.shape[1]] = g8[r0:r0 + nr]
        eng.stage_upload(slot, nr, r0)
    eng.score_resident(rows)
    check(eng.finish(offset=-0.5), want)
    eng.close()
    want = oracle(words, n, rows)
    eng = engine(nb, n, max_rows=128, n_slots=3)
    for r0 in range(0, len(rows), 17):
        eng.score_host(words, rows[r0:r0 + 17])
    check(eng.finish(), want)
    eng.close()
    stride = 16384
    dev = torch.zeros((V, stride), dtype=torch.uint8, device="cuda")
    dev[:, :g8.shape[1]] = torch.from_numpy(g8).cuda()
    torch.cuda.synchronize()
    eng = engine(nb, n, max_rows=256)
    eng.score_block_device(dev, stride, V, rows)
    check(eng.finish(), want)
    counts = torch.zeros((len(rows), 2), dtype=torch.int64, device="cuda")
    with pytest.raises(nb.NpcError, match="rc=-5"):
        eng.count_block_device(dev, stride, V, rows, counts)
    with pytest.raises(nb.NpcError, match="rc=-5"):
        eng.accumulate_block_device(dev, stride, V, rows, counts)
    eng.close()
    n = 1_300_000
    words = random_words(rng, n, 24, pad=0)                 # 4n is a multiple of the 128-byte row stride here
    rows = random_rows(rng, 24, n_rows=41, n_alt=1)
    eng = engine(nb, n, max_rows=64)
    eng.score_host(words, rows)
    check(eng.finish(), oracle(words, n, rows))
    eng.close()


def test_decisive_equals_int8_gt_and_multi(nb):
    """Decisive PLs with haploid samples score bit for bit as the same genotypes in int8 GT rows in exact order, records
    equal with neff as the bits of the count; three definitions through npc_score_resident_multi are scored one at a
    time (no contraction) and equal three separate contexts."""
    rng = np.random.default_rng(31)
    n, V = 2003, 60
    gt, alleles, ploidy = hard_cohort(rng, n, V, haploid_rate=0.3)
    words = np.stack([pack_words(*decisive_pl(alleles[v], ploidy[v], rng)) for v in range(V)])
    rows = random_rows(rng, V, n_rows=100, n_alt=1, nan_eaf_rate=0.0)
    for pol in (POLICIES[3], POLICIES[17], POLICIES[38]):
        pol = dict(pol, mincs=100, maxmis=0.05)
        a = engine(nb, n, max_rows=256, pol=pol)
        a.score_host(words, rows)
        got = a.finish(offset=0.5)
        b = engine(nb, n, max_rows=256, exact=True, pol=pol, width=1)
        b.score_host(gt, rows)
        ref = b.finish(offset=0.5)
        a.close(); b.close()
        assert got["nloci"] == ref["nloci"]
        want = ref["loci"].copy()
        want["neff"] = np.where(want["neff"] >= 0, want["neff"].astype(np.float64).view(np.int64), want["neff"])
        assert_loci_equal(got["loci"], want)
        assert np.array_equal(bits(got["scores"]), bits(ref["scores"]))
    lists = [rows, random_rows(rng, V, n_rows=40, n_alt=1), random_rows(rng, V, n_rows=90, n_alt=1)]
    eng = engine(nb, n, max_rows=256)
    assert eng.resident_reserve(V) >= V
    slot, view = eng.stage_acquire()
    g8 = words.view(np.uint8)
    view[:V, :g8.shape[1]] = g8
    eng.stage_upload(slot, V, 0)
    multi = eng.score_resident_multi(lists, [0.25, 0.0, -1.0])
    assert eng.multi_contractions == 0
    for (sc, nloci, loci), r, off in zip(multi, lists, [0.25, 0.0, -1.0]):
        check(dict(scores=sc, nloci=nloci, loci=loci), oracle(words, n, r, offset=off))
    eng.close()


# ---- host and CLI -------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def api(nb):
    from nimpress_b200 import api
    return api


def dataset(tmp, rng, decisive, n=803, V=240, haploid_rate=0.2):
    """make_dataset's cohort with haploid calls, split biallelic (records without an ALT dropped), with GT and PL
    (decisive: the calls' own PLs, and no NaN eaf in the score file), as BGZF VCF text and BCF, its score file and
    coverage BED."""
    from util_bgen_bits import split_records_keep_haploid
    from util_files import make_dataset
    d = make_dataset(tmp, rng, n=n, V=V, haploid_rate=haploid_rate)
    recs = [r for r in split_records_keep_haploid(d["records"]) if len(r["alts"]) == 1]      # PL rows: biallelic records only
    recs = with_pl(recs, n, rng, decisive=decisive)
    contigs = list(dict.fromkeys(r["contig"] for r in d["records"]))
    d["vcf"] = os.path.join(tmp, "pl.vcf.gz")
    write_vcf_pl(d["vcf"], d["samples"], recs, contigs)
    d["bcf"] = os.path.join(tmp, "pl.bcf")
    write_bcf_pl(d["bcf"], d["samples"], recs, contigs)
    d["recs"] = recs
    if decisive:
        # property 1 needs 0 < eaf < 1: a NaN eaf makes every sample of a PL row missing (DESIGN.md 4.10), while its GT calls
        # stay called, so the score file's NaN eafs become 0.5 here
        with open(d["score"]) as fh:
            lines = fh.read().split("\n")
        with open(d["score"], "w") as fh:
            fh.write("\n".join(ln[:-3] + "0.5" if ln.endswith("\tnan") else ln for ln in lines))
    return d


def test_host_decisive_equals_gt_and_cli(api, tmp_path):
    """On decisive PLs, --pl through nph_compute_polygenic_scores scores VCF and BCF as GT does in exact order, with and
    without --cov (records equal with neff as the bits of the count, WARN lines equal but for the AF-mismatch lines of
    tallied loci); and the CLI prints the same lines as --exact-order on the GTs."""
    rng = np.random.default_rng(41)
    d = dataset(str(tmp_path), rng, decisive=True)
    for cov in (None, d["bed"]):
        g = api.run(d["score"], d["vcf"], cov, exact_order=True)
        for geno in (d["vcf"], d["bcf"]):
            p = api.run(d["score"], geno, cov, pl=True)
            assert p.samples == g.samples and p.nloci == g.nloci
            assert p.warnings == AF_LINE.sub("", g.warnings)
            want = g.loci.copy()
            want["neff"] = np.where(want["neff"] >= 0, want["neff"].astype(np.float64).view(np.int64), want["neff"])
            assert_loci_equal(p.loci, want)
            assert np.array_equal(bits(p.scores), bits(g.scores))
    for geno in (d["vcf"], d["bcf"]):
        outs = [subprocess.run(args + [d["score"], geno], capture_output=True, text=True) for args in ([EXE, "--pl"], [EXE, "--exact-order"])]
        assert all(o.returncode == 0 for o in outs), [o.stderr for o in outs]
        assert outs[0].stdout == AF_LINE.sub("", outs[1].stdout)


def read_pl_rows(api, path, n, V, monkeypatch):
    monkeypatch.setenv("NIMPRESS_READ_PL", "1")
    L = api.load_host_library()
    out = np.zeros((V, 4 * n), np.uint8)
    nrec, ns, w, p = C.c_int64(), C.c_int64(), C.c_int32(), C.c_int32()
    assert L.nph_read_gt(os.fsencode(path), out.ctypes.data, out.shape[1], V, C.byref(nrec), C.byref(ns), C.byref(w), C.byref(p)) == 0
    monkeypatch.delenv("NIMPRESS_READ_PL")
    return out[:nrec.value].view("<u4")


def score_rows(entries, recs):
    """Score rows of the restatement for a score file whose entry i names record i (or nothing, i >= len(recs))."""
    rows = np.zeros(len(entries), dtype=orc.ROW_DTYPE)
    for i, e in enumerate(entries):
        hit = i < len(recs)
        rows[i] = (i if hit else -1, (0 if e[3] == e[2] else 1) if hit else -1, e[4], e[5], int(e[2] == e[3]), 0 if hit else 2)
    return rows


def test_host_random_pl_equals_restatement(api, tmp_path, monkeypatch):
    """Random PLs (ties, saturation, haploid and missing samples) through the host on VCF and BCF equal the restatement
    on the rows nph_read_gt returns, bit for bit, under three policies and with NIMPRESS_SPLIT=3 (three contexts, combined
    by npc_reduce) and NIMPRESS_SLAB_ROWS=7 (rounds) as well; no AF-mismatch line is written.  Three score files in one
    pass equal three separate runs."""
    rng = np.random.default_rng(43)
    n, V = 1203, 150
    samples = [f"s{i}" for i in range(n)]
    g = np.full((n, 2), 4, np.int8)
    recs = with_pl([dict(contig="X", pos=1000 + 10 * j, ref="A", alts=["C"], filter="PASS", gt=g) for j in range(V)], n, rng,
                   haploid_rate=0.3)
    vcf, bcf = str(tmp_path / "r.vcf.gz"), str(tmp_path / "r.bcf")
    write_vcf_pl(vcf, samples, recs, ["X"])
    write_bcf_pl(bcf, samples, recs, ["X"])
    words = read_pl_rows(api, vcf, n, V, monkeypatch)
    assert np.array_equal(words, read_pl_rows(api, bcf, n, V, monkeypatch))
    scores = []
    for k in range(3):
        entries = [("X", 1000 + 10 * j, "A", "A" if rng.random() < 0.3 else "C", round(float(rng.normal(0, 0.05)), 4),
                    round(float(rng.uniform(0.01, 0.6)), 4)) for j in range(V)]
        entries += [("X", 5, "A", "C", 0.1, 0.2)]
        path = str(tmp_path / f"s{k}.score")
        with open(path, "w") as fh:
            fh.write("S\nd\nc\nhs37d5\n0.125\n" + "\n".join("\t".join(str(x) for x in e) for e in entries) + "\n")
        scores.append((path, entries))
    path, entries = scores[0]
    rows = score_rows(entries, recs)
    for pol in (dict(), dict(imp_sample="int_fail", maxmis=0.03), dict(imp_locus="homref", imp_sample="ps", maxmis=0.02)):
        kw = dict(maxmis=pol.get("maxmis", 0.05), imp_locus=api.ImputeMethodLocus[pol.get("imp_locus", "ps")],
                  imp_sample=api.ImputeMethodSample[pol.get("imp_sample", "int_ps")])
        want = oracle(words, n, rows, offset=0.125, **pol)
        for geno in (vcf, bcf):
            b = api.run(path, geno, pl=True, **kw)
            assert b.nloci == want["nloci"]
            assert_loci_equal(b.loci, want["loci"])
            assert np.array_equal(bits(b.scores), bits(want["scores"]))
            assert AF_LINE.search(b.warnings) is None
    one = [api.run(p, bcf, pl=True) for p, _ in scores]
    many = api.run_multi([p for p, _ in scores], bcf, pl=True)
    for a, b in zip(one, many):
        assert a.nloci == b.nloci and np.array_equal(bits(a.scores), bits(b.scores))
        assert_loci_equal(a.loci, b.loci)
    monkeypatch.setenv("NIMPRESS_SPLIT", "3")
    b = api.run(path, vcf, pl=True)
    assert b.devices == 3
    assert b.nloci == one[0].nloci and np.allclose(b.scores, one[0].scores, rtol=1e-13, atol=1e-15)
    assert_loci_equal(b.loci, one[0].loci)
    monkeypatch.delenv("NIMPRESS_SPLIT")
    monkeypatch.setenv("NIMPRESS_SLAB_ROWS", "7")
    b = api.run(path, bcf, pl=True)
    assert b.rounds > 2
    assert np.allclose(b.scores, one[0].scores, rtol=1e-13, atol=1e-15)
    assert_loci_equal(b.loci, one[0].loci)


def test_cli_refusals_of_matched_records(tmp_path):
    """A matched record with several ALTs, without PL, or with a sample of 4 PL values exits 1 from the CLI naming the
    variant; unmatched, the file scores."""
    n = 5
    samples = [f"s{i}" for i in range(n)]
    score = str(tmp_path / "f.score")
    with open(score, "w") as fh:
        fh.write("S\nd\nc\nhs37d5\n0.0\n1\t100\tA\tG\t0.1\t0.2\n")
    g = np.full((n, 2), 4, np.int8)
    good = with_pl([dict(contig="1", pos=110, ref="A", alts=["G"], filter="PASS", gt=g)], n, np.random.default_rng(1))[0]
    cases = [(dict(good, alts=["G", "T"]), "biallelic records only"),
             ({k: v for k, v in good.items() if not k.startswith("pl")}, "has no PL field"),
             (dict(good, pltext=["0,1,2", "0,1,2,3", "0,1,2", ".", "0,1,2"]), "4 values")]
    for fmt in ("vcf", "bcf"):
        path = str(tmp_path / f"f.{fmt}")
        for bad, msg in cases:
            if fmt == "bcf" and "pltext" in bad:
                continue
            for pos, rc in ((100, 1), (105, 0)):
                recs = [dict(bad, pos=pos), good]
                (write_vcf_pl if fmt == "vcf" else write_bcf_pl)(path, samples, recs, ["1"])
                r = subprocess.run([EXE, "--pl", score, path], capture_output=True, text=True)
                assert r.returncode == rc and (rc == 0 or ("1:100" in r.stderr and msg in r.stderr)), (fmt, msg, r.returncode, r.stderr)
