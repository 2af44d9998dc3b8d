"""CPU tests of FORMAT/PL rows (DESIGN.md 4.10): the weight table against Python decimal, the word packer, the rows the
VCF text and BCF readers make (NIMPRESS_READ_PL=1), the refusals, and the numpy restatement the GPU tests pin the
kernels to, against the C oracle on decisive likelihoods.  No GPU needed: nothing here computes a score on a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import orc
from util_bgen_bits import hard_cohort
from util_cohort import assert_loci_equal, bits, random_rows
from util_pl import (MISSING_PL, TN, decisive_pl, dosages, ds_order_sum, pack_words, random_pl, reference_scores_pl,
                     weight, write_bcf_pl, write_vcf_pl)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
POLICIES = [dict(imp_locus=l, imp_missing=m, imp_sample=s) for l in ("ps", "homref", "fail", "ignore")
            for m in ("homref", "ignore") for s in ("ps", "homref", "fail", "int_ps", "int_fail")]


@pytest.fixture(scope="module")
def nb():
    import __graft_entry__ as g
    g.build()
    import nimpress_b200
    return nimpress_b200


@pytest.fixture(scope="module")
def api(nb):
    from nimpress_b200 import api
    api.load_host_library()
    return api


def test_weight_table_is_correctly_rounded(nb):
    """npc_pl_weight_table: every entry for x = 0 .. 4095 is 10^(-x/10) computed with decimal at 60 digits and rounded
    once (the same double at 90 digits), 0 from 3237 on, whose neighbour 3236 is the smallest subnormal."""
    T = nb.pl_weight_table(4096)
    want = np.array([weight(x) if x < TN else 0.0 for x in range(4096)])
    assert np.array_equal(bits(T), bits(want))
    assert all(weight(x, 90) == want[x] for x in range(0, TN, 7))
    assert T[0] == 1.0 and T[10] == 0.1 and T[TN - 1] == 2.0 ** -1074 and weight(TN) == 0.0
    naive = 10.0 ** (-np.arange(TN) / 10.0)                    # the rounded exponent moves the result: not the table
    assert (bits(naive) != bits(T[:TN])).sum() > 1000


def test_pack_words_by_hand():
    """a | b << 12 | j << 24 | ploidy << 26: ties take the first minimum, values saturate at 4095 above the minimum,
    a haploid sample has b = 0, a missing one is 0xFFFFFFFF."""
    pl = np.array([[0, 10, 100], [30, 0, 45], [7, 7, 0], [5, 5, 5], [9000, 20, 10000], [3, 0, 0], [0, 40, 0], [12, 0, 99],
                   [1, 2, 3]])
    cnt = np.array([3, 3, 3, 3, 3, 2, 2, 2, 3])
    miss = np.array([0, 0, 0, 0, 0, 0, 0, 0, 1], bool)
    w = pack_words(pl, cnt, miss)
    assert w.tolist() == [10 | 100 << 12 | 0 << 24 | 2 << 26, 30 | 45 << 12 | 1 << 24 | 2 << 26, 7 | 7 << 12 | 2 << 24 | 2 << 26,
                          0 | 0 << 12 | 0 << 24 | 2 << 26, 4095 | 4095 << 12 | 1 << 24 | 2 << 26, 3 | 1 << 24 | 1 << 26,
                          40 | 0 << 24 | 1 << 26, 12 | 1 << 24 | 1 << 26, MISSING_PL]


def read_pl(api, path, n, V, monkeypatch, threads=1):
    monkeypatch.setenv("NIMPRESS_READ_PL", "1")
    monkeypatch.setenv("NIMPRESS_THREADS", str(threads))
    L = api.load_host_library()
    out = np.full((V + 2, 4 * n), 0xAB, np.uint8)
    nrec, ns, w, p = C.c_int64(), C.c_int64(), C.c_int32(-1), C.c_int32()
    rc = L.nph_read_gt(os.fsencode(path), out.ctypes.data, out.shape[1], V + 2, C.byref(nrec), C.byref(ns), C.byref(w), C.byref(p))
    monkeypatch.delenv("NIMPRESS_READ_PL")
    err = L.nph_last_error().decode()
    return rc, err, out[:nrec.value].view("<u4"), w.value, p.value


def pl_records(rng, n, V, hi, haploid_rate=0.2):
    from util_pl import with_pl
    g = np.full((n, 2), 4, np.int8)
    recs = [dict(contig="1", pos=100 + 10 * j, ref="A", alts=["G"], filter="PASS", gt=g) for j in range(V)]
    return with_pl(recs, n, rng, haploid_rate=haploid_rate, hi=hi)


@pytest.mark.parametrize("threads", [1, 8])
def test_reader_rows_vcf_and_bcf(api, tmp_path, monkeypatch, threads):
    """VCF text (plain and BGZF) and BCF with PL as int8, int16 and int32 give the same rows, the packer's words: ties,
    saturated values, haploid samples, "." and one-"."-value missing samples; gt_width 10, ploidy 2."""
    rng = np.random.default_rng(threads)
    n, V = 37, 25
    for hi, widths in ((120, (1, 2, 4)), (70000, (4,))):
        recs = pl_records(rng, n, V, hi)
        want = np.stack([pack_words(r["pl"], r["plcnt"], r["plmiss"]) for r in recs])
        samples = [f"s{i}" for i in range(n)]
        paths = [str(tmp_path / "a.vcf"), str(tmp_path / "a.vcf.gz")]
        write_vcf_pl(paths[0], samples, recs, ["1"], compress=None)
        write_vcf_pl(paths[1], samples, recs, ["1"], compress="bgzf")
        for wd in widths:
            paths.append(str(tmp_path / f"a{wd}.bcf"))
            write_bcf_pl(paths[-1], samples, recs, ["1"], pl_width=wd)
        for path in paths:
            rc, err, rows, w, p = read_pl(api, path, n, V, monkeypatch, threads)
            assert rc == 0, (path, err)
            assert (w, p) == (10, 2) and rows.shape == (V, n)
            assert np.array_equal(rows, want), path


def test_reader_pl_only_format(api, tmp_path, monkeypatch):
    """PL as the only FORMAT field of a VCF text record, and PL after GT, give the same rows."""
    rng = np.random.default_rng(3)
    n, V = 20, 6
    recs = pl_records(rng, n, V, 300)
    a, b = str(tmp_path / "a.vcf"), str(tmp_path / "b.vcf")
    samples = [f"s{i}" for i in range(n)]
    write_vcf_pl(a, samples, recs, ["1"], compress=None)
    write_vcf_pl(b, samples, recs, ["1"], compress=None, with_gt=False)
    ra, rb = read_pl(api, a, n, V, monkeypatch), read_pl(api, b, n, V, monkeypatch)
    assert ra[0] == rb[0] == 0 and np.array_equal(ra[2], rb[2])


@pytest.mark.parametrize("fmt", ["vcf", "bcf"])
def test_reader_refusals(api, tmp_path, monkeypatch, fmt):
    """A sample with 1 or 4 PL values, or a negative one, is an input error naming the variant and the sample; text that
    is not an integer too (VCF text)."""
    n = 4
    samples = [f"s{i}" for i in range(n)]
    base = dict(contig="1", pos=100, ref="A", alts=["G"], filter="PASS", gt=np.full((n, 2), 4, np.int8),
                pl=np.array([[0, 10, 20]] * n), plcnt=np.full(n, 3), plmiss=np.zeros(n, bool), plpartial=np.zeros(n, bool))
    cases = [("1 values", ["0,10,20", "5", "0,1,2", "."]), ("4 values", ["0,10,20", "0,1,2,3", "0,1,2", "."]),
             ("negative value -3", ["0,10,20", "0,-3,2", "0,1,2", "."])]
    if fmt == "vcf":
        cases.append(("is not an integer", ["0,1x,2", "0,1,2", "0,1,2", "."]))
    for msg, texts in cases:
        path = str(tmp_path / f"r.{fmt}")
        rec = dict(base, pltext=texts)
        if fmt == "vcf":
            write_vcf_pl(path, samples, [rec], ["1"], compress=None)
        else:
            pl = np.zeros((n, 4), np.int64)
            cnt = np.zeros(n, np.int64)
            for i, t in enumerate(texts):
                vals = [] if t == "." else [int(x) for x in t.split(",")]
                pl[i, :len(vals)] = vals
                cnt[i] = len(vals)
            write_bcf_raw_pl(path, samples, rec, pl, cnt)
        rc, err, _, _, _ = read_pl(api, path, n, 1, monkeypatch)
        assert rc == -3 and msg in err and "1:100" in err and "sample s" in err, (msg, rc, err)


def write_bcf_raw_pl(path, samples, rec, pl, cnt):
    """One BCF record whose PL field has up to 4 int8 values per sample (vector_end padded; none = ".")."""
    from util_pl import write_bcf_pl
    n = len(samples)
    L = int(max(cnt.max(), 1))
    r = dict(rec, pl=pl[:, :L], plcnt=cnt, plmiss=cnt == 0, plpartial=np.zeros(n, bool))
    write_bcf_pl(path, samples, [r], ["1"], pl_width=1)


def test_cli_option_refusals(tmp_path):
    """--pl with --dosage, and --pl on a PLINK fileset or a BGEN file, exit 1 with the reason."""
    from util_bgen import write_bgen, genotype_block
    from util_plink import write_plink
    score = str(tmp_path / "s.score")
    with open(score, "w") as fh:
        fh.write("S\nd\nc\nhs37d5\n0.0\n1\t100\tA\tG\t0.1\t0.2\n")
    vcf = str(tmp_path / "a.vcf")
    n = 3
    samples = [f"s{i}" for i in range(n)]
    write_vcf_pl(vcf, samples, pl_records(np.random.default_rng(1), n, 2, 50), ["1"], compress=None)
    r = subprocess.run([EXE, "--pl", "--dosage", score, vcf], capture_output=True, text=True)
    assert r.returncode == 1 and "--pl and --dosage" in r.stderr, r.stderr
    probs, miss = np.full((n, 2), 0), np.zeros(n, bool)
    bg = write_bgen(str(tmp_path / "a.bgen"), samples, [dict(contig="1", pos=100, alleles=["A", "G"],
                                                           block=genotype_block(n, probs, miss, False))])
    r = subprocess.run([EXE, "--pl", score, bg], capture_output=True, text=True)
    assert r.returncode == 1 and "--pl: a BGEN file" in r.stderr, r.stderr
    bed = write_plink(str(tmp_path / "p"), samples, [dict(contig="1", pos=100, ref="A", alts=["G"], gt=np.full((n, 2), 4, np.int8))])
    r = subprocess.run([EXE, "--pl", score, bed], capture_output=True, text=True)
    assert r.returncode == 1 and "--pl: a PLINK fileset" in r.stderr, r.stderr


@pytest.mark.parametrize("n", [1, 9, 300, 1030])
def test_decisive_restatement_equals_oracle(n):
    """Property 1 of DESIGN.md 4.10: decisive PLs give d in {0, 1, 2} exactly.  The restatement on such rows equals the
    C oracle on the same genotypes as int8 GT rows (haploid samples included) bit for bit under all 40 policies, records
    equal with neff as the bits of the count; and, on a diploid cohort, the oracle's FORMAT/DS path on those dosages as
    fp32 DS rows, records and neff bits included (which pins the tally order)."""
    rng = np.random.default_rng(n)
    V = 40
    for haploid_rate in (0.3, 0.0):
        gt, alleles, ploidy = hard_cohort(rng, n, V, haploid_rate=haploid_rate)
        words = np.stack([pack_words(*decisive_pl(alleles[v], ploidy[v], rng)) for v in range(V)])
        rows = random_rows(rng, V, n_rows=70, n_alt=1, nan_eaf_rate=0.0)
        rows["eaf"] = np.clip(rows["eaf"], 0.01, 0.99)
        if haploid_rate == 0.0:
            ds = np.full((V, n), np.nan, np.float32)
            for v in range(V):
                d, called = dosages(words[v], 0.3, 1)
                assert set(np.unique(d[called])) <= {0.0, 1.0, 2.0}
                ds[v] = np.where(called, d, np.nan).astype(np.float32)
        for pol in POLICIES:
            pol = dict(pol, mincs=min(100, max(n - 2, 0)), maxmis=0.05 if n > 100 else 0.5)
            want = reference_scores_pl(words, n, rows, offset=0.25, **pol)
            ref = orc.score_matrix(gt, n, 2, rows, offset=0.25, **pol)
            assert want["nloci"] == ref["nloci"]
            assert np.array_equal(bits(want["scores"]), bits(ref["scores"]))
            loci = ref["loci"].copy()
            loci["neff"] = np.where(loci["neff"] >= 0, loci["neff"].astype(np.float64).view(np.int64), loci["neff"])
            assert_loci_equal(want["loci"], loci)
            if haploid_rate == 0.0:
                dsr = orc.score_matrix(ds, n, 2, rows, offset=0.25, **pol)
                assert want["nloci"] == dsr["nloci"]
                assert np.array_equal(bits(want["scores"]), bits(dsr["scores"]))
                assert_loci_equal(want["loci"], dsr["loci"])


def test_uninformative_gives_ps_and_ds_order():
    """Property 2: all-equal PLs give d within a few ulp of 2 eaf (eaf haploid), for ALT and REF effect alleles; and the
    DS-order sum of ds_order_sum is the chunked, butterflied, block-ordered sum."""
    for eaf in (1e-6, 0.01, 0.1234, 0.5, 0.77, 0.999999):
        for cnt in (3, 2):
            w = pack_words(np.full((1, 3), 17), [cnt], [False])
            for eaidx in (1, 0):                                       # eaf is the effect allele's frequency either way
                d, called = dosages(w, eaf, eaidx)
                assert called[0]
                want = (cnt - 1) * eaf
                assert abs(d[0] - want) <= 4 * np.spacing(want), (eaf, cnt, eaidx, d[0], want)
    rng = np.random.default_rng(2)
    d = rng.random(700)
    c = rng.random(700) < 0.9
    want = 0.0
    for b in range(3):
        v = []
        for lane in range(32):
            s = 0.0
            for k in range(8):
                i = b * 256 + lane * 8 + k
                if i < 700 and c[i]:
                    s += d[i]
            v.append(s)
        for o in (16, 8, 4, 2, 1):
            v = [v[i] + v[i ^ o] for i in range(32)]
        want += v[0]
    assert ds_order_sum(d, c) == want
