"""CPU tests of BGEN blocks at 1 to 16 bits per probability and with haploid samples (DESIGN.md 4.9): the writer of
tests/util_bgen_bits.py against the 8-bit one, the 32-bit dosage rows the reader makes (NIMPRESS_READ_DOSE32=1), the
refusals, and the numpy restatement the GPU tests pin the kernels to.  No GPU needed: nothing here computes a score."""
import ctypes as C
import os

import numpy as np
import pytest

from util_bgen import genotype_block, random_probs, write_bgen
from util_bgen_bits import (MISSING32, genotype_block_bits, hard_cohort, hard_values, numerators, pack_values,
                            random_values, reference_scores_dose32, refusal_blocks)

GT_DOSE32 = 32
POLICIES = [dict(imp_locus=l, imp_missing=m, imp_sample=s) for l in ("ps", "homref", "fail", "ignore")
            for m in ("homref", "ignore") for s in ("ps", "homref", "fail", "int_ps", "int_fail")]


@pytest.fixture(scope="module")
def api():
    import __graft_entry__ as g
    g.build()
    from nimpress_b200 import api
    api.load_host_library()
    return api


def read_gt(api, path, row_bytes, max_records=256):
    L = api.load_host_library()
    out = np.full((max_records, row_bytes), 0xAB, np.uint8)
    nrec, ns, w, pl = C.c_int64(), C.c_int64(), C.c_int32(-1), C.c_int32()
    rc = L.nph_read_gt(os.fsencode(path), out.ctypes.data, row_bytes, max_records, C.byref(nrec), C.byref(ns), C.byref(w), C.byref(pl))
    return rc, out[:nrec.value], ns.value, w.value, pl.value


def test_writer_at_8_and_16_bits():
    """At 8 bits the writer's bytes are util_bgen.genotype_block's; at 16 bits each value is a little-endian uint16; the
    bit stream is least-significant bit first."""
    rng = np.random.default_rng(1)
    for n in (1, 9, 100):
        for phased in (False, True):
            probs, miss = random_probs(rng, n, phased)
            assert genotype_block_bits(n, probs, np.full(n, 2), miss, phased, 8) == genotype_block(n, probs, miss, phased)
    vals, ploidy, miss = random_values(rng, 50, 16, False, haploid_rate=0.3, ploidy0_rate=0.1)
    blk = genotype_block_bits(50, vals, ploidy, miss, False, 16)
    stored = np.concatenate([vals[i, :ploidy[i]] for i in range(50)])
    assert blk[8 + 50 + 2:] == stored.astype("<u2").tobytes()
    assert pack_values([1, 0, 3, 5], 3) == bytes([0b11000001, 0b00001010])      # 001 000 011 101, low bit first
    assert pack_values([1], 1) == b"\x01"


def test_numerators_conventions():
    """Hand-worked words: unphased 2D - 2*b0 - b1, phased (D - h0) + (D - h1), haploid D - b0, each | ploidy << 24;
    missing and ploidy 0 are 0xFFFFFFFF."""
    vals = np.array([[3, 0], [0, 3], [1, 1], [2, 0], [0, 0], [1, 2]])
    ploidy = np.array([2, 2, 2, 1, 0, 2])
    miss = np.array([0, 0, 0, 0, 0, 1], bool)
    w = numerators(vals, ploidy, miss, False, 2)
    assert w.tolist() == [0 | 2 << 24, 3 | 2 << 24, 3 | 2 << 24, 1 | 1 << 24, MISSING32, MISSING32]
    w = numerators(vals, ploidy, miss, True, 2)
    assert w.tolist() == [3 | 2 << 24, 3 | 2 << 24, 4 | 2 << 24, 1 | 1 << 24, MISSING32, MISSING32]


def _variants(rng, n, B, V=12, **kw):
    variants, words = [], []
    for j in range(V):
        phased = bool(j % 2)
        vals, ploidy, miss = random_values(rng, n, B, phased, **kw)
        variants.append(dict(contig="1", pos=100 + j, alleles=["A", "G"], block=genotype_block_bits(n, vals, ploidy, miss, phased, B)))
        words.append(numerators(vals, ploidy, miss, phased, B))
    return variants, np.stack(words)


@pytest.mark.parametrize("B", [1, 2, 3, 7, 8, 9, 12, 15, 16])
@pytest.mark.parametrize("compression", ["none", "zlib"])
def test_read_dose32_rows(api, tmp_path, monkeypatch, B, compression):
    """nph_read_gt with NIMPRESS_READ_DOSE32=1: per block the row header (D = 2^B - 1, 12 zero bytes) and the words of
    numpy's numerators; phased and unphased, haploid, diploid, ploidy-0 and missing samples, in blocks whose samples are
    all diploid, all haploid or mixed; NIMPRESS_THREADS 1 and 8 give the same bytes; nothing is written past a row."""
    monkeypatch.setenv("NIMPRESS_READ_DOSE32", "1")
    rng = np.random.default_rng(B * 7 + len(compression))
    n = 301
    samples = [f"id{i}" for i in range(n)]
    v1, w1 = _variants(rng, n, B, haploid_rate=0.3, ploidy0_rate=0.05)
    v2, w2 = _variants(rng, n, B, V=4)
    v3, w3 = _variants(rng, n, B, V=4, haploid_rate=1.0)
    words = np.concatenate([w1, w2, w3])
    path = write_bgen(str(tmp_path / "b.bgen"), samples, v1 + v2 + v3, compression=compression)
    rb = 16 + 4 * n + 32
    outs = []
    for threads in ("1", "8"):
        monkeypatch.setenv("NIMPRESS_THREADS", threads)
        rc, rows, ns, w, pl = read_gt(api, path, rb)
        assert rc == 0 and ns == n and (w, pl) == (GT_DOSE32, 2) and rows.shape[0] == len(words)
        assert (rows[:, :4].copy().view("<u4")[:, 0] == (1 << B) - 1).all() and (rows[:, 4:16] == 0).all()
        assert np.array_equal(rows[:, 16:16 + 4 * n].copy().view("<u4"), words)
        assert (rows[:, 16 + 4 * n:] == 0xAB).all()
        outs.append(rows)
    assert np.array_equal(outs[0], outs[1])


def test_default_read_still_refuses(api, tmp_path, monkeypatch):
    """Without NIMPRESS_READ_DOSE32, nph_read_gt keeps 2-byte rows: a well-formed 16-bit or haploid block is refused,
    naming the variant and what the rows cannot hold."""
    monkeypatch.delenv("NIMPRESS_READ_DOSE32", raising=False)
    rng = np.random.default_rng(3)
    n = 9
    for B, hap, msg in ((16, 0.0, "16 bits"), (8, 0.5, "ploidy 1..2")):
        vals, ploidy, miss = random_values(rng, n, B, False, haploid_rate=hap)
        ploidy[:2] = (1, 2) if hap else 2
        path = write_bgen(str(tmp_path / "r.bgen"), [f"s{i}" for i in range(n)],
                          [dict(contig="1", pos=100, alleles=["A", "G"], block=genotype_block_bits(n, vals, ploidy, miss, False, B))])
        rc, *_ = read_gt(api, path, 2 * n + 16)
        err = api.load_host_library().nph_last_error().decode()
        assert rc == -3 and msg in err and "1:100 (v0)" in err, err


def test_refusals(api, tmp_path, monkeypatch):
    """A block that 32-bit rows cannot hold either is NPH_EINPUT from nph_read_gt with NIMPRESS_READ_DOSE32=1, naming the
    variant: K != 2, B of 0 or 17, Pmax > 2, a sample's ploidy outside [Pmin, Pmax], an unphased b0 + b1 > D, a stored N
    other than N, and a block too short for its samples (the message names the bit depth).  tests/test_bgen_bits_gpu.py
    checks the CLI's exit code on the same blocks."""
    n = 9
    samples = [f"s{i}" for i in range(n)]
    path = str(tmp_path / "f.bgen")
    good, cases = refusal_blocks(n, np.random.default_rng(4))
    rest = [dict(contig="1", pos=110 + 10 * j, alleles=["A", "G"], block=good) for j in range(3)]
    L = api.load_host_library()
    monkeypatch.setenv("NIMPRESS_READ_DOSE32", "1")
    write_bgen(path, samples, [dict(contig="1", pos=100, alleles=["A", "G"], block=good)] + rest)
    assert read_gt(api, path, 16 + 4 * n)[0] == 0
    for blk, msg in cases:
        write_bgen(path, samples, [dict(contig="1", pos=100, alleles=["A", "G"], block=blk)] + rest)
        rc, *_ = read_gt(api, path, 16 + 4 * n)
        err = L.nph_last_error().decode()
        assert rc == -3 and msg in err and "1:100 (v0)" in err, (msg, err)


@pytest.mark.parametrize("n", [1, 9, 130, 1001])
def test_restatement_equals_dose255_restatement(n):
    """On D = 255 rows of diploid samples, reference_scores_dose32 equals util_bgen.reference_scores under all 40
    policies: scores, nloci and records."""
    from util_bgen import reference_scores
    rng = np.random.default_rng(n)
    V = 30
    k = rng.integers(0, 511, size=(V, n))
    k[rng.random((V, n)) < 0.2] = 255 * rng.integers(0, 3, size=1)
    miss = rng.random((V, n)) < 0.04
    k[miss] = 0xFFFF
    words = np.where(miss, MISSING32, k | 2 << 24).astype(np.uint32)
    from util_cohort import random_rows
    rows = random_rows(rng, V, n_rows=50, n_alt=1)
    for pol in POLICIES:
        pol = dict(pol, mincs=min(100, max(n - 2, 0)), maxmis=0.05 if n > 100 else 0.5)
        a = reference_scores(k.astype(np.uint16), n, rows, offset=0.25, **pol)
        b = reference_scores_dose32(words, np.full(V, 255), n, rows, offset=0.25, **pol)
        assert a["nloci"] == b["nloci"]
        for f in ("klass", "used", "eaidx", "ngt", "nmiss", "neff"):
            assert np.array_equal(a["loci"][f], b["loci"][f]), f
        assert np.array_equal(np.isnan(a["loci"]["imputed"]), np.isnan(b["loci"]["imputed"]))
        ok = ~np.isnan(a["loci"]["imputed"])
        assert np.array_equal(a["loci"]["imputed"][ok], b["loci"]["imputed"][ok])
        assert np.array_equal(a["scores"].view(np.uint64), b["scores"].view(np.uint64))


@pytest.mark.parametrize("n", [1, 9, 130, 1001])
def test_restatement_equals_oracle_on_hard_calls(n):
    """reference_scores_dose32 equals the C oracle on the same hard calls as int8 GT rows, a haploid sample written as
    allele then vector_end, under all 40 policies, at 1, 3 and 16 bits: scores bit for bit, nloci, and records with
    neff = D x the GT neff."""
    import orc
    from util_cohort import random_rows
    rng = np.random.default_rng(n + 11)
    V = 40
    gt, alleles, ploidy = hard_cohort(rng, n, V, haploid_rate=0.3)
    rows = random_rows(rng, V, n_rows=70, n_alt=1)
    for B in (1, 3, 16):
        D = (1 << B) - 1
        words = np.stack([numerators(*hard_values(alleles[v], ploidy[v], bool(v % 2), B), bool(v % 2), B) for v in range(V)])
        for pol in POLICIES:
            pol = dict(pol, mincs=min(100, max(n - 2, 0)), maxmis=0.05 if n > 100 else 0.5)
            got = reference_scores_dose32(words, np.full(V, D), n, rows, offset=0.25, **pol)
            want = orc.score_matrix(gt, n, 2, rows.astype(orc.ROW_DTYPE), offset=0.25, **pol)
            assert got["nloci"] == want["nloci"]
            g, w = got["loci"], want["loci"]
            for f in ("klass", "used", "eaidx", "ngt", "nmiss"):
                assert np.array_equal(g[f], w[f]), f
            assert np.array_equal(g["neff"], np.where(w["neff"] >= 0, D * w["neff"], w["neff"]))
            assert np.array_equal(np.isnan(g["imputed"]), np.isnan(w["imputed"]))
            ok = ~np.isnan(w["imputed"])
            assert np.array_equal(g["imputed"][ok], w["imputed"][ok])
            assert np.array_equal(got["scores"].view(np.uint64), want["scores"].view(np.uint64))
