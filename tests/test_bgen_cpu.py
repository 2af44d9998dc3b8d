"""CPU tests of the BGEN v1.2 reader (DESIGN.md 4.8): the fixed-point dosage rows it makes, sample names, matching
against the equivalent all-PASS VCF, and the refusals with their exit codes.  No GPU needed: nothing here computes a
score."""
import ctypes as C
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

from util_bgen import (MISSING, genotype_block, hard_call_probs, make_split_dataset, numerators, random_probs,
                       write_bgen)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
GT_DOSE255 = 255


@pytest.fixture(scope="module")
def api():
    import __graft_entry__ as g
    g.build()
    from nimpress_b200 import api
    api.load_host_library()
    return api


def read_gt(api, path, row_bytes, max_records=4096):
    L = api.load_host_library()
    out = np.full((max_records, row_bytes), 0xAB, np.uint8)
    nrec, ns, w, pl = C.c_int64(), C.c_int64(), C.c_int32(-1), C.c_int32()
    rc = L.nph_read_gt(os.fsencode(path), out.ctypes.data, row_bytes, max_records, C.byref(nrec), C.byref(ns), C.byref(w), C.byref(pl))
    return rc, out[:nrec.value], ns.value, w.value, pl.value


def plan(api, score, geno, bed=None):
    L = api.load_host_library()
    p = api._Params(0, 0, 3, 0, int(bed is not None), 0, 0, 0, 100, 0.05, 0.001)
    kind = np.zeros(1 << 16, np.int32); ea = np.zeros(1 << 16, np.int32)
    n_rows, n_s = C.c_int64(), C.c_int64()
    rc = L.nph_plan(os.fsencode(score), os.fsencode(geno), os.fsencode(bed) if bed else None, C.byref(p),
                    kind.ctypes.data, ea.ctypes.data, len(kind), C.byref(n_rows), C.byref(n_s))
    assert rc == 0, (rc, L.nph_last_error())
    return kind[:n_rows.value].copy(), ea[:n_rows.value].copy(), n_s.value


def test_writer_conventions():
    """Hand-worked samples: unphased k = 510 - 2*P(hom allele 1) - P(het), phased k = (255 - h0) + (255 - h1), in units
    of 1/255 of an ALT dosage; a missing sample is 0xFFFF.  Hard calls of GT rows give 0, 255 and 510."""
    probs = np.array([[255, 0], [0, 255], [0, 0], [100, 55], [1, 2], [0, 0]], np.uint8)
    miss = np.array([0, 0, 0, 0, 0, 1], bool)
    assert numerators(probs, False, miss).tolist() == [0, 255, 510, 255, 506, MISSING]
    assert numerators(probs, True, miss).tolist() == [255, 255, 510, 355, 507, MISSING]
    raw = np.array([2, 2, 2, 4, 4, 4, 0, 0, 0, 4, 3, 5], np.int8)          # 0/0, 0/1, 1/1, ./., ./1, 0|1
    for phased in (False, True):
        p, m = hard_call_probs(raw, 6, phased)
        assert numerators(p, phased, m).tolist() == [0, 255, 510, MISSING, MISSING, 255]
    blk = genotype_block(2, np.array([[1, 2], [0, 0]]), np.array([0, 1], bool), False)
    assert blk == struct.pack("<IHBB", 2, 2, 2, 2) + bytes([2, 0x82, 0, 8, 1, 2, 0, 0])


@pytest.mark.parametrize("n", [1, 7, 8, 9, 301])
@pytest.mark.parametrize("compression", ["none", "zlib"])
def test_read_gt_returns_numerators(api, tmp_path, monkeypatch, n, compression):
    """nph_read_gt on a .bgen: per sample the uint16 numerator computed in numpy from the stored probabilities (width
    NPC_GT_DOSE255, ploidy 2), phased and unphased variants, missing samples at 0xFFFF; NIMPRESS_THREADS=1 and 8 give
    the same bytes; the sample count comes from the embedded identifiers or from the .sample file."""
    rng = np.random.default_rng(n * 10 + len(compression))
    samples = [f"id{i}" for i in range(n)]
    variants, want = [], []
    for k in range(40):
        phased = bool(rng.random() < 0.5)
        probs, miss = random_probs(rng, n, phased)
        variants.append(dict(contig=str(1 + k % 3), pos=100 + k, alleles=["A", "G"], probs=probs, missing=miss, phased=phased))
        want.append(numerators(probs, phased, miss))
    want = np.stack(want)
    rb = 2 * n + 32
    for embed in (True, False):
        path = write_bgen(str(tmp_path / f"c{int(embed)}.bgen"), samples, variants, compression=compression, embed_ids=embed)
        outs = []
        for threads in ("1", "8"):
            monkeypatch.setenv("NIMPRESS_THREADS", threads)
            rc, rows, ns, w, pl = read_gt(api, path, rb)
            assert rc == 0 and ns == n and (w, pl) == (GT_DOSE255, 2) and rows.shape[0] == len(variants)
            assert np.array_equal(rows[:, :2 * n].copy().view("<u2"), want)
            assert (rows[:, 2 * n:] == 0xAB).all()                        # nothing written past the row
            outs.append(rows)
        assert np.array_equal(outs[0], outs[1])


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_matching_equals_equivalent_vcf(api, tmp_path, seed):
    """nph_plan on the .bgen gives the kind and eaidx of the equivalent all-PASS VCF, with and without --cov, and the
    sample count of the .sample file when the identifiers are not embedded."""
    rng = np.random.default_rng(seed)
    d = make_split_dataset(str(tmp_path), rng, n=37, V=150, embed_ids=seed != 2, compression="none" if seed == 3 else "zlib")
    for bed in (None, d["bed"]):
        k_b, e_b, n_b = plan(api, d["score"], d["bgen"], bed)
        k_v, e_v, _ = plan(api, d["score"], d["vcf"], bed)
        assert np.array_equal(k_b, k_v) and np.array_equal(e_b, e_v) and n_b == 37
        assert set(np.unique(e_b[k_b == 0])) <= {0, 1}
    assert (k_b == 0).sum() > 20


def _file(tmp, n=9, V=5, **kw):
    rng = np.random.default_rng(0)
    variants = []
    for k in range(V):
        probs, miss = random_probs(rng, n, False, miss_rate=0.0)
        variants.append(dict(contig="1", pos=100 + 10 * k, alleles=["A", "G"], probs=probs, missing=miss, phased=False))
    path = os.path.join(tmp, "f.bgen")
    score = os.path.join(tmp, "f.score")
    with open(score, "w") as fh:
        fh.write("S\nd\nc\nhs37d5\n0.0\n1\t100\tA\tG\t0.1\t0.2\n")
    return path, score, variants, [f"s{i}" for i in range(n)]


def _run(*args):
    return subprocess.run([EXE, *args], capture_output=True, text=True)


def test_refusals(api, tmp_path):
    """Malformed files are InputError (exit 1): zstd, layout 1, LH < 20, offset < LH, a truncated file, fewer variant
    blocks than M, a .sample or embedded identifier count other than N.  A block with K != 2, ploidy other than 2,
    B != 8, a stored N other than N or an unphased b0 + b1 > 255 is InputError naming the variant.  A missing .sample is
    "could not open input" (exit 255)."""
    path, score, variants, samples = _file(str(tmp_path))
    n = len(samples)

    def refused(expect_rc, expect_msg, *extra):
        r = _run(*extra, score, path)
        assert r.returncode == expect_rc, (r.returncode, r.stdout, r.stderr)
        assert expect_msg in (r.stdout + r.stderr), (r.stdout, r.stderr)

    write_bgen(path, samples, variants)
    plan(api, score, path)
    good = open(path, "rb").read()
    write_bgen(path, samples, variants, compression="zstd")
    refused(1, "zstd")
    write_bgen(path, samples, variants, layout=1)
    refused(1, "layout 1")
    write_bgen(path, samples, variants, free=b"", header_len=16)
    refused(1, "< 20")
    write_bgen(path, samples, variants, embed_ids=False, offset_delta=-2)
    refused(1, "inside the header")
    # the variant blocks are walked while the file streams to the GPU: on the CPU, nph_plan (which walks them too)
    # reports a truncation as NPH_EINPUT; tests/test_bgen_gpu.py checks the CLI's exit code
    L = api.load_host_library()

    def plan_refused(msg):
        kind = np.zeros(16, np.int32); ea = np.zeros(16, np.int32); nr, ns = C.c_int64(), C.c_int64()
        rc = L.nph_plan(os.fsencode(score), os.fsencode(path), None, C.byref(api._Params(0, 0, 3, 0, 0, 0, 0, 0, 100, 0.05, 0.001)),
                        kind.ctypes.data, ea.ctypes.data, 16, C.byref(nr), C.byref(ns))
        assert rc == -3 and msg in L.nph_last_error().decode(), (rc, L.nph_last_error())

    open(path, "wb").write(good[:-7])
    plan_refused("truncated")
    write_bgen(path, samples, variants, n_variants=len(variants) + 1)
    plan_refused("truncated")
    write_bgen(path, samples, variants, embed_ids=False)
    with open(path[:-5] + ".sample", "a") as fh:
        fh.write("F99 extra 0\n")
    refused(1, ".sample")
    hdr = struct.unpack_from("<II", good, 0)                         # the embedded count field says N + 1
    ids = good[:4 + hdr[1] + 4] + struct.pack("<I", n + 1) + good[4 + hdr[1] + 8:]
    open(path, "wb").write(ids)
    refused(1, "sample identifiers")

    # a matched variant's block is converted while the file streams to the GPU: on the CPU, nph_read_gt (which converts
    # every block) reports the same InputError as NPH_EINPUT

    def block_refused(v, msg):
        write_bgen(path, samples, v)
        rc, *_ = read_gt(api, path, 2 * n + 16)
        assert rc == -3 and msg in L.nph_last_error().decode() and "1:100 (v0)" in L.nph_last_error().decode()

    probs, miss = variants[0]["probs"], variants[0]["missing"]
    for kw, msg in ((dict(K=3), "3 alleles"), (dict(pmin=1), "ploidy"), (dict(pmax=3), "ploidy"), (dict(bits=16), "16 bits"),
                    (dict(n_stored=n + 1), "samples")):
        block_refused([dict(variants[0], block=genotype_block(n, probs, miss, False, **kw))] + variants[1:], msg)
    block_refused([dict(variants[0], probs=np.full((n, 2), 200, np.uint8))] + variants[1:], "> 1")
    write_bgen(path, samples, variants, embed_ids=False)
    os.remove(path[:-5] + ".sample")
    refused(255, "FATAL Could not open input VCF file")
    # the refusals reach the C ABI as NPH_EINPUT / NPH_EOPEN_VCF too
    with pytest.raises(FileNotFoundError):
        api.run(score, path)
    write_bgen(path, samples, variants, layout=1)
    with pytest.raises(api.NimpressInputError, match="layout"):
        api.run(score, path)


def test_unmatched_malformed_blocks_are_never_read(api, tmp_path, monkeypatch):
    """Blocks of variants no score row needs are skipped by their length: K = 3 or B = 16 there is no refusal, and
    nph_plan, which reads no genotypes, matches the well-formed variant."""
    path, score, variants, samples = _file(str(tmp_path))
    n = len(samples)
    probs, miss = variants[1]["probs"], variants[1]["missing"]
    bad = [variants[0], dict(variants[1], alleles=["A", "G", "T"], block=genotype_block(n, probs, miss, False, K=3)),
           dict(variants[2], block=genotype_block(n, probs, miss, False, bits=16)), variants[3]]
    write_bgen(path, samples, bad)
    kind, ea, _ = plan(api, score, path)
    assert kind.tolist() == [0] and ea.tolist() == [1]
    rc, rows, *_ = read_gt(api, path, 2 * n + 16)                     # nph_read_gt converts every block: refused
    assert rc != 0


def test_usage_names_bgen(api):
    r = _run("--help")
    assert r.returncode == 0 and "<genotypes.bgen>" in r.stdout and "BGEN v1.2" in r.stdout


@pytest.mark.parametrize("n", [1, 9, 130, 1001])
def test_reference_restatement_equals_oracle_on_hard_calls(n):
    """The numpy restatement the GPU tests pin the dosage kernels to (util_bgen.reference_scores) equals the C oracle on
    the same genotypes as int8 GT rows, under every locus / missing / sample policy: scores bit for bit, nloci, and
    records with neff = 255 x the GT neff (fl(k/255) is the exact allele count for k = 0, 255, 510)."""
    import orc
    from util_bgen import reference_scores
    from util_cohort import random_cohort, random_rows
    rng = np.random.default_rng(n + 5)
    gt = random_cohort(rng, n, 40, miss_rate=0.04, n_alt=1, halfcall_rate=0.01)
    rows = random_rows(rng, 40, n_rows=70, n_alt=1)
    a = (gt[:, :2 * n].reshape(len(gt), n, 2).astype(np.int32) >> 1) - 1
    k = np.where((a < 0).any(axis=2), MISSING, 255 * (a == 1).sum(axis=2)).astype(np.uint16)
    for l in ("ps", "homref", "fail", "ignore"):
        for m in ("homref", "ignore"):
            for s in ("ps", "homref", "fail", "int_ps", "int_fail"):
                pol = dict(imp_locus=l, imp_missing=m, imp_sample=s, mincs=min(100, max(n - 2, 0)), maxmis=0.05 if n > 100 else 0.5)
                got = reference_scores(k, n, rows, offset=0.25, **pol)
                want = orc.score_matrix(gt, n, 2, rows.astype(orc.ROW_DTYPE), offset=0.25, **pol)
                assert got["nloci"] == want["nloci"]
                w = want["loci"]
                g = got["loci"]
                for f in ("klass", "used", "eaidx", "ngt", "nmiss"):
                    assert np.array_equal(g[f], w[f]), f
                assert np.array_equal(g["neff"], np.where(w["neff"] >= 0, 255 * w["neff"], w["neff"]))
                assert np.array_equal(np.isnan(g["imputed"]), np.isnan(w["imputed"]))
                ok = ~np.isnan(w["imputed"])
                assert np.array_equal(g["imputed"][ok], w["imputed"][ok])
                assert np.array_equal(got["scores"].view(np.uint64), want["scores"].view(np.uint64))
