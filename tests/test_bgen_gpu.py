"""GPU tests of fixed-point dosage rows from BGEN files (DESIGN.md 4.8): the C ABI bit for bit against the reference
restatement of tests/util_bgen.py (`oracle` here; pinned to the C oracle on hard calls by tests/test_bgen_cpu.py),
hard calls against int8 GT rows, and the whole host path on a .bgen against the equivalent VCF and BCF."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import orc
from util_bgen import genotype_block, make_split_dataset, random_probs, reference_scores as oracle, write_bgen
from util_cohort import assert_loci_equal, bits, random_cohort, random_rows
from util_files import derive_scores

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


def random_k(rng, n, V, pad_to=16):
    """Dosage rows uint16[V, cols]: fractional numerators, hard calls (0, 255, 510), missing samples as 0xFFFF and as
    other values above 510; the padding past sample n - 1 is garbage that must never be read."""
    cols = -(-2 * n // pad_to) * pad_to // 2
    k = rng.integers(0, 511, size=(V, cols))
    hard = rng.random((V, cols)) < 0.3
    k[hard] = 255 * rng.integers(0, 3, size=int(hard.sum()))
    miss = rng.random((V, cols)) < 0.03 * rng.uniform(0, 2, size=(V, 1))
    k[miss] = np.where(rng.random(int(miss.sum())) < 0.8, 0xFFFF, rng.integers(511, 0xFFFF, size=int(miss.sum())))
    k[:, n:] = rng.integers(0, 0x10000, size=(V, cols - n))
    return k.astype(np.uint16)


def engine(nb, n, max_rows=4096, n_slots=2, exact=False, pol=None, staging_rows=None):
    eng = nb.Engine(n, ploidy=2, gt_width=nb.GT_DOSE255, max_rows_per_block=max_rows, n_slots=n_slots, staging_rows=staging_rows)
    eng.set_policy(**(pol or {}))
    eng.set_exact_order(exact)
    eng.reset()
    return eng


def check(got, want):
    assert got["nloci"] == want["nloci"]
    assert_loci_equal(got["loci"], want["loci"])
    assert np.array_equal(bits(got["scores"]), bits(want["scores"]))     # NaN included: the same bits


def cohort(seed, n, V, n_rows):
    rng = np.random.default_rng(seed)
    return random_k(rng, n, V), random_rows(rng, V, n_rows=n_rows, n_alt=1)


@pytest.mark.parametrize("n", [1, 7, 8, 9, 130, 1001, 2050])
def test_abi_parity_every_policy(nb, n):
    """Scores, records and nloci equal the oracle bit for bit under every locus / missing / sample policy, exact order on
    and off alike; kernel_shape reports mode 5."""
    k, rows = cohort(n, n, 61, 83)
    for pol in POLICIES:
        pol = dict(pol, mincs=min(100, max(n - 2, 0)), maxmis=0.05 if n > 100 else 0.5)
        want = oracle(k, n, rows, offset=0.125, **pol)
        for exact in (False, True):
            eng = engine(nb, n, exact=exact, pol=pol)
            shape = eng.kernel_shape
            assert shape["fused"] == 5
            eng.score_host(k, rows)
            check(eng.finish(offset=0.125), want)
            eng.close()


def test_launch_cuts_ring_and_device_slabs(nb):
    """npc_score_resident cut at max_rows_per_block (37), blocks of 17 rows streamed through the staging ring, and
    npc_score_block_device on a torch slab: the sums carry across launches, the bits equal the oracle's."""
    import torch
    n, V = 3001, 90
    k, rows = cohort(9, n, V, 201)
    want = oracle(k, n, rows, offset=-0.5)
    for exact in (False, True):
        eng = engine(nb, n, max_rows=37, exact=exact)
        assert eng.resident_reserve(V) >= V
        for r0 in range(0, V, 37):
            slot, view = eng.stage_acquire()
            nr = min(37, V - r0)
            view[:nr, :k.shape[1] * 2] = k[r0:r0 + nr].view(np.uint8)
            eng.stage_upload(slot, nr, r0)
        eng.score_resident(rows)
        check(eng.finish(offset=-0.5), want)
        eng.close()
    want = oracle(k, n, rows)
    eng = engine(nb, n, max_rows=128, n_slots=3)
    for r0 in range(0, len(rows), 17):
        eng.score_host(k, rows[r0:r0 + 17])
    check(eng.finish(), want)
    eng.close()
    stride = 8192
    dev = torch.zeros((V, stride), dtype=torch.uint8, device="cuda")
    dev[:, :k.shape[1] * 2] = torch.from_numpy(k.view(np.uint8)).cuda()
    torch.cuda.synchronize()
    eng = engine(nb, n, max_rows=256)
    eng.score_block_device(dev, stride, V, rows)
    check(eng.finish(), want)
    eng.close()


def test_wide_cohort(nb):
    """1,300,000 samples: the same kernels, the same bits."""
    n = 1_300_000
    k, rows = cohort(13, n, 24, 41)
    eng = engine(nb, n, max_rows=64)
    eng.score_host(k, rows)
    check(eng.finish(), oracle(k, n, rows))
    eng.close()


def to_k(gt, n):
    """int8 biallelic diploid GT rows -> dosage numerators (255 x ALT alleles; a half call is missing)."""
    a = (gt[:, :2 * n].reshape(len(gt), n, 2).astype(np.int32) >> 1) - 1
    k = np.where((a < 0).any(axis=2), 0xFFFF, 255 * (a == 1).sum(axis=2))
    return k.astype(np.uint16)


@pytest.mark.parametrize("n", [9, 1001, 40000])
def test_hard_calls_equal_int8_gt(nb, n):
    """Hard-call dosage rows score bit for bit as the same genotypes in int8 GT rows in exact order; the records are
    equal except that neff is 255 x the GT neff."""
    rng = np.random.default_rng(n)
    gt = random_cohort(rng, n, 50, miss_rate=0.03, n_alt=1, halfcall_rate=0.01)
    rows = random_rows(rng, 50, n_rows=90, n_alt=1)
    k = to_k(gt, n)
    for pol in (POLICIES[3], POLICIES[17], POLICIES[38]):
        pol = dict(pol, mincs=min(100, n - 2), maxmis=0.05 if n > 100 else 0.5)
        a = engine(nb, n, exact=True, pol=pol)
        a.score_host(k, rows)
        got = a.finish(offset=0.5)
        b = nb.Engine(n, max_rows_per_block=4096, n_slots=2)
        b.set_policy(**pol); b.set_exact_order(True); b.reset()
        b.score_host(gt, rows)
        ref = b.finish(offset=0.5)
        a.close(); b.close()
        assert got["nloci"] == ref["nloci"]
        want = ref["loci"].copy()
        want["neff"] = np.where(want["neff"] >= 0, want["neff"] * 255, want["neff"])
        assert_loci_equal(got["loci"], want)
        assert np.array_equal(bits(got["scores"]), bits(ref["scores"]))


def test_refusals_and_one_by_one_multi(nb):
    """An effect allele other than REF / the ALT is NPC_EINVAL; the split count / accumulate calls NPC_EUNSUPPORTED;
    npc_score_resident_multi scores one definition at a time (no contraction) with the oracle's bits."""
    import torch
    n, V = 777, 30
    k, rows = cohort(17, n, V, 40)
    eng = engine(nb, n)
    bad = rows.copy()
    bad["kind"][0], bad["gt_row"][0], bad["eaidx"][0] = 0, 1, 2
    with pytest.raises(nb.NpcError, match="eaidx"):
        eng.score_host(k, bad)
    dev = torch.zeros((V, 2048), dtype=torch.uint8, device="cuda")
    counts = torch.zeros((len(rows), 2), dtype=torch.int64, device="cuda")
    with pytest.raises(nb.NpcError, match="rc=-5"):
        eng.count_block_device(dev, 2048, V, rows, counts)
    with pytest.raises(nb.NpcError, match="rc=-5"):
        eng.accumulate_block_device(dev, 2048, V, rows, counts)
    eng.close()
    eng = engine(nb, n)
    assert eng.resident_reserve(V) >= V
    slot, view = eng.stage_acquire()
    view[:V, :k.shape[1] * 2] = k.view(np.uint8)
    eng.stage_upload(slot, V, 0)
    rng = np.random.default_rng(3)
    lists = [rows, random_rows(rng, V, n_rows=25, n_alt=1), random_rows(rng, V, n_rows=60, n_alt=1)]
    offs = [0.25, 0.0, -1.0]
    multi = eng.score_resident_multi(lists, offs)
    assert eng.multi_contractions == 0
    for (sc, nloci, loci), r, off in zip(multi, lists, offs):
        check(dict(scores=sc, nloci=nloci, loci=loci), oracle(k, n, r, offset=off))
    eng.close()


# ---- host and CLI -------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def api(nb):
    from nimpress_b200 import api
    return api


def same(b, v, exact=True):
    """b on the .bgen, v on the equivalent VCF / BCF: the same samples, nloci, scores (exact order: bits), records with
    neff scaled by 255, and WARN lines once the AF-mismatch lines of tallied loci are removed."""
    assert b.samples == v.samples and b.nloci == v.nloci
    assert b.warnings == AF_LINE.sub("", v.warnings)
    want = v.loci.copy()
    want["neff"] = np.where(want["neff"] >= 0, want["neff"] * 255, want["neff"])
    assert_loci_equal(b.loci, want)
    if exact:
        assert np.array_equal(bits(b.scores), bits(v.scores))
    else:
        assert np.allclose(b.scores, v.scores, rtol=1e-12, atol=1e-15, equal_nan=True)


@pytest.mark.parametrize("seed", [41, 42])
def test_host_bgen_equals_vcf_and_bcf(api, tmp_path, seed, monkeypatch):
    """nph_compute_polygenic_scores on a hard-call .bgen equals the same call on the equivalent VCF and BCF in exact
    order -- without and with --cov, with NIMPRESS_SPLIT=3 and with NIMPRESS_SLAB_ROWS=7.  Seed 42: identifiers from
    the .sample file, uncompressed blocks, one worker thread."""
    rng = np.random.default_rng(seed)
    d = make_split_dataset(str(tmp_path), rng, n=1203, V=300, sorted_scores=seed != 42, embed_ids=seed != 42,
                           compression="zlib" if seed != 42 else "none")
    if seed == 42:
        monkeypatch.setenv("NIMPRESS_THREADS", "1")
    for cov in (None, d["bed"]):
        b = api.run(d["score"], d["bgen"], cov, exact_order=True)
        for geno in (d["vcf"], d["bcf"]):
            same(b, api.run(d["score"], geno, cov, exact_order=True))
        same(api.run(d["score"], d["bgen"], cov), api.run(d["score"], d["vcf"], cov, exact_order=True))   # every mode: the chain
    monkeypatch.setenv("NIMPRESS_SPLIT", "3")
    b = api.run(d["score"], d["bgen"], d["bed"], exact_order=True)
    assert b.devices == 3
    same(b, api.run(d["score"], d["bcf"], d["bed"], exact_order=True))
    monkeypatch.delenv("NIMPRESS_SPLIT")
    monkeypatch.setenv("NIMPRESS_SLAB_ROWS", "7")
    b = api.run(d["score"], d["bgen"], d["bed"], exact_order=True)
    v = api.run(d["score"], d["bcf"], d["bed"], exact_order=True)
    assert b.rounds > 2 and b.rounds == v.rounds
    same(b, v)


def test_three_score_files_and_cli(api, tmp_path):
    """Three score files in one pass over the .bgen equal the same pass over the VCF; `nimpress` prints the same stdout
    on the .bgen as on the VCF and BCF once the AF-mismatch lines are removed, and --dosage changes nothing."""
    rng = np.random.default_rng(7)
    d = make_split_dataset(str(tmp_path), rng, n=801, V=240)
    paths = [d["score"]] + derive_scores(str(tmp_path), rng, d["entries"], 2)
    bs = api.run_multi(paths, d["bgen"], d["bed"], exact_order=True)
    vs = api.run_multi(paths, d["vcf"], d["bed"], exact_order=True)
    for a, b in zip(bs, vs):
        same(a, b)
    for opts in ([], [f"--cov={d['bed']}", "--imp-sample=fail", "--maxmis=0.2"], ["--imp-locus=ignore", "--mincs=900"]):
        outs = [subprocess.run([EXE, "--exact-order", *opts, d["score"], g], capture_output=True, text=True)
                for g in (d["bgen"], d["vcf"], d["bcf"])]
        assert all(o.returncode == 0 for o in outs), [o.stderr for o in outs]
        assert outs[0].stdout == AF_LINE.sub("", outs[1].stdout) == AF_LINE.sub("", outs[2].stdout)
        o = subprocess.run([EXE, "--exact-order", "--dosage", *opts, d["score"], d["bgen"]], capture_output=True, text=True)
        assert o.returncode == 0 and o.stdout == outs[0].stdout
    o = subprocess.run([EXE, "--exact-order", ",".join(paths), d["bgen"]], capture_output=True, text=True)
    v = subprocess.run([EXE, "--exact-order", ",".join(paths), d["vcf"]], capture_output=True, text=True)
    assert o.returncode == 0 and o.stdout.replace(d["bgen"], "G") == AF_LINE.sub("", v.stdout.replace(d["vcf"], "G"))


def test_fractional_host_equals_oracle(api, tmp_path, monkeypatch):
    """A fractional .bgen through the host equals the oracle on the rows nph_read_gt returns, bit for bit, with the
    blocks converted on eight worker threads; no AF-mismatch line is written for its loci."""
    monkeypatch.setenv("NIMPRESS_THREADS", "8")
    rng = np.random.default_rng(5)
    n, V = 2003, 120
    samples = [f"s{i}" for i in range(n)]
    variants, entries = [], []
    for j in range(V):
        phased = bool(rng.random() < 0.5)
        probs, miss = random_probs(rng, n, phased)
        variants.append(dict(contig="1", pos=1000 + 10 * j, alleles=["A", "C"], probs=probs, missing=miss, phased=phased))
        ea = "A" if rng.random() < 0.3 else "C"
        entries.append(("1", 1000 + 10 * j, "A", ea, round(float(rng.normal(0, 0.05)), 4), round(float(rng.uniform(0.01, 0.5)), 4)))
    entries += [("1", 5, "A", "C", 0.1, 0.2), ("1", 1000, "A", "G", 0.1, 0.2)]                      # absent
    path = write_bgen(str(tmp_path / "f.bgen"), samples, variants)
    score = str(tmp_path / "f.score")
    with open(score, "w") as fh:
        fh.write("S\nd\nc\nhs37d5\n0.125\n" + "\n".join("\t".join(str(x) for x in e) for e in entries) + "\n")
    L = api.load_host_library()
    out = np.zeros((V, 2 * n), np.uint8)
    nrec, ns, w, pl = C.c_int64(), C.c_int64(), C.c_int32(), C.c_int32()
    assert L.nph_read_gt(os.fsencode(path), out.ctypes.data, 2 * n, V, C.byref(nrec), C.byref(ns), C.byref(w), C.byref(pl)) == 0
    k = out.view("<u2")
    rows = np.zeros(len(entries), dtype=orc.ROW_DTYPE)
    for i, e in enumerate(entries):
        hit = i < V
        rows[i] = (i if hit else -1, (0 if e[3] == "A" else 1) if hit else -1, e[4], e[5], int(e[2] == e[3]), 0 if hit else 2)
    for pol in (dict(), dict(imp_sample="int_fail", maxmis=0.03), dict(imp_locus="homref", imp_sample="ps", maxmis=0.02)):
        kw = dict(maxmis=pol.get("maxmis", 0.05), imp_locus=api.ImputeMethodLocus[pol.get("imp_locus", "ps")],
                  imp_sample=api.ImputeMethodSample[pol.get("imp_sample", "int_ps")])
        b = api.run(score, path, exact_order=bool(pol), **kw)
        want = oracle(k, n, rows, offset=0.125, **pol)
        assert b.nloci == want["nloci"]
        assert_loci_equal(b.loci, want["loci"])
        assert np.array_equal(bits(b.scores), bits(want["scores"]))
        assert AF_LINE.search(b.warnings) is None                         # no AF-mismatch test on dosage rows


def test_cli_refusals_of_streamed_blocks(tmp_path):
    """Refusals found while the file streams exit 1 from the CLI: a truncated file, fewer variant blocks than the header
    says, and a matched variant with K != 2, B != 8 or an unphased b0 + b1 > 255 (named in the message).  The same file
    with those blocks unmatched scores, and --dosage changes nothing."""
    rng = np.random.default_rng(11)
    n = 9
    samples = [f"s{i}" for i in range(n)]
    variants = []
    for j in range(4):
        probs, miss = random_probs(rng, n, False, miss_rate=0.0)
        variants.append(dict(contig="1", pos=100 + 10 * j, alleles=["A", "G"], probs=probs, missing=miss, phased=False))
    path = str(tmp_path / "f.bgen")
    score = str(tmp_path / "f.score")
    with open(score, "w") as fh:
        fh.write("S\nd\nc\nhs37d5\n0.0\n1\t100\tA\tG\t0.1\t0.2\n")

    def run(*extra):
        return subprocess.run([EXE, *extra, score, path], capture_output=True, text=True)

    write_bgen(path, samples, variants)
    good = open(path, "rb").read()
    ok = run()
    assert ok.returncode == 0 and run("--dosage").stdout == ok.stdout
    open(path, "wb").write(good[:-7])
    r = run()
    assert r.returncode == 1 and "truncated" in r.stderr
    write_bgen(path, samples, variants, n_variants=5)
    r = run()
    assert r.returncode == 1 and "truncated" in r.stderr
    p0, m0 = variants[0]["probs"], variants[0]["missing"]
    for v0, msg in ((dict(variants[0], block=genotype_block(n, p0, m0, False, K=3)), "3 alleles"),
                    (dict(variants[0], block=genotype_block(n, p0, m0, False, bits=16)), "16 bits"),
                    (dict(variants[0], probs=np.full((n, 2), 200, np.uint8)), "> 1")):
        write_bgen(path, samples, [v0] + variants[1:])
        r = run()
        assert r.returncode == 1 and msg in r.stderr and "1:100 (v0)" in r.stderr, (r.returncode, r.stderr)
        write_bgen(path, samples, variants[:1] + [dict(v0, pos=110)] + variants[2:])      # the bad block unmatched
        assert run().returncode == 0
