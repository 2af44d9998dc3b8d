"""GPU tests of PLINK 1 .bed rows (DESIGN.md 4.7): the C ABI on 2-bit rows against the oracle on the equivalent int8 GT
rows, and the whole host path on a fileset against the equivalent VCF and BCF."""
import os
import subprocess

import numpy as np
import pytest

import orc
from util_cohort import assert_loci_equal, assert_parity, bits, random_cohort, random_rows
from util_order import default_order_scores
from util_plink import make_split_dataset, pack_cohort
from util_files import derive_scores

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
LOC = ("ps", "homref", "fail", "ignore"); MIS = ("homref", "ignore"); SAM = ("ps", "homref", "fail", "int_ps", "int_fail")
POLICIES = [dict(imp_locus=l, imp_missing=m, imp_sample=s) for l in LOC for m in MIS for s in SAM]


@pytest.fixture(scope="module")
def nb():
    import __graft_entry__ as g
    g.build()
    import nimpress_b200
    return nimpress_b200


def cohort(seed, n, V, n_rows=None, miss_rate=0.03):
    """Random biallelic diploid int8 cohort (half calls included: missing, as the reference treats them), its .bed rows
    and random score rows naming REF or the ALT."""
    rng = np.random.default_rng(seed)
    gt = random_cohort(rng, n, V, miss_rate=miss_rate, n_alt=1, halfcall_rate=0.01)
    rows = random_rows(rng, V, n_rows=n_rows, n_alt=1)
    return gt, pack_cohort(gt, n), rows


def check(nb, eng, gt, n, rows, blocks, exact, offset, pol):
    got = eng.finish(offset=offset)
    want = orc.score_matrix(gt, n, 2, rows.astype(orc.ROW_DTYPE), offset=offset, **pol)
    assert got["nloci"] == want["nloci"]
    assert_loci_equal(got["loci"], want["loci"])
    if exact:
        assert_parity(got, want, exact=True)
    else:
        model = default_order_scores(gt, n, rows, want["loci"], want["nloci"], offset, blocks, lambda nb_: 1)
        a = got["scores"]
        assert np.array_equal(np.isnan(a), np.isnan(model))
        ok = ~np.isnan(a)
        assert np.array_equal(bits(a[ok]), bits(model[ok])), "default order differs from the model"
        assert_parity(got, want, exact=False)
    return got


def engine(nb, n, max_rows=4096, n_slots=2, exact=False, pol=None, staging_rows=None):
    eng = nb.Engine(n, ploidy=2, gt_width=nb.GT_BED, max_rows_per_block=max_rows, n_slots=n_slots, staging_rows=staging_rows)
    eng.set_policy(**(pol or {}))
    eng.set_exact_order(exact)
    eng.reset()
    return eng


@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
@pytest.mark.parametrize("n", [1, 3, 4, 5, 6, 7, 130, 1001, 2050])
def test_abi_parity_every_policy(nb, n, exact):
    """n = 0, 1, 2, 3 mod 4 (and n = 1, 3): records and nloci equal the oracle on the int8 rows; scores equal it bit
    for bit in exact order, and equal the one-row-group tile model bit for bit in the default order, under every
    sample / locus / missing policy.  Rows of every kind: constant and dropped rows sit inside tiles."""
    gt, bed, rows = cohort(n, n, 61, n_rows=83)
    for pol in POLICIES:
        pol = dict(pol, mincs=min(100, max(n - 2, 0)), maxmis=0.05 if n > 100 else 0.5)
        eng = engine(nb, n, exact=exact, pol=pol)
        assert eng.kernel_shape["fused"] == 4
        eng.score_host(bed, rows)
        check(nb, eng, gt, n, rows, [len(rows)], exact, 0.125, pol)
        eng.close()


@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
def test_padding_bits_are_ignored(nb, exact):
    """The codes past sample n - 1 in a row's last byte -- 00, 01, 10 or 11 -- change nothing."""
    n = 4 * 517 + 1
    gt, _, rows = cohort(5, n, 40, n_rows=70)
    outs = []
    for pad in range(4):
        eng = engine(nb, n, exact=exact)
        eng.score_host(pack_cohort(gt, n, pad_code=pad), rows)
        outs.append(check(nb, eng, gt, n, rows, [len(rows)], exact, 0.0, {}))
        eng.close()
    for o in outs[1:]:
        assert np.array_equal(bits(o["scores"]), bits(outs[0]["scores"]))


@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
def test_launch_cuts_ring_and_device_slabs(nb, exact):
    """npc_score_resident cut at max_rows_per_block (37), blocks of 17 rows streamed through the staging ring, and
    npc_score_block_device on a torch slab: each launch's tiles start at its own first row."""
    import torch
    n, V = 3001, 90
    gt, bed, rows = cohort(9, n, V, n_rows=201)
    # resident slab, launches of 37 rows
    eng = engine(nb, n, max_rows=37, exact=exact)
    assert eng.resident_reserve(V) >= V
    for r0 in range(0, V, 37):
        slot, view = eng.stage_acquire()
        nr = min(37, V - r0)
        view[:nr, :bed.shape[1]] = bed[r0:r0 + nr]
        eng.stage_upload(slot, nr, r0)
    eng.score_resident(rows)
    cut = [min(37, len(rows) - r0) for r0 in range(0, len(rows), 37)]
    check(nb, eng, gt, n, rows, cut, exact, -0.5, {})
    eng.close()
    # streaming: blocks of 17 score rows, each with the whole genotype block in its staging slot
    eng = engine(nb, n, max_rows=128, n_slots=3, exact=exact)
    blocks = []
    for r0 in range(0, len(rows), 17):
        eng.score_host(bed, rows[r0:r0 + 17])
        blocks.append(len(rows[r0:r0 + 17]))
    check(nb, eng, gt, n, rows, blocks, exact, 0.0, {})
    eng.close()
    # device slab with a wider row stride
    stride = 1024
    dev = torch.zeros((V, stride), dtype=torch.uint8, device="cuda")
    dev[:, :bed.shape[1]] = torch.from_numpy(bed).cuda()
    torch.cuda.synchronize()
    eng = engine(nb, n, max_rows=256, exact=exact)
    eng.score_block_device(dev, stride, V, rows)
    check(nb, eng, gt, n, rows, [len(rows)], exact, 0.0, {})
    eng.close()


@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
def test_wide_cohort(nb, exact):
    """1,300,000 samples (wider than one resident pass of the int8 tile kernel): the same kernels, same parity."""
    n = 1_300_000
    gt, bed, rows = cohort(13, n, 24, n_rows=41, miss_rate=0.01)
    eng = engine(nb, n, exact=exact)
    eng.score_host(bed, rows)
    check(nb, eng, gt, n, rows, [len(rows)], exact, 0.0, {})
    eng.close()


def test_refusals_and_one_by_one_multi(nb):
    """An effect allele other than REF / the ALT is NPC_EINVAL; the split count / accumulate calls NPC_EUNSUPPORTED;
    npc_score_resident_multi scores one definition at a time (no contraction) with the one-by-one results."""
    import torch
    n, V = 777, 30
    gt, bed, rows = cohort(17, n, V, n_rows=40)
    eng = engine(nb, n)
    bad = rows.copy()
    bad["kind"][0], bad["gt_row"][0], bad["eaidx"][0] = 0, 1, 2
    with pytest.raises(nb.NpcError, match="eaidx"):
        eng.score_host(bed, bad)
    dev = torch.zeros((V, 256), dtype=torch.uint8, device="cuda")
    counts = torch.zeros((len(rows), 2), dtype=torch.int64, device="cuda")
    with pytest.raises(nb.NpcError, match="rc=-5"):
        eng.count_block_device(dev, 256, V, rows, counts)
    with pytest.raises(nb.NpcError, match="rc=-5"):
        eng.accumulate_block_device(dev, 256, V, rows, counts)
    eng.close()
    eng = engine(nb, n)
    assert eng.resident_reserve(V) >= V
    slot, view = eng.stage_acquire()
    view[:V, :bed.shape[1]] = bed
    eng.stage_upload(slot, V, 0)
    rng = np.random.default_rng(3)
    lists = [rows, random_rows(rng, V, n_rows=25, n_alt=1), random_rows(rng, V, n_rows=60, n_alt=1)]
    multi = eng.score_resident_multi(lists, [0.25, 0.0, -1.0])
    assert eng.multi_contractions == 0
    for (sc, nloci, loci), r, off in zip(multi, lists, [0.25, 0.0, -1.0]):
        want = orc.score_matrix(gt, n, 2, r.astype(orc.ROW_DTYPE), offset=off)
        assert nloci == want["nloci"]
        assert_loci_equal(loci, want["loci"])
        model = default_order_scores(gt, n, r, want["loci"], want["nloci"], off, [len(r)], lambda nb_: 1)
        assert np.array_equal(bits(sc), bits(model))
    eng.close()


# ---- host and CLI -------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def api(nb):
    from nimpress_b200 import api
    return api


def same(a, b, exact=True):
    assert a.samples == b.samples and a.nloci == b.nloci and a.warnings == b.warnings
    assert_loci_equal(a.loci, b.loci)
    if exact:
        assert np.array_equal(bits(a.scores), bits(b.scores))


@pytest.mark.parametrize("seed", [41, 42])
def test_host_fileset_equals_vcf_and_bcf(api, tmp_path, seed, monkeypatch):
    """nph_compute_polygenic_scores on the fileset equals the same call on the equivalent VCF and BCF -- scores bit for
    bit in exact order, records, nloci, WARN lines -- without and with --cov, with NIMPRESS_SPLIT=3 (three contexts,
    contiguous score ranges), and with NIMPRESS_SLAB_ROWS forcing rounds.  The default order agrees too."""
    rng = np.random.default_rng(seed)
    d = make_split_dataset(str(tmp_path), rng, n=1203, V=300, sorted_scores=seed != 42)
    for cov in (None, d["bed"]):
        for exact in (True, False):
            p = api.run(d["score"], d["plink"], cov, exact_order=exact)
            for geno in (d["vcf"], d["bcf"]):
                same(p, api.run(d["score"], geno, cov, exact_order=exact), exact)
            assert p.rounds == 1
    monkeypatch.setenv("NIMPRESS_SPLIT", "3")
    p = api.run(d["score"], d["plink"], d["bed"], exact_order=True)
    assert p.devices == 3
    same(p, api.run(d["score"], d["bcf"], d["bed"], exact_order=True))
    monkeypatch.delenv("NIMPRESS_SPLIT")
    monkeypatch.setenv("NIMPRESS_SLAB_ROWS", "7")
    p = api.run(d["score"], d["plink"], d["bed"], exact_order=True)
    v = api.run(d["score"], d["bcf"], d["bed"], exact_order=True)
    assert p.rounds > 2 and p.rounds == v.rounds
    same(p, v)


def test_three_score_files_and_cli(api, tmp_path):
    """Three score files in one pass over the fileset equal the same pass over the VCF; `nimpress` on the fileset
    prints byte for byte what it prints on the VCF and BCF (exact order, with and without --cov)."""
    rng = np.random.default_rng(7)
    d = make_split_dataset(str(tmp_path), rng, n=801, V=240)
    paths = [d["score"]] + derive_scores(str(tmp_path), rng, d["entries"], 2)
    for exact in (True, False):
        ps = api.run_multi(paths, d["plink"], d["bed"], exact_order=exact)
        vs = api.run_multi(paths, d["vcf"], d["bed"], exact_order=exact)
        for a, b in zip(ps, vs):
            same(a, b, exact)
    for opts in ([], [f"--cov={d['bed']}", "--imp-sample=fail", "--maxmis=0.2"], ["--imp-locus=ignore", "--mincs=900"]):
        outs = [subprocess.run([EXE, "--exact-order", *opts, d["score"], g], capture_output=True, text=True)
                for g in (d["plink"], d["vcf"], d["bcf"])]
        assert all(o.returncode == 0 for o in outs), [o.stderr for o in outs]
        assert outs[0].stdout == outs[1].stdout == outs[2].stdout
    o = subprocess.run([EXE, "--exact-order", ",".join(paths), d["plink"]], capture_output=True, text=True)
    v = subprocess.run([EXE, "--exact-order", ",".join(paths), d["vcf"]], capture_output=True, text=True)
    assert o.returncode == 0 and o.stdout.replace(d["plink"], "G") == v.stdout.replace(d["vcf"], "G")
