"""GPU tests of the observed counts (DESIGN.md 4.13): per sample, the score rows of class OK at which the sample has a
called genotype.  Every layout at the C ABI against the numpy restatement of its tally's predicate (tests/util_observed.py)
over the engine's own records (which the other suites pin to the oracle); the counts add up to the OK records' ngt;
scores, records and launches are untouched; the host paths (--samples, several files, rounds, several contexts, several
score files) give what one plain run gives; the CLI prints set1's hand-derived counts."""
import os
import subprocess
import sys

import numpy as np
import pytest

from util_bcf import write_vcf
from util_cohort import assert_loci_equal, bits, random_cohort, random_rows
from util_files import derive_scores, make_dataset
from util_observed import (called_bed, called_dose32, called_dose255, called_ds, called_gt, called_pl, ngt_total,
                           observed, oracle_observed_files, oracle_observed_matrix)
from util_pl import pack_words, random_pl
from util_plink import pack_cohort
from util_split import by_contig, write_split

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S1 = os.path.join(ROOT, "tests", "golden", "set1")
CONTIGS = ["1", "2", "X"]


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


def pad16(a):
    a = np.ascontiguousarray(a).view(np.uint8).reshape(len(a), -1)
    out = np.zeros((len(a), -(-a.shape[1] // 16) * 16), np.uint8)
    out[:, :a.shape[1]] = a
    return out


def score(nb, slab, n, rows, width=1, ploidy=2, exact=False, obs=True, dosage=False, maxmis=0.5, max_rows=4096, split=False):
    """One context over the device slab: (finish() dict, observed counts or None, launches)."""
    import torch
    eng = nb.Engine(n, ploidy=ploidy, gt_width=width, max_rows_per_block=max_rows)
    eng.set_policy(maxmis=maxmis, mincs=5)
    eng.set_exact_order(exact)
    if dosage:
        eng.set_dosage_rows(True)
    if obs is not None:
        eng.set_observed(obs)
    eng.reset()
    dev = torch.from_numpy(slab).cuda()
    for r0 in range(0, len(rows), max_rows):
        blk = rows[r0:r0 + max_rows]
        if split:
            counts = torch.zeros((len(blk), 2), dtype=torch.int64, device="cuda")
            eng.count_block_device(dev.data_ptr(), slab.shape[1], len(slab), blk, counts.data_ptr())
            eng.accumulate_block_device(dev.data_ptr(), slab.shape[1], len(slab), blk, counts.data_ptr())
        else:
            eng.score_block_device(dev.data_ptr(), slab.shape[1], len(slab), blk)
    res = eng.finish()
    got = eng.observed() if obs else None
    launches = eng.launches
    eng.close()
    return res, got, launches


def check(nb, slab, n, rows, called_of, oracle_gt=None, **kw):
    """oracle_gt: the slab's rows as the oracle reads them (int GT or float32 DS rows): the counts are also checked against
    the oracle's own loop."""
    res, got, _ = score(nb, slab, n, rows, **kw)
    want = observed(called_of, rows, res["loci"], n)
    assert np.array_equal(got, want)
    if oracle_gt is not None:
        assert np.array_equal(got, oracle_observed_matrix(oracle_gt, n, kw.get("ploidy", 2), rows, maxmis=kw.get("maxmis", 0.5), mincs=5))
    assert int(got.sum()) == ngt_total(res["loci"])
    assert (res["loci"]["klass"] == 0).sum() > 0 and (got < res["nloci"]).any()
    return res, got


def gt_case(rng, n, V, width=1, ploidy=2):
    gt = random_cohort(rng, n, V, width=width, ploidy=ploidy, miss_rate=0.05, n_alt=2, halfcall_rate=0.02, sentinel_rate=0.03,
                       invalid_rate=0.002)
    dt = {1: np.int8, 2: np.int16, 4: np.int32}[width]
    slab = pad16(gt)
    return slab, random_rows(rng, V, n_rows=V + 20, n_alt=2), lambda r: called_gt(slab[r["gt_row"]], n, ploidy, dt), slab.view(dt)


@pytest.mark.parametrize("width,ploidy", [(1, 2), (1, 1), (1, 3), (2, 2), (4, 2), (2, 4)])
@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
def test_gt_layouts(nb, width, ploidy, exact):
    rng = np.random.default_rng(width * 10 + ploidy)
    slab, rows, called_of, ogt = gt_case(rng, 1037, 48, width, ploidy)
    check(nb, slab, 1037, rows, called_of, oracle_gt=ogt, width=width, ploidy=ploidy, exact=exact)


def test_unchanged_when_off_and_launches(nb):
    rng = np.random.default_rng(3)
    n = 3001
    slab, rows, _, _ = gt_case(rng, n, 40)
    never, _, l_never = score(nb, slab, n, rows, obs=None, max_rows=40)
    off, _, l_off = score(nb, slab, n, rows, obs=False, max_rows=40)
    on, _, l_on = score(nb, slab, n, rows, obs=True, max_rows=40)
    for r in (off, on):
        assert np.array_equal(bits(r["scores"]), bits(never["scores"])) and r["nloci"] == never["nloci"]
        assert_loci_equal(r["loci"], never["loci"])
    assert l_off == l_never
    assert l_on == l_never + -(-len(rows) // 40)          # one observed pass per scoring launch


def bed_rows(rng, n, V):
    gt = random_cohort(rng, n, V, miss_rate=0.06, halfcall_rate=0.02)
    return pad16(pack_cohort(gt, n, pad_code=1))


@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
def test_bed(nb, exact):
    rng = np.random.default_rng(11)
    n, V = 2051, 40
    slab = bed_rows(rng, n, V)
    rows = random_rows(rng, V, n_rows=V + 10)
    check(nb, slab, n, rows, lambda r: called_bed(slab[r["gt_row"]], n), width=nb.GT_BED, exact=exact)


def test_dose255(nb):
    rng = np.random.default_rng(12)
    n, V = 1999, 40
    k = rng.integers(0, 511, size=(V, n)).astype(np.uint16)
    k[rng.random((V, n)) < 0.05] = 0xFFFF
    k[rng.random((V, n)) < 0.01] = 511
    slab = pad16(k)
    rows = random_rows(rng, V, n_rows=V + 10)
    check(nb, slab, n, rows, lambda r: called_dose255(slab[r["gt_row"]], n), width=nb.GT_DOSE255)


@pytest.mark.parametrize("bits_", [8, 16])
def test_dose32_haploid(nb, bits_):
    from util_bgen_bits import dose32_rows
    rng = np.random.default_rng(bits_)
    n, V = 1501, 40
    D = (1 << bits_) - 1
    p = rng.choice([1, 2, 2, 2, 0, 3], size=(V, n), p=[0.2, 0.25, 0.25, 0.25, 0.025, 0.025])
    k = (rng.random((V, n)) * (np.maximum(p, 1) * D + 3)).astype(np.int64)
    w = (k | (p << 24)).astype(np.uint32)
    w[rng.random((V, n)) < 0.04] = 0xFFFFFFFF
    w[rng.random((V, n)) < 0.01] |= np.uint32(1 << 31)
    slab = dose32_rows(w, np.full(V, D))
    rows = random_rows(rng, V, n_rows=V + 10)
    check(nb, slab, n, rows, lambda r: called_dose32(slab[r["gt_row"]], n), width=nb.GT_DOSE32)


def test_ds(nb):
    rng = np.random.default_rng(13)
    n, V = 1003, 40
    ds = rng.uniform(0, 2, size=(V, n)).astype(np.float32)
    b = ds.view(np.uint32)
    b[rng.random((V, n)) < 0.03] = 0x7F800001
    b[rng.random((V, n)) < 0.02] = 0x7F800002
    b[rng.random((V, n)) < 0.02] = 0x7FC00000
    b[rng.random((V, n)) < 0.01] = 0xFF800005
    slab = pad16(ds)
    rows = random_rows(rng, V, n_rows=V + 10)
    check(nb, slab, n, rows, lambda r: called_ds(slab[r["gt_row"]], n), oracle_gt=slab.view(np.float32), width=4, ploidy=1,
          dosage=True)


def test_pl_with_odd_eaf(nb):
    rng = np.random.default_rng(14)
    n, V = 1201, 40
    words = np.zeros((V, n), np.uint32)
    for v in range(V):
        pl, cnt, miss = random_pl(rng, n, haploid_rate=float(rng.choice([0, 0.3, 1])), miss_rate=0.05)
        words[v] = pack_words(pl, cnt, miss)
    slab = pad16(words)
    rows = random_rows(rng, V, n_rows=V + 10, nan_eaf_rate=0.0)
    rows["eaf"][:6] = [np.nan, -0.25, 1.5, 0.0, 1.0, 0.5]
    rows["kind"][:6] = 0
    rows["gt_row"][:6] = np.arange(6)
    rows["eaidx"][:6] = [1, 0, 1, 0, 1, 0]
    check(nb, slab, n, rows, lambda r: called_pl(slab[r["gt_row"]], n, r["eaf"], r["eaidx"]), width=nb.GT_PL, maxmis=1.0)


def test_wide_cohort_mode3(nb):
    rng = np.random.default_rng(15)
    n, V = 1_300_000, 6
    slab, rows, called_of, ogt = gt_case(rng, n, V)
    eng = nb.Engine(n, max_rows_per_block=64)
    assert eng.kernel_shape["fused"] == 3
    eng.close()
    for exact in (False, True):
        check(nb, slab, n, rows, called_of, oracle_gt=ogt if exact else None, exact=exact)


def test_split_calls_equal_one_call(nb):
    rng = np.random.default_rng(16)
    n = 2000
    slab, rows, called_of, _ = gt_case(rng, n, 40)
    a, oa = check(nb, slab, n, rows, called_of, split=True)
    b, ob = check(nb, slab, n, rows, called_of)
    assert np.array_equal(oa, ob)


def resident_engine(nb, slab, n):
    eng = nb.Engine(n, max_rows_per_block=4096, n_slots=2, staging_rows=len(slab))
    eng.set_policy(maxmis=0.5, mincs=5)
    eng.reset()
    assert eng.resident_reserve(len(slab)) >= len(slab)
    slot, view = eng.stage_acquire()
    view[:len(slab), :slab.shape[1]] = slab
    eng.stage_upload(slot, len(slab), 0)
    return eng


@pytest.mark.parametrize("S", [2, 3, 18])
@pytest.mark.parametrize("multi", ["0", "1"])
def test_multi_equals_single(nb, monkeypatch, S, multi):
    monkeypatch.setenv("NPC_MULTI", multi)
    rng = np.random.default_rng(S)
    n, V = 2500, 60
    slab, _, called_of, _ = gt_case(rng, n, V)
    lists = [random_rows(rng, V, n_rows=int(rng.integers(30, 90))) for _ in range(S)]
    eng = resident_engine(nb, slab, n)
    eng.set_observed(True)                             # the context's own counts: a multi call resets them on either path
    eng.score_resident(lists[0])
    assert eng.observed().sum() > 0
    before = eng.multi_contractions
    out = eng.score_resident_multi(lists, [0.0] * S, observed=True)
    assert (eng.multi_contractions > before) == (multi == "1")
    for rows, (sc, nloci, loci, obs) in zip(lists, out):
        single, want, _ = score(nb, slab, n, rows)
        assert_loci_equal(loci, single["loci"])
        assert np.array_equal(obs, want)
        assert np.array_equal(obs, observed(called_of, rows, loci, n))
    assert not eng.observed().any()
    plain = eng.score_resident_multi(lists, [0.0] * S)
    for (sc, _, loci, _), (sc2, _, loci2) in zip(out, plain):
        assert np.array_equal(bits(sc), bits(sc2))
        assert_loci_equal(loci, loci2)
    eng.close()


# ---- host paths -------------------------------------------------------------------------------------------------------


def host_case(tmp_path, seed=0, n=240):
    rng = np.random.default_rng(seed)
    d = make_dataset(tmp_path, rng, n=n, V=90)
    return rng, d


def check_host(r):
    assert r.observed is not None and r.observed.dtype == np.int64
    assert int(r.observed.sum()) == ngt_total(r.loci)
    assert (r.observed <= r.nloci).all()


def test_cli_set1(tmp_path):
    want = [([], [3, 4, 2, 2, 2, 3]), (["--maxmis", "0.2"], [3, 3, 2, 2, 2, 3]), (["--ignorefilt"], [4, 5, 3, 2, 2, 3]),
            (["--cov", os.path.join(S1, "set1.bed")], [1, 1, 1, 0, 1, 1])]
    code = "import sys; from nimpress_b200 import api; sys.exit(api.main(sys.argv[1:]))"
    for extra, counts in want:
        args = ["--maxmis", "1.0"] + extra + [os.path.join(S1, "set1.score"), os.path.join(S1, "set1.vcf.gz")]
        plain = subprocess.run([sys.executable, "-c", code, *args], capture_output=True, text=True, cwd=ROOT, timeout=300)
        obs = subprocess.run([sys.executable, "-c", code, "--observed", *args], capture_output=True, text=True, cwd=ROOT, timeout=300)
        assert plain.returncode == 0 and obs.returncode == 0, obs.stderr
        p_lines, o_lines = plain.stdout.split("\n"), obs.stdout.split("\n")
        assert len(p_lines) == len(o_lines)
        rows = [(p, o) for p, o in zip(p_lines, o_lines) if p and not p.startswith("WARN")]
        assert all(p == o for p, o in zip(p_lines, o_lines) if not p or p.startswith("WARN"))
        assert [o for _, o in rows] == [p + "\t" + str(c) for (p, _), c in zip(rows, counts)] and len(rows) == len(counts)
        cov = extra[1] if extra[:1] == ["--cov"] else None
        oracle = oracle_observed_files(args[-2], args[-1], tmp_path, cov, maxmis=0.2 if "0.2" in extra else 1.0,
                                       ignorefilt="--ignorefilt" in extra)
        assert oracle.tolist() == counts


def test_host_unchanged_and_exact(api, tmp_path):
    _, d = host_case(tmp_path)
    for ex in (False, True):
        a = api.run(d["score"], d["bcf"], exact_order=ex)
        b = api.run(d["score"], d["bcf"], exact_order=ex, observed=True)
        assert a.observed is None
        assert np.array_equal(bits(a.scores), bits(b.scores)) and a.warnings == b.warnings
        assert_loci_equal(a.loci, b.loci)
        check_host(b)


def test_host_samples_equals_subset_file(api, tmp_path):
    rng, d = host_case(tmp_path, 1)
    keep = np.sort(rng.choice(len(d["samples"]), size=150, replace=False))
    lst = tmp_path / "keep.txt"
    lst.write_text("".join(d["samples"][i] + "\n" for i in keep))
    sub = [dict(r, gt=np.asarray(r["gt"])[keep]) for r in d["records"]]
    path = str(tmp_path / "sub.vcf.gz")
    write_vcf(path, [d["samples"][i] for i in keep], sub, contigs=CONTIGS, filters=("FAIL", "LowQ"), compress="bgzf")
    got = api.run(d["score"], d["vcf"], samples=str(lst), observed=True)
    want = api.run(d["score"], path, observed=True)
    check_host(got)
    assert np.array_equal(got.observed, want.observed) and np.array_equal(bits(got.scores), bits(want.scores))
    assert np.array_equal(got.observed, oracle_observed_files(d["score"], path, tmp_path))


def test_host_files_rounds_split_multi(api, tmp_path, monkeypatch):
    rng, d = host_case(tmp_path, 2)
    plain = api.run(d["score"], d["vcf"], observed=True)
    check_host(plain)
    assert np.array_equal(plain.observed, oracle_observed_files(d["score"], d["vcf"], tmp_path))
    parts, cat = write_split("vcf", tmp_path, "part", d["samples"], by_contig(d["records"]))
    split_files = api.run(d["score"], parts, observed=True)
    assert np.array_equal(split_files.observed, api.run(d["score"], cat, observed=True).observed)
    assert np.array_equal(split_files.observed, oracle_observed_files(d["score"], cat, tmp_path))
    with monkeypatch.context() as m:
        m.setenv("NIMPRESS_SLAB_ROWS", "7")
        r = api.run(d["score"], d["vcf"], observed=True)
        assert r.rounds > 1 and np.array_equal(r.observed, plain.observed)
    with monkeypatch.context() as m:
        m.setenv("NIMPRESS_SPLIT", "3")
        r = api.run(d["score"], d["vcf"], observed=True)
        assert r.devices == 3 and np.array_equal(r.observed, plain.observed)
    files = derive_scores(tmp_path, rng, d["entries"], 18)
    for multi in ("0", "1"):
        with monkeypatch.context() as m:
            m.setenv("NPC_MULTI", multi)
            for S in (2, 3, 18):
                got = api.run_multi(files[:S], d["vcf"], observed=True)
                for f, g in zip(files[:S], got):
                    w = api.run(f, d["vcf"], observed=True)
                    assert np.array_equal(g.observed, w.observed), (multi, S, f)
                    if multi == "1" and S == 3:
                        assert np.array_equal(g.observed, oracle_observed_files(f, d["vcf"], tmp_path))
                    assert_loci_equal(g.loci, w.loci)
