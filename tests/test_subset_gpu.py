"""GPU tests of --samples and subset contexts (DESIGN.md 4.11).  The oracle for every case is the same engine on a file
that the test writers produce with only the kept samples (same records, same order): scores bit for bit in the default
order and with --exact-order, per-locus records field by field, nloci, the WARN text and the sample names.  At the C ABI,
npc_create_subset against npc_create2 on rows compacted in numpy, and npc_gather_rows_device against a numpy gather."""
import numpy as np
import pytest

from util_bcf import write_bcf, write_vcf
from util_bgen import records_to_variants, write_bgen
from util_bgen_bits import VEND8, records_to_variants_bits, split_records_keep_haploid
from util_cohort import assert_loci_equal, bits, random_cohort, random_rows
from util_files import derive_scores, make_dataset
from util_pl import with_pl, write_bcf_pl, write_vcf_pl
from util_plink import split_records, write_plink

pytestmark = pytest.mark.gpu
CONTIGS = ["1", "2", "X"]
PER_SAMPLE = ("gt", "ds", "pl", "plcnt", "plmiss", "plpartial")


@pytest.fixture(scope="module")
def api():
    import __graft_entry__ as g
    g.build()
    from nimpress_b200 import api
    api.load_host_library()
    return api


@pytest.fixture(scope="module")
def nb():
    import nimpress_b200
    return nimpress_b200


def sub_records(records, keep):
    return [dict(r, **{k: np.asarray(r[k])[keep] for k in PER_SAMPLE if k in r}) for r in records]


def write_kind(kind, path, samples, records, seed=0):
    """The genotype file of one layout; the BGEN writers draw their phasing from `seed`, so that the full file and the
    subsetted one phase the same variants."""
    rng = np.random.default_rng(seed)
    if kind in ("vcf", "ds"):
        write_vcf(path, samples, records, contigs=CONTIGS, filters=("FAIL", "LowQ"), compress="bgzf")
    elif kind == "bcf":
        write_bcf(path, samples, records, contigs=CONTIGS, filters=("FAIL", "LowQ"), compress="bgzf")
    elif kind == "bed":
        return write_plink(path[:-4], samples, records)
    elif kind == "bgen8":
        write_bgen(path, samples, records_to_variants(records, len(samples), rng))
    elif kind == "bgen16":
        write_bgen(path, samples, records_to_variants_bits(records, len(samples), 16, rng))
    elif kind == "pl_vcf":
        write_vcf_pl(path, samples, records, CONTIGS)
    elif kind == "pl_bcf":
        write_bcf_pl(path, samples, records, CONTIGS)
    return path


EXT = dict(vcf=".vcf.gz", ds=".vcf.gz", bcf=".bcf", bed=".bed", bgen8=".bgen", bgen16=".bgen", pl_vcf=".vcf.gz", pl_bcf=".bcf")


def dataset(tmp, kind, n, seed):
    """(score path, samples, records) of one layout: int8 / int16 / triploid-with-haploid GT, FORMAT/DS, split biallelic
    records for .bed and BGEN (16-bit with haploid samples), random FORMAT/PL."""
    rng = np.random.default_rng(seed)
    kw = dict(gt_dtype=np.int16) if kind == "bcf16" else dict(ploidy=3, haploid_rate=0.2) if kind == "bcf3" else {}
    d = make_dataset(tmp, rng, n=n, V=90, **kw)
    recs = d["records"]
    if kind in ("ds", "bed", "bgen8", "pl_vcf", "pl_bcf"):
        recs = split_records(recs)
    if kind == "ds":
        for r in recs:
            r["ds"] = np.where(rng.random(n) < 0.03, np.nan, np.round(rng.uniform(0, 2, n), 3)).astype(np.float32)
    if kind == "bgen16":
        for r in recs:
            r["gt"] = np.where((rng.random(n) < 0.15)[:, None] & (np.arange(2) == 1), VEND8, r["gt"]).astype(np.int8)
        recs = split_records_keep_haploid(recs)
    if kind.startswith("pl"):
        recs = with_pl([r for r in recs if r["alts"]], n, rng, haploid_rate=0.1)        # FORMAT/PL: biallelic records only
    return d["score"], d["samples"], recs


def file_kind(kind):
    return "bcf" if kind in ("bcf16", "bcf3") else kind


def compare(api, score, full, sub, keep_names, tmp, exact=(False, True), multi=None, exclude=None, **kw):
    """--samples on `full` against the plain run on `sub`, in both summation orders."""
    lst = str(tmp / "keep.txt")
    with open(lst, "w") as fh:
        fh.write("\n".join(exclude if exclude is not None else keep_names) + "\n")
    for ex in exact:
        if multi:
            got = api.run_multi(multi, full, exact_order=ex, samples=lst, exclude_samples=exclude is not None, **kw)
            want = api.run_multi(multi, sub, exact_order=ex, **kw)
        else:
            got = [api.run(score, full, exact_order=ex, samples=lst, exclude_samples=exclude is not None, **kw)]
            want = [api.run(score, sub, exact_order=ex, **kw)]
        for g, w in zip(got, want):
            assert g.samples == w.samples == list(keep_names)
            assert g.nloci == w.nloci and g.warnings == w.warnings
            assert_loci_equal(g.loci, w.loci)
            assert np.array_equal(bits(g.scores), bits(w.scores))
    return got


def shapes(rng, n):
    """The subset shapes: a random 10 % and 50 %, all but one, a single sample, 37 samples (not a multiple of 4, 8 or
    16), a contiguous range."""
    return {"10%": np.sort(rng.choice(n, n // 10, replace=False)), "50%": np.sort(rng.choice(n, n // 2, replace=False)),
            "all_but_one": np.delete(np.arange(n), int(rng.integers(n))), "one": np.array([int(rng.integers(n))]),
            "37": np.sort(rng.choice(n, 37, replace=False)), "range": np.arange(n // 3, n // 3 + n // 4)}


@pytest.mark.parametrize("kind", ["vcf", "bcf", "bcf16", "bcf3", "ds", "bed", "bgen8", "bgen16", "pl_vcf", "pl_bcf"])
def test_every_layout_equals_subsetted_file(api, tmp_path, kind):
    """Every row layout (int8 GT from VCF text and BCF, int16 GT, triploid GT with haploid samples on the generic
    kernels, FORMAT/DS, .bed, 8-bit BGEN, 16-bit BGEN with haploid samples, FORMAT/PL from VCF text and BCF) under every
    subset shape scores as the file holding only the kept samples."""
    n = 203
    score, samples, recs = dataset(str(tmp_path), kind, n, seed=sum(map(ord, kind)))
    fk = file_kind(kind)
    full = write_kind(fk, str(tmp_path / ("full" + EXT[fk])), samples, recs, seed=3)
    kw = dict(dosage=True) if kind == "ds" else dict(pl=True) if kind.startswith("pl") else {}
    for name, keep in shapes(np.random.default_rng(11), n).items():
        sub = write_kind(fk, str(tmp_path / (f"sub_{name}" + EXT[fk])), [samples[i] for i in keep], sub_records(recs, keep), seed=3)
        compare(api, score, full, sub, [samples[i] for i in keep], tmp_path,
                exact=(False, True) if name in ("50%", "37") else (False,), **kw)


def test_every_sample_listed_is_the_plain_run(api, tmp_path):
    """A keep list naming every sample, and an exclude list naming only samples the file lacks, give what no list gives."""
    score, samples, recs = dataset(str(tmp_path), "bcf", 150, seed=4)
    full = write_kind("bcf", str(tmp_path / "full.bcf"), samples, recs)
    compare(api, score, full, full, samples, tmp_path)
    compare(api, score, full, full, samples, tmp_path, exclude=["ghost1", "ghost2"])


def test_exclude_list(api, tmp_path):
    """--samples=^FILE drops the listed samples; names the file lacks are ignored."""
    score, samples, recs = dataset(str(tmp_path), "bcf", 211, seed=5)
    full = write_kind("bcf", str(tmp_path / "full.bcf"), samples, recs)
    drop = np.sort(np.random.default_rng(2).choice(211, 30, replace=False))
    keep = np.setdiff1d(np.arange(211), drop)
    sub = write_kind("bcf", str(tmp_path / "sub.bcf"), [samples[i] for i in keep], sub_records(recs, keep))
    compare(api, score, full, sub, [samples[i] for i in keep], tmp_path, exclude=[samples[i] for i in drop] + ["withdrawn_elsewhere"])


@pytest.mark.parametrize("env", [dict(NIMPRESS_SPLIT="3"), dict(NIMPRESS_SLAB_ROWS="7")])
def test_split_contexts_and_rounds(api, tmp_path, monkeypatch, env):
    """Three contexts on one GPU (every one created with the subset, combined by npc_reduce), and scoring in rounds of
    seven resident rows."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    for kind in ("bcf", "bed"):
        score, samples, recs = dataset(str(tmp_path), kind, 251, seed=6)
        full = write_kind(kind, str(tmp_path / ("full" + EXT[kind])), samples, recs)
        keep = np.sort(np.random.default_rng(3).choice(251, 120, replace=False))
        sub = write_kind(kind, str(tmp_path / ("sub" + EXT[kind])), [samples[i] for i in keep], sub_records(recs, keep))
        got = compare(api, score, full, sub, [samples[i] for i in keep], tmp_path)
        if "NIMPRESS_SLAB_ROWS" in env:
            assert got[0].rounds > 1


def test_three_score_files(api, tmp_path):
    """Three score files in one pass (the tensor-core contraction on int8 diploid rows) equal the same call on the
    subsetted file."""
    rng = np.random.default_rng(7)
    d = make_dataset(str(tmp_path), rng, n=400, V=150)
    paths = [d["score"]] + derive_scores(str(tmp_path), rng, d["entries"], 3)
    keep = np.sort(rng.choice(400, 173, replace=False))
    sub = write_kind("bcf", str(tmp_path / "sub.bcf"), [d["samples"][i] for i in keep], sub_records(d["records"], keep))
    compare(api, None, d["bcf"], sub, [d["samples"][i] for i in keep], tmp_path, multi=paths)


def test_bgen_dropped_haploid_sample_restart(api, tmp_path, capfd, monkeypatch):
    """A BGEN file whose dropped sample is haploid: the full rows need 32-bit rows (the pass restarts with NPC_GT_DOSE32),
    the subsetted file takes 2-byte rows; D = 255 diploid rows score bit for bit as 2-byte rows (DESIGN.md 4.9)."""
    score, samples, recs = dataset(str(tmp_path), "bgen8", 160, seed=8)
    for r in recs:
        r["gt"] = r["gt"].copy()
        r["gt"][5, 1] = VEND8                                           # sample 5 is haploid everywhere
    rng = np.random.default_rng(1)
    full = str(tmp_path / "full.bgen")
    write_bgen(full, samples, records_to_variants_bits(recs, 160, 8, rng))
    keep = np.delete(np.arange(160), 5)
    sub = str(tmp_path / "sub.bgen")
    write_bgen(sub, [samples[i] for i in keep], records_to_variants_bits(sub_records(recs, keep), 159, 8, np.random.default_rng(1)))
    monkeypatch.setenv("NIMPRESS_TIMING", "1")
    capfd.readouterr()
    compare(api, score, full, sub, [samples[i] for i in keep], tmp_path)
    err = capfd.readouterr().err
    assert "restart with 32-bit dosage rows" in err


# ---- C ABI -------------------------------------------------------------------------------------------------------------

LAYOUTS = [(2, 1), (2, 2), (1, 4), (1, 1), (3, 1), (2, 4), (2, 255), (2, 32), (2, 10), (2, 0)]    # (ploidy, gt_width)


def numpy_gather(nb, rows, n_row, keep, ploidy, width):
    """Compact rows in numpy: the kept samples' bytes (the 16-byte header of NPC_GT_DOSE32 rows first; .bed codes
    repacked four to a byte)."""
    keep = np.asarray(keep)
    if width == nb.GT_BED:
        codes = (rows[:, :, None] >> (2 * np.arange(4))) & 3
        codes = codes.reshape(len(rows), -1)[:, keep]
        codes = np.pad(codes, ((0, 0), (0, -len(keep) % 4)))
        q = codes.reshape(len(rows), -1, 4).astype(np.uint8)
        return (q[..., 0] | (q[..., 1] << 2) | (q[..., 2] << 4) | (q[..., 3] << 6)).astype(np.uint8)
    hdr = 16 if width == nb.GT_DOSE32 else 0
    E = 2 if width == nb.GT_DOSE255 else 4 if width in (nb.GT_DOSE32, nb.GT_PL) else ploidy * width
    el = rows[:, hdr:hdr + n_row * E].reshape(len(rows), n_row, E)[:, keep].reshape(len(rows), -1)
    return np.concatenate([rows[:, :hdr], el], axis=1)


def test_gather_rows_device_equals_numpy(nb):
    """npc_gather_rows_device on random bytes, for every layout: the compact row's bytes equal a numpy gather (.bed: the
    codes of the kept samples; the padding codes of the last byte are free)."""
    import torch
    rng = np.random.default_rng(9)
    for ploidy, width in LAYOUTS:
        for n_row, n_keep in ((1, 1), (1000, 1), (1000, 999), (1003, 37), (4099, 2050), (70001, 7000)):
            keep = np.sort(rng.choice(n_row, n_keep, replace=False))
            eng = nb.Engine(0, ploidy=ploidy, gt_width=width, max_rows_per_block=64, keep=keep, n_row_samples=n_row)
            V = 5
            sb, db = nb.gt_row_bytes(n_row, ploidy, width), nb.gt_row_bytes(n_keep, ploidy, width)
            ss, ds = -(-sb // 16) * 16 + 16, -(-db // 16) * 16 + 32
            src = rng.integers(0, 256, size=(V, ss), dtype=np.uint8)
            d_src = torch.from_numpy(src).cuda()
            d_dst = torch.full((V, ds), 0xAB, dtype=torch.uint8, device="cuda")
            eng.gather_rows_device(d_src, ss, V, d_dst, ds)
            torch.cuda.synchronize()
            got = d_dst.cpu().numpy()
            want = numpy_gather(nb, src[:, :sb], n_row, keep, ploidy, width)
            if width == nb.GT_BED:
                full = n_keep // 4
                assert np.array_equal(got[:, :full], want[:, :full]), (ploidy, width, n_row, n_keep)
                if n_keep % 4:
                    m = (1 << (2 * (n_keep % 4))) - 1
                    assert np.array_equal(got[:, full] & m, want[:, full] & m)
            else:
                assert np.array_equal(got[:, :db], want), (ploidy, width, n_row, n_keep)
            eng.close()
    plain = nb.Engine(10, max_rows_per_block=8)
    with pytest.raises(nb.NpcError, match="rc=-4"):
        plain.gather_rows_device(0, 16, 0, 0, 16)
    plain.close()


def run_engine(nb, n, rows, gt, exact, keep=None, n_row=None, width=1, block=32, resident=False):
    eng = nb.Engine(n, gt_width=width, max_rows_per_block=max(block, len(rows)), n_slots=3, staging_rows=block, keep=keep,
                    n_row_samples=n_row)
    eng.set_policy()
    eng.set_exact_order(exact)
    eng.reset()
    V = gt.shape[0]
    if resident:
        assert eng.resident_reserve(V) >= V
        for v0 in range(0, V, block):
            slot, view = eng.stage_acquire()
            view[:min(block, V - v0), :gt.shape[1]] = gt[v0:v0 + block]
            eng.stage_upload(slot, min(block, V - v0), v0)
        eng.score_resident(rows)
    else:
        for v0 in range(0, V, block):                       # each block's score rows name its own genotype rows
            r = rows[(rows["gt_row"] >= v0) & (rows["gt_row"] < v0 + block)].copy()
            r["gt_row"] -= v0
            slot, view = eng.stage_acquire()
            view[:min(block, V - v0), :gt.shape[1]] = gt[v0:v0 + block]
            eng.score_block(slot, min(block, V - v0), r)
    out = eng.finish(offset=0.5)
    shape = eng.kernel_shape
    eng.close()
    return out, shape


def check(a, b):
    assert a["nloci"] == b["nloci"]
    assert_loci_equal(a["loci"], b["loci"])
    assert np.array_equal(bits(a["scores"]), bits(b["scores"]))


@pytest.mark.parametrize("width", [1, 0])
def test_create_subset_streaming_equals_create2_on_compact_rows(nb, width):
    """npc_create_subset with npc_score_block streaming and with npc_stage_upload into the resident slab equals
    npc_create2 on rows compacted in numpy: int8 diploid GT (the tile kernel) and .bed rows, both summation orders."""
    rng = np.random.default_rng(12)
    n_row, V = 3001, 96
    gt = random_cohort(rng, n_row, V, miss_rate=0.05)
    keep = np.sort(rng.choice(n_row, 1234, replace=False))
    rows = random_rows(rng, V, n_rows=V, shuffle_gt=False)
    rows = rows[np.argsort(np.where(rows["gt_row"] < 0, V, rows["gt_row"]), kind="stable")]
    if width == nb.GT_BED:
        from util_plink import pack_cohort
        rows["eaidx"] = np.where(rows["kind"] == 0, rows["eaidx"] % 2, rows["eaidx"])
        gt = pack_cohort(gt, n_row)
        compact = numpy_gather(nb, gt, n_row, keep, 2, width)
    else:
        compact = numpy_gather(nb, gt.view(np.uint8)[:, :2 * n_row], n_row, keep, 2, 1)
    for exact in (False, True):
        for resident in (False, True):
            a, sa = run_engine(nb, len(keep), rows, gt.view(np.uint8), exact, keep=keep, n_row=n_row, width=width, resident=resident)
            b, sb = run_engine(nb, len(keep), rows, compact, exact, width=width, resident=resident)
            check(a, b)
            assert sa == sb


def test_wide_cohort_takes_one_read_tile_kernel(nb):
    """n_row_samples = 1,300,000 with 500,000 kept: the subset context reports the one-read tile kernel (mode 2) where
    the whole cohort takes the two-read wide mode (3), and its scores equal a plain 500,000-sample context on the
    compacted rows."""
    rng = np.random.default_rng(13)
    n_row, n_keep, V = 1_300_000, 500_000, 24
    lut = np.select([np.arange(256) < 5, np.arange(256) < 120, np.arange(256) < 200], [0, 2, 3], 4).astype(np.int8)
    gt = lut[rng.integers(0, 256, size=(V, 2 * n_row), dtype=np.uint8)]      # ./., 0/0, 0|1 and 1/1 without numpy temporaries
    keep = np.sort(rng.choice(n_row, n_keep, replace=False))
    rows = random_rows(rng, V, n_rows=V, shuffle_gt=False)
    rows = rows[np.argsort(np.where(rows["gt_row"] < 0, V, rows["gt_row"]), kind="stable")]
    compact = numpy_gather(nb, gt.view(np.uint8)[:, :2 * n_row], n_row, keep, 2, 1)
    a, sa = run_engine(nb, n_keep, rows, gt.view(np.uint8), False, keep=keep, n_row=n_row, block=8, resident=True)
    b, sb = run_engine(nb, n_keep, rows, compact, False, block=8, resident=True)
    assert sa["fused"] == 2 and sa == sb
    whole = nb.Engine(n_row, max_rows_per_block=8)
    assert whole.kernel_shape["fused"] == 3
    whole.close()
    check(a, b)
