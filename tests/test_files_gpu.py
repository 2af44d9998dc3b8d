"""GPU tests of several genotype files read as their concatenation (DESIGN.md 4.12).  The oracle for every case is the
same engine on the one file that the test writers produce from the parts' records in order: scores bit for bit in the
default order and with --exact-order, per-locus records field by field, nloci, the WARN text, the sample names and
records_read.  At the C ABI, npc_set_keep between two staged "files" of different widths against npc_create2 on rows
compacted in numpy, and npc_gather_rows_device under each keep list against a numpy gather."""
import os
import subprocess

import numpy as np
import pytest

from util_cohort import assert_loci_equal, bits, random_cohort, random_rows
from util_files import derive_scores, make_dataset
from util_pl import with_pl
from util_plink import split_records
from util_split import by_contig, chunks, write_split

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
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


def dataset(tmp, kind, n, seed):
    """(score path, samples, records) of one layout: int8 / int16 / triploid-with-haploid GT, FORMAT/DS, split biallelic
    records for .bed and BGEN, random FORMAT/PL."""
    rng = np.random.default_rng(seed)
    kw = dict(gt_dtype=np.int16) if kind == "bcf16" else dict(ploidy=3, haploid_rate=0.2) if kind == "bcf3" else {}
    d = make_dataset(tmp, rng, n=n, V=90, **kw)
    recs = d["records"]
    if kind in ("ds", "bed", "bgen8", "bgen_last16", "pl_vcf", "pl_bcf"):
        recs = split_records(recs)
    if kind == "ds":
        for r in recs:
            r["ds"] = np.where(rng.random(n) < 0.03, np.nan, np.round(rng.uniform(0, 2, n), 3)).astype(np.float32)
    if kind.startswith("pl"):
        recs = with_pl([r for r in recs if r["alts"]], n, rng, haploid_rate=0.1)
    return d["score"], d["samples"], recs


def file_kind(kind):
    return "bcf" if kind in ("bcf16", "bcf3") else kind


def options(kind):
    return dict(dosage=True) if kind == "ds" else dict(pl=True) if kind.startswith("pl") else {}


def check_same(g, w):
    assert g.samples == w.samples
    assert g.nloci == w.nloci and g.warnings == w.warnings and g.records_read == w.records_read
    assert_loci_equal(g.loci, w.loci)
    assert np.array_equal(bits(g.scores), bits(w.scores))


def compare(api, score, parts, cat, exact=(False, True), multi=None, **kw):
    """The run over the parts against the run over their concatenation, in both summation orders."""
    out = []
    for ex in exact:
        if multi:
            got, want = api.run_multi(multi, parts, exact_order=ex, **kw), api.run_multi(multi, cat, exact_order=ex, **kw)
        else:
            got, want = [api.run(score, parts, exact_order=ex, **kw)], [api.run(score, cat, exact_order=ex, **kw)]
        for g, w in zip(got, want):
            check_same(g, w)
        out.append(got)
    return out


@pytest.mark.parametrize("kind", ["vcf", "bcf", "bcf16", "bcf3", "ds", "bed", "bgen8", "bgen_last16", "pl_vcf", "pl_bcf"])
def test_every_layout_equals_concatenation(api, tmp_path, kind, capfd, monkeypatch):
    """Every row layout, split per contig and in three chunks whose boundaries repeat a site (the earlier file's copy
    wins), scores as the concatenated file.  bgen_last16: 8-bit BGEN whose last file holds 16-bit blocks, so that the
    pass restarts once with 32-bit rows, from the first file."""
    score, samples, recs = dataset(str(tmp_path), kind, 157, seed=sum(map(ord, kind)))
    if kind == "bgen_last16":
        monkeypatch.setenv("NIMPRESS_TIMING", "1")
    for name, parts in (("contig", by_contig(recs)), ("chunk", chunks(recs, 3))):
        paths, cat = write_split(file_kind(kind), str(tmp_path), name, samples, parts, seed=3)
        exact = (False, True) if name == "chunk" else (False,)
        capfd.readouterr()
        compare(api, score, paths, cat, exact=exact, **options(kind))
        if kind == "bgen_last16":                                                   # one restart per run: parts, then file
            err = capfd.readouterr().err
            assert err.count("restart with 32-bit dosage rows") == 2 * len(exact), err


def test_int16_in_the_last_file_restarts_the_layout(api, tmp_path):
    """int8 GT in the first files and int16 in the last: the layout restart re-reads every file with int16 rows and
    scores as the concatenation (which restarts the same way)."""
    score, samples, recs = dataset(str(tmp_path), "bcf", 141, seed=9)
    parts = chunks(recs, 3, dup=False)
    parts[-1] = [dict(r, gt=np.asarray(r["gt"]).astype(np.int16)) for r in parts[-1]]
    paths, cat = write_split("bcf", str(tmp_path), "w", samples, parts)
    compare(api, score, paths, cat)


def test_permuted_file_order(api, tmp_path):
    """Per-contig files in another order: the same as their concatenation in that order, and, with no site in two
    files, bit for bit the same as the files in their first order (summation follows the score file)."""
    score, samples, recs = dataset(str(tmp_path), "bcf", 177, seed=10)
    parts = by_contig(recs)
    paths, _ = write_split("bcf", str(tmp_path), "p", samples, parts)
    first = [api.run(score, paths, exact_order=ex) for ex in (False, True)]
    perm = [2, 0, 1]
    ppaths, pcat = write_split("bcf", str(tmp_path), "q", samples, [parts[i] for i in perm])
    for ex, got in zip((False, True), compare(api, score, ppaths, pcat)):
        assert np.array_equal(bits(got[0].scores), bits(first[ex].scores))
        assert_loci_equal(got[0].loci, first[ex].loci)
        assert got[0].warnings == first[ex].warnings


def write_chrx_case(tmp, kind, n, seed):
    """Autosome files with all n samples and a last (chrX-like) file lacking four of them; a keep list of samples
    present in every file.  Returns (score, part paths, keep-list path, concatenated file of the kept samples)."""
    score, samples, recs = dataset(tmp, kind, n, seed)
    parts = by_contig(recs)
    rng = np.random.default_rng(seed)
    lacking = np.sort(rng.choice(n, 4, replace=False))
    x_keep = np.setdiff1d(np.arange(n), lacking)
    keep = np.sort(np.setdiff1d(x_keep, rng.choice(n, n // 5, replace=False)))
    sub = lambda rs, idx: [dict(r, **{f: np.asarray(r[f])[idx] for f in PER_SAMPLE if f in r}) for r in rs]
    x_samples = [samples[i] for i in x_keep]
    paths, _ = write_split(kind, tmp, "f", samples, parts[:-1] + [sub(parts[-1], x_keep)], seed=3,
                           part_samples=[samples] * (len(parts) - 1) + [x_samples])
    kept = [samples[i] for i in keep]
    _, cat = write_split(kind, tmp, "kept", kept, [sub(p, keep) for p in parts], seed=3)     # the same BGEN phasing draws
    lst = os.path.join(tmp, "keep.txt")
    with open(lst, "w") as fh:
        fh.write("\n".join(kept) + "\n")
    return score, paths, lst, cat


@pytest.mark.parametrize("kind", ["bcf", "bed", "bgen8"])
def test_chrx_file_lacking_samples_with_keep_list(api, tmp_path, kind):
    """A last file that lacks some samples, with --samples naming samples present in every file: each file is compacted
    with its own keep list (npc_set_keep) and the result is the concatenated file holding only the kept samples."""
    score, paths, lst, cat = write_chrx_case(str(tmp_path), kind, 203, seed=11)
    for ex in (False, True):
        check_same(api.run(score, paths, exact_order=ex, samples=lst), api.run(score, cat, exact_order=ex))


@pytest.mark.parametrize("env", [dict(NIMPRESS_SPLIT="3"), dict(NIMPRESS_SLAB_ROWS="7")])
def test_split_contexts_and_rounds_across_files(api, tmp_path, monkeypatch, env):
    """Three contexts on one GPU, and rounds of seven resident rows that straddle file boundaries: on plain files and on
    the chrX case with a keep list."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    score, samples, recs = dataset(str(tmp_path), "bcf", 191, seed=12)
    paths, cat = write_split("bcf", str(tmp_path), "c", samples, chunks(recs, 4))
    got = compare(api, score, paths, cat)
    if "NIMPRESS_SLAB_ROWS" in env:
        assert got[0][0].rounds > 1
    score, paths, lst, cat = write_chrx_case(str(tmp_path), "bcf", 163, seed=13)
    check_same(api.run(score, paths, samples=lst), api.run(score, cat))


def with_absent_tail(score, path):
    """The score file followed by twice its rows again on a contig no genotype file holds: the last third of the rows
    (the last device's range under NIMPRESS_SPLIT=3) never matches a record."""
    lines = open(score).read().rstrip("\n").split("\n")
    head, rows = lines[:5], lines[5:]
    tail = [f"absent\t{1000 + 7 * i}\tA\tG\t0.01\t0.2" for i in range(2 * len(rows))]
    with open(path, "w") as fh:
        fh.write("\n".join(head + rows + tail) + "\n")
    return path


def test_context_without_rows_under_samples(api, tmp_path, monkeypatch):
    """With --samples and three contexts on one GPU, the context whose range matches no record is opened only after the
    stream: on one file and on several (the chrX case), it is created with a valid keep list and the result equals
    the run on the file holding only the kept samples."""
    monkeypatch.setenv("NIMPRESS_SPLIT", "3")
    score, paths, lst, cat = write_chrx_case(str(tmp_path), "bcf", 173, seed=17)
    score = with_absent_tail(score, str(tmp_path / "tail.score"))
    for ex in (False, True):
        check_same(api.run(score, paths, exact_order=ex, samples=lst), api.run(score, cat, exact_order=ex))
    # one file with a keep list
    full_score, samples, recs = dataset(str(tmp_path), "bcf", 173, seed=18)
    full_score = with_absent_tail(full_score, str(tmp_path / "tail1.score"))
    keep = np.sort(np.random.default_rng(18).choice(173, 90, replace=False))
    _, full = write_split("bcf", str(tmp_path), "whole", samples, [recs])
    sub = [dict(r, gt=np.asarray(r["gt"])[keep]) for r in recs]
    _, only = write_split("bcf", str(tmp_path), "only", [samples[i] for i in keep], [sub])
    lst1 = str(tmp_path / "keep1.txt")
    with open(lst1, "w") as fh:
        fh.write("\n".join(samples[i] for i in keep) + "\n")
    for ex in (False, True):
        check_same(api.run(full_score, full, exact_order=ex, samples=lst1), api.run(full_score, only, exact_order=ex))


def test_three_score_files(api, tmp_path):
    """Three score files in one pass over four chunk files (the tensor-core contraction on int8 diploid rows)."""
    rng = np.random.default_rng(14)
    d = make_dataset(str(tmp_path), rng, n=400, V=150)
    multi = [d["score"]] + derive_scores(str(tmp_path), rng, d["entries"], 2)
    paths, cat = write_split("bcf", str(tmp_path), "m", d["samples"], chunks(d["records"], 4))
    compare(api, None, paths, cat, multi=multi)


@pytest.mark.parametrize("kind,k", [("bcf", 3), ("bgen8", 22)])
def test_cli_prints_what_the_concatenation_prints(api, tmp_path, kind, k):
    """nimpress score f1 ... fk prints byte for byte what nimpress score all prints: 3 BCF chunk files, and 22
    per-contig BGEN files."""
    rng = np.random.default_rng(15)
    contigs = tuple(str(c) for c in range(1, 23)) if k == 22 else ("1", "2", "X")
    d = make_dataset(str(tmp_path), rng, n=120, V=22 * 12, contigs=contigs)
    recs = split_records(d["records"]) if kind == "bgen8" else d["records"]
    parts = by_contig(recs) if k == 22 else chunks(recs, k)
    paths, cat = write_split(kind, str(tmp_path), "f", d["samples"], parts, seed=1)
    assert len(paths) == k
    a = subprocess.run([EXE, d["score"], *paths], capture_output=True)
    b = subprocess.run([EXE, d["score"], cat], capture_output=True)
    assert a.returncode == 0 and b.returncode == 0, a.stderr
    assert a.stdout == b.stdout and len(a.stdout) > 1000


# ---- C ABI -------------------------------------------------------------------------------------------------------------

def compact(rows, n_row, keep):
    """int8 diploid rows of n_row samples -> the kept samples' bytes."""
    return rows[:, :2 * n_row].reshape(len(rows), n_row, 2)[:, keep].reshape(len(rows), -1)


def test_set_keep_between_files_of_different_widths(nb):
    """A subset context over rows of 3001 samples scores 1234 of them; after npc_set_keep the next "file" carries 2500
    samples at the front of the same staging rows.  Scores, nloci and records equal npc_create2 on the rows compacted in
    numpy, resident and streaming, in both orders; npc_gather_rows_device follows each list."""
    import torch
    rng = np.random.default_rng(16)
    wide, narrow, m, V = 3001, 2500, 1234, 96
    ka = np.sort(rng.choice(wide, m, replace=False))
    kb = np.sort(rng.choice(narrow, m, replace=False))
    ga = random_cohort(rng, wide, V // 2, miss_rate=0.05).view(np.uint8)
    gb = random_cohort(rng, narrow, V // 2, miss_rate=0.05).view(np.uint8)
    comp = np.concatenate([compact(ga, wide, ka), compact(gb, narrow, kb)])
    rows = random_rows(rng, V, n_rows=V, shuffle_gt=False)
    rows = rows[np.argsort(np.where(rows["gt_row"] < 0, V, rows["gt_row"]), kind="stable")]
    for exact in (False, True):
        for resident in (False, True):
            outs = []
            for sub in (True, False):
                eng = nb.Engine(m, max_rows_per_block=V, n_slots=3, staging_rows=16, keep=ka if sub else None,
                                n_row_samples=wide if sub else None)
                eng.set_policy()
                eng.set_exact_order(exact)
                eng.reset()
                if resident:
                    assert eng.resident_reserve(V) >= V
                for v0 in range(0, V, 16):
                    if sub and v0 == V // 2:
                        eng.set_keep(kb)
                    src = (ga[v0:v0 + 16] if v0 < V // 2 else gb[v0 - V // 2:v0 - V // 2 + 16]) if sub else comp[v0:v0 + 16]
                    slot, view = eng.stage_acquire()
                    view[:len(src), :src.shape[1]] = src
                    if resident:
                        eng.stage_upload(slot, len(src), v0)
                    else:
                        r = rows[(rows["gt_row"] >= v0) & (rows["gt_row"] < v0 + 16)].copy()
                        r["gt_row"] -= v0
                        eng.score_block(slot, len(src), r)
                if resident:
                    eng.score_resident(rows)
                outs.append(eng.finish(offset=0.5))
                eng.close()
            a, b = outs
            assert a["nloci"] == b["nloci"]
            assert_loci_equal(a["loci"], b["loci"])
            assert np.array_equal(bits(a["scores"]), bits(b["scores"]))
    eng = nb.Engine(0, max_rows_per_block=16, keep=ka, n_row_samples=wide)
    src = rng.integers(0, 256, size=(5, 2 * wide + 14), dtype=np.uint8)
    d_src = torch.from_numpy(src).cuda()
    for keep, n_row in ((ka, wide), (kb, narrow), (ka, wide)):
        eng.set_keep(keep)
        d_dst = torch.full((5, 2 * m + 12), 0xAB, dtype=torch.uint8, device="cuda")
        eng.gather_rows_device(d_src, src.shape[1], 5, d_dst, d_dst.shape[1])
        torch.cuda.synchronize()
        assert np.array_equal(d_dst.cpu().numpy()[:, :2 * m], compact(src, n_row, keep))
    for bad in (ka[:-1], ka[::-1], np.append(ka[:-1], wide), np.append(ka[1:], ka[-1])):
        with pytest.raises(nb.NpcError, match="rc=-1"):
            eng.set_keep(bad)
    eng.close()
    plain = nb.Engine(10, max_rows_per_block=8)
    with pytest.raises(nb.NpcError, match="rc=-4"):
        plain.set_keep(np.arange(10))
    plain.close()
