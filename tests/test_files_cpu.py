"""CPU tests of several genotype files read as their concatenation (DESIGN.md 4.12): nph_plan_files over the parts
equals nph_plan_indexed over the concatenated file for VCF text, BCF, both mixed, PLINK filesets and BGEN; file order,
per-file index use, and every refusal through the command line.  None of this needs a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from util_bgen import make_split_dataset as bgen_split
from util_files import make_dataset
from util_split import by_contig, chunks, write_split

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")
NO_GPU = dict(os.environ, CUDA_VISIBLE_DEVICES="")


@pytest.fixture(scope="module")
def api():
    import __graft_entry__ as g
    g.build()
    from nimpress_b200 import api
    api.load_host_library()
    return api


def params(api, samples=None, exclude=False):
    p = api._Params(0, 0, 3, 0, 0, 0, 0, 0, 100, 0.05, 0.001)
    p.samples_path = os.fsencode(samples) if samples else None
    p.exclude_samples = int(exclude)
    return p


def plan_files(api, score, genos, samples=None):
    """nph_plan_files: (rc, kinds, eaidx, n_samples, records_read, index_seeks, error text)."""
    L = api.load_host_library()
    p = params(api, samples)
    kind = np.zeros(1 << 14, np.int32); ea = np.zeros(1 << 14, np.int32)
    n_rows, n_s, nrec, seeks = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
    arr = (C.c_char_p * len(genos))(*[os.fsencode(g) for g in genos])
    rc = L.nph_plan_files(os.fsencode(score), arr, len(genos), None, C.byref(p), kind.ctypes.data, ea.ctypes.data, len(kind),
                          C.byref(n_rows), C.byref(n_s), C.byref(nrec), C.byref(seeks))
    return (rc, kind[:n_rows.value].copy(), ea[:n_rows.value].copy(), n_s.value, nrec.value, seeks.value,
            L.nph_last_error().decode() if rc else "")


def plan_indexed(api, score, geno, samples=None):
    L = api.load_host_library()
    p = params(api, samples)
    kind = np.zeros(1 << 14, np.int32); ea = np.zeros(1 << 14, np.int32)
    n_rows, n_s, nrec, seeks = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
    rc = L.nph_plan_indexed(os.fsencode(score), os.fsencode(geno), None, C.byref(p), kind.ctypes.data, ea.ctypes.data, len(kind),
                            C.byref(n_rows), C.byref(n_s), C.byref(nrec), C.byref(seeks))
    assert rc == 0, L.nph_last_error()
    return kind[:n_rows.value].copy(), ea[:n_rows.value].copy(), n_s.value, nrec.value, seeks.value


def assert_same_plan(api, score, parts, cat):
    rc, k, e, n, nrec, _, err = plan_files(api, score, parts)
    assert rc == 0, err
    k2, e2, n2, nrec2, _ = plan_indexed(api, score, cat)
    assert np.array_equal(k, k2) and np.array_equal(e, e2) and n == n2 and nrec == nrec2
    return k, e


@pytest.fixture(scope="module")
def cohort(tmp_path_factory):
    d = make_dataset(str(tmp_path_factory.mktemp("files_cpu")), np.random.default_rng(21), n=23, V=150)
    s = bgen_split(str(tmp_path_factory.mktemp("files_cpu_split")), np.random.default_rng(22), n=23, V=150)
    assert s["samples"] == d["samples"]
    return dict(score=d["score"], samples=d["samples"], records=d["records"], split_score=s["score"],
                split_records=s["records"])


@pytest.mark.parametrize("kind", ["vcf", "bcf", "mixed", "bed", "bgen8"])
def test_plan_over_parts_equals_concatenation(api, cohort, kind, tmp_path):
    """Split per contig and in four chunks whose boundaries repeat a site: the kinds, eaidx, sample count and records
    read over the parts equal nph_plan_indexed over their concatenation (the earlier copy of a repeated site wins)."""
    split = kind in ("bed", "bgen8")
    score = cohort["split_score"] if split else cohort["score"]
    recs = cohort["split_records"] if split else cohort["records"]
    for name, parts in (("contig", by_contig(recs)), ("chunk", chunks(recs, 4))):
        kinds = ["vcf", "bcf"] * 2 if kind == "mixed" else None
        paths, cat = write_split("vcf" if kind == "mixed" else kind, str(tmp_path), f"{name}_", cohort["samples"], parts,
                                 kinds=kinds[:len(parts)] if kinds else None)
        assert_same_plan(api, score, paths, cat)


def test_file_order_does_not_matter(api, cohort, tmp_path):
    """With no site in two files, every order of the per-contig files gives the same plan."""
    parts = by_contig(cohort["records"])
    paths, _ = write_split("bcf", str(tmp_path), "c", cohort["samples"], parts)
    want = plan_files(api, cohort["score"], paths)
    assert want[0] == 0
    for perm in ([2, 0, 1], [1, 2, 0], [2, 1, 0]):
        got = plan_files(api, cohort["score"], [paths[i] for i in perm])
        assert got[0] == 0 and np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2]) and got[4] == want[4]


def test_index_decided_per_file(api, tmp_path, monkeypatch):
    """One BCF with a .csi and one without: the first takes the index-driven pass (index_seeks > 0, fewer records
    read), the second is streamed; the plan equals that of the concatenation streamed."""
    import util_bcf
    from util_bcf import write_bcf
    monkeypatch.setattr(util_bcf, "INDEX_BLOCK", 3000)
    rng = np.random.default_rng(3)
    d = make_dataset(str(tmp_path), rng, n=12, V=1500, index=True, spread=400)
    ents = open(d["score"]).read().split("\n")
    sparse = tmp_path / "sparse.score"
    sparse.write_text("\n".join(ents[:5] + [e for e in ents[5:] if e and rng.random() < 0.05]) + "\n")
    parts = by_contig(d["records"])
    a, b = str(tmp_path / "a.bcf"), str(tmp_path / "b.bcf")
    write_bcf(a, d["samples"], parts[0], contigs=["1", "2", "X"], filters=("FAIL", "LowQ"), index=True)
    write_bcf(b, d["samples"], [r for p in parts[1:] for r in p], contigs=["1", "2", "X"], filters=("FAIL", "LowQ"))
    assert os.path.exists(a + ".csi") and not os.path.exists(b + ".csi")
    monkeypatch.setenv("NIMPRESS_FORCE_INDEX", "1")
    rc, k, e, _, nrec, seeks, err = plan_files(api, str(sparse), [a, b])
    assert rc == 0, err
    assert seeks > 0 and nrec < len(d["records"])
    rc, k3, _, _, nrec3, seeks3, _ = plan_files(api, str(sparse), [b, a])         # the indexed file second
    assert rc == 0 and np.array_equal(k3, k) and seeks3 == seeks and nrec3 == nrec
    monkeypatch.setenv("NIMPRESS_NO_INDEX", "1")
    k2, e2, _, nrec2, seeks2 = plan_indexed(api, str(sparse), d["bcf"])
    assert seeks2 == 0 and nrec2 == len(d["records"])
    assert np.array_equal(k, k2) and np.array_equal(e, e2)


def cli(args):
    return subprocess.run([EXE, *args], capture_output=True, text=True, env=NO_GPU)


def test_refusals_through_the_cli(api, cohort, tmp_path):
    """Exit 1 naming both files for mixed kinds, naming the file and the first differing sample for other names or
    another order (suggesting --samples), for a keep name one file lacks and for kept sequences that differ; exit 255
    naming an unopenable second file.  All before any GPU is touched."""
    tmp, samples, recs, score = str(tmp_path), cohort["samples"], cohort["split_records"], cohort["split_score"]
    parts = by_contig(recs)
    bcfs, _ = write_split("bcf", tmp, "b", samples, parts)
    beds, _ = write_split("bed", tmp, "p", samples, parts)
    bgens, _ = write_split("bgen8", tmp, "g", samples, parts)
    for a, b in ((bcfs[0], beds[1]), (beds[0], bgens[1]), (bgens[0], bcfs[1])):
        r = cli([score, a, b])
        assert r.returncode == 1 and a in r.stderr and b in r.stderr and "different kinds" in r.stderr, r.stderr
        assert plan_files(api, score, [a, b])[0] == -3
    renamed = samples[:5] + ["Z9"] + samples[6:]
    reordered = samples[1:2] + samples[:1] + samples[2:]
    for other, first in ((renamed, "Z9"), (reordered, samples[1]), (samples[:-2], "none")):
        odd, _ = write_split("bcf", tmp, "odd", other, [parts[1]])
        r = cli([score, bcfs[0], odd[0]])
        assert r.returncode == 1 and odd[0] in r.stderr and first in r.stderr and "--samples" in r.stderr, r.stderr
    # chrX-like: the last file lacks two samples
    short = [s for i, s in enumerate(samples) if i not in (3, 8)]
    x, _ = write_split("bcf", tmp, "x", short, [[dict(r, gt=np.delete(r["gt"], [3, 8], axis=0)) for r in parts[2]]],
                       part_samples=[short])
    keep_all = tmp_path / "all.txt"
    keep_all.write_text("\n".join(samples) + "\n")
    r = cli([f"--samples={keep_all}", score, bcfs[0], bcfs[1], x[0]])
    assert r.returncode == 1 and x[0] in r.stderr and samples[3] in r.stderr, r.stderr
    rc, _, _, n, _, _, err = plan_files(api, score, [bcfs[0], bcfs[1], x[0]], samples=str(keep_all))
    assert rc == -3 and x[0] in err
    keep_short = tmp_path / "short.txt"
    keep_short.write_text("\n".join(short) + "\n")
    rc, _, _, n, _, _, err = plan_files(api, score, [bcfs[0], bcfs[1], x[0]], samples=str(keep_short))
    assert rc == 0 and n == len(short), err
    # kept sequences that differ: an exclude list that drops sample 3 from every file, but file x lacks sample 8 too
    drop = tmp_path / "drop.txt"
    drop.write_text(samples[3] + "\n")
    r = cli([f"--samples=^{drop}", score, bcfs[0], x[0]])
    assert r.returncode == 1 and x[0] in r.stderr and "--samples" in r.stderr, r.stderr
    # an unopenable second file: FATAL naming it, exit 255
    r = cli([score, bcfs[0], str(tmp_path / "missing.bcf"), bcfs[1]])
    assert r.returncode == 255 and r.stdout == f"FATAL Could not open input VCF file {tmp_path / 'missing.bcf'}\n", r.stdout
    # one file: the usual FATAL; the short usage line names the new form
    r = cli([score])
    assert r.returncode == 1 and "<genotypes> [<genotypes> ...]" in r.stderr
    assert "<genotypes> [<genotypes> ...]" in cli(["--help"]).stdout


def test_python_run_takes_a_list(api, cohort, tmp_path):
    """api.run / run_multi take a list of genotype paths; a refusal surfaces as NimpressInputError without a GPU."""
    parts = by_contig(cohort["split_records"])
    bcfs, _ = write_split("bcf", str(tmp_path), "b", cohort["samples"], parts)
    beds, _ = write_split("bed", str(tmp_path), "p", cohort["samples"], parts)
    with pytest.raises(api.NimpressInputError, match="different kinds"):
        api.run(cohort["split_score"], [bcfs[0], beds[1]])
    with pytest.raises(api.NimpressInputError, match="different kinds"):
        api.run_multi([cohort["split_score"]], (beds[0], bcfs[1]))
    with pytest.raises(FileNotFoundError, match="nope.bcf"):
        api.run(cohort["split_score"], [bcfs[0], str(tmp_path / "nope.bcf")])


def test_set_keep_refuses_without_a_context(api):
    """npc_set_keep returns NPC_EINVAL for a NULL context, before touching a device.  Every other refusal needs a
    context, which needs a device: NPC_ESTATE for a plain context and NPC_EINVAL for bad lists are checked in
    test_files_gpu.py."""
    L = api.load_library()
    k = np.arange(4, dtype=np.int64)
    assert L.npc_set_keep(None, k.ctypes.data, 4) == -1
