"""CPU tests of the PLINK 1 fileset reader (DESIGN.md 4.7): rows as stored, sample names, matching against the
equivalent all-PASS VCF, and the refusals with their exit codes.  No GPU needed: nothing here computes a score."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from util_plink import BED_MAGIC, bed_codes, make_split_dataset, pack_codes, write_plink

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")


@pytest.fixture(scope="module")
def api():
    import __graft_entry__ as g
    g.build()
    from nimpress_b200 import api
    api.load_host_library()
    return api


def read_gt(api, path, row_bytes, max_records=4096):
    L = api.load_host_library()
    out = np.zeros((max_records, row_bytes), np.uint8)
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


def test_codes_and_packing():
    """The writer's own conventions: 00 hom A1 (= ALT), 01 missing (a half call too), 10 het, 11 hom A2 (= REF),
    four samples per byte, low bits first."""
    raw = np.array([4, 4, 2, 4, 2, 2, 0, 0, 0, 4, 3, 5], np.int8)          # 1/1, 0/1, 0/0, ./., ./1, 0|1
    assert list(bed_codes(raw, 6)) == [0, 2, 3, 1, 1, 2]
    assert pack_codes(np.array([[0, 2, 3, 1, 1, 2]]), pad_code=3).tolist() == [[0b01111000, 0b11111001]]


@pytest.mark.parametrize("n", [1, 3, 4, 5, 6, 7, 301])
def test_read_gt_returns_packed_rows(api, tmp_path, n):
    """nph_read_gt on a fileset: the .bed rows as stored (width 0 = NPC_GT_BED, ploidy 2), sample names = IIDs."""
    rng = np.random.default_rng(n)
    d = make_split_dataset(str(tmp_path), rng, n=n, V=30, with_traps=n > 4)
    rb = (n + 3) // 4
    rc, rows, ns, w, pl = read_gt(api, d["plink"], 64 + rb)
    assert rc == 0 and ns == n and (w, pl) == (0, 2)
    raw = np.fromfile(d["plink"], np.uint8)
    assert raw[:3].tobytes() == BED_MAGIC
    want = raw[3:].reshape(-1, rb)
    assert rows.shape[0] == want.shape[0] == len(d["records"])
    assert np.array_equal(rows[:, :rb], want) and not rows[:, rb:].any()
    # sample names: the .fam's second column, even when FID differs
    fam = d["plink"][:-4] + ".fam"
    with open(fam, "w") as fh:
        fh.write("".join(f"FAM{i} {s}  0 0 1 -9\n" for i, s in enumerate(d["samples"])))
    assert plan(api, d["score"], d["plink"])[2] == n


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_matching_equals_equivalent_vcf(api, tmp_path, seed):
    """nph_plan on the fileset gives the kind and eaidx of the equivalent all-PASS VCF: an ALT2 effect allele matches
    its own split line at eaidx 1; REF effect alleles at eaidx 0; a line without ALT (A1 = 0) matches REF only."""
    rng = np.random.default_rng(seed)
    d = make_split_dataset(str(tmp_path), rng, n=37, V=150)
    for bed in (None, d["bed"]):
        k_p, e_p, _ = plan(api, d["score"], d["plink"], bed)
        k_v, e_v, _ = plan(api, d["score"], d["vcf"], bed)
        assert np.array_equal(k_p, k_v) and np.array_equal(e_p, e_v)
        assert set(np.unique(e_p[k_p == 0])) <= {0, 1}
    assert (k_p == 0).sum() > 20


def _fileset(tmp, n=9, V=5):
    rng = np.random.default_rng(0)
    recs = [dict(contig="1", pos=100 + 10 * k, ref="A", alts=["G"], filter="PASS",
                 gt=(((rng.random((n, 2)) < 0.3).astype(np.int64) + 1) << 1).astype(np.int8)) for k in range(V)]
    prefix = os.path.join(tmp, "f")
    write_plink(prefix, [f"s{i}" for i in range(n)], recs)
    score = os.path.join(tmp, "f.score")
    with open(score, "w") as fh:
        fh.write("S\nd\nc\nhs37d5\n0.0\n1\t100\tA\tG\t0.1\t0.2\n")
    return prefix, score


def _run(*args):
    return subprocess.run([EXE, *args], capture_output=True, text=True)


def test_refusals(api, tmp_path):
    """Malformed filesets: InputError (exit 1) for an individual-major mode byte, a .bed shorter or longer than the
    .bim and .fam say, a .bim line with fewer than 6 columns or a bad POS; a missing .fam or .bim is "could not open
    input VCF" (exit 255); --dosage with a fileset exits 1.  The well-formed fileset parses."""
    prefix, score = _fileset(str(tmp_path))
    bed = prefix + ".bed"
    plan(api, score, bed)
    good = open(bed, "rb").read()

    def refused(expect_rc, expect_msg, *extra):
        r = _run(*extra, score, bed)
        assert r.returncode == expect_rc, (r.returncode, r.stdout, r.stderr)
        assert expect_msg in (r.stdout + r.stderr), (r.stdout, r.stderr)

    open(bed, "wb").write(good[:2] + b"\x00" + good[3:])
    refused(1, "individual-major")
    open(bed, "wb").write(good[:-1])
    refused(1, "need")
    open(bed, "wb").write(good + b"\x00")
    refused(1, "need")
    open(bed, "wb").write(good)
    bim = open(prefix + ".bim").read()
    lines = bim.splitlines()
    open(prefix + ".bim", "w").write("\n".join(lines[:2] + ["1\tv9\t0\t130\tG"] + lines[3:]) + "\n")
    refused(1, "fewer than 6 columns")
    open(prefix + ".bim", "w").write("\n".join(lines[:2] + ["1\tv9\t0\t1x0\tG\tA"] + lines[3:]) + "\n")
    refused(1, "POS")
    open(prefix + ".bim", "w").write(bim)
    refused(1, "--dosage", "--dosage")
    shutil.move(prefix + ".fam", prefix + ".fam.x")
    refused(255, "FATAL Could not open input VCF file")
    shutil.move(prefix + ".fam.x", prefix + ".fam")
    shutil.move(prefix + ".bim", prefix + ".bim.x")
    refused(255, "FATAL Could not open input VCF file")
    shutil.move(prefix + ".bim.x", prefix + ".bim")
    # the refusals reach the C ABI as NPH_EINPUT / NPH_EOPEN_VCF too
    with pytest.raises(api.NimpressInputError, match="individual-major"):
        open(bed, "wb").write(good[:2] + b"\x00" + good[3:])
        api.run(score, bed)
    open(bed, "wb").write(good)
    os.remove(prefix + ".fam")
    with pytest.raises(FileNotFoundError):
        api.run(score, bed)


def test_usage_names_the_fileset(api):
    r = _run("--help")
    assert r.returncode == 0 and "<genotypes.vcf|.bcf|.bed>" in r.stdout
