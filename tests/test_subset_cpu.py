"""CPU tests of --samples (DESIGN.md 4.11): resolution of keep and ^exclude lists against the sample names of VCF text,
BCF, a PLINK fileset and BGEN files (embedded identifiers and .sample ID_2), the list format, and every refusal.  The
list is resolved right after the genotype file is opened, before any GPU context, so none of this needs a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from util_bcf import write_vcf
from util_bgen import make_split_dataset as bgen_split, records_to_variants, write_bgen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "nimpress_b200", "bin", "nimpress")


@pytest.fixture(scope="module")
def api():
    import __graft_entry__ as g
    g.build()
    from nimpress_b200 import api
    api.load_host_library()
    return api


def plan(api, score, geno, samples=None, exclude=False):
    """nph_plan and nph_plan_indexed with a sample list: (rc, kinds, eaidx, n_samples_out, error text)."""
    L = api.load_host_library()
    p = api._Params(0, 0, 3, 0, 0, 0, 0, 0, 100, 0.05, 0.001)
    p.samples_path = os.fsencode(samples) if samples else None
    p.exclude_samples = int(exclude)
    out = []
    for fn in ("nph_plan", "nph_plan_indexed"):
        kind = np.zeros(1 << 14, np.int32); ea = np.zeros(1 << 14, np.int32)
        n_rows, n_s = C.c_int64(), C.c_int64()
        args = [os.fsencode(score), os.fsencode(geno), None, C.byref(p), kind.ctypes.data, ea.ctypes.data, len(kind), C.byref(n_rows), C.byref(n_s)]
        if fn == "nph_plan_indexed":
            args += [None, None]
        rc = getattr(L, fn)(*args)
        out.append((rc, kind[:n_rows.value].copy(), ea[:n_rows.value].copy(), n_s.value, L.nph_last_error().decode() if rc else ""))
    assert out[0][0] == out[1][0] and out[0][3] == out[1][3]
    return out[0]


def write_list(path, names, nl="\n"):
    with open(path, "w", newline="") as fh:
        fh.write(nl.join(names) + nl)
    return str(path)


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    """One cohort of 57 samples (some names with spaces) as VCF text, BCF, a PLINK fileset and BGEN with embedded
    identifiers and with a .sample file."""
    tmp = str(tmp_path_factory.mktemp("subset_cpu"))
    rng = np.random.default_rng(5)
    d = bgen_split(tmp, rng, n=57, V=40)
    names = [f"S {i}" if i % 7 == 3 else f"S{i}" for i in range(57)]      # VCF / BCF / BGEN names may hold spaces
    d["names"] = names
    write_vcf(d["vcf"][:-7] + "_sp.vcf.gz", names, d["records"], contigs=["1", "2", "X"], compress="bgzf")
    d["vcf_sp"] = d["vcf"][:-7] + "_sp.vcf.gz"
    d["bgen_ids"] = write_bgen(os.path.join(tmp, "ids.bgen"), names, records_to_variants(d["records"], 57))
    d["bgen_sample"] = write_bgen(os.path.join(tmp, "sfile.bgen"), d["samples"], records_to_variants(d["records"], 57), embed_ids=False)
    return d


def test_keep_and_exclude_on_every_reader(api, files, tmp_path):
    """A keep list of 20 names gives n_samples_out 20 and the kinds / eaidx of the whole file; the exclude list of the
    same names gives 37; on VCF text, BCF, the PLINK fileset (.fam IID) and BGEN (embedded ids, .sample ID_2)."""
    rng = np.random.default_rng(1)
    pick = sorted(rng.choice(57, 20, replace=False))
    for geno, names in ((files["vcf_sp"], files["names"]), (files["bcf"], files["samples"]), (files["plink"], files["samples"]),
                        (files["bgen_ids"], files["names"]), (files["bgen_sample"], files["samples"])):
        lst = write_list(tmp_path / "keep.txt", [names[i] for i in pick[::-1]])          # list order does not matter
        rc0, k0, e0, n0, _ = plan(api, files["score"], geno)
        assert rc0 == 0 and n0 == 57
        rc, k, e, n, err = plan(api, files["score"], geno, lst)
        assert rc == 0, err
        assert n == 20 and np.array_equal(k, k0) and np.array_equal(e, e0)
        rc, k, e, n, err = plan(api, files["score"], geno, lst, exclude=True)
        assert rc == 0 and n == 37 and np.array_equal(k, k0), err


def test_list_format_crlf_blank_lines_and_spaces(api, files, tmp_path):
    """CRLF line ends are stripped, blank lines skipped, a name is the whole line (spaces included); a name padded with a
    space is another name."""
    names = files["names"]
    lst = tmp_path / "crlf.txt"
    lst.write_bytes(b"\r\n".join([b"", names[3].encode(), b"", names[10].encode(), b"", names[0].encode()]) + b"\r\n\r\n")
    rc, _, _, n, err = plan(api, files["score"], files["vcf_sp"], str(lst))
    assert rc == 0 and n == 3, err
    assert " " in names[3]
    rc, _, _, _, err = plan(api, files["score"], files["vcf_sp"], write_list(tmp_path / "pad.txt", [names[3] + " "]))
    assert rc == -3 and "S 3 " in err
    no_nl = tmp_path / "nonl.txt"
    no_nl.write_text(names[1] + "\n" + names[2])                                          # no newline at the end
    assert plan(api, files["score"], files["vcf_sp"], str(no_nl))[3] == 2


def test_every_sample_listed_and_exclude_unknown(api, files, tmp_path):
    """A keep list naming every sample and an exclude list naming none of the file's samples (unknown names are
    ignored, as plink --remove does) both score all 57."""
    all_list = write_list(tmp_path / "all.txt", files["samples"])
    assert plan(api, files["score"], files["bcf"], all_list)[3] == 57
    other = write_list(tmp_path / "other.txt", ["nobody", "X1", "S999"])
    assert plan(api, files["score"], files["bcf"], other, exclude=True)[3] == 57
    part = write_list(tmp_path / "part.txt", ["nobody", files["samples"][4], "S999"])
    assert plan(api, files["score"], files["bcf"], part, exclude=True)[3] == 56


def test_refusals(api, files, tmp_path):
    """nph_plan: NPH_EINPUT and a message naming the sample for an unknown keep name, a twice-listed name, a name the file
    holds twice (keep or exclude); an empty subset and an unreadable list are NPH_EINPUT too."""
    s = files["samples"]
    cases = [(write_list(tmp_path / "unk.txt", [s[1], "ghost"]), False, "ghost"),
             (write_list(tmp_path / "dup.txt", [s[2], s[5], s[2]]), False, f"{s[2]} is listed twice"),
             (write_list(tmp_path / "allx.txt", s), True, "no sample"),
             (str(tmp_path / "missing.txt"), False, "missing.txt")]
    for path, exclude, needle in cases:
        rc, _, _, _, err = plan(api, files["score"], files["bcf"], path, exclude)
        assert rc == -3 and needle in err, (path, err)
    dup_names = list(s)
    dup_names[9] = s[4]
    vcf = str(tmp_path / "dupnames.vcf")
    write_vcf(vcf, dup_names, files["records"], contigs=["1", "2", "X"])
    for exclude in (False, True):
        rc, _, _, _, err = plan(api, files["score"], vcf, write_list(tmp_path / "d.txt", [s[4]]), exclude)
        assert rc == -3 and f"{s[4]} occurs more than once" in err
    assert plan(api, files["score"], vcf, write_list(tmp_path / "ok.txt", [s[5]]))[3] == 1    # unlisted duplicates are fine


def test_cli_refusals_and_usage(api, files, tmp_path):
    """nimpress exits 1 and names the sample for each refusal, before any GPU is touched; --help lists both forms."""
    s = files["samples"]
    cases = [([f"--samples={write_list(tmp_path / 'u.txt', ['ghost'])}"], "ghost"),
             (["--samples", write_list(tmp_path / "t.txt", [s[3], s[3]])], f"{s[3]} is listed twice"),
             ([f"--samples=^{write_list(tmp_path / 'a.txt', s)}"], "no sample"),
             ([f"--samples={tmp_path / 'none.txt'}"], "none.txt"),
             (["--samples="], "--samples")]
    for args, needle in cases:
        r = subprocess.run([EXE, *args, files["score"], files["bcf"]], capture_output=True, text=True,
                           env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
        assert r.returncode == 1 and needle in r.stderr, (args, r.returncode, r.stderr)
        assert r.stdout == ""
    out = subprocess.run([EXE, "--help"], capture_output=True, text=True).stdout
    assert "--samples=<file>" in out and "--samples=^<file>" in out


def test_python_run_refuses_without_gpu(api, files, tmp_path):
    """api.run(samples=...) raises NimpressInputError for a bad list whether or not a GPU is present."""
    with pytest.raises(api.NimpressInputError, match="ghost"):
        api.run(files["score"], files["bcf"], samples=write_list(tmp_path / "g.txt", ["ghost"]))
    with pytest.raises(api.NimpressInputError, match="no sample"):
        api.run_multi([files["score"]], files["bcf"], samples=write_list(tmp_path / "e.txt", files["samples"]), exclude_samples=True)


def test_create_subset_refuses_bad_keep_lists(api):
    """npc_create_subset returns NPC_EINVAL, before touching a device, for a keep list that is not ascending, repeats an
    index, reaches n_row_samples or below 0, is empty, or for rows too wide for int32 indices."""
    L = api.load_library()
    for n_row, keep in ((10, [3, 2]), (10, [2, 2, 5]), (10, [1, 10]), (10, [-1, 4]), (10, []), (1 << 31, [0, 1])):
        h = C.c_void_p()
        k = np.array(keep, np.int64)
        rc = L.npc_create_subset(C.byref(h), 0, n_row, k.ctypes.data if len(k) else None, len(k), 2, 1, 16, 2, 16)
        assert rc == -1 and not h.value, (n_row, keep)
        assert b"npc_create_subset" in L.npc_last_error(None)
