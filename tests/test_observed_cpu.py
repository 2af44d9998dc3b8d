"""CPU checks of --observed (DESIGN.md 4.13): the option parses and is documented, the symbol tables carry the new
calls, and on tests/golden/set1 the counts the CPU oracle's own loop gives (every score row on its own under --imp-sample
fail: a NaN score is a sample without a call) equal the values derived by hand from SURVEY Appendix B's raw dosages, as
does the numpy restatement of the tally's predicate over the oracle's records."""
import os
import subprocess
import sys

import numpy as np
import pytest

from util_observed import called_gt, ngt_total, observed, oracle_observed_files, oracle_observed_matrix
from util_vcf import build_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S1 = os.path.join(ROOT, "tests", "golden", "set1")

# S1..S6 under each option set: (maxmis, ignorefilt, cov)
SET1 = [
    (1.0, False, False, [3, 4, 2, 2, 2, 3]),
    (0.2, False, False, [3, 3, 2, 2, 2, 3]),          # 2:400 becomes MAXMIS
    (1.0, True, False, [4, 5, 3, 2, 2, 3]),
    (1.0, False, True, [1, 1, 1, 0, 1, 1]),           # only 3:500 is OK
]


@pytest.fixture(scope="module")
def api():
    import __graft_entry__ as g
    g.build()
    from nimpress_b200 import api
    api.load_host_library()
    return api


def cli(*args):
    code = "import sys; from nimpress_b200 import api; sys.exit(api.main(sys.argv[1:]))"
    return subprocess.run([sys.executable, "-c", code, *args], capture_output=True, text=True, cwd=ROOT, timeout=300)


def test_usage_and_parse(api):
    r = cli("--help")
    assert r.returncode == 0
    i = r.stdout.index("--observed")
    assert "(not a reference option)" in r.stdout[i:i + 400] and "not alleles" in r.stdout[i:i + 400]
    # parsed: the run gets as far as opening the genotype file (an unknown option would exit 1 first)
    r = cli("--observed", os.path.join(S1, "set1.score"), "/nonexistent.vcf")
    assert r.returncode == 255 and r.stdout.startswith("FATAL Could not open input VCF file"), (r.stdout, r.stderr)
    assert cli("--observd", os.path.join(S1, "set1.score"), "/nonexistent.vcf").returncode == 1


def test_symbol_tables(api):
    import nimpress_b200 as nb
    L = nb.load_library()
    for s in ("npc_set_observed", "npc_observed", "npc_score_resident_multi_observed"):
        assert s in L._npc_symbols and hasattr(L, s)
    assert "nph_result_observed" in api.load_host_library()._nph_symbols
    assert [f[0] for f in api._Params._fields_][-1] == "observed"


@pytest.mark.parametrize("maxmis,ignorefilt,cov,want", SET1, ids=["maxmis1", "maxmis0.2", "ignorefilt", "cov"])
def test_set1_oracle_counts(maxmis, ignorefilt, cov, want, tmp_path):
    import orc
    bed = os.path.join(S1, "set1.bed") if cov else None
    files = oracle_observed_files(os.path.join(S1, "set1.score"), os.path.join(S1, "set1.vcf.gz"), tmp_path, bed, maxmis=maxmis,
                                  ignorefilt=ignorefilt)
    assert files.tolist() == want
    samples, _, gt, rows = build_block(os.path.join(S1, "set1.score"), os.path.join(S1, "set1.vcf.gz"), bed, ignorefilt=ignorefilt)
    n = len(samples)
    assert oracle_observed_matrix(gt, n, 2, rows, maxmis=maxmis).tolist() == want
    ref = orc.score_matrix(gt, n, 2, rows.astype(orc.ROW_DTYPE), maxmis=maxmis)
    got = observed(lambda r: called_gt(gt[r["gt_row"]], n, 2, np.int8), rows, ref["loci"], n)
    assert got.tolist() == want
    assert int(got.sum()) == ngt_total(ref["loci"])


@pytest.mark.parametrize("width,ploidy", [(1, 2), (1, 1), (1, 3), (2, 2), (4, 2), (2, 4)])
def test_gt_predicate_equals_oracle_loop(width, ploidy):
    """The GT predicate the GPU tests use (called_gt) against the oracle's own loop on cohorts with half calls, short
    calls, missing / vector_end sentinels and invalid negative values."""
    import orc
    from util_cohort import random_cohort, random_rows
    rng = np.random.default_rng(100 + 10 * width + ploidy)
    n, V = 301, 30
    gt = random_cohort(rng, n, V, width=width, ploidy=ploidy, miss_rate=0.05, n_alt=2, halfcall_rate=0.03, sentinel_rate=0.05,
                       invalid_rate=0.01)
    rows = random_rows(rng, V, n_rows=V + 10, n_alt=2)
    ref = orc.score_matrix(gt, n, ploidy, rows.astype(orc.ROW_DTYPE), maxmis=0.5, mincs=5)
    want = oracle_observed_matrix(gt, n, ploidy, rows, maxmis=0.5, mincs=5)
    got = observed(lambda r: called_gt(gt[r["gt_row"]], n, ploidy, gt.dtype), rows, ref["loci"], n)
    assert np.array_equal(got, want) and int(want.sum()) == ngt_total(ref["loci"])
