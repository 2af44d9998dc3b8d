"""The multi-score tensor-core contraction (npc_multi.cuh, DESIGN section 4.5) against the EXACT sum of the
addends the reference adds, under a bound proven from its documented arithmetic.

Reference.  For one definition, the reference adds per sample, row by row, fl(d*beta) for a called sample of
an OK row and fl(imputed*beta) for a missing sample or a constant row (src/nimpress.nim:639-641).  The addend
matrix A[row, sample] is built from the genotypes and the oracle's per-locus records (util_order.addends), is
self-checked against the oracle (A summed serially in row order == orc.score_matrix, bit for bit), and the
expectation per sample is math.fsum of its column: the correctly rounded exact sum.

Bound.  The contraction scales each definition's coefficients c (beta and cm = fl(imputed*beta) of its OK
rows) by 2^F, F = 52 - ex where max|c| = m * 2^ex, 0.5 <= m < 1, and rounds them to integers; everything
after that is integer-exact until one conversion to fp64.  A coefficient is off by at most half a quantum,
2^(ex-53) <= 2^-52 * max|c|, with equality when max|c| is a power of two and c sits on a half quantum.  A row
contributes its coefficient times its plane value w (the dosage 0, 1, 2 of a called sample, 1 for a missing
one), so per sample
    |got - exact| <= 2^-52 * max|c| * W   (W = sum of w over the OK rows)   + fp64 roundings,
where the roundings are the constant rows' chain, the int64 -> fp64 conversion, the k-split adds and the
normalisation, each at most 2^-53 of a value no larger than the sum of |addends|.  Scores are taken as raw sums
(offsets = None) so that no offset hides an absolute error.

Inputs that fall back to the fused kernel (npc_multi_contractions says which path ran) are checked against the
same exact sum under the bound of any fp64 summation of the addends, (R + 2) * 2^-53 * sum|addends|."""
import math
from fractions import Fraction

import numpy as np
import pytest

import orc
import util_order
from util_cohort import assert_loci_equal, bits

U = 2.0 ** -53
DBL_MAX = np.finfo(np.float64).max
MAX_PARTS = 4                 # the library splits a tile's k-blocks into at most 4 parts unless NPC_MULTI_PARTS says more


# ---- CPU helpers: the exact reference and the bound ---------------------------------------------------------

def fixed_point_exponent(maxc):
    """F of a definition (npc_api.cu, multi_contract): 52 - ex with max|c| = m * 2^ex, 0.5 <= m < 1."""
    return 52 - math.frexp(maxc)[1] if maxc > 0 else 0


def quantise(c, F):
    """round(c * 2^F), ties to even (__double2ll_rn of scalbn): Python's round of a float is exact."""
    return round(math.ldexp(c, F))


def terms(gt, n, rows, loci):
    """What the bound needs of one definition, from the oracle's records:
      A     [R, n] addends in row order (0.0 for an unused row);
      W     [n] plane values summed over the OK (decoded) rows with a beta that is not NaN: the dosage, 1 for a
            missing sample;
      maxc  max |beta|, |cm| over the OK rows, NaN coefficients excluded (k_multi_scale);
      n_const, c_abs: number of constant rows and the sum of their |addends|."""
    A = np.zeros((len(rows), n))
    W = np.zeros(n)
    maxc, n_const, c_abs = 0.0, 0, 0.0
    with np.errstate(invalid="ignore", over="ignore"):
        for i, (a, row, rec) in enumerate(zip(util_order.addends(gt, n, rows, loci), rows, loci)):
            A[i] = a
            if not rec["used"]:
                continue
            if rec["klass"] != orc.CLASS_OK:
                n_const += 1
                c_abs += abs(float(a))
                continue
            beta = float(row["beta"])
            if beta != beta:                             # a NaN beta makes every sample NaN: no coefficient
                continue
            codes = util_order.dosage_codes(gt[int(row["gt_row"])], n, gt.dtype.itemsize, int(row["eaidx"]))
            W += np.where(codes == 3, 1, codes)
            cm = float(np.float64(rec["imputed"]) * np.float64(beta))
            maxc = max(maxc, abs(beta), abs(cm) if cm == cm else 0.0)
    return dict(A=A, W=W, maxc=maxc, n_const=n_const, c_abs=c_abs)


def serial_sums(A):
    """The reference's chain over the addends: +0.0, then every row in order."""
    s = np.zeros(A.shape[1])
    with np.errstate(invalid="ignore"):
        for a in A:
            s = s + a
    return s


def exact_sums(A, cols):
    """Correctly rounded exact column sums at the sample indices `cols` (NaN elsewhere)."""
    out = np.full(A.shape[1], np.nan)
    At = A.T
    for s in np.nonzero(cols)[0]:
        col = At[s].tolist()
        try:
            out[s] = math.fsum(col)
        except OverflowError:                          # an intermediate beyond DBL_MAX: exact rationals
            try:
                out[s] = float(sum(map(Fraction, col)))
            except OverflowError:
                out[s] = math.copysign(math.inf, sum(map(Fraction, col)))
    return out


def contraction_bound(t, parts=MAX_PARTS):
    """Per-sample bound on |contraction - exact sum| (module docstring).  The int64 -> fp64 conversion of the low
    digit sum |lo| <= 2^32 * W quanta adds at most 2^-53 * 2^32 * W * 2^-F <= 2^-72 * max|c| * W."""
    q = 2.0 ** -52 * t["maxc"] * t["W"]
    s_abs = np.abs(t["A"]).sum(axis=0)
    return q + 2.0 ** -72 * t["maxc"] * t["W"] + U * (t["n_const"] * t["c_abs"] + (parts + 3) * (s_abs + q))


def summation_bound(t):
    """Any fp64 summation of the R addends: (R + 2) * 2^-53 * sum|addends| (the fused kernel's tile order)."""
    return (len(t["A"]) + 2) * U * np.abs(t["A"]).sum(axis=0)


def check_definition(got, gt, n, rows, pol, contracted, parts=MAX_PARTS):
    """One definition's raw sums against the oracle (records, nloci, NaN / inf pattern) and the exact sum (finite
    samples, within the bound of the path that ran).  Returns the worst |error| / bound."""
    sc, nloci, loci = got
    want = orc.score_matrix(gt, n, 2, rows, offset=0.0, **pol)
    assert nloci == want["nloci"] > 0
    assert_loci_equal(loci, want["loci"])
    t = terms(gt, n, rows, want["loci"])
    ser = util_order.finalize(serial_sums(t["A"]), nloci, 0.0)   # self-check of the addends against the oracle's chain
    b = want["scores"]
    assert np.array_equal(np.isnan(ser), np.isnan(b)) and np.array_equal(bits(ser[~np.isnan(b)]), bits(b[~np.isnan(b)]))
    assert np.array_equal(np.isnan(sc), np.isnan(b)), (np.isnan(sc).sum(), np.isnan(b).sum())
    inf = np.isinf(b)
    assert np.array_equal(np.isinf(sc), inf) and np.array_equal(sc[inf], b[inf])
    ok = np.isfinite(b)
    if not ok.any():
        return 0.0
    exact = exact_sums(t["A"], ok)
    bound = contraction_bound(t, parts) if contracted else summation_bound(t)
    err = np.abs(sc[ok] - exact[ok])
    bad = np.nonzero(err > bound[ok])[0]
    assert bad.size == 0, f"{bad.size} samples over the bound, worst {float((err / bound[ok])[bad].max()):.3g}x"
    return float((err / np.maximum(bound[ok], 1e-300)).max())


# ---- inputs -------------------------------------------------------------------------------------------------

def dosage_cohort(rng, n, V, miss=0.01, miss_rows=1.0):
    """int8 GT rows (REF = allele 0, ALT = allele 1) with random dosages of ALT; `miss` of the samples of a fraction
    `miss_rows` of the rows are './.'.  Row bytes padded to 16; padding holds allele codes no sample reads."""
    af = rng.uniform(0.05, 0.95, size=(V, 1))
    a = (rng.random((V, n, 2)) < af[:, :, None]).astype(np.int64)
    raw = (a + 1) << 1
    m = (rng.random((V, n)) < miss) & (rng.random((V, 1)) < miss_rows)
    raw[m] = 0
    gt = np.zeros((V, -(-2 * n // 16) * 16), np.int8)
    gt[:, :2 * n] = raw.reshape(V, 2 * n)
    gt[:, 2 * n:] = 4
    return gt


def gt_rows(gt_row, beta, eaf=0.3):
    """GT rows with effect allele ALT (eaidx 1)."""
    r = np.zeros(len(gt_row), dtype=orc.ROW_DTYPE)
    r["gt_row"] = gt_row
    r["eaidx"] = 1
    r["beta"] = beta
    r["eaf"] = eaf
    return r


def const_rows(beta, eaf=0.3):
    """Not-covered rows: under --imp-locus=ps each adds fl(2*eaf*beta) to every sample."""
    r = gt_rows(np.full(len(beta), -1), beta, eaf)
    r["kind"] = 1                                        # NOTCOV
    r["eaidx"] = -1
    return r


def wide_betas(rng, k, lo=-60, hi=4):
    """Betas of both signs spanning the binades 2^lo .. 2^hi."""
    return rng.choice([-1.0, 1.0], k) * np.exp2(rng.uniform(lo, hi, k))


def score(nb, gt, n, lists, pol, block=256):
    eng = nb.Engine(n, max_rows_per_block=block, n_slots=2)
    eng.set_policy(**pol)
    V = gt.shape[0]
    assert eng.resident_reserve(V) >= V
    for r0 in range(0, V, block):
        slot, view = eng.stage_acquire()
        m = min(block, V - r0)
        view[:m, :gt.shape[1]] = gt[r0:r0 + m].view(np.uint8)
        eng.stage_upload(slot, m, r0)
    got = eng.score_resident_multi(lists, None)
    ran = eng.multi_contractions
    eng.close()
    return got, ran


@pytest.fixture(scope="module")
def nb():
    import __graft_entry__ as g
    g.build()
    import nimpress_b200 as nb
    return nb


# ---- CPU tests of the helpers ---------------------------------------------------------------------------------

@pytest.mark.parametrize("k", [-849, -60, -1, 0, 4, 951])
def test_quantisation_bound_is_attained_at_powers_of_two(k):
    """The model of F and round(c * 2^F): every |c| <= max|c| is off by at most 2^-52 * max|c|; with max|c| a power
    of two the largest quantised value is 2^51 and c = 2^-52 * max|c| (half a quantum, ties to even -> 0) is off by
    exactly the bound; one ulp below the power of two the quantum halves and so does the worst error."""
    rng = np.random.default_rng(k & 0xFFFF)
    for maxc, worst in ((math.ldexp(1.0, k), 1.0), (math.nextafter(math.ldexp(1.0, k), 0.0), 0.5)):
        F = fixed_point_exponent(maxc)
        assert 2 ** 51 <= quantise(maxc, F) <= 2 ** 52
        cs = [maxc * float(u) for u in rng.uniform(-1, 1, 2000)] + [maxc, -maxc, math.ldexp(maxc, -52), 5e-324, -0.0]
        ratio = max(abs(Fraction(quantise(c, F)) * Fraction(2) ** -F - Fraction(c)) / (Fraction(maxc) / 2 ** 52) for c in cs)
        assert ratio <= worst * (1 + 2.0 ** -50)
        if worst == 1.0:
            assert quantise(maxc, F) == 2 ** 51 and ratio == 1
    assert fixed_point_exponent(math.ldexp(1.0, -849)) == 900 and fixed_point_exponent(math.nextafter(math.ldexp(1.0, -849), 0)) == 901
    assert fixed_point_exponent(math.nextafter(math.ldexp(1.0, 952), 0)) == -900 and fixed_point_exponent(math.ldexp(1.0, 952)) == -901


def model_contraction(gt, n, rows, loci, t):
    """The contraction's value per sample in exact rationals: sum of w * round(c * 2^F) * 2^-F over the OK rows plus
    the exact constant sum (no fp64 rounding anywhere)."""
    F = fixed_point_exponent(t["maxc"])
    tot = [Fraction(0)] * n
    for row, rec, a in zip(rows, loci, t["A"]):
        if not rec["used"]:
            continue
        if rec["klass"] != orc.CLASS_OK:
            tot = [x + Fraction(float(a[0])) for x in tot]
            continue
        codes = util_order.dosage_codes(gt[int(row["gt_row"])], n, 1, int(row["eaidx"]))
        qb = quantise(float(row["beta"]), F)
        qm = quantise(float(np.float64(rec["imputed"]) * row["beta"]), F)
        tot = [x + Fraction(qm if c == 3 else int(c) * qb) / Fraction(2) ** F for x, c in zip(tot, codes)]
    return tot


def test_reference_and_bound_on_the_aligned_case():
    """The exact reference equals the oracle's chain bit for bit, fsum is the exact sum rounded once, and on the
    aligned case -- beta = 1 at dosage 0 plus 1000 betas of 0.49 * 2^-51 at dosage 2, which round to nothing -- the
    modelled contraction is 0.98 of the bound away from the exact sum: the bound is tight.  The error is also over
    a hundred times the oracle parity floor (8 eps sum|beta| / nloci), which an offset check never saw."""
    rng = np.random.default_rng(3)
    n, V = 40, 1002
    gt = dosage_cohort(rng, n, V, miss=0.0)
    gt[0, :2 * n] = 2                                   # the beta = 1 row: dosage 0 everywhere
    gt[1:1001, :2 * n] = 4                              # the small rows: dosage 2 everywhere
    gt[1001, :2 * n] = np.where(np.arange(2 * n) < n, 4, 0)    # one row missing for half the samples
    rows = np.concatenate([gt_rows([0], [1.0]), gt_rows(np.arange(1, 1001), np.full(1000, 0.49 * 2.0 ** -51)),
                           gt_rows([1001], [2.0 ** -52]), const_rows(np.array([2.0 ** -10, -3e-5]))])
    want = orc.score_matrix(gt, n, 2, rows, offset=0.0, maxmis=1.0)
    t = terms(gt, n, rows, want["loci"])
    ser = util_order.finalize(serial_sums(t["A"]), want["nloci"], 0.0)
    assert np.array_equal(bits(ser), bits(want["scores"]))
    ex = exact_sums(t["A"], np.ones(n, bool))
    for s in range(n):
        assert ex[s] == float(sum(map(Fraction, t["A"][:, s].tolist())))
    model = model_contraction(gt, n, rows, want["loci"], t)
    bound = contraction_bound(t, parts=1)
    q = 2.0 ** -52 * t["maxc"] * t["W"]
    ratio = [abs(m - Fraction(e)) / Fraction(q[s]) for s, (m, e) in enumerate(zip(model, ex))]
    assert all(abs(float(m) - e) <= bound[s] for s, (m, e) in enumerate(zip(model, ex)))
    assert max(ratio) <= 1 and min(ratio) > Fraction(97, 100)
    floor = orc.abs_floor(rows["beta"], want["nloci"]) * 2 * want["nloci"]     # the parity floor in raw-sum units
    assert float(min(abs(m - Fraction(e)) for m, e in zip(model, ex))) > 100 * floor


def test_bound_helpers_on_non_finite_and_constant_rows():
    """terms() takes max|c| over OK rows only (constant and unused rows are not coefficients), skips NaN betas and NaN
    cm, and counts a missing sample as plane value 1; exact_sums survives intermediates beyond DBL_MAX."""
    rng = np.random.default_rng(4)
    n = 8
    gt = dosage_cohort(rng, n, 3, miss=0.0)
    gt[0, :2 * n] = [0, 0] + [4, 4] * (n - 1)            # sample 0 missing, others dosage 2
    rows = np.concatenate([gt_rows([0], [0.5]), gt_rows([1], [np.nan]), const_rows(np.array([1e6])), gt_rows([2], [0.25], eaf=0.9)])
    want = orc.score_matrix(gt, n, 2, rows, offset=0.0, imp_sample="ps", maxmis=1.0)
    t = terms(gt, n, rows, want["loci"])
    assert t["maxc"] == 0.5 and t["n_const"] == 1 and t["c_abs"] == 0.6e6
    d2 = util_order.dosage_codes(gt[2], n, 1, 1)
    assert np.array_equal(t["W"], np.r_[1, np.full(n - 1, 2)] + d2)
    A = np.array([[DBL_MAX, 1.0], [DBL_MAX, 0.0], [-DBL_MAX, 0.0]])
    e = exact_sums(A, np.array([True, True]))
    assert e[0] == DBL_MAX and e[1] == 1.0


# ---- GPU: coefficient range ------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_coefficient_range(nb):
    """Seven definitions over one slab in one contraction, raw sums: the aligned case (beta 1 and betas of
    0.49 * 2^-51, which round to nothing), max|c| exactly a power of two with betas on half quanta (2^-52: off by
    exactly the bound; 2^-51: exact at this F, off by twice the bound at a quantum twice as coarse), max|c| one ulp
    below a power of two, betas spanning 2^-60 .. 2^4, subnormal betas and -0.0 next to 2^-849, cm > max|beta|
    (neff / ngt near 2 under int_ps), and 2-4 repeats of one entry with opposite signs."""
    rng = np.random.default_rng(11)
    n, V = 300, 1200
    gt = dosage_cohort(rng, n, V, miss=0.01)
    pol = dict(imp_sample="ps")                          # imputed = 2 * eaf: 0.6 (cm < beta) unless eaf says otherwise
    perm = rng.permutation(V)
    lists = [
        np.concatenate([gt_rows([perm[0]], [1.0]), gt_rows(perm[1:1001], np.full(1000, 0.49 * 2.0 ** -51))]),
        np.concatenate([gt_rows([perm[0]], [-1.0]), gt_rows(perm[1:301], np.full(300, 2.0 ** -52))]),
        np.concatenate([gt_rows([perm[0]], [1.0]), gt_rows(perm[301:601], np.full(300, 2.0 ** -51)),
                        gt_rows(perm[601:700], rng.normal(0, 0.1, 99)), const_rows(np.array([0.5, -0.25]))]),
        np.concatenate([gt_rows([perm[5]], [math.nextafter(1.0, 0.0)]), gt_rows(perm[10:500], rng.uniform(-1, 1, 490))]),
        np.concatenate([gt_rows(perm[:1100], wide_betas(rng, 1100)), const_rows(wide_betas(rng, 5))]),
        gt_rows(perm[200:400], np.r_[2.0 ** -849, -2.0 ** -849 * rng.uniform(0, 1, 99), rng.choice([5e-324, -5e-324, 2.2e-310, -0.0, 0.0], 100)]),
        gt_rows(perm[1100:1150], rng.normal(0, 0.05, 50), eaf=0.995),
        gt_rows(np.repeat(perm[700:760], [2, 3, 4, 1] * 15), np.r_[[1.5, -1.5, 0.7, -0.7, 0.7 / 3, 2.0 ** -40, -2.0 ** -40, 3.0, -1.0, 1e-9] * 15]),
    ]
    got, ran = score(nb, gt, n, lists, pol)
    assert ran == 1
    ratios = [check_definition(got[k], gt, n, rows, pol, True) for k, rows in enumerate(lists)]
    assert ratios[0] > 0.9 and ratios[1] > 0.9           # the bound is reached, not merely safe
    print("worst error / bound per definition:", " ".join(f"{r:.3f}" for r in ratios))


# ---- GPU: scale guards -----------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("maxc,contracts", [(2.0 ** -849, True), (math.nextafter(2.0 ** -849, 0.0), False),
                                             (math.nextafter(2.0 ** 952, 0.0), True), (2.0 ** 952, False)],
                         ids=["F900", "F901", "F-900", "F-901"])
def test_scale_guards(nb, maxc, contracts):
    """|F| <= 900 contracts, one step past falls back to the fused kernel; both sides against the exact sum.  cm
    stays below max|beta| (imputed = 2 * eaf = 0.6)."""
    rng = np.random.default_rng(12)
    n, V = 257, 400
    gt = dosage_cohort(rng, n, V, miss=0.02)
    pol = dict(imp_sample="ps")
    scaled = np.r_[maxc, -maxc, [maxc * float(u) for u in rng.uniform(-1, 1, 150)], rng.choice([5e-324, -0.0], 20)]
    lists = [gt_rows(rng.permutation(V)[:len(scaled)], scaled), gt_rows(np.arange(100), rng.normal(0, 0.2, 100)),
             gt_rows(np.arange(150, 400), wide_betas(rng, 250))]
    got, ran = score(nb, gt, n, lists, pol)
    assert ran == int(contracts)
    for k, rows in enumerate(lists):
        check_definition(got[k], gt, n, rows, pol, contracts)


# ---- GPU: non-finite coefficients -------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("beta", [math.inf, -math.inf, DBL_MAX, -DBL_MAX, 1.7975e308, -1.7975e308, 9e307, "cm-inf", math.nan],
                         ids=["inf", "-inf", "DBL_MAX", "-DBL_MAX", "1.7975e308", "-1.7975e308", "9e307", "cm-inf", "nan"])
def test_non_finite_betas(nb, beta):
    """A decoded row whose beta is +-inf or too large for fixed point (or whose cm = fl(imputed * beta) overflows:
    beta 1e10 at eaf 1e300 under --imp-sample=ps) sends the call to the fused kernel, which gives +-inf where the
    dosage is not 0 and NaN where it is, as the reference does.  A NaN beta makes its whole definition NaN, which the
    contraction gives itself."""
    rng = np.random.default_rng(13)
    n, V = 300, 200
    gt = dosage_cohort(rng, n, V, miss=0.01)
    pol = dict(imp_sample="ps")
    gt[7, :4] = [0, 0, 4, 4]                             # the large row: sample 0 missing, sample 1 dosage 2
    big = gt_rows([7], [1e10], eaf=1e300) if beta == "cm-inf" else gt_rows([7], [beta])
    lists = [np.concatenate([gt_rows(np.arange(20, 120), rng.normal(0, 0.1, 100)), big]),
             gt_rows(np.arange(50, 150), rng.normal(0, 0.1, 100)), gt_rows(np.arange(100, 200), wide_betas(rng, 100))]
    got, ran = score(nb, gt, n, lists, pol)
    assert ran == (1 if beta != beta else 0)
    for k, rows in enumerate(lists):
        check_definition(got[k], gt, n, rows, pol, bool(ran))
    if beta != beta:
        assert np.isnan(got[0][0]).all()
    else:
        assert np.isinf(got[0][0]).any()


# ---- GPU: shapes -------------------------------------------------------------------------------------------------

SHAPES = [  # n, entries, definitions, NaN-counter rows (imp_sample=fail), NPC_MULTI_PARTS
    (1, 63, 3, False, None), (255, 64, 16, True, None), (256, 65, 17, True, None), (257, 1300, 18, False, None),
    (257, 1300, 19, False, None), (256, 64, 18, True, None), (4099, 65, 3, False, None), (30011, 65, 3, True, None),
    (2100, 1300, 5, True, "1"), (2100, 1300, 5, False, "2"), (2100, 1300, 5, True, "3"), (2100, 1300, 5, False, "4"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,E,S,fail,parts", SHAPES, ids=[f"n{s[0]}-E{s[1]}-S{s[2]}{'-nan' if s[3] else ''}{'-p' + s[4] if s[4] else ''}"
                                                           for s in SHAPES])
def test_contraction_shapes(nb, monkeypatch, n, E, S, fail, parts):
    """Tile edges (1, 255, 256, 257, 4099, 30011 samples), k-block edges (63, 64, 65, 1300 entries), launch
    boundaries (18 definitions of 7 rows, 16 of 8 with the NaN counter rows, one more each) and the k-split
    (NPC_MULTI_PARTS 1-4), every definition with betas across 2^-40 .. 2^2 and a few constant rows."""
    if parts:
        monkeypatch.setenv("NPC_MULTI_PARTS", parts)
    rng = np.random.default_rng(1000 + n + E + S)
    gt = dosage_cohort(rng, n, E, miss=0.003, miss_rows=0.1 if fail else 1.0)
    pol = dict(imp_sample="fail", maxmis=1.0) if fail else dict()
    lists = [np.concatenate([gt_rows(np.arange(E), wide_betas(rng, E, -40, 2)), const_rows(wide_betas(rng, 3, -20, 0))])]
    for _ in range(S - 1):
        m = int(rng.integers(1, E + 1))
        lists.append(gt_rows(rng.permutation(E)[:m], wide_betas(rng, m, -40, 2)))
    got, ran = score(nb, gt, n, lists, pol, block=512)
    assert ran == 1
    worst = max(check_definition(got[k], gt, n, rows, pol, True, max(MAX_PARTS, int(parts or 1))) for k, rows in enumerate(lists))
    if fail:
        assert any(np.isnan(g[0]).any() for g in got) and any(np.isfinite(g[0]).any() for g in got)
    print(f"worst error / bound {worst:.3f}")


# ---- GPU: the int32 accumulator edge, in closed form -------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("E,contracts", [(1 << 22, True), ((1 << 22) + 1, False)], ids=["2^22", "2^22+1"])
def test_int32_accumulator_edge(nb, monkeypatch, E, contracts):
    """256 samples, all 1/1 (dosage 2), one definition forced through the contraction, one part, E distinct slab rows
    (2 GB).  One beta is 1 + 2^-44 (max|c|: F = 51) and E - 1 are 2^-44, so every quantised coefficient is 128 mod
    256: digit 0 is -128 on every entry and its accumulator reaches -2 * 128 * E = -2^30 at E = 2^22, the most the
    contraction takes.  The raw sum is 2 + E * 2^-43, exact in any fp64 association; one entry more falls back to
    the fused kernel with the same bits."""
    monkeypatch.setenv("NPC_MULTI", "1")
    monkeypatch.setenv("NPC_MULTI_PARTS", "1")
    n, block = 256, 1 << 16
    assert fixed_point_exponent(1 + 2.0 ** -44) == 51 and quantise(2.0 ** -44, 51) == 128 and quantise(1 + 2.0 ** -44, 51) % 256 == 128
    rows = gt_rows(np.arange(E), np.full(E, 2.0 ** -44))
    rows["beta"][E // 2] = 1 + 2.0 ** -44
    eng = nb.Engine(n, max_rows_per_block=block, n_slots=2)
    eng.set_policy(imp_sample="homref")                  # imputed 0: cm = 0, max|c| is the largest beta
    assert eng.resident_reserve(E) >= E
    for r0 in range(0, E, block):
        slot, view = eng.stage_acquire()
        m = min(block, E - r0)
        view[:m, :2 * n] = 4                             # allele code of ALT on both alleles
        eng.stage_upload(slot, m, r0)
    (sc, nloci, loci), = eng.score_resident_multi([rows], None)
    assert eng.multi_contractions == int(contracts)
    eng.close()
    assert nloci == E and (loci["klass"] == orc.CLASS_OK).all() and (loci["neff"] == 2 * n).all()
    want = 2.0 + E * 2.0 ** -43
    assert want == float(2 + Fraction(E, 2 ** 43))
    assert np.array_equal(bits(sc), bits(np.full(n, want)))
