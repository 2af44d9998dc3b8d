"""Every compiled instance of the tile kernel that the shape planner launches, against the oracle, and the default
mode's summation order pinned bit for bit.

The planner (npc_plan_shape, host arithmetic) picks, per cohort size, GT width, mode and launch length, one of a
handful of kernel instances: K chunks per consumer thread, 16 / 24 / 28 consumer warps per instance, decided-mode
slabs above ~1.2 M samples, the generic two-kernel path where no tile shape fits.  CASES names one cohort per instance
and states the plan it must get; the CPU tests check those plans and that every (width, mode, K, instance) the planner
can produce has a case, so that a new instance or a planner change without a parity case fails here.

The GPU tests score each case in both modes with adversarial rows (tally fields at their maximum, every chunk on the
exact decode, the only non-REF sample at a slab's first or the cohort's last sample): records and nloci bit-equal to
the oracle, exact-mode scores bit-equal to the oracle's serial chain, default-mode scores bit-equal to the documented
tile order (util_order.default_order_scores, DESIGN 4.1) -- a check the 1e-12 tolerance of assert_parity cannot make:
a dropped or doubled small row, or a wrong tile or row-group boundary, stays inside the tolerance."""
import numpy as np
import pytest

import orc
from nimpress_b200 import cuda
from util_cohort import random_cohort, random_rows, assert_parity, assert_loci_equal, bits
from util_order import serial_scores, default_order_scores

OFFSET = 0.25


def plan(mode, K=0, instance=0, slabs=0, groups=0, warps=0, wide=1):
    """Expected plan: mode (0 generic, 1 exact, 2 default, 3 decided), chunks per thread, instance warps, sample slabs x
    planned row groups, consumer warps, decided-mode slabs."""
    return dict(mode=mode, chunks_per_thread=K, instance_warps=instance, sample_slabs=slabs, row_groups=groups,
                consumer_warps=warps, wide_slabs=wide if mode else 0)


GENERIC = plan(0, wide=0)

# name: (samples, GT width, score rows per launch, default plan, exact plan).  Rows: at least 3 turns of the index ring
# (12 x index_tiles), never a multiple of 4 (the last tile is partial), and a last decider group that is short.
CASES = {
    "bench_launch":       (500_000, 1, 1667, plan(2, 1, 28, 74, 2, 27), plan(1, 1, 16, 148, 1, 14)),   # long launch: >= 1,611 rows
    "int8_28warp":        (1_000_000, 1, 135, plan(2, 1, 28, 148, 1, 27), plan(1, 1, 28, 148, 1, 27)),
    "int8_24warp":        (850_000, 1, 171, plan(2, 1, 24, 148, 1, 23), plan(1, 1, 24, 148, 1, 23)),
    "int8_16warp":        (100_003, 1, 387, plan(2, 1, 16, 29, 5, 14), plan(1, 1, 16, 148, 1, 3)),
    "int8_k2_row_groups": (400_000, 1, 303, plan(2, 2, 16, 49, 3, 16), plan(1, 1, 16, 148, 1, 11)),
    "int8_k2_resident":   (1_150_000, 1, 135, plan(2, 2, 16, 148, 1, 16), plan(1, 2, 16, 148, 1, 16)),
    "decided_24warp":     (1_300_000, 1, 195, plan(3, 1, 24, 148, 1, 18, 2), plan(3, 1, 24, 148, 1, 18, 2)),
    "decided_28warp":     (2_000_000, 1, 135, plan(3, 1, 28, 148, 1, 27, 2), plan(3, 1, 28, 148, 1, 27, 2)),
    "decided_k2":         (2_200_000, 1, 135, plan(3, 2, 16, 148, 1, 15, 2), plan(3, 2, 16, 148, 1, 15, 2)),
    "int16_16warp":       (100_003, 2, 387, plan(2, 1, 16, 29, 5, 14), plan(1, 1, 16, 148, 1, 3)),
    "int16_k2":           (700_000, 2, 163, plan(2, 2, 16, 148, 1, 10), plan(1, 2, 16, 148, 1, 10)),
    "int16_generic":      (1_000_000, 2, 135, GENERIC, GENERIC),
}


def case_plan(name, exact):
    n, width, rows = CASES[name][:3]
    return cuda.plan_shape(n, width, n_rows=rows, exact=exact)


def instance(width, exact, p):
    return (width, bool(exact), p["mode"], p["chunks_per_thread"], p["instance_warps"])


# ---- CPU: the plans, the coverage of the planner's instances, the serial model ------------------------------------

@pytest.mark.parametrize("name", list(CASES))
def test_case_plans(name):
    n, width, rows, want_default, want_exact = CASES[name]
    for exact, want in ((False, want_default), (True, want_exact)):
        p = case_plan(name, exact)
        assert {k: p[k] for k in want} == want, (exact, p)
        if p["mode"] == 0:
            continue
        tiles = -(-rows // 4)
        assert rows % 4 and rows >= 12 * p["index_tiles"], p
        groups = max(1, min(p["row_groups"], tiles // 16))
        assert any((tiles * (g + 1) // groups - tiles * g // groups) % p["decider_tiles"] for g in range(groups)), p


def sweep():
    """(width, exact, mode, K, instance warps) -> first (samples, rows per launch) the planner gives it: cohorts of
    1,000 to 2.4 M samples, short (64 rows) and long (2^20 rows) launches, and the cohort sizes of the parity tests."""
    sizes = list(range(1000, 2_400_001, 997)) + [1, 7, 8, 9, 255, 256, 257, 3001, 4099, 5003, 20011, 40009, 100003,
                                                 157_929, 250_000, 500_000, 850_000, 1_150_000, 1_300_000, 2_000_000]
    seen = {}
    for width in (1, 2):
        for exact in (False, True):
            for n_rows in (64, 1 << 20):
                for n in sizes:
                    seen.setdefault(instance(width, exact, cuda.plan_shape(n, width, n_rows=n_rows, exact=exact)), (n, n_rows))
    return seen


def test_every_planned_instance_has_a_case():
    covered = {}
    for name, (n, width, rows, _, _) in CASES.items():
        for exact in (False, True):
            covered.setdefault(instance(width, exact, case_plan(name, exact)), name)
    missing = {t: at for t, at in sweep().items() if t not in covered}
    assert not missing, f"planned kernel instances without a parity case in CASES (instance: samples, rows): {missing}"


@pytest.mark.parametrize("width", [1, 2])
def test_serial_model_is_the_oracle(width):
    """util_order's decode and addends, summed in row order, are the oracle's scores bit for bit: random cohorts with
    sentinels, invalid bytes and alleles past ALT3, several policies, beta in {0, -0.0, 1e-9} on rows of every kind.
    A beta of +-inf on a decoded row makes every sample non-finite -- NaN where fl(0 * inf) is added, +-inf elsewhere
    -- so it is checked on its own, by that pattern; a NaN beta only on a row the policy drops, where it must not
    poison a score.  The default-order model of the same rows stays within assert_parity's tolerance of the oracle but
    is not its bits."""
    rng = np.random.default_rng(40 + width)
    n, V = 5003, 40
    gt = random_cohort(rng, n, V, width=width, miss_rate=0.04, n_alt=5, sentinel_rate=0.01, invalid_rate=0.002)
    rows = random_rows(rng, V, n_rows=97, n_alt=5, nan_eaf_rate=0.0)
    rows["beta"][[3, 10, 20, 50, 60, 70]] = [0.0, -0.0, 1e-9, 0.0, -0.0, 1e-9]
    odd = np.nonzero(rows["kind"] == 0)[0][::7]
    rows["eaidx"][odd], rows["ref_is_ea"][odd] = 6, 0
    # policies under which most scores stay finite
    for pol in (dict(), dict(imp_sample="int_ps", mincs=0), dict(imp_locus="homref", imp_missing="ignore", maxmis=0.02, mincs=4000),
                dict(imp_sample="ps", maxmis=1.0), dict(imp_locus="ignore", imp_sample="int_fail", mincs=0),
                dict(imp_locus="homref", imp_sample="homref", maxmis=0.0)):
        want = orc.score_matrix(gt, n, 2, rows, offset=OFFSET, **pol)
        assert np.isfinite(want["scores"]).sum() > n // 2, pol
        assert_bits_equal(serial_scores(gt, n, rows, want["loci"], want["nloci"], OFFSET), want["scores"])
    dec = np.nonzero((rows["kind"] == 0) & (rows["eaidx"] == 1))[0][0]
    for b in (np.inf, -np.inf):                            # NaN on samples with dosage 0, +-inf on the others
        r2 = rows.copy()
        r2["beta"][dec] = b
        want = orc.score_matrix(gt, n, 2, r2, offset=OFFSET, maxmis=1.0)
        nan = np.isnan(want["scores"]).sum()
        assert 0 < nan < n and (want["scores"] == b).sum() > 0
        assert_bits_equal(serial_scores(gt, n, r2, want["loci"], want["nloci"], OFFSET), want["scores"])
    r2 = rows.copy()
    nc = np.nonzero(r2["kind"] == 1)[0]
    r2["beta"][nc] = np.nan                                # not-covered rows under --imp-locus ignore: dropped
    pol = dict(imp_locus="ignore")
    want = orc.score_matrix(gt, n, 2, r2, offset=OFFSET, **pol)
    assert nc.size and np.isfinite(want["scores"]).all()
    assert_bits_equal(serial_scores(gt, n, r2, want["loci"], want["nloci"], OFFSET), want["scores"])
    want = orc.score_matrix(gt, n, 2, rows, offset=OFFSET, imp_sample="ps")
    model = default_order_scores(gt, n, rows, want["loci"], want["nloci"], OFFSET, [len(rows)], lambda r: 1)
    assert_parity(dict(scores=model, nloci=want["nloci"], loci=want["loci"]), want, exact=False)
    ok = np.isfinite(model)
    assert ok.sum() > n // 2 and (bits(model[ok]) != bits(want["scores"][ok])).sum() > 0


def assert_bits_equal(got, want, what="scores"):
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN pattern differs"
    ok = ~np.isnan(want)
    bad = np.nonzero(bits(got[ok]) != bits(want[ok]))[0]
    assert bad.size == 0, f"{what}: {bad.size} of {ok.sum()} differ in bits, first {got[ok][bad[:3]]} vs {want[ok][bad[:3]]}"


# ---- GPU: every case in both modes ----------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def nb():
    import __graft_entry__ as g
    g.build()
    import nimpress_b200
    return nimpress_b200


def slab_starts(n, p):
    """First sample of every CTA's share of the sample axis (npc_fused5.cuh:152-155); in decided mode, of every wide
    slab and of the CTA shares inside the first one."""
    n_slab = p["wide_samples"] if p["mode"] == 3 else n
    C, gs = -(-n_slab // 8), max(p["sample_slabs"], 1)
    q, rem = divmod(C, gs)
    starts = [8 * (s * q + min(s, rem)) for s in range(gs)]
    if p["mode"] == 3:
        starts += [p["wide_samples"] * s for s in range(1, p["wide_slabs"])]
    return starts


ADV = 8                                                    # adversarial genotype rows per case


def adversarial_rows(n, width, stride, p, p_exact, rng):
    """Genotype rows at the limits of the packed tallies and the decode paths: every sample homozygous ALT1
    (neff = 2n: every 6-bit field at its per-group maximum), every sample missing, every sample a half call, one ALT3
    in every chunk (the exact decode everywhere), and rows whose only non-REF sample is the cohort's last sample, the
    first sample of a CTA's slab in the middle of the default plan's grid, of its last (wide) slab, or of the exact
    plan's middle slab (its grid splits the samples differently)."""
    dt = {1: np.int8, 2: np.int16}[width]
    base = np.full((ADV, 2 * n), 2, dt)                    # 0|0
    base[0] = 4 | rng.integers(0, 2, size=2 * n)           # 1|1, either phase
    base[1] = rng.integers(0, 2, size=2 * n)               # ./.
    base[2, 0::2] = 0                                      # ./1
    base[2, 1::2] = 4
    base[3] = np.where(rng.random(2 * n) < 0.2, 4, 2)
    base[3, 0::16] = 8                                     # ALT3 in the first sample of every chunk of 8
    base[4, 2 * n - 1] = 4
    starts = slab_starts(n, p)
    base[5, 2 * starts[len(starts) // 2]] = 4
    base[6, 2 * starts[-1] + 1] = 4
    starts = slab_starts(n, p_exact)
    base[7, 2 * starts[len(starts) // 2] + 1] = 4
    out = np.zeros((ADV, stride // width), dt)
    out[:, :2 * n] = base
    return out


def build_case(name, rng):
    """Cohort (host array, rows x stride bytes) and score rows of a case."""
    n, width, R = CASES[name][:3]
    stride = -(-2 * n * width // 128) * 128
    if width == 1:
        V = 40
        gt = np.zeros((V + ADV, stride), np.int8)
        orc.synth_fill(gt[:V], n, 0, 0x6E696D70 + n, (rng.uniform(0.01, 0.5, V) * 65536).astype(np.uint32),
                       (rng.uniform(0, 0.1, V) * (1 << 24)).astype(np.uint32), rng.integers(1, 4, V).astype(np.int32))
        for r in range(4):                                 # sentinels and invalid bytes: the exact decode in scattered chunks
            at = rng.choice(2 * n, size=max(n // 500, 4), replace=False)
            gt[r, at] = rng.choice([-128, -127, -3, 126], size=at.size)
    else:
        V = 24
        gt = np.zeros((V + ADV, stride // 2), np.int16)
        for r in range(0, V, 8):                           # in slices: random_cohort holds int64 temporaries
            gt[r:r + 8] = random_cohort(rng, n, 8, width=2, miss_rate=0.03, n_alt=4 if r else 90, sentinel_rate=0.003,
                                        invalid_rate=0.0005, pad_to=128)
    gt[V:] = adversarial_rows(n, width, stride, case_plan(name, False), case_plan(name, True), rng)
    rows = random_rows(rng, V + ADV, n_rows=R, n_alt=3, nan_eaf_rate=0.0)
    gt_rows = np.nonzero(rows["kind"] == 0)[0]
    rows["eaidx"][gt_rows[::9]] = rng.integers(4, 8, size=gt_rows[::9].size)     # no allele matches: the T >= 4 table
    rows["ref_is_ea"][gt_rows[::9]] = 0
    # each adversarial row several times, ending the block, in every position of a tile, with the effect alleles that
    # make it extreme (ALT1; REF for the all-missing / half-call rows too)
    at = np.concatenate([[R - 1], rng.choice(R - 1, size=3 * ADV - 3, replace=False)])
    a = np.arange(at.size) % ADV
    rows["kind"][at], rows["gt_row"][at] = 0, V + a
    rows["eaidx"][at] = np.where(np.isin(a, (1, 2)) & (np.arange(at.size) >= ADV), 0, 1)
    rows["ref_is_ea"][at] = rows["eaidx"][at] == 0
    rows["beta"][at] = np.round(rng.normal(0, 0.05, at.size), 4)
    rows["eaf"][at[np.isin(a, (0, 4, 5, 6, 7))]] = np.nan    # no missing calls: the tallies impute, a NaN eaf is never read
    rows["beta"][at[:3]] = [1e-9, -0.0, 3.0]
    return gt, rows


_cache = {}


def case_data(name):
    """Cohort, rows and oracle result of one case (the last one only: the bench launch's cohort is the large one)."""
    if name not in _cache:
        _cache.clear()
        n = CASES[name][0]
        gt, rows = build_case(name, np.random.default_rng(sum(map(ord, name))))
        _cache[name] = (gt, rows, orc.score_matrix(gt, n, 2, rows, offset=OFFSET, threads=1))
    return _cache[name]


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", [(c, m) for c in CASES for m in ("default", "exact")])
def test_instance_parity(nb, name, mode):
    import torch
    n, width, R = CASES[name][:3]
    exact = mode == "exact"
    want_plan = CASES[name][4 if exact else 3]
    gt, rows, want = case_data(name)
    assert np.isfinite(want["scores"]).all()
    eng = nb.Engine(n, gt_width=width, max_rows_per_block=R)
    eng.set_policy(); eng.set_exact_order(exact); eng.reset()
    shape = eng.kernel_shape_for(R)
    assert shape["fused"] == want_plan["mode"], shape
    p = case_plan(name, exact)                             # the context reports the launch the planner chose
    for k in ("decider_warps", "decider_tiles", "lag", "raw_stages", "index_tiles", "smem_bytes"):
        assert shape[k] == p[k], (k, shape, p)
    if want_plan["mode"]:
        for k in ("chunks_per_thread", "consumer_warps"):
            assert shape[k] == want_plan[k], (k, shape)
        assert shape["row_groups"] == (want_plan["row_groups"] if want_plan["mode"] == 2 else 1), shape
        assert shape["grid"] == want_plan["sample_slabs"] * shape["row_groups"], shape
    d = torch.from_numpy(gt.view(np.uint8)).cuda()
    eng.score_block_device(d, d.shape[1], gt.shape[0], rows)
    got = eng.finish(offset=OFFSET)
    eng.close()
    del d
    assert got["nloci"] == want["nloci"]
    assert_loci_equal(got["loci"], want["loci"])
    if exact or want_plan["mode"] == 0:                    # the exact-order kernel, the generic kernels: the oracle's chain
        assert_bits_equal(got["scores"], want["scores"])
    else:
        assert_parity(got, want, exact=False)
        model = default_order_scores(gt, n, rows, want["loci"], want["nloci"], OFFSET, [R], lambda r: shape["row_groups"])
        assert_bits_equal(got["scores"], model, "scores against the default tile order")


# ---- GPU: the default order on cheap shapes -------------------------------------------------------------------------

CHEAP = {
    "GR=1":               (40_009, dict(NPC_TILE_GR="1"), 1029, "device"),
    "GR=3":               (100_003, dict(NPC_TILE_GR="3"), 1029, "device"),
    "GR=4":               (100_003, dict(NPC_TILE_GR="4"), 1029, "device"),
    "GR=16":              (40_009, dict(NPC_TILE_GR="16"), 1029, "device"),
    "K=2":                (100_003, dict(NPC_TILE_K="2"), 1029, "device"),
    "LONG_MB=1":          (40_009, dict(NPC_TILE_LONG_MB="1"), 1029, "device"),
    "blocks_of_17":       (100_003, dict(), 1029, "staged"),
    "resident_split":     (40_009, dict(), 1029, "resident"),
    "row_group_cap":      (40_009, dict(), 135, "device"),     # 12 planned row groups, 34 tiles: 2 launched
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CHEAP))
def test_default_order_cheap_shapes(nb, name, monkeypatch):
    """The default tile kernel's scores are the documented order's bits under forced row-group counts, two chunks per
    thread, the long-launch split, streaming blocks of 17 rows and npc_score_resident's cut at max_rows_per_block."""
    n, env, R, how = CHEAP[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(sum(map(ord, name)))
    V = 203
    gt = random_cohort(rng, n, V, miss_rate=0.03, n_alt=9, sentinel_rate=0.003, invalid_rate=0.0005)
    rows = random_rows(rng, V, n_rows=R, n_alt=9, nan_eaf_rate=0.0)    # a NaN eaf on a constant row makes every score NaN
    want = orc.score_matrix(gt, n, 2, rows, offset=OFFSET)
    assert np.isfinite(want["scores"]).all()
    max_rows = {"device": max(R, V), "staged": max(R, V), "resident": 300}[how]
    eng = nb.Engine(n, max_rows_per_block=max_rows, n_slots=0 if how == "device" else 2)
    eng.set_policy(); eng.reset()
    if how == "device":
        import torch
        d = torch.from_numpy(gt.view(np.uint8).reshape(V, -1)).cuda()
        eng.score_block_device(d, d.shape[1], V, rows)
        blocks = [R]
    elif how == "staged":
        for r0 in range(0, R, 17):
            eng.score_host(gt, rows[r0:r0 + 17])
        blocks = [min(17, R - r0) for r0 in range(0, R, 17)]
    else:
        assert eng.resident_reserve(V) >= V
        slot, view = eng.stage_acquire()
        g8 = gt.view(np.uint8).reshape(V, -1)
        view[:V, :g8.shape[1]] = g8
        eng.stage_upload(slot, V, 0)
        eng.score_resident(rows)
        blocks = [min(max_rows, R - r0) for r0 in range(0, R, max_rows)]
    shapes = {b: eng.kernel_shape_for(b) for b in set(blocks)}
    got = eng.finish(offset=OFFSET)
    eng.close()
    for b, s in shapes.items():
        assert s["fused"] == 2, (b, s)
        if "NPC_TILE_GR" in env:
            assert s["row_groups"] == int(env["NPC_TILE_GR"]), s
        if "NPC_TILE_K" in env:
            assert s["chunks_per_thread"] == 2, s
    if name == "LONG_MB=1":
        assert shapes[R]["row_groups"] == cuda.plan_shape(n, n_rows=1 << 30)["row_groups"] != cuda.plan_shape(n, n_rows=1)["row_groups"]
    assert_parity(got, want, exact=False)
    model = default_order_scores(gt, n, rows, want["loci"], want["nloci"], OFFSET, blocks, lambda b: shapes[b]["row_groups"])
    assert_bits_equal(got["scores"], model, "scores against the default tile order")
