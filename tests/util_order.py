"""Tests-only: the two summation orders of the tile kernel, restated in numpy so that scores can be checked bit for bit.

Both orders add the same addends -- the reference's rounded products fl(dosage*beta) (src/nimpress.nim:640) -- and differ
only in their association:

  * serial_scores: the reference's chain, scores[i] += dosages[i]*beta row by row (:639-640), then the epilogue
    (:643-649).  It is the oracle's order, the exact mode's and the generic kernels'.
  * default_order_scores: the default tile kernel (npc_fused5.cuh, DESIGN 4.1): tiles of four rows counted from each
    launch's first row, sum = (sum + (v0 + v1)) + (v2 + v3); the launch's row groups each sum their contiguous tiles,
    group 0 onto the running sums and groups g > 0 from 0.0, and k_add_partials adds the groups in order.

The addends come from the oracle's per-locus records (klass, used, imputed), so the model needs no decide logic of its
own: a wrong record is caught by the record comparison, a wrong order by the score bits.  Every array is a vector over
the samples -- never rows x samples, which at the bench launch (1,664 rows x 500,000 samples) would be 6.6 GB."""
import numpy as np

import orc

_SENT = {1: (-128, -127), 2: (-32768, -32767), 4: (-2147483648, -2147483647)}   # (missing, vector_end) per width


def dosage_codes(gt_row, n, width, eaidx):
    """Per-sample dosage code of one diploid genotype row: 0, 1, 2, or 3 for a missing call.  decode_sample
    (npc_kernels.cuh:56-67), i.e. getRawDosages (:384-391) on the stored integers: a vector_end ends the sample, a
    missing sentinel is skipped, allele value (raw >> 1) - 1 (raw itself when negative) == eaidx adds 1, == -1 makes
    the sample missing (sticky: a NaN stays NaN under a later += 1)."""
    miss_s, vend = _SENT[width]
    a = np.asarray(gt_row)[:2 * n].reshape(n, 2).astype(np.int32)
    d = np.zeros(n, np.int32)
    miss = np.zeros(n, bool)
    ended = np.zeros(n, bool)
    for k in range(2):
        raw = a[:, k]
        ended |= raw == vend
        live = ~ended & (raw != miss_s)
        val = np.where(raw < 0, raw, (raw >> 1) - 1)
        hit = live & (val == eaidx)
        d += hit
        miss |= live & ~hit & (val == -1)
    return np.where(miss, 3, d)


def addends(gt, n, rows, loci):
    """What each score row adds to every sample, in row order: a float64 vector over the samples, or a float64 scalar
    where every sample gets the same value.  decide_row (npc_kernels.cuh:236-283) from the oracle's record of the row:
      * not used (used == 0): 0.0 -- the tile kernel's dropped row (npc_fused5.cuh:281);
      * constant (klass != OK: not covered, absent, FILTER, over --maxmis): fl(imputed * beta) (:280);
      * decoded (klass == OK): [fl(0*b), fl(1*b), fl(2*b), fl(imputed*b)][code] (:273-276)."""
    width = gt.dtype.itemsize
    for row, rec in zip(rows, loci):
        beta = np.float64(row["beta"])
        if not rec["used"]:
            yield np.float64(0.0)
        elif rec["klass"] != orc.CLASS_OK:
            yield np.float64(rec["imputed"]) * beta
        else:
            table = np.array([np.float64(0.0) * beta, np.float64(1.0) * beta, np.float64(2.0) * beta,
                              np.float64(rec["imputed"]) * beta])
            yield table[dosage_codes(gt[int(row["gt_row"])], n, width, int(row["eaidx"]))]


def finalize(sums, nloci, offset):
    """k_finalize (npc_kernels.cuh:431-437), the reference's epilogue: one rounded divide by fl(nloci * 2), one rounded
    add of the offset (0/0 = NaN, x/0 = +-inf)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return sums / (np.float64(nloci) * 2.0) + np.float64(offset)


def serial_scores(gt, n, rows, loci, nloci, offset):
    """The reference's chain: every row's addend onto the running sum, rows in score-file order.  A row that is not used
    adds +0.0 here where the reference skips it: the same bits, since a sum that starts at +0.0 never becomes -0.0."""
    sums = np.zeros(n, np.float64)
    for a in addends(gt, n, rows, loci):
        sums = sums + a
    return finalize(sums, nloci, offset)


def default_order_scores(gt, n, rows, loci, nloci, offset, blocks, row_groups_of):
    """The default tile kernel's order.  blocks: score rows per launch, in order (the caller's blocks, or
    npc_score_resident's cut at max_rows_per_block); row_groups_of(n_rows): the planned row groups of a launch of that
    many rows (Engine.kernel_shape_for(n_rows)["row_groups"]).  Per launch:
      * tiles of four rows from the launch's first row; rows past its end add +0.0 (npc_fused5.cuh:274, 281);
      * gr = max(1, min(planned, tiles // 16)) row groups (npc_api.cu:657-659); group g owns tiles
        [tiles*g // gr, tiles*(g+1) // gr) (npc_fused5.cuh:148-149);
      * per tile T01 = v0 + v1, T23 = v2 + v3 (:315), then sum = (sum + T01) + T23 (:475-476); group 0 starts from the
        running sums, groups g > 0 from 0.0 (:352);
      * k_add_partials: sums = ((sums + p1) + p2) + ... in group order (npc_fused.cuh:126-132)."""
    assert sum(blocks) == len(rows)
    sums = np.zeros(n, np.float64)
    it = addends(gt, n, rows, loci)
    zero = np.float64(0.0)
    for nb in blocks:
        tiles = (nb + 3) // 4
        gr = max(1, min(int(row_groups_of(nb)), tiles // 16))
        parts = []
        for g in range(gr):                       # groups own consecutive tiles: the addends are taken in row order
            acc = sums if g == 0 else np.zeros(n, np.float64)
            for t in range(tiles * g // gr, tiles * (g + 1) // gr):
                v0, v1, v2, v3 = (next(it) if 4 * t + r < nb else zero for r in range(4))
                acc = (acc + (v0 + v1)) + (v2 + v3)
            parts.append(acc)
        sums = parts[0]
        for p in parts[1:]:
            sums = sums + p
    return finalize(sums, nloci, offset)
