"""Tests-only: BGEN v1.2 layout-2 genotype blocks at any bit depth B (1 to 16), with per-sample ploidy 0, 1 or 2 and
missing samples, written with numpy; util_bgen.write_bgen writes the file around them.

Conventions (DESIGN.md 4.9): D = 2^B - 1 and a stored value v is the probability v / D.  Each sample stores `ploidy`
values, packed back to back least-significant bit first (value i at bits i*B .. i*B+B-1 of the little-endian stream):
unphased diploid b0 = P(hom allele 1), b1 = P(het); phased diploid h0, h1 = P(haplotype carries allele 1); haploid b0 =
P(allele 1).  A missing sample has bit 7 of its ploidy byte set and zero values.  The engine's 32-bit dosage row is a
16-byte header (uint32 D, 12 zero bytes) and one uint32 word per sample: k | ploidy << 24 with k = D x the expected
ALT dosage, 0xFFFFFFFF for a missing sample or ploidy 0."""
import struct

import numpy as np

from util_bgen import LOCUS, LOCUS_DTYPE, MISSING_POL, SAMPLE

MISSING32 = 0xFFFFFFFF
VEND8 = -127                                     # int8 vector_end: a haploid call in a diploid GT row


def pack_values(values, B):
    """B-bit values, least-significant bit first, into bytes (the last byte zero-padded)."""
    v = np.asarray(values, np.int64).reshape(-1)
    bits = ((v[:, None] >> np.arange(B)) & 1).astype(np.uint8).reshape(-1)
    return np.packbits(bits, bitorder="little").tobytes()


def genotype_block_bits(n, vals, ploidy, missing, phased, bits, K=2, pmin=None, pmax=None, n_stored=None):
    """Uncompressed probability data of one variant: sample i stores vals[i, :ploidy[i]] at `bits` bits each."""
    ploidy = np.asarray(ploidy, np.int64)
    vals = np.asarray(vals, np.int64)
    pmin = int(ploidy.min()) if pmin is None else pmin
    pmax = int(ploidy.max()) if pmax is None else pmax
    pb = (ploidy | np.where(np.asarray(missing, bool), 0x80, 0)).astype(np.uint8)
    stored = np.concatenate([vals[i, :ploidy[i]] for i in range(n)]) if n else np.zeros(0, np.int64)
    head = struct.pack("<IHBB", n if n_stored is None else n_stored, K, pmin, pmax)
    return head + pb.tobytes() + struct.pack("<BB", int(bool(phased)), bits) + pack_values(stored, bits)


def numerators(vals, ploidy, missing, phased, bits):
    """uint32 words of the engine's 32-bit dosage row for one variant."""
    D = (1 << bits) - 1
    v = np.asarray(vals, np.int64)
    p = np.asarray(ploidy, np.int64)
    k2 = 2 * D - v[:, 0] - v[:, 1] if phased else 2 * D - 2 * v[:, 0] - v[:, 1]
    k = np.where(p == 1, D - v[:, 0], k2)
    miss = np.asarray(missing, bool) | (p == 0)
    return np.where(miss, MISSING32, k | (p << 24)).astype(np.uint32)


def random_values(rng, n, bits, phased, haploid_rate=0.0, ploidy0_rate=0.0, miss_rate=0.05, hard_rate=0.2):
    """Random fractional values at `bits` bits, hard calls mixed in -> (vals int64[n, 2], ploidy[n], missing[n]).  A
    haploid sample uses vals[:, 0] only; a missing sample's values are zero."""
    D = (1 << bits) - 1
    ploidy = np.where(rng.random(n) < haploid_rate, 1, 2)
    ploidy[rng.random(n) < ploidy0_rate] = 0
    if phased:
        vals = rng.integers(0, D + 1, size=(n, 2))
        hard = rng.random((n, 2)) < hard_rate
        vals = np.where(hard, D * rng.integers(0, 2, size=(n, 2)), vals)
    else:
        b0 = rng.integers(0, D + 1, size=n)
        b1 = np.minimum((rng.random(n) * (D + 1 - b0)).astype(np.int64), D - b0)     # b0 + b1 <= D
        vals = np.stack([b0, b1], axis=1)
        hard = rng.random(n) < hard_rate
        vals[hard] = np.array([[D, 0], [0, D], [0, 0]])[rng.integers(0, 3, size=int(hard.sum()))]
    hap = ploidy == 1
    vals[hap, 0] = np.where(rng.random(int(hap.sum())) < hard_rate, D * rng.integers(0, 2, size=int(hap.sum())), vals[hap, 0])
    vals[hap, 1] = 0
    vals[ploidy == 0] = 0
    missing = rng.random(n) < miss_rate
    vals[missing] = 0
    return vals, ploidy, missing


def dose32_rows(words, D, pad_to=16, rng=None):
    """The engine's rows uint8[V, 16 + 4 cols]: header with D[v], then words[v] (cols = words.shape[1], which may run
    past n: those words must never be read)."""
    words = np.asarray(words, np.uint32)
    V, cols = words.shape
    width = -(-(16 + 4 * cols) // pad_to) * pad_to
    out = np.zeros((V, width), np.uint8)
    out[:, :4] = np.asarray(D, np.uint32).reshape(V, 1).view(np.uint8)
    out[:, 16:16 + 4 * cols] = words.view(np.uint8).reshape(V, 4 * cols)
    if rng is not None and width > 16 + 4 * cols:
        out[:, 16 + 4 * cols:] = rng.integers(0, 256, size=(V, width - 16 - 4 * cols))
    return out


def refusal_blocks(n, rng):
    """A well-formed 12-bit block with haploid and diploid samples, and blocks that no dosage row holds, each with a part
    of the message that refuses it -> (good, [(block, message), ...])."""
    vals, ploidy, miss = random_values(rng, n, 12, False, haploid_rate=0.3, miss_rate=0.0)
    ploidy[:2] = (1, 2)
    good = genotype_block_bits(n, vals, ploidy, miss, False, 12)
    over = vals.copy()
    over[ploidy == 2] = [4000, 100]                                     # b0 + b1 > 4095
    h = 8 + n                                                           # offset of the phased flag
    return good, [(genotype_block_bits(n, vals, ploidy, miss, False, 12, K=3), "3 alleles"),
                  (good[:h + 1] + b"\x00" + good[h + 2:], "0 bits"),
                  (good[:h + 1] + b"\x11" + good[h + 2:], "17 bits"),
                  (genotype_block_bits(n, vals, ploidy, miss, False, 12, pmax=3), "ploidy 1..3"),
                  (genotype_block_bits(n, vals, ploidy, miss, False, 12, pmin=1, pmax=1), "sample 1: ploidy 2 outside 1..1"),
                  (genotype_block_bits(n, over, ploidy, miss, False, 12), "> 1"),
                  (genotype_block_bits(n, vals, ploidy, miss, False, 12, n_stored=n + 1), "samples"),
                  (good[:-3], f"too short for {n} samples at 12 bits")]


# ---- hard calls -----------------------------------------------------------------------------------------------------


def hard_cohort(rng, n, V, haploid_rate=0.1, miss_rate=0.03, halfcall_rate=0.01, pad_to=16):
    """Biallelic hard calls -> (gt int8[V, cols] raw BCF GT rows, a haploid sample written as allele then vector_end;
    alleles int64[V, n, 2] with -1 missing; ploidy[V, n])."""
    af = rng.uniform(0.01, 0.5, size=(V, 1, 1))
    al = (rng.random((V, n, 2)) < af).astype(np.int64)
    raw = ((al + 1) << 1) | (rng.random((V, n, 2)) < 0.3)
    miss = rng.random((V, n)) < miss_rate * rng.uniform(0, 2, size=(V, 1))
    raw[miss] &= 1
    half = rng.random((V, n)) < halfcall_rate
    raw[half, 0] &= 1
    ploidy = np.where(rng.random((V, n)) < haploid_rate, 1, 2)
    raw[..., 1] = np.where(ploidy == 1, VEND8, raw[..., 1])
    cols = -(-2 * n // pad_to) * pad_to
    gt = np.zeros((V, cols), np.int8)
    gt[:, :2 * n] = raw.reshape(V, 2 * n).astype(np.int8)
    gt[:, 2 * n:] = rng.integers(0, 6, size=(V, cols - 2 * n)).astype(np.int8)
    alleles = np.where((raw & ~1) == 0, -1, (raw >> 1) - 1)
    alleles[..., 1] = np.where(ploidy == 1, 0, alleles[..., 1])
    return gt, alleles, ploidy


def hard_values(alleles, ploidy, phased, bits):
    """One variant's hard calls (alleles[n, 2], -1 missing; ploidy[n]) as BGEN values -> (vals, ploidy, missing)."""
    D = (1 << bits) - 1
    a = np.asarray(alleles, np.int64)
    p = np.asarray(ploidy, np.int64)
    missing = (a[:, 0] < 0) | ((p == 2) & (a[:, 1] < 0))
    if phased:
        vals = np.where(a == 0, D, 0)
    else:
        n_alt = (a == 1).sum(axis=1)
        vals = np.stack([np.where(n_alt == 0, D, 0), np.where(n_alt == 1, D, 0)], axis=1)
    vals = np.where((p == 1)[:, None], np.stack([np.where(a[:, 0] == 0, D, 0), np.zeros_like(a[:, 0])], axis=1), vals)
    vals[missing] = 0
    return vals, p, missing


def split_records_keep_haploid(records):
    """util_plink.split_records, with each haploid call (allele, vector_end) kept as one."""
    from util_plink import split_records
    out = []
    for r in records:
        for o in split_records([r]):
            g = np.asarray(r["gt"])
            o["gt"] = np.where(g == VEND8, VEND8, o["gt"]).astype(g.dtype)
            out.append(o)
    return out


def records_to_variants_bits(records, n, bits, rng=None):
    """Split biallelic records with haploid calls -> hard-call BGEN variants at `bits` bits; with rng, some phased."""
    out = []
    for r in records:
        phased = bool(rng is not None and rng.random() < 0.4)
        g = np.asarray(r["gt"]).reshape(n, 2).astype(np.int64)
        ploidy = np.where(g[:, 1] == VEND8, 1, 2)
        a = np.where((g & ~1) == 0, -1, (g >> 1) - 1)
        a[:, 1] = np.where(ploidy == 1, 0, a[:, 1])
        vals, p, miss = hard_values(a, ploidy, phased, bits)
        out.append(dict(contig=r["contig"], pos=r["pos"], alleles=[r["ref"], r["alts"][0] if r["alts"] else "."],
                        block=genotype_block_bits(n, vals, p, miss, phased, bits)))
    return out


# ---- reference restatement of scoring on 32-bit dosage rows (DESIGN.md 4.9) ----------------------------------------


def reference_scores_dose32(words, D, n, rows, offset=0.0, imp_locus="ps", imp_missing="homref", imp_sample="int_ps",
                            maxmis=0.05, mincs=100):
    """computePolygenicScores (src/nimpress.nim:592-649) on 32-bit dosage rows words[V, >= n] with denominators D[V],
    restated per score row in the reference's order with numpy's correctly rounded fp64 operations, as
    util_bgen.reference_scores does for 2-byte rows: a word is called when bit 31 is clear, its ploidy p (bits 24-25) is
    1 or 2 and k (bits 0-23) <= p*D; k' = p*D - k for eaidx 0; raw dosage fl(k'/D); tallies nmiss and neff_num = sum k'
    as integers, neff = fl(neff_num / D); the --maxmis rule, imputeLocusDosages and imputeSampleDosages as the reference
    has them; scores = fl(scores + fl(dosage * beta)) row after row; then / fl(nloci * 2) and + offset.  The record's
    neff is neff_num."""
    words = np.asarray(words, np.uint32)
    D = np.asarray(D, np.int64).reshape(-1)
    scores = np.zeros(n, np.float64)
    loci = np.zeros(len(rows), dtype=LOCUS_DTYPE)
    nloci = 0

    def locus_value(r):                                   # imputeLocusDosages (:417-447); None: the locus is dropped
        m = LOCUS[imp_locus]
        if m == 3:
            return None
        return float(r["eaf"]) * 2.0 if m == 0 else (2.0 if r["ref_is_ea"] else 0.0) if m == 1 else float("nan")

    for i, r in enumerate(rows):
        rec = loci[i]
        rec["eaidx"], rec["ngt"], rec["nmiss"], rec["neff"], rec["imputed"] = -1, -1, -1, -1, np.nan
        dos = None
        kind = int(r["kind"])
        if kind == 1:                                                           # not covered (:526-531)
            rec["klass"] = 1
            v = locus_value(r)
        elif kind == 3:                                                         # FILTER (:553-558)
            rec["klass"], rec["eaidx"] = 3, r["eaidx"]
            v = locus_value(r)
        elif kind == 2 or r["gt_row"] < 0:                                      # absent (:536-551)
            rec["klass"] = 2
            v = (2.0 if r["ref_is_ea"] else 0.0) if MISSING_POL[imp_missing] == 0 else None
        else:
            rec["eaidx"] = r["eaidx"]
            d = int(D[r["gt_row"]])
            w = words[r["gt_row"], :n].astype(np.int64)
            p = (w >> 24) & 3
            k = w & 0xFFFFFF
            miss = ~(((w >> 31) == 0) & ((p == 1) | (p == 2)) & (k <= p * d))
            kk = np.where(r["eaidx"] == 0, p * d - k, k)
            nmiss = int(miss.sum())
            num = int(kk[~miss].sum())
            ngt = n - nmiss
            rec["ngt"], rec["nmiss"], rec["neff"] = ngt, nmiss, num
            neff = float(num) / float(d)
            if float(nmiss) / float(n) > maxmis:                                # :565-571
                rec["klass"] = 4
                v = locus_value(r)
            else:                                                               # :582, imputeSampleDosages :450-481
                rec["klass"] = 0
                m = SAMPLE[imp_sample]
                if m == 0:
                    v = float(r["eaf"]) * 2.0
                elif m == 1:
                    v = 2.0 if r["ref_is_ea"] else 0.0
                elif m == 2:
                    v = float("nan")
                elif float(ngt) >= float(mincs):
                    v = neff / float(ngt)
                else:
                    v = float(r["eaf"]) * 2.0 if m == 3 else float("nan")
                dos = np.where(miss, v, kk.astype(np.float64) / float(d))
        rec["used"] = v is not None
        if v is None:
            continue
        rec["imputed"] = v
        if dos is None:
            dos = np.full(n, v, np.float64)
        scores = scores + dos * float(r["beta"])                                # :639-641
        nloci += 1
    with np.errstate(divide="ignore", invalid="ignore"):
        scores = scores / (float(nloci) * 2.0) + offset                           # :643-649
    return dict(scores=scores, loci=loci, nloci=nloci)
