"""Tests-only: BGEN v1.2 files (layout 2, 8-bit probabilities) written with numpy and zlib.

Conventions (DESIGN.md 4.8): allele 1 = REF, allele 2 = the one ALT; a record without ALT is written with allele 2 = "."
(which no score row names).  Unphased: per sample b0 = P(hom allele 1), b1 = P(het); phased: h0, h1 = P(haplotype
carries allele 1).  A missing sample has ploidy byte 0x82 and zero probabilities.  The dosage numerator the engine
derives is k = 510 - 2*b0 - b1 (unphased) or 510 - h0 - h1 (phased), 0xFFFF for a missing sample."""
import os
import struct
import zlib

import numpy as np

MISSING = 0xFFFF


def numerators(probs, phased, missing):
    """uint16 k per sample from the stored probability bytes probs[n, 2]."""
    p = np.asarray(probs, np.int64)
    k = 510 - p[:, 0] - p[:, 1] if phased else 510 - 2 * p[:, 0] - p[:, 1]
    return np.where(np.asarray(missing, bool), MISSING, k).astype(np.uint16)


def random_probs(rng, n, phased, miss_rate=0.05, hard_rate=0.2):
    """Random fractional 8-bit probabilities (hard calls mixed in) -> (probs uint8[n, 2], missing bool[n])."""
    if phased:
        probs = rng.integers(0, 256, size=(n, 2))
        hard = rng.random((n, 2)) < hard_rate
        probs = np.where(hard, 255 * rng.integers(0, 2, size=(n, 2)), probs)
    else:
        b0 = rng.integers(0, 256, size=n)
        b1 = (rng.random(n) * (256 - b0)).astype(np.int64)          # b0 + b1 <= 255
        probs = np.stack([b0, b1], axis=1)
        hard = rng.random(n) < hard_rate
        probs[hard] = np.array([[255, 0], [0, 255], [0, 0]])[rng.integers(0, 3, size=int(hard.sum()))]
    missing = rng.random(n) < miss_rate
    probs[missing] = 0
    return probs.astype(np.uint8), missing


def hard_call_probs(gt_row, n, phased):
    """Probabilities of the hard calls of one biallelic diploid int8 GT row (raw BCF values); a half call is missing."""
    a = (np.asarray(gt_row)[:2 * n].reshape(n, 2).astype(np.int32) >> 1) - 1        # allele index, -1 missing
    missing = (a < 0).any(axis=1)
    if phased:
        probs = np.where(a == 0, 255, 0)
    else:
        n_alt = (a == 1).sum(axis=1)
        probs = np.stack([np.where(n_alt == 0, 255, 0), np.where(n_alt == 1, 255, 0)], axis=1)
    probs[missing] = 0
    return probs.astype(np.uint8), missing


def genotype_block(n, probs, missing, phased, K=2, bits=8, pmin=2, pmax=2, n_stored=None):
    """Uncompressed probability data of one variant (layout 2)."""
    ploidy = np.where(np.asarray(missing, bool), 0x82, 2).astype(np.uint8)
    head = struct.pack("<IHBB", n if n_stored is None else n_stored, K, pmin, pmax)
    return head + ploidy.tobytes() + struct.pack("<BB", int(bool(phased)), bits) + np.asarray(probs, np.uint8).tobytes()


def _s16(s):
    b = s.encode()
    return struct.pack("<H", len(b)) + b


def write_bgen(path, samples, variants, compression="zlib", embed_ids=True, sample_file=True, layout=2, free=b"free",
               header_len=None, offset_delta=0, n_variants=None):
    """variants: dicts with contig, pos, alleles, and either `block` (raw probability data) or probs / missing / phased.
    compression: "none", "zlib" or "zstd" (the flag only: the blocks are then zlib, for the refusal test).  Without
    embedded identifiers a sibling X.sample is written when sample_file is true.  Returns path."""
    n = len(samples)
    comp = {"none": 0, "zlib": 1, "zstd": 2}[compression]
    flags = comp | (layout << 2) | (0x80000000 if embed_ids else 0)
    LH = 20 + len(free) if header_len is None else header_len
    sblock = b""
    if embed_ids:
        ids = b"".join(_s16(s) for s in samples)
        sblock = struct.pack("<II", 8 + len(ids), n) + ids
    offset = LH + len(sblock) + offset_delta
    out = [struct.pack("<IIII", offset, LH, len(variants) if n_variants is None else n_variants, n), b"bgen", free,
           struct.pack("<I", flags), sblock]
    for k, v in enumerate(variants):
        block = v.get("block")
        if block is None:
            block = genotype_block(n, v["probs"], v["missing"], v["phased"])
        if comp:
            z = zlib.compress(block, 6)
            g = struct.pack("<II", len(z) + 4, len(block)) + z
        else:
            g = struct.pack("<I", len(block)) + block
        alleles = v["alleles"]
        out.append(_s16(v.get("id", f"v{k}")) + _s16(v.get("rsid", f"rs{k}")) + _s16(v["contig"]) +
                   struct.pack("<IH", v["pos"], len(alleles)) +
                   b"".join(struct.pack("<I", len(a)) + a.encode() for a in alleles) + g)
    with open(path, "wb") as fh:
        fh.write(b"".join(out))
    if not embed_ids and sample_file:
        with open(path[:-5] + ".sample" if path.endswith(".bgen") else path + ".sample", "w") as fh:
            fh.write("ID_1 ID_2 missing\n0 0 0\n")
            fh.write("".join(f"F{i} {s} 0\n" for i, s in enumerate(samples)))
    return path


def records_to_variants(records, n, rng=None):
    """Split biallelic diploid records (util_plink.split_records) -> hard-call BGEN variants; with rng, some phased."""
    out = []
    for r in records:
        phased = bool(rng is not None and rng.random() < 0.4)
        probs, missing = hard_call_probs(np.asarray(r["gt"]).reshape(-1), n, phased)
        out.append(dict(contig=r["contig"], pos=r["pos"], alleles=[r["ref"], r["alts"][0] if r["alts"] else "."],
                        probs=probs, missing=missing, phased=phased))
    return out


def make_split_dataset(tmp, rng, n=300, V=120, compression="zlib", embed_ids=True, **kw):
    """util_plink.make_split_dataset's cohort (biallelic, all PASS; VCF, BCF and PLINK fileset), also as a hard-call
    BGEN file: d["bgen"]."""
    from util_plink import make_split_dataset as plink_split
    d = plink_split(tmp, rng, n=n, V=V, **kw)
    d["bgen"] = write_bgen(os.path.join(tmp, "split.bgen"), d["samples"], records_to_variants(d["records"], n, rng),
                           compression=compression, embed_ids=embed_ids)
    return d


# ---- reference restatement of scoring on dosage rows (DESIGN.md 4.8) -------------------------------------------------

LOCUS = {"ps": 0, "homref": 1, "fail": 2, "ignore": 3}
MISSING_POL = {"homref": 0, "ignore": 1}
SAMPLE = {"ps": 0, "homref": 1, "fail": 2, "int_ps": 3, "int_fail": 4}
LOCUS_DTYPE = np.dtype([("klass", "<i4"), ("used", "<i4"), ("eaidx", "<i4"), ("reserved", "<i4"),
                        ("ngt", "<i8"), ("nmiss", "<i8"), ("neff", "<i8"), ("imputed", "<f8")], align=True)


def reference_scores(k, n, rows, offset=0.0, imp_locus="ps", imp_missing="homref", imp_sample="int_ps", maxmis=0.05,
                     mincs=100):
    """computePolygenicScores (src/nimpress.nim:592-649) on dosage rows k[V, >= n] (uint16, 255 x the ALT dosage, above
    510 missing), restated per score row in the reference's order with numpy's correctly rounded fp64 operations:
    raw dosage fl(k'/255) (k' = 510 - k for eaidx 0), NaN when missing; tallies nmiss and neff_num = sum k' as integers,
    neff = fl(neff_num / 255); the --maxmis rule, imputeLocusDosages and imputeSampleDosages as the reference has them;
    scores = fl(scores + fl(dosage * beta)) row after row; then / fl(nloci * 2) and + offset.  The record's neff is
    neff_num.  rows: records of the npc_row layout (gt_row, eaidx, beta, eaf, ref_is_ea, kind)."""
    k = np.asarray(k)
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
            row = k[r["gt_row"], :n].astype(np.int64)
            miss = row > 510
            kk = np.where(r["eaidx"] == 0, 510 - row, row)
            nmiss = int(miss.sum())
            num = int(kk[~miss].sum())
            ngt = n - nmiss
            rec["ngt"], rec["nmiss"], rec["neff"] = ngt, nmiss, num
            neff = float(num) / 255.0
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
                dos = np.where(miss, v, kk.astype(np.float64) / 255.0)
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
