"""Tests-only: FORMAT/PL rows (DESIGN.md 4.10).  The word packer, VCF text and BCF writers of records with GT and PL, and
reference_scores_pl, a numpy restatement of scoring on PL rows in the reference's order.

A sample's PL values come as (pl int64[n, 3], cnt[n] in {2, 3}, missing[n]): a diploid sample has 3 values (0/0, 0/1,
1/1), a haploid one 2 (pl[:, 2] unused).  Its word in an NPC_GT_PL row: m = the smallest PL, j = the index of its first
occurrence, a and b = the other genotypes' PL - m in genotype order, saturated at 4095 (b = 0 for a haploid sample):
a | b << 12 | j << 24 | ploidy << 26, 0xFFFFFFFF for a missing sample."""
import decimal
import functools
import struct

import numpy as np

from util_bcf import _desc, _typed_int, _typed_str, _typed_ints, bgzf_compress
from util_bgen import LOCUS, LOCUS_DTYPE, MISSING_POL, SAMPLE

MISSING_PL = 0xFFFFFFFF
TN = 3237                                        # T[x] = 0 from here on


def weight(x, digits=60):
    """fl(10^(-x/10)) correctly rounded: Python decimal at `digits` significant digits, then one rounding to double."""
    ctx = decimal.Context(prec=digits, Emin=-10000, Emax=10000)
    return float(ctx.power(decimal.Decimal(10), ctx.divide(decimal.Decimal(-int(x)), decimal.Decimal(10))))


@functools.lru_cache(None)
def weight_table(n=4096):
    return np.array([weight(x) if x < TN else 0.0 for x in range(n)], np.float64)


def pack_words(pl, cnt, missing):
    """Per sample (pl[n, 3], cnt[n] = 2 or 3, missing[n]) -> uint32 words of an NPC_GT_PL row."""
    pl = np.asarray(pl, np.int64).reshape(-1, 3)
    cnt = np.asarray(cnt, np.int64)
    v = np.where(np.arange(3) < cnt[:, None], pl, np.iinfo(np.int64).max)
    j = np.argmin(v, axis=1)                                           # first occurrence of the minimum
    m = v[np.arange(len(v)), j]
    x = np.minimum(v - m[:, None], 4095)
    other = np.array([[1, 2], [0, 2], [0, 1]])[j]                      # the genotypes other than j, in order
    a = x[np.arange(len(v)), other[:, 0]]
    b = np.where(cnt == 3, x[np.arange(len(v)), other[:, 1]], 0)
    w = a | b << 12 | j << 24 | (cnt - 1) << 26
    return np.where(np.asarray(missing, bool), MISSING_PL, w).astype(np.uint32)


def random_pl(rng, n, haploid_rate=0.1, miss_rate=0.03, hi=6000):
    """Random PL values -> (pl int64[n, 3], cnt[n], missing[n]): a mix of decisive samples (every other PL >= 3237 above
    the minimum, or hi / 2 when hi <= 3237), uninformative ones (all equal), moderate values, ties and values past the
    4095 saturation."""
    cnt = np.where(rng.random(n) < haploid_rate, 2, 3)
    kind = rng.integers(0, 5, size=n)
    base = rng.integers(0, 40, size=(n, 1))
    pl = np.where(kind[:, None] == 0, rng.integers(0, 60, size=(n, 3)),                       # moderate
         np.where(kind[:, None] == 1, rng.integers(0, hi, size=(n, 3)),                       # anything, often saturated
         np.where(kind[:, None] == 2, np.repeat(base, 3, axis=1),                             # uninformative
         np.where(kind[:, None] == 3, rng.integers(0, 3, size=(n, 3)) * 7,                    # ties
                  rng.integers(TN if hi > TN else hi // 2, hi, size=(n, 3))))))            # decisive (one set to 0 below)
    g = rng.integers(0, 3, size=n)
    g = np.where(cnt == 2, g % 2, g)
    pl[np.arange(n), g] = np.where(kind == 4, 0, pl[np.arange(n), g])
    pl[:, 2] = np.where(cnt == 2, 0, pl[:, 2])
    missing = rng.random(n) < miss_rate
    return pl, cnt, missing


def decisive_pl(alleles, ploidy, rng):
    """Hard calls (alleles[n, 2] with -1 missing, ploidy[n]) as decisive PLs: 0 for the called genotype, every other at
    least 3237 above it (some saturated) -> (pl, cnt, missing)."""
    a = np.asarray(alleles, np.int64)
    p = np.asarray(ploidy, np.int64)
    n = len(p)
    missing = (a[:, 0] < 0) | ((p == 2) & (a[:, 1] < 0))
    g = np.where(p == 2, (a == 1).sum(axis=1), (a[:, 0] == 1).astype(np.int64))
    pl = rng.integers(TN, 9000, size=(n, 3)) + rng.integers(0, 50, size=(n, 1))
    base = rng.integers(0, 30, size=n)
    pl = pl + base[:, None]
    pl[np.arange(n), np.clip(g, 0, 2)] = base
    pl[:, 2] = np.where(p == 1, 0, pl[:, 2])
    return pl, np.where(p == 1, 2, 3), missing


# ---- the posterior dosage and the tally order (DESIGN.md 4.10) ------------------------------------------------------


def dosages(words, eaf, eaidx, T=None):
    """One row's words -> (d float64[n], called bool[n]) with numpy's correctly rounded fp64 operations."""
    T = weight_table() if T is None else T
    w = np.asarray(words, np.uint32).astype(np.int64)
    a, b, j, P = w & 0xFFF, (w >> 12) & 0xFFF, (w >> 24) & 3, (w >> 26) & 3
    ok = ((w >> 31) == 0) & ((P == 1) | (P == 2)) & (j <= P)
    p = float(eaf)
    q = 1.0 - p
    pi = np.array([q * q, 2.0 * (p * q), p * p])
    alt = eaidx != 0
    g = pi if alt else pi[::-1]
    h = np.array([q, p]) if alt else np.array([p, q])
    wa, wb = T[np.minimum(a, TN)], T[np.minimum(b, TN)]
    w0 = np.where(j == 0, 1.0, wa)
    w1 = np.where(j == 0, wa, np.where(j == 1, 1.0, wb))
    w2 = np.where(j == 2, 1.0, wb)
    dip = P == 2
    u0 = np.where(dip, g[0], h[0]) * w0
    u1 = np.where(dip, g[1], h[1]) * w1
    u2 = np.where(dip, g[2] * w2, 0.0)
    den = (u0 + u1) + u2
    num = np.where(dip, u1 + 2.0 * (u2 if alt else u0), u1 if alt else u0)
    with np.errstate(divide="ignore", invalid="ignore"):
        d = num / den
    called = ok & (den > 0) & (0.0 <= p <= 1.0)
    return d, called


def ds_order_sum(d, called):
    """The fp64 sum of the called d in the order of FORMAT/DS rows: chunks of 8 samples left to right from +0.0, the
    butterfly v[i] = v[i] + v[i ^ o] (o = 16, 8, 4, 2, 1) over the 32 chunks of a block of 256 (lane 0's value), block
    sums left to right."""
    n = len(d)
    nb = -(-n // 256)
    x = np.zeros(nb * 256)
    x[:n] = np.where(called, d, 0.0)
    c = np.zeros(nb * 256, bool)
    c[:n] = called
    x = x.reshape(nb, 32, 8)
    c = c.reshape(nb, 32, 8)
    v = np.zeros((nb, 32))
    for k in range(8):
        v = np.where(c[:, :, k], v + x[:, :, k], v)
    lanes = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = v + v[:, lanes ^ o]
    total = 0.0
    for s in v[:, 0]:
        total = total + float(s)
    return total


def reference_scores_pl(words, n, rows, offset=0.0, imp_locus="ps", imp_missing="homref", imp_sample="int_ps", maxmis=0.05,
                        mincs=100):
    """computePolygenicScores (src/nimpress.nim:592-649) on PL rows words[V, >= n], restated per score row in the
    reference's order as util_bgen.reference_scores does: per sample the posterior expected dosage d (dosages), missing
    when not called; nmiss an integer, neff = ds_order_sum; the --maxmis rule, imputeLocusDosages and
    imputeSampleDosages as the reference has them; scores = fl(scores + fl(dosage * beta)) row after row; then
    / fl(nloci * 2) and + offset.  The record's neff holds the bits of neff."""
    words = np.asarray(words, np.uint32)
    scores = np.zeros(n, np.float64)
    loci = np.zeros(len(rows), dtype=LOCUS_DTYPE)
    nloci = 0

    def locus_value(r):
        m = LOCUS[imp_locus]
        if m == 3:
            return None
        return float(r["eaf"]) * 2.0 if m == 0 else (2.0 if r["ref_is_ea"] else 0.0) if m == 1 else float("nan")

    for i, r in enumerate(rows):
        rec = loci[i]
        rec["eaidx"], rec["ngt"], rec["nmiss"], rec["neff"], rec["imputed"] = -1, -1, -1, -1, np.nan
        dos = None
        kind = int(r["kind"])
        if kind == 1:
            rec["klass"] = 1
            v = locus_value(r)
        elif kind == 3:
            rec["klass"], rec["eaidx"] = 3, r["eaidx"]
            v = locus_value(r)
        elif kind == 2 or r["gt_row"] < 0:
            rec["klass"] = 2
            v = (2.0 if r["ref_is_ea"] else 0.0) if MISSING_POL[imp_missing] == 0 else None
        else:
            rec["eaidx"] = r["eaidx"]
            d, called = dosages(words[r["gt_row"], :n], r["eaf"], int(r["eaidx"]))
            nmiss = int((~called).sum())
            neff = ds_order_sum(d, called)
            ngt = n - nmiss
            rec["ngt"], rec["nmiss"] = ngt, nmiss
            rec["neff"] = np.float64(neff).view(np.int64)
            if float(nmiss) / float(n) > maxmis:
                rec["klass"] = 4
                v = locus_value(r)
            else:
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
                dos = np.where(called, d, v)
        rec["used"] = v is not None
        if v is None:
            continue
        rec["imputed"] = v
        if dos is None:
            dos = np.full(n, v, np.float64)
        scores = scores + dos * float(r["beta"])
        nloci += 1
    with np.errstate(divide="ignore", invalid="ignore"):
        scores = scores / (float(nloci) * 2.0) + offset
    return dict(scores=scores, loci=loci, nloci=nloci)


# ---- files ------------------------------------------------------------------------------------------------------------


def pl_text(pl, cnt, missing, partial=False):
    """One sample's PL sub-field: "." when missing (or, with partial, one value written as ".")."""
    if missing and not partial:
        return "."
    vals = [str(int(x)) for x in pl[:cnt]]
    if missing:
        vals[1] = "."
    return ",".join(vals)


def with_pl(records, n, rng, decisive=False, haploid_rate=0.1, miss_rate=0.03, hi=6000):
    """Records with GT (dict as util_bcf.write_vcf takes) -> the same with pl, plcnt, plmiss and plpartial (missing
    samples written with one "." value).  decisive: the PLs of the record's hard calls (vector_end second allele =
    haploid), else random_pl."""
    out = []
    for r in records:
        g = np.asarray(r["gt"]).reshape(n, -1).astype(np.int64)
        if decisive:
            ploidy = np.where(g[:, 1] == -127, 1, 2) if g.shape[1] > 1 else np.ones(n, np.int64)
            a = np.where((g & ~1) == 0, -1, (g >> 1) - 1)
            if g.shape[1] > 1:
                a[:, 1] = np.where(ploidy == 1, 0, a[:, 1])
            pl, cnt, miss = decisive_pl(a, ploidy, rng)
        else:
            pl, cnt, miss = random_pl(rng, n, haploid_rate, miss_rate, hi)
        out.append(dict(r, pl=pl, plcnt=cnt, plmiss=miss, plpartial=miss & (rng.random(n) < 0.5)))
    return out


def write_vcf_pl(path, samples, records, contigs, compress="bgzf", with_gt=True):
    """VCF text with FORMAT GT:PL (PL only without with_gt); a record without "pl" has GT alone."""
    from util_bcf import gt_text
    lines = ["##fileformat=VCFv4.2", '##FILTER=<ID=FAIL,Description="x">', '##FILTER=<ID=LowQ,Description="x">']
    lines += [f"##contig=<ID={c}>" for c in contigs]
    lines += ['##INFO=<ID=END,Number=1,Type=Integer,Description="End">',
              '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
              '##FORMAT=<ID=PL,Number=G,Type=Integer,Description="Phred-scaled genotype likelihoods">']
    lines.append("\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + list(samples)))
    for r in records:
        g = np.asarray(r["gt"])
        cols = [r["contig"], str(r["pos"]), ".", r["ref"], ",".join(r["alts"]) if r["alts"] else ".", ".", r["filter"], r.get("info", ".")]
        gts = [gt_text(g[i], g.dtype.itemsize) for i in range(len(samples))]
        if "pl" not in r:
            cols.append("GT")
            cols += gts
        else:
            pls = [r["pltext"][i] if "pltext" in r else pl_text(r["pl"][i], r["plcnt"][i], r["plmiss"][i], r["plpartial"][i])
                   for i in range(len(samples))]
            cols.append("GT:PL" if with_gt else "PL")
            cols += [f"{a}:{b}" for a, b in zip(gts, pls)] if with_gt else pls
        lines.append("\t".join(cols))
    data = ("\n".join(lines) + "\n").encode()
    if compress == "bgzf":
        data = bgzf_compress(data)
    open(path, "wb").write(data)


def write_bcf_pl(path, samples, records, contigs, pl_width=None):
    """BCF2.2 with FORMAT GT then PL as typed integers of pl_width bytes (1, 2 or 4; None: the narrowest that holds the
    record's values), missing = MIN and vector_end = MIN + 1 of the width: a haploid sample is two values then
    vector_end, a missing one "." then vector_end (or one value missing, with plpartial)."""
    ids = ["PASS", "FAIL", "LowQ", "END", "GT", "PL"]
    idx = {s: i for i, s in enumerate(ids)}
    cidx = {c: i for i, c in enumerate(contigs)}
    lines = ["##fileformat=VCFv4.2", '##FILTER=<ID=PASS,Description="All filters passed">', '##FILTER=<ID=FAIL,Description="x">',
             '##FILTER=<ID=LowQ,Description="x">']
    lines += [f"##contig=<ID={c}>" for c in contigs]
    lines += ['##INFO=<ID=END,Number=1,Type=Integer,Description="End">',
              '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
              '##FORMAT=<ID=PL,Number=G,Type=Integer,Description="Phred-scaled genotype likelihoods">']
    lines.append("\t".join(["#CHROM", "POS", "ID", "REF", "ALT", "QUAL", "FILTER", "INFO", "FORMAT"] + list(samples)))
    text = ("\n".join(lines) + "\n").encode() + b"\0"
    out = bytearray(b"BCF\2\2" + struct.pack("<I", len(text)) + text)
    n = len(samples)
    for r in records:
        g = np.ascontiguousarray(r["gt"])
        alleles = [r["ref"]] + list(r["alts"])
        flt = [] if r["filter"] == "." else [idx[f] for f in r["filter"].split(";")]
        rlen, info, n_info = len(r["ref"]), b"", 0
        if r.get("info", ".").startswith("END="):
            end = int(r["info"][4:])
            rlen, info, n_info = end - r["pos"] + 1, _typed_int(idx["END"]) + _typed_ints([end]), 1
        shared = struct.pack("<iiif", cidx[r["contig"]], r["pos"] - 1, rlen, float("nan"))
        n_fmt = 2 if "pl" in r else 1
        shared += struct.pack("<II", (len(alleles) << 16) | n_info, (n_fmt << 24) | n)
        shared += _desc(0, 7)
        for a in alleles:
            shared += _typed_str(a)
        shared += _typed_ints(flt) + info
        t = {1: 1, 2: 2, 4: 3}[g.dtype.itemsize]
        indiv = _typed_int(idx["GT"]) + _desc(g.shape[1], t) + g.tobytes()
        if "pl" in r:
            pl = np.asarray(r["pl"], np.int64)
            L = int(max(2, np.max(r["plcnt"])))
            width = pl_width or (1 if pl.max() <= 127 else 2 if pl.max() <= 32767 else 4)
            dt = {1: np.int8, 2: np.int16, 4: np.int32}[width]
            lo = int(np.iinfo(dt).min)
            v = np.full((n, L), lo + 1, np.int64)                               # vector_end
            for i in range(n):
                c = int(r["plcnt"][i])
                if r["plmiss"][i] and not r["plpartial"][i]:
                    v[i, 0] = lo
                else:
                    v[i, :c] = pl[i, :c]
                    if r["plmiss"][i]:
                        v[i, 1] = lo
            assert v.max() <= np.iinfo(dt).max
            indiv += _typed_int(idx["PL"]) + _desc(L, {1: 1, 2: 2, 4: 3}[width]) + v.astype(dt).tobytes()
        out += struct.pack("<II", len(shared), len(indiv)) + shared + indiv
    open(path, "wb").write(bgzf_compress(bytes(out)))
