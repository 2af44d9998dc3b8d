"""Tests-only: PLINK 1 binary filesets (.bed/.bim/.fam) written with numpy from the cohorts the VCF/BCF writers take.

Conventions (DESIGN.md 4.7): A2 = REF (.bim column 6), A1 = the one ALT (column 5, "0" when there is none); a
multi-allelic site is split into one biallelic line per ALT as `bcftools norm -m-` does (the other ALTs' alleles
become REF); per sample a 2-bit code, low bits first: 00 hom A1, 01 missing, 10 het, 11 hom A2.  A half call ("./a")
is missing, as the reference treats it."""
import os

import numpy as np

from util_bcf import write_bcf, write_vcf

BED_MAGIC = bytes([0x6C, 0x1B, 0x01])


def bed_codes(gt_row, n):
    """2-bit codes of one biallelic diploid int8 GT row (raw BCF values (allele+1)<<1|phase)."""
    a = (np.asarray(gt_row)[:2 * n].reshape(n, 2).astype(np.int32) >> 1) - 1        # allele index, -1 missing
    miss = (a < 0).any(axis=1)
    n_alt = (a == 1).sum(axis=1)
    code = np.select([miss, n_alt == 2, n_alt == 1], [1, 0, 2], default=3)
    return code.astype(np.uint8)


def pack_codes(codes, pad_code=0):
    """codes[V, n] (0..3) -> .bed rows uint8[V, ceil(n/4)]; the padding codes of the last byte are pad_code."""
    codes = np.atleast_2d(codes)
    V, n = codes.shape
    nb = (n + 3) // 4
    full = np.full((V, nb * 4), pad_code & 3, np.uint8)
    full[:, :n] = codes
    q = full.reshape(V, nb, 4).astype(np.uint8)
    return (q[..., 0] | (q[..., 1] << 2) | (q[..., 2] << 4) | (q[..., 3] << 6)).astype(np.uint8)


def pack_cohort(gt, n, pad_code=0):
    """An int8 biallelic diploid cohort gt[V, cols] -> .bed rows."""
    return pack_codes(np.stack([bed_codes(r, n) for r in gt]) if len(gt) else np.zeros((0, n), np.uint8), pad_code)


def split_records(records):
    """`bcftools norm -m-`: one record per ALT, in ALT order; on line j the alleles of other ALTs become REF.  FILTER is
    set to PASS and INFO dropped, since a .bim carries neither (a PLINK fileset is the all-PASS VCF's equivalent)."""
    out = []
    for r in records:
        alts = r["alts"] or [None]
        for j, alt in enumerate(alts, start=1):
            g = np.asarray(r["gt"]).astype(np.int64)
            a = (g >> 1) - 1
            phase = g & 1
            na = np.where(a < 0, -1, np.where(a == j, 1, 0))
            raw = np.where(na < 0, phase, ((na + 1) << 1) | phase)
            out.append(dict(contig=r["contig"], pos=r["pos"], ref=r["ref"], alts=[alt] if alt else [], filter="PASS",
                            gt=raw.astype(r["gt"].dtype)))
    return out


def write_plink(prefix, samples, records, pad_code=0):
    """prefix.bed / .bim / .fam of biallelic diploid records (dicts as util_bcf takes them); returns prefix.bed."""
    n = len(samples)
    with open(prefix + ".fam", "w") as fh:
        for s in samples:
            fh.write(f"{s} {s} 0 0 0 -9\n")
    with open(prefix + ".bim", "w") as fh:
        for k, r in enumerate(records):
            a1 = r["alts"][0] if r["alts"] else "0"
            fh.write(f"{r['contig']}\tv{k}\t0\t{r['pos']}\t{a1}\t{r['ref']}\n")
    rows = pack_codes(np.stack([bed_codes(r["gt"].reshape(-1), n) for r in records]), pad_code) if records else np.zeros((0, (n + 3) // 4), np.uint8)
    with open(prefix + ".bed", "wb") as fh:
        fh.write(BED_MAGIC)
        fh.write(rows.tobytes())
    return prefix + ".bed"


def make_split_dataset(tmp, rng, n=300, V=120, **kw):
    """make_dataset's cohort and score file, its records split biallelic and all-PASS, written three ways: the
    equivalent VCF (BGZF), BCF and PLINK fileset.  Returns make_dataset's dict with vcf / bcf / plink replaced."""
    from util_files import make_dataset
    d = make_dataset(tmp, rng, n=n, V=V, **kw)
    recs = split_records(d["records"])
    contigs = list(dict.fromkeys(r["contig"] for r in d["records"]))
    d["records"] = recs
    d["vcf"] = os.path.join(tmp, "split.vcf.gz")
    write_vcf(d["vcf"], d["samples"], recs, contigs=contigs, compress="bgzf")
    d["bcf"] = os.path.join(tmp, "split.bcf")
    write_bcf(d["bcf"], d["samples"], recs, contigs=contigs, compress="bgzf")
    d["plink"] = write_plink(os.path.join(tmp, "split"), d["samples"], recs)
    return d
