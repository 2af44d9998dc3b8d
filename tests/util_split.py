"""Tests-only: one cohort's records written as several genotype files (per contig, or in chunks with a site repeated
across a chunk boundary) and as the one file that is their concatenation (DESIGN.md 4.12), for every kind the engine
reads."""
import os

import numpy as np

from util_bcf import write_bcf, write_vcf
from util_bgen import records_to_variants, write_bgen
from util_bgen_bits import records_to_variants_bits
from util_pl import write_bcf_pl, write_vcf_pl
from util_plink import write_plink

CONTIGS = ["1", "2", "X"]
EXT = dict(vcf=".vcf.gz", ds=".vcf.gz", bcf=".bcf", bed=".bed", bgen8=".bgen", bgen16=".bgen", bgen_last16=".bgen",
           pl_vcf=".vcf.gz", pl_bcf=".bcf")


def by_contig(records):
    """One part per contig, in order of first appearance (a contig's records keep their order)."""
    parts = {}
    for r in records:
        parts.setdefault(r["contig"], []).append(r)
    return list(parts.values())


def chunks(records, k, dup=True):
    """k contiguous parts; with dup, each part after the first starts with a copy of the previous part's last record
    whose genotypes are rolled by one sample: the same site in two files, where the earlier one must win."""
    bounds = np.linspace(0, len(records), k + 1).astype(int)
    parts = [list(records[a:b]) for a, b in zip(bounds[:-1], bounds[1:])]
    if dup:
        for i in range(1, k):
            r = dict(parts[i - 1][-1])
            for f in ("gt", "ds", "pl", "plcnt", "plmiss", "plpartial"):
                if f in r:
                    r[f] = np.roll(np.asarray(r[f]), 1, axis=0)
            parts[i] = [r] + parts[i]
    return parts


def _write(kind, path, samples, records, variants=None):
    if kind in ("vcf", "ds"):
        write_vcf(path, samples, records, contigs=CONTIGS, filters=("FAIL", "LowQ"), compress="bgzf")
    elif kind == "bcf":
        write_bcf(path, samples, records, contigs=CONTIGS, filters=("FAIL", "LowQ"), compress="bgzf")
    elif kind == "bed":
        return write_plink(path[:-4], samples, records)
    elif kind.startswith("bgen"):
        write_bgen(path, samples, variants)
    elif kind == "pl_vcf":
        write_vcf_pl(path, samples, records, CONTIGS)
    elif kind == "pl_bcf":
        write_bcf_pl(path, samples, records, CONTIGS)
    return path


def write_split(kind, tmp, stem, samples, parts, seed=0, part_samples=None, kinds=None):
    """Writes every part as a file of `kind` (kinds: one kind per part, e.g. VCF text and BCF mixed) and the
    concatenation of all parts as one file of kind kinds[0] or `kind`.  part_samples[i]: the samples of part i
    (their records are then subsetted to them by the caller).  bgen_last16: 8-bit BGEN, 16-bit in the last part only.
    Returns (part paths, concatenated path)."""
    n = len(samples)
    kinds = kinds or [kind] * len(parts)
    variants = [None] * len(parts)
    if kind.startswith("bgen"):                        # one phasing draw over all records, sliced per part
        rng = np.random.default_rng(seed)
        for i, p in enumerate(parts):
            ns = len(part_samples[i]) if part_samples else n
            if kind == "bgen8":
                variants[i] = records_to_variants(p, ns, rng)
            else:
                bits = 16 if kind == "bgen16" or i == len(parts) - 1 else 8
                variants[i] = records_to_variants_bits(p, ns, bits, rng)
    paths = [_write(kinds[i], os.path.join(tmp, f"{stem}{i}{EXT[kinds[i]]}"), part_samples[i] if part_samples else samples,
                    p, variants[i]) for i, p in enumerate(parts)]
    cat = None
    if not part_samples:
        cat = _write(kinds[0], os.path.join(tmp, f"{stem}_all{EXT[kinds[0]]}"), samples, [r for p in parts for r in p],
                     [v for vs in variants for v in vs] if kind.startswith("bgen") else None)
    return paths, cat
