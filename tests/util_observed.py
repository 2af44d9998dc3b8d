"""The observed counts (DESIGN.md 4.13) restated two ways: per sample, the score rows of class OK (klass 0, used) at which
the sample has a called genotype -- one the layout's tally does not count in nmiss.

- From the CPU oracle's own loop (oracle_observed_*): each score row is scored on its own with beta 1 and
  --imp-sample fail.  The reference's getRawDosages gives a missing sample a NaN dosage, which `fail` keeps, so at an OK
  row a sample's score is NaN exactly when its genotype was not called.  Nothing here decodes a genotype.
- From numpy predicates of each layout's tally (called_*), for the layouts the oracle does not read."""
import os

import numpy as np

import orc

from util_pl import dosages


def called_gt(row, n, ploidy, dtype):
    """GT row of any width and ploidy: getRawDosages gives a non-NaN dosage -- no allele before a vector_end decodes to -1
    (a sample of missing / vector_end sentinels only is called, dosage 0)."""
    info = np.iinfo(dtype)
    a = np.asarray(row).view(dtype)[:n * ploidy].reshape(n, ploidy).astype(np.int64)
    ended, missing = np.zeros(n, bool), np.zeros(n, bool)
    for k in range(ploidy):
        raw = a[:, k]
        ended |= raw == info.min + 1
        val = np.where(raw < 0, raw, (raw >> 1) - 1)
        missing |= ~ended & (raw != info.min) & (val == -1)
    return ~missing


def called_bed(row, n):
    b = np.asarray(row, np.uint8)
    s = np.arange(n)
    return ((b[s >> 2] >> (2 * (s & 3))) & 3) != 1


def called_dose255(row, n):
    return np.asarray(row, np.uint8).view(np.uint16)[:n] <= 510


def called_dose32(row, n):
    r = np.asarray(row, np.uint8)
    D = int(r[:4].view(np.uint32)[0])
    w = r[16:16 + 4 * n].view(np.uint32).astype(np.int64)
    p, k = (w >> 24) & 3, w & 0xFFFFFF
    return ((w >> 31) == 0) & ((p == 1) | (p == 2)) & (k <= p * D)


def called_ds(row, n):
    b = np.asarray(row, np.uint8).view(np.uint32)[:n].astype(np.int64)
    return ~((b == 0x7F800001) | (b == 0x7F800002) | ((b & 0x7FFFFFFF) > 0x7F800000))


def called_pl(row, n, eaf, eaidx):
    return dosages(np.asarray(row, np.uint8).view(np.uint32)[:n], eaf, eaidx)[1]


def observed(called_of, rows, loci, n):
    """called_of(npc_row) -> bool[n] of the row's slab row; rows / loci: one definition's rows and records, in order."""
    out = np.zeros(n, np.int64)
    for r, rec in zip(rows, loci):
        if rec["klass"] == 0 and rec["used"] and r["kind"] == 0 and r["gt_row"] >= 0:
            out += called_of(r)
    return out


def ngt_total(loci):
    """Sum of ngt over the OK records: what the observed counts add up to."""
    ok = (loci["klass"] == 0) & (loci["used"] != 0)
    return int(loci["ngt"][ok].sum())


def _oracle_called(res):
    """(row is OK, called bool[n]) from the oracle's run of one score row with beta 1 and --imp-sample fail."""
    rec = res["loci"][0]
    return bool(rec["klass"] == orc.CLASS_OK and rec["used"]), ~np.isnan(res["scores"])


def oracle_observed_matrix(gt, n, ploidy, rows, **kw):
    """orc_score_matrix (GT rows of int8 / int16 / int32 gt[V, >= n * ploidy], or float32 FORMAT/DS rows), one score row
    at a time.  kw: the policy (maxmis, mincs, ...); imp_sample is set to fail."""
    out = np.zeros(n, np.int64)
    for r in np.ascontiguousarray(rows, dtype=orc.ROW_DTYPE):
        one = np.array([r], dtype=orc.ROW_DTYPE)
        one["beta"] = 1.0
        ok, called = _oracle_called(orc.score_matrix(gt, n, ploidy, one, **dict(kw, imp_sample="fail")))
        if ok:
            out += called
    return out


def oracle_observed_files(score, vcf, tmp, bed=None, **kw):
    """orc_compute_scores_files over the score file one entry at a time (its own file under tmp, beta 1, offset 0)."""
    lines = open(score).read().split("\n")
    head, ents = lines[:5], [l for l in lines[5:] if l.strip()]
    out = None
    for j, e in enumerate(ents):
        f = e.rstrip().split("\t")
        f[4] = "1"
        path = os.path.join(str(tmp), f"observed_row{j}.score")
        with open(path, "w") as fh:
            fh.write("\n".join(head[:4] + ["0"] + ["\t".join(f)]) + "\n")
        ok, called = _oracle_called(orc.compute_scores_files(path, vcf, bed, **dict(kw, imp_sample="fail")))
        out = np.zeros(len(called), np.int64) if out is None else out
        if ok:
            out += called
    return out
