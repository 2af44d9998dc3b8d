"""Python mirror of the reference's public procs for the scoring path, over libnimpress_host.so
(C++ host + CUDA engine).  Names, argument order and meaning follow src/nimpress.nim so that
tests/test_set1.py reads like the reference's tests/test_set1.nim:

    scoreFile = ScoreFile(); open_score(scoreFile, "tests/set1.score")
    genotypeVcf = VCF();     open_vcf(genotypeVcf, "tests/set1.vcf.gz")
    coveredBed = GenomeIntervals(); loadBedIntervals(coveredBed, "tests/set1.bed")
    scores = []
    computePolygenicScores(scores, scoreFile, genotypeVcf, False, coveredBed,
                           ImputeMethodLocus.ps, ImputeMethodMissing.homref, ImputeMethodSample.fail,
                           maxMissingRate=1.0, afMismatchPthresh=1.0, minGtForInternalImput=100,
                           ignoreFilterField=False)

There is no CPU fallback: without the CUDA library and a B200 the call raises."""
import ctypes as C
import enum
import os

import numpy as np

from .cuda import LOCUS_DTYPE, NpcError, load_library

_HERE = os.path.dirname(os.path.abspath(__file__))


class ImputeMethodLocus(enum.IntEnum):      # src/nimpress.nim:412
    ps = 0
    homref = 1
    fail = 2
    ignore = 3


class ImputeMethodMissing(enum.IntEnum):    # :413
    homref = 0
    ignore = 1


class ImputeMethodSample(enum.IntEnum):     # :414
    ps = 0
    homref = 1
    fail = 2
    int_ps = 3
    int_fail = 4


class NimpressInputError(ValueError):
    """Malformed input: where the reference raises ValueError / fails a doAssert."""


class _Params(C.Structure):
    _fields_ = [("imp_locus", C.c_int32), ("imp_missing", C.c_int32), ("imp_sample", C.c_int32),
                ("ignorefilt", C.c_int32), ("use_cov", C.c_int32), ("device", C.c_int32),
                ("exact_order", C.c_int32), ("device_mask", C.c_int32),
                ("mincs", C.c_int64), ("maxmis", C.c_double), ("afmisp", C.c_double),
                ("use_ds", C.c_int32), ("use_pl", C.c_int32), ("samples_path", C.c_char_p), ("exclude_samples", C.c_int32),
                ("observed", C.c_int32)]


_host = None


def host_library_path():
    return os.path.join(_HERE, "lib", "libnimpress_host.so")


def load_host_library():
    global _host
    if _host is not None:
        return _host
    load_library()                                   # libnimpress_cuda.so first (same directory, rpath $ORIGIN)
    path = host_library_path()
    if not os.path.exists(path):
        raise NpcError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = C.CDLL(path)
    vp, i32, i64, f64, cp = C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_char_p
    sig = {
        "nph_compute_polygenic_scores": (C.c_int, [cp, cp, cp, C.POINTER(_Params), C.POINTER(vp)]),
        "nph_compute_polygenic_scores_multi": (C.c_int, [C.POINTER(cp), C.c_int32, cp, cp, C.POINTER(_Params), C.POINTER(vp)]),
        "nph_compute_polygenic_scores_files": (C.c_int, [C.POINTER(cp), C.c_int32, C.POINTER(cp), C.c_int32, cp, C.POINTER(_Params),
                                                         C.POINTER(vp)]),
        "nph_result_n_samples": (i64, [vp]), "nph_result_n_loci": (i64, [vp]), "nph_result_nloci_used": (i64, [vp]),
        "nph_result_rounds": (i64, [vp]), "nph_result_devices": (i64, [vp]), "nph_result_scores": (vp, [vp]), "nph_result_loci": (vp, [vp]),
        "nph_result_sample": (cp, [vp, i64]), "nph_result_observed": (vp, [vp]), "nph_result_warnings": (cp, [vp]), "nph_result_free": (None, [vp]),
        "nph_last_error": (cp, []),
        "nph_plan": (C.c_int, [cp, cp, cp, C.POINTER(_Params), vp, vp, i64, C.POINTER(i64), C.POINTER(i64)]),
        "nph_fast_inflate": (C.c_int, [vp, i64, vp, i64]),
        "nph_plan_indexed": (C.c_int, [cp, cp, cp, C.POINTER(_Params), vp, vp, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
        "nph_plan_files": (C.c_int, [cp, C.POINTER(cp), C.c_int32, cp, C.POINTER(_Params), vp, vp, i64, C.POINTER(i64), C.POINTER(i64),
                                     C.POINTER(i64), C.POINTER(i64)]),
        "nph_result_records_read": (i64, [vp]), "nph_result_index_seeks": (i64, [vp]),
        "nph_read_gt": (C.c_int, [cp, vp, i64, i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i32), C.POINTER(i32)]),
        "nph_dbinom": (f64, [i64, i64, f64]), "nph_pbinom": (f64, [i64, i64, f64]), "nph_betai": (f64, [f64, f64, f64]),
        "nph_binom_test": (f64, [i64, i64, f64]), "nph_format_float": (C.c_int, [f64, cp, i32]),
        "nph_main": (C.c_int, [C.c_int, C.POINTER(cp)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    L._nph_symbols = sorted(sig)
    _host = L
    return L


# ---- objects of the reference ----------------------------------------------------------------------

class ScoreFile:
    """ScoreFile (src/nimpress.nim:195-219); `open_score` = `open` (:233-244)."""
    path = None


class VCF:
    """hts-nim VCF handle as the reference uses it: a path, sample names after the first run."""
    path = None
    samples = None


class GenomeIntervals:
    """GenomeIntervals (src/nimpress.nim:272-275); empty until loadBedIntervals."""
    path = None


def open_score(scoreFile, path):
    if not os.path.exists(path):
        return False
    scoreFile.path = path
    return True


def open_vcf(vcf, path):
    if not os.path.exists(path):
        return False
    vcf.path = path
    return True


def loadBedIntervals(ivals, path):
    if not os.path.exists(path):
        return False
    ivals.path = path
    return True


class Result:
    def __init__(self, scores, loci, nloci, samples, warnings, rounds, records_read=0, index_seeks=0, observed=None):
        self.scores, self.loci, self.nloci, self.samples, self.warnings, self.rounds = scores, loci, nloci, samples, warnings, rounds
        self.records_read, self.index_seeks = records_read, index_seeks     # index_seeks > 0: the .tbi / .csi index was used
        self.observed = observed            # int64 per sample with observed=True (DESIGN.md 4.13), else None


def run(score_path, genotype_path, bed_path=None, imp_locus=ImputeMethodLocus.ps, imp_missing=ImputeMethodMissing.homref,
        imp_sample=ImputeMethodSample.int_ps, maxmis=0.05, afmisp=0.001, mincs=100, ignorefilt=False, device=0,
        exact_order=False, devices=None, dosage=False, pl=False, samples=None, exclude_samples=False, observed=False):
    """nph_compute_polygenic_scores -> Result (scores, per-locus records, WARN text).  devices: list of CUDA
    device indices to split the score rows over (npc_reduce combines their partial sums).  dosage: score FORMAT/DS;
    pl: score FORMAT/PL as posterior expected dosages at the score file's eaf (DESIGN.md 4.10).  samples: path of a
    list of sample names to score (one per line; DESIGN.md 4.11), exclude_samples: score the others instead.
    genotype_path: one path, or a list of them (e.g. one file per chromosome) scored as their concatenation (DESIGN.md 4.12).
    observed: also fill Result.observed, per sample the OK loci at which it has a called genotype (DESIGN.md 4.13)."""
    L = load_host_library()
    mask = sum(1 << int(d) for d in set(devices)) if devices else 0
    p = _Params(int(imp_locus), int(imp_missing), int(imp_sample), int(ignorefilt), int(bed_path is not None), device,
                int(bool(exact_order)), mask, int(mincs), float(maxmis), float(afmisp), int(bool(dosage)), int(bool(pl)),
                os.fsencode(samples) if samples else None, int(bool(exclude_samples)), int(bool(observed)))
    if not isinstance(genotype_path, (str, bytes, os.PathLike)):
        return _run_files([score_path], genotype_path, bed_path, p)[0]
    h = C.c_void_p()
    rc = L.nph_compute_polygenic_scores(os.fsencode(score_path), os.fsencode(genotype_path),
                                        os.fsencode(bed_path) if bed_path else None, C.byref(p), C.byref(h))
    _check(L, rc)
    return _take_result(L, h)


def run_multi(score_paths, genotype_path, bed_path=None, imp_locus=ImputeMethodLocus.ps, imp_missing=ImputeMethodMissing.homref,
              imp_sample=ImputeMethodSample.int_ps, maxmis=0.05, afmisp=0.001, mincs=100, ignorefilt=False, device=0,
              exact_order=False, pl=False, samples=None, exclude_samples=False, observed=False):
    """nph_compute_polygenic_scores_multi: several score files over one pass of the genotype file
    -> [Result], each equal to run() on that file alone.  genotype_path: one path or a list of them, as for run()."""
    L = load_host_library()
    p = _Params(int(imp_locus), int(imp_missing), int(imp_sample), int(ignorefilt), int(bed_path is not None), device,
                int(bool(exact_order)), 0, int(mincs), float(maxmis), float(afmisp), 0, int(bool(pl)),
                os.fsencode(samples) if samples else None, int(bool(exclude_samples)), int(bool(observed)))
    if not isinstance(genotype_path, (str, bytes, os.PathLike)):
        return _run_files(score_paths, genotype_path, bed_path, p)
    paths = (C.c_char_p * len(score_paths))(*[os.fsencode(s) for s in score_paths])
    hs = (C.c_void_p * len(score_paths))()
    rc = L.nph_compute_polygenic_scores_multi(paths, len(score_paths), os.fsencode(genotype_path),
                                              os.fsencode(bed_path) if bed_path else None, C.byref(p), hs)
    _check(L, rc)
    return [_take_result(L, C.c_void_p(h)) for h in hs]


def _run_files(score_paths, genotype_paths, bed_path, p):
    """nph_compute_polygenic_scores_files: the score files over the genotype files read as their concatenation."""
    L = load_host_library()
    genotype_paths = list(genotype_paths)
    paths = (C.c_char_p * len(score_paths))(*[os.fsencode(s) for s in score_paths])
    geno = (C.c_char_p * len(genotype_paths))(*[os.fsencode(g) for g in genotype_paths])
    hs = (C.c_void_p * len(score_paths))()
    rc = L.nph_compute_polygenic_scores_files(paths, len(score_paths), geno, len(genotype_paths),
                                              os.fsencode(bed_path) if bed_path else None, C.byref(p), hs)
    _check(L, rc)
    return [_take_result(L, C.c_void_p(h)) for h in hs]


def _check(L, rc):
    if rc == -3:
        raise NimpressInputError(L.nph_last_error().decode())
    if rc in (-1, -2):
        raise FileNotFoundError(L.nph_last_error().decode())
    if rc:
        raise NpcError(f"rc={rc}: {L.nph_last_error().decode()}")


def _take_result(L, h):
    try:
        n, nl = L.nph_result_n_samples(h), L.nph_result_n_loci(h)
        scores = np.ctypeslib.as_array(C.cast(L.nph_result_scores(h), C.POINTER(C.c_double)), (n,)).copy() if n else np.zeros(0)
        loci = np.frombuffer(C.string_at(L.nph_result_loci(h), nl * LOCUS_DTYPE.itemsize), dtype=LOCUS_DTYPE).copy() if nl \
            else np.zeros(0, LOCUS_DTYPE)
        samples = [L.nph_result_sample(h, i).decode() for i in range(n)]
        op = L.nph_result_observed(h)
        observed = np.ctypeslib.as_array(C.cast(op, C.POINTER(C.c_int64)), (n,)).copy() if op and n else \
            (np.zeros(0, np.int64) if op is not None else None)
        r = Result(scores, loci, L.nph_result_nloci_used(h), samples, L.nph_result_warnings(h).decode(),
                   L.nph_result_rounds(h), L.nph_result_records_read(h), L.nph_result_index_seeks(h), observed)
        r.devices = L.nph_result_devices(h)
        return r
    finally:
        L.nph_result_free(h)


def computePolygenicScores(scores, scoreFile, genotypeVcf, restrictToCoveredRgns, coveredIvals, imputeMethodLocus,
                           imputeMethodMissing, imputeMethodSample, maxMissingRate, afMismatchPthresh,
                           minGtForInternalImput, ignoreFilterField, exactOrder=False):
    """computePolygenicScores* (src/nimpress.nim:592-599): fills `scores` (a list, resized to the
    number of samples like the reference's `var seq[float]`).  exactOrder is this engine's only
    extra: the reference's summation order bit for bit."""
    r = run(scoreFile.path, genotypeVcf.path, coveredIvals.path if restrictToCoveredRgns else None,
            imputeMethodLocus, imputeMethodMissing, imputeMethodSample, maxMissingRate, afMismatchPthresh,
            minGtForInternalImput, ignoreFilterField, exact_order=exactOrder)
    genotypeVcf.samples = r.samples
    scores[:] = r.scores.tolist()
    return r


def main(argv):
    """main() of the reference (src/nimpress.nim:652-753): returns the exit code; output on stdout."""
    L = load_host_library()
    args = [b"nimpress"] + [os.fsencode(a) for a in argv]
    arr = (C.c_char_p * len(args))(*args)
    return L.nph_main(len(args), arr)
