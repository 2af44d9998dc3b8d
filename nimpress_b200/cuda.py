"""ctypes binding of libnimpress_cuda.so (include/nimpress_cuda.h).

Fails loudly: a missing library or a missing sm_100 device raises; nothing here computes on
the CPU."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

LOCUS = {"ps": 0, "homref": 1, "fail": 2, "ignore": 3}          # ImputeMethodLocus  (src/nimpress.nim:412)
MISSING = {"homref": 0, "ignore": 1}                             # ImputeMethodMissing (:413)
SAMPLE = {"ps": 0, "homref": 1, "fail": 2, "int_ps": 3, "int_fail": 4}   # ImputeMethodSample (:414)
KIND_GT, KIND_NOTCOV, KIND_ABSENT, KIND_FILTER, CLASS_MAXMIS = range(5)
GT_BED = 0        # gt_width of a context over PLINK 1 .bed rows (2 bits per sample, ploidy 2): NPC_GT_BED
GT_DOSE255 = 255  # gt_width of a context over fixed-point dosage rows of BGEN files (uint16 255 x dosage, ploidy 2): NPC_GT_DOSE255
GT_DOSE32 = 32    # gt_width of a context over 32-bit fixed-point dosage rows of BGEN files at any bit depth (ploidy 2): NPC_GT_DOSE32
GT_PL = 10        # gt_width of a context over FORMAT/PL rows (one packed uint32 per sample, ploidy 2): NPC_GT_PL


def gt_row_bytes(n_samples, ploidy, gt_width):
    """npc_gt_row_bytes: bytes of one genotype row in a layout."""
    return int(load_library().npc_gt_row_bytes(int(n_samples), int(ploidy), int(gt_width)))

ROW_DTYPE = np.dtype([("gt_row", "<i4"), ("eaidx", "<i4"), ("beta", "<f8"), ("eaf", "<f8"),
                      ("ref_is_ea", "<i4"), ("kind", "<i4")], align=True)
LOCUS_DTYPE = np.dtype([("klass", "<i4"), ("used", "<i4"), ("eaidx", "<i4"), ("reserved", "<i4"),
                        ("ngt", "<i8"), ("nmiss", "<i8"), ("neff", "<i8"), ("imputed", "<f8")], align=True)
assert ROW_DTYPE.itemsize == 32 and LOCUS_DTYPE.itemsize == 48


class NpcError(RuntimeError):
    pass


class _Policy(C.Structure):
    _fields_ = [("imp_locus", C.c_int32), ("imp_missing", C.c_int32), ("imp_sample", C.c_int32),
                ("reserved", C.c_int32), ("mincs", C.c_int64), ("maxmis", C.c_double)]


def library_path():
    return os.path.join(_HERE, "lib", "libnimpress_cuda.so")


_lib = None


def load_library():
    """dlopen libnimpress_cuda.so and declare every export of include/nimpress_cuda.h."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise NpcError(f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)")
    L = C.CDLL(path)
    vp, i32, i64, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    pi64 = C.POINTER(C.c_int64)
    sig = {
        "npc_create": (C.c_int, [C.POINTER(vp), C.c_int, i64, i32, i32, i64, i32]),
        "npc_create2": (C.c_int, [C.POINTER(vp), C.c_int, i64, i32, i32, i64, i32, i64]),
        "npc_create_subset": (C.c_int, [C.POINTER(vp), C.c_int, i64, vp, i64, i32, i32, i64, i32, i64]),
        "npc_gather_rows_device": (C.c_int, [vp, vp, i64, i64, vp, i64]),
        "npc_set_keep": (C.c_int, [vp, vp, i64]),
        "npc_destroy": (None, [vp]),
        "npc_last_error": (C.c_char_p, [vp]),
        "npc_set_stream": (C.c_int, [vp, vp]),
        "npc_set_policy": (C.c_int, [vp, C.POINTER(_Policy)]),
        "npc_set_cohort_size": (C.c_int, [vp, i64]),
        "npc_reset": (C.c_int, [vp]),
        "npc_stage_acquire": (C.c_int, [vp, C.POINTER(i32), C.POINTER(vp), pi64]),
        "npc_score_block": (C.c_int, [vp, i32, i64, vp, i64]),
        "npc_score_block_device": (C.c_int, [vp, vp, i64, i64, vp, i64, i32]),
        "npc_count_block_device": (C.c_int, [vp, vp, i64, i64, vp, i64, i32, vp]),
        "npc_accumulate_block_device": (C.c_int, [vp, vp, i64, i64, vp, i64, i32, vp]),
        "npc_resident_reserve": (C.c_int, [vp, i64, pi64]),
        "npc_stage_upload": (C.c_int, [vp, i32, i64, i64]),
        "npc_resident_adopt": (C.c_int, [vp, vp, i64, i64]),
        "npc_score_resident": (C.c_int, [vp, vp, i64]),
        "npc_multi_contractions": (C.c_int64, [vp]),
        "npc_score_resident_multi": (C.c_int, [vp, i32, vp, vp, vp, vp, vp, vp]),
        "npc_finish": (C.c_int, [vp, f64, vp, pi64, vp, i64, pi64]),
        "npc_partial": (C.c_int, [vp, vp, pi64, vp, i64, pi64]),
        "npc_partial_device_ptr": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
        "npc_normalise": (None, [vp, i64, i64, f64]),
        "npc_reduce": (C.c_int, [C.POINTER(vp), i32, C.POINTER(f64), vp, pi64]),
        "npc_comm_unique_id": (C.c_int, [vp]),
        "npc_comm_init": (C.c_int, [vp, vp, i32, i32]),
        "npc_comm_combine": (C.c_int, [vp, C.POINTER(f64), vp, pi64]),
        "npc_combined_device_ptr": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
        "npc_comm_sum_counts": (C.c_int, [vp, vp, i64]),
        "npc_launch_count": (i64, [vp]),
        "npc_kernel_shape": (C.c_int, [vp, C.POINTER(i32 * 8)]),
        "npc_kernel_shape2": (C.c_int, [vp, i64, C.POINTER(i32 * 8)]),
        "npc_plan_shape": (C.c_int, [i64, i32, i32, i32, i64, i32, C.POINTER(i32 * 16)]),
        "npc_trace": (C.c_int, [vp, C.POINTER(C.c_uint64 * 8)]),
        "npc_set_exact_order": (C.c_int, [vp, i32]),
        "npc_set_dosage_rows": (C.c_int, [vp, i32]),
        "npc_synth_fill_device": (C.c_int, [vp, vp, i64, i64, i64, C.c_uint64, vp, vp, vp]),
        "npc_gt_row_bytes": (i64, [i64, i32, i32]),
        "npc_pl_weight_table": (C.c_int, [vp, i32]),
        "npc_version": (C.c_int, []),
        "npc_warmup": (C.c_int, [C.c_int]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)          # AttributeError if the symbol is missing
        fn.restype, fn.argtypes = res, args
    L._npc_symbols = sorted(sig)
    _lib = L
    return L


def _ptr(x):
    """device pointer of a torch tensor / int, or host pointer of a numpy array"""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return x.data_ptr()


PLAN_KEYS = ("mode", "sample_slabs", "row_groups", "chunks_per_thread", "consumer_warps", "slab_bytes", "raw_stages", "index_tiles",
             "lag", "decider_warps", "decider_tiles", "smem_bytes", "threads", "instance_warps", "wide_slabs", "wide_samples")


def plan_shape(n_samples, gt_width=1, num_sms=148, max_smem=232448, n_rows=0, exact=False):
    """npc_plan_shape: the launch shape a context of this size would choose on such a GPU -- host arithmetic, no device."""
    a = (C.c_int32 * 16)()
    rc = load_library().npc_plan_shape(int(n_samples), int(gt_width), int(num_sms), int(max_smem), int(n_rows), int(bool(exact)), C.byref(a))
    if rc != 0:
        raise NpcError(f"npc_plan_shape: error {rc}")
    return dict(zip(PLAN_KEYS, list(a)))


def pl_weight_table(n=4096):
    """npc_pl_weight_table: T[x] = fl(10^(-x/10)) correctly rounded for x = 0 .. n - 1 (0 from 3237 on), the weights of
    FORMAT/PL rows -- host only, no device."""
    out = np.zeros(n, np.float64)
    rc = load_library().npc_pl_weight_table(out.ctypes.data, int(n))
    if rc != 0:
        raise NpcError(f"npc_pl_weight_table: error {rc}")
    return out


def reduce_contexts(engines, offset=None):
    """npc_reduce over Engine objects in score-file order of their row ranges: (scores, nloci)."""
    L = load_library()
    arr = (C.c_void_p * len(engines))(*[e.h for e in engines])
    scores = np.empty(engines[0].n, dtype=np.float64)
    nloci = C.c_int64()
    off = C.byref(C.c_double(float(offset))) if offset is not None else None
    rc = L.npc_reduce(arr, len(engines), off, scores.ctypes.data, C.byref(nloci))
    if rc:
        raise NpcError(f"npc_reduce rc={rc}: {L.npc_last_error(engines[0].h).decode()}")
    return scores, nloci.value


class Engine:
    """One scoring context on one GPU: the state of one computePolygenicScores call
    (src/nimpress.nim:592-649) -- per-sample fp64 sums, nloci and the per-locus log."""

    def __init__(self, n_samples, ploidy=2, gt_width=1, max_rows_per_block=4096, n_slots=0, device=0, staging_rows=None,
                 keep=None, n_row_samples=None):
        """keep: indices of the samples to score among the n_row_samples that staged rows carry (npc_create_subset; the
        context then holds len(keep) samples and n_samples is ignored)."""
        self.L = load_library()
        self.ploidy, self.gt_width, self.max_rows = int(ploidy), int(gt_width), int(max_rows_per_block)
        h = C.c_void_p()
        self.staging_rows = int(staging_rows) if staging_rows else self.max_rows
        if keep is None:
            self.n = int(n_samples)
            rc = self.L.npc_create2(C.byref(h), device, self.n, ploidy, gt_width, max_rows_per_block, n_slots, self.staging_rows)
        else:
            keep = np.ascontiguousarray(keep, dtype=np.int64)
            self.n = len(keep)
            rc = self.L.npc_create_subset(C.byref(h), device, int(n_row_samples), keep.ctypes.data, self.n, ploidy, gt_width,
                                          max_rows_per_block, n_slots, self.staging_rows)
        if rc:
            raise NpcError(f"npc_create rc={rc}: {self.L.npc_last_error(None).decode()}")
        self.h = h

    def _ck(self, rc):
        if rc:
            raise NpcError(f"rc={rc}: {self.L.npc_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.L.npc_destroy(self.h)
            self.h = None

    __del__ = close

    def set_stream(self, cuda_stream):
        self._ck(self.L.npc_set_stream(self.h, cuda_stream))

    def set_policy(self, imp_locus="ps", imp_missing="homref", imp_sample="int_ps", maxmis=0.05, mincs=100):
        p = _Policy(LOCUS[imp_locus], MISSING[imp_missing], SAMPLE[imp_sample], 0, int(mincs), float(maxmis))
        self._ck(self.L.npc_set_policy(self.h, C.byref(p)))

    def set_exact_order(self, on=True):
        self._ck(self.L.npc_set_exact_order(self.h, int(bool(on))))

    def set_dosage_rows(self, on=True):
        self._ck(self.L.npc_set_dosage_rows(self.h, int(bool(on))))

    def set_cohort_size(self, n_total):
        self._ck(self.L.npc_set_cohort_size(self.h, int(n_total)))

    def reset(self):
        self._ck(self.L.npc_reset(self.h))

    def gather_rows_device(self, src, src_stride, n_rows, dst, dst_stride):
        """npc_gather_rows_device: compact n_rows device rows of the staged width into dst (asynchronous)."""
        self._ck(self.L.npc_gather_rows_device(self.h, _ptr(src), int(src_stride), int(n_rows), _ptr(dst), int(dst_stride)))

    def set_keep(self, keep):
        """npc_set_keep: compact rows uploaded from now on with this keep list (same length, ascending)."""
        keep = np.ascontiguousarray(keep, dtype=np.int64)
        self._ck(self.L.npc_set_keep(self.h, keep.ctypes.data, len(keep)))

    # -- host blocks through the pinned ring
    def stage_acquire(self):
        slot, ptr, stride = C.c_int32(), C.c_void_p(), C.c_int64()
        self._ck(self.L.npc_stage_acquire(self.h, C.byref(slot), C.byref(ptr), C.byref(stride)))
        buf = (C.c_uint8 * (stride.value * self.staging_rows)).from_address(ptr.value)
        view = np.frombuffer(buf, dtype=np.uint8).reshape(self.staging_rows, stride.value)
        return slot.value, view

    def score_block(self, slot, n_gt_rows, rows):
        rows = np.ascontiguousarray(rows, dtype=ROW_DTYPE)
        self._ck(self.L.npc_score_block(self.h, slot, int(n_gt_rows), rows.ctypes.data, len(rows)))

    def score_host(self, gt, rows):
        """Convenience: one block from a host array gt[n_gt_rows, >= n*ploidy*width bytes]."""
        gt = np.ascontiguousarray(gt)
        g8 = gt.view(np.uint8).reshape(gt.shape[0], -1) if gt.size else np.zeros((0, 0), np.uint8)
        slot, view = self.stage_acquire()
        if g8.shape[0]:
            view[:g8.shape[0], :g8.shape[1]] = g8
        self.score_block(slot, g8.shape[0], rows)

    # -- resident slab: upload as records stream past, score later in score-file order
    def resident_reserve(self, capacity_rows):
        g = C.c_int64()
        self._ck(self.L.npc_resident_reserve(self.h, int(capacity_rows), C.byref(g)))
        return g.value

    def resident_adopt(self, gt_dev, row_stride, n_gt_rows):
        self._ck(self.L.npc_resident_adopt(self.h, _ptr(gt_dev), int(row_stride), int(n_gt_rows)))

    def stage_upload(self, slot, n_gt_rows, dst_row):
        self._ck(self.L.npc_stage_upload(self.h, slot, int(n_gt_rows), int(dst_row)))

    def score_resident(self, rows):
        rows = np.ascontiguousarray(rows, dtype=ROW_DTYPE)
        self._ck(self.L.npc_score_resident(self.h, rows.ctypes.data, len(rows)))

    def score_resident_multi(self, rows_list, offsets, scores=None, loci=None):
        """npc_score_resident_multi -> [(scores, nloci, loci)] per score definition.  scores / loci:
        optional preallocated output arrays (e.g. views of pinned memory), one per definition."""
        S = len(rows_list)
        rows_list = [np.ascontiguousarray(r, dtype=ROW_DTYPE) for r in rows_list]
        rp = (C.c_void_p * S)(*[r.ctypes.data for r in rows_list])
        nr = np.array([len(r) for r in rows_list], dtype=np.int64)
        off = np.array(offsets, dtype=np.float64) if offsets is not None else None      # None: raw partial sums
        scores = scores if scores is not None else [np.zeros(self.n, dtype=np.float64) for _ in range(S)]
        loci = loci if loci is not None else [np.zeros(len(r), dtype=LOCUS_DTYPE) for r in rows_list]
        sp = (C.c_void_p * S)(*[a.ctypes.data for a in scores])
        lp = (C.c_void_p * S)(*[a.ctypes.data for a in loci])
        nloci = np.zeros(S, dtype=np.int64)
        self._ck(self.L.npc_score_resident_multi(self.h, S, rp, nr.ctypes.data, off.ctypes.data if off is not None else None, sp, nloci.ctypes.data, lp))
        return [(scores[k], int(nloci[k]), loci[k]) for k in range(S)]

    @property
    def multi_contractions(self):
        return self.L.npc_multi_contractions(self.h)

    # -- device-resident blocks
    def score_block_device(self, gt_dev, row_stride, n_gt_rows, rows, n_rows=None):
        if isinstance(rows, np.ndarray):
            rows = np.ascontiguousarray(rows, dtype=ROW_DTYPE)
            self._ck(self.L.npc_score_block_device(self.h, _ptr(gt_dev), row_stride, n_gt_rows, rows.ctypes.data,
                                                   len(rows), 0))
        else:
            self._ck(self.L.npc_score_block_device(self.h, _ptr(gt_dev), row_stride, n_gt_rows, _ptr(rows), n_rows, 1))

    def count_block_device(self, gt_dev, row_stride, n_gt_rows, rows, counts_dev, n_rows=None):
        on_dev = not isinstance(rows, np.ndarray)
        if not on_dev:
            rows = np.ascontiguousarray(rows, dtype=ROW_DTYPE)
            n_rows = len(rows)
        self._ck(self.L.npc_count_block_device(self.h, _ptr(gt_dev), row_stride, n_gt_rows, _ptr(rows), n_rows,
                                               int(on_dev), _ptr(counts_dev)))

    def accumulate_block_device(self, gt_dev, row_stride, n_gt_rows, rows, counts_dev, n_rows=None):
        on_dev = not isinstance(rows, np.ndarray)
        if not on_dev:
            rows = np.ascontiguousarray(rows, dtype=ROW_DTYPE)
            n_rows = len(rows)
        self._ck(self.L.npc_accumulate_block_device(self.h, _ptr(gt_dev), row_stride, n_gt_rows, _ptr(rows), n_rows,
                                                    int(on_dev), _ptr(counts_dev)))

    # -- results
    def finish(self, offset=0.0, want_loci=True, loci_cap=None):
        scores = np.empty(self.n, dtype=np.float64)
        nloci, nlog = C.c_int64(), C.c_int64()
        cap = loci_cap
        if want_loci and cap is None:
            # ask for the log length first (cheap: no loci copy)
            tmp = np.empty(self.n, dtype=np.float64)
            self._ck(self.L.npc_partial(self.h, tmp.ctypes.data, C.byref(nloci), None, 0, C.byref(nlog)))
            cap = nlog.value
        loci = np.zeros(cap if want_loci else 0, dtype=LOCUS_DTYPE)
        self._ck(self.L.npc_finish(self.h, float(offset), scores.ctypes.data, C.byref(nloci),
                                   loci.ctypes.data if want_loci else None, len(loci), C.byref(nlog)))
        return dict(scores=scores, nloci=nloci.value, loci=loci[:nlog.value])

    def partial(self, want_loci=False):
        sums = np.empty(self.n, dtype=np.float64)
        nloci, nlog = C.c_int64(), C.c_int64()
        self._ck(self.L.npc_partial(self.h, sums.ctypes.data, C.byref(nloci), None, 0, C.byref(nlog)))
        loci = None
        if want_loci:
            loci = np.zeros(nlog.value, dtype=LOCUS_DTYPE)
            self._ck(self.L.npc_partial(self.h, sums.ctypes.data, C.byref(nloci), loci.ctypes.data, len(loci),
                                        C.byref(nlog)))
        return dict(sums=sums, nloci=nloci.value, loci=loci)

    # -- several GPUs
    @staticmethod
    def comm_unique_id():
        """128 bytes that rank 0 hands to the other ranks (npc_comm_unique_id)."""
        buf = (C.c_uint8 * 128)()
        rc = load_library().npc_comm_unique_id(buf)
        if rc:
            raise NpcError(f"npc_comm_unique_id rc={rc}: {load_library().npc_last_error(None).decode()}")
        return bytes(buf)

    def comm_init(self, unique_id, rank, world):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self._ck(self.L.npc_comm_init(self.h, buf, int(rank), int(world)))

    def comm_combine(self, offset=None, want_scores=True):
        """npc_comm_combine: (scores or None, nloci) -- normalised when offset is given, raw sums otherwise.
        want_scores=False with offset=None queues the combine on the stream and returns nothing."""
        off = C.byref(C.c_double(float(offset))) if offset is not None else None
        if not want_scores:
            self._ck(self.L.npc_comm_combine(self.h, off, None, None))
            return None, None
        scores = np.empty(self.n, dtype=np.float64)
        nloci = C.c_int64()
        self._ck(self.L.npc_comm_combine(self.h, off, scores.ctypes.data, C.byref(nloci)))
        return scores, nloci.value

    def comm_sum_counts(self, counts_dev, n_rows):
        self._ck(self.L.npc_comm_sum_counts(self.h, _ptr(counts_dev), int(n_rows)))

    def combined_device_ptr(self):
        a, b = C.c_void_p(), C.c_void_p()
        self._ck(self.L.npc_combined_device_ptr(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def partial_device_ptr(self):
        a, b = C.c_void_p(), C.c_void_p()
        self._ck(self.L.npc_partial_device_ptr(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def normalise(self, sums, nloci, offset):
        sums = np.ascontiguousarray(sums, dtype=np.float64).copy()
        self.L.npc_normalise(sums.ctypes.data, len(sums), int(nloci), float(offset))
        return sums

    @property
    def kernel_shape(self):
        return self.kernel_shape_for(0)

    def kernel_shape_for(self, n_rows):
        """Launch shape of a block of n_rows score rows (long launches may split the grid differently)."""
        a = (C.c_int32 * 8)()
        self._ck(self.L.npc_kernel_shape2(self.h, int(n_rows), C.byref(a)))
        keys = ("fused", "grid", "consumer_warps", "chunks_per_thread", "rows_per_tile", "stages", "lag", "smem_bytes")
        d = dict(zip(keys, list(a)))
        d["decider_warps"], d["decider_tiles"], d["lag"] = d["lag"] % 10, d["lag"] % 100 // 10, d["lag"] // 100
        d["raw_stages"], d["index_tiles"] = d["stages"] // 1000, d["stages"] % 1000
        del d["stages"]
        if d["fused"] in (1, 2, 3):              # tile kernel: grid = sample slabs x (max) row groups
            d["row_groups"], d["grid"] = d["grid"] % 1000, d["grid"] // 1000
            d["grid"] *= d["row_groups"]
        return d

    def trace(self):
        a = (C.c_uint64 * 8)()
        self._ck(self.L.npc_trace(self.h, C.byref(a)))
        return list(a)

    @property
    def launches(self):
        return self.L.npc_launch_count(self.h)

    def synth_fill_device(self, gt_dev, row_stride, v0, n_rows, seed, af_thr16_dev, miss_thr24_dev, alt_code_dev):
        self._ck(self.L.npc_synth_fill_device(self.h, _ptr(gt_dev), row_stride, v0, n_rows, seed, _ptr(af_thr16_dev),
                                              _ptr(miss_thr24_dev), _ptr(alt_code_dev)))
