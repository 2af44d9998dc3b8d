"""nimpress_b200 -- B200 (sm_100a) engine for the scoring path of mpinese/nimpress.

The product is ``libnimpress_cuda.so`` (C ABI in ``include/nimpress_cuda.h``) plus the C++
host in ``nimpress_b200/host``; this package is the thin ctypes layer over the C ABI that the
tests and ``bench.py`` use.  There is no CPU fallback anywhere in this package."""
from .cuda import (Engine, NpcError, LOCUS, MISSING, SAMPLE, ROW_DTYPE, LOCUS_DTYPE, KIND_GT, KIND_NOTCOV,
                   KIND_ABSENT, KIND_FILTER, CLASS_MAXMIS, GT_BED, GT_DOSE255, GT_DOSE32, GT_PL, gt_row_bytes, pl_weight_table, load_library, library_path, reduce_contexts)

__all__ = ["Engine", "NpcError", "LOCUS", "MISSING", "SAMPLE", "ROW_DTYPE", "LOCUS_DTYPE", "KIND_GT",
           "KIND_NOTCOV", "KIND_ABSENT", "KIND_FILTER", "CLASS_MAXMIS", "GT_BED", "GT_DOSE255", "GT_DOSE32", "GT_PL", "gt_row_bytes", "pl_weight_table", "load_library", "library_path", "reduce_contexts"]
