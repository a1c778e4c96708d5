"""ctypes binding of libdsoft.so - every symbol include/dsoft.h declares, nothing else.

There is no fallback: if the library is missing the import of this module's `lib()` raises."""
from __future__ import annotations

import ctypes as C
import os
import threading

from . import _build

DSOFT_F_SOFT, DSOFT_F_TEXT, DSOFT_F_SOFT_LOCAL, DSOFT_F_ROW_ONLY, DSOFT_F_GMAT = 1, 2, 4, 8, 16
DSOFT_F_WEIGHTED, DSOFT_F_WSYM = 32, 64
DSOFT_F_SIGLIP = 128
DSOFT_F_DISTILL = 256
DBG_N = 32
DT_F32, DT_BF16, DT_F16 = 0, 1, 2


class Shape(C.Structure):
    """dsoft_shape_t (include/dsoft.h)."""

    _fields_ = [
        ("b", C.c_int32), ("world", C.c_int32), ("rank", C.c_int32),
        ("D", C.c_int32), ("Dp", C.c_int32), ("Dd", C.c_int32),
        ("flags", C.c_uint32), ("teacher_temp", C.c_float), ("text_temp", C.c_float),
        ("rho", C.c_float), ("c_clip", C.c_float),
    ]

    def key(self):
        return tuple(getattr(self, f) for f, _ in self._fields_)


# name -> (restype, argtypes); kept in one table so tests can check it against the header
PROTOTYPES = {
    "dsoft_version": (C.c_int, []),
    "dsoft_last_error": (C.c_char_p, []),
    "dsoft_plan_create": (C.c_int, [C.POINTER(Shape), C.POINTER(C.c_void_p)]),
    "dsoft_plan_destroy": (None, [C.c_void_p]),
    "dsoft_plan_gathered_row_elems": (C.c_size_t, [C.c_void_p]),
    "dsoft_plan_gathered_bytes": (C.c_size_t, [C.c_void_p]),
    "dsoft_plan_state_bytes": (C.c_size_t, [C.c_void_p]),
    "dsoft_plan_scratch_bytes": (C.c_size_t, [C.c_void_p]),
    "dsoft_plan_forward_scratch_bytes": (C.c_size_t, [C.c_void_p]),
    "dsoft_plan_algorithmic_flops": (C.c_double, [C.c_void_p]),
    "dsoft_plan_kernel_flops": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int]),
    "dsoft_profile_enable": (C.c_int, [C.c_int]),
    "dsoft_set_concurrency": (C.c_int, [C.c_int]),
    "dsoft_plan_concurrency": (C.c_int, [C.c_void_p]),
    "dsoft_profile_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_int]),
    "dsoft_plan_launches_forward": (C.c_int, [C.c_void_p]),
    "dsoft_plan_launches_backward": (C.c_int, [C.c_void_p]),
    "dsoft_plan_dino_col_offset": (C.c_size_t, [C.c_void_p]),
    "dsoft_gather_rows": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_int32,
                                    C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    "dsoft_pack": (C.c_int, [C.c_void_p,
                             C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_int64,
                             C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_int64,
                             C.c_void_p, C.c_void_p]),
    "dsoft_pair_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                   C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int32, C.c_void_p, C.c_float,
                                   C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "dsoft_retrieval_scratch_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "dsoft_retrieval_ranks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dsoft_knn_scratch_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "dsoft_knn_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dsoft_geometry_scratch_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "dsoft_geometry": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dsoft_siglip_g_bytes": (C.c_size_t, [C.c_void_p]),
    "dsoft_siglip_forward": (C.c_int, [C.c_void_p] * 9),
    "dsoft_siglip_backward": (C.c_int, [C.c_void_p] * 11),
    "dsoft_distill_g_bytes": (C.c_size_t, [C.c_void_p]),
    "dsoft_distill_forward": (C.c_int, [C.c_void_p] * 9),
    "dsoft_distill_backward": (C.c_int, [C.c_void_p] * 11),
    "dsoft_head_forward": (C.c_int, [C.c_void_p] * 6 + [C.c_int32, C.c_void_p, C.c_void_p]),
    "dsoft_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)] + [C.c_void_p] * 6),
    "dsoft_backward": (C.c_int, [C.c_void_p] * 6 + [C.POINTER(C.c_float)] + [C.c_void_p] * 5),
    "dsoft_forward_phase": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)] + [C.c_void_p] * 6
                            + [C.c_int]),
    "dsoft_backward_phase": (C.c_int, [C.c_void_p] * 6 + [C.POINTER(C.c_float)] + [C.c_void_p] * 5 + [C.c_int]),
    "dsoft_plan_symw_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong), C.c_int]),
    "dsoft_plan_wsigma_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong), C.c_int]),
    "dsoft_plan_lse_rows": (C.c_int, [C.c_void_p]),
    "dsoft_selftest_gemm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "dsoft_selftest_chain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
}

_lock = threading.Lock()
_lib = None


class DsoftError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load (once) the in-tree libdsoft.so.  Raises if it has not been built - no silent fallback."""
    global _lib
    with _lock:
        if _lib is None:
            # DSOFT_LIB: another build of the same sources (kernel A/B runs, scripts/build_variant.py)
            path = os.environ.get("DSOFT_LIB") or _build.LIB_PATH
            if not os.path.exists(path):
                raise DsoftError(
                    f"{path} is missing: the CUDA extension has not been built. Run "
                    "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
                    "This package has no CPU or PyTorch fallback for the loss kernels."
                )
            handle = C.CDLL(path)
            for name, (res, args) in PROTOTYPES.items():
                fn = getattr(handle, name)  # AttributeError here == header/library mismatch
                fn.restype = res
                fn.argtypes = args
            _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().dsoft_last_error()
        raise DsoftError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")
