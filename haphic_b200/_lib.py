"""ctypes binding of libhaphic_b200.so (the C ABI declared in include/haphic_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is
present every entry point raises.
"""

from __future__ import annotations

import ctypes as C
import weakref
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libhaphic_b200.so")

HH_MEM_HOST, HH_MEM_DEVICE = 0, 1


class HHError(RuntimeError):
    pass


class LinksInfo(C.Structure):
    _fields_ = [("n_records", C.c_int64), ("n_used", C.c_int64), ("nnz_full", C.c_int64), ("nnz_flank", C.c_int64),
                ("table_slots", C.c_int64)]


class MclResult(C.Structure):
    _fields_ = [("rounds", C.c_int32), ("converged", C.c_int32), ("nnz", C.c_int64), ("products", C.c_int64),
                ("bytes", C.c_int64)]


class PreexpInfo(C.Structure):
    _fields_ = [("mode", C.c_int32), ("a_planes", C.c_int32), ("passes", C.c_int32), ("cta_group", C.c_int32),
                ("stages", C.c_int32), ("chunk_kb", C.c_int32), ("total_ms", C.c_float), ("densify_ms", C.c_float),
                ("gemm_ms", C.c_float), ("clip_ms", C.c_float), ("flops", C.c_double), ("products", C.c_int64),
                ("clip", C.c_float), ("b_planes", C.c_int32), ("fmt_a", C.c_int32), ("fmt_b", C.c_int32), ("k_chunks", C.c_int32)]


HH_PREEXP_AUTO, HH_PREEXP_SPARSE, HH_PREEXP_DENSE = 0, 1, 2

# name -> (restype, argtypes): every symbol include/haphic_b200.h declares
_P = C.c_void_p
_SIGNATURES = {
    "hh_version": (C.c_int, []),
    "hh_last_error": (C.c_char_p, []),
    "hh_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "hh_ctx_destroy": (C.c_int, [_P]),
    "hh_ctx_sync": (C.c_int, [_P]),
    "hh_ctx_stream": (_P, [_P]),
    "hh_ctx_device": (C.c_int, [_P]),
    "hh_ctx_sm_count": (C.c_int, [_P]),
    "hh_ctx_launches": (C.c_int64, [_P]),
    "hh_links_create": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_int64, C.c_int64, C.POINTER(_P)]),
    "hh_links_create_frags": (C.c_int, [_P, C.c_int32, _P, _P, C.c_int32, _P, _P, _P, C.c_int64, C.c_int64, C.c_int64,
                                        C.POINTER(_P)]),
    "hh_links_add": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int]),
    "hh_links_add_async": (C.c_int, [_P, _P, C.c_int64, C.c_int64]),
    "hh_links_finish": (C.c_int, [_P, C.POINTER(LinksInfo)]),
    "hh_links_fetch": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    "hh_links_fetch_ctg": (C.c_int, [_P, _P]),
    "hh_links_export": (C.c_int, [_P, _P, _P]),
    "hh_links_merge": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int64, C.c_int64]),
    "hh_links_route": (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int, _P, _P, _P]),
    "hh_links_add_routed": (C.c_int, [_P, _P, _P, C.c_int64]),
    "hh_links_finish_partition": (C.c_int, [_P, _P]),
    "hh_links_adopt": (C.c_int, [_P, _P, C.c_int64, _P, C.c_int64, C.c_int64, C.c_int64]),
    "hh_links_destroy": (C.c_int, [_P]),
    "hh_links_linked_index": (C.c_int, [_P, _P, _P, C.POINTER(C.c_int32)]),
    "hh_matrix_from_links": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int, C.c_int, C.POINTER(_P)]),
    "hh_matrix_rank_sums": (C.c_int, [_P, C.c_int, _P]),
    "hh_matrix_from_csc": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.POINTER(_P)]),
    "hh_matrix_info": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "hh_matrix_fetch_csc": (C.c_int, [_P, _P, _P, _P]),
    "hh_matrix_destroy": (C.c_int, [_P]),
    "hh_mcl_create": (C.c_int, [_P, C.c_int, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "hh_mcl_create_ex": (C.c_int, [_P, C.c_int, C.c_int32, C.c_int32, C.c_int, C.POINTER(_P)]),
    "hh_mcl_preexp_info": (C.c_int, [_P, C.POINTER(PreexpInfo)]),
    "hh_mcl_info": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                              C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "hh_mcl_fetch_m0": (C.c_int, [_P, _P, _P, _P]),
    "hh_mcl_fetch_m1": (C.c_int, [_P, _P]),
    "hh_mcl_run": (C.c_int, [_P, C.c_double, C.c_int, C.c_double, C.POINTER(MclResult), _P, _P, _P, _P]),
    "hh_mcl_fetch_result": (C.c_int, [_P, _P, _P, _P]),
    "hh_mcl_begin": (C.c_int, [_P, C.c_double, C.c_double]),
    "hh_mcl_step": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_float),
                              C.POINTER(C.c_float)]),
    "hh_mcl_pack": (C.c_int, [_P, _P, _P, _P]),
    "hh_mcl_unpack": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, C.c_int64]),
    "hh_mcl_commit": (C.c_int, [_P]),
    "hh_mcl_set_block": (C.c_int, [_P, C.c_int32, C.c_int32]),
    "hh_mcl_destroy": (C.c_int, [_P]),
    "hh_pairs_open": (C.c_int, [C.c_char_p, _P, C.c_int32, C.c_char_p, C.c_int, C.c_int, C.POINTER(_P)]),
    "hh_pairs_next": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "hh_pairs_close": (C.c_int, [_P]),
    "hh_pairs_write": (C.c_int, [C.c_char_p, _P, C.c_int32, _P, C.c_int64, C.c_int64, C.c_int, C.c_int]),
    "hh_bam_open": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int32, C.c_int, C.c_int, C.POINTER(_P)]),
    "hh_bam_header_text": (C.c_int, [_P, C.POINTER(C.c_char_p), C.POINTER(C.c_int64)]),
    "hh_bam_next": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "hh_bam_close": (C.c_int, [_P]),
    "hh_pickle_links": (C.c_int, [C.c_char_p, _P, C.c_int32, _P, _P, C.c_int64, _P, _P, _P]),
    "hh_clm_from_records": (C.c_int, [C.c_char_p, _P, C.c_int32, _P, C.c_int64, _P, _P, C.c_int]),
    "hh_correct_create": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.POINTER(_P)]),
    "hh_correct_add": (C.c_int, [_P, _P, C.c_int64, C.c_int]),
    "hh_correct_info": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "hh_correct_fetch": (C.c_int, [_P, _P, _P, _P]),
    "hh_correct_detect": (C.c_int, [_P, C.c_int32, _P, _P, _P, C.c_double, C.c_double, C.c_int64, _P, _P, _P, C.c_int64,
                                    C.POINTER(C.c_int64)]),
    "hh_correct_detect_segments": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, _P, _P, _P, C.c_double, C.c_double,
                                             C.c_int64, _P, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "hh_correct_split": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int32]),
    "hh_correct_set_pieces": (C.c_int, [_P, C.c_int32, _P, _P, _P]),
    "hh_correct_remap": (C.c_int, [_P, _P, C.c_int64, C.c_int]),
    "hh_correct_destroy": (C.c_int, [_P]),
}

_lib = None


def exported_symbols():
    return sorted(_SIGNATURES)


def load():
    """Load the shared library (once).  Raises HHError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HHError(
            "{} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `python -m haphic_b200.build`). haphic_b200 has no CPU fallback.".format(LIB_PATH))
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = ABI mismatch, surface it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        msg = load().hh_last_error()
        raise HHError("libhaphic_b200 error {}: {}".format(rc, msg.decode() if msg else "?"))


def ptr(x):
    """void* of a numpy array (host), a torch tensor (host or device) or None."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data_as(C.c_void_p)
    if hasattr(x, "data_ptr"):
        return C.c_void_p(x.data_ptr())
    if isinstance(x, int):
        return C.c_void_p(x)
    raise TypeError("cannot take the address of {!r}".format(type(x)))


class Context:
    """One GPU + one CUDA stream (hh_ctx)."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        lib = load()
        check(lib.hh_ctx_create(int(device), C.byref(self._h)))
        self.device = int(device)
        self._children = weakref.WeakSet()      # LinkTable / LinkMatrix / Mcl objects living on this context

    def adopt(self, obj):
        """Register an object whose library handle dies with this context: close() destroys it first, so a handle that
        outlives its context (e.g. kept alive by a traceback) is never passed to the library again."""
        self._children.add(obj)

    @property
    def handle(self):
        if not self._h:
            raise HHError("context already closed")
        return self._h

    def sync(self):
        check(load().hh_ctx_sync(self.handle))

    @property
    def stream(self) -> int:
        return int(load().hh_ctx_stream(self.handle) or 0)

    @property
    def sm_count(self) -> int:
        return load().hh_ctx_sm_count(self.handle)

    @property
    def launches(self) -> int:
        return int(load().hh_ctx_launches(self.handle))

    def close(self):
        if self._h:
            for obj in sorted(self._children, key=lambda o: -getattr(o, "_close_order", 0)):
                obj.close()
            load().hh_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
