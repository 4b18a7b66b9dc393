"""ctypes binding of libnsr_b200.so (the C ABI declared in include/normalisr_b200.h).

The product path has no CPU fallback: if the library is missing or the device is not a
B200-class (sm_100) GPU, calls raise."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnsr_b200.so")

MODE_COEX, MODE_DE, MODE_RAW, MODE_COEX_UPPER, MODE_COEX_RECT = 0, 1, 2, 3, 4
ENGINE_UMMA, ENGINE_SIMT = 0, 1
TILE = 128
KBLOCK = 128
MAX_RANK = 64
MAX_SPLITS = 64
MAX_SLICES = 4

_lib = None

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_vp = ctypes.c_void_p
c_dbl = ctypes.c_double
c_up = ctypes.c_size_t           # uintptr_t

_SIGNATURES = {
    "nsr_version": (c_int, []),
    "nsr_last_error": (ctypes.c_char_p, []),
    "nsr_ctx_create": (c_int, [c_int, ctypes.POINTER(c_vp)]),
    "nsr_ctx_destroy": (c_int, [c_vp]),
    "nsr_padded_cells": (c_i64, [c_i64]),
    "nsr_set_option": (c_int, [ctypes.c_char_p, c_int]),
    "nsr_cell_splits": (c_int, [c_i64]),
    "nsr_pair_tiles": (c_i64, [c_vp, c_i64, c_int, c_vp]),
    "nsr_residualize": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_i64, c_int, c_vp,
                                c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "nsr_contract": (c_int, [c_vp, c_up, c_int, c_int,
                             c_vp, c_i64, c_i64, c_vp, c_vp,
                             c_vp, c_i64, c_i64, c_vp, c_vp,
                             c_i64, c_i64, c_int, c_int, c_vp, c_i64, c_dbl, c_vp, c_vp, c_i64, c_i64]),
    "nsr_contract_ab": (c_int, [c_vp, c_up, c_int, c_int,
                                c_vp, c_i64, c_i64, c_int, c_vp, c_vp,
                                c_vp, c_i64, c_i64, c_int, c_vp, c_vp,
                                c_i64, c_i64, c_int, c_vp, c_i64, c_dbl, c_vp, c_vp, c_i64, c_i64]),
    "nsr_contract_segments": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_vp, c_vp, c_i64, c_i64, c_int, c_int,
                                      c_vp, c_int, c_vp, c_i64, c_dbl, c_vp, c_vp, c_i64, c_i64]),
    "nsr_stream_signal": (c_int, [c_vp, c_up, c_vp, ctypes.c_uint32]),
    "nsr_stream_wait_geq": (c_int, [c_vp, c_up, c_vp, ctypes.c_uint32]),
    "nsr_residualize_exact": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_i64, c_vp,
                                      c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "nsr_gram_f64": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_vp, c_i64]),
    "nsr_gram_correct": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_vp, c_int]),
    "nsr_de4_solve": (c_int, [c_vp, c_up, c_vp, c_int, c_vp, c_i64, c_i64, c_vp, c_i64, c_int, c_int, c_dbl, c_int,
                              c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "nsr_tsv_shape": (c_int, [ctypes.c_char_p, ctypes.c_char, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]),
    "nsr_tsv_read": (c_int, [ctypes.c_char_p, ctypes.c_char, c_vp, c_i64, c_i64, c_i64, c_int]),
    "nsr_tsv_write": (c_int, [ctypes.c_char_p, ctypes.c_char, c_vp, c_i64, c_i64, c_i64, c_int, c_int]),
    "nsr_mtx_shape": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64), ctypes.POINTER(c_i64),
                              ctypes.POINTER(c_int)]),
    "nsr_mtx_read": (c_int, [ctypes.c_char_p, c_i64, c_vp, c_vp, c_vp, ctypes.POINTER(c_int), c_int]),
    "nsr_pvalue": (c_int, [c_vp, c_up, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "nsr_copy2d": (c_int, [c_vp, c_up, c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_int]),
    "nsr_host_copy2d": (c_int, [c_vp, c_i64, c_vp, c_i64, c_i64, c_i64, c_int]),
    "nsr_copy_peer": (c_int, [c_vp, c_up, c_vp, c_vp, c_int, c_i64]),
    "nsr_unslice": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp]),
    "nsr_binnet": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_i64, c_dbl, c_vp, c_i64, c_vp]),
    "nsr_binnet_count": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_i64, c_dbl, c_vp, c_vp, c_vp]),
    "nsr_binnet_csr_fill": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_int, c_vp, c_i64,
                                    c_vp, c_vp, c_vp]),
    "nsr_project_coef": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_i64, c_vp, c_vp]),
    "nsr_group_stats": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_vp, c_int, c_i64, c_vp, c_int, c_vp]),
    "nsr_normvar_width": (c_int, [c_int]),
    "nsr_normvar_stats": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_i64, c_vp, c_vp, c_vp]),
    "nsr_normvar_rhs": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "nsr_normvar_apply": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_vp,
                                  c_vp, c_i64]),
    "nsr_sym_pinv": (c_int, [c_vp, c_up, c_vp, c_i64, c_int, c_dbl, c_vp, c_vp]),
    "nsr_single1_finish": (c_int, [c_vp, c_up, c_vp, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                   c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "nsr_last_refined": (c_int, [c_vp, c_up, c_i64, c_vp]),
    "nsr_lcpm_scan": (c_int, [c_vp, c_up, c_vp, c_int, c_i64, c_i64, c_i64, c_vp]),
    "nsr_lcpm_colstats": (c_int, [c_vp, c_up, c_vp, c_int, c_i64, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64,
                                  ctypes.c_uint64, c_i64, c_vp, c_vp]),
    "nsr_lcpm_apply": (c_int, [c_vp, c_up, c_vp, c_int, c_i64, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64,
                               ctypes.c_uint64, c_i64, c_vp, c_vp, c_i64]),
    "nsr_lcpm_colstats_csr": (c_int, [c_vp, c_up, c_vp, c_vp, c_vp, c_int, c_i64, c_i64, c_vp, c_vp, c_i64, c_vp,
                                      c_vp, c_i64, ctypes.c_uint64, c_i64, c_vp, c_vp]),
    "nsr_lcpm_apply_csr": (c_int, [c_vp, c_up, c_vp, c_vp, c_vp, c_int, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64,
                                   ctypes.c_uint64, c_i64, c_vp, c_vp, c_i64]),
    "nsr_colvar": (c_int, [c_vp, c_up, c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "nsr_cov_gram": (c_int, [c_vp, c_up, c_vp, c_int, c_i64, c_i64, c_vp]),
    "nsr_cov_apply": (c_int, [c_vp, c_up, c_vp, c_int, c_int, c_vp, c_i64, c_i64, c_vp, c_i64]),
}


MAX_SEGMENTS = 10


class Segment(ctypes.Structure):
    """struct nsr_segment (include/normalisr_b200.h)."""
    _fields_ = [("b_slices", c_vp), ("rows_b", c_i64), ("rows_alloc_b", c_i64), ("quantum_b", c_vp), ("var_b", c_vp),
                ("col0", c_i64), ("diagonal", ctypes.c_int32), ("ready_value", ctypes.c_uint32), ("ready", c_vp),
                ("done", c_vp), ("mirror_P", c_vp), ("mirror_out2", c_vp), ("ld_mirror", c_i64)]


class NsrError(RuntimeError):
    pass


def load():
    """Load the shared library (building it first if sources are newer and nvcc exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NsrError(
            "normalisr_b200: %s is missing. Build it with `python -m normalisr_b200._build` "
            "(needs nvcc; sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(status, what):
    if status != 0:
        msg = load().nsr_last_error()
        raise NsrError("%s failed (status %d): %s" % (what, status, msg.decode() if msg else "?"))
