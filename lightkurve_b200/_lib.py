"""ctypes binding of ``liblkb200.so`` (the C ABI declared in ``include/lkb200.h``).

There is deliberately NO fallback here: if the shared library is missing, or no
B200 is visible, every compute call raises.  (The reference's arithmetic lives in
astropy/scipy; this engine replaces it with CUDA and nothing else.)
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblkb200.so")

OK, E_ARG, E_CUDA, E_OOM, E_SINGULAR, E_UNSUPPORTED, E_NCCL, E_VERIFY = 0, -1, -2, -3, -4, -5, -6, -7
NCCL_ID_BYTES = 128
MEM_HOST, MEM_DEVICE = 0, 1
DTYPE_F32, DTYPE_F64 = 0, 1
LS_NORM_PSD_RAW, LS_NORM_PSD_SCALE, LS_NORM_AMPLITUDE = 0, 1, 2
LS_ALGO_AUTO, LS_ALGO_SIMT, LS_ALGO_TCGEN05, LS_ALGO_NUFFT = 0, 1, 2, 3
BLS_LIKELIHOOD, BLS_SNR = 0, 1

c_int, c_i64, c_dbl, c_vp = ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p

# name -> (restype, argtypes); pointers are passed as void* so that host numpy
# buffers and raw device addresses go through the same entry points.
SIGNATURES = {
    "lkb_last_error": (ctypes.c_char_p, []),
    "lkb_version": (c_int, []),
    "lkb_device_count": (c_int, []),
    "lkb_init": (c_int, [c_int]),
    "lkb_shutdown": (c_int, []),
    "lkb_sm_count": (c_int, []),
    "lkb_launch_count": (c_i64, []),
    "lkb_ls_last_algo": (c_int, []),
    "lkb_ls_last_escalated": (c_int, []),
    "lkb_profile_enable": (c_int, [c_int]),
    "lkb_profile_read": (c_int, [c_vp, c_int]),
    "lkb_ws_read": (c_int, [c_int, c_i64, c_i64, c_vp]),
    "lkb_ls_power": (c_int, [c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_int, c_vp]),
    "lkb_ls_power_ex": (c_int, [c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_int, c_vp,
                                c_int]),
    "lkb_ls_power_chi2": (c_int, [c_vp, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp,
                                  c_int, c_vp]),
    "lkb_ls_power_shared": (c_int, [c_vp, c_vp, c_int, c_int, c_i64, c_vp, c_i64, c_int, c_vp, c_vp, c_int,
                                    c_vp, c_int]),
    "lkb_bls_power": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_i64, c_vp, c_int, c_int, c_int,
                              c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp]),
    "lkb_bls_power_slow": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_i64, c_vp, c_int, c_int, c_int,
                                   c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp]),
    "lkb_bls_bin_index": (c_int, [c_vp, c_i64, c_dbl, c_dbl, c_dbl, c_vp, c_int, c_vp]),
    "lkb_flatten": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_dbl, c_int, c_dbl,
                            c_vp, c_vp, c_vp, c_int, c_vp]),
    "lkb_regress": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_i64, c_int, c_dbl, c_int,
                            c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp]),
    "lkb_savgol_tables": (c_int, [c_int, c_int, c_vp, c_vp]),
    "lkb_nanmedian_std": (c_int, [c_vp, c_vp, c_int, c_vp, c_vp, c_int, c_vp]),
    "lkb_pg_logmedian": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp, c_int, c_dbl, c_vp, c_int, c_vp]),
    "lkb_nccl_version": (c_int, []),
    "lkb_nccl_unique_id": (c_int, [c_vp]),
    "lkb_nccl_init": (c_int, [c_int, c_int, c_vp]),
    "lkb_nccl_shutdown": (c_int, []),
    "lkb_nccl_rank": (c_int, []),
    "lkb_nccl_world_size": (c_int, []),
    "lkb_allgather_f32": (c_int, [c_vp, c_i64, c_vp, c_vp]),
}

_lib = None


class EngineError(RuntimeError):
    """Raised for any non-zero status of the C ABI (message from lkb_last_error)."""

    def __init__(self, status, message):
        super().__init__("liblkb200 status %d: %s" % (status, message))
        self.status = status


class SingularMatrixError(EngineError, np.linalg.LinAlgError):
    """LKB_E_SINGULAR: the analogue of numpy.linalg.LinAlgError('Singular matrix')."""


def load():
    """Load liblkb200.so (no CUDA call is made).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C lightkurve_b200/csrc`.  lightkurve_b200 has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status):
    if status == OK:
        return
    msg = load().lkb_last_error().decode("utf-8", "replace")
    if status == E_SINGULAR:
        raise SingularMatrixError(status, msg or "Singular matrix")
    if status == E_ARG:
        raise ValueError(msg)
    raise EngineError(status, msg)


def ptr(x):
    """void* of a contiguous numpy array, a torch tensor, an int address, or None."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array passed to liblkb200 must be C-contiguous")
        return x.ctypes.data
    if isinstance(x, int):
        return x
    if hasattr(x, "data_ptr"):
        if not x.is_contiguous():
            raise ValueError("tensor passed to liblkb200 must be contiguous")
        return x.data_ptr()
    raise TypeError("cannot take a pointer of %r" % type(x))
