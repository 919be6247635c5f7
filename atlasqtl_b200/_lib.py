"""ctypes binding of libatlasqtl_b200.so (include/atlasqtl_b200.h).  Fails loudly: there is no fallback."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# (AQ_LIB: development knob to load another build of the same library, e.g. for A/B timing of a kernel variant)
LIB_PATH = os.environ.get("AQ_LIB") or os.path.join(_HERE, "libatlasqtl_b200.so")
_DP = ctypes.POINTER(ctypes.c_double)
_IP = ctypes.POINTER(ctypes.c_int32)

EXPORTS = ["aq_last_error", "aq_version", "aq_device_info", "aq_create", "aq_destroy", "aq_dims", "aq_set_order",
           "aq_set_state", "aq_get_state", "aq_get_residual", "aq_get_tables", "aq_refresh_tables", "aq_sweep", "aq_rowsums_zpart",
           "aq_rowsums_zpart_dev", "aq_launch_count", "aq_last_sweep_ms", "aq_last_ms", "aq_sync", "aq_coreDualLoop",
           "aq_set_missing", "aq_set_state_mis", "aq_sweep_mis", "aq_ppi_count_sum", "aq_ppi_next_above", "aq_ppi_collect",
           "aq_prep_x", "aq_prep_geno", "aq_prep_result", "aq_prep_destroy", "aq_prep_launch_count", "aq_create_prepared",
           "aq_get_x", "aq_get_y", "aq_snapshot", "aq_snapshot_fetch", "aq_coreDualMisLoop", "aq_sweep_plan",
           "aq_test_logistic", "aq_prep_dims", "aq_release_x"]


class AtlasqtlB200Error(RuntimeError):
    pass


_lib = None


def load():
    """Load the CUDA library; raise (never fall back) if it is missing or unloadable."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AtlasqtlB200Error(f"{LIB_PATH} not found: build it with `python -m atlasqtl_b200.build` "
                                "(there is no CPU fallback for the CAVI sweep)")
    lib = ctypes.CDLL(LIB_PATH)
    lib.aq_last_error.restype = ctypes.c_char_p
    lib.aq_launch_count.restype = ctypes.c_int64
    lib.aq_launch_count.argtypes = [ctypes.c_void_p]
    lib.aq_prep_launch_count.restype = ctypes.c_int64
    lib.aq_prep_launch_count.argtypes = [ctypes.c_void_p]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise AtlasqtlB200Error(f"atlasqtl_b200 error {rc}: {load().aq_last_error().decode()}")


def dptr(a):
    if a is None:
        return None
    assert isinstance(a, np.ndarray) and a.dtype == np.float64
    return a.ctypes.data_as(_DP)


def iptr(a):
    if a is None:
        return None
    assert isinstance(a, np.ndarray) and a.dtype == np.int32 and a.flags.c_contiguous
    return a.ctypes.data_as(_IP)


def fmat(a):
    """Column-major float64 view/copy (R layout)."""
    return np.asfortranarray(a, dtype=np.float64)
