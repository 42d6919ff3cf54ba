"""ctypes binding of libbmf_b200.so (include/pybmf_b200.h).

There is NO fallback: if the library is missing or no sm_100 GPU is visible the
product path raises.  PyTorch is used only as the device allocator / stream owner.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbmf_b200.so")

_p = C.c_void_p
_i64 = C.c_int64
_i32 = C.c_int32
_f64 = C.c_double
_i8 = C.c_int8

# name -> argtypes, mirrors include/pybmf_b200.h one to one
SIGNATURES = {
    "bmf_abi_version": [],
    "bmf_device_info": [_p, _p, _p],
    "bmf_fill_zero": [_p, _i64, _p],
    "bmf_pack_csr": [_p, _p, _i64, _i64, C.c_int, _p, _i64, _p],
    "bmf_expand_bits_i8": [_p, _p, _i64, _i64, _i64, _i8, _i8, _i8, _p, _i64, _i64, _p],
    "bmf_assoc_counts_popc": [_p, _i64, _i64, _p, _i64, _p],
    "bmf_gemm_i8_nt": [_p, _i64, _p, _i64, _i64, _p, _i64, _p],
    "bmf_assoc_counts_i8": [_p, _i64, _i64, _i64, _p, _i64, _p],
    "bmf_basis_threshold": [_p, _i64, _i64, _f64, _p, _i64, _p, _i64, _p, _p, _p],
    "bmf_cover_score_popc": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _i32, _i32, _f64, _f64, _p, _p, _p],
    "bmf_cover_score_i8": [_p, _i64, _p, _i64, _i64, _i32, _p, _i32, _p, _p],
    "bmf_expand_bits_pq": [_p, _p, _i64, _i64, _i64, _p, _i64, _p],
    "bmf_cover_score_i8_general": [_p, _i64, _p, _i64, _i64, _p, _p, _p, _f64, _f64, _p, _p, _p],
    "bmf_cover_apply_general": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _f64, _f64, _p, _i64, _p, _p, _p],
    "bmf_e2m1_code": [_i32],
    "bmf_expand_bits_f4": [_p, _p, _i64, _i64, _i64, _i32, _i32, _i32, _p, _i64, _i64, _p],
    "bmf_gemm_f4_nt": [_p, _i64, _p, _i64, _i64, _p, _i64, _i32, _p],
    "bmf_cover_score_f4": [_p, _i64, _p, _i64, _i64, _p, _i32, _p, _p],
    "bmf_cover_apply_f4": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i32, _i32, _p, _i64, _i32, _p, _p, _p],
    "bmf_expand_bits_pq_f4": [_p, _p, _i64, _i64, _i64, _p, _i64, _p],
    "bmf_cover_score_f4_general": [_p, _i64, _p, _i64, _i64, _p, _p, _p, _f64, _f64, _p, _p, _p],
    "bmf_cover_apply_f4_general": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _f64, _f64, _p, _i64, _p, _p, _p],
    "bmf_select_first_max": [_p, _p, _p, _i64, _i32, _i32, _i64, _f64, _f64, _f64, _i64, _i64, _f64, _p, _p],
    "bmf_cover_apply": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i32, _i32, _f64, _f64, _p, _i64, _i8, _p, _p, _p],
    "bmf_bool_product": [_p, _i64, _i64, _p, _i64, _i64, _p, _p],
    "bmf_residual_factors": [_p, _i64, _i64, _p, _i64, _p, _i64, _p, _p],
    "bmf_confusion_factors": [_p, _i64, _i64, _p, _i64, _p, _i64, _i64, _p, _p, _p, _p],
    "bmf_confusion_bits": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p],
    "bmf_confusion_entries_bits": [_p, _p, _p, _i64, _i64, _p, _p],
    "bmf_confusion_entries_factors": [_p, _p, _i64, _i64, _p, _i64, _p, _i64, _p, _p],
    "bmf_bits_combine": [_p, _p, _i64, _i64, C.c_int, _p, _p],
    "bmf_confusion_triplets": [_p, _p, _p, _i64, _p, _i64, _p, _p, _p],
    "bmf_greedy_select": [_p, _p, _p, _p, _p, _i64, _i32, _i32, _f64, _f64, _f64, _i32, _p, _p, _p, _p, _p, _p],
    "bmf_cover_apply_compact": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p,
                                _i64, _i64, _i32, _p, _p, _p, _i64, _i32, _p, _p, _p],
    "bmf_cover_rescore_f4": [_p, _i64, _p, _i64, _i64, _p, _i32, _p, _i32, _p, _p],
    "bmf_cover_rescore_i8": [_p, _i64, _p, _i64, _i64, _i32, _p, _i32, _p, _i32, _p, _p],
    "bmf_cover_apply_compact_general": [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p, _p, _f64, _f64, _i32, _p, _p, _i64, _i64, _p,
                                        _p, _p, _p, _p, _p, _p, _p],
    "bmf_cover_rescore_f4_general": [_p, _i64, _p, _i64, _i64, _p, _p, _p, _f64, _f64, _p, _i32, _p, _p, _p],
    "bmf_cover_rescore_i8_general": [_p, _i64, _p, _i64, _i64, _p, _p, _p, _f64, _f64, _p, _i32, _p, _p, _p],
    "bmf_basis_threshold_rows": [_p, _i64, _i64, _i64, _i64, _i32, _f64, _p, _i64, _p, _p, _p],
    "bmf_expand_scores": [_p, _p, _i64, _i64, _p, _p, _f64, _f64, _p, _p, _p],
    "bmf_expand_init": [_p, _p, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p],
    "bmf_expand_step_rows": [_p, _p, _i64, _i64, _i64, _i64, _p, _p, _f64, _f64, _p, _p, _p, _i64, _i64, _p],
    "bmf_expand_step_decide": [_p, _i64, _i64, _p, _p, _f64, _f64, _p, _p, _p, _i64, _p, _i64, _p],
    "bmf_expand_col_scores": [_p, _i64, _p, _f64, _f64, _p, _p, _p],
    "bmf_optimal_rows":[_p, _i64, _i64, _p, _i64, _f64, _f64, _p, _p, _p],
    "bmf_random_bits": [_p, _i64, _i64, _i64, _i64, C.c_uint64, C.c_uint64, _f64, _p],
    "bmf_noise_bits": [_p, _i64, _i64, _i64, _i64, C.c_uint64, _f64, _f64, _p],
    "bmf_transpose_bits": [_p, _i64, _i64, _i64, _p, _i64, _p],
    "bmf_split_bits": [_p, _i64, _i64, _i64, _i64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64,
                       C.c_uint64, _p, _p],
    "bmf_probe_mma_rate": [_i32, _i32, _p, _p],
    "bmf_refine_column": [_p, _i64, _i64, _i64, _p, _i64, _p, _i64, _i64, _i32, _i32, _f64, _f64, _p, _p],
    "bmf_refine_sweep": [_p, _i64, _i64, _i64, _p, _i64, _p, _i64, _i64, _i64, _i32, _i32, _f64, _f64, _p, _p],
}


class NativeError(RuntimeError):
    pass


_lib = None


def load():
    """Load the library (building is the job of `python -m pybmf_b200.build` / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError("%s not found: run `python -m pybmf_b200.build` (nvcc, sm_100a). "
                          "pybmf_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.bmf_last_error.restype = C.c_char_p
    lib.bmf_last_error.argtypes = []
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    if lib.bmf_abi_version() != 1:
        raise NativeError("libbmf_b200.so ABI version mismatch")
    _lib = lib
    return lib


def _ptr(t):
    """Device pointer of a torch tensor (or None / int passthrough)."""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    return t.data_ptr()


def call(name, *args):
    """Call an entry point on torch's current stream; raise NativeError on a non-zero status."""
    import torch
    lib = load()
    stream = torch.cuda.current_stream().cuda_stream
    conv = [_ptr(a) if (hasattr(a, "data_ptr") or a is None) else a for a in args]
    rc = getattr(lib, name)(*conv, stream)
    if rc != 0:
        msg = lib.bmf_last_error().decode("utf-8", "replace")
        if rc < 0:
            raise ValueError("%s failed (%d): %s" % (name, rc, msg))
        raise NativeError("%s failed (cudaError %d): %s" % (name, rc, msg))


def require_gpu():
    """Fail loudly unless a B200-class (sm_100) device is visible."""
    import torch
    if not torch.cuda.is_available():
        raise NativeError("pybmf_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    lib = load()
    sm, maj, mnr = C.c_int(), C.c_int(), C.c_int()
    rc = lib.bmf_device_info(C.byref(sm), C.byref(maj), C.byref(mnr))
    if rc != 0:
        raise NativeError(lib.bmf_last_error().decode())
    return sm.value, maj.value, mnr.value
