"""ctypes binding of libdecaf377_b200.so (the C ABI of include/decaf377_b200.h).

There is deliberately no fallback: a missing library or a missing GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

HERE = Path(__file__).resolve().parent
# D377_DEBUG_LIB=1 loads the build that checks every point the kernels produce against the
# reference's OnCurve predicate (decaf377_b200/build.py --debug)
DEBUG = os.environ.get("D377_DEBUG_LIB", "0") not in ("", "0")
LIB_PATH = HERE / ("libdecaf377_b200_dbg.so" if DEBUG else "libdecaf377_b200.so")

OK = 0
ERR_INVALID_ARG = -1
ERR_CUDA = -2
ERR_NOT_INITIALISED = -3
ERR_SCALAR_RANGE = -4
ERR_INVALID_ENCODING = -5

PT_ELEMENT, PT_ENCODING, PT_AFFINE, PT_XYZ, PT_BASES = 0, 1, 2, 3, 4
OUT_ELEMENT, OUT_ENCODING = 0, 1
PT_WIDTH = {PT_ELEMENT: 128, PT_ENCODING: 32, PT_AFFINE: 64, PT_XYZ: 96}   # bytes per point
OUT_WIDTH = {OUT_ELEMENT: PT_WIDTH[PT_ELEMENT], OUT_ENCODING: PT_WIDTH[PT_ENCODING]}   # bytes per result
SCALARS_MONTGOMERY = 0x100   # OR into point_format (out_format for fixed_base_mul / fixed_bases_mul)

u8p = C.c_void_p
_SIGS = {
    "d377_init": [C.c_int],
    "d377_init_multi": [C.POINTER(C.c_int), C.c_int],
    "d377_set_device": [C.c_int],
    "d377_get_device": [],
    "d377_device_list": [C.POINTER(C.c_int), C.c_int],
    "d377_shutdown": [],
    "d377_sync": [],
    "d377_join": [],
    "d377_msm_set_tail_overlap": [C.c_int],
    "d377_debug_build": [],
    "d377_debug_counts": [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)],
    "d377_batch_encode_to_curve_wide": [u8p, C.c_size_t, C.c_size_t, u8p, C.c_int],
    "d377_batch_hash_to_curve_wide": [u8p, u8p, C.c_size_t, C.c_size_t, u8p, C.c_int],
    "d377_fq_batch_from_le_bytes_mod_order": [u8p, C.c_size_t, C.c_size_t, u8p],
    "d377_batch_sub": [u8p, u8p, C.c_size_t, u8p],
    "d377_batch_neg": [u8p, C.c_size_t, u8p],
    "d377_batch_double": [u8p, C.c_size_t, u8p],
    "d377_batch_on_curve": [u8p, C.c_size_t, C.c_int, u8p],
    "d377_element_sum_result_dev": [u8p, C.c_size_t, u8p, u8p],
    "d377_msm_dev_async": [u8p, u8p, C.c_int, C.c_size_t, u8p, u8p, C.c_int],
    "d377_msm_multi": [u8p, u8p, C.c_int, C.c_size_t, C.c_int, u8p, u8p],
    "d377_msm_multi_dev": [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                           C.POINTER(C.c_size_t), C.c_int, u8p, u8p],
    "d377_msm_multi_dev_async": [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int,
                                 C.POINTER(C.c_size_t), C.c_int, u8p, u8p],
    "d377_multi_sync": [],
    "d377_batch_msm": [u8p, u8p, C.c_int, u8p, C.c_size_t, u8p, C.c_int, u8p],
    "d377_batch_msm_dev": [u8p, u8p, C.c_int, u8p, C.c_size_t, C.c_size_t, u8p, C.c_int, u8p],
    "d377_msm_segmented": [u8p, u8p, C.c_int, u8p, C.c_size_t, u8p, C.c_int, u8p],
    "d377_msm_segmented_last": [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t)],
    "d377_msm_set_window": [C.c_int],
    "d377_msm_set_host_chunks": [C.c_int],
    "d377_host_free": [C.c_void_p],
    "d377_batch_decompress": [u8p, C.c_size_t, u8p, u8p],
    "d377_batch_compress": [u8p, C.c_size_t, u8p],
    "d377_batch_decompress_fmt": [u8p, C.c_size_t, C.c_int, u8p, u8p],
    "d377_batch_compress_fmt": [u8p, C.c_int, C.c_size_t, u8p],
    "d377_batch_encode_to_curve": [u8p, C.c_size_t, u8p, C.c_int],
    "d377_batch_hash_to_curve": [u8p, u8p, C.c_size_t, u8p, C.c_int],
    "d377_batch_scalar_mul": [u8p, C.c_int, u8p, C.c_size_t, u8p, C.c_int, u8p],
    "d377_fixed_base_mul": [u8p, C.c_size_t, u8p, C.c_int],
    "d377_batch_add": [u8p, u8p, C.c_size_t, u8p],
    "d377_batch_element_eq": [u8p, u8p, C.c_size_t, u8p],
    "d377_element_sum": [u8p, C.c_size_t, u8p, u8p],
    "d377_msm": [u8p, u8p, C.c_int, C.c_size_t, u8p, u8p],
    "d377_msm_submit": [u8p, u8p, C.c_int, C.c_size_t, C.c_int],
    "d377_msm_bases_create": [u8p, C.c_int, C.c_size_t, C.POINTER(C.c_void_p)],
    "d377_msm_bases_destroy": [C.c_void_p],
    "d377_msm_bases_create_windowed": [u8p, C.c_int, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)],
    "d377_msm_bases_info": [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_int),
                            C.POINTER(C.c_size_t)],
    "d377_msm_last_windowed": [C.POINTER(C.c_int)],
    "d377_fixed_bases_create": [u8p, C.c_int, C.c_size_t, C.POINTER(C.c_void_p)],
    "d377_fixed_bases_info": [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)],
    "d377_fixed_bases_destroy": [C.c_void_p],
    "d377_fixed_bases_mul": [C.c_void_p, u8p, C.c_size_t, u8p, C.c_int],
    "d377_msm_wait": [C.c_int, u8p, u8p],
    "d377_fq_batch_op": [C.c_int, u8p, u8p, C.c_size_t, u8p],
    "d377_fq_batch_isqrt": [u8p, C.c_size_t, u8p, u8p],
    "d377_fq_batch_sqrt_ratio_zeta": [u8p, u8p, C.c_size_t, u8p, u8p],
    "d377_field_batch_deserialize": [C.c_int, u8p, C.c_size_t, u8p, u8p],
    "d377_batch_normalize": [u8p, C.c_size_t, u8p],
    "d377_imad_peak": [C.POINTER(C.c_double)],
    "d377_msm_stage_info": [C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_int),
                            C.POINTER(C.c_uint64)],
    "d377_msm_last_mode": [C.POINTER(C.c_int)],
    "d377_msm_timeline": [C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_int)],
    "d377_msm_set_normalize": [C.c_int],
    "d377_msm_set_groups": [C.c_int],
}
# every host entry point above except the field/debug ones has a `_dev` twin
for _n in ["d377_batch_decompress", "d377_batch_compress", "d377_batch_encode_to_curve",
           "d377_batch_hash_to_curve", "d377_batch_scalar_mul", "d377_fixed_base_mul",
           "d377_batch_add", "d377_batch_element_eq", "d377_element_sum", "d377_msm",
           "d377_fq_batch_isqrt", "d377_fq_batch_sqrt_ratio_zeta", "d377_field_batch_deserialize",
           "d377_batch_normalize", "d377_msm_bases_create", "d377_msm_bases_create_windowed",
           "d377_fixed_bases_create", "d377_fixed_bases_mul",
           "d377_batch_encode_to_curve_wide",
           "d377_batch_hash_to_curve_wide", "d377_fq_batch_from_le_bytes_mod_order",
           "d377_batch_sub", "d377_batch_neg", "d377_batch_double", "d377_batch_on_curve",
           "d377_batch_decompress_fmt", "d377_batch_compress_fmt", "d377_msm_segmented"]:
    _SIGS[_n + "_dev"] = _SIGS[_n]

EXPORTS = sorted(list(_SIGS) + ["d377_stream", "d377_result_stream", "d377_last_error",
                                 "d377_launch_count", "d377_host_alloc"])

_lib = None


class D377Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("decaf377_b200 error %d: %s" % (code, msg))
        self.code = code


def load() -> C.CDLL:
    """Load the shared library (no GPU needed for this step)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            "%s is missing: build it with `python -m decaf377_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(str(LIB_PATH), mode=os.RTLD_LOCAL)
    for name, args in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.d377_stream.argtypes = []
    lib.d377_stream.restype = C.c_void_p
    lib.d377_result_stream.argtypes = []
    lib.d377_result_stream.restype = C.c_void_p
    lib.d377_host_alloc.argtypes = [C.c_size_t]
    lib.d377_host_alloc.restype = C.c_void_p
    lib.d377_last_error.argtypes = []
    lib.d377_last_error.restype = C.c_char_p
    lib.d377_launch_count.argtypes = []
    lib.d377_launch_count.restype = C.c_uint64
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != OK:
        raise D377Error(rc, load().d377_last_error().decode(errors="replace"))
