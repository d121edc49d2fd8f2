"""ctypes binding of libsimdjson_b200.so (include/simdjson_b200.h).  No fallback: a missing library raises."""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libsimdjson_b200.so")

FLAG_VALIDATE_UTF8 = 1
FLAG_NO_UTF8 = 4
FLAG_TIMING = 8

# every symbol include/simdjson_b200.h declares: (restype, argtypes)
_vp, _u64, _u32, _i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32
_pu32, _pi32, _pu64 = C.POINTER(C.c_uint32), C.POINTER(C.c_int32), C.POINTER(C.c_uint64)
SIGNATURES = {
    "sjb200_version": (_i32, []),
    "sjb200_device_count": (_i32, []),
    "sjb200_ctx_create": (_i32, [_i32, _u64, _u64, _u32, C.POINTER(_vp)]),
    "sjb200_ctx_destroy": (_i32, [_vp]),
    "sjb200_ctx_set_stream": (_i32, [_vp, _vp]),
    "sjb200_ctx_set_warps": (_i32, [_vp, _i32]),
    "sjb200_ctx_set_kernel": (_i32, [_vp, _i32]),
    "sjb200_ctx_reserve": (_i32, [_vp, _u64, _u32]),
    "sjb200_ctx_set_chunk_bytes": (_i32, [_vp, _u64]),
    "sjb200_stage1": (_i32, [_vp, _vp, _u64, _vp, _u64, _pu32, _pi32, _u32]),
    "sjb200_structural_bytes_device_async": (_i32, [_vp, _vp, _u64, _vp, _u64, _vp]),
    "sjb200_document_starts_device_async": (_i32, [_vp, _vp, _u64, _vp, _vp, _u64]),
    "sjb200_stage1_device_async": (_i32, [_vp, _vp, _u64, _vp, _u64, _u32]),
    "sjb200_stage1_finish": (_i32, [_vp, _pu32, _pu32, _pi32]),
    "sjb200_stage1_device": (_i32, [_vp, _vp, _u64, _vp, _u64, _pu32, _pi32, _u32]),
    "sjb200_sync": (_i32, [_vp]),
    "sjb200_last_elapsed_ms": (C.c_float, [_vp]),
    "sjb200_launch_count": (_u64, [_vp]),
    "sjb200_pinned_alloc": (_i32, [_u64, C.POINTER(_vp)]),
    "sjb200_pinned_free": (_i32, [_vp]),
    "sjb200_device_alloc": (_i32, [_vp, _u64, C.POINTER(_vp)]),
    "sjb200_device_free": (_i32, [_vp, _vp]),
    "sjb200_copy_to_device": (_i32, [_vp, _vp, _vp, _u64]),
    "sjb200_copy_to_host": (_i32, [_vp, _vp, _vp, _u64]),
    "sjb200_batch_split_device": (_i32, [_vp, _vp, _u64, _u64, _pu64, _u32, _pu32]),
    "sjb200_batch_split_host": (_i32, [_vp, _u64, _u64, _pu64, _u32, _pu32]),
    "sjb200_batch_run_device_async": (_i32, [_vp, _vp, _pu64, _u32, _u32, _vp, _pu64, _u64, _vp, _u32]),
    "sjb200_batch_run_device": (_i32, [_vp, _vp, _pu64, _u32, _u32, _vp, _pu64, _u64, _pu32, _pi32, _pi32, _u32]),
    "sjb200_batch_unique_id": (_i32, [_vp]),
    "sjb200_batch_create": (_i32, [_i32, _pi32, _u64, _u64, _u32, _u32, C.POINTER(_vp)]),
    "sjb200_batch_create_rank": (_i32, [_i32, _i32, _i32, _vp, _u64, _u64, _u32, _u32, C.POINTER(_vp)]),
    "sjb200_batch_destroy": (_i32, [_vp]),
    "sjb200_batch_local_gpus": (_i32, [_vp]),
    "sjb200_batch_ctx": (_i32, [_vp, _i32, C.POINTER(_vp)]),
    "sjb200_batch_run": (_i32, [_vp, _vp, _u64, _vp, _u64, _pu64, _pu64, _pu32, _pi32, _u32, _pu32, _pi32, _u32]),
    "sjb200_batch_plan_resident": (_i32, [_vp, _i32, _vp, _u64, _pu64, _pu64, _pu32]),
    "sjb200_batch_run_resident_async": (_i32, [_vp, C.POINTER(_vp), _pu64, _u32]),
    "sjb200_batch_finish": (_i32, [_vp, _pi32, _pi32]),
    "sjb200_stage2": (_i32, [_vp, _vp, _u64, _vp, _u64, _pu64, _pu64, _pu64]),
    "sjb200_stage2_tape_device_async": (_i32, [_vp, _vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _u64, _vp]),
    "sjb200_stage2_primitives_device_async": (_i32, [_vp, _vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _u64, _vp]),
    "sjb200_stage2_stream_device_async": (_i32, [_vp, _vp, _u64, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _u64, _vp, _vp, _vp, _vp]),
    "sjb200_stage2_stream": (_i32, [_vp, _vp, _u64, _vp, _u64, _vp, _vp, _vp, _u64, _pu64, _pu64, _pu64, _pu64, _pu64]),
    "sjb200_at_pointers_device_async": (_i32, [_vp, _vp, _u64, _vp, _u64, _vp, _vp, _u64, _vp, _pu64, _u64, _vp, _vp, _vp]),
    "sjb200_stage2_stream_at_pointers": (_i32, [_vp, _vp, _pu64, _u64, _vp, _vp, _vp, _u64, _vp, _u64, _pu64, _pu64]),
    "sjb200_string_columns_device_async": (_i32, [_vp, _vp, _vp, _u64, _u64, _vp, _u64, _vp, _vp, _u64, _vp]),
}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m mojo_simdjson_b200.build` "
                "(there is no CPU fallback for the stage-1 path)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)  # AttributeError if the library does not export what the header declares
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib
