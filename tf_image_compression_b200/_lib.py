"""ctypes binding of the C-ABI library (include/tic.h).  There is no CPU fallback: if libtic.so is
missing or no B200 is visible, loading / tic_create fails loudly."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libtic.so"
RC_LIB_PATH = _HERE / "librangecoder.so"

OK = 0
ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_NOMEM, ERR_UNSUPPORTED = -1, -2, -3, -4, -5
GRAPH_ENCODER, GRAPH_DECODER, GRAPH_POSTFILTER = 0, 1, 2
CONV, DECONV = 0, 1
ACT_IDENTITY, ACT_RELU = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1
U8, F32 = 0, 1
COMPUTE_FP32, COMPUTE_TENSOR_3XTF32, COMPUTE_TENSOR_TF32, COMPUTE_TENSOR_F16X3 = 0, 1, 2, 3


class LayerDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("cin", C.c_int32), ("cout", C.c_int32), ("stride", C.c_int32),
                ("act", C.c_int32), ("res_begin", C.c_int32), ("res_end", C.c_int32)]


# name -> (restype, argtypes); every symbol include/tic.h declares
SIGNATURES = {
    "tic_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "tic_destroy": (None, [C.c_void_p]),
    "tic_last_error": (C.c_char_p, [C.c_void_p]),
    "tic_create_error": (C.c_char_p, []),
    "tic_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tic_set_compute_mode": (C.c_int, [C.c_void_p, C.c_int]),
    "tic_set_chunk_patches": (C.c_int, [C.c_void_p, C.c_int]),
    "tic_set_graph": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(LayerDesc), C.c_int]),
    "tic_load_weights": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tic_set_norm": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "tic_set_quantizer": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "tic_bottleneck_shape": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tic_encode_patches": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "tic_encode_images": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "tic_decode_patches": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "tic_decode_images": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "tic_roundtrip_images": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_int, C.c_int]),
    "tic_postfilter_patches": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int]),
    "tic_postfilter_images": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int]),
    "tic_run_layers": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "tic_round_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int]),
    "tic_hist_reset": (C.c_int, [C.c_void_p]),
    "tic_hist_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "tic_hist_device_ptr": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "tic_position_sums": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int]),
    "tic_position_sums_batched": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int]),
    "tic_check_status": (C.c_int, [C.c_void_p]),
    "tic_entropy_bound": (C.c_int64, [C.c_int64]),
    "tic_entropy_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_int]),
    "tic_entropy_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                     C.c_int64, C.c_int]),
    "tic_evaluate_images": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "tic_launch_count": (C.c_int64, [C.c_void_p]),
    "tic_last_kernel_ms": (C.c_float, [C.c_void_p]),
    "tic_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "tic_profile_reset": (C.c_int, [C.c_void_p]),
    "tic_profile_read": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "tic_crc32c": (C.c_uint32, [C.c_char_p, C.c_uint64]),
    "tic_version": (C.c_char_p, []),
}

_lib = None


def load():
    """dlopen libtic.so and type every entry point.  Raises (never falls back) if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  tf_image_compression_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(str(LIB_PATH), mode=getattr(os, "RTLD_NOW", 2))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
