"""ctypes binding of the C ABI declared in include/zeekstd_b200.h.

The product library is zeekstd_b200/libzeekstd_b200.so (nvcc, sm_100a).  There is NO fallback:
if it is missing, or no CUDA device is usable, loading / context creation raises.
Tests may load another build of the SAME sources explicitly by path (tests/emul: device code
interpreted on the CPU) through `load(path)`; nothing in this package ever does so on its own.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import (POINTER, c_char_p, c_float, c_int32, c_int64, c_size_t, c_uint8, c_uint32, c_uint64,
                    c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
PRODUCT_SO = os.path.join(_HERE, "libzeekstd_b200.so")

u8p = POINTER(c_uint8)
u32p = POINTER(c_uint32)
u64p = POINTER(c_uint64)
i32p = POINTER(c_int32)


class CompressionProgress(ctypes.Structure):
    _fields_ = [("in_progress", c_size_t), ("out_progress", c_size_t)]


class EpilogueProgress(ctypes.Structure):
    _fields_ = [("out_progress", c_size_t), ("data_left", c_size_t)]


SET_OFFSET_FN = ctypes.CFUNCTYPE(c_int64, c_void_p, c_int32, c_int64)
READ_FN = ctypes.CFUNCTYPE(c_int64, c_void_p, u8p, c_size_t)
WRITE_FN = ctypes.CFUNCTYPE(c_int32, c_void_p, u8p, c_size_t)
FLUSH_FN = ctypes.CFUNCTYPE(c_int32, c_void_p)


class Seekable(ctypes.Structure):
    _fields_ = [("user", c_void_p), ("set_offset", SET_OFFSET_FN), ("read", READ_FN)]


_SIGS = {
    "zk_error_name": (c_char_p, [c_int32]),
    "zk_version": (c_char_p, []),
    "zk_last_cuda_error": (c_char_p, []),
    "zk_ctx_create": (c_int32, [c_int32, c_uint32, POINTER(c_void_p)]),
    "zk_ctx_destroy": (None, [c_void_p]),
    "zk_ctx_kernel_launches": (c_uint64, [c_void_p]),
    "zk_ctx_last_device_ms": (c_float, [c_void_p]),
    "zk_compress_bound": (c_size_t, [c_size_t, c_uint32]),
    "zk_ctx_profile": (None, [c_void_p, c_int32]),
    "zk_ctx_profile_read": (None, [c_void_p, POINTER(c_float), u32p]),
    "zk_ctx_set_cparameter": (c_int32, [c_void_p, c_int32, c_int32]),
    "zk_ctx_set_dparameter": (c_int32, [c_void_p, c_int32, c_int32]),
    "zk_compress_frames": (c_int32, [c_void_p, c_void_p, c_size_t, c_uint32, c_int32, c_int32, c_void_p, c_size_t,
                                     u32p, u32p, c_uint32, u32p, POINTER(c_size_t)]),
    "zk_decompress_frames": (c_int32, [c_void_p, c_void_p, u64p, u64p, c_uint32, c_void_p, c_int32, i32p]),
    "zk_decompress_frames_upto": (c_int32, [c_void_p, c_void_p, u64p, u64p, c_uint32, c_void_p, u32p, c_int32, i32p]),
    "zk_compress_frames_prefix": (c_int32, [c_void_p, c_void_p, c_size_t, c_uint32, c_int32, c_int32, c_void_p, c_size_t, c_void_p, c_size_t,
                                            u32p, u32p, c_uint32, u32p, POINTER(c_size_t)]),
    "zk_decompress_frames_prefix": (c_int32, [c_void_p, c_void_p, u64p, u64p, c_uint32, c_void_p, u32p, c_int32, i32p, c_void_p, c_size_t]),
    "zk_compress_frames_dev": (c_int32, [c_void_p, c_void_p, c_size_t, c_uint32, c_int32, c_int32, c_void_p, c_size_t,
                                         u32p, u32p, c_uint32, u32p, POINTER(c_size_t), c_void_p]),
    "zk_decompress_frames_dev": (c_int32, [c_void_p, c_void_p, u64p, u64p, c_uint32, c_void_p, c_int32, i32p,
                                           c_void_p]),
    # seek table
    "zk_seek_table_new": (c_void_p, []),
    "zk_seek_table_free": (None, [c_void_p]),
    "zk_seek_table_clone": (c_void_p, [c_void_p]),
    "zk_seek_table_from_bytes": (c_int32, [c_void_p, c_size_t, c_int32, POINTER(c_void_p)]),
    "zk_seek_table_log_frame": (c_int32, [c_void_p, c_uint32, c_uint32]),
    "zk_seek_table_num_frames": (c_uint32, [c_void_p]),
    "zk_seek_table_frame_index_comp": (c_uint32, [c_void_p, c_uint64]),
    "zk_seek_table_frame_index_decomp": (c_uint32, [c_void_p, c_uint64]),
    "zk_seek_table_frame_start_comp": (c_int32, [c_void_p, c_uint32, u64p]),
    "zk_seek_table_frame_start_decomp": (c_int32, [c_void_p, c_uint32, u64p]),
    "zk_seek_table_frame_end_comp": (c_int32, [c_void_p, c_uint32, u64p]),
    "zk_seek_table_frame_end_decomp": (c_int32, [c_void_p, c_uint32, u64p]),
    "zk_seek_table_frame_size_comp": (c_int32, [c_void_p, c_uint32, u64p]),
    "zk_seek_table_frame_size_decomp": (c_int32, [c_void_p, c_uint32, u64p]),
    "zk_seek_table_max_frame_size_comp": (c_uint64, [c_void_p]),
    "zk_seek_table_max_frame_size_decomp": (c_uint64, [c_void_p]),
    "zk_seek_table_size_comp": (c_uint64, [c_void_p]),
    "zk_seek_table_size_decomp": (c_uint64, [c_void_p]),
    "zk_seek_table_offsets": (c_uint32, [c_void_p, u64p, u64p, c_uint32]),
    "zk_seek_table_into_serializer": (c_void_p, [c_void_p, c_int32]),
    "zk_serializer_free": (None, [c_void_p]),
    "zk_serializer_write_into": (c_size_t, [c_void_p, c_void_p, c_size_t]),
    "zk_serializer_reset": (None, [c_void_p]),
    "zk_serializer_encoded_len": (c_size_t, [c_void_p]),
    # encoder
    "zk_encode_options_new": (c_void_p, [c_void_p]),
    "zk_encode_options_free": (None, [c_void_p]),
    "zk_encode_options_frame_size_policy": (None, [c_void_p, c_int32, c_uint32]),
    "zk_encode_options_checksum_flag": (None, [c_void_p, c_int32]),
    "zk_encode_options_compression_level": (None, [c_void_p, c_int32]),
    "zk_encode_options_into_raw_encoder": (c_int32, [c_void_p, POINTER(c_void_p)]),
    "zk_encode_options_into_encoder": (c_int32, [c_void_p, WRITE_FN, FLUSH_FN, c_void_p, POINTER(c_void_p)]),
    "zk_raw_encoder_free": (None, [c_void_p]),
    "zk_raw_encoder_compress": (c_int32, [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t,
                                          POINTER(CompressionProgress)]),
    "zk_raw_encoder_compress_with_prefix": (c_int32, [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t, c_void_p, c_size_t,
                                                      POINTER(CompressionProgress)]),
    "zk_raw_encoder_end_frame": (c_int32, [c_void_p, c_void_p, c_size_t, POINTER(EpilogueProgress)]),
    "zk_raw_encoder_seek_table": (c_void_p, [c_void_p]),
    "zk_raw_encoder_into_seek_table": (c_void_p, [c_void_p]),
    "zk_raw_encoder_reset_frame": (None, [c_void_p]),
    "zk_raw_encoder_reset_seek_table": (None, [c_void_p]),
    "zk_encoder_free": (None, [c_void_p]),
    "zk_encoder_compress": (c_int32, [c_void_p, c_void_p, c_size_t, POINTER(c_size_t)]),
    "zk_encoder_compress_with_prefix": (c_int32, [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t, POINTER(c_size_t)]),
    "zk_encoder_end_frame": (c_int32, [c_void_p, POINTER(c_size_t)]),
    "zk_encoder_flush": (c_int32, [c_void_p]),
    "zk_encoder_finish": (c_int32, [c_void_p, u64p]),
    "zk_encoder_finish_format": (c_int32, [c_void_p, c_int32, u64p]),
    "zk_encoder_written_compressed": (c_uint64, [c_void_p]),
    "zk_encoder_seek_table": (c_void_p, [c_void_p]),
    # decoder
    "zk_decode_options_new_bytes": (c_void_p, [c_void_p, c_void_p, c_size_t]),
    "zk_decode_options_new_seekable": (c_void_p, [c_void_p, Seekable]),
    "zk_decode_options_free": (None, [c_void_p]),
    "zk_decode_options_seek_table": (None, [c_void_p, c_void_p]),
    "zk_decode_options_lower_frame": (None, [c_void_p, c_uint32]),
    "zk_decode_options_upper_frame": (None, [c_void_p, c_uint32]),
    "zk_decode_options_offset": (None, [c_void_p, c_uint64]),
    "zk_decode_options_offset_limit": (None, [c_void_p, c_uint64]),
    "zk_decode_options_into_decoder": (c_int32, [c_void_p, POINTER(c_void_p)]),
    "zk_decoder_free": (None, [c_void_p]),
    "zk_decoder_decompress": (c_int32, [c_void_p, c_void_p, c_size_t, POINTER(c_size_t)]),
    "zk_decoder_decompress_with_prefix": (c_int32, [c_void_p, c_void_p, c_size_t, c_void_p, c_size_t, POINTER(c_size_t)]),
    "zk_decoder_reset": (None, [c_void_p]),
    "zk_decoder_set_lower_frame": (c_int32, [c_void_p, c_uint32, u64p]),
    "zk_decoder_set_upper_frame": (c_int32, [c_void_p, c_uint32, u64p]),
    "zk_decoder_set_offset": (c_int32, [c_void_p, c_uint64]),
    "zk_decoder_set_offset_limit": (c_int32, [c_void_p, c_uint64]),
    "zk_decoder_read_compressed": (c_uint64, [c_void_p]),
    "zk_decoder_offset": (c_uint64, [c_void_p]),
    "zk_decoder_offset_limit": (c_uint64, [c_void_p]),
    "zk_decoder_seek_table": (c_void_p, [c_void_p]),
    "zk_decoder_seek": (c_int32, [c_void_p, c_int32, c_int64, u64p]),
}

EXPORTED_SYMBOLS = sorted(_SIGS)

_libs: dict[str, ctypes.CDLL] = {}
_default: ctypes.CDLL | None = None


def load(path: str | None = None, require_all: bool = True) -> ctypes.CDLL:
    """load a build of the native library and attach prototypes. Raises if it cannot be loaded."""
    path = os.path.abspath(path or PRODUCT_SO)
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build it with `python -m zeekstd_b200.build` (nvcc, sm_100a). "
            "zeekstd_b200 has no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, (res, args) in _SIGS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            if require_all:
                raise ImportError(f"{path} does not export {name} (declared in include/zeekstd_b200.h)")
            continue
        fn.restype = res
        fn.argtypes = args
    _libs[path] = lib
    return lib


def default_lib() -> ctypes.CDLL:
    global _default
    if _default is None:
        _default = load(PRODUCT_SO)
    return _default


def set_default_lib(lib: ctypes.CDLL) -> None:
    """tests only: route the Python mirror classes to an explicitly loaded build"""
    global _default
    _default = lib
