"""Loader for libaurora_cuda.so (the C ABI of include/aurora_cuda.h).  There is no CPU fallback: a missing
library or a missing B200 raises."""
import ctypes as C
import os

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# AURORA_CUDA_LIB: developer override to load an alternate build of the same library (tools/build_variant.sh)
LIB_PATH = os.environ.get("AURORA_CUDA_LIB") or os.path.join(_HERE, "libaurora_cuda.so")

# every symbol include/aurora_cuda.h declares
EXPORTS = [
    "aurora_init", "aurora_shutdown", "aurora_device_count", "aurora_ctx_device_count", "aurora_abi_version",
    "aurora_last_error_string", "aurora_status_string", "aurora_pinned_alloc", "aurora_pinned_free",
    "aurora_lz_props_window", "aurora_lz_props_bits", "aurora_codec_opts_init", "aurora_decoded_size_batch",
    "aurora_is_match_batch", "aurora_scan_offsets", "aurora_decode_batch", "aurora_encode_bound", "aurora_encode_batch",
    "aurora_decode_batch_device", "aurora_encode_batch_device", "aurora_decoded_size_batch_device", "aurora_is_match_batch_device",
    "aurora_scan_offsets_device", "aurora_scan_decode_device", "aurora_kernel_launch_count",
]

_LIB = None


class AuroraLibraryError(ImportError):
    pass


def load():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise AuroraLibraryError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C auroralib/compression_b200/csrc).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz, i32, u32, u64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint32, C.c_uint64
    opts = C.POINTER(_abi.CodecOpts)
    L.aurora_init.restype = vp
    L.aurora_init.argtypes = [u32]
    L.aurora_shutdown.argtypes = [vp]
    L.aurora_device_count.restype = i32
    L.aurora_ctx_device_count.restype = i32
    L.aurora_ctx_device_count.argtypes = [vp]
    L.aurora_abi_version.restype = i32
    L.aurora_last_error_string.restype = C.c_char_p
    L.aurora_last_error_string.argtypes = [vp]
    L.aurora_status_string.restype = C.c_char_p
    L.aurora_status_string.argtypes = [i32]
    L.aurora_pinned_alloc.restype = vp
    L.aurora_pinned_alloc.argtypes = [sz]
    L.aurora_pinned_free.argtypes = [vp]
    L.aurora_lz_props_window.argtypes = [C.POINTER(_abi.LzProps), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    L.aurora_lz_props_bits.argtypes = [C.POINTER(_abi.LzProps), C.c_int32, C.c_int32, C.c_int32]
    L.aurora_codec_opts_init.argtypes = [opts]
    L.aurora_decoded_size_batch.restype = i32
    L.aurora_decoded_size_batch.argtypes = [vp, i32, opts, sz, vp, vp, vp, i32, vp, vp]
    L.aurora_is_match_batch.restype = i32
    L.aurora_is_match_batch.argtypes = [vp, i32, opts, sz, vp, vp, vp, vp]
    L.aurora_scan_offsets.restype = i32
    L.aurora_scan_offsets.argtypes = [vp, i32, opts, vp, u64, vp]
    L.aurora_decode_batch.restype = i32
    L.aurora_decode_batch.argtypes = [vp, i32, opts, sz, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.aurora_encode_bound.restype = u64
    L.aurora_encode_bound.argtypes = [i32, u64]
    L.aurora_encode_batch.restype = i32
    L.aurora_encode_batch.argtypes = [vp, i32, opts, sz, vp, vp, vp, vp, vp, vp, vp, vp]
    L.aurora_decode_batch_device.restype = i32
    L.aurora_decode_batch_device.argtypes = [vp, i32, i32, opts, sz, vp, u64, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.aurora_encode_batch_device.restype = i32
    L.aurora_encode_batch_device.argtypes = [vp, i32, i32, opts, sz, vp, u64, vp, vp, vp, vp, vp, vp, vp, vp]
    L.aurora_decoded_size_batch_device.restype = i32
    L.aurora_decoded_size_batch_device.argtypes = [vp, i32, i32, opts, sz, vp, u64, vp, vp, i32, vp, vp, vp]
    L.aurora_is_match_batch_device.restype = i32
    L.aurora_is_match_batch_device.argtypes = [vp, i32, i32, opts, sz, vp, vp, vp, vp, vp]
    L.aurora_scan_offsets_device.restype = i32
    L.aurora_scan_offsets_device.argtypes = [vp, i32, i32, opts, vp, u64, vp, vp]
    L.aurora_scan_decode_device.restype = i32
    L.aurora_scan_decode_device.argtypes = [vp, i32, i32, opts, vp, u64, u64, u64, sz, vp, vp, vp, vp, u64, vp, vp, vp, vp]
    L.aurora_kernel_launch_count.restype = u64
    L.aurora_kernel_launch_count.argtypes = [vp]
    _LIB = L
    return L
