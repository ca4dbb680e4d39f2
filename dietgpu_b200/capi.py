"""ctypes binding of libdietgpu_b200.so (the C ABI in include/dietgpu_b200.h).

There is NO fallback: if the CUDA library has not been built (or cannot be
loaded) importing this module raises, and every call needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DIETGPU_B200_LIB selects an experiment build of the same library (tools/ only); default = the shipped one
LIB_PATH = os.environ.get("DIETGPU_B200_LIB") or os.path.join(_HERE, "libdietgpu_b200.so")

OK, ERR_INVALID_ARG, ERR_TEMP_TOO_SMALL, ERR_CUDA, ERR_CHECKSUM, ERR_TOO_LARGE = range(6)
FLOAT16, BFLOAT16, FLOAT32 = 1, 2, 3

# every symbol include/dietgpu_b200.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "dgb_version", "dgb_error_string", "dgb_last_cuda_error",
    "dgb_ans_max_compressed_size", "dgb_float_max_compressed_size",
    "dgb_ans_encode_temp_bytes", "dgb_ans_decode_temp_bytes",
    "dgb_float_compress_temp_bytes", "dgb_float_decompress_temp_bytes",
    "dgb_ans_encode_pointer", "dgb_ans_encode_stride", "dgb_ans_encode_split_size",
    "dgb_ans_decode_pointer", "dgb_ans_decode_stride", "dgb_ans_decode_split_size",
    "dgb_ans_get_compressed_info",
    "dgb_float_compress_pointer", "dgb_float_compress_split_size",
    "dgb_float_decompress_pointer", "dgb_float_decompress_split_size",
    "dgb_float_get_compressed_info",
    "dgb_copy_async", "dgb_copy_rows_async", "dgb_archives_pull",
    "dgb_set_option", "dgb_get_option", "dgb_set_thread_option", "dgb_clear_thread_options", "dgb_kernel_times",
]


class DietGpuError(RuntimeError):
    def __init__(self, code: int, what: str):
        super().__init__(f"dietgpu_b200: {what} failed: {error_string(code)} (code {code}"
                         + (f", cudaError {lib().dgb_last_cuda_error()}" if code == ERR_CUDA else "") + ")")
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C dietgpu_b200/csrc`. dietgpu_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    u32, i32, vp, sz = C.c_uint32, C.c_int, C.c_void_p, C.c_size_t
    L.dgb_version.restype = i32
    L.dgb_error_string.restype = C.c_char_p
    L.dgb_error_string.argtypes = [i32]
    L.dgb_last_cuda_error.restype = i32
    L.dgb_ans_max_compressed_size.restype = u32
    L.dgb_ans_max_compressed_size.argtypes = [u32]
    L.dgb_float_max_compressed_size.restype = u32
    L.dgb_float_max_compressed_size.argtypes = [i32, u32]
    L.dgb_ans_encode_temp_bytes.restype = sz
    L.dgb_ans_encode_temp_bytes.argtypes = [u32, u32]
    L.dgb_ans_decode_temp_bytes.restype = sz
    L.dgb_ans_decode_temp_bytes.argtypes = [u32]
    L.dgb_float_compress_temp_bytes.restype = sz
    L.dgb_float_compress_temp_bytes.argtypes = [i32, u32, u32]
    L.dgb_float_decompress_temp_bytes.restype = sz
    L.dgb_float_decompress_temp_bytes.argtypes = [i32, u32, u32]
    L.dgb_ans_encode_pointer.restype = i32
    L.dgb_ans_encode_pointer.argtypes = [vp, sz, i32, i32, u32, vp, vp, vp, vp, vp, vp]
    L.dgb_ans_encode_stride.restype = i32
    L.dgb_ans_encode_stride.argtypes = [vp, sz, i32, i32, u32, vp, u32, u32, vp, vp, u32, vp, vp]
    L.dgb_ans_encode_split_size.restype = i32
    L.dgb_ans_encode_split_size.argtypes = [vp, sz, i32, i32, u32, vp, vp, vp, vp, u32, vp, vp]
    L.dgb_ans_decode_pointer.restype = i32
    L.dgb_ans_decode_pointer.argtypes = [vp, sz, i32, i32, u32, vp, vp, vp, vp, vp, vp, vp]
    L.dgb_ans_decode_stride.restype = i32
    L.dgb_ans_decode_stride.argtypes = [vp, sz, i32, i32, u32, vp, u32, vp, u32, u32, vp, vp, vp, vp]
    L.dgb_ans_decode_split_size.restype = i32
    L.dgb_ans_decode_split_size.argtypes = [vp, sz, i32, i32, u32, vp, vp, vp, vp, vp, vp, vp]
    L.dgb_ans_get_compressed_info.restype = i32
    L.dgb_ans_get_compressed_info.argtypes = [vp, sz, vp, i32, u32, vp, vp, vp]
    L.dgb_float_compress_pointer.restype = i32
    L.dgb_float_compress_pointer.argtypes = [vp, sz, i32, i32, i32, u32, vp, vp, vp, vp, vp]
    L.dgb_float_compress_split_size.restype = i32
    L.dgb_float_compress_split_size.argtypes = [vp, sz, i32, i32, i32, u32, vp, vp, vp, u32, vp, vp]
    L.dgb_float_decompress_pointer.restype = i32
    L.dgb_float_decompress_pointer.argtypes = [vp, sz, i32, i32, i32, u32, vp, vp, vp, vp, vp, vp, vp]
    L.dgb_float_decompress_split_size.restype = i32
    L.dgb_float_decompress_split_size.argtypes = [vp, sz, i32, i32, i32, u32, vp, vp, vp, vp, vp, vp, vp]
    L.dgb_float_get_compressed_info.restype = i32
    L.dgb_float_get_compressed_info.argtypes = [vp, sz, vp, i32, u32, vp, vp, vp, vp]
    L.dgb_set_option.restype = i32
    L.dgb_set_option.argtypes = [C.c_char_p, i32]
    L.dgb_get_option.restype = i32
    L.dgb_get_option.argtypes = [C.c_char_p, C.POINTER(i32)]
    L.dgb_set_thread_option.restype = i32
    L.dgb_set_thread_option.argtypes = [C.c_char_p, i32]
    L.dgb_clear_thread_options.restype = i32
    L.dgb_clear_thread_options.argtypes = []
    L.dgb_copy_async.restype = i32
    L.dgb_copy_async.argtypes = [vp, vp, sz, vp]
    L.dgb_copy_rows_async.restype = i32
    L.dgb_copy_rows_async.argtypes = [vp, sz, vp, sz, sz, sz, vp]
    L.dgb_archives_pull.restype = i32
    L.dgb_archives_pull.argtypes = [i32, u32, vp, vp, vp, vp, vp]
    L.dgb_kernel_times.restype = i32
    L.dgb_kernel_times.argtypes = [vp, vp, i32]
    _lib = L
    return L


def error_string(code: int) -> str:
    return lib().dgb_error_string(code).decode()


def check(code: int, what: str) -> None:
    if code != OK:
        raise DietGpuError(code, what)


def set_option(name: str, value: int) -> None:
    check(lib().dgb_set_option(name.encode(), int(value)), f"set_option({name})")


def set_thread_option(name: str, value: int) -> None:
    """Override for codec calls made by the calling thread only (dgb_set_thread_option)."""
    check(lib().dgb_set_thread_option(name.encode(), int(value)), f"set_thread_option({name})")


def clear_thread_options() -> None:
    check(lib().dgb_clear_thread_options(), "clear_thread_options")


def get_option(name: str) -> int:
    v = C.c_int()
    check(lib().dgb_get_option(name.encode(), C.byref(v)), f"get_option({name})")
    return v.value


def ptr_array(ptrs):
    return (C.c_void_p * len(ptrs))(*[C.c_void_p(int(p)) for p in ptrs])


def u32_array(vals):
    return (C.c_uint32 * len(vals))(*[int(v) for v in vals])


# slot numbers are C ABI: 2 and 5 are retired and always report 0
KERNEL_SLOTS = ["stats", "encode", "retired_2", "decode", "checksum", "retired_5", "pull"]


def kernel_times():
    """(ms, launches) per kernel slot since the last call (option "timing" must be 1)."""
    ms = (C.c_float * len(KERNEL_SLOTS))()
    cnt = (C.c_int * len(KERNEL_SLOTS))()
    check(lib().dgb_kernel_times(ms, cnt, len(KERNEL_SLOTS)), "kernel_times")
    return {k: (ms[i], cnt[i]) for i, k in enumerate(KERNEL_SLOTS)}
