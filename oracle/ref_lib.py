"""ctypes binding of oracle/_ref/libdietgpu_ref.so -- the UNMODIFIED reference
(facebookresearch/dietgpu) compiled for sm_100a by oracle/build_ref.sh, behind
the C veneer oracle/ref_harness.cu.  TEST / BASELINE infrastructure only: used
by tests/golden/make_ref_golden.py and by `bench.py --impl reference`.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libdietgpu_ref.so")


def available() -> bool:
    return os.path.exists(LIB_PATH)


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(LIB_PATH)
        u32, i32, vp, sz = C.c_uint32, C.c_int, C.c_void_p, C.c_size_t
        L.ref_ans_max_compressed_size.restype = u32
        L.ref_ans_max_compressed_size.argtypes = [u32]
        L.ref_float_max_compressed_size.restype = u32
        L.ref_float_max_compressed_size.argtypes = [i32, u32]
        L.ref_ans_encode_pointer.restype = i32
        L.ref_ans_encode_pointer.argtypes = [vp, sz, i32, i32, u32, vp, vp, vp, vp, vp]
        L.ref_ans_decode_pointer.restype = i32
        L.ref_ans_decode_pointer.argtypes = [vp, sz, i32, i32, u32, vp, vp, vp, vp, vp, vp]
        L.ref_float_compress.restype = i32
        L.ref_float_compress.argtypes = [vp, sz, i32, i32, i32, u32, vp, vp, vp, vp, vp]
        L.ref_float_decompress.restype = i32
        L.ref_float_decompress.argtypes = [vp, sz, i32, i32, i32, i32, u32, vp, vp, vp, vp, vp, vp]
        _lib = L
    return _lib


def _parr(ptrs):
    return (C.c_void_p * len(ptrs))(*[C.c_void_p(int(p)) for p in ptrs])


def _uarr(vals):
    return (C.c_uint32 * len(vals))(*[int(v) for v in vals])


class RefCodec:
    """Drives the reference through torch tensors (device memory only)."""

    def __init__(self, temp_bytes: int, device="cuda"):
        import torch
        self.torch = torch
        self.temp = torch.empty(temp_bytes, dtype=torch.uint8, device=device)

    def _stream(self):
        return self.torch.cuda.current_stream().cuda_stream

    def ans_encode(self, ts, comp, sizes, pb=10, checksum=False):
        n = len(ts)
        row = comp.size(1)
        return lib().ref_ans_encode_pointer(
            self.temp.data_ptr(), self.temp.numel(), pb, int(checksum), n,
            _parr([t.data_ptr() for t in ts]), _uarr([t.numel() * t.element_size() for t in ts]),
            _parr([comp.data_ptr() + i * row for i in range(n)]), sizes.data_ptr(), self._stream())

    def ans_decode(self, comps, outs, status=None, sizes=None, pb=10, checksum=False):
        n = len(comps)
        return lib().ref_ans_decode_pointer(
            self.temp.data_ptr(), self.temp.numel(), pb, int(checksum), n,
            _parr([t.data_ptr() for t in comps]), _parr([t.data_ptr() for t in outs]),
            _uarr([t.numel() * t.element_size() for t in outs]),
            status.data_ptr() if status is not None else None,
            sizes.data_ptr() if sizes is not None else None, self._stream())

    def float_compress(self, ft, ts, comp, sizes, pb=10, checksum=False):
        n = len(ts)
        row = comp.size(1)
        return lib().ref_float_compress(
            self.temp.data_ptr(), self.temp.numel(), ft, pb, int(checksum), n,
            _parr([t.data_ptr() for t in ts]), _uarr([t.numel() for t in ts]),
            _parr([comp.data_ptr() + i * row for i in range(n)]), sizes.data_ptr(), self._stream())

    def float_decompress(self, ft, comps, outs, status=None, sizes=None, pb=10, checksum=False, aligned16=True):
        n = len(comps)
        return lib().ref_float_decompress(
            self.temp.data_ptr(), self.temp.numel(), ft, pb, int(checksum), int(aligned16), n,
            _parr([t.data_ptr() for t in comps]), _parr([t.data_ptr() for t in outs]),
            _uarr([t.numel() for t in outs]),
            status.data_ptr() if status is not None else None,
            sizes.data_ptr() if sizes is not None else None, self._stream())
