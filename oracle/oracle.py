"""ctypes binding of the CPU oracle (oracle/dietgpu_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  The product package
(dietgpu_b200/) never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libdietgpu_oracle.so")

F16, BF16, F32 = 1, 2, 3
OK, ERR_BAD_MAGIC, ERR_BAD_PROBBITS, ERR_CAPACITY, ERR_CHECKSUM, ERR_BAD_FLOAT_TYPE, ERR_CORRUPT = range(7)


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "dietgpu_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "libdietgpu_oracle.so"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        u32, i32, vp = C.c_uint32, C.c_int, C.c_void_p
        L.dgo_ans_overhead.restype = u32
        L.dgo_ans_overhead.argtypes = [u32]
        L.dgo_ans_max_compressed_size.restype = u32
        L.dgo_ans_max_compressed_size.argtypes = [u32]
        L.dgo_float_noncomp_bytes.restype = u32
        L.dgo_float_noncomp_bytes.argtypes = [i32, u32]
        L.dgo_float_max_compressed_size.restype = u32
        L.dgo_float_max_compressed_size.argtypes = [i32, u32]
        L.dgo_histogram.argtypes = [vp, u32, vp]
        L.dgo_checksum.restype = u32
        L.dgo_checksum.argtypes = [vp, u32]
        L.dgo_normalize.argtypes = [vp, u32, i32, vp]
        L.dgo_ans_encode.restype = u32
        L.dgo_ans_encode.argtypes = [vp, u32, i32, i32, vp, vp]
        L.dgo_ans_info.restype = i32
        L.dgo_ans_info.argtypes = [vp] + [vp] * 5
        L.dgo_ans_decode.restype = i32
        L.dgo_ans_decode.argtypes = [vp, i32, i32, vp, u32, vp]
        L.dgo_float_compress.restype = u32
        L.dgo_float_compress.argtypes = [i32, vp, u32, i32, i32, vp]
        L.dgo_float_info.restype = i32
        L.dgo_float_info.argtypes = [vp, vp, vp, vp]
        L.dgo_float_decompress.restype = i32
        L.dgo_float_decompress.argtypes = [i32, vp, i32, i32, vp, u32, vp]
        L.dgo_div_magic.argtypes = [u32, vp, vp]
        L.dgo_batch_roundtrip.restype = i32
        L.dgo_batch_roundtrip.argtypes = [i32, vp, vp, u32, i32, vp, vp, vp, vp]
        L.dgo_num_threads.restype = i32
        L.dgo_set_threads.argtypes = [i32]
        _lib = L
    return _lib


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _bytes(a) -> np.ndarray:
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(-1)


def ans_max_compressed_size(n: int) -> int:
    return lib().dgo_ans_max_compressed_size(n)


def float_max_compressed_size(ft: int, n: int) -> int:
    return lib().dgo_float_max_compressed_size(ft, n)


def ans_overhead(nb: int) -> int:
    return lib().dgo_ans_overhead(nb)


def float_noncomp_bytes(ft: int, n: int) -> int:
    return lib().dgo_float_noncomp_bytes(ft, n)


def histogram(data) -> np.ndarray:
    d = _bytes(data)
    h = np.zeros(256, np.uint32)
    lib().dgo_histogram(_ptr(d), d.size, _ptr(h))
    return h


def checksum(data, nbytes: int | None = None) -> int:
    d = _bytes(data)
    return lib().dgo_checksum(_ptr(d), d.size if nbytes is None else nbytes)


def normalize(hist, total: int, pb: int) -> np.ndarray:
    h = np.ascontiguousarray(hist, np.uint32)
    pdf = np.zeros(256, np.uint32)
    lib().dgo_normalize(_ptr(h), total, pb, _ptr(pdf))
    return pdf


def div_magic(pdf: int):
    m, s = C.c_uint32(), C.c_uint32()
    lib().dgo_div_magic(pdf, C.byref(m), C.byref(s))
    return m.value, s.value


def ans_encode(data, pb: int = 10, use_checksum: bool = False, hist=None) -> np.ndarray:
    d = _bytes(data)
    out = np.zeros(ans_max_compressed_size(d.size) + 1024, np.uint8)
    hp = None if hist is None else _ptr(np.ascontiguousarray(hist, np.uint32))
    n = lib().dgo_ans_encode(_ptr(d), d.size, pb, int(use_checksum), hp, _ptr(out))
    return out[:n].copy()


def ans_info(arch) -> dict:
    a = _bytes(arch)
    size, unc, cks = C.c_uint32(), C.c_uint32(), C.c_uint32()
    pb, hc = C.c_int(), C.c_int()
    rc = lib().dgo_ans_info(_ptr(a), C.byref(size), C.byref(unc), C.byref(cks), C.byref(pb), C.byref(hc))
    return dict(rc=rc, size=size.value, uncompressed=unc.value, checksum=cks.value,
                prob_bits=pb.value, has_checksum=bool(hc.value))


def ans_decode(arch, pb: int = 10, capacity: int | None = None, verify_checksum: bool = False):
    a = _bytes(arch)
    info = ans_info(a)
    cap = info["uncompressed"] if capacity is None else capacity
    out = np.zeros(max(cap, 1), np.uint8)
    got = C.c_uint32()
    rc = lib().dgo_ans_decode(_ptr(a), pb, int(verify_checksum), _ptr(out), cap, C.byref(got))
    return rc, out[:min(cap, got.value)].copy(), got.value


_WORD = {F16: np.uint16, BF16: np.uint16, F32: np.uint32}


def float_compress(ft: int, words, pb: int = 10, use_checksum: bool = False) -> np.ndarray:
    w = np.ascontiguousarray(words).view(_WORD[ft]).reshape(-1)
    out = np.zeros(float_max_compressed_size(ft, w.size) + 1024, np.uint8)
    n = lib().dgo_float_compress(ft, _ptr(w), w.size, pb, int(use_checksum), _ptr(out))
    return out[:n].copy()


def float_info(arch) -> dict:
    a = _bytes(arch)
    n, cks = C.c_uint32(), C.c_uint32()
    ft = C.c_int()
    rc = lib().dgo_float_info(_ptr(a), C.byref(n), C.byref(ft), C.byref(cks))
    return dict(rc=rc, size=n.value, float_type=ft.value, checksum=cks.value)


def float_decompress(ft: int, arch, pb: int = 10, capacity: int | None = None,
                     verify_checksum: bool = False):
    a = _bytes(arch)
    info = float_info(a)
    cap = info["size"] if capacity is None else capacity
    out = np.zeros(max(cap, 1), _WORD[ft])
    got = C.c_uint32()
    rc = lib().dgo_float_decompress(ft, _ptr(a), pb, int(verify_checksum), _ptr(out), cap, C.byref(got))
    return rc, out[:min(cap, got.value)].copy(), got.value


def batch_roundtrip(ft: int, arrays, pb: int = 10):
    """Whole-batch encode then decode with every phase spread over all host cores (the CPU baseline
    of bench.py).  ft: 0 = raw bytes (uint8 arrays), else F16/BF16 (uint16 arrays) / F32 (uint32).
    Returns (archives, decoded arrays, encode seconds, decode seconds)."""
    n = len(arrays)
    arrs = [np.ascontiguousarray(a) for a in arrays]
    sizes = np.array([a.size for a in arrs], dtype=np.uint32)
    caps = [float_max_compressed_size(ft, int(k)) if ft else ans_max_compressed_size(int(k)) for k in sizes]
    archs = [np.empty(c, dtype=np.uint8) for c in caps]
    outs = [np.empty_like(a) for a in arrs]
    P = C.c_void_p * n
    in_p = P(*[a.ctypes.data for a in arrs])
    ar_p = P(*[a.ctypes.data for a in archs])
    out_p = P(*[a.ctypes.data for a in outs])
    asz = np.zeros(n, dtype=np.uint32)
    t = (C.c_double * 2)()
    rc = lib().dgo_batch_roundtrip(ft, in_p, _ptr(sizes), n, pb, ar_p, _ptr(asz), out_p, t)
    assert rc == 0, f"dgo_batch_roundtrip: error {rc}"
    return [a[:int(k)] for a, k in zip(archs, asz)], outs, t[0], t[1]


def num_threads() -> int:
    return lib().dgo_num_threads()


def set_threads(n: int) -> None:
    lib().dgo_set_threads(n)


# ---- archive dissection helpers used by the parity tests (field-wise compare,
# masking the bits the reference leaves undefined, SURVEY B3) ----

def parse_ans(arch) -> dict:
    a = _bytes(arch)
    hdr = a[:32].view(np.uint32)
    nb = int(hdr[1])
    pdf = a[32:544].view(np.uint16).copy()
    states = a[544:544 + 128 * nb].view(np.uint32).reshape(nb, 32).copy()
    o = 544 + 128 * nb
    bw = a[o:o + 8 * nb].view(np.uint32).reshape(nb, 2).copy()
    o += 8 * ((nb + 1) // 2 * 2)
    data = a[o:o + 2 * int(hdr[3])].view(np.uint16)
    streams = [data[int(off):int(off) + int(x & 0xffff)].copy() for x, off in bw]
    return dict(magic=int(hdr[0]), num_blocks=nb, uncompressed=int(hdr[2]), total_words=int(hdr[3]),
                prob_bits=int(hdr[4] & 0xf), use_checksum=bool(hdr[4] & 0x10), checksum=int(hdr[5]),
                pdf=pdf, states=states, block_words=bw, streams=streams,
                size=o + 2 * int(hdr[3]))


def assert_same_ans(mine, ref, what: str = "") -> None:
    """Semantic equality of two ANS archives: every defined field and every block's stream equal;
    only the ORDER of the streams inside the data section (blockWords[k].y) may differ, since the
    decoder addresses streams through those offsets.  Total size must match to the byte."""
    a, b = parse_ans(mine), parse_ans(ref)
    for k in ("magic", "num_blocks", "uncompressed", "total_words", "prob_bits", "use_checksum", "size"):
        assert a[k] == b[k], f"{what}: field {k}: {a[k]} != {b[k]}"
    if b["use_checksum"]:
        assert a["checksum"] == b["checksum"], f"{what}: checksum"
    assert np.array_equal(a["pdf"], b["pdf"]), f"{what}: pdf"
    assert np.array_equal(a["states"], b["states"]), f"{what}: lane states"
    assert np.array_equal(a["block_words"][:, 0], b["block_words"][:, 0]), f"{what}: block sizes"
    # offsets: multiples of 8 words; the non-empty streams tile the data section exactly (an empty
    # stream may sit at any offset inside it)
    if a["num_blocks"]:
        off = a["block_words"][:, 1].astype(np.int64)
        ln = (((a["block_words"][:, 0] & 0xffff).astype(np.int64) + 7) // 8) * 8
        assert np.all(off % 8 == 0), f"{what}: unaligned stream offset"
        assert np.all(off + ln <= a["total_words"]), f"{what}: stream beyond the data section"
        nz = ln > 0
        o2, l2 = off[nz], ln[nz]
        order = np.argsort(o2, kind="stable")
        starts, ends = o2[order], o2[order] + l2[order]
        if starts.size:
            assert starts[0] == 0 and np.all(starts[1:] == ends[:-1]) and ends[-1] == a["total_words"], \
                f"{what}: streams do not tile the data section"
        else:
            assert a["total_words"] == 0, f"{what}: total_words without streams"
    for i, (x, y) in enumerate(zip(a["streams"], b["streams"])):
        assert np.array_equal(x, y), f"{what}: stream of block {i}"


def defined_fields(arch, ft: int = 0) -> dict:
    """The parts of an archive that the format defines, as bytes, under stable names: exactly what
    assert_same_ans (ft = 0, a raw-byte archive) or the float comparison of the parity tests looks at.
    Streams are concatenated in block order, so their placement inside the data section does not count.
    Stored as digests, these let an archive be compared with one that is too large to keep."""
    a = _bytes(arch)
    out = {}
    if ft:
        n = int(a[4:8].view(np.uint32)[0])
        out["float_header"] = bytes(a[:8]) + bytes([int(a[8]) & 0x1F]) + bytes(a[12:16])
        if ft == F32:
            o1 = 16 + 2 * ((n + 7) // 8 * 8)
            out["float_planes"] = bytes(a[16:16 + 2 * n]) + bytes(a[o1:o1 + n])
        else:
            out["float_planes"] = bytes(a[16:16 + n])
        a = a[16 + float_noncomp_bytes(ft, n):]
    p = parse_ans(a)
    hdr = [p[k] for k in ("magic", "num_blocks", "uncompressed", "total_words", "prob_bits", "use_checksum", "size")]
    out["ans_header"] = np.array(hdr + [p["checksum"] if p["use_checksum"] else 0], np.uint32).tobytes()
    out["pdf"] = p["pdf"].tobytes()
    out["states"] = p["states"].tobytes()
    out["block_sizes"] = p["block_words"][:, 0].tobytes()
    out["streams"] = b"".join(s.tobytes() for s in p["streams"])
    return out


def assert_same_float(mine, ref, ft: int, what: str = "") -> None:
    """Float archives: header and stored planes byte-equal, ANS part semantically equal."""
    m, r = _bytes(mine), _bytes(ref)
    assert m.size == r.size, f"{what}: size {m.size} != {r.size}"
    n = int(r[4:8].view(np.uint32)[0])
    nc = float_noncomp_bytes(ft, n)
    assert np.array_equal(m[:16 + nc], r[:16 + nc]), f"{what}: float header / stored planes"
    assert_same_ans(m[16 + nc:], r[16 + nc:], what)
