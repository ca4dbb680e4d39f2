"""CPU tests of the boundary: the C-ABI library loads here (no GPU), exports every symbol the header
declares, its size functions agree with the oracle, and misuse returns error codes (never aborts)."""
import ctypes as C
import os
import re

import pytest

from dietgpu_b200 import capi
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "dietgpu_b200.h")).read()
    declared = set(re.findall(r"\b(dgb_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(capi.SYMBOLS), declared ^ set(capi.SYMBOLS)
    L = capi.lib()
    for s in declared:
        assert getattr(L, s) is not None
    assert L.dgb_version() == 1


def test_size_functions_match_oracle():
    L = capi.lib()
    for n in (0, 1, 4095, 4096, 4097, 1 << 20, 4 << 20, 123456789):
        assert L.dgb_ans_max_compressed_size(n) == O.ans_max_compressed_size(n)
        for ft in (capi.FLOAT16, capi.BFLOAT16, capi.FLOAT32):
            assert L.dgb_float_max_compressed_size(ft, n) == O.float_max_compressed_size(ft, n)
    assert L.dgb_float_max_compressed_size(7, 100) == 0  # unknown float type


def test_temp_sizes_are_sane():
    L = capi.lib()
    a = L.dgb_ans_encode_temp_bytes(64, 4 << 20)
    f = L.dgb_float_compress_temp_bytes(capi.BFLOAT16, 64, 2 << 20)
    # no per-element scratch any more (the coder reads the raw words; round 1 kept a coded-byte row per
    # member): both are the spill area + tables, well below the input size
    assert 0 < a < (100 << 20) and 0 < f < (100 << 20)
    assert L.dgb_ans_decode_temp_bytes(64) < (1 << 20)
    # small batches need small scratch (the reference's scratch scales with the batch)
    assert L.dgb_ans_encode_temp_bytes(1, 4096) < (1 << 20)
    assert L.dgb_float_compress_temp_bytes(capi.FLOAT16, 3, 10000) < (1 << 20)


def test_error_codes_and_option_names_without_gpu():
    L = capi.lib()
    assert capi.error_string(capi.OK) == "ok"
    assert "temporary" in capi.error_string(capi.ERR_TEMP_TOO_SMALL)
    # empty batches are no-ops and need no device
    assert L.dgb_ans_encode_pointer(None, 0, 10, 0, 0, None, None, None, None, None, None) == capi.OK
    assert L.dgb_ans_decode_pointer(None, 0, 10, 0, 0, None, None, None, None, None, None, None) == capi.OK
    # invalid arguments are reported, not asserted
    one = (C.c_void_p * 1)(C.c_void_p(256))
    sz = (C.c_uint32 * 1)(16)
    assert L.dgb_ans_encode_pointer(None, 0, 12, 0, 1, one, sz, None, one, None, None) == capi.ERR_INVALID_ARG
    assert L.dgb_float_compress_pointer(None, 0, 9, 10, 0, 1, one, sz, one, None, None) == capi.ERR_INVALID_ARG
    assert L.dgb_ans_encode_pointer(None, 0, 10, 0, 1, one, sz, None, one, None, None) == capi.ERR_TEMP_TOO_SMALL
    assert L.dgb_set_option(b"no_such_option", 1) == capi.ERR_INVALID_ARG
    capi.set_option("inline_members", 1)
    assert capi.get_option("inline_members") == 1
    # retired kernel variants: their options are unknown names now
    for name in ("encode_fused", "decode_fused", "fused_stage", "fused_stats_every", "fused_chunk_blocks",
                 "stats_stage", "stats_stage_kb", "encode_k2_ctas", "first_part_pct", "last_part_pct"):
        assert L.dgb_set_option(name.encode(), 1) == capi.ERR_INVALID_ARG, name
        v = C.c_int(0)
        assert L.dgb_get_option(name.encode(), C.byref(v)) == capi.ERR_INVALID_ARG, name


def test_product_does_not_import_oracle():
    # the shipped package must never route through the CPU oracle
    pkg = os.path.join(ROOT, "dietgpu_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), f"{f} mentions the oracle"


def test_ops_raise_without_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import dietgpu_b200 as dg

    with pytest.raises(RuntimeError):
        dg.compress_data(False, [torch.zeros(16, dtype=torch.uint8)])


def test_thread_options_override_only_their_thread():
    # dgb_set_thread_option: a per-thread copy of the tuning set; other threads keep the process-wide one
    import threading

    from dietgpu_b200 import capi

    base = capi.get_option("encode_warps")
    seen = {}

    def worker():
        capi.set_thread_option("encode_warps", base + 3)
        seen["worker"] = capi.get_option("encode_warps")
        capi.set_option("decode_warps", capi.get_option("decode_warps"))  # process-wide set still works from here
        capi.clear_thread_options()
        seen["worker_cleared"] = capi.get_option("encode_warps")

    t = threading.Thread(target=worker)
    t.start()
    t.join()
    assert seen == {"worker": base + 3, "worker_cleared": base}
    assert capi.get_option("encode_warps") == base
    with pytest.raises(capi.DietGpuError):
        capi.set_thread_option("no_such_option", 1)
