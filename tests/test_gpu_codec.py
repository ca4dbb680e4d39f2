"""GPU parity tests: the CUDA path (through the C ABI, via dietgpu_b200.ops) against the CPU oracle.
Bit-exact everywhere: sizes, pdf, lane states, every block's stream and every decoded byte must equal
the oracle's.  In the default encoder the ORDER of the streams inside an archive's data section is
completion order (the format addresses streams by offset); with option encode_canonical=1 archives
equal the oracle's byte for byte, which test_canonical_layout_is_byte_exact checks."""
import numpy as np
import pytest
import torch

from conftest import exp_bytes, normal_words, zipf_bytes
from oracle import oracle as O

pytestmark = pytest.mark.gpu

KINDS = {"f16": (O.F16, torch.float16, np.uint16), "bf16": (O.BF16, torch.bfloat16, np.uint16),
         "f32": (O.F32, torch.float32, np.uint32)}


def dg():
    import dietgpu_b200

    return dietgpu_b200


def to_dev_bytes(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def words_to_tensor(w, kind):
    _, tdt, _ = KINDS[kind]
    t = torch.from_numpy(w.view(np.int16 if w.dtype == np.uint16 else np.int32).copy())
    return t.view(tdt).cuda()


def ans_roundtrip(arrays, pb, checksum=False):
    ts = [to_dev_bytes(a) for a in arrays]
    comp, sizes, _ = dg().compress_data(False, ts, checksum, prob_bits=pb)
    hs = sizes.cpu().tolist()
    rows = []
    for i, a in enumerate(arrays):
        want = O.ans_encode(a, pb, checksum)
        got = comp[i, :hs[i]].cpu().numpy()
        assert hs[i] == want.size, f"member {i}: size {hs[i]} != oracle {want.size}"
        assert hs[i] % 16 == 0  # ans/ANSTest.cu:131-135
        O.assert_same_ans(got, want, f"member {i}")
        rows.append(comp[i, :hs[i]].clone())  # exactly-truncated buffers (ans_test.py:21-26)
    outs = [torch.empty_like(t) for t in ts]
    status = torch.zeros(len(ts), dtype=torch.uint8, device="cuda")
    osz = torch.zeros(len(ts), dtype=torch.int32, device="cuda")
    dg().decompress_data(False, rows, outs, checksum, None, status, osz, prob_bits=pb)
    assert status.cpu().tolist() == [1] * len(ts)
    assert osz.cpu().tolist() == [a.size for a in arrays]
    for t, o in zip(ts, outs):
        assert torch.equal(t, o)


@pytest.mark.parametrize("pb", [9, 10, 11])
@pytest.mark.parametrize("lam", [1.0, 10.0, 100.0, 1000.0])
def test_ans_batch_pointer(pb, lam):
    # size lists of ans/ANSTest.cu:248-260 (BatchPointer), checksum on as there (:121)
    for sizes in ([1], [1, 1], [4096, 4095, 4096], [1234, 2345, 3456], [10000, 10013, 10000]):
        arrays = [exp_bytes(n, lam, 10 + i) for i, n in enumerate(sizes)]
        ans_roundtrip(arrays, pb, checksum=True)


def test_ans_zero_sized():
    # ans/ANSTest.cu:243-246 ZeroSized, alone and inside a batch
    ans_roundtrip([np.zeros(0, np.uint8)], 10)
    ans_roundtrip([exp_bytes(5000, 20, 1), np.zeros(0, np.uint8), exp_bytes(77, 5, 2)], 10, checksum=True)


def test_ans_batch_large():
    # ans/ANSTest.cu:262-275 BatchPointerLarge: 100 members of 100..10000 bytes
    rng = np.random.default_rng(3)
    sizes = rng.integers(100, 10000, 100)
    ans_roundtrip([exp_bytes(int(n), 20.0, 100 + i) for i, n in enumerate(sizes)], 10)


def test_ans_block_boundaries_and_distributions():
    arrays = []
    for n in (31, 32, 33, 4064, 4095, 4096, 4097, 8191, 8192, 8193, 65536 + 17):
        arrays.append(zipf_bytes(n, 1.0, n))
    arrays.append(np.full(10000, 7, np.uint8))                      # single symbol: pdf == 2^pb
    arrays.append(np.random.default_rng(5).integers(0, 256, 50000, dtype=np.uint8))  # incompressible
    arrays.append((np.random.default_rng(6).integers(100, 160, 30000)).astype(np.uint8))  # SURVEY B1 quirk
    for pb in (9, 10, 11):
        ans_roundtrip(arrays, pb)


def test_ans_config1_uniform_1mib():
    # BASELINE configs[0]: 1 MiB uniform random bytes, batch 1, prec 10
    a = np.random.default_rng(1234).integers(0, 256, 1 << 20, dtype=np.uint8)
    ans_roundtrip([a], 10)


def test_ans_unaligned_inputs():
    # inputs need only 4 B alignment (ans/GpuANSCodec.h:16); exercise odd offsets too
    base = to_dev_bytes(zipf_bytes(40000, 1.2, 9))
    for off in (0, 1, 3, 4, 12, 20):
        t = base[off:off + 20000]
        comp, sizes, _ = dg().compress_data(False, [t])
        n = int(sizes[0])
        want = O.ans_encode(t.cpu().numpy(), 10)
        assert n == want.size
        O.assert_same_ans(comp[0, :n].cpu().numpy(), want)
        out = torch.empty(20000 + 8, dtype=torch.uint8, device="cuda")[off % 8:][:20000]
        dg().decompress_data(False, [comp[0, :n]], [out])
        assert torch.equal(out, t)


def test_ans_decode_oracle_archives():
    # archives produced by the oracle (== reference format) decode bit-exactly
    arrays = [exp_bytes(12345, 30, 1), zipf_bytes(70000, 1.5, 2), exp_bytes(1, 1, 3)]
    for pb in (9, 10, 11):
        rows = [to_dev_bytes(O.ans_encode(a, pb)) for a in arrays]
        outs = [torch.empty(a.size, dtype=torch.uint8, device="cuda") for a in arrays]
        dg().decompress_data(False, rows, outs, prob_bits=pb)
        for a, o in zip(arrays, outs):
            assert np.array_equal(o.cpu().numpy(), a)


def test_ans_capacity_and_bad_header():
    a = exp_bytes(10000, 20, 1)
    row = to_dev_bytes(O.ans_encode(a, 10))
    bad = row.clone()
    bad[0] = 0  # break the magic
    outs = [torch.zeros(9999, dtype=torch.uint8, device="cuda"), torch.zeros(10000, dtype=torch.uint8, device="cuda"),
            torch.zeros(10000, dtype=torch.uint8, device="cuda")]
    status = torch.full((3,), 9, dtype=torch.uint8, device="cuda")
    osz = torch.zeros(3, dtype=torch.int32, device="cuda")
    dg().decompress_data(False, [row, row, bad], outs, False, None, status, osz)
    # ans/GpuANSDecode.cuh:326-341: too-small capacity -> success 0, size = required; member skipped
    assert status.cpu().tolist() == [0, 1, 0]
    assert osz.cpu().tolist() == [10000, 10000, 0]
    assert int(outs[0].sum()) == 0 and int(outs[2].sum()) == 0
    assert np.array_equal(outs[1].cpu().numpy(), a)
    # wrong precision is rejected per member rather than asserted
    status.fill_(9)
    dg().decompress_data(False, [row], [outs[1]], False, None, status[:1], osz[:1], prob_bits=11)
    assert int(status[0]) == 0


def test_ans_checksum_mismatch_detected():
    a = exp_bytes(20000, 20, 1)
    arch = O.ans_encode(a, 10, True)
    arch[20] ^= 0x5A  # stored checksum field
    out = torch.empty(a.size, dtype=torch.uint8, device="cuda")
    with pytest.raises(RuntimeError, match="checksum mismatch"):
        dg().decompress_data(False, [to_dev_bytes(arch)], [out], True)


def test_ans_split_size_api():
    # ans_test.py:100-139 split-size compress / decompress
    sizes = [4096, 8000, 12, 20000, 5]  # interior sizes multiples of 4
    arrays = [exp_bytes(n, 15, 40 + i) for i, n in enumerate(sizes)]
    flat = to_dev_bytes(np.concatenate(arrays))
    splits = torch.tensor(sizes, dtype=torch.int32)
    rows, csz, _ = dg().compress_data_split_size(False, flat, splits, True)
    for i, a in enumerate(arrays):
        O.assert_same_ans(rows[i].cpu().numpy(), O.ans_encode(a, 10, True))
    out = torch.empty_like(flat)
    status = torch.zeros(len(sizes), dtype=torch.uint8, device="cuda")
    dg().decompress_data_split_size(False, rows, out, splits, True, None, status, None)
    assert status.cpu().tolist() == [1] * len(sizes)
    assert torch.equal(out, flat)


def test_ans_stride_api():
    # ans/ANSTest.cu:277-282 BatchStride: 13 members of 8208 bytes
    import ctypes as C

    from dietgpu_b200 import capi

    n, size = 13, 8208
    stride_in = 8208 + 48
    arrays = [exp_bytes(size, 25, 60 + i) for i in range(n)]
    buf = torch.zeros(n * stride_in, dtype=torch.uint8, device="cuda")
    for i, a in enumerate(arrays):
        buf[i * stride_in:i * stride_in + size] = to_dev_bytes(a)
    L = capi.lib()
    ostride = L.dgb_ans_max_compressed_size(size)
    comp = torch.zeros(n * ostride, dtype=torch.uint8, device="cuda")
    csz = torch.zeros(n, dtype=torch.int32, device="cuda")
    tb = L.dgb_ans_encode_temp_bytes(n, size)
    temp = torch.empty(tb + 256, dtype=torch.uint8, device="cuda")
    tp = temp.data_ptr() + (-temp.data_ptr()) % 256
    st = torch.cuda.current_stream().cuda_stream
    capi.check(L.dgb_ans_encode_stride(tp, tb, 10, 1, n, buf.data_ptr(), size, stride_in, None,
                                       comp.data_ptr(), ostride, csz.data_ptr(), st), "encode_stride")
    hs = csz.cpu().tolist()
    for i, a in enumerate(arrays):
        O.assert_same_ans(comp[i * ostride:i * ostride + hs[i]].cpu().numpy(), O.ans_encode(a, 10, True))
    out = torch.zeros(n * stride_in, dtype=torch.uint8, device="cuda")
    status = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mism = (C.c_uint8 * n)()
    capi.check(L.dgb_ans_decode_stride(tp, tb, 10, 1, n, comp.data_ptr(), ostride, out.data_ptr(), stride_in,
                                       size, status.data_ptr(), None, mism, st), "decode_stride")
    assert status.cpu().tolist() == [1] * n and list(mism) == [0] * n
    assert torch.equal(out, buf)


# ------------------------------------------------------------------ floats ----

def float_roundtrip(kind, word_arrays, pb=10, checksum=False, offsets=None):
    ft, tdt, _ = KINDS[kind]
    ts = []
    for i, w in enumerate(word_arrays):
        off = 0 if offsets is None else offsets[i]
        full = words_to_tensor(np.concatenate([np.zeros(off, w.dtype), w]), kind)
        ts.append(full[off:])  # element-aligned but possibly not 16 B aligned (float/FloatTest.cu:276-282)
    comp, sizes, _ = dg().compress_data(True, ts, checksum, prob_bits=pb)
    hs = sizes.cpu().tolist()
    rows = []
    for i, w in enumerate(word_arrays):
        want = O.float_compress(ft, w, pb, checksum)
        assert hs[i] == want.size, f"member {i}: size {hs[i]} != oracle {want.size}"
        O.assert_same_float(comp[i, :hs[i]].cpu().numpy(), want, ft, f"member {i}")
        rows.append(comp[i, :hs[i]].clone())
    outs = []
    for i, t in enumerate(ts):
        off = 0 if offsets is None else (offsets[i] + 1) % 5
        outs.append(torch.empty(t.numel() + off, dtype=tdt, device="cuda")[off:])
    status = torch.zeros(len(ts), dtype=torch.uint8, device="cuda")
    osz = torch.zeros(len(ts), dtype=torch.int32, device="cuda")
    dg().decompress_data(True, rows, outs, checksum, None, status, osz, prob_bits=pb)
    assert status.cpu().tolist() == [1] * len(ts)
    assert osz.cpu().tolist() == [w.size for w in word_arrays]
    it = torch.int16 if kind != "f32" else torch.int32
    for t, o in zip(ts, outs):
        assert torch.equal(t.view(it), o.view(it))


@pytest.mark.parametrize("kind", ["f16", "bf16", "f32"])
@pytest.mark.parametrize("pb", [9, 10])
def test_float_batch(kind, pb):
    # float/FloatTest.cu:270-311: B in {1,3,16,23}, sizes 1..10000, with and without 16 B alignment
    rng = np.random.default_rng(11)
    for b in (1, 3, 16, 23):
        sizes = [int(x) for x in rng.integers(1, 10000, b)]
        arrs = [normal_words(n, kind, 10 + n) for n in sizes]
        float_roundtrip(kind, arrs, pb, checksum=True)
        float_roundtrip(kind, arrs, pb, offsets=[int(x) for x in rng.integers(0, 9, b)])


@pytest.mark.parametrize("kind", ["f16", "bf16", "f32"])
def test_float_large_batch_and_sizes(kind):
    # FloatTest LargeBatch (B = 256 > the reference's inline-parameter limit) and a 512 Ki member
    arrs = [normal_words(1000 + 7 * i, kind, i) for i in range(256)]
    float_roundtrip(kind, arrs, 10)
    float_roundtrip(kind, [normal_words(512 * 1024, kind, 5), normal_words(0, kind, 6), normal_words(1, kind, 7)], 10, checksum=True)


@pytest.mark.parametrize("kind", ["f16", "bf16"])
def test_float_relu_sparse(kind):
    # BASELINE configs[3] shape: ~50 % exact zeros
    float_roundtrip(kind, [normal_words(300000, kind, 3, relu=True) for _ in range(3)], 10)


def test_float_simple_api_shrinks():
    # float_test.py:50-92: compress_data_simple must actually shrink N(0,1) data
    for kind in ("bf16", "f16", "f32"):
        _, tdt, _ = KINDS[kind]
        ts = [words_to_tensor(normal_words(n, kind, n), kind) for n in (10000, 100000, 1000000)]
        comp = dg().compress_data_simple(True, ts, True)
        for t, c in zip(ts, comp):
            assert c.numel() < t.numel() * t.element_size()
        outs = dg().decompress_data_simple(True, comp, True)
        it = torch.int16 if kind != "f32" else torch.int32
        for t, o in zip(ts, outs):
            assert o.dtype == tdt and torch.equal(t.view(it), o.view(it))


def test_float_split_size_api():
    # float_test.py:94-178 split-size with and without 16 B alignment
    for kind in ("bf16", "f16", "f32"):
        sizes = [4096, 12345, 7, 100000]
        arrs = [normal_words(n, kind, 70 + i) for i, n in enumerate(sizes)]
        flat = words_to_tensor(np.concatenate(arrs), kind)
        splits = torch.tensor(sizes, dtype=torch.int32)
        rows, _, _ = dg().compress_data_split_size(True, flat, splits, True)
        ft = KINDS[kind][0]
        for r, a in zip(rows, arrs):
            O.assert_same_float(r.cpu().numpy(), O.float_compress(ft, a, 10, True), ft)
        out = torch.empty_like(flat)
        dg().decompress_data_split_size(True, rows, out, splits, True)
        it = torch.int16 if kind != "f32" else torch.int32
        assert torch.equal(out.view(it), flat.view(it))


def test_float_capacity_failure():
    w = normal_words(5000, "bf16", 1)
    row = to_dev_bytes(O.float_compress(O.BF16, w, 10))
    outs = [torch.zeros(4999, dtype=torch.bfloat16, device="cuda"), torch.zeros(5000, dtype=torch.bfloat16, device="cuda")]
    status = torch.full((2,), 9, dtype=torch.uint8, device="cuda")
    osz = torch.zeros(2, dtype=torch.int32, device="cuda")
    dg().decompress_data(True, [row, row], outs, False, None, status, osz)
    assert status.cpu().tolist() == [0, 1] and osz.cpu().tolist() == [5000, 5000]
    assert np.array_equal(outs[1].view(torch.int16).cpu().numpy().view(np.uint16), w)


# ------------------------------------------- full-size configs (properties) ----

def test_config2_zipf_256mib_roundtrip():
    # BASELINE configs[1]: 64 x 4 MiB Zipf bytes, prec 10 and 11: round trip + size == oracle on a sample
    members = [to_dev_bytes(zipf_bytes(4 << 20, 1.0 if i % 2 == 0 else 1.5, 1234 + i)) for i in range(8)]
    ts = [members[i % 8] for i in range(64)]
    for pb in (10, 11):
        comp, sizes, _ = dg().compress_data(False, ts, prob_bits=pb)
        hs = sizes.cpu().tolist()
        for i in (0, 1):
            want = O.ans_encode(members[i].cpu().numpy(), pb)
            assert hs[i] == want.size
            O.assert_same_ans(comp[i, :hs[i]].cpu().numpy(), want)
        assert hs[:8] * 8 == hs
        outs = [torch.empty_like(t) for t in ts]
        dg().decompress_data(False, [comp[i, :hs[i]] for i in range(64)], outs, prob_bits=pb)
        for i in range(64):
            assert torch.equal(outs[i], ts[i])


@pytest.mark.parametrize("kind,batch,relu", [("bf16", 64, False), ("f16", 256, True)])
def test_config3_4_float_256mib_roundtrip(kind, batch, relu):
    # BASELINE configs[2]/[3]: 256 MiB of 16-bit floats; round trip + oracle equality on one member
    per = (128 << 20) // batch
    uniq = [normal_words(per, kind, 1234 + i, relu=relu) for i in range(4)]
    dev = [words_to_tensor(u, kind) for u in uniq]
    ts = [dev[i % 4] for i in range(batch)]
    comp, sizes, _ = dg().compress_data(True, ts)
    hs = sizes.cpu().tolist()
    want = O.float_compress(KINDS[kind][0], uniq[0], 10)
    assert hs[0] == want.size
    O.assert_same_float(comp[0, :hs[0]].cpu().numpy(), want, KINDS[kind][0])
    outs = [torch.empty_like(t) for t in ts]
    dg().decompress_data(True, [comp[i, :hs[i]] for i in range(batch)], outs)
    for i in range(batch):
        assert torch.equal(outs[i].view(torch.int16), ts[i].view(torch.int16))


def test_single_member_256mib_bf16():
    # bs = 1 x 128 Mi floats: 32768 blocks in one member (look-back across many tickets)
    w = words_to_tensor(normal_words(128 << 20, "bf16", 99), "bf16")
    comp, sizes, _ = dg().compress_data(True, [w])
    n = int(sizes[0])
    ratio = n / (w.numel() * 2)
    assert 0.66 < ratio < 0.69  # README: ~0.673
    out = torch.empty_like(w)
    dg().decompress_data(True, [comp[0, :n]], [out])
    assert torch.equal(out.view(torch.int16), w.view(torch.int16))


def test_canonical_layout_is_byte_exact():
    # option encode_canonical: streams packed in block order -> archives equal the oracle's byte for byte
    from dietgpu_b200 import capi

    capi.set_option("encode_canonical", 1)
    try:
        arrays = [zipf_bytes(300000, 1.1, 5), exp_bytes(4097, 50, 6), exp_bytes(70000, 10, 7), np.zeros(0, np.uint8)]
        for pb in (9, 10, 11):
            ts = [to_dev_bytes(a) for a in arrays]
            comp, sizes, _ = dg().compress_data(False, ts, True, prob_bits=pb)
            hs = sizes.cpu().tolist()
            for i, a in enumerate(arrays):
                assert np.array_equal(comp[i, :hs[i]].cpu().numpy(), O.ans_encode(a, pb, True))
        for kind in ("bf16", "f16", "f32"):
            ws = [normal_words(n, kind, n) for n in (100000, 4096, 33)]
            ts = [words_to_tensor(w, kind) for w in ws]
            comp, sizes, _ = dg().compress_data(True, ts, True)
            hs = sizes.cpu().tolist()
            for i, w in enumerate(ws):
                assert np.array_equal(comp[i, :hs[i]].cpu().numpy(), O.float_compress(KINDS[kind][0], w, 10, True))
            outs = [torch.empty_like(t) for t in ts]
            dg().decompress_data(True, [comp[i, :hs[i]] for i in range(len(ts))], outs, True)
            it = torch.int16 if kind != "f32" else torch.int32
            for t, o in zip(ts, outs):
                assert torch.equal(t.view(it), o.view(it))
    finally:
        capi.set_option("encode_canonical", 0)


def test_small_staging_slot_spills():
    # the fast encoder's staging slot can be smaller than a block's worst-case stream; force the
    # spill path with the smallest slot on incompressible and on ragged inputs
    from dietgpu_b200 import capi

    capi.set_option("encode_slot_words", 776)
    try:
        arrays = [np.random.default_rng(5).integers(0, 256, 300000, dtype=np.uint8), zipf_bytes(123457, 1.0, 3),
                  exp_bytes(4097, 2, 4), exp_bytes(31, 1, 5)]
        for pb in (9, 10, 11):
            ans_roundtrip(arrays, pb, checksum=True)
        float_roundtrip("f32", [np.random.default_rng(6).integers(0, 2**32, 100000, dtype=np.uint32)], 10)
        float_roundtrip("bf16", [np.random.default_rng(7).integers(0, 2**16, 200001, dtype=np.uint16)], 11)
    finally:
        capi.set_option("encode_slot_words", 0)


def test_sub_batch_streams():
    # large batches are cut into sub-batches that run on internal streams; force 1/2/4 parts on
    # batches of 1, 3 and many members (incl. empty members) and check parity each time
    from dietgpu_b200 import capi

    try:
        for parts in (1, 2, 4):
            capi.set_option("parts", parts)
            ans_roundtrip([zipf_bytes(50000, 1.0, 1)], 10)
            ans_roundtrip([exp_bytes(9000, 5, 2), np.zeros(0, np.uint8), exp_bytes(70000, 50, 3)], 10, checksum=True)
            ans_roundtrip([exp_bytes(1000 + 513 * i, 20, i) for i in range(37)], 11)
            float_roundtrip("bf16", [normal_words(3000 + 1111 * i, "bf16", i) for i in range(19)], 10, checksum=True)
            float_roundtrip("f32", [normal_words(5000, "f32", 1), normal_words(0, "f32", 2)], 10)
    finally:
        capi.set_option("parts", 0)


def test_two_host_threads_with_sub_batches():
    # two host threads, each on its own CUDA stream, both forcing sub-batch streams: the internal
    # fork/join streams and events are per thread, so the calls must not disturb each other
    import threading

    from dietgpu_b200 import capi

    errs = []

    def worker(seed):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                for it in range(6):
                    float_roundtrip("bf16", [normal_words(60000 + 1000 * i, "bf16", seed + i) for i in range(9)], 10,
                                    checksum=True)
                    ans_roundtrip([exp_bytes(30000 + 4097 * i, 20, seed + i) for i in range(7)], 10)
        except Exception as e:  # noqa: BLE001
            errs.append(repr(e))

    try:
        capi.set_option("parts", 3)
        th = [threading.Thread(target=worker, args=(100 * k,)) for k in range(2)]
        for t in th:
            t.start()
        for t in th:
            t.join()
    finally:
        capi.set_option("parts", 0)
    assert not errs, errs


def test_encoder_table_formats():
    # the encoder symbol table has a 16-byte and an 8-byte entry format (chosen by data kind);
    # force each one on every kind, all precisions, incl. pdf == 1 symbols and a single-symbol input
    from dietgpu_b200 import capi

    try:
        for wide in (0, 1):
            capi.set_option("encode_wide_table", wide)
            for pb in (9, 10, 11):
                ans_roundtrip([zipf_bytes(200000, 1.0, 1), exp_bytes(4097, 3, 2), np.full(5000, 7, np.uint8),
                               np.random.default_rng(3).integers(0, 256, 70001, dtype=np.uint8)], pb, checksum=True)
            for ft in ("f16", "bf16", "f32"):
                float_roundtrip(ft, [normal_words(100000 + 7 * i, ft, i) for i in range(3)], 10, checksum=True)
    finally:
        capi.set_option("encode_wide_table", -1)


def test_tuning_options_agree():
    # every tuning variant produces identical results: warps per CTA in both directions, canonical
    # packing, member table in the kernel parameters or in scratch
    from dietgpu_b200 import capi

    a = [zipf_bytes(300000, 1.1, 5), exp_bytes(4097, 50, 6), zipf_bytes(1, 1.0, 7), np.zeros(0, np.uint8)]
    f = [normal_words(50000 + 13 * i, "bf16", i) for i in range(5)]
    names = ("encode_warps", "encode_canonical", "inline_members", "decode_warps")
    defaults = {k: capi.get_option(k) for k in names}
    variants = [
        {},
        dict(encode_warps=2),
        dict(encode_warps=4),
        dict(encode_canonical=1),
        dict(decode_warps=20),  # byte archives: 20-warp decoder CTAs (auto only for long members)
        dict(decode_warps=8),
        dict(inline_members=0),  # member table uploaded to scratch instead of travelling in the kernel parameters
    ]
    try:
        for v in variants:
            for k, d in defaults.items():
                capi.set_option(k, v.get(k, d))
            ans_roundtrip(a, 10)
            float_roundtrip("bf16", f, 10)
    finally:
        for k, d in defaults.items():
            capi.set_option(k, d)


def test_more_members_than_fit_the_kernel_parameters():
    # batches above 64 members read the member table from scratch, up to 64 from the kernel parameters:
    # both sides of the boundary, bytes and floats, against the oracle
    for n in (63, 64, 65, 130):
        ans_roundtrip([zipf_bytes(3000 + 37 * i, 1.2, i) for i in range(n)], 10)
        float_roundtrip("f16", [normal_words(2500 + 11 * i, "f16", i) for i in range(n)], 10)


def test_calls_can_be_captured_into_a_cuda_graph():
    # with the member table in the kernel parameters a call reads no host memory after it returns, so
    # compress + decompress can be captured once and replayed on new data in the same buffers
    from dietgpu_b200 import ops

    n, per = 6, 40000 + 17
    ts = [torch.zeros(per, dtype=torch.bfloat16, device="cuda") for _ in range(n)]
    outs = [torch.empty_like(t) for t in ts]
    _, cols = ops.max_float_compressed_output_size(ts)
    comp = torch.empty((n, cols), dtype=torch.uint8, device="cuda")
    sizes = torch.zeros(n, dtype=torch.int32, device="cuda")
    temp = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    rows = [comp[i] for i in range(n)]

    def step():
        ops.compress_data(True, ts, False, temp, comp, sizes)
        ops.decompress_data(True, rows, outs, False, temp)

    step()  # warm-up outside capture (function attributes, occupancy queries)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    for seed in (1, 2, 3):
        gen = torch.Generator(device="cuda").manual_seed(seed)
        for t in ts:
            t.copy_(torch.randn(per, generator=gen, device="cuda").to(torch.bfloat16) * (seed * 3.0))
        g.replay()
        torch.cuda.synchronize()
        for t, o in zip(ts, outs):
            assert torch.equal(t.view(torch.int16), o.view(torch.int16))
        want = [len(O.float_compress(O.BF16, t.view(torch.int16).cpu().numpy().view(np.uint16), 10)) for t in ts]
        assert sizes.cpu().tolist() == want


def test_archive_mover_copies_exactly_the_archive():
    # dgb_archives_pull: each archive is copied as long as its header says (sizes read on the device), the rest
    # of the destination row is left alone; bad headers arrive as 32 bytes and fail in the decoder
    from dietgpu_b200 import ops

    for as_float, dt in ((True, torch.bfloat16), (True, torch.float32), (False, torch.uint8)):
        if as_float:
            ts = [torch.randn(30000 + 4097 * i, device="cuda").to(dt) for i in range(5)]
        else:
            ts = [to_dev_bytes(zipf_bytes(50000 + 977 * i, 1.2, i)) for i in range(5)]
        comp, sizes, _ = ops.compress_data(as_float, ts)
        hs = sizes.cpu().tolist()
        dst = torch.full_like(comp, 0xAB)
        got = torch.zeros(len(ts), dtype=torch.int32, device="cuda")
        ops.pull_archives(as_float, [comp[i] for i in range(len(ts))], [dst[i] for i in range(len(ts))], dt, got)
        assert got.cpu().tolist() == hs
        for i, k in enumerate(hs):
            assert torch.equal(dst[i, :k], comp[i, :k])
            assert bool((dst[i, k:] == 0xAB).all())
        outs = [torch.empty_like(t) for t in ts]
        st = torch.zeros(len(ts), dtype=torch.uint8, device="cuda")
        ops.decompress_data(as_float, [dst[i] for i in range(len(ts))], outs, False, None, st)
        assert bool(st.all())
        for a, b in zip(ts, outs):
            assert torch.equal(a.view(torch.uint8), b.view(torch.uint8))
        # a corrupted magic: 32 bytes arrive, the decoder reports the member
        bad = comp.clone()
        bad[2, 0] ^= 0xFF
        dst.fill_(0)
        ops.pull_archives(as_float, [bad[i] for i in range(len(ts))], [dst[i] for i in range(len(ts))], dt, got)
        assert got.cpu().tolist()[2] == 32 and not bool(dst[2, 32:].any())
        st.zero_()
        ops.decompress_data(as_float, [dst[i] for i in range(len(ts))], outs, False, None, st)
        assert st.cpu().tolist() == [1, 1, 0, 1, 1]
        # a destination shorter than the archive: cut at the capacity, nothing written behind it
        small = torch.zeros(hs[0] + 64, dtype=torch.uint8, device="cuda")
        ops.pull_archives(as_float, [comp[0]], [small[:hs[0] - 160]], dt)
        assert torch.equal(small[:hs[0] - 160], comp[0, :hs[0] - 160]) and not bool(small[hs[0] - 160:].any())


def test_members_near_the_format_limit():
    # one member of 1.5 Gi + 1 symbols: the largest round size whose worst-case archive still fits the format's
    # 32-bit sizes (dgb_*_max_compressed_size != 0); 393 217 blocks, block offsets above 2^31 bytes in the
    # float output.  Round trip, status, reported size against the archive's own header fields.
    from dietgpu_b200 import ops

    n = (3 << 29) + 1
    gen = torch.Generator(device="cuda").manual_seed(11)
    for as_float in (False, True):
        if as_float:
            x = torch.empty(n, dtype=torch.bfloat16, device="cuda")
            for a in range(0, n, 1 << 28):
                b = min(n, a + (1 << 28))
                x[a:b] = torch.randn(b - a, generator=gen, device="cuda").to(torch.bfloat16)
        else:
            x = torch.empty(n, dtype=torch.uint8, device="cuda")
            for a in range(0, n, 1 << 28):
                b = min(n, a + (1 << 28))
                x[a:b] = (torch.randn(b - a, generator=gen, device="cuda") * 12).abs().clamp(max=255).to(torch.uint8)
        comp, sizes, _ = ops.compress_data(as_float, [x])
        size = int(sizes[0]) & 0xffffffff  # the operator's size tensor is int32 (DietGpu.cpp:139); the C ABI writes u32
        words = comp[0, :size]
        if as_float:
            fh = words[:16].view(torch.int32).cpu().tolist()
            assert (fh[0] & 0xffffffff) == 0xf00f0001 and fh[1] == n
            ans = words[16 + ((n + 15) // 16) * 16:]
        else:
            ans = words
        h = ans[:16].view(torch.int32).cpu().tolist()
        nb = (n + 4095) // 4096
        assert (h[0] & 0xffffffff) == 0xd00d0001 and h[1] == nb and h[2] == n
        total_words = h[3] & 0xffffffff
        overhead = 32 + 512 + 128 * nb + 8 * ((nb + 1) // 2 * 2)
        assert ans.numel() == overhead + 2 * total_words
        assert 0.2 * n < 2 * total_words < 1.0 * n
        out = torch.empty_like(x)
        st = torch.zeros(1, dtype=torch.uint8, device="cuda")
        osz = torch.zeros(1, dtype=torch.int32, device="cuda")
        ops.decompress_data(as_float, [words], [out], False, None, st, osz)
        assert st.item() == 1 and osz.item() == n
        for a in range(0, n, 1 << 28):  # chunked compare keeps the temporaries small
            b = min(n, a + (1 << 28))
            assert torch.equal(x[a:b].view(torch.uint8 if not as_float else torch.int16), out[a:b].view(torch.uint8 if not as_float else torch.int16))
        del x, out, comp, words, ans


def test_get_compressed_info_matches_oracle():
    # dgb_{ans,float}_get_compressed_info (ans/GpuANSInfo.cu:14-49, float/GpuFloatInfo.cu:17-64) against
    # dgo_ans_info / dgo_float_info on the same archives: uncompressed sizes, float types, stored checksums
    import ctypes as C

    from dietgpu_b200 import capi

    L = capi.lib()
    arrays = [zipf_bytes(50000 + 977 * i, 1.2, i) for i in range(5)] + [np.zeros(0, np.uint8)]
    ts = [to_dev_bytes(a) for a in arrays]
    comp, sizes, _ = dg().compress_data(False, ts, True)
    hs = sizes.cpu().tolist()
    n = len(ts)
    ptrs = capi.ptr_array([comp[i].data_ptr() for i in range(n)])
    o_sz = torch.zeros(n, dtype=torch.int32, device="cuda")
    o_ck = torch.zeros(n, dtype=torch.int32, device="cuda")
    tmp = torch.empty(8 * n + 512, dtype=torch.uint8, device="cuda")
    tp = tmp.data_ptr() + (-tmp.data_ptr()) % 256
    capi.check(L.dgb_ans_get_compressed_info(tp, 8 * n + 256, ptrs, 0, n, o_sz.data_ptr(), o_ck.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream), "ans info")
    for i in range(n):
        info = O.ans_info(comp[i, :hs[i]].cpu().numpy())
        assert info["rc"] == O.OK and info["size"] == hs[i]
        assert o_sz[i].item() == info["uncompressed"] == arrays[i].size
        assert (o_ck[i].item() & 0xffffffff) == info["checksum"] == O.ans_info(O.ans_encode(arrays[i], 10, True))["checksum"]
    # the device-array form returns the same
    dptrs = torch.tensor([comp[i].data_ptr() for i in range(n)], dtype=torch.int64, device="cuda")
    o_sz2 = torch.zeros_like(o_sz)
    capi.check(L.dgb_ans_get_compressed_info(None, 0, C.c_void_p(dptrs.data_ptr()), 1, n, o_sz2.data_ptr(), None,
                                             torch.cuda.current_stream().cuda_stream), "ans info (device array)")
    assert torch.equal(o_sz, o_sz2)

    for kind, (ft, _, _) in KINDS.items():
        words = [normal_words(30000 + 501 * i, kind, i) for i in range(4)]
        fts = [words_to_tensor(w, kind) for w in words]
        comp, sizes, _ = dg().compress_data(True, fts, True)
        hs = sizes.cpu().tolist()
        n = len(fts)
        ptrs = capi.ptr_array([comp[i].data_ptr() for i in range(n)])
        o_sz = torch.zeros(n, dtype=torch.int32, device="cuda")
        o_ty = torch.zeros(n, dtype=torch.int32, device="cuda")
        o_ck = torch.zeros(n, dtype=torch.int32, device="cuda")
        capi.check(L.dgb_float_get_compressed_info(tp, 8 * n + 256, ptrs, 0, n, o_sz.data_ptr(), o_ty.data_ptr(),
                                                   o_ck.data_ptr(), torch.cuda.current_stream().cuda_stream), "float info")
        for i in range(n):
            info = O.float_info(comp[i, :hs[i]].cpu().numpy())
            assert info["rc"] == O.OK
            assert o_sz[i].item() == info["size"] == words[i].size
            assert o_ty[i].item() == info["float_type"] == ft
            assert (o_ck[i].item() & 0xffffffff) == info["checksum"] == O.float_info(O.float_compress(ft, words[i], 10, True))["checksum"]


@pytest.mark.parametrize("kind", ["f16", "bf16", "f32"])
def test_float_members_not_16_byte_aligned(kind):
    # split sizes that push every following member off the 16 B grid (dgb_float_compress_split_size lays
    # members back to back): the statistics pass peels a scalar head and keeps its vector body, and the
    # planes are written at shifted offsets -- archives must still equal the oracle's
    ft, tdt, _ = KINDS[kind]
    sizes = [40003, 8191, 65537, 5, 33001, 12345]
    words = [normal_words(n, kind, i) for i, n in enumerate(sizes)]
    big = words_to_tensor(np.concatenate(words), kind)
    comps, csz, _ = dg().compress_data_split_size(True, big, torch.tensor(sizes, dtype=torch.int32))
    hs = csz.cpu().tolist()
    for i, w in enumerate(words):
        want = O.float_compress(ft, w, 10)
        assert hs[i] == want.size
        O.assert_same_float(comps[i][:hs[i]].cpu().numpy(), want, ft, f"member {i}")
    out = torch.empty_like(big)
    dg().decompress_data_split_size(True, [comps[i][:hs[i]] for i in range(len(sizes))], out,
                                    torch.tensor(sizes, dtype=torch.int32))
    idt = torch.int32 if kind == "f32" else torch.int16
    assert torch.equal(out.view(idt), big.view(idt))
