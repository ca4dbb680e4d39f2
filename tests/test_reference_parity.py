"""GPU parity against the REFERENCE ITSELF (facebookresearch/dietgpu, unmodified, sm_100a build).  Pins what
the reference's own tests leave unpinned (SURVEY 8c): byte-exact compressed sizes, field-exact archives
(masking only the bits the reference leaves undefined), and cross-decoding.

What the reference produced is stored under tests/golden/ (tests/golden/make_ref_golden.py writes it):
ref_parity.npz holds, for the inputs below, the reference's compressed sizes, row widths and max-size table,
and a SHA-256 digest of every defined field of every archive (oracle.defined_fields); ref_golden.npz holds
whole reference archives of smaller inputs, which our decoder must read back.  Where the reference itself
decoded our archives, the CPU oracle does: it reads archives the way the reference does and is pinned to the
reference by tests/test_oracle.py."""
import hashlib
import os

import numpy as np
import pytest
import torch

from conftest import exp_bytes, normal_words, zipf_bytes
from oracle import oracle as O

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KINDS = {"f16": (1, torch.float16), "bf16": (2, torch.bfloat16), "f32": (3, torch.float32)}
MAX_SIZE_NS = (0, 1, 4095, 4096, 4097, 1 << 20, 4 << 20, 123456789, 0x7fffffff // 2)


def ans_inputs():
    return [exp_bytes(10013, 10, 1), zipf_bytes(300000, 1.0, 2), exp_bytes(4096, 100, 3), exp_bytes(1, 1, 4),
            np.random.default_rng(5).integers(100, 160, 30000).astype(np.uint8),  # SURVEY B1: 'add' branch by symbol id
            np.random.default_rng(6).integers(0, 256, 70000, dtype=np.uint8)]


def float_inputs(kind):
    return [normal_words(n, kind, 20 + i) for i, n in enumerate((10000, 123457, 4096, 1, 524288))]


def field_digests(arch, ft=0):
    return {k: hashlib.sha256(v).digest() for k, v in O.defined_fields(arch, ft).items()}


@pytest.fixture(scope="module")
def parity():
    return np.load(os.path.join(GOLD, "ref_parity.npz"))


@pytest.fixture(scope="module")
def ref_archives():
    return np.load(os.path.join(GOLD, "ref_golden.npz"))


def dg():
    import dietgpu_b200

    return dietgpu_b200


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_fields_match(mine, parity, key, ft=0):
    want = {k[len(key) + 1:]: parity[k].tobytes() for k in parity.files if k.startswith(key + "/")}
    got = field_digests(mine, ft)
    assert got.keys() == want.keys(), (key, sorted(got), sorted(want))
    differ = [k for k in got if got[k] != want[k]]
    assert not differ, f"{key}: fields differ from the reference archive: {differ}"


@pytest.mark.parametrize("pb", [9, 10, 11])
def test_ans_matches_reference(parity, ref_archives, pb):
    arrays = ans_inputs()
    ts = [dev(a) for a in arrays]
    n = len(ts)
    comp, sizes, _ = dg().compress_data(False, ts, True, prob_bits=pb)
    assert comp.size(1) == int(parity["ans/cols"])
    hs = sizes.cpu().tolist()
    assert hs == parity[f"ans/pb{pb}/sizes"].tolist(), "compressed sizes differ from the reference"
    for i in range(n):
        mine = comp[i, :hs[i]].cpu().numpy()
        assert_fields_match(mine, parity, f"ans/pb{pb}/{i}")
        O.assert_same_ans(mine, O.ans_encode(arrays[i], pb, True))
        rc, out, _ = O.ans_decode(mine, pb, verify_checksum=True)
        assert rc == O.OK and np.array_equal(out, arrays[i])
    # ours <- archives written by the reference
    names = sorted({k.rsplit("/", 1)[0] for k in ref_archives.files if k.startswith("ans/")})
    ins = [ref_archives[b + "/in"] for b in names]
    outs = [torch.empty(x.size, dtype=torch.uint8, device="cuda") for x in ins]
    dg().decompress_data(False, [dev(ref_archives[f"{b}/pb{pb}"]) for b in names], outs, True, prob_bits=pb)
    for b, x, o in zip(names, ins, outs):
        assert np.array_equal(o.cpu().numpy(), x), b


@pytest.mark.parametrize("kind", ["f16", "bf16", "f32"])
def test_float_matches_reference(parity, ref_archives, kind):
    ft, tdt = KINDS[kind]
    words = float_inputs(kind)
    it, wt = (torch.int16, np.int16) if kind != "f32" else (torch.int32, np.int32)
    ts = [torch.from_numpy(w.view(wt).copy()).view(tdt).cuda() for w in words]
    comp, sizes, _ = dg().compress_data(True, ts, True)
    assert comp.size(1) == int(parity[f"float/{kind}/cols"])
    hs = sizes.cpu().tolist()
    assert hs == parity[f"float/{kind}/sizes"].tolist(), "float compressed sizes differ from the reference"
    for i, w in enumerate(words):
        mine = comp[i, :hs[i]].cpu().numpy()
        assert_fields_match(mine, parity, f"float/{kind}/{i}", ft)
        O.assert_same_float(mine, O.float_compress(ft, w, 10, True), ft, f"member {i}")
        rc, out, _ = O.float_decompress(ft, mine, 10, verify_checksum=True)
        assert rc == O.OK and np.array_equal(out, w)
    # ours <- archives written by the reference
    names = sorted({k.rsplit("/", 1)[0] for k in ref_archives.files if k.startswith(f"float/{kind}/")})
    ins = [ref_archives[b + "/in"] for b in names]
    outs = [torch.empty(x.size, dtype=tdt, device="cuda") for x in ins]
    dg().decompress_data(True, [dev(ref_archives[b + "/pb10"]) for b in names], outs, True)
    for b, x, o in zip(names, ins, outs):
        assert np.array_equal(o.view(it).cpu().numpy().view(x.dtype), x), b


def test_max_sizes_match_reference(parity):
    L = dg().capi.lib()
    ref_ans, ref_float = parity["max_sizes/ans"], parity["max_sizes/float"]
    for j, n in enumerate(MAX_SIZE_NS):
        assert L.dgb_ans_max_compressed_size(n) == ref_ans[j]
        for ft in (1, 2, 3):
            mine = L.dgb_float_max_compressed_size(ft, n)
            if mine == 0:
                # the exact bound does not fit 32 bits: the reference returns the wrapped sum, this ABI
                # reports "too large" (0) instead of a value a caller would under-allocate from
                assert 16 + L.dgb_ans_max_compressed_size(n) + (3 if ft == 3 else 1) * n > 0xffffffff
                continue
            assert mine == ref_float[ft - 1, j]
