"""Writes the golden data taken from the UNMODIFIED reference, which must have been compiled for sm_100a
into oracle/_ref/ (oracle/build_ref.sh); needs a GPU.
  ref_golden.npz: small seeded inputs with the reference's archives of them (checksum on).  CPU tests compare
                  the oracle with them field by field; GPU tests decode them with the library.
  ref_parity.npz: for the inputs of tests/test_reference_parity.py, the reference's compressed sizes, row
                  widths, max-size table and SHA-256 digests of every defined archive field.
Usage:  python tests/golden/make_ref_golden.py [OUT_DIR]     (default: tests/golden)"""
import hashlib
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import test_reference_parity as P  # noqa: E402
from conftest import exp_bytes, normal_words, zipf_bytes  # noqa: E402

from oracle import oracle as O  # noqa: E402
from oracle import ref_lib  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else HERE
ref = ref_lib.RefCodec(512 << 20)
L = ref_lib.lib()
KINDS = {"f16": (1, torch.float16, np.int16), "bf16": (2, torch.bfloat16, np.int16), "f32": (3, torch.float32, np.int32)}


def ans_archives(arrays, pb):
    ts = [torch.from_numpy(a).cuda() for a in arrays]
    comp = torch.zeros((len(ts), L.ref_ans_max_compressed_size(max(a.size for a in arrays))), dtype=torch.uint8,
                       device="cuda")
    sz = torch.zeros(len(ts), dtype=torch.int32, device="cuda")
    assert ref.ans_encode(ts, comp, sz, pb, True) == 0
    torch.cuda.synchronize()
    return comp.size(1), [comp[i, :n].cpu().numpy() for i, n in enumerate(sz.cpu().tolist())]


def float_archives(kind, words):
    ft, tdt, wt = KINDS[kind]
    ts = [torch.from_numpy(w.view(wt).copy()).view(tdt).cuda() for w in words]
    comp = torch.zeros((len(ts), L.ref_float_max_compressed_size(ft, max(w.size for w in words))), dtype=torch.uint8,
                       device="cuda")
    sz = torch.zeros(len(ts), dtype=torch.int32, device="cuda")
    assert ref.float_compress(ft, ts, comp, sz, 10, True) == 0
    torch.cuda.synchronize()
    return comp.size(1), [comp[i, :n].cpu().numpy() for i, n in enumerate(sz.cpu().tolist())]


# ---- ref_golden.npz: whole archives, members small enough to keep the file well under 1 MB ----
golden = {}
cases = {
    "exp20_10013": exp_bytes(10013, 20, 1), "zipf1_20000": zipf_bytes(20000, 1.0, 2), "one": exp_bytes(1, 1, 3),
    "quirk_ids_100_160": np.random.default_rng(4).integers(100, 160, 12000).astype(np.uint8),
    "uniform_12000": np.random.default_rng(5).integers(0, 256, 12000, dtype=np.uint8),
    "single_symbol": np.full(10000, 9, np.uint8),
    "exp100_163841": exp_bytes(163841, 100, 6),  # 41 blocks: the decoder's multi-block path on reference archives
}
for name, data in cases.items():
    golden[f"ans/{name}/in"] = data
    for pb in (9, 10, 11):
        golden[f"ans/{name}/pb{pb}"] = ans_archives([data], pb)[1][0]
for kind in ("bf16", "f16", "f32"):
    for n in (1, 4099, 12289):
        w = normal_words(n, kind, 100 + n)
        golden[f"float/{kind}/{n}/in"] = w
        golden[f"float/{kind}/{n}/pb10"] = float_archives(kind, [w])[1][0]

# ---- ref_parity.npz: field digests of the archives of the parity tests' (larger) inputs ----
parity = {}


def add_digests(key, archives, ft=0):
    parity[key + "/sizes"] = np.array([a.size for a in archives], np.int64)
    for i, a in enumerate(archives):
        for field, v in O.defined_fields(a, ft).items():
            parity[f"{key}/{i}/{field}"] = np.frombuffer(hashlib.sha256(v).digest(), np.uint8)


for pb in (9, 10, 11):
    cols, archives = ans_archives(P.ans_inputs(), pb)
    parity["ans/cols"] = np.int64(cols)
    add_digests(f"ans/pb{pb}", archives)
for kind, (ft, _, _) in KINDS.items():
    cols, archives = float_archives(kind, P.float_inputs(kind))
    parity[f"float/{kind}/cols"] = np.int64(cols)
    add_digests(f"float/{kind}", archives, ft)
parity["max_sizes/ans"] = np.array([L.ref_ans_max_compressed_size(n) for n in P.MAX_SIZE_NS], np.int64)
parity["max_sizes/float"] = np.array([[L.ref_float_max_compressed_size(ft, n) for n in P.MAX_SIZE_NS]
                                      for ft in (1, 2, 3)], np.int64)

os.makedirs(OUT, exist_ok=True)
np.savez_compressed(os.path.join(OUT, "ref_golden.npz"), **golden)
np.savez_compressed(os.path.join(OUT, "ref_parity.npz"), **parity)
print("wrote", len(golden), "+", len(parity), "arrays to", OUT)
