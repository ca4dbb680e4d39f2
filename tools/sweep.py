"""Kernel-variant sweep on one workload: python tools/sweep.py <workload> 'opt=val,opt=val' ...
Prints encode/decode GB/s and per-kernel ms for each variant (C ABI called with cached arrays)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from dietgpu_b200 import capi  # noqa: E402

wl = sys.argv[1]
variants = sys.argv[2:] or [""]
kind, batch, per, desc = bench.WORKLOADS[wl]
dev = torch.device("cuda", 0)
ts = bench.make_batch(torch, kind, batch, per, 1234, dev)
ub = sum(t.numel() * t.element_size() for t in ts)
it = torch.int16 if kind != "bytes" else torch.uint8
for v in variants:
    opts = dict(kv.split("=") for kv in v.split(",") if kv)
    for k, val in opts.items():
        capi.set_option(k, int(val))
    codec = bench.OursCodec(torch, kind, ts)
    codec.encode(); hs = codec.bind_rows(); codec.decode(); torch.cuda.synchronize()
    ok = all(torch.equal(a.view(it), b.view(it)) for a, b in zip(ts, codec.outs))
    for _ in range(3):
        codec.encode(); codec.decode()
    capi.set_option("timing", 1); capi.kernel_times()
    n = 10
    for _ in range(n):
        codec.encode(); codec.decode()
    kt = capi.kernel_times(); capi.set_option("timing", 0)
    ms = {k: kt[k][0] / max(kt[k][1], 1) for k in kt}
    enc = ms["stats"] + ms["encode"]; dec = ms["decode"]
    print(f"{wl} [{v}] ok={ok} ratio={sum(hs)/ub:.4f} stats={ms['stats']*1e3:.1f}us encode={ms['encode']*1e3:.1f}us "
          f"decode={ms['decode']*1e3:.1f}us | enc {ub/enc/1e6:.0f} GB/s dec {ub/dec/1e6:.0f} GB/s (kernel-only)", flush=True)
    for k in opts:
        pass
