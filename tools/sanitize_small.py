"""Small round trips of every kernel flavour, meant to run under compute-sanitizer (memcheck / racecheck /
synccheck / initcheck): python tools/sanitize_small.py.  Sizes are a few 4 KiB blocks per member so that the
instrumented kernels finish in seconds; every result is checked (bit-exact round trip)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from dietgpu_b200 import capi, ops  # noqa: E402

dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(5)


def floats(n, dt, off=0):
    base = torch.randn(n + off, generator=g, device=dev)
    if dt == torch.float32:
        return base[off:]
    return base.to(dt)[off:]


def bytes_(n, off=0):
    return (torch.randn(n + off, generator=g, device=dev) * 9).abs().clamp(max=255).to(torch.uint8)[off:]


VARIANTS = [
    {},
    {"encode_canonical": 1},
    {"inline_members": 0},
    {"decode_warps": 20},
    {"encode_warps": 2, "decode_slot_words": 512, "encode_slot_words": 512},
]
if os.environ.get("SAN_QUICK") == "1":
    VARIANTS = VARIANTS[:1]
cases = 0
for v in VARIANTS:
    saved = {k: capi.get_option(k) for k in v}
    for k, val in v.items():
        capi.set_option(k, val)
    try:
        for as_float, dt, pb in ((False, torch.uint8, 10), (False, torch.uint8, 9), (False, torch.uint8, 11),
                                 (True, torch.bfloat16, 10), (True, torch.float16, 10), (True, torch.float32, 10)):
            for checksum in (False, True):
                sizes = (0, 1, 31, 4096, 4097, 12345, 3 * 4096 + 5)
                if as_float:
                    ts = [floats(n, dt, off=i % 3) for i, n in enumerate(sizes) if n]
                else:
                    ts = [bytes_(n, off=4 * (i % 2)) for i, n in enumerate(sizes)]
                comp, csz, _ = ops.compress_data(as_float, ts, checksum, prob_bits=pb)
                hs = csz.cpu().tolist()
                outs = [torch.empty_like(t) for t in ts]
                st = torch.zeros(len(ts), dtype=torch.uint8, device=dev)
                ops.decompress_data(as_float, [comp[i, :hs[i]] for i in range(len(ts))], outs, checksum, None, st, prob_bits=pb)
                assert bool(st.all()), (v, dt, pb, checksum, st.tolist())
                for a, b in zip(ts, outs):
                    assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), (v, dt, pb, checksum)
                cases += 1
        # archive mover
        ts = [floats(9000 + 13 * i, torch.bfloat16) for i in range(3)]
        comp, csz, _ = ops.compress_data(True, ts)
        dst = torch.zeros_like(comp)
        ops.pull_archives(True, [comp[i] for i in range(3)], [dst[i] for i in range(3)], torch.bfloat16)
        for i, k in enumerate(csz.cpu().tolist()):
            assert torch.equal(dst[i, :k], comp[i, :k])
    finally:
        for k, val in saved.items():
            capi.set_option(k, val)
torch.cuda.synchronize()
print(f"sanitize_small: {cases} round-trip cases over {len(VARIANTS)} kernel variants OK")
