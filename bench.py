#!/usr/bin/env python
"""bench.py -- encode+decode throughput of the batched rANS / float codec.

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--workload c3|c2|c4|c3x1]
                    [--dump-outputs DIR]

A "step" = one pass of the hot path over one batch: compress the whole batch,
then decompress it.  metric = uncompressed GB/s through encode+decode
= 2 * uncompressed_bytes / (t_encode + t_decode)   [the reference's convention
is uncompressed bytes / time, benchmark.py:156-157].

Workloads (BASELINE.json configs; MiB-based like the reference's benchmark.py):
  c3    64 x 2 Mi bf16 N(0,1)            (256 MiB)  <- default / headline
  c2    64 x 4 MiB Zipf(s=1) bytes, pb10 (256 MiB)
  c4    256 x 512 Ki fp16 ReLU(N(0,1))   (256 MiB)
  c3x1  1 x 128 Mi bf16 N(0,1)           (256 MiB, batch 1 -- the published A100 curve point)

N > 1 (torchrun, one rank per GPU): every rank codes its own batch (seed offset
1000*rank): weak scaling, no data-path collective (batch members are
independent); NCCL is only used for the barrier / max-over-ranks timing and one
all-gather of the compressed sizes.

--impl reference runs the UNMODIFIED reference (oracle/_ref/libdietgpu_ref.so,
built from /root/reference for sm_100a by oracle/build_ref.sh) through the same
harness on the GPU.  DietGPU has no CPU implementation, so "the reference's own
implementation of the path" is its CUDA code; the host-CPU number both arms
report under `cpu_baseline` is the oracle port (oracle/dietgpu_oracle.c,
OpenMP over all host cores).  If oracle/_ref is missing the reference arm falls
back to timing that CPU port.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the source tree may be read-only; the bench writes nothing into it

MIB = 1 << 20
WORKLOADS = {
    # name: (kind, batch, elems per member, description)
    "c3": ("bf16", 64, 2 * MIB, "64 x 2Mi bf16 N(0,1) = 256 MiB, prec 10 (BASELINE configs[2])"),
    "c2": ("bytes", 64, 4 * MIB, "64 x 4MiB Zipf(s=1) bytes = 256 MiB, prec 10 (BASELINE configs[1])"),
    "c2p11": ("bytes", 64, 4 * MIB, "64 x 4MiB Zipf(s=1) bytes = 256 MiB, prec 11 (BASELINE configs[1])"),
    "c4": ("f16", 256, 512 * 1024, "256 x 512Ki fp16 ReLU(N(0,1)) = 256 MiB, prec 10 (BASELINE configs[3])"),
    "c3x1": ("bf16", 1, 128 * MIB, "1 x 128Mi bf16 N(0,1) = 256 MiB, batch 1, prec 10"),
}
PROB_BITS = {"c2p11": 11}  # every other workload codes at the reference's default precision, 10


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML in a thread DURING the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.thread = None
        self.max_mhz = None

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv = None
            self.err = str(e)
            return
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.samples), "reasons": sorted(self.reasons)}


def bind_to_gpu_numa_node(index: int):
    """Run this rank on the CPUs of its GPU's NUMA node, so that the pinned staging buffers (first touch)
    and the copy-issuing thread sit next to the GPU's PCIe root (both arms of the bench do this)."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus) > 12:  # nvml: 00000000:3b:00.0, sysfs: 0000:3b:00.0
            bus = bus[-12:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            if "-" in part:
                lo, hi = part.split("-")
                cpus |= set(range(int(lo), int(hi) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"node": node, "cpus": len(cpus)}
    except Exception:  # noqa: BLE001
        pass
    return None


def make_batch(torch, kind, batch, per, seed, device):
    g = torch.Generator(device=device).manual_seed(seed)
    ts = []
    if kind == "bytes":
        p = 1.0 / torch.arange(1, 257, dtype=torch.float64, device=device)
        p = (p / p.sum()).float()
        for _ in range(batch):
            ts.append(torch.multinomial(p, per, replacement=True, generator=g).to(torch.uint8))
    else:
        dt = torch.bfloat16 if kind == "bf16" else torch.float16
        for _ in range(batch):
            x = torch.randn(per, generator=g, device=device, dtype=torch.float32)
            if kind == "f16":
                x = torch.relu(x)
            ts.append(x.to(dt))
    return ts


class OursCodec:
    """Device-resident codec calls through the C ABI (include/dietgpu_b200.h) with the host-side
    pointer/size arrays prepared once, so the timed region measures the library, not Python list
    handling.  `api_*` go through the public operator mirror (dietgpu_b200.ops) for the e2e leg."""
    name = "ours"

    def __init__(self, torch, kind, ts, pb=10):
        import dietgpu_b200 as dg
        self.dg, self.torch, self.kind, self.ts, self.pb = dg, torch, kind, ts, pb
        self.as_float = kind != "bytes"
        n = self.n = len(ts)
        dev = ts[0].device
        _, cols = (dg.max_float_compressed_output_size(ts) if self.as_float else dg.max_any_compressed_output_size(ts))
        self.comp = torch.empty((n, cols), dtype=torch.uint8, device=dev)
        self.sizes = torch.zeros(n, dtype=torch.int32, device=dev)
        self.outs = [torch.empty_like(t) for t in ts]
        L = self.L = dg.capi.lib()
        mx = max(t.numel() for t in ts)
        if self.as_float:
            self.ft = dg.ops._float_type(ts[0])
            need = max(L.dgb_float_compress_temp_bytes(self.ft, n, mx), L.dgb_float_decompress_temp_bytes(self.ft, n, mx))
        else:
            need = max(L.dgb_ans_encode_temp_bytes(n, mx), L.dgb_ans_decode_temp_bytes(n))
        self.temp = torch.empty(need + 512, dtype=torch.uint8, device=dev)
        self.tp = self.temp.data_ptr() + (-self.temp.data_ptr()) % 256
        self.tb = need
        capi = dg.capi
        self.in_ptrs = capi.ptr_array([t.data_ptr() for t in ts])
        self.in_sizes = capi.u32_array([t.numel() if self.as_float else t.numel() * t.element_size() for t in ts])
        self.row_ptrs = capi.ptr_array([self.comp.data_ptr() + i * cols for i in range(n)])
        self.out_ptrs = capi.ptr_array([t.data_ptr() for t in self.outs])
        self.rows = None

    def _stream(self):
        return self.torch.cuda.current_stream().cuda_stream

    def encode(self):
        L = self.L
        if self.as_float:
            rc = L.dgb_float_compress_pointer(self.tp, self.tb, self.ft, self.pb, 0, self.n, self.in_ptrs, self.in_sizes,
                                              self.row_ptrs, self.sizes.data_ptr(), self._stream())
        else:
            rc = L.dgb_ans_encode_pointer(self.tp, self.tb, self.pb, 0, self.n, self.in_ptrs, self.in_sizes, None,
                                          self.row_ptrs, self.sizes.data_ptr(), self._stream())
        assert rc == 0, rc

    def bind_rows(self):
        hs = self.sizes.cpu().tolist()
        self.rows = [self.comp[i, :hs[i]] for i in range(self.n)]
        return hs

    def decode(self):
        L = self.L
        if self.as_float:
            rc = L.dgb_float_decompress_pointer(self.tp, self.tb, self.ft, self.pb, 0, self.n, self.row_ptrs, self.out_ptrs,
                                                self.in_sizes, None, None, None, self._stream())
        else:
            rc = L.dgb_ans_decode_pointer(self.tp, self.tb, self.pb, 0, self.n, self.row_ptrs, self.out_ptrs, self.in_sizes,
                                          None, None, None, self._stream())
        assert rc == 0, rc

    def api_encode(self):
        self.dg.compress_data(self.as_float, self.ts, False, self.temp, self.comp, self.sizes, prob_bits=self.pb)

    def api_decode(self):
        self.dg.decompress_data(self.as_float, self.rows, self.outs, False, self.temp, prob_bits=self.pb)


class RefGpuCodec:
    name = "reference"

    def __init__(self, torch, kind, ts, pb=10):
        from oracle import ref_lib
        self.torch, self.kind, self.ts, self.pb = torch, kind, ts, pb
        self.as_float = kind != "bytes"
        self.ft = {"bf16": 2, "f16": 1}.get(kind, 0)
        n = len(ts)
        dev = ts[0].device
        L = ref_lib.lib()
        mx = max(t.numel() for t in ts)
        cols = L.ref_float_max_compressed_size(self.ft, mx) if self.as_float else L.ref_ans_max_compressed_size(mx)
        self.comp = torch.empty((n, cols), dtype=torch.uint8, device=dev)
        self.sizes = torch.zeros(n, dtype=torch.int32, device=dev)
        self.outs = [torch.empty_like(t) for t in ts]
        total = sum(t.numel() * t.element_size() for t in ts)
        self.codec = ref_lib.RefCodec(int(2.0 * total) + 256 * MIB, dev)  # no cudaMalloc fallback
        self.rows = None

    def _prep(self):
        from oracle import ref_lib
        if getattr(self, "_ready", False):
            return
        self.RL = ref_lib.lib()
        n = self.n = len(self.ts)
        row = self.comp.size(1)
        self.a_in = ref_lib._parr([t.data_ptr() for t in self.ts])
        self.a_sz = ref_lib._uarr([t.numel() if self.as_float else t.numel() * t.element_size() for t in self.ts])
        self.a_rows = ref_lib._parr([self.comp.data_ptr() + i * row for i in range(n)])
        self.a_out = ref_lib._parr([t.data_ptr() for t in self.outs])
        self.tptr, self.tbytes = self.codec.temp.data_ptr(), self.codec.temp.numel()
        self._ready = True

    def _stream(self):
        return self.torch.cuda.current_stream().cuda_stream

    def encode(self):
        self._prep()
        if self.as_float:
            self.RL.ref_float_compress(self.tptr, self.tbytes, self.ft, self.pb, 0, self.n, self.a_in, self.a_sz, self.a_rows,
                                       self.sizes.data_ptr(), self._stream())
        else:
            self.RL.ref_ans_encode_pointer(self.tptr, self.tbytes, self.pb, 0, self.n, self.a_in, self.a_sz, self.a_rows,
                                           self.sizes.data_ptr(), self._stream())

    def bind_rows(self):
        hs = self.sizes.cpu().tolist()
        self.rows = [self.comp[i, :hs[i]] for i in range(len(self.ts))]
        return hs

    def decode(self):
        self._prep()
        if self.as_float:
            self.RL.ref_float_decompress(self.tptr, self.tbytes, self.ft, self.pb, 0, 1, self.n, self.a_rows, self.a_out,
                                         self.a_sz, None, None, self._stream())
        else:
            self.RL.ref_ans_decode_pointer(self.tptr, self.tbytes, self.pb, 0, self.n, self.a_rows, self.a_out, self.a_sz,
                                           None, None, self._stream())

    def api_encode(self):
        self.encode()

    def api_decode(self):
        self.decode()

    launches_per_step = 0


DUMP_SAMPLES = 4 * MIB  # values sampled from the archives and from the decoded batch: 2 x 16 MiB of float32


def dump_outputs(out_dir, torch, codec, kind):
    """Writes what the last codec step returned to its caller, so that two builds can be compared on the
    same inputs: the compressed sizes (float64) and a fixed, seeded sample of the archives and of the
    decoded batch (float32, both exact).  The format leaves some archive bytes free (where each block's
    stream sits in the data section, padding), and they differ from run to run, so each archive is first
    reduced to its defined fields in a fixed order (oracle.defined_fields).  Sample positions are drawn over
    the whole row width, which depends on the input sizes only; a position past that reduced archive reads -1."""
    import numpy as np

    from oracle import oracle as O

    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(2024)
    n, cols = codec.comp.shape
    k = DUMP_SAMPLES // n
    hs = codec.sizes.cpu().tolist()
    ft = {"bf16": O.BF16, "f16": O.F16}.get(kind, 0)
    arch = np.full((n, k), -1, np.float32)
    for i, h in enumerate(hs):
        fields = O.defined_fields(codec.comp[i, :h].cpu().numpy(), ft)
        canon = np.frombuffer(b"".join(fields.values()), np.uint8)
        pos = np.sort(rng.integers(0, cols, k))
        inside = pos < canon.size
        arch[i, inside] = canon[pos[inside]]
    dec = [o[torch.from_numpy(np.sort(rng.integers(0, o.numel(), k))).to(o.device)].float() for o in codec.outs]
    np.save(os.path.join(out_dir, "compressed_sizes.npy"), np.array(hs, np.float64))
    np.save(os.path.join(out_dir, "compressed_sample.npy"), arch)
    np.save(os.path.join(out_dir, "decompressed_sample.npy"), torch.stack(dec).cpu().numpy())


def cpu_baseline(kind, batch, per, budget_s=12.0, pb=10):
    """Oracle port on the host cores, bounded sample of the same workload.  One C call takes the whole
    sample batch and spreads split / histogram / block coding / packing (and the inverse) over all
    cores (oracle/dietgpu_oracle.c dgo_batch_roundtrip); the data is generated outside the timing."""
    import numpy as np
    import torch

    from oracle import oracle as O

    cores = O.num_threads()
    g = torch.Generator().manual_seed(4321)
    # enough members to give every core work, capped so that generation stays a few seconds
    members = max(1, min(batch, max(8, min(64, cores)), (512 * MIB) // max(1, per * (1 if kind == "bytes" else 2))))
    arrs = []
    for i in range(members):
        if kind == "bytes":
            p = 1.0 / np.arange(1, 257)
            p /= p.sum()
            arrs.append(np.random.default_rng(4321 + i).choice(256, size=per, p=p).astype(np.uint8))
        else:
            x = torch.randn(per, generator=g)
            if kind == "f16":
                arrs.append(torch.relu(x).to(torch.float16).view(torch.int16).numpy().view(np.uint16))
            else:
                arrs.append(x.to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16))
    ft = {"bf16": O.BF16, "f16": O.F16}.get(kind, 0)
    nbytes = sum(a.nbytes for a in arrs)
    t_enc = t_dec = 0.0
    reps = 0
    t0 = time.perf_counter()
    while reps < 2 or (time.perf_counter() - t0 < budget_s and reps < 50):
        _, outs, te, td = O.batch_roundtrip(ft, arrs, pb)
        if reps == 0:
            assert all(np.array_equal(o, a) for o, a in zip(outs, arrs))  # first pass also warms the pages
        else:
            t_enc += te
            t_dec += td
        reps += 1
    total = nbytes * (reps - 1)
    return {
        "value": round(2 * total / (t_enc + t_dec) / 1e9, 3), "unit": "GB/s", "cores": cores, "kind": "port",
        "encode_gbs": round(total / t_enc / 1e9, 3), "decode_gbs": round(total / t_dec / 1e9, 3),
        "sample": f"{members} members x {reps - 1} timed reps of the workload ({nbytes / MIB:.0f} MiB per rep), "
                  f"oracle/dietgpu_oracle.c dgo_batch_roundtrip: every phase OpenMP-parallel over members x blocks",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--all-workloads", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--no-detail", action="store_true", help="skip the short runs of the other BASELINE workloads")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0: compressed sizes, a seeded "
                         "sample of the archives and of the decoded batch) to DIR/<name>.npy; inputs are seeded, so "
                         "runs with the same arguments can be compared")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device; dietgpu_b200 has no CPU fallback"}))
        sys.exit(1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from oracle import ref_lib
    use_ref_gpu = args.impl == "reference" and ref_lib.available()
    if args.impl == "reference" and not use_ref_gpu:
        # no compiled reference here: the reference arm is the CPU port
        if args.dump_outputs:
            ap.error("--dump-outputs: the CPU port that stands in for a missing reference build has no outputs to dump")
        if rank == 0:
            kind, batch, per, desc = WORKLOADS[args.workload]
            cb = cpu_baseline(kind, batch, per, budget_s=60.0, pb=PROB_BITS.get(args.workload, 10))
            line = {"metric": "encode+decode GB/s (uncompressed bytes / time)", "value": cb["value"], "unit": "GB/s",
                    "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "u8/u32 integer", "data": "synthetic", "config": {"workload": desc},
                    "cpu_baseline": cb,
                    "e2e": {"value": cb["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
            print(json.dumps(line))
        return

    def run_workload(name, steps, warmup, full):
        kind, batch, per, desc = WORKLOADS[name]
        pb = PROB_BITS.get(name, 10)
        ts = make_batch(torch, kind, batch, per, 1234 + 1000 * rank, dev)
        codec = RefGpuCodec(torch, kind, ts, pb) if use_ref_gpu else OursCodec(torch, kind, ts, pb)
        ubytes = sum(t.numel() * t.element_size() for t in ts)
        stream = torch.cuda.current_stream()

        codec.encode()
        hs = codec.bind_rows()
        codec.decode()
        torch.cuda.synchronize()
        it = torch.int16 if kind != "bytes" else torch.uint8
        verified = all(torch.equal(a.view(it), b.view(it)) for a, b in zip(ts, codec.outs))
        cbytes = int(sum(hs))

        for _ in range(warmup):
            codec.encode()
            codec.decode()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local)
        if full and rank == 0:
            sampler.start()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps + 1)]
        launches0 = 0
        if not use_ref_gpu:
            from dietgpu_b200 import capi as _capi
            launches0 = _capi.get_option("launches")  # the library's own count of its kernel launches
        ev[0].record(stream)
        for i in range(steps):
            codec.encode()
            ev[2 * i + 1].record(stream)
            codec.decode()
            ev[2 * i + 2].record(stream)
        torch.cuda.synchronize()
        launches = (_capi.get_option("launches") - launches0) if not use_ref_gpu else 0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        clocks = sampler.stop() if (full and rank == 0) else None
        t_enc = sum(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(steps)) / 1e3
        t_dec = sum(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(steps)) / 1e3
        t_tot = ev[0].elapsed_time(ev[2 * steps]) / 1e3
        if world > 1:
            tt = torch.tensor([t_tot, t_enc, t_dec], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_tot, t_enc, t_dec = tt.tolist()
            # plumbing only: every rank learns every archive size
            allsz = torch.empty(world * len(hs), dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(allsz, codec.sizes)
            cbytes_all = int(allsz.sum().item())
        else:
            cbytes_all = cbytes
        res = {
            "desc": desc, "kind": kind, "batch": batch, "ubytes": ubytes, "cbytes": cbytes,
            "ratio": round(cbytes / ubytes, 4), "verified": bool(verified),
            "t_tot": t_tot, "t_enc": t_enc, "t_dec": t_dec,
            "encode_gbs": world * ubytes * steps / t_enc / 1e9, "decode_gbs": world * ubytes * steps / t_dec / 1e9,
            "value": world * 2 * ubytes * steps / t_tot / 1e9, "clocks": clocks, "cbytes_all": cbytes_all,
            "launches": launches, "prob_bits": pb,
        }
        if full and args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, torch, codec, kind)
        if not full:
            return res

        # ---- per-kernel durations (CUDA events around every launch, same stream) ----
        if not use_ref_gpu:
            from dietgpu_b200 import capi
            capi.set_option("timing", 1)
            capi.kernel_times()
            for _ in range(steps):
                codec.encode()
                codec.decode()
            kt = capi.kernel_times()
            capi.set_option("timing", 0)
            res["kernels"] = {k: {"ms_avg": v[0] / max(v[1], 1), "launches": v[1]} for k, v in kt.items() if v[1]}

            # ---- the same step captured once into a CUDA graph and replayed (a batch of <= 64 members carries its
            #      member table in the kernel parameters, so a call reads no host memory after it returns) ----
            try:
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    codec.encode()
                    codec.decode()
                for _ in range(warmup):
                    g.replay()
                torch.cuda.synchronize()
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record(stream)
                for _ in range(steps):
                    g.replay()
                g1.record(stream)
                torch.cuda.synchronize()
                tg = g0.elapsed_time(g1) / 1e3
                okg = all(torch.equal(a.view(it), b.view(it)) for a, b in zip(ts, codec.outs))
                res["graph_replay"] = {"value": round(2 * ubytes * steps / tg / 1e9, 2), "unit": "GB/s (this rank)",
                                       "ms_per_step": round(tg / steps * 1e3, 4), "verified": bool(okg),
                                       "note": "encode+decode of the step captured into one CUDA graph, replayed; not the headline"}
                del g
            except Exception as ex:  # noqa: BLE001
                res["graph_replay"] = {"unavailable": str(ex)[:160]}

        # ---- end to end through the public API with HOST buffers ----
        # host staging: the members are slices of ONE pinned buffer each way (both arms)
        def pinned_like(tensors):
            flat = torch.empty(sum(t.numel() * t.element_size() for t in tensors), dtype=torch.uint8, pin_memory=True)
            out, off = [], 0
            for t in tensors:
                nb = t.numel() * t.element_size()
                out.append(flat[off:off + nb].view(t.dtype).view(t.shape))
                off += nb
            return out

        pin_in = pinned_like(ts)
        for p, t in zip(pin_in, ts):
            p.copy_(t)
        pin_comp = torch.empty(codec.comp.shape, dtype=torch.uint8, pin_memory=True)
        pin_out = pinned_like(ts)
        e2e_steps = max(2, min(steps, 5))
        h2d = d2h = 0

        def e2e_step():
            nonlocal h2d, d2h
            for t, p in zip(ts, pin_in):          # host -> device: the step's inputs
                t.copy_(p, non_blocking=True)
            codec.api_encode()
            hs2 = codec.sizes.cpu().tolist()      # device -> host: sizes, then the archives
            for i, n in enumerate(hs2):
                pin_comp[i, :n].copy_(codec.comp[i, :n], non_blocking=True)
            torch.cuda.synchronize()
            for i, n in enumerate(hs2):           # host -> device: the archives
                codec.comp[i, :n].copy_(pin_comp[i, :n], non_blocking=True)
            codec.rows = [codec.comp[i, :n] for i, n in enumerate(hs2)]
            codec.api_decode()
            for o, p in zip(codec.outs, pin_out):  # device -> host: the decoded floats
                p.copy_(o, non_blocking=True)
            torch.cuda.synchronize()
            h2d = ubytes + sum(hs2)
            d2h = sum(hs2) + 4 * len(hs2) + ubytes

        def timed(step_fn):
            step_fn()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                step_fn()
            torch.cuda.synchronize()
            t = time.perf_counter() - t0
            if world > 1:
                tt = torch.tensor([t], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t = tt.item()
            ok = all(torch.equal(a.view(it), b.view(it).to(dev)) for a, b in zip(ts, pin_out))
            for p in pin_out:
                p.zero_()
            return t, ok

        t_plain, ok_plain = timed(e2e_step)
        plain = {"value": round(world * 2 * ubytes * e2e_steps / t_plain / 1e9, 3), "unit": "GB/s",
                 "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                 "verified": bool(ok_plain),
                 "note": "device-tensor operators, one stream: pinned host input -> H2D -> compress -> D2H archives "
                         "-> H2D archives -> decompress -> D2H output (what the reference's API affords)"}
        if use_ref_gpu:
            res["e2e"] = plain
            return res

        # ours: the host-buffer front end (dietgpu_b200.HostCodec), same bytes over the link.
        #  e2e_sync : compress(...) then decompress(...), each a blocking call; inside each call upload /
        #             codec / download of different member groups overlap (H2D and D2H run at once)
        #  e2e      : the same calls through the async API, software-pipelined ACROSS steps: while step i
        #             is decompressed (archives up, floats down), step i+1 is already being compressed
        #             (floats up, archives down), so both directions of the link stay busy.  Every step
        #             still moves all of its bytes inside the timed region, and the last step's output
        #             is verified.
        import dietgpu_b200 as dg
        hc = dg.HostCodec(kind != "bytes", pin_in, device=dev, groups=8, prob_bits=pb)
        pin_comp2 = [torch.empty((len(ts), hc.max_archive_bytes()), dtype=torch.uint8, pin_memory=True) for _ in range(2)]

        def host_step():
            nonlocal h2d, d2h
            hs3 = hc.compress(pin_in, pin_comp2[0])
            hc.decompress([pin_comp2[0][i, :n] for i, n in enumerate(hs3)], pin_out)
            h2d = ubytes + sum(hs3)
            d2h = sum(hs3) + 4 * len(hs3) + ubytes + len(hs3)

        t_host, ok_host = timed(host_step)
        sync = {"value": round(world * 2 * ubytes * e2e_steps / t_host / 1e9, 3), "unit": "GB/s",
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                "verified": bool(ok_host),
                "note": "dietgpu_b200.HostCodec.compress() then .decompress(), blocking calls: pinned host input -> "
                        "archives in pinned host memory -> pinned host output; 8 member groups pipelined over "
                        "upload / codec / download streams inside each call"}

        def pipelined(nsteps):
            # step i = compress batch -> archives (host) -> decompress -> output (host); compress of step i+1
            # is enqueued before decompress of step i is awaited
            pend = hc.compress_async(pin_in, pin_comp2[0])
            for i in range(nsteps):
                hs3 = pend.finish()
                rows = [pin_comp2[i & 1][j, :n] for j, n in enumerate(hs3)]
                pd = hc.decompress_async(rows, pin_out)
                if i + 1 < nsteps:
                    pend = hc.compress_async(pin_in, pin_comp2[(i + 1) & 1])
                    pend.finish()
                pd.finish()
            return hs3

        pipelined(2)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for p in pin_out:
            p.zero_()
        psteps = max(4, 2 * e2e_steps)
        t0 = time.perf_counter()
        hs4 = pipelined(psteps)
        torch.cuda.synchronize()
        t_pipe = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([t_pipe], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_pipe = tt.item()
        ok_pipe = all(torch.equal(a.view(it), b.view(it).to(dev)) for a, b in zip(ts, pin_out))
        res["e2e"] = {"value": round(world * 2 * ubytes * psteps / t_pipe / 1e9, 3), "unit": "GB/s",
                      "h2d_bytes_per_step": int(ubytes + sum(hs4)), "d2h_bytes_per_step": int(sum(hs4) + 4 * len(hs4) + ubytes + len(hs4)),
                      "steps": psteps, "verified": bool(ok_pipe),
                      "note": "dietgpu_b200.HostCodec async API (compress_async / decompress_async + finish), steps "
                              "software-pipelined: compress of step i+1 overlaps decompress of step i, so H2D and D2H "
                              "run concurrently (link measured full duplex: profiles/r02_pcie_duplex.txt); every step "
                              "uploads its inputs and downloads its archives and outputs inside the timed region"}
        res["e2e_sync"] = sync
        res["e2e_plain"] = plain
        return res

    main_res = run_workload(args.workload, args.steps, args.warmup, True)
    kind = main_res["kind"]
    peak, peak_src = load_peaks()
    ubytes, cbytes, steps = main_res["ubytes"], main_res["cbytes"], args.steps

    # ---- roofline (algorithmic bytes per launch / event-timed duration of that kernel) ----
    roofline = None
    roofline_all = {}
    if "kernels" in main_res:
        # compulsory bytes per launch (DESIGN.md section 5): the statistics kernel is a pure read of the raw
        # input (U); the coder reads the raw input again and writes the whole archive (U + C: stored planes + ANS
        # part for float kinds); the decoder reads the archive and writes the output (C + U).  The single-launch
        # (fused) encoder does the statistics read and the coder's work in one launch (counted U + C, SURVEY 8d).
        alg = {"stats": ubytes, "encode": ubytes + cbytes, "decode": cbytes + ubytes, "encode_fused": ubytes + cbytes}
        for k, v in main_res["kernels"].items():
            if k in alg:
                a = alg[k] / (v["ms_avg"] / 1e3) / 1e9
                roofline_all[k] = {"bound": "hbm", "achieved": round(a, 1), "peak": peak, "unit": "GB/s",
                                   "frac": round(a / peak, 4), "ms": round(v["ms_avg"], 4),
                                   "algorithmic_bytes": int(alg[k])}
        # DRAM traffic per launch from the committed `ncu --set full` captures of the same workload
        # (profiles/r*_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum), else null
        traffic = {}
        try:
            import glob
            tf = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))[-1]
            for k, v in json.load(open(tf)).items():
                if v.get("workload") == args.workload:
                    traffic[k] = int(v["traffic"])
        except Exception:  # noqa: BLE001
            pass
        for k in roofline_all:
            roofline_all[k]["traffic"] = traffic.get(k)
        dom = max(roofline_all, key=lambda k: roofline_all[k]["ms"])
        roofline = dict(roofline_all[dom])
        roofline.update({"kernel": dom, "peak_source": peak_src})
        # direction-level figures (SURVEY 8d: encode = decode = 2F + C_f algorithmic bytes)
        for d, t in (("encode_direction", main_res["t_enc"]), ("decode_direction", main_res["t_dec"])):
            a = (ubytes + cbytes) * steps / t / 1e9
            roofline_all[d] = {"achieved": round(a, 1), "frac": round(a / peak, 4), "unit": "GB/s"}

    # every BASELINE config in the same line (north_star: bytes prec 10/11, fp16, bf16, at every N):
    # short runs of the other workloads, same timing rules, every rank takes part
    detail = {}
    if not args.no_detail:
        dsteps = max(5, args.steps // 5)
        for w in sorted(WORKLOADS):
            if w == args.workload:
                r, st = main_res, args.steps
            else:
                torch.cuda.empty_cache()
                r, st = run_workload(w, dsteps, 3, False), dsteps
            alg_dir = (r["ubytes"] + r["cbytes"]) * world  # SURVEY 8d: U + C per direction
            detail[w] = {"desc": r["desc"], "prob_bits": r["prob_bits"], "steps": st,
                         "encode_gbs": round(r["encode_gbs"], 1), "decode_gbs": round(r["decode_gbs"], 1),
                         "value": round(r["value"], 1), "ratio": r["ratio"], "verified": r["verified"],
                         "encode_roofline_frac": round(alg_dir * st / r["t_enc"] / 1e9 / (peak * world), 4),
                         "decode_roofline_frac": round(alg_dir * st / r["t_dec"] / 1e9 / (peak * world), 4)}

    cb = None
    if rank == 0 and world == 1 and not args.no_cpu:
        kind_, batch_, per_, _ = WORKLOADS[args.workload]
        cb = cpu_baseline(kind_, batch_, per_, pb=PROB_BITS.get(args.workload, 10))

    if rank == 0:
        line = {
            "metric": "encode+decode GB/s (uncompressed bytes / time)",
            "value": round(main_res["value"], 2), "unit": "GB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(main_res["t_tot"] / args.steps * 1e3, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 integer state machine on u8 symbols", "data": "synthetic",
            "config": {"workload": main_res["desc"], "batch": main_res["batch"],
                       "uncompressed_bytes_per_gpu": ubytes, "compressed_bytes_per_gpu": cbytes,
                       "ratio": main_res["ratio"], "prob_bits": main_res["prob_bits"], "checksum": False,
                       "l2": "inputs (256 MiB) + archives (~172 MiB) exceed the 126 MB L2; no explicit flush",
                       "parallelism": f"batch shard x{world}, no data-path collective",
                       "host_binding": numa},
            "encode_gbs": round(main_res["encode_gbs"], 2), "decode_gbs": round(main_res["decode_gbs"], 2),
            "verified_roundtrip": main_res["verified"],
            "gpu_launches": main_res["launches"],  # counted by the library (stats/encode/plan/decode kernels)
            "clocks": main_res["clocks"],
            "e2e": main_res.get("e2e"),
        }
        for k in ("e2e_sync", "e2e_plain", "graph_replay"):
            if main_res.get(k):
                line[k] = main_res[k]
        if use_ref_gpu:
            line["impl"] = "reference"
            line["reference_kind"] = "reference CUDA path (oracle/_ref/libdietgpu_ref.so, sm_100a build of /root/reference)"
        if roofline:
            line["roofline"] = roofline
            line["roofline_all"] = roofline_all
        if cb:
            line["cpu_baseline"] = cb
        if detail:
            line["detail"] = detail
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
