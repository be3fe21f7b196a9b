#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's configuration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--blocks B] [--cls E50] [--dump-outputs DIR]

metric  : "GB/s encode+decode on batched 64KiB blocks" -- raw (uncompressed) bytes per second through one encode pass
          plus one decode pass over the batch (the reference's convention: throughput numerator = uncompressed bytes in
          both directions, src/LZ4.Tests.Helpers/TimedMethod.cs:66-69).  GB = 1e9 bytes.
step    : one pass of the hot path over the whole batch: ONE fast-encode launch over all blocks (raw -> fixed-stride
          slots, both resident in HBM), then the known-size decode of every block (slots -> a reused wave buffer).
workload: configs[1] of BASELINE.json: 2^20 x 64 KiB independent blocks per GPU (64 GiB raw, > 500x the L2, so every
          timed iteration streams from HBM), synthetic entropy class E50 (SURVEY.md 8d) unless --cls says otherwise.
value   : whole-job throughput over all ranks, device-timed (CUDA events, barrier + synchronize on both sides, max over
          ranks), inputs already in HBM.
e2e     : the same metric through the reference-facing C ABI with HOST buffers (pinned), H2D/D2H inside the timed region.
roofline: algorithmic bytes (raw + compressed, SURVEY.md 8d) / CUDA-event duration of the launches, for the kernel that
          dominates the step (the fast encoder -- latency-bound by the exact greedy parse) and, as "roofline_decode",
          for the decoder, the kernel north_star sets the HBM target on.
cpu_baseline / --impl reference: the reference's own original/lz4.c (oracle/_ref, built from /root/reference by
          oracle/Makefile; the oracle port if that file is absent) timed on the host cores with a static block partition.

Multi-GPU: one process per GPU under torch.distributed.run; blocks are independent (doc/compatibility.md:4-7), so ranks
own disjoint block ranges and there is no data-path collective -- "scaling": "weak" (per-GPU work fixed).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BLOCK = 65536
GB = 1e9


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--blocks", type=int, default=1 << 20, help="64 KiB blocks per GPU (default 2^20 = BASELINE configs[1])")
    p.add_argument("--cls", default="E50", choices=["E0", "E50", "E100", "ETEXT"])
    p.add_argument("--wave", type=int, default=1 << 18, help="blocks per decode wave (output buffer reuse)")
    p.add_argument("--e2e-blocks", type=int, default=1 << 14)
    p.add_argument("--cpu-blocks", type=int, default=1 << 15)
    p.add_argument("--lanes", type=int, default=0, help="decode lanes per block (4/8/16/32, +100 staged, 1/2 lane-per-block); 0 = library default (picked per batch)")
    p.add_argument("--stream-gib", type=float, default=16.0, help="BASELINE configs[3]: size of the stream that starts on rank 0")
    p.add_argument("--no-stream", action="store_true")
    p.add_argument("--no-numa", action="store_true")
    p.add_argument("--enc-ctas", type=int, default=0)
    p.add_argument("--no-sweep", action="store_true")
    p.add_argument("--no-hc", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--sweep-blocks", type=int, default=1 << 17)
    p.add_argument("--hc-blocks", type=int, default=1 << 17)
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write what the last timed step returned as DIR/<name>.npy (rank 0's blocks), to compare two builds")
    args = p.parse_args()
    if args.dump_outputs and args.impl == "reference":
        p.error("--dump-outputs dumps the GPU path's outputs; --impl reference has none")
    return args


# ------------------------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md: sample DURING the timed region)
# ------------------------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index; self.samples = []; self.proc = None; self.th = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True); self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# CPU side: the reference's own code on the host cores
# ------------------------------------------------------------------------------------------------------------------
def cpu_codec(cls: str, n_blocks: int, threads: int, repeats: int = 3):
    """Encode + decode n_blocks 64 KiB blocks of class cls with the reference's C code on `threads` host threads."""
    import numpy as np
    import oracle
    from lz4net_b200 import synth
    impl, kind = ("ref", "reference") if oracle.have_ref() else ("port", "port")
    raw = synth.make_blocks(cls, n_blocks, BLOCK, seed=1).reshape(-1)
    slot = oracle.bound(BLOCK)
    so = np.arange(n_blocks, dtype=np.int64) * BLOCK
    do = np.arange(n_blocks, dtype=np.int64) * slot
    sl = np.full(n_blocks, BLOCK, np.int32); dc = np.full(n_blocks, slot, np.int32)
    comp = np.zeros(n_blocks * slot + 64, np.uint8)
    out = np.zeros(n_blocks * BLOCK + 64, np.uint8)
    best_e = best_d = 1e30
    clen = None
    for _ in range(repeats):
        te, clen = oracle.mt_run("encode", impl, raw, so, sl, comp, do, dc, threads)
        td, used = oracle.mt_run("decode", impl, comp, do, clen, out, so, sl, threads)
        best_e, best_d = min(best_e, te), min(best_d, td)
    assert (used == clen).all() and np.array_equal(out[:raw.size], raw), "CPU reference round trip failed"
    nbytes = n_blocks * BLOCK
    return {"kind": kind, "encode_gbs": nbytes / best_e / GB, "decode_gbs": nbytes / best_d / GB,
            "roundtrip_gbs": nbytes / (best_e + best_d) / GB, "ratio": float(clen.sum()) / nbytes,
            "t_enc": best_e, "t_dec": best_d}


def cpu_hc(cls: str, n_blocks: int, threads: int):
    """LZ4HC encode of a small sample with the reference's C code on all host threads (GB/s raw)."""
    import numpy as np
    import oracle
    from lz4net_b200 import synth
    impl = "ref" if oracle.have_ref() else "port"
    raw = synth.make_blocks(cls, n_blocks, BLOCK, seed=3).reshape(-1)
    slot = oracle.bound(BLOCK)
    so = np.arange(n_blocks, dtype=np.int64) * BLOCK; do = np.arange(n_blocks, dtype=np.int64) * slot
    sl = np.full(n_blocks, BLOCK, np.int32); dc = np.full(n_blocks, slot, np.int32)
    comp = np.zeros(n_blocks * slot + 64, np.uint8)
    best = min(oracle.mt_run("encode_hc", impl, raw, so, sl, comp, do, dc, threads)[0] for _ in range(2))
    return n_blocks * BLOCK / best / GB


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path, all host threads, same metric and config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = min(args.cpu_blocks, args.blocks)
    for _ in range(max(args.warmup, 1) - 1):
        cpu_codec(args.cls, min(n, 4096), threads, repeats=1)
    vals = []
    t0 = time.time()
    for _ in range(args.steps):
        r = cpu_codec(args.cls, n, threads, repeats=1)
        vals.append(r)
    ms = (time.time() - t0) * 1e3 / max(args.steps, 1)
    nbytes = n * BLOCK
    t = sum(v["t_enc"] + v["t_dec"] for v in vals) / len(vals)
    value = nbytes / t / GB
    sample = f"{n} x 64 KiB blocks of class {args.cls} per step ({nbytes / 2**20:.0f} MiB raw), encode then decode, static partition over {threads} threads"
    line = {
        "impl": "reference", "metric": "GB/s encode+decode on batched 64KiB blocks", "value": round(value, 3), "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{args.blocks} x 64KiB independent blocks per GPU, class {args.cls} (BASELINE configs[1]); CPU arm times a bounded sample",
                   "block_size": BLOCK, "class": args.cls},
        "encode_gbs": round(sum(v["encode_gbs"] for v in vals) / len(vals), 3),
        "decode_gbs": round(sum(v["decode_gbs"] for v in vals) / len(vals), 3),
        "cpu_baseline": {"value": round(value, 3), "unit": "GB/s", "cores": threads, "kind": vals[0]["kind"], "sample": sample},
        "e2e": {"value": round(value, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# host placement: run this rank's threads (and first-touch its pinned staging) on the NUMA node its GPU hangs off
# ------------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(index: int):
    """Returns a dict describing what was done.  PCIe traffic of GPUs on the far socket crosses the inter-socket link; with 8
    ranks each streaming raw + compressed bytes both ways that link, not PCIe, is what the e2e numbers hit first."""
    info = {"bound": False}
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return info
        dom, rest = bus.split(":", 1)
        dev = f"{dom[-4:]}:{rest}"
        node = int(open(f"/sys/bus/pci/devices/{dev}/numa_node").read().strip())
        info.update({"pci": dev, "numa_node": node})
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            info.update({"bound": True, "cpus": len(cpus)})
    except Exception as e:                       # placement is an optimisation, never a reason to fail the run
        info["error"] = str(e)[:100]
    return info


# ------------------------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------------------------
class Workload:
    """Device-resident batch: raw blocks, fixed-stride encoder slots, a reused decode wave buffer."""

    def __init__(self, ctx, n_blocks, cls, wave, seed=1, first_block=0):
        import torch
        from lz4net_b200 import batch, synth
        self.torch, self.batch, self.ctx = torch, batch, ctx
        self.n, self.cls = n_blocks, cls
        self.slot = BLOCK + BLOCK // 255 + 16
        self.wave = min(wave, n_blocks)
        dev = "cuda"
        self.raw = torch.empty(n_blocks * BLOCK, dtype=torch.uint8, device=dev)
        chunk = 1 << 16
        for b0 in range(0, n_blocks, chunk):
            m = min(chunk, n_blocks - b0)
            batch.synth_fill(ctx, self.raw[b0 * BLOCK:], m, BLOCK, synth.CLASS_ID[cls], seed=seed, first_block=first_block + b0)
        self.slots = torch.empty(n_blocks * self.slot, dtype=torch.uint8, device=dev)
        self.out = torch.empty(self.wave * BLOCK, dtype=torch.uint8, device=dev)
        idx = torch.arange(n_blocks, dtype=torch.int64, device=dev)
        self.raw_off = idx * BLOCK
        self.slot_off = idx * self.slot
        self.out_off = (idx % self.wave) * BLOCK
        self.raw_len = torch.full((n_blocks,), BLOCK, dtype=torch.int32, device=dev)
        self.slot_cap = torch.full((n_blocks,), self.slot, dtype=torch.int32, device=dev)
        self.clen = torch.zeros(n_blocks, dtype=torch.int32, device=dev)
        self.used = torch.zeros(n_blocks, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()

    def encode(self, hc=False):
        self.batch.encode(self.ctx, self.raw, self.raw_off, self.raw_len, self.slots, self.slot_off, self.slot_cap, self.clen, hc=hc)

    def decode_wave(self, w):
        b0 = w * self.wave; b1 = min(self.n, b0 + self.wave)
        s = slice(b0, b1)
        self.batch.decode(self.ctx, self.slots, self.slot_off[s], self.clen[s], self.out, self.out_off[s], self.raw_len[s], self.used[s], known=True)
        return b0, b1

    @property
    def n_waves(self):
        return (self.n + self.wave - 1) // self.wave

    def verify(self):
        """Round trip over the full batch: every decoded wave equals its raw blocks, every stream fully consumed."""
        torch = self.torch
        self.encode()
        for w in range(self.n_waves):
            b0, b1 = self.decode_wave(w)
            torch.cuda.synchronize()
            assert torch.equal(self.out[: (b1 - b0) * BLOCK], self.raw[b0 * BLOCK: b1 * BLOCK]), f"decode mismatch in wave {w}"
        assert torch.equal(self.used, self.clen), "decoder did not consume exactly the encoder's bytes"
        assert int((self.clen <= 0).sum()) == 0
        return int(self.clen.sum())

    def timed_step(self, ev):
        """Enqueue one step; ev = list of (start, end) CUDA event pairs: [encode, decode...]."""
        ev[0][0].record(); self.encode(); ev[0][1].record()
        for w in range(self.n_waves):
            ev[1 + w][0].record(); self.decode_wave(w); ev[1 + w][1].record()


DUMP_SAMPLE_BLOCKS = 64


def dump_outputs(work, out_dir):
    """Writes what the last step returned to its caller as float32 arrays (byte values and lengths are exact in float32):
    every block's compressed length and the bytes the decoder consumed, and, for a fixed seeded sample of the blocks whose
    decoded bytes are still in the reused decode buffer (the last wave), their compressed bytes (zero past the length)
    and decoded bytes.  40 MiB at the default 2^20 blocks."""
    import numpy as np
    torch = work.torch
    torch.cuda.synchronize()
    first = (work.n_waves - 1) * work.wave
    blocks = np.sort(np.random.default_rng(0).choice(np.arange(first, work.n), min(DUMP_SAMPLE_BLOCKS, work.n - first), replace=False))
    idx = torch.from_numpy(blocks).to(work.clen.device)
    comp = work.slots.view(work.n, work.slot)[idx]
    comp[torch.arange(work.slot, device=idx.device)[None, :] >= work.clen[idx].unsqueeze(1)] = 0
    arrays = {"compressed_lengths": work.clen, "decode_consumed": work.used, "sample_blocks": blocks,
              "compressed_sample": comp, "decoded_sample": work.out.view(work.wave, BLOCK)[idx - first]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a if isinstance(a, np.ndarray) else a.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if name == "sample_blocks" else np.float32))


def measure_pair(work, steps, warmup, hc=False):
    """Device-timed encode and decode of a workload (used by the sweep / HC sections). Returns seconds per pass."""
    torch = work.torch
    for _ in range(warmup):
        work.encode(hc=hc)
        for w in range(work.n_waves):
            work.decode_wave(w)
    torch.cuda.synchronize()
    te = td = 0.0
    for _ in range(steps):
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(); work.encode(hc=hc); e1.record()
        for w in range(work.n_waves):
            work.decode_wave(w)
        e2.record(); torch.cuda.synchronize()
        te += e0.elapsed_time(e1) * 1e-3; td += e1.elapsed_time(e2) * 1e-3
    return te / steps, td / steps


class E2E:
    """The metric through the C ABI with HOST buffers: lz4b200_encode_batch_packed + lz4b200_decode_batch (MEM_HOST), every
    H2D / D2H copy inside the timed calls.  kind: "pinned" (cudaHostAlloc), "pageable" (plain numpy -- what a `fixed` byte[]
    of a managed caller is), "registered" (pageable, page-locked once with lz4b200_host_register)."""

    def __init__(self, device, cls, n_blocks, kind="pinned", seed=7):
        import numpy as np
        import torch
        import lz4net_b200
        from lz4net_b200 import native, synth
        self.np, self.torch, self.native = np, torch, native
        self.ctx = lz4net_b200.Context(device)
        self.n, self.kind = n_blocks, kind
        slot = BLOCK + BLOCK // 255 + 16
        def buf(nbytes):
            if kind == "pinned":
                return torch.empty(nbytes, dtype=torch.uint8).pin_memory()
            t = torch.from_numpy(np.empty(nbytes, np.uint8))
            if kind == "registered":
                native.check(native.lib().lz4b200_host_register(t.data_ptr(), nbytes), "host_register")
            return t
        self.raw, self.comp, self.out = buf(n_blocks * BLOCK), buf(n_blocks * slot), buf(n_blocks * BLOCK)
        for b0 in range(0, n_blocks, 1024):
            m = min(1024, n_blocks - b0)
            self.raw[b0 * BLOCK:(b0 + m) * BLOCK] = torch.from_numpy(synth.make_blocks(cls, m, BLOCK, seed=seed, first_block=b0).reshape(-1))
        self.so = np.arange(n_blocks, dtype=np.int64) * BLOCK
        self.sl = np.full(n_blocks, BLOCK, np.int32); self.dc = np.full(n_blocks, slot, np.int32)
        self.clen = np.zeros(n_blocks, np.int32); self.used = np.zeros(n_blocks, np.int32); self.coff = np.zeros(n_blocks + 1, np.int64)

    def encode(self):
        self.ctx.encode_batch_packed_ptr(self.raw.data_ptr(), self.so.ctypes.data, self.sl.ctypes.data, self.dc.ctypes.data, self.comp.data_ptr(),
                                         self.comp.numel(), self.coff.ctypes.data, self.clen.ctypes.data, self.n, hc=False)

    def decode(self):
        self.ctx.decode_batch_ptr(self.comp.data_ptr(), self.coff.ctypes.data, self.clen.ctypes.data, self.out.data_ptr(), self.so.ctypes.data,
                                  self.sl.ctypes.data, self.used.ctypes.data, self.n, known=True, device=False)

    def check(self):
        assert self.torch.equal(self.out, self.raw) and (self.used == self.clen).all(), "e2e round trip failed"

    def close(self):
        if self.kind == "registered":
            for t in (self.raw, self.comp, self.out):
                self.native.lib().lz4b200_host_unregister(t.data_ptr())
        self.ctx.close()


def e2e_sequential(device, cls, n_blocks, steps, warmup, kind="pinned"):
    """encode then decode, one call after the other (one caller thread)."""
    w = E2E(device, cls, n_blocks, kind)
    te = td = 0.0
    for i in range(warmup + steps):
        t0 = time.perf_counter(); w.encode(); t1 = time.perf_counter(); w.decode(); t2 = time.perf_counter()
        if i >= warmup:
            te += t1 - t0; td += t2 - t1
    w.check()
    csum = int(w.clen.sum()); nbytes = n_blocks * BLOCK
    w.close()
    return {"t_enc": te / steps, "t_dec": td / steps, "bytes": nbytes, "h2d": nbytes + csum, "d2h": csum + nbytes}


def e2e_pipelined(device, cls, n_blocks, steps, warmup):
    """Two caller threads with a context each (the library's contexts serialise their callers): the encode of step i+1 runs
    while step i is decoded, so both PCIe directions carry raw + compressed bytes at the same time instead of one direction
    idling per call.  Returns seconds per step (one step = one encode + one decode of n_blocks blocks)."""
    a, b = E2E(device, cls, n_blocks, "pinned", seed=7), E2E(device, cls, n_blocks, "pinned", seed=8)
    a.encode(); b.encode()                       # both batches hold valid streams before the pipeline starts
    def run(k):
        # step 2j uses batch a, step 2j+1 batch b; decode(i) overlaps encode(i+1)
        t = [None]
        def enc(w): w.encode()
        for i in range(k):
            cur, nxt = (a, b) if i % 2 == 0 else (b, a)
            th = threading.Thread(target=enc, args=(nxt,)); th.start()
            cur.decode(); th.join()
    run(max(warmup, 1) * 2)
    t0 = time.perf_counter(); run(steps * 2); dt = time.perf_counter() - t0
    a.check(); b.check()
    csum = int(a.clen.sum()); nbytes = n_blocks * BLOCK
    a.close(); b.close()
    # 2 * steps decodes and 2 * steps encodes ran: per step (one encode + one decode) that is dt / (2 * steps)
    return {"t_step": dt / (2 * steps), "bytes": nbytes, "h2d": nbytes + csum, "d2h": csum + nbytes}


def stream_section(ctx, args, rank, world, dev):
    """BASELINE configs[3]: ONE stream that starts on rank 0, chunked into 64 KiB blocks, encoded by all ranks, payloads back
    on rank 0 in stream order -- and the mirror image.  Strong scaling: the stream is the same size whatever the world size.
    Device-timed per phase (CUDA events on the stream the NCCL calls are ordered with), max over ranks."""
    import torch
    import torch.distributed as dist
    from lz4net_b200 import batch, shard, synth
    nb = int(args.stream_gib * (1 << 30)) // BLOCK
    torch.cuda.empty_cache()
    enc, dec = shard.gpu_codec(ctx, BLOCK)
    raw = None
    win, werr = None, None
    if world > 1:                                               # set up once, like the communicator
        try:
            win = shard.StreamWindow(nb, BLOCK, rank, world, device=dev)
        except RuntimeError as e:                               # (raised on every rank alike: peer memory not available here)
            werr = str(e)[:300]
    if rank == 0:
        raw = win.raw if win is not None else torch.empty(nb * BLOCK, dtype=torch.uint8, device=dev)
        for b0 in range(0, nb, 65536):
            batch.synth_fill(ctx, raw[b0 * BLOCK:], min(65536, nb - b0), BLOCK, synth.CLASS_ID[args.cls], seed=6, first_block=b0)
    def ev():
        return torch.cuda.Event(enable_timing=True)
    best = None
    for it in range(2):                                         # the first pass warms NCCL's connections up
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        if world > 1:
            lens, off, packed = shard.encode_stream_sharded(raw, nb, BLOCK, enc, rank, world, device=dev)
        else:
            packed, lens = enc(raw, nb)
        e1.record()
        if world > 1:
            back = shard.decode_stream_sharded(packed, lens, nb, BLOCK, dec, rank, world, device=dev)
        else:
            back = dec(packed, lens, nb)
        e2.record(); torch.cuda.synchronize()
        te, td = shard.reduce_max([e0.elapsed_time(e1) * 1e-3, e1.elapsed_time(e2) * 1e-3], device="cuda")
        best = (te, td)
    # ---- the same job over peer memory: the stream's buffers are a CUDA-IPC window on the root, the peers pull / push
    # their ranges with copy-engine transfers (lz4b200_peer_copy) that overlap the codec kernels piece by piece
    wres = {"unavailable": werr} if werr else None
    if win is not None:
        keep = raw.clone() if rank == 0 else None               # (the decode overwrites win.raw: compare against a copy)
        for it in range(2):
            torch.cuda.synchronize(); dist.barrier()
            e0, e1, d0, d1 = ev(), ev(), ev(), ev()
            e0.record()
            wl, wo, wp = shard.encode_stream_window(win, enc, pieces=4)
            e1.record()
            if rank == 0 and it == 1:
                wsame = bool(torch.equal(wl, lens)) and bool(torch.equal(wp, packed))
                win.raw.zero_()
            torch.cuda.synchronize(); dist.barrier()
            d0.record()
            wback = shard.decode_stream_window(win, dec, pieces=4)
            d1.record(); torch.cuda.synchronize()
            wte, wtd = shard.reduce_max([e0.elapsed_time(e1) * 1e-3, d0.elapsed_time(d1) * 1e-3], device="cuda")
        if rank == 0:
            n_ = nb * BLOCK
            wres = {"transport": "CUDA IPC window on rank 0 + copy-engine peer copies (lz4b200_peer_copy), 4 pieces per rank, overlapped with the kernels",
                    "encode_gbs": round(n_ / wte / GB, 1), "decode_gbs": round(n_ / wtd / GB, 1), "roundtrip_gbs": round(n_ / (wte + wtd) / GB, 1),
                    "identical_to_send_recv_result": wsame, "roundtrip_exact": bool(torch.equal(wback, keep))}
            raw.copy_(keep)
        del keep
    # ---- the same stream with the limiter removed: the blocks LAND sharded (rank r holds its contiguous block range, as a
    # multi-GPU producer would leave them) and stay sharded; the only exchange is 4 bytes of length per block (all-gather).
    a, b = shard.strong_range(rank, world, nb)
    mine = torch.empty(max(b - a, 1) * BLOCK, dtype=torch.uint8, device=dev)
    for b0 in range(a, b, 65536):
        batch.synth_fill(ctx, mine[(b0 - a) * BLOCK:], min(65536, b - b0), BLOCK, synth.CLASS_ID[args.cls], seed=6, first_block=b0)
    for it in range(2):                                         # (the first pass pays for the allocations)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        rp, rl = enc(mine[: (b - a) * BLOCK], b - a)
        if world > 1 and nb % world == 0:
            lens_all = [torch.empty(shard.strong_range(r, world, nb)[1] - shard.strong_range(r, world, nb)[0], dtype=torch.int32, device=dev) for r in range(world)]
            dist.all_gather(lens_all, rl)                           # (block counts differ by at most one: equal here, 2^18 blocks)
        e1.record()
        rback = dec(rp, rl, b - a)
        e2.record(); torch.cuda.synchronize()
        rte, rtd = shard.reduce_max([e0.elapsed_time(e1) * 1e-3, e1.elapsed_time(e2) * 1e-3], device="cuda")
    rok, = shard.reduce_sum([0.0 if torch.equal(rback, mine[: (b - a) * BLOCK]) else 1.0], device="cuda")
    del mine, rback, rp
    res = None
    if rank == 0:
        ok = bool(torch.equal(back, raw))
        # sampled byte identity with the one-GPU encode of the same blocks (rank 0 encodes the sample by itself)
        idx = list(range(0, nb, max(nb // 64, 1)))[:64]
        sample = torch.cat([raw[i * BLOCK:(i + 1) * BLOCK] for i in idx])
        sp, sl = enc(sample, len(idx))
        so = torch.zeros(len(idx) + 1, dtype=torch.int64, device=dev); so[1:] = torch.cumsum(sl.to(torch.int64), 0)
        offs = torch.zeros(nb + 1, dtype=torch.int64, device=dev); offs[1:] = torch.cumsum(lens.to(torch.int64), 0)
        same = True
        for j, i in enumerate(idx):
            a0, a1 = int(offs[i]), int(offs[i + 1]); b0, b1 = int(so[j]), int(so[j + 1])
            same = same and (a1 - a0 == b1 - b0) and bool(torch.equal(packed[a0:a1], sp[b0:b1]))
        n = nb * BLOCK; comp = int(packed.numel())
        far = (world - 1) / world
        te, td = best
        res = {"workload": f"{args.stream_gib:g} GiB stream of class {args.cls} on rank 0, 64 KiB blocks: NCCL scatter -> encode on {world} GPU(s) -> gather; and back",
               "scaling": "strong", "n_gpus": world, "ratio": round(comp / n, 4),
               "encode_gbs": round(n / te / GB, 1), "decode_gbs": round(n / td / GB, 1), "roundtrip_gbs": round(n / (te + td) / GB, 1),
               "roundtrip_exact": ok, "stream_parity": bool(same), "stream_parity_blocks": len(idx),
               # what crosses the root's NVLink ports per direction and phase, and the rate that alone would allow
               "root_link": {"encode_out_bytes": int(n * far), "encode_in_bytes": int(comp * far), "decode_out_bytes": int(comp * far), "decode_in_bytes": int(n * far),
                             "decode_in_gbs_if_only_transfer": None if world == 1 else round(n * far / td / GB, 1)},
               "limiter": "none (one GPU: no transfer)" if world == 1 else
                          "encode: the kernels (1/N of the one-GPU time) plus the transfers a send/recv kernel cannot overlap with them; decode: the root's NVLink ingress -- every decoded byte comes back through it (see 'window' for the overlapped transport)",
               "window": wres,
               # the limiter removed: the same stream landed sharded, outputs left sharded, 4 bytes per block exchanged
               "resident": {"encode_gbs": round(n / rte / GB, 1), "decode_gbs": round(n / rtd / GB, 1), "roundtrip_gbs": round(n / (rte + rtd) / GB, 1),
                            "roundtrip_exact": rok == 0.0, "exchange": "all-gather of int32 lengths only"}}
    del raw
    if win is not None:
        wl = wo = wp = wback = None
        win.close()
    torch.cuda.empty_cache()
    return res


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = {"bound": False} if args.no_numa else bind_to_gpu_numa(local)     # before any pinned allocation (first touch)
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: lz4net_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import lz4net_b200
    ctx = lz4net_b200.Context(local)
    # The headline runs the library's DEFAULTS: for device batches the decoder is picked per batch on the device from the
    # compression ratio.  TUNED_LANES (tools/sweep.py) is what a caller who knows the data could set by hand; the entropy
    # sweep reports both side by side.
    TUNED_LANES = {"E0": 32, "E50": 108, "E100": 16, "ETEXT": 104}
    if args.lanes:
        ctx.set_option("decode_lanes", args.lanes)
    if args.enc_ctas:
        ctx.set_option("encode_ctas_per_sm", args.enc_ctas)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_hbm = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"

    # ---- headline workload -------------------------------------------------------------------------------------------
    from lz4net_b200 import shard
    first_block, _ = shard.weak_range(rank, args.blocks)        # rank r owns global blocks [r*B, (r+1)*B): no exchange step
    work = Workload(ctx, args.blocks, args.cls, args.wave, seed=1, first_block=first_block)
    csum = work.verify()                                   # correctness first: full-batch round trip on the device
    raw_bytes = args.blocks * BLOCK
    nw = work.n_waves
    for _ in range(args.warmup):
        work.encode()
        for w in range(nw):
            work.decode_wave(w)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = Clocks(local); clocks.start()
    launches0 = ctx.launches
    evs = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(1 + nw)] for _ in range(args.steps)]
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    for s in range(args.steps):
        work.timed_step(evs[s])
    t_end.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clk = clocks.stop()
    launches = ctx.launches - launches0
    elapsed = t_start.elapsed_time(t_end) * 1e-3
    t_enc = sum(e[0][0].elapsed_time(e[0][1]) for e in evs) * 1e-3 / args.steps
    t_dec = sum(sum(p[0].elapsed_time(p[1]) for p in e[1:]) for e in evs) * 1e-3 / args.steps
    elapsed, t_enc, t_dec = shard.reduce_max([elapsed, t_enc, t_dec], device="cuda")     # the slowest rank defines the job
    csum_all, = shard.reduce_sum([float(csum)], device="cuda")
    total_raw = raw_bytes * world
    value = total_raw * args.steps / elapsed / GB
    enc_gbs = total_raw / t_enc / GB; dec_gbs = total_raw / t_dec / GB
    # roofline (per GPU): algorithmic bytes = raw + compressed, both directions of each kernel (SURVEY.md 8d)
    alg = (total_raw + csum_all) / world
    # DRAM traffic per launch: NOT measured in this run -- scaled per block from the committed ncu --set full capture
    # (profiles/ncu_traffic.json, class E50 only), labelled as such
    traffic_dec = traffic_enc = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        if args.cls == "E50":
            traffic_dec = int(tj["lz4_decode_kernel"]["dram_bytes"] / tj["blocks"] * min(args.wave, args.blocks))
            traffic_enc = int(tj["lz4_encode_fast_kernel"]["dram_bytes"] / tj["blocks"] * args.blocks)
    except Exception:
        pass
    tsrc = "static: profiles/ncu_traffic.json (ncu --set full, bytes per block x blocks per launch), not measured in this run"
    roof_dec = {"kernel": "lz4_decode_lpb_kernel (whole waves of the batch) + lz4_decode_kernel<8> (the rest), as picked on the device", "bound": "hbm", "achieved": round(alg / t_dec / GB, 1), "peak": peak_hbm, "unit": "GB/s",
                "frac": round(alg / t_dec / GB / peak_hbm, 4), "traffic": traffic_dec, "traffic_source": tsrc, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": int(alg / nw), "launch_ms": round(t_dec / nw * 1e3, 3)}
    roof_enc = {"kernel": "lz4_encode_fast_kernel", "bound": "hbm", "achieved": round(alg / t_enc / GB, 1), "peak": peak_hbm, "unit": "GB/s",
                "frac": round(alg / t_enc / GB / peak_hbm, 4), "traffic": traffic_enc, "traffic_source": tsrc, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": int(alg), "launch_ms": round(t_enc * 1e3, 3)}
    if args.dump_outputs and rank == 0:
        dump_outputs(work, args.dump_outputs)
    del work
    torch.cuda.empty_cache()

    # ---- end to end through the C ABI with host buffers (every rank, concurrently) -----------------------------------
    e2e = None
    if not args.no_e2e:
        nb_e = min(args.e2e_blocks, args.blocks); st_e = max(2, args.steps // 4)
        if world > 1:
            dist.barrier()
        r = e2e_sequential(local, args.cls, nb_e, st_e, 1, "pinned")
        if world > 1:
            dist.barrier()
        pl = e2e_pipelined(local, args.cls, nb_e, st_e, 1)
        if world > 1:
            dist.barrier()
        pg = e2e_sequential(local, args.cls, min(nb_e, 4096), 2, 1, "pageable")
        if world > 1:
            dist.barrier()
        rg = e2e_sequential(local, args.cls, min(nb_e, 4096), 2, 1, "registered")
        te, td, tp, tpg, trg = shard.reduce_max([r["t_enc"], r["t_dec"], pl["t_step"], pg["t_enc"] + pg["t_dec"], rg["t_enc"] + rg["t_dec"]], device="cuda")
        seq = r["bytes"] * world / (te + td) / GB; pip = r["bytes"] * world / tp / GB
        mine_e2e = {"rank": rank, "numa_node": numa.get("numa_node"), "bound": numa.get("bound"),
                    "sequential_gbs": round(r["bytes"] / (r["t_enc"] + r["t_dec"]) / GB, 2), "pipelined_gbs": round(r["bytes"] / pl["t_step"] / GB, 2)}
        per_rank = [None] * world
        if world > 1:
            dist.all_gather_object(per_rank, mine_e2e)
        else:
            per_rank = [mine_e2e]
        e2e = {"value": round(max(seq, pip), 3), "unit": "GB/s", "h2d_bytes_per_step": int(r["h2d"]), "d2h_bytes_per_step": int(r["d2h"]),
               "sequential_gbs": round(seq, 3), "pipelined_gbs": round(pip, 3),
               "encode_gbs": round(r["bytes"] * world / te / GB, 3), "decode_gbs": round(r["bytes"] * world / td / GB, 3),
               "pageable_gbs": round(pg["bytes"] * world / tpg / GB, 3), "registered_gbs": round(rg["bytes"] * world / trg / GB, 3),
               "numa": numa, "per_rank": per_rank,
               "sample": f"{nb_e} x 64 KiB blocks per GPU through lz4b200_encode_batch_packed + lz4b200_decode_batch (MEM_HOST), wall clock, every copy inside the calls. "
                         "value = the better of: sequential (one caller thread: encode, then decode) and pipelined (two caller threads, a context each: the encode of step i+1 "
                         "overlaps the decode of step i, both PCIe directions busy). pinned host memory; pageable_gbs / registered_gbs: the sequential form from plain "
                         "malloc'ed memory (what a managed caller's fixed byte[] is) and from the same memory page-locked once with lz4b200_host_register (4096 blocks)"}

    # ---- entropy sweep (BASELINE configs[4]) on every rank: library defaults and hand-tuned decode lanes side by side ----
    extras = {}
    if not args.no_sweep:
        sweep = {}
        for cls in ("E0", "E50", "E100", "ETEXT"):
            w = Workload(ctx, min(args.sweep_blocks, args.blocks), cls, args.wave, seed=2, first_block=rank * min(args.sweep_blocks, args.blocks))
            ctx.set_option("decode_lanes_auto", 1)
            cs = w.verify()
            te, td = measure_pair(w, 3, 2)
            ctx.set_option("decode_lanes", TUNED_LANES[cls])
            _, td_t = measure_pair(w, 3, 1)
            ctx.set_option("decode_lanes_auto", 1)
            te, td, td_t = shard.reduce_max([te, td, td_t], device="cuda")
            cs_all, = shard.reduce_sum([float(cs)], device="cuda")
            rb = w.n * BLOCK * world
            sweep[cls] = {"ratio": round(cs_all / rb, 4), "encode_gbs": round(rb / te / GB, 1), "decode_gbs": round(rb / td / GB, 1),
                          "decode_roofline_frac": round((rb + cs_all) / td / GB / peak_hbm / world, 4),
                          "encode_roofline_frac": round((rb + cs_all) / te / GB / peak_hbm / world, 4), "blocks_per_gpu": w.n,
                          "decode_tuned_gbs": round(rb / td_t / GB, 1), "decode_tuned_lanes": TUNED_LANES[cls],
                          "decode_tuned_roofline_frac": round((rb + cs_all) / td_t / GB / peak_hbm / world, 4)}
            del w; torch.cuda.empty_cache()
        if args.lanes:
            ctx.set_option("decode_lanes", args.lanes)
        extras["entropy_sweep"] = sweep
        extras["entropy_sweep_note"] = f"aggregate over {world} GPU(s), device-timed, max over ranks; decode_gbs = library default (decoder picked on the device per batch), decode_tuned_gbs = decode_lanes set by hand"

    # ---- BASELINE configs[3]: one stream, N GPUs, NCCL scatter / gather ------------------------------------------------
    if not args.no_stream:
        st = stream_section(ctx, args, rank, world, dev)
        if st is not None:
            extras["stream"] = st

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rank 0, N=1 extras: HC (config 3), CPU baseline ---------------------------------------------------------------
    if world == 1 and not args.no_hc:
        hc = {}
        for cls in ("E50", "ETEXT"):
            # (ETEXT gains nothing from more than 65 536 blocks in flight: half the batch keeps the default run short)
            w = Workload(ctx, min(args.hc_blocks if cls == "E50" else args.hc_blocks // 2, args.blocks), cls, args.wave, seed=3)
            # the library's default HC kernel first (its output is what the round trip below checks), then the others
            # (hc_kernel 0: a thread per block; 1 / 2: a warp per block on a static index, block in shared memory / through L1)
            default_kernel = ctx.get_option("hc_kernel")
            te, _ = measure_pair(w, 1, 1, hc=True)
            torch.cuda.synchronize()
            cs = int(w.clen.sum()); rb = w.n * BLOCK
            for wv in range(w.n_waves):
                b0, b1 = w.decode_wave(wv); torch.cuda.synchronize()
                assert torch.equal(w.out[: (b1 - b0) * BLOCK], w.raw[b0 * BLOCK: b1 * BLOCK]), "HC round trip failed"
            hc[cls] = {"ratio": round(cs / rb, 4), "encode_gbs": round(rb / te / GB, 2), "blocks": w.n, "hc_kernel": default_kernel,
                       "roofline_frac": round((rb + cs) / te / GB / peak_hbm, 5), "kernels": {}}
            lens_default = w.clen.clone()
            for k in (0, 1, 2):
                if k == default_kernel:
                    hc[cls]["kernels"][str(k)] = hc[cls]["encode_gbs"]; continue
                ctx.set_option("hc_kernel", k)
                try:
                    tk, _ = measure_pair(w, 1, 1, hc=True)
                    torch.cuda.synchronize()
                    assert torch.equal(w.clen, lens_default), "HC kernels disagree on the compressed lengths"
                    hc[cls]["kernels"][str(k)] = round(rb / tk / GB, 2)
                finally:
                    ctx.set_option("hc_kernel", default_kernel)
            if not args.no_cpu:
                hc[cls]["cpu_reference_gbs"] = round(cpu_hc(cls, 1024 if cls == "ETEXT" else 4096, os.cpu_count() or 1), 3)
            del w; torch.cuda.empty_cache()
        # natural text (not a BASELINE class; blocks cut from this repository's own documents and sources, tiled): what LZ4HC
        # is used on in practice -- hash buckets of 20 - 60 positions, between E50's 4 and ETEXT's 240
        try:
            nb = min(16384, args.blocks)
            data = b""
            for name in ("SURVEY.md", "DESIGN.md", "BASELINE.md", "INTEGRATION.md", "README.md", "bench.py", "lz4net_b200/csrc/capi.cu"):
                fp = os.path.join(os.path.dirname(os.path.abspath(__file__)), name)
                if os.path.exists(fp):
                    data += open(fp, "rb").read()
            k = len(data) // BLOCK
            if k >= 1:
                w = Workload(ctx, nb, "E0", nb, seed=3)
                t = torch.frombuffer(bytearray(data[: k * BLOCK]), dtype=torch.uint8).cuda().view(k, BLOCK)
                w.raw = t.repeat((nb + k - 1) // k, 1)[:nb].contiguous().view(-1)
                te, _ = measure_pair(w, 1, 1, hc=True)
                torch.cuda.synchronize()
                cs = int(w.clen.sum()); rb = w.n * BLOCK
                row = {"ratio": round(cs / rb, 4), "encode_gbs": round(rb / te / GB, 2), "blocks": w.n, "distinct_blocks": k,
                       "hc_kernel": ctx.get_option("hc_kernel"), "kernels": {}}
                ctx.set_option("hc_kernel", 0)
                try:
                    tk, _ = measure_pair(w, 1, 1, hc=True)
                    torch.cuda.synchronize()
                    row["kernels"]["0"] = round(rb / tk / GB, 2)
                finally:
                    ctx.set_option("hc_kernel", row["hc_kernel"])
                hc["TEXT"] = row
                del w; torch.cuda.empty_cache()
        except Exception as e:                      # an extra, never the reason the bench line is lost
            hc["TEXT"] = {"error": repr(e)[:200]}
        extras["hc"] = hc
    cpu = None
    if world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        n = min(args.cpu_blocks, args.blocks)
        r = cpu_codec(args.cls, n, threads, repeats=3)
        r1 = cpu_codec(args.cls, min(n, 2048), 1, repeats=2)
        cpu = {"value": round(r["roundtrip_gbs"], 3), "unit": "GB/s", "cores": threads, "kind": r["kind"],
               "sample": f"{n} x 64 KiB blocks of class {args.cls} ({n * BLOCK / 2**20:.0f} MiB raw), encode then decode, best of 3, static partition",
               "encode_gbs": round(r["encode_gbs"], 3), "decode_gbs": round(r["decode_gbs"], 3),
               "single_thread": {"encode_gbs": round(r1["encode_gbs"], 3), "decode_gbs": round(r1["decode_gbs"], 3)}}

    line = {
        "metric": "GB/s encode+decode on batched 64KiB blocks", "value": round(value, 3), "unit": "GB/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(elapsed / args.steps * 1e3, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": f"{args.blocks} x 64KiB independent blocks per GPU, class {args.cls} (BASELINE configs[1]): one fast-encode launch + {nw} known-size decode launches per step",
                   "block_size": BLOCK, "class": args.cls, "blocks_per_gpu": args.blocks, "ratio": round(csum_all / total_raw, 4),
                   "decode_lanes": args.lanes or "library default: picked per batch on the device from the compression ratio",
                   "decode_wave_blocks": work_wave(args), "l2": "inputs (64 GiB raw + slots per GPU) are far larger than the 126 MB L2; no flush needed",
                   "parallelism": f"independent blocks sharded over {world} GPU(s), no data-path collective", "gb": "1e9 bytes"},
        "encode_gbs": round(enc_gbs, 2), "decode_gbs": round(dec_gbs, 2),
        "roofline": roof_enc, "roofline_decode": roof_dec,
        "clocks": clk, "gpu_launches": int(launches),
        "e2e": e2e, "cpu_baseline": cpu,
    }
    line.update(extras)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def work_wave(args):
    return min(args.wave, args.blocks)


if __name__ == "__main__":
    main()
