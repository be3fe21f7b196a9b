"""LZ4Stream framing on device memory against the host framing, on a stream far larger than L2.

    python tools/stream_device.py [--gib 4] [--warmup 3] [--reps 10] [--out FILE]

For each class (E50, ETEXT, E0; fast encoder) and block size (64 KiB, 1 MiB), on one stream synthesised on the device:
  encode_device        host clock around lz4b200_stream_encode_device (synchronous), GB/s of raw bytes
  encode_batch         the encode batch alone on the same chunks (one device batch, CUDA events): the framing's overhead
                       is the difference
  decoded_size_device  the serial header walk: total and per chunk
  decode_device        host clock around lz4b200_stream_decode_device; decode_batch = the compressed chunks' batch alone
  host_encode          D2H of the raw bytes into pinned memory + lz4b200_stream_encode from there (what a GPU producer
                       does without the device framing); host_decode the mirror image (stream_decode from pinned
                       memory + H2D of the result)
The device wire is compared with the host wire byte for byte, and the device decode with the input, in the same run.
Medians of --reps runs after --warmup runs.  Prints one JSON line (and writes it to --out when given).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import lz4net_b200
from lz4net_b200 import batch, native, synth

SYNTH_BLOCK = 65536


def card():
    """Name and power limit, read-only query (no setting is changed)."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def event_timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    return statistics.median(ts)


def chunk_table(wire):
    """(payload offset, compressed length, output offset, raw length) of every compressed chunk; number of chunks."""
    out, p, o, k = [], 0, 0, 0
    def varint():
        nonlocal p
        v = sh = 0
        while True:
            x = int(wire[p]); p += 1; v |= (x & 0x7F) << sh; sh += 7
            if not x & 0x80:
                return v
    while p < len(wire):
        f = varint(); r = varint(); c = varint() if f & 1 else r
        if f & 1:
            out.append((p, c, o, r))
        p += c; o += r; k += 1
    return out, k


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=4.0)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lib = native.lib()
    ctx = lz4net_b200.Context(torch.cuda.current_device())
    st = torch.cuda.current_stream().cuda_stream
    n = int(args.gib * (1 << 30)) // SYNTH_BLOCK * SYNTH_BLOCK
    dev = torch.device("cuda", torch.cuda.current_device())
    raw = torch.empty(n, dtype=torch.uint8, device=dev)
    cap = int(lib.lz4b200_stream_bound(n, 65536))
    wire = torch.empty(cap, dtype=torch.uint8, device=dev)
    back = torch.empty(n, dtype=torch.uint8, device=dev)
    slots = torch.empty(n, dtype=torch.uint8, device=dev)
    h_raw = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h_wire = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
    res = {"tool": "tools/stream_device.py", "card": card(), "bytes": n, "warmup": args.warmup, "reps": args.reps,
           "timing": "host clock around synchronous calls; *_batch_s: CUDA events around one device batch", "runs": []}
    for cls in ("E50", "ETEXT", "E0"):
        batch.synth_fill(ctx, raw, n // SYNTH_BLOCK, SYNTH_BLOCK, synth.CLASS_ID[cls], seed=7)
        torch.cuda.synchronize()
        for bs in (65536, 1 << 20):
            r = {"class": cls, "block_size": bs, "chunks": (n + bs - 1) // bs}
            w = [0]
            def enc_dev():
                w[0] = int(lib.lz4b200_stream_encode_device(ctx.handle, raw.data_ptr(), n, bs, 0, wire.data_ptr(), cap, st))
                assert w[0] > 0, (w[0], native.last_error())
            t = timed(enc_dev, args.warmup, args.reps)
            W = w[0]
            r.update(wire_bytes=W, encode_device_s=t, encode_device_gbs=n / t / 1e9)
            # the encode batch alone: the same chunks, one slot per chunk with capacity == its length
            m = r["chunks"]
            so = torch.arange(m, dtype=torch.int64, device=dev) * bs
            sl = torch.clamp(n - so, max=bs).to(torch.int32)
            out = torch.zeros(m, dtype=torch.int32, device=dev)
            t = event_timed(lambda: ctx.encode_batch_ptr(raw.data_ptr(), so.data_ptr(), sl.data_ptr(), slots.data_ptr(), so.data_ptr(),
                                                         sl.data_ptr(), out.data_ptr(), m, hc=False, device=True, stream=st),
                            args.warmup, args.reps)
            r.update(encode_batch_s=t, encode_batch_gbs=n / t / 1e9)
            # the serial walk
            def size():
                assert int(lib.lz4b200_stream_decoded_size_device(ctx.handle, wire.data_ptr(), W, st)) == n
            t = timed(size, args.warmup, args.reps)
            r.update(decoded_size_device_s=t, walk_us_per_chunk=t / m * 1e6)
            def dec_dev():
                assert int(lib.lz4b200_stream_decode_device(ctx.handle, wire.data_ptr(), W, back.data_ptr(), n, st)) == n
            t = timed(dec_dev, args.warmup, args.reps)
            r.update(decode_device_s=t, decode_device_gbs=n / t / 1e9)
            r["roundtrip_exact"] = bool(torch.equal(back, raw))
            # the decode batch alone, on the compressed chunks of the same wire
            h_wire[:W].copy_(wire[:W]); torch.cuda.synchronize()
            tab, k = chunk_table(h_wire[:W].numpy())
            assert k == m
            r["compressed_chunks"] = len(tab)
            if tab:
                tt = torch.tensor(tab, dtype=torch.int64).to(dev)
                d_so, d_sl, d_do, d_dc = tt[:, 0].contiguous(), tt[:, 1].to(torch.int32), tt[:, 2].contiguous(), tt[:, 3].to(torch.int32)
                d_out = torch.zeros(len(tab), dtype=torch.int32, device=dev)
                t = event_timed(lambda: ctx.decode_batch_ptr(wire.data_ptr(), d_so.data_ptr(), d_sl.data_ptr(), back.data_ptr(), d_do.data_ptr(),
                                                             d_dc.data_ptr(), d_out.data_ptr(), len(tab), known=True, device=True, stream=st),
                                args.warmup, args.reps)
                r.update(decode_batch_s=t, decode_batch_gbs=n / t / 1e9)
            # host framing from pinned memory, with the PCIe transfer a device-resident producer / consumer pays
            hw = [0]
            def enc_host():
                h_raw.copy_(raw); torch.cuda.synchronize()
                hw[0] = int(lib.lz4b200_stream_encode(ctx.handle, h_raw.data_ptr(), n, bs, 0, h_wire.data_ptr(), cap))
                assert hw[0] > 0
            t = timed(enc_host, args.warmup, args.reps)
            r.update(host_encode_s=t, host_encode_gbs=n / t / 1e9)
            r["wire_identical_to_host"] = hw[0] == W and bool(torch.equal(wire[:W], h_wire[:W].to(dev)))
            def dec_host():
                assert int(lib.lz4b200_stream_decode(ctx.handle, h_wire.data_ptr(), W, h_raw.data_ptr(), n)) == n
                back.copy_(h_raw); torch.cuda.synchronize()
            t = timed(dec_host, args.warmup, args.reps)
            r.update(host_decode_s=t, host_decode_gbs=n / t / 1e9)
            r = {k: (round(v, 6) if isinstance(v, float) else v) for k, v in r.items()}
            res["runs"].append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
