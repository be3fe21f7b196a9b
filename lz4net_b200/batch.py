"""Device-memory batches: torch owns the HBM buffers, the work is done by liblz4b200.so on raw pointers.

A batch is the GPU-native unit of work of this codec (the reference handles one block per call; LZ4Stream dispatches
one block at a time, src/LZ4/LZ4Stream.cs:239-269).  Layouts:

* raw blocks      uint8[n_blocks * block_size], block i at i * block_size
* encoder slots   uint8[n_blocks * slot], slot = MaximumOutputLength(block_size) (or block_size for LZ4Stream/Wrap caps)
* packed payload  uint8[sum(len)], block i at off[i] (exclusive prefix sum, int64[n_blocks + 1])
"""
from __future__ import annotations

import torch

from . import native
from .codec import Context


def _p(t: torch.Tensor) -> int:
    return t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def uniform_layout(n_blocks: int, block_size: int, slot: int, device):
    idx = torch.arange(n_blocks, dtype=torch.int64, device=device)
    return idx * block_size, idx * slot, torch.full((n_blocks,), block_size, dtype=torch.int32, device=device), \
        torch.full((n_blocks,), slot, dtype=torch.int32, device=device)


def synth_fill(ctx: Context, dst: torch.Tensor, n_blocks: int, block_size: int, cls: int, seed: int = 1, first_block: int = 0):
    native.check(native.lib().lz4b200_synth_fill(ctx.handle, _p(dst), n_blocks, block_size, cls, seed, first_block, _stream()),
                 "synth_fill")


def encode(ctx: Context, raw: torch.Tensor, src_off, src_len, slots: torch.Tensor, dst_off, dst_cap, out_len, hc: bool = False):
    """Asynchronous on the current torch stream."""
    ctx.encode_batch_ptr(_p(raw), _p(src_off), _p(src_len), _p(slots), _p(dst_off), _p(dst_cap), _p(out_len),
                         src_off.numel(), hc=hc, device=True, stream=_stream())


def decode(ctx: Context, comp: torch.Tensor, src_off, src_len, out: torch.Tensor, dst_off, dst_cap, out_len, known: bool = True):
    ctx.decode_batch_ptr(_p(comp), _p(src_off), _p(src_len), _p(out), _p(dst_off), _p(dst_cap), _p(out_len),
                         src_off.numel(), known=known, device=True, stream=_stream())


def compact(ctx: Context, slots: torch.Tensor, slot_off, lens, packed, out_off):
    """out_off: int64[n+1]; packed may be None to compute only the offsets."""
    native.check(native.lib().lz4b200_compact(ctx.handle, _p(slots), _p(slot_off), _p(lens),
                                              _p(packed) if packed is not None else 0, _p(out_off), lens.numel(), _stream()),
                 "compact")


# ---- LZ4Stream framing on device memory --------------------------------------------------------------------------
def _check_bytes(ctx: Context, t, what: str) -> int:
    if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8:
        raise TypeError(f"{what} must be a torch.uint8 tensor")
    if t.device.type != "cuda" or t.device.index != ctx.device:
        raise ValueError(f"{what} must be on cuda:{ctx.device}, the context's device (got {t.device})")
    if t.dim() != 1 or not t.is_contiguous():
        raise ValueError(f"{what} must be a 1-D contiguous tensor")
    return t.numel()


def stream_encode(ctx: Context, raw: torch.Tensor, block_size: int = 1 << 20, high_compression: bool = False) -> torch.Tensor:
    """The LZ4Stream bytes of `raw` (what Context.stream_encode returns for the same bytes), built in device memory on the
    current torch stream.  Returns a tensor of exactly the stream's length."""
    n = _check_bytes(ctx, raw, "raw")
    l = native.lib()
    cap = int(l.lz4b200_stream_bound(n, block_size))
    if cap < 0:
        raise ValueError(f"block_size must be >= 1 (got {block_size})")
    out = torch.empty(cap, dtype=torch.uint8, device=raw.device)
    w = int(l.lz4b200_stream_encode_device(ctx.handle, _p(raw), n, block_size, int(high_compression), _p(out), cap,
                                           torch.cuda.current_stream(raw.device).cuda_stream))
    if w < 0:
        raise native.Lz4B200Error(f"stream_encode failed ({w}): {native.last_error()}")
    return out[:w]


def stream_decode(ctx: Context, wire: torch.Tensor) -> torch.Tensor:
    """Decode an LZ4Stream held in device memory, on the current torch stream.  Errors as Context.stream_decode:
    a malformed chunk header raises EOFError, a chunk that does not decode ValueError."""
    n = _check_bytes(ctx, wire, "wire")
    l = native.lib()
    st = torch.cuda.current_stream(wire.device).cuda_stream
    total = int(l.lz4b200_stream_decoded_size_device(ctx.handle, _p(wire), n, st))
    if total == native.E_FORMAT:
        raise EOFError("LZ4Stream: unexpected end of stream / corrupt chunk header")     # EndOfStreamException
    if total < 0:
        raise native.Lz4B200Error(f"stream_decoded_size failed ({total}): {native.last_error()}")
    out = torch.empty(total, dtype=torch.uint8, device=wire.device)
    r = int(l.lz4b200_stream_decode_device(ctx.handle, _p(wire), n, _p(out), total, st))
    if r == native.E_FORMAT:
        raise ValueError("LZ4 block has been corrupted")
    if r < 0:
        raise native.Lz4B200Error(f"stream_decode failed ({r}): {native.last_error()}")
    return out
