"""CPU-only checks of the device-memory LZ4Stream calls (lz4b200_stream_*_device): they refuse to run without a context
or a device -- there is no host fallback -- and the chunk-header step they share with the host framing
(lz4net_b200/csrc/lz4_stream.cuh) never reads a byte behind the end of its input."""
import ctypes as C
import mmap

import numpy as np
import pytest

import oracle
from tests import cases


@pytest.fixture(scope="module")
def lib():
    from lz4net_b200 import build, native
    build.build()
    return native.lib()


def _varint(v):
    out = bytearray()
    while True:
        b = v & 0x7F; v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _wire(data, bs, hc):
    """LZ4Stream bytes made with the oracle (src/LZ4/LZ4Stream.cs:239-269)."""
    out = bytearray()
    for o in range(0, len(data), bs):
        blk = data[o:o + bs]
        r, c = (oracle.encode_hc if hc else oracle.encode)(blk, cap=len(blk))
        comp = 0 < r < len(blk)
        out += _varint((1 if comp else 0) | (2 if hc else 0)) + _varint(len(blk))
        out += _varint(r) + c[:r] if comp else blk
    return bytes(out)


def _py_decoded_size(b):
    """The reader's header walk (LZ4Stream.cs:274-312), restated: total raw size, or None when malformed."""
    p = total = 0
    def varint():
        nonlocal p
        v = sh = 0
        while True:
            if p >= len(b):
                return None
            x = b[p]; p += 1; v += (x & 0x7F) << sh; sh += 7
            if not x & 0x80 or sh >= 64:
                return v
    while p < len(b):
        f = varint(); r = varint() if f is not None else None
        if r is None:
            return None
        c = varint() if f & 1 else r
        if c is None:
            return None
        ri = (r & 0xFFFFFFFF) - ((r & 0x80000000) << 1); ci = (c & 0xFFFFFFFF) - ((c & 0x80000000) << 1)
        if ri < 0 or ci < 0 or ci > ri or p + ci > len(b) or (f & 1 and f >> 2):
            return None
        p += ci; total += ri
    return total


def test_device_entry_points_refuse_without_context_or_device(lib):
    from lz4net_b200 import native
    src = np.frombuffer(bytes([0, 5]) + b"hello" + b"\0" * 16, np.uint8)
    dst = np.zeros(64, np.uint8)
    p, q = src.ctypes.data, dst.ctypes.data
    # a null context is an argument error, even where the host call would succeed on the same bytes
    assert lib.lz4b200_stream_decoded_size(p, 7) == 5
    assert lib.lz4b200_stream_decoded_size_device(None, p, 7, None) == native.E_ARG
    assert lib.lz4b200_stream_decode_device(None, p, 7, q, 64, None) == native.E_ARG
    assert lib.lz4b200_stream_encode_device(None, p, 7, 4, 0, q, 64, None) == native.E_ARG
    # negative sizes
    for n in (-1, -(1 << 40)):
        assert lib.lz4b200_stream_decoded_size_device(None, p, n, None) == native.E_ARG
        assert lib.lz4b200_stream_decode_device(None, p, n, q, 64, None) == native.E_ARG
        assert lib.lz4b200_stream_encode_device(None, p, n, 4, 0, q, 64, None) == native.E_ARG
    import torch
    if not torch.cuda.is_available():
        # without a device there is no context to pass: creation fails, so nothing can run on the host instead
        h = C.c_void_p()
        assert lib.lz4b200_create(C.byref(h), 0) == native.E_NODEVICE
        assert not h.value


def test_header_walk_never_reads_past_the_input(lib):
    """Every prefix of a real stream ends on the last readable byte of a page; the next page is PROT_NONE, so a read of
    even one byte behind the input would kill the process.  The verdict matches the walk restated in Python."""
    data = b"".join(cases.content(m, n, seed=5).tobytes() for m, n in (("ETEXT", 1500), ("E0", 700), ("mixed", 900)))
    wires = [_wire(data, 256, False), _wire(data, 1000, True),
             _varint(0) + _varint(0) + _varint(0) + _varint(3) + b"abc" + _varint(2) + _varint(200) + bytes(200) +  # zero-length, stored (HC flag)
             _varint(1) + _varint(1 << 31) + _varint(4) + b"wxyz"]                                                # rawLen >= 2^31
    page = mmap.PAGESIZE
    npages = (max(len(w) for w in wires) + page - 1) // page + 1
    m = mmap.mmap(-1, (npages + 1) * page)
    base = C.addressof(C.c_char.from_buffer(m))
    libc = C.CDLL(None, use_errno=True)
    libc.mprotect.argtypes = [C.c_void_p, C.c_size_t, C.c_int]
    end = npages * page
    assert libc.mprotect(base + end, page, 0) == 0
    try:
        for w in wires:
            for L in range(len(w) + 1):
                m[end - L:end] = w[:L]
                got = lib.lz4b200_stream_decoded_size(base + end - L, L)
                want = _py_decoded_size(w[:L])
                assert got == (-5 if want is None else want), (L, got, want)
    finally:
        assert libc.mprotect(base + end, page, 3) == 0
    assert _py_decoded_size(wires[0]) == len(data)
