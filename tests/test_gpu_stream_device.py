"""LZ4Stream framing on device memory (lz4b200_stream_*_device, lz4net_b200.batch.stream_encode / stream_decode) on the
B200: the wire is byte-identical to the host framing (framing.cpp) and to the reference format built from the oracle,
and every decode verdict -- malformed inputs included -- is the host's."""
import functools

import numpy as np
import pytest

import oracle
from tests import cases

pytestmark = pytest.mark.gpu

E_ARG, E_FORMAT = -1, -5
BLOCK_SIZES = (65536, 1 << 20, 1000, 16, 65547, 70001)


@pytest.fixture(scope="module")
def ctx():
    import lz4net_b200
    return lz4net_b200.default_context()


@pytest.fixture(scope="module")
def lib():
    from lz4net_b200 import native
    return native.lib()


@pytest.fixture(params=[-1, 0, 1, 2], ids=["hc-auto", "hc-thread", "hc-warp-smem", "hc-warp-l1"])
def hck(ctx, request):
    """Every LZ4HC kernel of the library, set for the test and restored after it."""
    prev = ctx.get_option("hc_kernel")
    ctx.set_option("hc_kernel", request.param)
    yield request.param
    ctx.set_option("hc_kernel", prev)


def _varint(v):
    out = bytearray()
    while True:
        b = v & 0x7F; v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _ref_stream(data, block_size, hc):
    """The LZ4Stream wire bytes, built from the oracle (src/LZ4/LZ4Stream.cs:225-269)."""
    out = bytearray()
    for o in range(0, len(data), block_size):
        blk = data[o:o + block_size]
        r, c = (oracle.encode_hc if hc else oracle.encode)(blk, cap=len(blk))
        comp = 0 < r < len(blk)
        out += _varint((1 if comp else 0) | (2 if hc else 0)) + _varint(len(blk))
        if comp:
            out += _varint(r)
        out += c if comp else blk
    return bytes(out)


@functools.lru_cache(maxsize=None)
def _mixed():
    """Compressible text, incompressible (stored E0) chunks and a short last chunk, as in the host wire-format test."""
    return b"".join(cases.content(m, n, seed=9).tobytes() for m, n in
                    (("ETEXT", 200000), ("E0", 70000), ("E100", 130000), ("mixed", 65536), ("lowent", 12345)))


@functools.lru_cache(maxsize=None)
def _case(bs, hc):
    d = _mixed() if bs >= 1000 else _mixed()[:3000]
    return d, _ref_stream(d, bs, hc)


def _dev(b):
    import torch
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda() if len(b) else torch.empty(0, dtype=torch.uint8, device="cuda")


def _stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _check_encode_parity(ctx, hc):
    from lz4net_b200 import batch
    for bs in BLOCK_SIZES:
        d, ref = _case(bs, hc)
        wire = batch.stream_encode(ctx, _dev(d), bs, hc)
        assert wire.numel() == len(ref), bs
        got = wire.cpu().numpy().tobytes()
        assert got == ref, bs
        assert got == ctx.stream_encode(d, bs, hc), bs
        assert batch.stream_decode(ctx, wire).cpu().numpy().tobytes() == d, bs               # device-made wire
        assert batch.stream_decode(ctx, _dev(ref)).cpu().numpy().tobytes() == d, bs          # host/reference-made wire
    assert batch.stream_encode(ctx, _dev(b""), 65536, hc).numel() == 0
    assert batch.stream_decode(ctx, _dev(b"")).numel() == 0


def test_encode_fast_matches_host_and_reference(ctx):
    _check_encode_parity(ctx, False)


def test_encode_hc_matches_host_and_reference(ctx, hck):
    _check_encode_parity(ctx, True)


def test_decode_hand_built_streams(ctx):
    from lz4net_b200 import batch
    blk = cases.content("ETEXT", 5000, seed=3).tobytes()
    r, c = oracle.encode(blk, cap=len(blk))
    assert 0 < r < len(blk)
    wire = (_varint(0) + _varint(0) +                                   # zero-length stored chunk
            _varint(1) + _varint(0) + _varint(0) +                       # zero-length compressed chunk
            _varint(2) + _varint(7) + b"stored!" +                       # stored chunk carrying the HC flag
            _varint(3) + _varint(len(blk)) + _varint(r) + c +            # compressed, HC flag
            _varint(0) + _varint(0))
    want = b"stored!" + blk
    assert ctx.stream_decode(wire) == want
    assert batch.stream_decode(ctx, _dev(wire)).cpu().numpy().tobytes() == want
    # a Flush ends the current chunk: a stream is the concatenation of independently framed segments
    d = _mixed()
    cuts = [0, 1, 4097, 70000, 70001, 200000, 333333, len(d)]
    for hc in (False, True):
        wire = b"".join(_ref_stream(d[a:b], 4096, hc) for a, b in zip(cuts, cuts[1:]))
        assert batch.stream_decode(ctx, _dev(wire)).cpu().numpy().tobytes() == d


def _same_verdicts(ctx, lib, wire, prefixes, mutations, seed):
    """decoded_size_device / decode_device against the host calls on the same bytes, input by input."""
    import torch
    cap = 1 << 20
    hdst = np.zeros(cap + 16, np.uint8)
    ddst = torch.zeros(cap + 16, dtype=torch.uint8, device="cuda")
    st = _stream_ptr()

    def check(hsrc, dsrc, n):
        hs = lib.lz4b200_stream_decoded_size(hsrc.ctypes.data, n)
        ds = lib.lz4b200_stream_decoded_size_device(ctx.handle, dsrc.data_ptr(), n, st)
        assert ds == hs, (n, ds, hs)
        dc = max(hs, 0)
        if dc > cap:
            return
        hr = lib.lz4b200_stream_decode(ctx.handle, hsrc.ctypes.data, n, hdst.ctypes.data, dc)
        dr = lib.lz4b200_stream_decode_device(ctx.handle, dsrc.data_ptr(), n, ddst.data_ptr(), dc, st)
        assert dr == hr, (n, dr, hr)
        if hr > 0:
            assert np.array_equal(ddst[:hr].cpu().numpy(), hdst[:hr]), n

    hsrc = np.frombuffer(wire + b"\0" * 16, np.uint8)
    dsrc = _dev(wire)
    for n in prefixes:
        check(hsrc, dsrc, n)
    if not mutations:
        return
    rng = np.random.default_rng(seed)
    heads, p = [], 0                                       # chunk header positions: headers are hit as often as payloads
    while p < len(wire):
        heads.append(p)
        p = _skip_chunk(wire, p)
    for k in range(mutations):
        b = bytearray(wire)
        pos = heads[int(rng.integers(0, len(heads)))] + int(rng.integers(0, 4)) if k % 2 == 0 else int(rng.integers(0, len(wire)))
        pos = min(pos, len(wire) - 1)
        b[pos] = int(rng.integers(0, 256)) if k % 3 else b[pos] ^ (1 << int(rng.integers(0, 8)))
        mb = bytes(b)
        check(np.frombuffer(mb + b"\0" * 16, np.uint8), _dev(mb), len(mb))


def _skip_chunk(w, p):
    def varint(p):
        v = sh = 0
        while True:
            x = w[p]; p += 1; v |= (x & 0x7F) << sh; sh += 7
            if not x & 0x80:
                return v, p
    f, p = varint(p); r, p = varint(p)
    c, p = varint(p) if f & 1 else (r, p)
    return p + c


@pytest.mark.parametrize("hc", [False, True])
def test_decode_verdicts_match_host(ctx, lib, hc):
    data = b"".join(cases.content(m, n, seed=21).tobytes() for m, n in (("ETEXT", 9000), ("E0", 5000), ("mixed", 6000)))
    wire = _ref_stream(data, 4096, hc)
    _same_verdicts(ctx, lib, wire, range(len(wire) + 1), 400, seed=7 + hc)


def test_decode_explicit_malformed_cases(ctx, lib):
    cases_ = [
        (b"", 0),
        (bytes([0, 5]) + b"hello", 5),                                  # stored chunk
        (bytes([0, 5]) + b"hell", E_FORMAT),                            # truncated payload
        (bytes([1, 5, 6]) + b"xxxxxx", E_FORMAT),                       # compLen > rawLen
        (bytes([0x80]), E_FORMAT),                                      # truncated varint
        (bytes([5, 100, 3]) + b"abc", E_FORMAT),                        # passes != 0
        (bytes([4, 3]) + b"abc", 3),                                    # passes bits on a stored chunk are ignored
        (_varint(0) + _varint(1 << 31) + b"x", E_FORMAT),               # rawLen >= 2^31: negative after the (int) cast
        (_varint(0) + _varint((1 << 32) + 3) + b"abc", 3),              # the cast keeps the low 32 bits
        (bytes([0, 0, 0, 0]), 0),                                       # zero-length chunks
    ]
    st = _stream_ptr()
    for b, want in cases_:
        h = np.frombuffer(b + b"\0", np.uint8)
        assert lib.lz4b200_stream_decoded_size(h.ctypes.data, len(b)) == want, b
        d = _dev(b)
        assert lib.lz4b200_stream_decoded_size_device(ctx.handle, d.data_ptr(), len(b), st) == want, b
    for b, _ in cases_:
        _same_verdicts(ctx, lib, b, [len(b)], 0, seed=1)


def test_capacity_and_guards(ctx, lib):
    import torch
    st = _stream_ptr()
    d, ref = _case(65536, False)
    n = len(d)
    bound = lib.lz4b200_stream_bound(n, 65536)
    src = _dev(d)
    dst = torch.full((bound + 64,), 0xEE, dtype=torch.uint8, device="cuda")
    assert lib.lz4b200_stream_encode_device(ctx.handle, src.data_ptr(), n, 65536, 0, dst.data_ptr(), bound - 1, st) == E_ARG
    assert bool((dst == 0xEE).all())
    w = lib.lz4b200_stream_encode_device(ctx.handle, src.data_ptr(), n, 65536, 0, dst.data_ptr(), bound, st)
    assert w == len(ref) and dst[:w].cpu().numpy().tobytes() == ref
    assert bool((dst[w:] == 0xEE).all())                                   # nothing behind the returned length
    wire = _dev(ref)
    out = torch.full((n + 64,), 0xEE, dtype=torch.uint8, device="cuda")
    assert lib.lz4b200_stream_decode_device(ctx.handle, wire.data_ptr(), len(ref), out.data_ptr(), n - 1, st) == E_ARG
    assert bool((out == 0xEE).all())
    assert lib.lz4b200_stream_decode_device(ctx.handle, wire.data_ptr(), len(ref), out.data_ptr(), n, st) == n
    assert out[:n].cpu().numpy().tobytes() == d and bool((out[n:] == 0xEE).all())
    # null pointers with work to do
    assert lib.lz4b200_stream_encode_device(ctx.handle, None, n, 65536, 0, dst.data_ptr(), bound, st) == E_ARG
    assert lib.lz4b200_stream_decode_device(ctx.handle, wire.data_ptr(), len(ref), None, n, st) == E_ARG
    assert lib.lz4b200_stream_encode_device(ctx.handle, src.data_ptr(), n, 0, 0, dst.data_ptr(), bound, st) == E_ARG


@pytest.mark.parametrize("hc", [False, True])
def test_any_byte_alignment(ctx, lib, hc):
    import torch
    st = _stream_ptr()
    for bs in (65536, 1000):
        d, ref = _case(bs, hc)
        d = d[:150000] if bs >= 1000 else d
        ref = _ref_stream(d, bs, hc)
        n = len(d)
        bound = lib.lz4b200_stream_bound(n, bs)
        for k in range(1, 16):
            src = torch.zeros(n + 64, dtype=torch.uint8, device="cuda")
            src[k:k + n] = _dev(d)
            dst = torch.full((bound + 64,), 0xEE, dtype=torch.uint8, device="cuda")
            w = lib.lz4b200_stream_encode_device(ctx.handle, src.data_ptr() + k, n, bs, int(hc), dst.data_ptr() + 16 - k, bound, st)
            assert w == len(ref), (bs, k)
            hb = dst.cpu().numpy()
            assert hb[16 - k:16 - k + w].tobytes() == ref, (bs, k)
            assert (hb[:16 - k] == 0xEE).all() and (hb[16 - k + w:] == 0xEE).all(), (bs, k)
            out = torch.full((n + 64,), 0xEE, dtype=torch.uint8, device="cuda")
            wire = torch.zeros(w + 64, dtype=torch.uint8, device="cuda")
            wire[k:k + w] = dst[16 - k:16 - k + w]
            assert lib.lz4b200_stream_decode_device(ctx.handle, wire.data_ptr() + k, w, out.data_ptr() + k, n, st) == n
            ho = out.cpu().numpy()
            assert ho[k:k + n].tobytes() == d and (ho[:k] == 0xEE).all() and (ho[k + n:] == 0xEE).all(), (bs, k)


def test_python_layer_errors(ctx):
    import torch
    from lz4net_b200 import batch
    with pytest.raises(TypeError):
        batch.stream_encode(ctx, torch.zeros(10, dtype=torch.int32, device="cuda"))
    with pytest.raises(TypeError):
        batch.stream_decode(ctx, b"abc")
    with pytest.raises(ValueError):
        batch.stream_encode(ctx, torch.zeros(10, dtype=torch.uint8))                      # host tensor
    with pytest.raises(ValueError):
        batch.stream_encode(ctx, torch.zeros(20, dtype=torch.uint8, device="cuda")[::2])  # not contiguous
    d, ref = _case(65536, False)
    with pytest.raises(EOFError):
        batch.stream_decode(ctx, _dev(ref[:-1]))
    bad = bytearray(ref)
    p = len(_varint(1)) + len(_varint(65536)) + len(_varint(1))                            # first chunk's LZ4 payload
    assert ref[0] & 1
    bad[p + 5:p + 40] = bytes(35)
    with pytest.raises(ValueError):
        ctx.stream_decode(bytes(bad))
    with pytest.raises(ValueError):
        batch.stream_decode(ctx, _dev(bytes(bad)))


def test_ordered_on_the_callers_stream(ctx):
    """Input filled by synth_fill on a side stream is encoded on that stream, with no synchronisation in between."""
    import torch
    from lz4net_b200 import batch
    s = torch.cuda.Stream()
    nb, bs = 512, 65536
    with torch.cuda.stream(s):
        raw = torch.empty(nb * bs, dtype=torch.uint8, device="cuda")
        batch.synth_fill(ctx, raw, nb, bs, 3, seed=5)                     # ETEXT
        wire = batch.stream_encode(ctx, raw, bs)
        back = batch.stream_decode(ctx, wire)
        same = bool(torch.equal(back, raw))
    s.synchronize()
    assert same
    host = raw.cpu().numpy().tobytes()
    assert wire.cpu().numpy().tobytes() == ctx.stream_encode(host, bs)


@pytest.mark.parametrize("bs", [65536, 1 << 20])
def test_larger_than_one_encode_group(ctx, bs):
    """600 MiB of E50: the encoder works through 256 MiB groups of chunks; the wire equals the host's and round-trips."""
    import torch
    from lz4net_b200 import batch
    n = 600 << 20
    raw = torch.empty(n, dtype=torch.uint8, device="cuda")
    batch.synth_fill(ctx, raw, n // 65536, 65536, 1, seed=3)
    wire = batch.stream_encode(ctx, raw, bs)
    host = raw.cpu().numpy().tobytes()
    assert wire.cpu().numpy().tobytes() == ctx.stream_encode(host, bs)
    assert bool(torch.equal(batch.stream_decode(ctx, wire), raw))
