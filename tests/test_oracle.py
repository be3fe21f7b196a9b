"""CPU-only: pins the port oracle (oracle/lz4_oracle.c) to the reference's own sources through committed golden data:
golden_v1.json and reference_results.json, both written by tests/golden/make_golden.py from the reference's code
(oracle/_ref).  Mirrors src/LZ4.Tests/ConformanceTests.cs (all encoders byte-identical, all decoders round-trip) and
original/fuzzer.c:146-233 (size +-1 invariants)."""
import functools
import hashlib
import json
import os

import numpy as np
import pytest

import oracle
from tests import cases

GOLD = os.path.join(os.path.dirname(__file__), "golden", "golden_v1.json")
REF_RESULTS = os.path.join(os.path.dirname(__file__), "golden", "reference_results.json")


@functools.cache
def reference_results():
    with open(REF_RESULTS) as f:
        return json.load(f)


def _sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def digest(*parts) -> str:
    """16 hex digits of SHA-256 over a sequence of ints and byte strings (results too many to store whole)."""
    h = hashlib.sha256()
    for p in parts:
        if isinstance(p, bytes):
            h.update(len(p).to_bytes(8, "little")); h.update(p)
        else:
            h.update(int(p).to_bytes(8, "little", signed=True))
    return h.hexdigest()[:16]


def test_bound():
    for n in (0, 1, 254, 255, 256, 65536, 1 << 20):
        assert oracle.bound(n) == oracle.port().lz4o_bound(n) == n + n // 255 + 16
    assert oracle.bound(65536) == 65809            # src/LZ4/LZ4Codec.cs:313-316


def test_golden_vectors_port():
    """The port reproduces every committed golden vector (made from oracle/_ref by make_golden.py)."""
    g = json.load(open(GOLD))
    assert len(g["cases"]) >= 40
    for c in g["cases"]:
        data = cases.AUTOTEST if c["model"] == "autotest" else cases.content(c["model"], c["n"], c["seed"]).tobytes()
        assert _sha(data) == c["input_sha256"], c["name"]
        for mode, fn in (("fast", oracle.encode), ("hc", oracle.encode_hc)):
            r, out = fn(data, impl="port")
            assert r == c[mode]["len"], (c["name"], mode)
            assert _sha(out) == c[mode]["sha256"], (c["name"], mode)
            if "hex" in c[mode]:
                assert out.hex() == c[mode]["hex"]
            rr, dec = oracle.decode_known(out, len(data), impl="port")
            assert rr == r and dec == data
            # LZ4Stream / Wrap pass cap = n (src/LZ4/LZ4Stream.cs:243-246): the stored-raw decision is part of parity
            r2, _ = fn(data, cap=len(data), impl="port")
            assert r2 == c[mode]["len_cap_n"], (c["name"], mode)


# ---- the port against the reference's own results (reference_results.json).  The functions below compute the results
# with either implementation: make_golden.py stores the reference's, the tests compare the port's with them. -----------
def random_length_inputs(model):
    lens = cases.random_lengths(60, 200_000, seed=7) + list(cases.BOUNDARY_LENGTHS)
    out = []
    for i, n in enumerate(lens):
        if model in ("mixed",) and n > 70_000:
            n = n % 70_000
        out.append((n, cases.content(model, n, seed=i).tobytes()))
    return out


def encode_results(data, impl):
    """Both encoders on one input.  Returns the digest of every return value and output byte (at the bound, and with
    the output limited to exactly enough, one short and cap = n: fuzzer.c:212-227; LZ4Stream.cs:243-246) and the
    (return value, bytes) of each encoder at the bound."""
    n = len(data)
    parts, full = [], []
    for fn in (oracle.encode, oracle.encode_hc):
        r, out = fn(data, impl=impl)
        full.append((r, out)); parts += [r, out]
        for cap in sorted({r, r - 1, n, max(0, n - 1), r // 2}):
            if cap >= 0:
                parts += [cap, *fn(data, cap=cap, impl=impl)]
    return digest(*parts), full


@pytest.mark.parametrize("model", cases.MODELS)
def test_port_equals_reference_random_lengths(model):
    want = reference_results()["random_lengths"][model]
    inputs = random_length_inputs(model)
    assert [n for n, _ in inputs] == [n for n, _ in want]
    for (n, data), (_, ref_digest) in zip(inputs, want):
        port_digest, full = encode_results(data, "port")
        assert port_digest == ref_digest, (model, n)
        for r, out in full:
            d1 = oracle.decode_known(out, n, impl="port")
            d2 = oracle.decode_unknown(out, n, impl="port")
            assert d1 == (r, data) and d2 == (n if n else d2[0], data)


def accept_reject_inputs():
    """(fuz, data): fuz marks the upstream generator, for which the +-1 invariants are strict (fuzzer.c:176-210)."""
    rng = np.random.default_rng(3)
    from lz4net_b200 import synth
    out = []
    for i in range(48):
        fuz = i % 6 == 5
        data = (synth.fuz_block(i, 4096) if fuz else
                cases.content(cases.MODELS[i % len(cases.MODELS)], int(rng.integers(20, 40000)), seed=100 + i)).tobytes()
        out.append((fuz, data))
    return out


def unknown_size_cases(clen, n):
    """(input size, output capacity) pairs the unknown-size decoder is tried with."""
    return ((clen, n + 1), (clen, n), (clen, n - 1), (clen - 1, n), (clen + 1, n))


def unknown_result(comp, cap, impl):
    r, out = oracle.decode_unknown(comp, cap, impl=impl)
    return [r, digest(out) if r >= 0 else None]


def accept_reject_results(comp, n, impl):
    """The decoders' verdicts on a stream of n bytes: known-size at n, n - 1, n + 1; unknown-size at unknown_size_cases."""
    clen = len(comp)
    known = [oracle.decode_known(comp, osize, impl=impl)[0] for osize in (n, n - 1, n + 1)]
    unknown = [unknown_result((comp if isz <= clen else comp + b"\x00")[:isz], osz, impl)
               for isz, osz in unknown_size_cases(clen, n)]
    return {"comp": digest(comp), "known": known, "unknown": unknown}


def test_decoders_accept_reject_like_reference():
    """fuzzer.c:176-210: exact size works, size +-1 must fail; the port takes the same decisions as the reference."""
    want = reference_results()["accept_reject"]
    for i, ((fuz, data), ref) in enumerate(zip(accept_reject_inputs(), want, strict=True)):
        n = len(data)
        _, comp = oracle.encode(data, impl="port")
        clen = len(comp)
        port = accept_reject_results(comp, n, "port")
        assert port["comp"] == ref["comp"], i                   # the decoders see the reference's stream
        for osize, a, b in zip((n, n - 1, n + 1), ref["known"], port["known"]):
            assert (a < 0) == (b < 0) and (a < 0 or a == b), (i, osize, a, b)
            assert (osize == n) == (a >= 0)
        for (isz, osz), a, b in zip(unknown_size_cases(clen, n), ref["unknown"], port["unknown"]):
            assert (a[0] < 0) == (b[0] < 0), (i, isz, osz, a[0], b[0])
            if a[0] >= 0:
                assert a == b
            if fuz or isz == clen:
                # (on arbitrary data a truncated stream can, rarely, still parse: the match-length loop stops at
                #  iend-6 and re-reads its last byte as a token, original/lz4.c:986-999)
                assert (a[0] >= 0) == (isz == clen and osz >= n)


def corrupt_streams(impl):
    """300 fast-encoded blocks with 1-3 bit flips each.  Returns (the encoded blocks, [(raw size, flipped stream)])."""
    rng = np.random.default_rng(11)
    comps, streams = [], []
    for i in range(300):
        data = cases.content("mixed", 3000, seed=i).tobytes()
        _, comp = oracle.encode(data, impl=impl)
        c = bytearray(comp)
        for _ in range(int(rng.integers(1, 4))):
            c[int(rng.integers(0, len(c)))] ^= 1 << int(rng.integers(0, 8))
        comps.append(comp); streams.append((len(data), bytes(c)))
    return comps, streams


def test_corrupt_streams_same_verdict():
    """Bit-flipped streams: the port must never crash and must agree with the reference on accept/reject
    (and on the bytes when both accept), except for offset-0 matches which the port rejects by design."""
    want = reference_results()["corrupt_streams"]
    comps, streams = corrupt_streams("port")
    assert digest(*comps) == want["comp"]                       # the flips hit the reference's streams
    agree = 0
    for (n, c), a in zip(streams, want["verdicts"], strict=True):
        b = unknown_result(c, n, "port")
        if (a[0] < 0) == (b[0] < 0):
            agree += 1
            if a[0] >= 0:
                assert a == b
        else:
            assert a[0] >= 0 and b[0] < 0          # only the documented tightening (offset == 0)
    assert agree >= 290


def test_fuz_generator_roundtrip():
    from lz4net_b200 import synth
    for seed in range(4):
        data = synth.fuz_block(seed, 8192).tobytes()
        r, c = oracle.encode(data)
        rh, ch = oracle.encode_hc(data)
        assert oracle.decode_known(c, len(data)) == (r, data)
        assert oracle.decode_known(ch, len(data)) == (rh, data)
        assert oracle.decode_known(c, len(data) - 1)[0] < 0 and oracle.decode_known(c, len(data) + 1)[0] < 0
