"""CPU-only logic tests of the CUDA kernel source, run through the warp emulator (tests/simt_emu).

The kernels' algorithms (lz4net_b200/csrc/lz4_decode.cuh, lz4_encode.cuh, lz4_copy.cuh) are compiled with g++ in
emulation mode and compared with the oracle -- the same checks the `-m gpu` parity tests make on the B200 through the
C ABI, at sizes the emulator finishes in seconds.  Shape: lz4net's ConformanceTests (byte-identical encoders, every
decoder round-trips, src/LZ4.Tests/ConformanceTests.cs:57-148) + the upstream fuzzer's size +-1 invariants
(original/fuzzer.c:176-227)."""
import numpy as np
import pytest

import oracle
from tests import cases, emu
from tests.test_oracle import reference_results


def _enc_check(blocks, caps=None, **kw):
    res, outs = emu.encode(blocks, caps, **kw)
    for i, b in enumerate(blocks):
        cap = None if caps is None else caps[i]
        r, o = oracle.encode(b, cap=cap)
        assert (res[i], outs[i]) == (r, o), (i, len(b), cap, res[i], r)


@pytest.mark.parametrize("model", cases.MODELS)
def test_encode_matches_oracle_64k_and_random_lengths(model):
    lens = [65536] + cases.random_lengths(10, 65546, seed=21) + [65546, 65535]
    blocks = [cases.content(model, n, seed=300 + i).tobytes() for i, n in enumerate(lens)]
    _enc_check(blocks, sched_seed=5)


def test_encode_boundary_lengths():
    blocks = []
    for n in cases.BOUNDARY_LENGTHS:
        if n <= 65546:
            for m in ("lowent", "periodic", "E50"):
                blocks.append(cases.content(m, n, seed=n).tobytes())
    _enc_check(blocks, sched_seed=9)


def test_encode_limited_output():
    """cap = exactly enough / one short / n (LZ4Stream, Wrap) / tiny: same return value and bytes, no overrun."""
    blocks, caps = [], []
    for i, m in enumerate(cases.MODELS):
        for n in (200, 3000, 65536):
            d = cases.content(m, n, seed=40 + i).tobytes()
            r, _ = oracle.encode(d)
            for cap in (r, r - 1, n, n - 1, r // 2, 0, 1, 7, 8, 13):
                if cap >= 0:
                    blocks.append(d); caps.append(cap)
    _enc_check(blocks, caps, sched_seed=3)


def test_encode_output_limit_inside_every_emission_batch():
    """The encoder evaluates the reference's output-limit checks for 32 parked sequences at a time: sweep the capacity
    over the whole compressed size so that the first failing sequence falls at every position of such a batch."""
    for model, n in (("ETEXT", 1500), ("lowent", 1200), ("E50", 2500)):
        d = cases.content(model, n, seed=5).tobytes()
        r, _ = oracle.encode(d)
        caps = list(range(0, r + 3))
        _enc_check([d] * len(caps), caps, sched_seed=8)


def test_encode_never_reads_past_the_input():
    """The block ends on the last byte of a mapped page (next page PROT_NONE): a load of any word that holds no input
    byte would fault.  Covers the unaligned 32-bit reads of the parse, the match-length count up to matchlimit, the
    literal copies and the long-match / long-literal paths."""
    for model, n in (("E50", 65536), ("ETEXT", 65536), ("E100", 65536), ("E0", 8192), ("lowent", 4096), ("periodic", 65536),
                     ("runs", 20000), ("mixed", 12), ("mixed", 16), ("ETEXT", 70000)):
        d = cases.content(model, n, seed=n % 97).tobytes()
        assert emu.encode_guarded(d, sched_seed=3) == oracle.encode(d), (model, n)
    # every source alignment and every position of the block end inside its last word
    for n in (4093, 4094, 4095, 4096, 13, 14, 15):
        for pad in range(4):
            if (n + pad) % 4 == 0 or pad == 0:
                d = cases.content("lowent", n, seed=n + pad).tobytes()
                e = (4 - n % 4) % 4 if pad else 0
                assert emu.encode_guarded(d, sched_seed=4, end_pad=e) == oracle.encode(d), (n, e)


def test_encode_general_variant_above_64k():
    """n >= 65547 takes LZ4_compressCtx (original/lz4.c:345-562): 12-bit hash, u32 table, distance checks."""
    blocks = [cases.content(m, n, seed=7).tobytes()
              for m, n in (("ETEXT", 65547), ("lowent", 70001), ("E50", 150000), ("periodic", 140000), ("mixed", 69999),
                           ("E100", 200000), ("runs", 131072), ("E0", 66000))]
    _enc_check(blocks, sched_seed=2)
    caps = [oracle.encode(b)[0] - 1 for b in blocks]
    _enc_check(blocks, caps, sched_seed=4)


@pytest.mark.parametrize("skew", [1, 3, 7, 13])
def test_encode_unaligned_buffers(skew):
    blocks = [cases.content(m, 5000 + skew, seed=skew).tobytes() for m in cases.MODELS]
    res, outs = emu.encode(blocks, sched_seed=skew, src_skew=skew, dst_skew=16 - skew)
    for b, r, o in zip(blocks, res, outs):
        assert (r, o) == oracle.encode(b)


@pytest.mark.parametrize("variant", [1])
def test_encode_other_duplicate_detectors(variant):
    """The always-exact (vote-per-hash-bit, 32 iterations per round) form of the round gives the same bytes as the default."""
    blocks = [cases.content(m, n, seed=90 + i).tobytes() for i, m in enumerate(cases.MODELS) for n in (65536, 4097)]
    _enc_check(blocks, sched_seed=6, variant=variant)


@pytest.mark.parametrize("tune", [(0, 0, 0), (64, 1000, 1000), (32, 0, 1000), (0, 1000, 0)])
def test_encode_heuristics_never_change_the_bytes(tune):
    """lane_copy_max / probe_max / wide_min only choose between equivalent code paths (per-lane or cooperative literal
    copies, probe-first or fused round, 32 or 64 iterations per round): every extreme setting emits the oracle's bytes."""
    blocks = [cases.content(m, n, seed=70 + i).tobytes() for i, m in enumerate(cases.MODELS) for n in (65536, 3001)]
    _enc_check(blocks, sched_seed=7, tune=tune)


def test_encode_fuzz_small_blocks():
    """Random content model, length, capacity, buffer alignment, lane schedule, round variant and heuristics: the
    encoder's return value and bytes are the oracle's, and it never writes outside [dst, dst + cap)."""
    rng = np.random.default_rng(2024)
    for trial in range(40):
        blocks, caps = [], []
        for _ in range(8):
            n = int(rng.choice([int(rng.integers(0, 64)), int(rng.integers(64, 3000)), int(rng.integers(3000, 9000))]))
            d = cases.content(str(rng.choice(cases.MODELS)), n, seed=int(rng.integers(1 << 30))).tobytes()
            r, _ = oracle.encode(d)
            cap = int(rng.choice([n + n // 255 + 16, r, max(r - 1, 0), n, int(rng.integers(0, max(r, 1) + 8))]))
            blocks.append(d); caps.append(cap)
        tune = (int(rng.choice([0, 12, 64])), int(rng.choice([0, 8, 1000])), int(rng.choice([0, 24, 1000])))
        res, outs = emu.encode(blocks, caps, sched_seed=int(rng.integers(1, 1 << 20)), src_skew=int(rng.integers(0, 8)),
                               dst_skew=int(rng.integers(0, 16)), variant=int(rng.choice([1, 2])), tune=tune)
        for b, c, r, o in zip(blocks, caps, res, outs):
            assert (r, o) == oracle.encode(b, cap=c), (trial, len(b), c, tune)


def test_encode_schedule_independent():
    """Lanes are scheduled in different orders: the result may not depend on lock-step luck."""
    blocks = [cases.content("lowent", 20000, seed=1).tobytes(), cases.content("mixed", 20000, seed=2).tobytes()]
    for seed in range(1, 6):
        _enc_check(blocks, sched_seed=seed)


@pytest.mark.parametrize("lanes", [32, 16, 8, 4, 132, 116, 108, 104, 1, 2])
@pytest.mark.parametrize("known", [True, False])
def test_decode_matches_oracle(lanes, known):
    blocks, raws = [], []
    for i, m in enumerate(cases.MODELS):
        for n in (65536, 1, 12, 13, 700, 33000):
            d = cases.content(m, n, seed=60 + i).tobytes()
            for fn in (oracle.encode, oracle.encode_hc):
                blocks.append(fn(d)[1]); raws.append(d)
    res, outs = emu.decode(blocks, [len(r) for r in raws], lanes=lanes, known=known, sched_seed=lanes)
    for c, d, r, o in zip(blocks, raws, res, outs):
        assert r == (len(c) if known else len(d)), (len(d), r)
        assert o == d


@pytest.mark.parametrize("lanes", [32, 8, 116, 1, 2])
def test_decode_size_invariants(lanes):
    """fuzzer.c:176-210 -- exact size works; size +-1 fails; verdicts equal the oracle's (which is pinned to the reference)."""
    from lz4net_b200 import synth
    comp, caps, known_flags, expect = [], [], [], []
    for seed in range(6):
        d = synth.fuz_block(seed, 6000).tobytes()
        c = oracle.encode(d)[1]
        n = len(d)
        for osz in (n, n - 1, n + 1):
            comp.append(c); caps.append(osz); known_flags.append(True); expect.append(oracle.decode_known(c, osz)[0])
        for cc, osz in ((c, n + 1), (c, n), (c, n - 1), (c[:-1], n), (c + b"\0", n)):
            comp.append(cc); caps.append(osz); known_flags.append(False); expect.append(oracle.decode_unknown(cc, osz)[0])
    for known in (True, False):
        idx = [i for i, k in enumerate(known_flags) if k == known]
        res, _ = emu.decode([comp[i] for i in idx], [caps[i] for i in idx], lanes=lanes, known=known, sched_seed=11)
        for i, r in zip(idx, res):
            assert (r < 0) == (expect[i] < 0), (i, r, expect[i])
            if expect[i] >= 0:
                assert r == expect[i]


@pytest.mark.parametrize("known", [True, False])
def test_decode_corrupt_streams_never_escape(known):
    """Bit flips / truncations: same accept-reject verdict as the oracle, identical bytes when accepted, and no write
    outside [dst, dst+cap) (emu.decode asserts the red zones)."""
    rng = np.random.default_rng(5)
    comp, caps = [], []
    for i in range(120):
        d = cases.content("mixed", 2500, seed=i).tobytes()
        c = bytearray(oracle.encode(d)[1])
        kind = i % 3
        if kind == 0:
            for _ in range(int(rng.integers(1, 4))):
                c[int(rng.integers(0, len(c)))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:
            c = c[: int(rng.integers(1, len(c)))]
        else:
            c[int(rng.integers(0, len(c)))] = 0xFF
        comp.append(bytes(c)); caps.append(len(d))
    res, outs = emu.decode(comp, caps, lanes=32, known=known, sched_seed=13)
    for other in (108, 1, 2):                                   # output-staged variant with 8 lanes; lane-per-block decoder
        res2, outs2 = emu.decode(comp, caps, lanes=other, known=known, sched_seed=14)
        assert [r < 0 for r in res2] == [r < 0 for r in res] and [r for r in res2 if r >= 0] == [r for r in res if r >= 0]
        assert [o for r, o in zip(res2, outs2) if r >= 0] == [o for r, o in zip(res, outs) if r >= 0]
    for c, cap, r, o in zip(comp, caps, res, outs):
        er, eo = (oracle.decode_known if known else oracle.decode_unknown)(c, cap)
        assert (r < 0) == (er < 0), (r, er)
        if er >= 0:
            assert r == er and o[:len(eo)] == eo


@pytest.mark.parametrize("skew", [1, 5, 15])
def test_decode_unaligned_stream_start(skew):
    raws = [cases.content(m, 9000, seed=skew).tobytes() for m in cases.MODELS]
    comp = [oracle.encode(d)[1] for d in raws]
    for lanes in (16, 116, 108, 1, 2):
        res, outs = emu.decode(comp, [len(d) for d in raws], lanes=lanes, known=True, sched_seed=skew, src_skew=skew)
        assert outs == raws and res == [len(c) for c in comp]


def test_decode_long_overlapping_matches():
    """RLE-style matches (offset < length), every small offset, long enough to take the wide path (SURVEY 7.2-H4)."""
    raws = []
    for off in list(range(1, 40)) + [63, 64, 65, 255, 256, 511, 512, 527, 528, 529, 1000]:
        rng = np.random.default_rng(off)
        pat = rng.integers(0, 256, off, dtype=np.uint8)
        raws.append(np.tile(pat, 9000 // off + 2)[:9000].tobytes())
    comp = [oracle.encode(d)[1] for d in raws]
    for lanes in (32, 16, 8, 4, 132, 116, 108, 104, 1, 2):
        res, outs = emu.decode(comp, [len(d) for d in raws], lanes=lanes, known=True, sched_seed=lanes)
        assert outs == raws


def test_decode_lane_per_block_fuzz():
    """The lane-per-block decoder over random content models, lengths, stream / output alignments, ring geometries and
    lane schedules, for both decoders and both encoders' streams: every lane walks its own block, so blocks of very
    different cost share a warp (literal runs and matches longer than 64 bytes go through the warp-wide copy)."""
    rng = np.random.default_rng(77)
    for trial in range(24):
        raws = []
        for _ in range(int(rng.integers(20, 70))):
            n = int(rng.choice([int(rng.integers(1, 40)), int(rng.integers(40, 2000)), int(rng.integers(2000, 20000))]))
            raws.append(cases.content(str(rng.choice(cases.MODELS)), n, seed=int(rng.integers(1 << 30))).tobytes())
        comp = [(oracle.encode_hc if rng.integers(2) else oracle.encode)(d)[1] for d in raws]
        known = bool(rng.integers(2))
        caps = [len(d) if known else len(d) + int(rng.integers(0, 40)) for d in raws]
        res, outs = emu.decode(comp, caps, lanes=int(rng.choice([1, 2])), known=known, sched_seed=int(rng.integers(1, 1 << 20)),
                               src_skew=int(rng.integers(0, 16)), dst_skew=int(rng.integers(0, 16)))
        for c, d, cap, r, o in zip(comp, raws, caps, res, outs):
            assert r == (len(c) if known else len(d)), (trial, len(d), r)
            assert o[:len(d)] == d, (trial, len(d))


# ---- LZ4HC (one thread per block: the device source compiled as plain scalar code) ------------------------------------
@pytest.mark.parametrize("model", cases.MODELS)
def test_encode_hc_matches_oracle(model):
    """Byte-identical to the reference's LZ4_compressHC_limitedOutput (original/lz4hc.c:745-755) through the oracle."""
    for i, n in enumerate([65536, 0, 1, 12, 13, 64, 4097] + cases.random_lengths(3, 65546, seed=5)):
        d = cases.content(model, n, seed=500 + i).tobytes()
        assert emu.encode_hc(d) == oracle.encode_hc(d), (model, n)


def test_encode_hc_limited_output_and_alignment():
    for i, m in enumerate(("ETEXT", "lowent", "E50", "periodic")):
        d = cases.content(m, 5000, seed=40 + i).tobytes()
        r, _ = oracle.encode_hc(d)
        for cap in (r, r - 1, len(d), r // 2, 0, 1, 7, 13):
            assert emu.encode_hc(d, cap=cap) == oracle.encode_hc(d, cap=cap), (m, cap)
        for skew in (1, 2, 3):
            assert emu.encode_hc(d, src_skew=skew) == oracle.encode_hc(d), (m, skew)


def test_encode_hc_above_64k():
    for m, n in (("ETEXT", 70001), ("periodic", 140000), ("E100", 200000), ("mixed", 131072)):
        d = cases.content(m, n, seed=9).tobytes()
        assert emu.encode_hc(d) == oracle.encode_hc(d), (m, n)


# ---- LZ4HC, one WARP per block on a static index (lz4hc_warp.cuh) -----------------------------------------------------
def _hcw_check(d, cap=None, **kw):
    """The warp kernel either emits the reference's bytes or hands the block back (never anything else); both placements
    of the block (staged in shared memory / read through the read-only path) take the same decision."""
    want = oracle.encode_hc(d, cap=cap)
    verdicts = []
    for smem in (True, False):
        r, o = emu.encode_hcw(d, cap=cap, smem=smem, **kw)
        verdicts.append(r == emu.HCW_FALLBACK)
        if r != emu.HCW_FALLBACK:
            assert (r, o) == want, (len(d), cap, smem, kw)
    assert verdicts[0] == verdicts[1]
    return not verdicts[0]


@pytest.mark.parametrize("model", cases.MODELS)
def test_encode_hcw_matches_oracle(model):
    """Byte-identical to LZ4_compressHC_limitedOutput (original/lz4hc.c:745-755): the chain walks of :423-433 / :477-514
    replaced by gathers from the sorted hash buckets."""
    done = 0
    for i, n in enumerate([65536, 4097] + cases.random_lengths(2, 65536, seed=5)):
        d = cases.content(model, n, seed=500 + i).tobytes()
        done += _hcw_check(d, sched_seed=3 + i)
    assert done >= 3, "the static index should describe (nearly) every block"


def test_encode_hcw_boundary_lengths():
    for n in cases.BOUNDARY_LENGTHS:
        if n <= 65536:
            for m in (("lowent", "periodic", "E50", "E100") if n < 4000 else ("periodic", "E50")):
                assert _hcw_check(cases.content(m, n, seed=n).tobytes(), sched_seed=n + 1), (m, n)


def test_encode_hcw_limited_output_and_alignment():
    for i, m in enumerate(("ETEXT", "lowent", "E50", "periodic", "runs", "E0")):
        d = cases.content(m, 3000, seed=40 + i).tobytes()
        r, _ = oracle.encode_hc(d)
        for cap in (r, r - 1, len(d), len(d) - 1, r // 2, 0, 1, 7, 8, 13):
            assert _hcw_check(d, cap=cap), (m, cap)
        for skew in (1, 2, 3, 7, 13):
            assert _hcw_check(d, src_skew=skew, dst_skew=(skew * 5) % 16, sched_seed=skew), (m, skew)
    # the capacity swept over a whole compressed block: every limit check of :529 / :541 / :731 fails once
    d = cases.content("ETEXT", 700, seed=5).tobytes()
    r, _ = oracle.encode_hc(d)
    for cap in range(0, r + 3):
        assert _hcw_check(d, cap=cap), cap


def test_encode_hcw_fuzz():
    """Random models / lengths / capacities / alignments / lane schedules."""
    rng = np.random.default_rng(20260924)
    handed_back = 0
    for trial in range(40):
        m = cases.MODELS[int(rng.integers(len(cases.MODELS)))]
        n = int(np.exp(rng.random() * np.log(65536)))
        d = cases.content(m, n, seed=int(rng.integers(1 << 30))).tobytes()
        cap = None
        if rng.integers(3) == 0:
            cap = int(rng.integers(0, oracle.encode_hc(d)[0] + 4))
        handed_back += not _hcw_check(d, cap=cap, src_skew=int(rng.integers(16)), dst_skew=int(rng.integers(16)),
                                      sched_seed=int(rng.integers(1, 1 << 20)))
    assert handed_back <= 2


def test_encode_hcw_upstream_fuzzer_buffers():
    for seed in range(6):
        from lz4net_b200 import synth
        d = synth.fuz_block(seed, 20000).tobytes()
        assert _hcw_check(d, sched_seed=seed + 1), seed


def _hash15(b4):
    return ((int.from_bytes(b4, "little") * 2654435761) & 0xFFFFFFFF) >> 17


def test_encode_hcw_hands_back_what_the_static_index_does_not_describe():
    """Larger than 64 KiB; and a run of period 3 two of whose strings share a hash bucket: the reference's repeat detector
    (original/lz4hc.c:437-455) writes chain deltas of 3 across positions whose real predecessor in the bucket is 1 back."""
    assert emu.encode_hcw(cases.content("ETEXT", 65537, seed=1).tobytes())[0] == emu.HCW_FALLBACK
    found = None
    for a in range(1, 256):
        for b in range(a + 1, 256):
            for c in range(b + 1, 256):
                s0, s1, s2 = bytes([a, b, c, a]), bytes([b, c, a, b]), bytes([c, a, b, c])
                if _hash15(s1) == _hash15(s2) and _hash15(s0) != _hash15(s1):
                    found = (a, b, c); break
            if found: break
        if found: break
    assert found, "no colliding triple"
    rng = np.random.default_rng(3)
    d = rng.integers(0, 256, 500, dtype=np.uint8).tobytes() + bytes(found) * 200 + rng.integers(0, 256, 500, dtype=np.uint8).tobytes()
    assert emu.encode_hcw(d)[0] == emu.HCW_FALLBACK
    # the same run with a triple that does not collide is encoded here
    assert _hcw_check(rng.integers(0, 256, 500, dtype=np.uint8).tobytes() + bytes([1, 2, 3]) * 200 + bytes(500))


def test_encode_hc_gives_up_at_the_bound_like_the_reference():
    """r93's LZ4HC can return 0 with a destination of LZ4_compressBound(n) bytes: incompressible data with one late match
    (about one random 64 KiB block in 400).  The reference compiled in place, the port and every kernel agree on it."""
    from lz4net_b200 import synth
    d = synth.make_blocks("E0", 1, 65536, seed=3, first_block=1268)[0].tobytes()
    cap = oracle.bound(len(d))
    assert oracle.encode_hc(d, cap=cap)[0] == 0 and oracle.encode_hc(d, cap=cap + 4096)[0] == 65794
    # the reference's own return values on this block at cap and cap + 4096 (tests/golden/make_golden.py)
    assert reference_results()["encode_hc_gives_up_at_the_bound"] == [0, 65794]
    assert emu.encode_hc(d, cap=cap)[0] == 0
    for smem in (True, False):
        assert emu.encode_hcw(d, cap=cap, smem=smem)[0] == 0
        assert emu.encode_hcw(d, cap=cap + 4096, smem=smem) == oracle.encode_hc(d, cap=cap + 4096)
