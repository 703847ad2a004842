"""Kernel LOGIC on the CPU simulator (tests/sim): the same .cu sources compiled with -DBZ_SIM.
Parity is checked against the oracle; the real-GPU parity tests are in test_gpu_parity.py."""
import os
import numpy as np
import pytest

from conftest import fixture_bytes

RNG = np.random.default_rng(11)
SMALL = {
    "empty": b"", "one": b"Q", "aaaa": b"aaaa", "aaaaa": b"aaaaa", "a256": b"a" * 256, "a255x": b"a" * 255 + b"x",
    "zeros1000": bytes(1000), "abab": b"abab", "abc3": b"abcabcabc", "sample0": b"This is a test\n",
    "text5k": (b"the quick brown fox jumps over the lazy dog. " * 120)[:5000],
    "rand3k": RNG.integers(0, 256, 3000, dtype=np.uint8).tobytes(),
    "rand4sym": RNG.integers(0, 4, 20000, dtype=np.uint8).tobytes(),
    "two_sym_d1": bytes(RNG.integers(0, 2, 6000, dtype=np.uint8)),
}


@pytest.mark.parametrize("name", sorted(SMALL))
def test_compress_parity_small(sim_engine, oracle, name):
    data = SMALL[name]
    exp, st = oracle.compress(data, 9, return_stats=True)
    assert sim_engine.compressFile(data, None, 9) == exp
    if not st.d1_triggered:
        assert sim_engine.decompressFile(exp) == data


def test_bwt_group_classes(sim_engine, oracle):
    """Small (counting), medium (dense shared-memory radix) and big (global radix, passed through) groups of the
    doubling rounds, alone and mixed inside one tile; periodic blocks end with the descending-index tie rule."""
    rng = np.random.default_rng(5)
    cases = {
        "ab5000": b"ab" * 5000, "abc3000": b"abc" * 3000, "two50k": bytes(rng.integers(0, 2, 50000, dtype=np.uint8)),
        "mix": b"ab" * 3000 + bytes(rng.integers(97, 123, 20000, dtype=np.uint8)) + b"xyz" * 2500 + bytes(rng.integers(0, 2, 9000, dtype=np.uint8)),
        "period97": bytes(rng.integers(97, 123, 97, dtype=np.uint8)) * 400,
        "three": bytes(rng.integers(0, 3, 30000, dtype=np.uint8)),
    }
    for name, data in cases.items():
        assert sim_engine.compressFile(data, None, 9) == oracle.compress(data, 9), name


def test_compress_parity_multiblock_level1(sim_engine, oracle):
    data = fixture_bytes("sample5.ref")[:230_000]
    exp = oracle.compress(data, 1)
    assert sim_engine.compressFile(data, None, 1) == exp
    assert sim_engine.stats().n_blocks == 3


def test_stage_dumps_match_oracle(sim_engine, oracle):
    data = fixture_bytes("sample1.ref")[:40_000]
    sim_engine.compressFile(data, None, 9)
    recs, metas = sim_engine.block_table(), sim_engine.block_meta()
    blk, used, crc = oracle.rle1_block(data, 899981)
    assert (recs[0].s, recs[0].p, recs[0].n, recs[0].crc) == (0, used, len(blk), crc)
    assert sim_engine.debug_fetch(1, 0, recs[0].n).tobytes() == blk.tobytes()
    st = oracle.block_stages(blk)
    assert sim_engine.debug_fetch(2, 0, recs[0].n).tobytes() == st["U"].tobytes() and recs[0].orig_ptr == st["orig_ptr"]
    A = np.frombuffer(sim_engine.debug_fetch(3, 0, 2 * metas[0].m).tobytes(), dtype=np.uint16)
    assert np.array_equal(A, st["A"]) and metas[0].alpha == st["alpha"]
    assert (metas[0].n_groups, metas[0].n_sel, metas[0].bits) == (st["n_groups"], st["n_sel"], st["bits"] + 80)


def _runny(rng, n, nsym, plong):
    out = bytearray()
    while len(out) < n:
        v = int(rng.integers(0, nsym))
        r = rng.random()
        if r < plong:
            L = int(rng.choice([4, 5, 6, 7, 8, 254, 255, 256, 257, 258, 259, 260, 509, 510, 511, 512, 513, 700, 1500]))
        elif r < plong + 0.2:
            L = int(rng.integers(2, 6))
        else:
            L = 1
        out += bytes([v]) * L
    return bytes(out[:n])


def test_cut_points_stress_tiny_blocks(sim_engine, oracle):
    """Runs straddling a cut, blocks ending on the 4th run byte / on the count byte, 255-byte chunking:
    thousands of cuts by overriding the block capacity in both the oracle and the kernels."""
    rng = np.random.default_rng(7)
    try:
        for it in range(12):
            cap = int(rng.choice([8, 9, 10, 11, 12, 13, 17, 50, 64, 100, 255, 256, 1000]))
            data = _runny(rng, int(rng.integers(1, 5000)), int(rng.choice([1, 2, 3, 200])), float(rng.choice([0.02, 0.2, 0.6])))
            oracle.set_block_cap(cap)
            sim_engine.debug_set_block_cap(cap)
            exp = oracle.compress(data, 9)
            got = sim_engine.compressFile(data, None, 9)
            assert got == exp, f"cap={cap} n={len(data)}"
            starts, lens, crcs = oracle.cut_points(data, 9)
            recs = sim_engine.block_table()
            assert [(r.s, r.n, r.crc) for r in recs] == list(zip(starts[:-1], lens, crcs))
    finally:
        oracle.set_block_cap(0)
        sim_engine.debug_set_block_cap(0)


def test_cut_points_many_tiles_speculation(sim_engine, oracle):
    """More blocks than the cut kernel speculates per round, spread over many 4 KiB tiles: text-like stretches
    (every speculated link holds), stretches of long runs (links break) and mixed."""
    rng = np.random.default_rng(19)
    text = rng.integers(97, 123, 120_000, dtype=np.uint8).tobytes()
    runs = _runny(rng, 60_000, 3, 0.5)
    zeros = bytes(70_000)
    data = text[:50_000] + runs[:30_000] + zeros + text[50_000:] + runs[30_000:] + b"x" * 9000 + text[:20_000]
    try:
        for cap in (997, 4099, 20_011):
            oracle.set_block_cap(cap)
            sim_engine.debug_set_block_cap(cap)
            starts, lens, crcs = oracle.cut_points(data, 9)
            sim_engine.compressFile(data, None, 9)
            recs = sim_engine.block_table()
            assert [(r.s, r.n, r.crc) for r in recs] == list(zip(starts[:-1], lens, crcs)), f"cap={cap}"
    finally:
        oracle.set_block_cap(0)
        sim_engine.debug_set_block_cap(0)


def _shards_stitched(eng, data, world, halo):
    """the shard protocol driven in-process: `world` shards compressed one after the other, stitched on the host"""
    n = len(data)
    slice_len = (n + world - 1) // world
    start, bitpos, segs, infos = 0, 32, [], []
    for r in range(world):
        base = r * slice_len
        own = max(0, min(slice_len, n - base))
        eng.shard_begin(data[base:min(n, base + own + halo)], 9)
        info = eng.shard_cut(max(start - base, 0), own, r == world - 1)
        assert info.complete
        start = max(base + info.next_start, start)
        eng.shard_compress(info)
        segs.append(eng.shard_emit(info, bitpos & 7))
        infos.append(info)
        bitpos += info.bits
    return eng.stitch_shards(9, segs, infos)


def test_batched_blocks_same_stream(sim_engine, oracle):
    """More blocks than one batch holds: the batches are stitched behind one another at the running bit offset, for a
    whole stream and for the shard segments of the shard protocol and of the stream compressor."""
    import io
    data = fixture_bytes("sample5.ref")[:150_000] + bytes(3000) + b"ab" * 4000
    try:
        oracle.set_block_cap(9000)
        sim_engine.debug_set_block_cap(9000)
        exp = oracle.compress(data, 9)
        for per in (1, 3, 7, 100):
            sim_engine.debug_set_batch_blocks(per)
            assert sim_engine.compressFile(data, None, 9) == exp, per
            starts, lens, crcs = oracle.cut_points(data, 9)
            assert [(r.s, r.n, r.crc) for r in sim_engine.block_table()] == list(zip(starts[:-1], lens, crcs))
            assert sim_engine.compressStream(io.BytesIO(data), None, 9, chunk_bytes=60_000) == exp, per
            assert _shards_stitched(sim_engine, data, 2, 20_000) == exp, per
    finally:
        oracle.set_block_cap(0)
        sim_engine.debug_set_block_cap(0)
        sim_engine.debug_set_batch_blocks(0)


def test_compress_stream_equals_whole(sim_engine, oracle):
    """Stream flavour (SURVEY 8f N2): chunks of every size, sources with read() / readByte, sinks with write() /
    writeByte / none -- always the bytes compressFile gives for the whole input."""
    import io
    rng = np.random.default_rng(3)
    data = (bytes(rng.integers(97, 123, 14000, dtype=np.uint8)) + bytes(3000) + b"ab" * 1500 +
            bytes(np.repeat(rng.integers(0, 4, 700, dtype=np.uint8), rng.choice([1, 2, 5, 300], 700))))

    class ByteSrc:
        def __init__(self, b):
            self.b, self.i = b, 0

        def readByte(self):
            self.i += 1
            return self.b[self.i - 1] if self.i <= len(self.b) else -1

    class ByteSink:
        def __init__(self):
            self.out = bytearray()

        def writeByte(self, b):
            self.out.append(b)

    try:
        for cap in (300, 4000):
            oracle.set_block_cap(cap)
            sim_engine.debug_set_block_cap(cap)
            exp = oracle.compress(data, 9)
            for chunk in (1000, 7777):
                assert sim_engine.compressStream(io.BytesIO(data), None, 9, chunk_bytes=chunk) == exp, (cap, chunk)
            sink = io.BytesIO()
            assert sim_engine.compressStream(ByteSrc(data), sink, 9, chunk_bytes=20000) is sink and sink.getvalue() == exp
            bs = ByteSink()
            sim_engine.compressStream(data, bs, 9, chunk_bytes=30000)
            assert bytes(bs.out) == exp
    finally:
        oracle.set_block_cap(0)
        sim_engine.debug_set_block_cap(0)
    for d in (b"", b"Q", b"aaaa", b"This is a test\n"):
        assert sim_engine.compressStream(io.BytesIO(d), None, 1, chunk_bytes=5) == oracle.compress(d, 1)
    with pytest.raises(ValueError, match="Invalid block size multiplier"):
        sim_engine.compressStream(io.BytesIO(b"x"), None, 10)


def test_decode_fixtures_and_random_access(sim_engine):
    for n in (0, 3):
        assert sim_engine.decompressFile(fixture_bytes(f"sample{n}.bz2")) == fixture_bytes(f"sample{n}.ref")
    s2 = fixture_bytes("sample2.bz2")
    rows = []
    sim_engine.table(s2, lambda p, s: rows.append(f"{p}\t{s}\n"))
    assert "".join(rows) == fixture_bytes("sample2.bzt").decode()
    assert sim_engine.decompressBlock(s2, 544888) == fixture_bytes("sample2.544888")


def test_decode_many_blocks(sim_engine, oracle):
    """Hundreds of small blocks in one stream (groups shorter and longer than one parse step)."""
    rng = np.random.default_rng(4)
    data = bytes(rng.integers(97, 123, 60_000, dtype=np.uint8)) + fixture_bytes("sample1.ref")[:30_000]
    try:
        oracle.set_block_cap(250)
        comp = oracle.compress(data, 9)
    finally:
        oracle.set_block_cap(0)
    assert sim_engine.decompressFile(comp) == data


def test_decode_periodic_and_runs(sim_engine, oracle):
    rng = np.random.default_rng(2)
    cases = [b"abab" * 10, b"aaaab" * 50, bytes(5000), b"abc" * 700,
             bytes(np.repeat(rng.integers(0, 3, 400, dtype=np.uint8), rng.integers(1, 12, 400))),
             _runny(rng, 4000, 2, 0.5)]
    for data in cases:
        assert sim_engine.decompressFile(oracle.compress(data, 9)) == data


def test_decode_errors_match_oracle(sim_engine, oracle):
    from compressjs_flattened_b200.bzip2 import Bzip2Error
    good = oracle.compress(b"hello world, hello world")
    flipped = bytearray(good)
    flipped[20] ^= 0x10
    bad_crc = bytearray(good)
    bad_crc[-1] ^= 0x01
    for blob in (b"", b"BZ", b"BZh0xxxx", b"XXXXXXXX", good[:-3], good[:20], bytes(flipped), bytes(bad_crc)):
        try:
            exp = ("ok", oracle.decompress(blob))
        except oracle.OracleError as e:
            exp = ("err", e.errorCode)
        try:
            got = ("ok", sim_engine.decompressFile(blob))
        except Bzip2Error as e:
            got = ("err", e.errorCode)
        assert got == exp


def test_multistream(sim_engine, oracle):
    ms = oracle.compress(b"first stream ") + oracle.compress(b"second stream", 1)
    assert sim_engine.decompressFile(ms, None, True) == b"first stream second stream" == oracle.decompress(ms, True)
    assert sim_engine.decompressFile(ms) == b"first stream "


def test_api_mirror_coercions(sim_engine):
    """Same argument coercions as Util.coerceInputStream/OutputStream (BJ:178-272)."""
    data = b"This is a test\n"

    class Src:
        def __init__(self, b):
            self.b, self.i = b, 0

        def readByte(self):
            if self.i >= len(self.b):
                return -1
            self.i += 1
            return self.b[self.i - 1]

    class Sink:
        def __init__(self):
            self.out, self.flushed = bytearray(), False

        def writeByte(self, b):
            self.out.append(b)

        def flush(self):
            self.flushed = True

    ref = sim_engine.compressFile(data)
    assert sim_engine.compressFile(list(data)) == ref == sim_engine.compressFile(Src(data)) == sim_engine.compressFile(np.frombuffer(data, np.uint8))
    assert sim_engine.compressFile(data, None, "not a number") == ref  # non-number props -> level 9 (BJ:2204)
    sink = Sink()
    assert sim_engine.compressFile(data, sink) is sink and bytes(sink.out) == ref and sink.flushed
    assert sim_engine.decompressFile(ref, len(data)) == data
    with pytest.raises(TypeError, match="outputsize does not match decoded input"):
        sim_engine.decompressFile(ref, len(data) + 1)
    buf = bytearray(len(data))
    assert sim_engine.decompressFile(ref, buf) is buf and bytes(buf) == data
    for bad in (0, 10, -1, 2.5):
        with pytest.raises(ValueError, match="Invalid block size multiplier"):
            sim_engine.compressFile(data, None, bad)


def _decode_outcome(engine_or_oracle, blob, err_type):
    try:
        if hasattr(engine_or_oracle, "decompressFile"):
            return ("ok", engine_or_oracle.decompressFile(blob))
        return ("ok", engine_or_oracle.decompress(blob))
    except err_type as e:
        return ("err", e.errorCode)


def _selector_region(blob):
    """Bit range [start, start + 8 * bits) of the selector list of the first block (SURVEY appendix A layout)."""
    bits = int.from_bytes(blob[:64], "big")
    total = 64 * 8
    used_map = (bits >> (total - (32 + 48 + 32 + 1 + 24) - 16)) & 0xFFFF
    k = bin(used_map).count("1")
    return 32 + 48 + 32 + 1 + 24 + 16 + 16 * k + 3 + 15


@pytest.mark.parametrize("parse_mode", ["1", "2"])
def test_decode_header_mutations_match_oracle(oracle, parse_mode, monkeypatch):
    """Both parse kernels against the oracle on streams whose selector list / code lengths / first symbols are damaged
    (runs of 1 bits longer than nGroups, the j == nGroups quirk of BJ:1488-1490, shifted lists, truncation)."""
    from compressjs_flattened_b200 import _native
    from compressjs_flattened_b200.bzip2 import Bzip2Engine, Bzip2Error
    from compressjs_flattened_b200.corpus import gen_text
    monkeypatch.setenv("BZ2B200_PARSE", parse_mode)
    eng = Bzip2Engine(0, _native.Library(os.path.join(os.path.dirname(__file__), "sim", "libbz2b200_sim.so")))
    rng = np.random.default_rng(11)
    good = oracle.compress(gen_text(40_000, 5).tobytes(), 9)
    assert eng.decompressFile(good) == oracle.decompress(good)
    s0 = _selector_region(good)
    cases = []
    for _ in range(24):  # single and double bit flips inside the selector list and the code lengths behind it
        b = bytearray(good)
        for pos in rng.integers(s0, s0 + 2500, rng.integers(1, 3)):
            b[pos >> 3] ^= 0x80 >> (pos & 7)
        cases.append(bytes(b))
    for _ in range(12):  # flips in the symbol data: other symbols, invalid codes, an early end-of-block
        b = bytearray(good)
        pos = int(rng.integers(8 * len(good) // 3, 8 * len(good) - 200))
        b[pos >> 3] ^= 0x80 >> (pos & 7)
        cases.append(bytes(b))
    for cut in (s0 // 8 + 3, s0 // 8 + 40, s0 // 8 + 200, len(good) - 9):
        cases.append(good[:cut])
    ones = bytearray(good)  # a run of 1 bits across a whole 32-bit word of the selector list
    for pos in range(s0 + 64, s0 + 64 + 70):
        ones[pos >> 3] |= 0x80 >> (pos & 7)
    cases.append(bytes(ones))
    for blob in cases:
        assert _decode_outcome(eng, blob, Bzip2Error) == _decode_outcome(oracle, blob, oracle.OracleError)
    # the same without the block CRC comparison on either side: what the damaged streams decode TO must agree as well
    eng.debug_set_ignore_block_crc(True)
    oracle.set_ignore_block_crc(True)
    try:
        outcomes = [_decode_outcome(oracle, blob, oracle.OracleError) for blob in cases]
        for blob, exp in zip(cases, outcomes):
            assert _decode_outcome(eng, blob, Bzip2Error) == exp
        assert sum(1 for o in outcomes if o[0] == "ok") >= 3 and sum(1 for o in outcomes if o[0] == "err") >= 3
    finally:
        oracle.set_ignore_block_crc(False)


def test_decode_many_selectors_multi_chunk(oracle, monkeypatch):
    """A block with ~5 000 selectors: the selector scan of the CTA parse kernel (256 threads = 8 192 bits per chunk) takes
    several chunks; both kernels must agree with the oracle, also when the list is damaged late."""
    from compressjs_flattened_b200 import _native
    from compressjs_flattened_b200.bzip2 import Bzip2Engine, Bzip2Error
    from compressjs_flattened_b200.corpus import gen_text
    data = gen_text(420_000, 6).tobytes()
    good = oracle.compress(data, 9)
    s0 = _selector_region(good)
    late = bytearray(good)
    late[(s0 + 9000) >> 3] ^= 0x10
    for mode in ("1", "2"):
        monkeypatch.setenv("BZ2B200_PARSE", mode)
        eng = Bzip2Engine(0, _native.Library(os.path.join(os.path.dirname(__file__), "sim", "libbz2b200_sim.so")))
        assert eng.decompressFile(good) == data
        assert _decode_outcome(eng, bytes(late), Bzip2Error) == _decode_outcome(oracle, bytes(late), oracle.OracleError)


class _BitW:
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, nbits, val):
        self.v = (self.v << nbits) | (val & ((1 << nbits) - 1))
        self.n += nbits

    def bytes(self):
        pad = -self.n % 8
        return ((self.v << pad).to_bytes((self.n + pad) // 8, "big"))


def crafted_run_overflow_stream(deep_total=1023, tail_literals=1000):
    """ADVICE r1 (high): a hand-built block whose RUNA/RUNB run lengths sum past 2^32.  Two used bytes (alphabet RUNA, RUNB,
    literal, end-of-block; two tables of 2-bit codes); two runs of 21 shallow RUNA digits followed by `deep` RUNB digits.
    With u32 sums and 0x400000 per deep digit (the round-1 kernel) the total wrapped to a small count that passed the dbuf
    check while per-symbol offsets ran to 4 GiB.  The reference rejects the first run at BJ:1647 (Data error)."""
    syms = []
    for deep in (deep_total // 2 + deep_total % 2, deep_total // 2):
        syms += [0] * 21 + [1] * deep + [2]
    syms += [2] * tail_literals + [3]
    w = _BitW()
    for ch in b"BZh9":
        w.put(8, ch)
    w.put(48, 0x314159265359)
    w.put(32, 0)                 # block CRC (never reached)
    w.put(1, 0)
    w.put(24, 5)                 # origPtr
    w.put(16, 0x8000)            # range 0 used
    w.put(16, 0xC000)            # bytes 0 and 1 used
    nsel = (len(syms) + 49) // 50
    w.put(3, 2)
    w.put(15, nsel)
    for _ in range(nsel):
        w.put(1, 0)              # selector MTF index 0
    for _ in range(2):           # two tables: every symbol 2 bits
        w.put(5, 2)
        for _ in range(4):
            w.put(1, 0)
    for s in syms:
        w.put(2, s)              # canonical codes of four 2-bit symbols: 00 01 10 11
    w.put(48, 0x177245385090)
    w.put(32, 0)
    wrapped = (2 * ((1 << 21) - 1) + deep_total * 0x400000 + 2 + tail_literals) % (1 << 32)
    return w.bytes(), wrapped


def test_decode_run_length_sum_cannot_wrap(sim_engine, oracle):
    from compressjs_flattened_b200.bzip2 import Bzip2Error
    blob, wrapped = crafted_run_overflow_stream()
    assert wrapped <= 900_000   # the old u32 sum would have passed the dbuf check
    assert _decode_outcome(oracle, blob, oracle.OracleError) == ("err", -5)
    assert _decode_outcome(sim_engine, blob, Bzip2Error) == ("err", -5)


def test_device_allocator_matches_reference_vectors(sim_engine, oracle):
    """the product's copy of the code-length allocator (huff.cuh ha_allocate) against NPM/test/huffman.js:16-76 directly,
    not only through whole-stream parity"""
    from test_oracle_golden import HUFF_VECTORS
    rng = np.random.default_rng(3)
    for freqs, limit, expect in HUFF_VECTORS:
        assert sim_engine.debug_huffman_lengths(freqs, limit) == list(expect)
    for _ in range(40):   # and against the oracle's copy on random histograms (limit 20 as in BJ:1342)
        n = int(rng.integers(3, 259))
        f = sorted(int(x) for x in rng.integers(0, 1 << int(rng.integers(1, 20)), n))
        assert sim_engine.debug_huffman_lengths(f, 20) == oracle.huff_alloc(f, 20)


def test_stream_objects_feed_and_finish(sim_engine, oracle):
    """csrc/stream_abi.inl: zstream == compressFile on the concatenation for any piece / chunk size (incl. blocks that need
    more than a chunk of input), dstream == decompressFile with the stream arriving in crumbs; multistream; errors"""
    import io
    from compressjs_flattened_b200.bzip2 import Bzip2Error
    rng = np.random.default_rng(17)
    from compressjs_flattened_b200.corpus import gen_text
    text = gen_text(40_000, 2).tobytes()
    runny = _runny(rng, 20_000, 3, 0.6)
    sim_engine.debug_set_block_cap(901)
    oracle.set_block_cap(901)
    try:
        for data in (text[:25_000], runny[:15_000], b"", b"q" * 7000):
            exp = oracle.compress(data, 9)
            for chunk, piece in ((4000, 1000), (1500, 7), (100_000, 100_000)):
                assert sim_engine.compressStream(io.BytesIO(data), None, 9, chunk_bytes=chunk, piece_bytes=piece) == exp, (len(data), chunk, piece)
            for chunk, piece in ((3000, 800), (200, 13), (1 << 20, 1 << 20)):
                assert sim_engine.decompressStream(io.BytesIO(exp), None, False, chunk_bytes=chunk, piece_bytes=piece) == data
        ms = oracle.compress(text, 9) + oracle.compress(runny, 9) + oracle.compress(b"end")
        assert sim_engine.decompressStream(io.BytesIO(ms), None, True, chunk_bytes=2500, piece_bytes=999) == text + runny + b"end"
        assert sim_engine.decompressStream(io.BytesIO(ms), None, False, chunk_bytes=2500, piece_bytes=999) == text
        good = oracle.compress(text, 9)
        bad = bytearray(good)
        bad[len(good) * 2 // 3] ^= 0x22
        sink = io.BytesIO()
        with pytest.raises(Bzip2Error) as e:
            sim_engine.decompressStream(io.BytesIO(bytes(bad)), sink, False, chunk_bytes=2000, piece_bytes=500)
        assert e.value.errorCode == -5 and 0 < len(sink.getvalue()) < len(text) and text.startswith(sink.getvalue())
        for blob in (good[:len(good) // 2], b"BZ", b"XYZW" + good[4:]):
            assert _decode_outcome(oracle, blob, oracle.OracleError)[0] == "err"
            with pytest.raises(Bzip2Error) as e:
                sim_engine.decompressStream(io.BytesIO(blob), None, False, chunk_bytes=1000, piece_bytes=300)
            assert ("err", e.value.errorCode) == _decode_outcome(oracle, blob, oracle.OracleError)
    finally:
        oracle.set_block_cap(0)
        sim_engine.debug_set_block_cap(0)


def test_command_line_like_the_reference(sim_engine, oracle, tmp_path, capsys):
    """NPM/bin/compressjs:7-58,163-180: -z is the default, level 7 by default, -d decodes the first stream only, -b extracts
    one block, the same complaints for contradictory flags"""
    from compressjs_flattened_b200.__main__ import main
    from compressjs_flattened_b200.corpus import gen_text
    data = gen_text(250_000, 12).tobytes()
    src, z7, z1, back, blk = (str(tmp_path / n) for n in ("in.txt", "z7.bz2", "z1.bz2", "back.txt", "blk.bin"))
    open(src, "wb").write(data)
    assert main([src, z7], engine=sim_engine) == 0 and open(z7, "rb").read() == oracle.compress(data, 7)
    assert main(["-z", "-1", src, z1], engine=sim_engine) == 0 and open(z1, "rb").read() == oracle.compress(data, 1)
    assert main(["-d", z1, back], engine=sim_engine) == 0 and open(back, "rb").read() == data
    two = str(tmp_path / "two.bz2")
    open(two, "wb").write(open(z1, "rb").read() + oracle.compress(b"second"))
    assert main(["-d", two, back], engine=sim_engine) == 0 and open(back, "rb").read() == data            # first stream only
    assert main(["-d", "--multistream", two, back], engine=sim_engine) == 0 and open(back, "rb").read() == data + b"second"
    pos, size = oracle.table(open(z1, "rb").read())[1]
    assert main(["-d", "-b", str(pos), z1, blk], engine=sim_engine) == 0
    assert open(blk, "rb").read() == oracle.decompress_block(open(z1, "rb").read(), pos) and len(open(blk, "rb").read()) == size
    assert main(["-d", "-z", src], engine=sim_engine) == 1
    assert main(["-z", "-b", "32", src], engine=sim_engine) == 1
    assert main(["-3", "-4", src], engine=sim_engine) == 1
    assert main(["-d", "-5", z1], engine=sim_engine) == 1
    assert main(["-t", "lzp3", src], engine=sim_engine) == 1
    err = capsys.readouterr().err
    assert "Must specify either -d or -z." in err and "--block can only be used with decompression" in err and "Can't specify both -3 and -4" in err


@pytest.mark.parametrize("parse_mode", ["1", "2"])
def test_decode_foreign_libbz2_streams(sim_engine, parse_mode, monkeypatch):
    """Streams made by libbz2 (Python's bz2: other table choices, code lengths up to 17, several streams back to back) on both
    parse kernels: what any encoder wrote must come back (SURVEY N3; the reference decodes foreign streams, BJ:1769-1796)."""
    import bz2
    from compressjs_flattened_b200 import _native
    from compressjs_flattened_b200.bzip2 import Bzip2Engine
    from compressjs_flattened_b200.corpus import gen_html, gen_text
    monkeypatch.setenv("BZ2B200_PARSE", parse_mode)
    eng = Bzip2Engine(0, _native.Library(os.path.join(os.path.dirname(__file__), "sim", "libbz2b200_sim.so")))
    rng = np.random.default_rng(3)
    skew = rng.choice(256, 50_000, p=np.arange(1, 257)[::-1] ** 3.0 / (np.arange(1, 257) ** 3.0).sum()).astype(np.uint8).tobytes()
    cases = [gen_text(70_000, 2).tobytes(), gen_html(40_000, 3).tobytes(), skew, bytes(30_000), b"a", b""]
    for data in cases:
        for level in (1, 9):
            assert eng.decompressFile(bz2.compress(data, level)) == data
    two = bz2.compress(cases[0][:20_000], 5) + bz2.compress(cases[2][:9_000], 2)
    assert eng.decompressFile(two, None, True) == cases[0][:20_000] + cases[2][:9_000]
    assert eng.decompressFile(two) == cases[0][:20_000]          # the reference stops after the first stream (multistream off)
