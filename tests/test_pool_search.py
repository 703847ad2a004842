"""Fixed-string search of ONE stream over the lanes of a pool: Bzip2Pool.search / bz2b200_pool_search (include/bz2b200.h).

Every result is compared field for field with Bzip2Engine.search on one context and with the Python model of
test_search.py.  The streams are cut into small blocks, and the slices are forced down to a few hundred bytes of stream
(smaller than a block, so that every block boundary is a slice boundary and some slices own no block), so that matches,
newlines and lines meet the slice boundaries the cases aim at; each case asserts that it reaches them.  On the simulator
every case runs on two pools, with both parse kernels and with 256-byte and default search tiles; on the GPU (-m gpu) on
two lanes of one device and on two devices when two are visible, then at full size: the 100 MB bench stream and a
50 MB line."""
import bz2
import ctypes as C

import numpy as np
import pytest

from compressjs_flattened_b200 import _native
from compressjs_flattened_b200.bzip2 import MATCH_FIRST_IN_LINE, Bzip2Engine
from compressjs_flattened_b200.corpus import gen_text
from compressjs_flattened_b200.pool import Bzip2Pool
from test_recover import damage_field, make
from test_search import RARE, SIM_SO, WORDS16, bench_stream, err_code, model  # noqa: F401  (bench_stream: a fixture)

SLICES = (0, 150, 400, 1500)   # bytes of stream per slice; 0 = as decompressFile picks them
TILES = (256, 0)


def _ngpu():
    import torch
    return torch.cuda.device_count()


POOLS = [pytest.param(("sim", (0, 0), 2, "1"), id="sim-2x2-parse1"), pytest.param(("sim", (0, 0), 2, "2"), id="sim-2x2-parse2"),
         pytest.param(("sim", (0,), 3, "1"), id="sim-1x3-parse1"), pytest.param(("sim", (0,), 3, "2"), id="sim-1x3-parse2"),
         pytest.param(("gpu", (0,), 2, ""), id="gpu-1x2", marks=pytest.mark.gpu),
         pytest.param(("gpu", (0, 1), 2, ""), id="gpu-2x2", marks=pytest.mark.gpu)]


@pytest.fixture(params=POOLS)
def pe(request, monkeypatch):
    """(pool, engine on one context) over the same library"""
    where, devices, lanes, parse = request.param
    if parse:
        monkeypatch.setenv("BZ2B200_PARSE", parse)   # read when a context is created
    if where == "sim":
        request.getfixturevalue("sim_engine")         # builds the simulator library when it is stale
        lib = _native.Library(SIM_SO)
    else:
        if len(devices) > _ngpu():
            pytest.skip(f"needs {len(devices)} GPUs")
        lib = None
    pool, eng = Bzip2Pool(list(devices), lanes, library=lib), Bzip2Engine(0, lib)
    yield pool, eng
    pool.close()
    eng.close()


def slice_starts(oracle, comp, sb, multistream=False):
    """output offsets at which the slices of `sb` bytes of stream start (0 excluded; a slice that owns no block repeats
    the offset of the next one): a slice owns the blocks whose signature starts in it"""
    if sb == 0:
        return []
    pos = oracle.table(comp, multistream)
    out, starts = 0, []
    k = 0
    for j in range(1, (len(comp) + sb - 1) // sb):
        while k < len(pos) and pos[k][0] < 8 * j * sb:
            out += pos[k][1]
            k += 1
        starts.append(out)
    return starts


def slice_sizes(oracle, comp, sb, total, multistream=False):
    s = [0] + slice_starts(oracle, comp, sb, multistream) + [total]
    return [b - a for a, b in zip(s, s[1:])]


def check(pe, comp, data, patterns, ignore_case=False, max_matches=None, multistream=False, slices=SLICES, tiles=TILES):
    """pool search with every slice size and tile size == one context == the model; returns {slice_bytes: result}"""
    pool, eng = pe
    want, total, lines, text = model(data, patterns, ignore_case, max_matches)
    out = {}
    for tile in tiles:
        pool.debug_set_search_tile(tile)
        eng.debug_set_search_tile(tile)
        try:
            one = eng.search(comp, patterns, ignore_case, max_matches, multistream, lines=True)
            n_blocks = eng.stats().n_blocks
            for sb in slices:
                r = pool.search(comp, patterns, ignore_case, max_matches, multistream, lines=True, slice_bytes=sb)
                assert (r.total_matches, r.total_lines, r.out_bytes) == (total, lines, len(data)), (tile, sb)
                assert np.array_equal(r.matches, want), (tile, sb)
                assert r.lines == text, (tile, sb)
                assert np.array_equal(r.matches, one.matches) and r.lines == one.lines
                assert (r.total_matches, r.total_lines, r.out_bytes) == (one.total_matches, one.total_lines, one.out_bytes)
                st = pool.stats()
                assert (st.in_bytes, st.out_bytes, st.n_blocks) == (len(comp), len(data), n_blocks)
                out[sb] = r
        finally:
            pool.debug_set_search_tile(0)
            eng.debug_set_search_tile(0)
    return out


def blocky(oracle, data, cap=300):
    """a stream of blocks of `cap` bytes and the output offsets where its blocks start (0 excluded); blocks of 300 bytes
    of text take 194 bytes of stream and more, so that at 150 bytes every block boundary is a slice boundary"""
    comp, _ = make(oracle, data, cap)
    sizes = [s for _, s in oracle.table(comp)]
    return comp, np.cumsum(sizes).tolist()[:-1]


def text_without_runs(n, seed):
    """text in which no byte repeats 4 times in a row: block sizes then depend on the block cap only"""
    t = bytearray(gen_text(n, seed).tobytes())
    for i in range(3, len(t)):
        if t[i] == t[i - 1] == t[i - 2] == t[i - 3]:
            t[i] = ord("x") if t[i] != ord("x") else ord("y")
    return t


def spans(r, L, cuts):
    """cuts c that some match of length L crosses (starts before c, ends after it)"""
    off = r.matches["offset"].astype(np.int64)
    return [c for c in cuts if ((off < c) & (off + L > c)).any()]


# ---- matches across slices ----
def test_matches_across_slices(pe, oracle):
    data = bytes(text_without_runs(6000, 61))
    comp, cuts = blocky(oracle, data, 100)            # blocks of 100 bytes, 86 bytes of stream and more: a slice of 60 owns one or none
    sizes = slice_sizes(oracle, comp, 60, len(data))
    assert 0 in sizes and any(0 < s < 255 for s in sizes)
    pats = [data[c - 3:c + 4] for c in cuts[5:40:6]] + [data[cuts[20] - 10:cuts[20] + 246], data[cuts[30] - 1:cuts[30] + 1]]
    res = check(pe, comp, data, pats, slices=(0, 60, 150, 1500))
    starts = slice_starts(oracle, comp, 60)
    assert len(spans(res[60], 7, starts)) >= 5                         # a 7-byte match crosses a slice boundary
    s0 = next(s for s in starts if s > cuts[20] - 10)
    inside = [b - a for a, b in zip(starts, starts[1:]) if a >= s0 and b <= cuts[20] + 246 and b > a]
    assert inside and min(inside) < 255                                 # the 256-byte match crosses a slice of < 255 bytes


def test_boundaries_at_newline_and_at_match_edges(pe, oracle):
    t = text_without_runs(9000, 62)
    comp0, cuts = blocky(oracle, bytes(t), 300)
    assert len(cuts) >= 25
    at_nl, after_nl, before_m, after_m, mid = cuts[2:6], cuts[7:11], cuts[12:16], cuts[17:21], cuts[22:25]
    for c in at_nl:
        t[c] = 10                                        # the slice starts on a '\n'
    for c in after_nl:
        t[c - 1] = 10                                    # the slice starts just after one
    for c in before_m:
        t[c - 3:c] = b"QZK"                              # a match ends just before the slice
    for c in after_m:
        t[c:c + 3] = b"QZK"                              # a match starts at the slice's first byte
    data = bytes(t)
    comp, cuts2 = blocky(oracle, data, 300)
    assert cuts2 == cuts
    pats = [b"QZK", b"\n", b"K\n", data[mid[0] - 128:mid[0] + 128], data[mid[1] - 255:mid[1] + 1], data[mid[2] - 1:mid[2] + 255]]
    res = check(pe, comp, data, pats)
    starts = set(slice_starts(oracle, comp, 150))
    assert set(cuts) <= starts                           # every block boundary is a slice boundary at 150 bytes
    off = set(res[150].matches["offset"].tolist())
    assert all(c in off for c in at_nl + after_m) and all(c - 3 in off for c in before_m) and all(c - 1 in off for c in after_nl)
    assert mid[0] in set(spans(res[150], 256, cuts))


# ---- lines ----
@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_line_across_many_slices(pe, oracle, where):
    long_line = bytes(text_without_runs(2400, 63)).replace(b"\n", b" ")
    at = {"first": 100, "middle": 1200, "last": 2300}[where]
    long_line = long_line[:at] + b"NEEDLE" + long_line[at + 6:]
    data = b"a b\nNEEDLE one\n" + long_line + b"\nlast NEEDLE line\nend"
    comp, cuts = blocky(oracle, data, 300)
    res = check(pe, comp, data, [b"NEEDLE"])
    lo, hi = data.index(long_line), data.index(long_line) + len(long_line)
    starts = slice_starts(oracle, comp, 150)
    assert len([s for s in starts if lo < s < hi]) >= 3                 # the line spans three slices and more
    m = res[150].matches
    assert len(m) == 3 and m["offset"][1] == lo + at and m["line_begin"][1] == lo and m["line_end"][1] == hi
    assert long_line + b"\n" in res[150].lines


def test_second_match_of_a_line_in_a_later_slice(pe, oracle):
    long_line = bytes(text_without_runs(2000, 64)).replace(b"\n", b" ")
    long_line = long_line[:50] + b"NEEDLE" + long_line[56:1500] + b"NEEDLE" + long_line[1506:]
    data = b"head\n" + long_line + b"\ntail\n"
    comp, cuts = blocky(oracle, data, 300)
    res = check(pe, comp, data, [b"NEEDLE", b"tail"])
    m = res[150].matches
    assert m["flags"].tolist() == [MATCH_FIRST_IN_LINE, 0, MATCH_FIRST_IN_LINE]
    starts = slice_starts(oracle, comp, 150)
    assert any(m["offset"][0] < s <= m["offset"][1] for s in starts)   # the second match is in a later slice


# ---- counts and truncation ----
def test_max_matches(pe, oracle):
    data = bytes(text_without_runs(5000, 65))
    comp, cuts = blocky(oracle, data, 300)
    pats = [b"e", b"th"]
    want = model(data, pats)[0]
    off = want["offset"].astype(np.int64)
    starts = slice_starts(oracle, comp, 150)
    at_cut = int((off < starts[len(starts) // 2]).sum())    # the last returned match is the last of a slice
    assert 0 < at_cut < len(want) and off[at_cut] >= starts[len(starts) // 2] > off[at_cut - 1]
    inside = at_cut + 3                                     # ... and cut inside the next slice
    for mm in (0, 1, inside, at_cut, len(want) - 1, None):
        res = check(pe, comp, data, pats, max_matches=mm, slices=(0, 150), tiles=(256,))
        assert len(res[150].matches) == (len(want) if mm is None else mm)
    r = pe[0].search(comp, pats, max_matches=0)
    assert len(r.matches) == 0 and r.lines is None and r.total_matches == len(want)


def test_ignore_case_one_byte_and_newline_patterns(pe, oracle):
    data = bytes(text_without_runs(4000, 66)).replace(b"the", b"THE", 20)
    comp, _ = blocky(oracle, data, 300)
    pats = [b"The", b"e", b"\n", b".\nT", b"x", b"\n<"]
    check(pe, comp, data, pats, ignore_case=True)
    check(pe, comp, data, pats, ignore_case=False, tiles=(256,))


# ---- shapes of the output ----
def test_no_newline_last_line_empty_and_multistream(pe, oracle):
    flat = bytes(text_without_runs(3000, 67)).replace(b"\n", b" ") + b" tail"
    comp, _ = blocky(oracle, flat, 300)
    res = check(pe, comp, flat, [b"the", b"tail"])
    assert res[150].lines == flat + b"\n" and res[150].total_lines == 1
    last = b"first\n" + flat
    comp, _ = blocky(oracle, last, 300)
    assert check(pe, comp, last, [b"tail", b"first"], slices=(0, 150))[150].lines == last + b"\n"
    empty = oracle.compress(b"", 9)
    assert check(pe, empty, b"", [b"a", b"ab"], slices=(0, 150))[0].out_bytes == 0
    parts = [make(oracle, gen_text(2_000, 68).tobytes(), 400, 1)[0], make(oracle, gen_text(2_500, 69).tobytes(), 300, 5)[0],
             bz2.compress(gen_text(1_500, 70).tobytes(), 1)]
    blob = b"".join(parts)
    full = oracle.decompress(blob, True)
    cuts = np.cumsum([s for _, s in oracle.table(blob, True)]).tolist()[:-1]
    pats = [full[c - 3:c + 4] for c in cuts] + [b"the"]
    res = check(pe, blob, full, pats, multistream=True)
    assert len(spans(res[150], 7, slice_starts(oracle, blob, 150, True))) >= 5
    check(pe, blob, oracle.decompress(parts[0]), pats[:4], multistream=False, slices=(0, 150))


# ---- errors ----
def test_damaged_streams_give_decoder_codes(pe, oracle):
    pool, eng = pe
    src = gen_text(12_000, 71).tobytes()
    comp, pos = make(oracle, src, 1500)
    rng = np.random.default_rng(72)
    cases = [damage_field(oracle, comp, pos, 3, "crc", rng), damage_field(oracle, comp, pos, 5, "sel", rng), comp[:len(comp) // 2], comp[:3],
             b"BZh0" + comp[4:], comp[:-2]]
    for d in cases:
        code = err_code(lambda: eng.search(d, [b"the"], lines=True))
        assert code != 0
        for sb in (0, 150, 700):
            assert err_code(lambda: pool.decompressFile(d, None, False, sb)) == code
            assert err_code(lambda: pool.search(d, [b"the"], lines=True, slice_bytes=sb)) == code


def pool_c_search(pool, comp, packed, lens, flags=0, max_matches=10):
    """bz2b200_pool_search called directly: the return code"""
    a = np.frombuffer(comp, dtype=np.uint8)
    pats = np.frombuffer(packed, dtype=np.uint8) if packed else np.zeros(1, dtype=np.uint8)
    ln = np.array(lens, dtype=np.uint32) if len(lens) else np.zeros(1, dtype=np.uint32)
    mp, nm, tot = C.POINTER(_native.Match)(), C.c_size_t(), _native.SearchTotals()
    rc = pool._L.bz2b200_pool_search(pool._p, a.ctypes.data, a.size, 0, pats.ctypes.data, ln.ctypes.data, len(lens), flags, max_matches, 0,
                                     C.byref(mp), C.byref(nm), C.byref(tot), None, None)
    if rc == 0:
        pool._L.bz2b200_free(mp)
    return rc


def test_bad_arguments_same_code_and_text(pe, oracle):
    from test_search import c_search
    pool, eng = pe
    comp = oracle.compress(gen_text(3000, 73).tobytes(), 9)
    assert pool_c_search(pool, comp, b"ab", [2]) == 0
    for packed, lens, flags in ((b"", [], 0), (b"a" * 257, [1] * 257, 0), (b"ab", [0, 2], 0), (b"a" * 257, [257], 0), (b"ab", [2], 2)):
        assert pool_c_search(pool, comp, packed, lens, flags) == c_search(eng, comp, packed, lens, flags) == _native.E_ARG
        assert pool._L.bz2b200_pool_last_error(pool._p) == eng._L.bz2b200_last_error(eng._ctx) != b""
    for pats in ([], [b""], [b"a"] * 257, [b"a" * 257], [b"ok", b""]):
        with pytest.raises(ValueError):
            pool.search(comp, pats)
    with pytest.raises(ValueError):
        pool.search(comp, b"a", max_matches=-1)
    with pytest.raises(RuntimeError):
        pool.debug_set_search_tile(100)


# ---- GPU only: sizes a user searches ----
def _gpu_pools():
    pools = [Bzip2Pool([0], 2)]
    if _ngpu() >= 2:
        pools.append(Bzip2Pool(list(range(_ngpu())), 2))
    return pools


def _full_check(eng, pools, comp, data, pats, ignore_case=False, max_matches=None, lines=False, slices=(0,)):
    want, total, nlines, text = model(data, pats, ignore_case, max_matches)
    one = eng.search(comp, pats, ignore_case, max_matches, False, lines)
    assert np.array_equal(one.matches, want) and (one.total_matches, one.total_lines) == (total, nlines)
    for pool in pools:
        for sb in slices:
            r = pool.search(comp, pats, ignore_case, max_matches, False, lines, slice_bytes=sb)
            assert np.array_equal(r.matches, want), sb
            assert (r.total_matches, r.total_lines, r.out_bytes) == (total, nlines, len(data)), sb
            assert r.lines == (text if lines else None), sb


@pytest.mark.gpu
def test_bench_stream_on_pools(gpu_engine, bench_stream):
    comp, full = bench_stream
    pools = _gpu_pools()
    try:
        _full_check(gpu_engine, pools, comp, full, [RARE], lines=True, slices=(0, 3_000_000))
        _full_check(gpu_engine, pools, comp, full, WORDS16, lines=True, slices=(0, 5_000_000))
        words = sorted({w for w in full[:2_000_000].split() if 6 <= len(w) <= 12 and w.isalpha()})[:256]
        assert len(words) == 256
        _full_check(gpu_engine, pools, comp, full, words, ignore_case=True, max_matches=2_000_000, lines=True, slices=(0,))
    finally:
        for p in pools:
            p.close()


@pytest.mark.gpu
def test_fifty_megabyte_line_on_pools(gpu_engine):
    body = gen_text(50_000_000, 52).tobytes().replace(b"\n", b" ")
    data = b"head\n" + body[:20_000_000] + b" NEEDLE " + body[20_000_000:] + b"tail\nafter"
    comp = gpu_engine.compressFile(data, None, 9)
    pools = _gpu_pools()
    try:
        _full_check(gpu_engine, pools, comp, data, [b"NEEDLE"], lines=True, slices=(0, 2_000_000))
        _full_check(gpu_engine, pools, comp, data, [b"head", b"tail", b"Paris"], lines=True, slices=(0, 2_000_000))
        r = pools[0].search(comp, [b"NEEDLE"], lines=True, slice_bytes=2_000_000)
        assert len(r.lines) >= 50_000_000 and len(comp) // 2_000_000 >= 5   # the line crosses several slices
    finally:
        for p in pools:
            p.close()
