"""Fixed-string search of the decompressed output: Bzip2Engine.search, bz2b200_search (include/bz2b200.h) and the --grep
command line.

Expected values come only from the oracle's (or libbz2's) decoded bytes and the Python model below: every occurrence by
bytes.find stepping one byte at a time, case folded with bytes.lower(), the line fields from the positions of '\\n', the
lines from data.split(b"\\n").  Every case runs on the simulator (both parse kernels) and on the GPU (-m gpu, both parse
kernels), each with 256-byte search tiles (so that a few KB of output spans many tiles) and with the default tiles; the
100 MB bench stream, 10^7 matches and a 50 MB line run on the GPU only."""
import bz2
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from compressjs_flattened_b200 import _native
from compressjs_flattened_b200.bzip2 import MATCH_DTYPE, MATCH_FIRST_IN_LINE, Bzip2Engine, Bzip2Error, Err
from compressjs_flattened_b200.corpus import gen_text
from test_recover import damage_field, make

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_SO = os.environ.get("BZ2B200_SIM_LIB") or os.path.join(HERE, "sim", "libbz2b200_sim.so")

ENGINES = [pytest.param(("sim", "1"), id="sim-parse1"), pytest.param(("sim", "2"), id="sim-parse2"),
           pytest.param(("gpu", "1"), id="gpu-parse1", marks=pytest.mark.gpu),
           pytest.param(("gpu", "2"), id="gpu-parse2", marks=pytest.mark.gpu)]
TILES = (256, 0)   # bytes per search tile; 0 = the default
# words of the bench text (gen_text(100 MB, seed 8)): one that is rare there, and 16 of every frequency
RARE = b"hbfiednrewd"
WORDS16 = [b"the", b"of", b"and", b"dtzat", b"tenwntne", b"ntbpsdlon", b"luooler", b"dveutseu", b"trocftecsa", b"tnnef", b"dlitcnm",
           b"qsmilplhnt", b"cihoes", b"<title>", b"[[", RARE]


@pytest.fixture(params=ENGINES)
def eng(request, monkeypatch):
    where, mode = request.param
    monkeypatch.setenv("BZ2B200_PARSE", mode)   # read when the context is created
    if where == "sim":
        request.getfixturevalue("sim_engine")   # builds the simulator library when it is stale
        e = Bzip2Engine(0, _native.Library(SIM_SO))
    else:
        e = Bzip2Engine(0)
    yield e
    e.close()


# ---- the model ----
def model(data, patterns, ignore_case=False, max_matches=None):
    """(matches as a MATCH_DTYPE array, total matches, total lines, expected lines) of searching `data`"""
    d = data.lower() if ignore_case else data
    found = []
    for j, p in enumerate(patterns):
        q = p.lower() if ignore_case else p
        i = d.find(q)
        while i >= 0:
            found.append((i, j))
            i = d.find(q, i + 1)
    found.sort()
    off = np.array([o for o, _ in found], dtype=np.int64)
    nl = np.flatnonzero(np.frombuffer(data, dtype=np.uint8) == 10)
    line = np.searchsorted(nl, off, side="left")                     # '\n' bytes before the offset
    begin = np.where(line > 0, nl[np.maximum(line - 1, 0)] + 1 if len(nl) else 0, 0)
    end = np.where(line < len(nl), nl[np.minimum(line, max(len(nl) - 1, 0))] if len(nl) else len(data), len(data))
    first = np.ones(len(found), dtype=bool)
    first[1:] = line[1:] != line[:-1]
    m = np.zeros(len(found), dtype=MATCH_DTYPE)
    m["offset"], m["line"], m["line_begin"], m["line_end"] = off, line, begin, end
    m["pattern"] = [j for _, j in found]
    m["flags"] = np.where(first, MATCH_FIRST_IN_LINE, 0)
    k = len(found) if max_matches is None else min(max_matches, len(found))
    rows = data.split(b"\n")
    text = b"".join(rows[i] + b"\n" for i in line[:k][first[:k]].tolist())
    return m[:k], len(found), int(first.sum()), text


def check(eng, comp, data, patterns, ignore_case=False, max_matches=None, multistream=False, tiles=TILES):
    """search `comp` with every tile size and compare everything with the model of `data`; returns the result"""
    want, total, lines, text = model(data, patterns, ignore_case, max_matches)
    for tile in tiles:
        eng.debug_set_search_tile(tile)
        try:
            r = eng.search(comp, patterns, ignore_case, max_matches, multistream, lines=True)
        finally:
            eng.debug_set_search_tile(0)
        assert r.matches.dtype == MATCH_DTYPE
        assert (r.total_matches, r.total_lines, r.out_bytes) == (total, lines, len(data)), tile
        assert np.array_equal(r.matches, want), tile
        assert r.lines == text, tile
        st = eng.stats()
        assert st.out_bytes == len(data) and st.in_bytes == len(comp)
    return r


def c_search(eng, comp, packed, lens, flags=0, max_matches=10):
    """bz2b200_search called directly: the return code"""
    a = np.frombuffer(comp, dtype=np.uint8)
    pats = np.frombuffer(packed, dtype=np.uint8) if packed else np.zeros(1, dtype=np.uint8)
    ln = np.array(lens, dtype=np.uint32) if len(lens) else np.zeros(1, dtype=np.uint32)
    mp, nm, tot = C.POINTER(_native.Match)(), C.c_size_t(), _native.SearchTotals()
    rc = eng._L.bz2b200_search(eng._ctx, a.ctypes.data, a.size, 0, pats.ctypes.data, ln.ctypes.data, len(lens), flags, max_matches,
                               C.byref(mp), C.byref(nm), C.byref(tot), None, None)
    if rc == 0:
        eng._L.bz2b200_free(mp)
    return rc


def err_code(fn):
    try:
        fn()
    except Bzip2Error as e:
        return e.errorCode
    return 0


@pytest.fixture(scope="module")
def text(oracle):
    data = gen_text(12_000, 41).tobytes()
    return oracle.compress(data, 9), data


# ---- match positions ----
def test_first_and_last_byte_and_tile_ends(eng, oracle):
    body = bytearray(gen_text(6_000, 42).tobytes().replace(b"Q", b"q"))
    for k in range(1, 20):   # "QQQQQ" across every 256-byte tile end, a 256-byte pattern across one
        body[256 * k - 3:256 * k + 2] = b"QQQQQ"
    data = b"Qstart" + bytes(body) + b"the end Qstart"
    comp = oracle.compress(data, 9)
    check(eng, comp, data, [b"Qstart", b"QQQQQ", b"QQ", data[1800:2056], b"Q"])
    check(eng, comp, data, [data[-1:], data[:1], data[-256:], data[:256]])


def test_block_and_stream_boundaries(eng, oracle):
    parts = [make(oracle, gen_text(7_000, 43).tobytes(), 997, 1)[0], make(oracle, gen_text(9_000, 44).tobytes(), 2500, 5)[0],
             make(oracle, gen_text(6_000, 45).tobytes(), 1800, 9)[0], bz2.compress(gen_text(5_000, 46).tobytes(), 1)]
    blob = b"".join(parts)
    full = oracle.decompress(blob, True)
    assert full[-5000:] == bz2.decompress(parts[-1])
    cuts = np.cumsum([s for _, s in oracle.table(blob, True)]).tolist()[:-1]
    assert len(cuts) > 12
    pats = [full[o - 3:o + 4] for o in cuts] + [full[o - 1:o + 1] for o in cuts[:5]]
    check(eng, blob, full, pats, multistream=True)
    first = oracle.decompress(parts[0])
    check(eng, blob, first, pats[:8], multistream=False)   # the first stream only


# ---- pattern sets ----
def test_overlaps_prefixes_duplicates_one_byte(eng, oracle):
    data = b"aaaa\nabcd abc ab a\nthe then thx th\n" * 40 + b"zz"
    comp = oracle.compress(data, 9)
    r = check(eng, comp, data, [b"aa"])
    assert r.matches["offset"][:3].tolist() == [0, 1, 2] and r.total_matches == 120
    check(eng, comp, data, [b"abcd", b"abc", b"ab", b"a"])              # prefixes of one another
    check(eng, comp, data, [b"ab", b"the", b"ab", b"z", b"z"])          # duplicates
    check(eng, comp, data, [b"a", b"\n", b" ", b"z"])                   # one byte
    check(eng, comp, data, [b"thx", b"then", b"th", b"the"])            # the same first two bytes


def test_newline_and_nul_in_patterns(eng, oracle):
    data = (b"x\0y\0\0z\nline\n\nend\0" * 30) + b"\0"
    comp = oracle.compress(data, 9)
    check(eng, comp, data, [b"\0", b"\0\0", b"\n\n", b"e\n\ne", b"\0x\0", b"\nline\n"])


def test_256_patterns_of_256_bytes(eng, oracle, text):
    comp, data = text
    rng = np.random.default_rng(47)
    pats = [data[s:s + 256] for s in rng.integers(0, len(data) - 256, 200).tolist()]
    pats += [pats[0][:255] + bytes([b]) for b in range(56)]   # the same 255 bytes, then 56 different last bytes
    assert len(pats) == 256 and all(len(p) == 256 for p in pats)
    r = check(eng, comp, data, pats, tiles=(256,))
    assert r.total_matches >= 200


def test_ignore_case_ascii_edges(eng, oracle):
    edges = b"@AZ[`az{"
    rng = np.random.default_rng(48)
    alphabet = np.frombuffer(edges + b"\x80\xc0\xc1\xda\xe0\xe1\xfa\xff\n ", dtype=np.uint8)
    data = rng.choice(alphabet, 6000).tobytes()
    comp = oracle.compress(data, 9)
    pats = [b"@", b"[", b"`", b"{", b"A", b"z", b"Z[", b"`a", b"@a", b"z{", b"\xc1", b"\xe1", b"\xc0a", b"Az", b"aZ"]
    check(eng, comp, data, pats, ignore_case=True)
    check(eng, comp, data, pats, ignore_case=False)
    r = eng.search(comp, [b"["], ignore_case=True)
    assert r.total_matches == data.count(b"[") and r.total_matches != data.count(b"[") + data.count(b"{")


# ---- lines ----
def test_lines_empty_last_long_and_many_matches(eng, oracle):
    long_line = b"needle " + gen_text(3000, 49).tobytes().replace(b"\n", b" ") + b" needle"
    data = b"\n\nneedle\n\n" + long_line + b"\nneedle needle needle\n\nlast needle"
    comp = oracle.compress(data, 9)
    r = check(eng, comp, data, [b"needle", b"e"])
    long_row = r.matches[r.matches["line"] == 4]
    assert long_row["line_begin"].tolist() == [10] * len(long_row) and long_row["line_end"][0] == 10 + len(long_line)
    assert int((long_row["flags"] != 0).sum()) == 1
    three = r.matches[(r.matches["line"] == 5) & (r.matches["pattern"] == 0)]
    assert len(three) == 3 and int((r.matches[r.matches["line"] == 5]["flags"] != 0).sum()) == 1
    assert r.lines.endswith(b"last needle\n") and r.matches["line_end"][-1] == len(data)
    check(eng, comp, data, [b"\n"])   # a match on every '\n', also of the empty lines


# ---- counts and truncation ----
def test_max_matches_and_totals(eng, text):
    comp, data = text
    pats = [b"e", b"the", b" "]
    total = model(data, pats)[1]
    for mm in (0, 1, 2, total - 1, total, total + 5):
        r = check(eng, comp, data, pats, max_matches=mm)
        assert len(r.matches) == min(mm, total) and r.total_matches == total
    r = eng.search(comp, pats, max_matches=0)
    assert len(r.matches) == 0 and r.lines is None and r.total_lines == model(data, pats)[2]


def test_no_match_and_empty_output(eng, oracle, text):
    comp, data = text
    r = check(eng, comp, data, [b"\xff\xfe", b"\x01"])
    assert r.total_matches == 0 and r.lines == b""
    empty = oracle.compress(b"", 9)
    r = check(eng, empty, b"", [b"a", b"ab"])
    assert (r.total_matches, r.out_bytes) == (0, 0)


# ---- errors ----
def test_limits_give_e_arg(eng, text):
    comp, _ = text
    assert c_search(eng, comp, b"ab", [2]) == 0
    for packed, lens, flags in ((b"", [], 0), (b"a" * 257, [1] * 257, 0), (b"ab", [0, 2], 0), (b"a" * 257, [257], 0), (b"ab", [2], 2)):
        assert c_search(eng, comp, packed, lens, flags) == _native.E_ARG
        assert eng._L.bz2b200_last_error(eng._ctx)
    assert c_search(eng, comp, b"a" * 256 * 256, [256] * 256) == 0
    for pats in ([], [b""], [b"a"] * 257, [b"a" * 257], [b"ok", b""]):
        with pytest.raises(ValueError):
            eng.search(comp, pats)
    with pytest.raises(ValueError):
        eng.search(comp, b"a", max_matches=-1)
    assert eng.search(comp, "the").total_matches == eng.search(comp, [b"the"]).total_matches   # a str is UTF-8


def test_damaged_streams_give_decompress_codes(eng, oracle):
    src = gen_text(24_000, 50).tobytes()
    comp, pos = make(oracle, src, 2500)
    rng = np.random.default_rng(51)
    cases = [damage_field(oracle, comp, pos, 3, "crc", rng), damage_field(oracle, comp, pos, 4, "sel", rng), comp[:len(comp) // 2], comp[:3],
             b"BZh0" + comp[4:], comp[:-2]]
    for d in cases:
        code = err_code(lambda: eng.decompressFile(d))
        assert code != 0
        assert err_code(lambda: eng.search(d, [b"the"], lines=True)) == code


# ---- the command line ----
def test_command_line_grep(sim_engine, oracle, tmp_path, capsys):
    from compressjs_flattened_b200.__main__ import main
    data = b"alpha Beta\ngamma\n\nBETA beta delta\nlast beta"
    src, out = tmp_path / "in.bz2", tmp_path / "out"
    src.write_bytes(oracle.compress(data, 9))
    assert main(["-d", "--grep", "beta", str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == b"BETA beta delta\nlast beta\n"
    assert main(["-d", "--grep", "beta", "--ignore-case", "--line-number", str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == b"1:alpha Beta\n4:BETA beta delta\n5:last beta\n"
    assert main(["--grep", "gamma", "--grep", "delta", "--line-number", str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == b"2:gamma\n4:BETA beta delta\n"
    assert main(["-d", "--grep", "a", "--count", str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == b"4\n"
    assert main(["-d", "--grep", "zeta", str(src), str(out)], engine=sim_engine) == 1
    assert out.read_bytes() == b""
    assert main(["-d", "--grep", "zeta", "--count", str(src), str(out)], engine=sim_engine) == 1
    assert out.read_bytes() == b"0\n"
    capsys.readouterr()
    for argv, msg in ((["-z", "--grep", "a"], "--grep can only be used without -z"), (["-d", "--grep", "a", "-b", "32"], "--grep and --block can't be used together"),
                      (["--grep", "a", "--recover"], "--grep and --recover can't be used together"),
                      (["-d", "--grep", "a", "-9"], "Compression level has no effect when searching."),
                      (["-d", "--grep", "a", "--list"], "--list and --grep can't be used together"),
                      (["-d", "--grep", "a", "--range", "0:1"], "--range and --grep can't be used together"),
                      (["-d", "--count"], "--count can only be used with --grep"), (["-d", "--ignore-case"], "--ignore-case can only be used with --grep"),
                      (["-d", "--line-number"], "--line-number can only be used with --grep")):
        assert main(argv + [str(src), str(out)], engine=sim_engine) == 1
        assert capsys.readouterr().err.strip() == msg


# ---- GPU only: sizes a user searches ----
@pytest.fixture(scope="module")
def bench_stream():
    g = json.load(open(os.path.join(HERE, "golden", "corpus_goldens.json")))["text:100000000:8:L9"]
    src = gen_text(100_000_000, 8).tobytes()
    comp = Bzip2Engine(0).compressFile(src, None, 9)
    assert hashlib.sha256(comp).hexdigest() == g["out_sha256"]
    return comp, src


@pytest.mark.gpu
def test_bench_stream(gpu_engine, bench_stream):
    comp, full = bench_stream
    assert gpu_engine.decompressFile(comp) == full
    check(gpu_engine, comp, full, [RARE], tiles=(0,))
    check(gpu_engine, comp, full, WORDS16, max_matches=3_000_000, tiles=(0,))
    check(gpu_engine, comp, full, [b"the"], max_matches=100_000, tiles=(0,))
    check(gpu_engine, comp, full, [b"the", b"THE"], ignore_case=True, max_matches=500_000, tiles=(0,))


@pytest.mark.gpu
def test_ten_million_matches(gpu_engine, oracle):
    data = b"a" * 10_000_000
    comp = oracle.compress(data, 9)
    r = gpu_engine.search(comp, b"a", lines=True)
    assert r.total_matches == 10_000_000 and r.total_lines == 1 and r.lines == data + b"\n"
    assert np.array_equal(r.matches["offset"], np.arange(10_000_000, dtype=np.uint64))
    assert (r.matches["line_end"] == 10_000_000).all() and int((r.matches["flags"] != 0).sum()) == 1
    r = gpu_engine.search(comp, [b"aa", b"a"], max_matches=7)
    assert r.total_matches == 19_999_999 and r.matches["offset"].tolist() == [0, 0, 1, 1, 2, 2, 3]
    assert r.matches["pattern"].tolist() == [0, 1, 0, 1, 0, 1, 0]


@pytest.mark.gpu
def test_fifty_megabyte_line(gpu_engine):
    body = gen_text(50_000_000, 52).tobytes().replace(b"\n", b" ")
    data = b"head\n" + body + b"tail"
    comp = gpu_engine.compressFile(data, None, 9)
    want = model(data, [b"head", b"tail", b"Paris"], max_matches=None)
    r = gpu_engine.search(comp, [b"head", b"tail", b"Paris"], lines=True)
    assert np.array_equal(r.matches, want[0]) and (r.total_matches, r.total_lines) == want[1:3]
    assert r.lines == want[3] and r.lines.endswith(b"tail\n") and len(r.lines) == len(data) + 1
