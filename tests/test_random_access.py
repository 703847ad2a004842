"""Random access to the decompressed bytes: Bzip2Engine.index / decompressRanges / decompressRange / open, the --list and
--range command line (bz2b200_index and bz2b200_decompress_ranges in include/bz2b200.h).

Expected values come from the oracle and libbz2, never from the code under test: the block positions and sizes from
oracle.table, the end bits from the signatures the bit helpers find, the stored CRCs from the 32 bits after each signature,
the bytes from oracle.decompress / oracle.decompress_block.  Every case runs on the simulator (both parse kernels) and on
the GPU (-m gpu, both parse kernels); the 100 MB bench stream runs on the GPU only."""
import bz2
import ctypes as C
import io
import json
import os
import hashlib

import numpy as np
import pytest

from compressjs_flattened_b200 import _native
from compressjs_flattened_b200.bzip2 import INDEX_DTYPE, Bzip2Engine, Bzip2Error, Bzip2Index, Err
from compressjs_flattened_b200.corpus import gen_text
from test_recover import MAGIC_BLOCK, MAGIC_END, damage_field, flip, footer_pos, get_bits, make, oracle_block

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_SO = os.environ.get("BZ2B200_SIM_LIB") or os.path.join(HERE, "sim", "libbz2b200_sim.so")   # e.g. an -fsanitize=address build

ENGINES = [pytest.param(("sim", "1"), id="sim-parse1"), pytest.param(("sim", "2"), id="sim-parse2"),
           pytest.param(("gpu", "1"), id="gpu-parse1", marks=pytest.mark.gpu),
           pytest.param(("gpu", "2"), id="gpu-parse2", marks=pytest.mark.gpu)]


@pytest.fixture(params=ENGINES)
def eng(request, monkeypatch):
    where, mode = request.param
    monkeypatch.setenv("BZ2B200_PARSE", mode)   # read when the context is created
    if where == "sim":
        request.getfixturevalue("sim_engine")   # builds the simulator library when it is stale
        e = Bzip2Engine(0, _native.Library(SIM_SO))
    else:
        e = Bzip2Engine(0)
    e.on_gpu = where == "gpu"
    yield e
    e.close()


# ---- inputs and the expected index ----
def expected_index(oracle, streams, multistream=True):
    """the index of the concatenation of `streams` [(bytes, level)] from the oracle's table and the bit helpers"""
    blob = b"".join(s for s, _ in streams)
    rows = oracle.table(blob, multistream)
    bounds, at = [], 0
    for s, lv in streams:
        bounds.append((8 * at, 8 * (at + len(s)), lv, 8 * at + footer_pos(s)))
        at += len(s)
    out, off = [], 0
    for i, (p, size) in enumerate(rows):
        k = next(k for k, b in enumerate(bounds) if b[0] <= p < b[1])
        nxt = rows[i + 1][0] if i + 1 < len(rows) else None
        end = nxt if nxt is not None and nxt < bounds[k][1] else bounds[k][3]
        assert get_bits(blob, p, 48) == MAGIC_BLOCK and get_bits(blob, end, 48) in (MAGIC_BLOCK, MAGIC_END)
        out.append((p, end, off, size, get_bits(blob, p + 48, 32), k, bounds[k][2]))
        off += size
    return blob, np.array(out, dtype=INDEX_DTYPE)


@pytest.fixture(scope="module")
def three(oracle):
    """three streams of levels 1, 5 and 9, small block caps (many blocks)"""
    parts = [(make(oracle, gen_text(7_000, 21).tobytes(), 997, 1)[0], 1), (make(oracle, gen_text(9_000, 22).tobytes(), 2500, 5)[0], 5),
             (make(oracle, gen_text(6_000, 23).tobytes(), 1800, 9)[0], 9)]
    blob, ix = expected_index(oracle, parts)
    return blob, ix, oracle.decompress(blob, True)


def equal_index(got, want):
    assert got.entries.dtype == INDEX_DTYPE
    assert got.entries.tolist() == want.tolist()


def err_code(fn):
    try:
        fn()
    except Bzip2Error as e:
        return e.errorCode
    return 0


def c_ranges(eng, blob, entries, starts, lens):
    """bz2b200_decompress_ranges called directly (no clipping): (rc, bytes)"""
    a = np.frombuffer(blob, dtype=np.uint8)
    ent = np.ascontiguousarray(entries, dtype=INDEX_DTYPE)
    s, ln = np.array(starts, dtype=np.uint64), np.array(lens, dtype=np.uint64)
    out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
    rc = eng._L.bz2b200_decompress_ranges(eng._ctx, a.ctypes.data, a.size, ent.ctypes.data, len(ent), s.ctypes.data, ln.ctypes.data, len(s),
                                          C.byref(out), C.byref(n))
    return rc, (eng._take(out, n.value) if rc == 0 else None)


def covering(ix, ranges):
    """blocks that cover any range, and the bytes of their spans (runs of consecutive blocks, whole bytes)"""
    ends = (ix["out_offset"] + ix["out_bytes"]).tolist()
    cov = sorted({i for s, ln in ranges if ln for i in range(len(ix)) if ix["out_offset"][i] < s + ln and ends[i] > s})
    spans, first = 0, None
    for j, i in enumerate(cov):
        if first is None:
            first = i
        if j + 1 == len(cov) or cov[j + 1] != i + 1:
            spans += ((int(ix["bit_end"][i]) + 7) >> 3) - (int(ix["bit_begin"][first]) >> 3)
            first = None
    return cov, spans


# ---- 1. the index ----
def test_index_matches_oracle_three_streams(eng, oracle, three):
    blob, want, full = three
    ix = eng.index(blob, True)
    equal_index(ix, want)
    assert ix.total == len(full) and len(ix) == len(want)
    assert sorted(set(ix.entries["level"].tolist())) == [1, 5, 9] and ix.entries["stream"].tolist()[-1] == 2
    first_stream = [r for r in want.tolist() if r[5] == 0]
    equal_index(eng.index(blob, False), np.array(first_stream, dtype=INDEX_DTYPE))
    rows = []
    eng.table(blob, lambda p, s: rows.append((p, s)), True)
    assert rows == [(r[0], r[3]) for r in want.tolist()]


def test_index_single_stream_and_libbz2(eng, oracle):
    src = gen_text(20_000, 24).tobytes()
    comp, _ = make(oracle, src, 1500, 3)
    blob, want = expected_index(oracle, [(comp, 3)], False)
    equal_index(eng.index(comp), want)
    lib = bz2.compress(gen_text(230_000, 25).tobytes(), 1)
    blob, want = expected_index(oracle, [(lib, 1)], False)
    assert len(want) >= 3
    ix = eng.index(lib)
    equal_index(ix, want)
    assert eng.decompressRanges(lib, ix, [(0, ix.total)]) == [bz2.decompress(lib)]


def test_index_errors_equal_table(eng, oracle, three):
    blob, want, _ = three
    comp, pos = make(oracle, gen_text(12_000, 26).tobytes(), 2500)
    rng = np.random.default_rng(3)
    cases = [comp[:len(comp) // 2], comp[:3], b"", b"BZh0" + comp[4:], flip(comp, pos[2] + 5), damage_field(oracle, comp, pos, 1, "data", rng),
             damage_field(oracle, comp, pos, 3, "crc", rng), blob[:len(blob) - 40], blob + b"BZh"]
    for multistream in (False, True):
        for d in cases:
            t = err_code(lambda: eng.table(d, lambda p, s: None, multistream))
            assert err_code(lambda: eng.index(d, multistream)) == t
    assert err_code(lambda: eng.index(comp[:len(comp) // 2])) == Err.UNEXPECTED_INPUT_EOF


# ---- 2. ranges ----
def test_ranges_random_and_edges(eng, oracle, three):
    blob, want, full = three
    ix = Bzip2Index(want)
    total = len(full)
    rng = np.random.default_rng(7)
    rand = [(int(s), int(rng.integers(0, 3000))) for s in rng.integers(0, total, 200)]
    rand = [(s, min(ln, total - s)) for s, ln in rand]
    got = eng.decompressRanges(blob, ix, rand)
    assert got == [full[s:s + ln] for s, ln in rand]
    offs = want["out_offset"].tolist() + [total]
    edges = []
    for o in offs[1:-1]:
        edges += [(o, 10), (o - 10, 10), (o - 1, 2), (0, o), (o, total - o)]
    edges += [(0, 0), (total, 0), (5, 0), (offs[3], 0)]
    stream_ends = np.cumsum([len(oracle.decompress(s)) for s in split_streams(blob, want)]).tolist()[:-1]
    edges += [(e - 100, 200) for e in stream_ends] + [(stream_ends[0] - 5, stream_ends[1] - stream_ends[0] + 10)]
    edges += [(100, 500), (100, 500), (300, 1000), (0, total)]
    edges += edges[::-1]
    assert eng.decompressRanges(blob, ix, edges) == [full[s:s + ln] for s, ln in edges]
    st = eng.stats()
    assert (st.n_blocks, st.out_bytes) == (len(want), sum(ln for _, ln in edges))
    assert eng.decompressRange(blob, ix, 0, total) == full


def split_streams(blob, want):
    """the streams of blob, cut at the first block of each stream (stream k starts 32 bits before it)"""
    starts = [int(want["bit_begin"][i]) // 8 - 4 for i in range(len(want)) if i == 0 or want["stream"][i] != want["stream"][i - 1]]
    return [blob[a:b] for a, b in zip(starts, starts[1:] + [len(blob)])]


def test_ranges_first_stream_blocks_equal_decompress_block(eng, oracle, three):
    blob, want, _ = three
    ix = Bzip2Index(want)
    for e in want.tolist():
        if e[5] == 0:
            assert eng.decompressRange(blob, ix, e[2], e[3]) == oracle.decompress_block(blob, e[0])


def test_ranges_python_clipping_equals_slicing(eng, three):
    blob, want, full = three
    ix = Bzip2Index(want)
    total = len(full)
    rng = np.random.default_rng(8)
    cases = [(int(s), int(ln)) for s, ln in zip(rng.integers(-2 * total, 2 * total, 100), rng.integers(-500, total + 500, 100))]
    cases += [(-10, 20), (total - 5, 100), (total + 5, 10), (0, -1), (-total - 10, 30), (3, 0)]
    assert eng.decompressRanges(blob, ix, cases) == [full[s:s + ln] for s, ln in cases]


def test_ranges_c_argument_checks(eng, three):
    blob, want, full = three
    total = len(full)
    assert c_ranges(eng, blob, want, [0, total - 3], [10, 3]) == (0, full[:10] + full[-3:])
    assert c_ranges(eng, blob, want, [total], [0]) == (0, b"")
    for s, ln in ((total, 1), (total + 1, 0), (total - 3, 4), (2 ** 63, 2 ** 63)):
        assert c_ranges(eng, blob, want, [s], [ln])[0] == _native.E_ARG
    bad = []
    e = want.copy(); e[[2, 3]] = e[[3, 2]]; bad.append(e)                        # not sorted
    e = want.copy(); e["out_offset"][4:] += 1; bad.append(e)                    # not contiguous
    e = want.copy(); e["out_offset"] += 7; bad.append(e)                        # not from 0
    e = want.copy(); e["level"][1] = 0; bad.append(e)
    e = want.copy(); e["level"][1] = 10; bad.append(e)
    e = want.copy(); e["bit_end"][2] = e["bit_begin"][2]; bad.append(e)
    e = want.copy(); e["bit_end"][-1] = 8 * len(blob) + 1; bad.append(e)
    for e in bad:
        assert c_ranges(eng, blob, e, [0], [1])[0] == _native.E_ARG
        with pytest.raises(RuntimeError):
            eng.decompressRange(blob, Bzip2Index(e), 0, 1)
    assert c_ranges(eng, blob, want[:0], [0], [0]) == (0, b"")


# ---- 3. only the covering blocks ----
def test_ranges_stats_count_covering_blocks(eng, three):
    blob, want, full = three
    ix = Bzip2Index(want)
    rng = np.random.default_rng(9)
    for trial in range(6):
        rs = [(int(s), int(rng.integers(0, 800))) for s in rng.integers(0, len(full) - 800, int(rng.integers(1, 8)))]
        got = eng.decompressRanges(blob, ix, rs)
        assert got == [full[s:s + ln] for s, ln in rs]
        cov, spans = covering(want, rs)
        st = eng.stats()
        assert (st.n_blocks, st.in_bytes, st.out_bytes) == (len(cov), spans, sum(ln for _, ln in rs))


def test_ranges_damage_outside_is_not_read(eng, oracle):
    src = gen_text(24_000, 27).tobytes()
    comp, pos = make(oracle, src, 2500)
    _, want = expected_index(oracle, [(comp, 9)], False)
    ix = Bzip2Index(want)
    rng = np.random.default_rng(10)
    k = 4
    for field in ("data", "sel", "crc"):
        d = damage_field(oracle, comp, pos, k, field, rng)
        o = want["out_offset"].tolist()
        rs = [(o[k - 1], o[k] - o[k - 1]), (o[k + 1], 100), (0, 10)]
        assert eng.decompressRanges(d, ix, rs) == [src[s:s + ln] for s, ln in rs]
        assert eng.stats().n_blocks == 3


@pytest.mark.parametrize("field", ["crc", "orig", "sel", "lens", "data"])
def test_ranges_damaged_block_gives_oracle_code(eng, oracle, field):
    src = gen_text(24_000, 28).tobytes()
    comp, pos = make(oracle, src, 2500)
    _, want = expected_index(oracle, [(comp, 9)], False)
    ix = Bzip2Index(want)
    k = 5
    d = damage_field(oracle, comp, pos, k, field, np.random.default_rng(hash(field) & 0xffff))
    what, code = oracle_block(oracle, d, pos[k])
    assert what == "err"
    o = want["out_offset"].tolist()
    assert err_code(lambda: eng.decompressRanges(d, ix, [(o[k] + 10, 5)])) == code
    assert err_code(lambda: eng.decompressRanges(d, ix, [(o[k + 1], 10), (o[k - 1], o[k + 1] - o[k - 1])])) == code


def test_ranges_first_failing_block_in_index_order_wins(eng, oracle):
    src = gen_text(24_000, 29).tobytes()
    comp, pos = make(oracle, src, 2500)
    _, want = expected_index(oracle, [(comp, 9)], False)
    ix = Bzip2Index(want)
    o = want["out_offset"].tolist()
    crc_hit = damage_field(oracle, comp, pos, 6, "crc", np.random.default_rng(11))
    d1 = flip(crc_hit, pos[2] + 20)      # block 2: no signature; block 6: bad CRC
    d2 = flip(damage_field(oracle, comp, pos, 2, "crc", np.random.default_rng(12)), pos[6] + 20)
    rs = [(o[6], 10), (o[7], 3), (o[2], 10), (o[0], 1)]   # the later block asked for first
    for batch in (0, 3):
        eng._L.bz2b200_debug_set_decode_batch(eng._ctx, None, batch)
        try:
            assert err_code(lambda: eng.decompressRanges(d1, ix, rs)) == Err.NOT_BZIP_DATA
            assert err_code(lambda: eng.decompressRanges(d2, ix, rs)) == Err.DATA_ERROR
            assert err_code(lambda: eng.decompressRanges(d1, ix, rs[:2])) == Err.DATA_ERROR
        finally:
            eng._L.bz2b200_debug_set_decode_batch(eng._ctx, None, 0)


def test_ranges_index_of_another_file(eng, oracle):
    comp, _ = make(oracle, gen_text(24_000, 30).tobytes(), 2500)
    other, _ = make(oracle, gen_text(12_000, 31).tobytes(), 2000)
    _, theirs = expected_index(oracle, [(other, 9)], False)
    ix = Bzip2Index(theirs)
    o = theirs["out_offset"].tolist()
    assert int(theirs["bit_begin"][0]) == 32   # both files have a signature there: a stale end bit or size
    assert err_code(lambda: eng.decompressRange(comp, ix, 0, 10)) == Err.DATA_ERROR
    assert "index does not match" in eng._L.bz2b200_last_error(eng._ctx).decode()
    for k in range(1, len(theirs)):
        if get_bits(comp, int(theirs["bit_begin"][k]), 48) != MAGIC_BLOCK:
            assert err_code(lambda: eng.decompressRange(comp, ix, o[k], 10)) == Err.NOT_BZIP_DATA


# ---- 4. batches ----
def test_ranges_in_small_batches(eng, three):
    blob, want, full = three
    ix = Bzip2Index(want)
    rng = np.random.default_rng(12)
    rs = [(int(s), 1500) for s in rng.integers(0, len(full) - 1500, 12)] + [(0, len(full))]
    eng._L.bz2b200_debug_set_decode_batch(eng._ctx, None, 3)
    try:
        assert eng.decompressRanges(blob, ix, rs) == [full[s:s + ln] for s, ln in rs]
        assert eng.stats().n_blocks == len(want) > 3
        rs = rs[:-1]
        assert eng.decompressRanges(blob, ix, rs) == [full[s:s + ln] for s, ln in rs]
        cov, spans = covering(want, rs)
        assert (eng.stats().n_blocks, eng.stats().in_bytes) == (len(cov), spans) and len(cov) > 3
    finally:
        eng._L.bz2b200_debug_set_decode_batch(eng._ctx, None, 0)


# ---- 5. the reader ----
def run_reader(f, full, seed, ops=500):
    ref = io.BytesIO(full)
    rng = np.random.default_rng(seed)
    total = len(full)
    assert f.readable() and f.seekable()
    for _ in range(ops):
        op = rng.random()
        if op < 0.25:
            p = int(rng.integers(0, total + 50))
            assert f.seek(p) == ref.seek(p)
        elif op < 0.35:
            d = int(rng.integers(-min(ref.tell(), 3000), 3000))
            assert f.seek(d, io.SEEK_CUR) == ref.seek(d, io.SEEK_CUR)
        elif op < 0.42:
            d = -int(rng.integers(0, min(total, 5000)))
            assert f.seek(d, io.SEEK_END) == ref.seek(d, io.SEEK_END)
        elif op < 0.47:
            assert f.read() == ref.read()
        elif op < 0.52:
            b1 = bytearray(int(rng.integers(0, 4000)))
            b2 = bytearray(len(b1))
            assert f.readinto(b1) == ref.readinto(b2) and b1 == b2
        else:
            k = int(rng.integers(0, 5000))
            assert f.read(k) == ref.read(k)
        assert f.tell() == ref.tell()


def test_reader_random_operations(eng, oracle, three, tmp_path):
    blob, want, full = three
    with eng.open(blob, Bzip2Index(want)) as f:
        run_reader(f, full, 13)
    path = tmp_path / "three.bz2"
    path.write_bytes(blob)
    with eng.open(str(path), multistream=True) as f:   # the index is built first
        run_reader(f, full, 14)
    with eng.open(path) as f:
        assert f.read() == oracle.decompress(blob)


def test_reader_whole_file_in_one_call(eng, three):
    blob, want, full = three
    with eng.open(blob, Bzip2Index(want)) as f:
        f.seek(100)
        assert f.read() == full[100:]
        assert eng.stats().out_bytes == len(full) - 100
        assert f.read() == b"" and f.read(10) == b""


# ---- 6. the command line ----
def test_command_line_list_and_range(sim_engine, oracle, three, tmp_path, capsys):
    from compressjs_flattened_b200.__main__ import main
    blob, want, full = three
    src, out, ixf = tmp_path / "three.bz2", tmp_path / "out", tmp_path / "three.idx"
    src.write_bytes(blob)
    assert main(["-d", "--list", "--multistream", str(src)], engine=sim_engine) == 0
    text = capsys.readouterr().out
    assert text.splitlines()[0] == "# bzip2 block index v1" and len(text.splitlines()) == len(want) + 1
    equal_index(Bzip2Index.from_text(text), want)
    assert Bzip2Index.from_text(text).to_text() == text
    assert main(["-d", "--list", str(src), str(out)], engine=sim_engine) == 0
    assert len(Bzip2Index.from_text(out.read_text())) == int((want["stream"] == 0).sum())
    ixf.write_text(text)
    s, ln = 5000, 9000
    assert main(["-d", "--range", f"{s}:{ln}", "--index", str(ixf), str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == full[s:s + ln]
    assert main(["-d", "--multistream", "--range", f"{s}:{ln}", str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == full[s:s + ln]
    assert main(["--range", f"{len(full) - 10}:100", "--index", str(ixf), str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == full[-10:]
    capsys.readouterr()
    for argv, msg in ((["-z", "--list"], "--list can only be used without -z"), (["-d", "--list", "-b", "32"], "--list and --block can't be used together"),
                      (["--list", "--recover"], "--list and --recover can't be used together"),
                      (["-d", "--list", "-9"], "Compression level has no effect when listing."),
                      (["-z", "--range", "0:1"], "--range can only be used without -z"),
                      (["-d", "--range", "0:1", "-b", "32"], "--range and --block can't be used together"),
                      (["--range", "0:1", "--recover"], "--range and --recover can't be used together"),
                      (["-d", "--range", "0:1", "-1"], "Compression level has no effect when reading a range."),
                      (["-d", "--range", "12"], "--range takes START:LEN, not 12"),
                      (["-d", "--list", "--range", "0:1"], "--list and --range can't be used together"),
                      (["-d", "--index", str(ixf)], "--index can only be used with --range")):
        assert main(argv + [str(src), str(out)], engine=sim_engine) == 1
        assert capsys.readouterr().err.strip() == msg


def test_index_text_rejects_malformed():
    good = Bzip2Index(np.array([(32, 9000, 0, 2500, 0xdeadbeef, 0, 9), (9000, 17000, 2500, 2000, 0x1234, 0, 9)], dtype=INDEX_DTYPE))
    text = good.to_text()
    assert text.splitlines()[1] == "0\t9\t32\t9000\t0\t2500\tdeadbeef"
    equal_index(Bzip2Index.from_text(text), good.entries)
    assert len(Bzip2Index.from_text(Bzip2Index.HEADER + "\n")) == 0
    lines = text.splitlines()
    for bad in ("", "# bzip2 block index v2\n" + "\n".join(lines[1:]), text.replace("\t9\t", "\t9 \t", 1), text + "1\t2\t3\n",
                text.replace("deadbeef", "xyz"), text.replace("\t2500\t", "\t-2500\t", 1), text.replace("\t2500\t", "\t4294967296\t", 1),
                text + "\n", lines[1] + "\n"):
        with pytest.raises(ValueError):
            Bzip2Index.from_text(bad)


# ---- 7. the 100 MB bench stream (GPU) ----
@pytest.mark.gpu
def test_bench_stream_ranges(gpu_engine):
    g = json.load(open(os.path.join(HERE, "golden", "corpus_goldens.json")))["text:100000000:8:L9"]
    comp = gpu_engine.compressFile(gen_text(100_000_000, 8), None, 9)
    assert hashlib.sha256(comp).hexdigest() == g["out_sha256"]
    full = gpu_engine.decompressFile(comp)
    ix = gpu_engine.index(comp)
    rows = []
    gpu_engine.table(comp, lambda p, s: rows.append((p, s)))
    assert list(zip(ix.entries["bit_begin"].tolist(), ix.entries["out_bytes"].tolist())) == rows and len(rows) == g["n_blocks"]
    assert ix.total == len(full) and (ix.entries["bit_end"][:-1] == ix.entries["bit_begin"][1:]).all()
    rng = np.random.default_rng(15)
    rs = [(int(s), int(rng.integers(0, 2_000_000))) for s in rng.integers(0, len(full), 200)]
    assert gpu_engine.decompressRanges(comp, ix, rs) == [full[s:s + ln] for s, ln in rs]
    rs = [(int(s), 4096) for s in rng.integers(0, len(full) - 4096, 4096)]
    assert gpu_engine.decompressRanges(comp, ix, rs) == [full[s:s + 4096] for s, _ in rs]
    assert gpu_engine.stats().out_bytes == 4096 * 4096
