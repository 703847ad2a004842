"""Lines by number: Bzip2Engine.lineIndex / decompressLines / lineSpans, the --line-index and --lines command line
(bz2b200_line_index and bz2b200_decompress_lines in include/bz2b200.h).

Expected values come from the oracle and libbz2, never from the code under test: the output from oracle.decompress, the
lines from data.split(b"\\n") with the '\\n' put back and an empty tail dropped, the '\\n' bytes of every block from
oracle.decompress_block of each row of oracle.table, the block index from test_random_access.expected_index.  Every case
runs on the simulator (both parse kernels) and on the GPU (-m gpu, both parse kernels); small block caps and 256-byte
directory tiles make small inputs span many blocks and tiles."""
import bz2
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from compressjs_flattened_b200 import _native
from compressjs_flattened_b200.bzip2 import INDEX_DTYPE, Bzip2Engine, Bzip2Error, Bzip2Index, Bzip2LineIndex, Err
from compressjs_flattened_b200.corpus import gen_text
from test_random_access import equal_index
from test_recover import damage_field, make

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_SO = os.environ.get("BZ2B200_SIM_LIB") or os.path.join(HERE, "sim", "libbz2b200_sim.so")
TILES = (0, 256)

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


# ---- the model ----
def model_lines(data):
    lines = [ln + b"\n" for ln in data.split(b"\n")]
    lines[-1] = lines[-1][:-1]
    if not lines[-1]:
        lines.pop()
    return lines


def model_counts(oracle, comp, multistream):
    return [oracle.decompress_block(comp, p).count(b"\n") for p, _ in oracle.table(comp, multistream)]


def model_spans(lines, reqs, total_lines):
    starts = np.concatenate([[0], np.cumsum([len(x) for x in lines], dtype=np.uint64)]).astype(np.uint64)
    out = []
    for f, k in reqs:
        a, b = slice(f, f + k).indices(total_lines)[:2]
        b = max(a, b)
        out.append((int(starts[a]), int(starts[b] - starts[a])))
    return out


def check_index(eng, oracle, comp, multistream, tiles=TILES):
    data = oracle.decompress(comp, multistream)
    lines = model_lines(data)
    counts = model_counts(oracle, comp, multistream)
    for tile in tiles:
        eng.debug_set_line_tile(tile)
        li = eng.lineIndex(comp, multistream)
        equal_index(li.blocks, eng.index(comp, multistream).entries)
        assert li.newlines.dtype == np.uint32 and li.newlines.tolist() == counts, tile
        assert (li.total_lines, li.total) == (len(lines), len(data)), tile
    eng.debug_set_line_tile(0)
    return li, data, lines


def check_reads(eng, comp, li, lines, reqs, tiles=TILES):
    want = [b"".join(lines[f:f + k]) for f, k in reqs]
    spans = model_spans(lines, reqs, li.total_lines)
    for tile in tiles:
        eng.debug_set_line_tile(tile)
        assert eng.decompressLines(comp, li, reqs) == want, tile
        got = eng.lineSpans(comp, li, reqs)
        assert got.dtype == np.uint64 and got.shape == (len(reqs), 2) and [tuple(r) for r in got.tolist()] == spans, tile
    eng.debug_set_line_tile(0)
    assert eng.decompressRanges(comp, li.blocks, spans) == want
    return spans


def block_starts(li):
    return li.blocks.entries["out_offset"].tolist()


@pytest.fixture(scope="module")
def three(oracle):
    """three streams of levels 1, 5 and 9; the first ends with '\\n', the second starts with one, the last has none at its end"""
    a = gen_text(7_000, 41).tobytes().rstrip(b"\n") + b"\n"
    b = b"\n" + gen_text(9_000, 42).tobytes()
    c = gen_text(6_000, 43).tobytes().rstrip(b"\n") + b" end"
    parts = [make(oracle, a, 997, 1)[0], make(oracle, b, 2500, 5)[0], make(oracle, c, 1800, 9)[0]]
    return b"".join(parts), (a, b, c)


# ---- 1. the line index ----
def test_line_index_three_streams_and_single(eng, oracle, three):
    blob, (a, b, c) = three
    li, data, lines = check_index(eng, oracle, blob, True)
    assert sorted(set(li.blocks.entries["level"].tolist())) == [1, 5, 9] and len(li) >= 12
    s_end = len(a)   # '\n' as the last byte of stream 0 and the first of stream 1
    assert data[s_end - 1:s_end + 1] == b"\n\n" and s_end in block_starts(li)
    check_index(eng, oracle, blob, False)
    li, _, lines = check_index(eng, oracle, make(oracle, gen_text(20_000, 44).tobytes(), 1500, 3)[0], False)
    assert len(li) >= 10 and len(lines) > 50
    lib = bz2.compress(gen_text(230_000, 45).tobytes(), 1)
    li = eng.lineIndex(lib)
    assert li.newlines.tolist() == model_counts(oracle, lib, False) and li.total_lines == len(model_lines(bz2.decompress(lib)))


def test_line_index_ends_empty_and_no_newline(eng, oracle):
    text = gen_text(12_000, 46).tobytes()
    for data in (text.rstrip(b"\n") + b"\n", text.rstrip(b"\n") + b"tail", b"x", b"\n"):
        li, _, lines = check_index(eng, oracle, make(oracle, data, 2500)[0], False)
        assert li.total_lines == data.count(b"\n") + (not data.endswith(b"\n"))
    empty = oracle.compress(b"", 9)
    li, _, _ = check_index(eng, oracle, empty, False)
    assert (len(li), li.total_lines, li.total) == (0, 0, 0)
    flat = text.replace(b"\n", b" ")
    comp = make(oracle, flat, 2500)[0]
    li, _, _ = check_index(eng, oracle, comp, False)
    assert li.total_lines == 1 and len(li) >= 4 and not li.newlines.any()
    check_reads(eng, comp, li, [flat], [(0, 1), (-1, 1), (0, 0), (1, 0)])


def test_line_index_only_newlines_and_crlf(eng, oracle):
    run = b"\n" * (30_000_000 if eng.on_gpu else 200_000)
    comp = oracle.compress(run, 9)
    li, _, _ = check_index(eng, oracle, comp, False, tiles=(0,))
    assert len(li) == 1 and li.total_lines == len(run) == int(li.newlines[0])   # one run block
    check_reads(eng, comp, li, [b"\n"] * len(run), [(0, 1), (len(run) - 1, 1), (12345, 3), (0, len(run))], tiles=(0,))
    crlf = gen_text(15_000, 47).tobytes().replace(b"\n", b"\r\n")
    comp = make(oracle, crlf, 2000)[0]
    li, _, lines = check_index(eng, oracle, comp, False)
    assert all(x.endswith(b"\r\n") for x in lines[:-1])
    check_reads(eng, comp, li, lines, [(0, 1), (3, 2), (-1, 1), (len(lines) - 1, 1)])


def test_newline_at_block_and_tile_edges(eng, oracle):
    # 10-byte lines and 2500-byte blocks: every block ends with '\n'; shifted by one, every block starts with one.
    # 16-byte lines: '\n' at 255 and 256 + 15 (the last byte of a 256-byte tile); shifted by one at 256 (its first)
    for line, shift in ((b"abcdefghi\n", 0), (b"abcdefghi\n", 1), (b"abcdefghijklmno\n", 0), (b"abcdefghijklmno\n", 1)):
        data = (b"\n" if shift else b"") + line * 1500
        comp = make(oracle, data, 2500)[0]
        li, _, lines = check_index(eng, oracle, comp, False)
        offs = block_starts(li)[1:]
        assert len(offs) >= 4
        if len(line) == 10:
            assert all(data[o - 1 + shift:o + shift] == b"\n" for o in offs)   # last byte of a block (shift 0) / first (shift 1)
        else:
            assert data[255 + shift] == ord("\n") and data[511 + shift] == ord("\n")
        k = len(lines) // 2
        reqs = [(0, 1), (k, 1), (k - 1, 3), (len(lines) - 1, 1)] + [(i, 1) for i in range(0, len(lines), 37)]
        at_block = [(o + shift) // len(line) for o in offs] if len(line) == 10 else []   # lines that start exactly at a block boundary
        spans = check_reads(eng, comp, li, lines, reqs + [(i, 1) for i in at_block] + [(i, 2) for i in at_block])
        if at_block and not shift:
            assert [sp[0] for sp in spans[len(reqs):len(reqs) + len(at_block)]] == offs


def test_command_line_line_index(sim_engine, oracle, three, tmp_path, capsys):
    from compressjs_flattened_b200.__main__ import main
    blob, _ = three
    src, out = tmp_path / "three.bz2", tmp_path / "out"
    src.write_bytes(blob)
    assert main(["-d", "--line-index", "--multistream", str(src)], engine=sim_engine) == 0
    text = capsys.readouterr().out
    li = sim_engine.lineIndex(blob, True)
    assert text == li.to_text() and text.splitlines()[:2] == ["# bzip2 line index v1", f"# lines {li.total_lines}"]
    back = Bzip2LineIndex.from_text(text)
    equal_index(back.blocks, li.blocks.entries)
    assert back.newlines.tolist() == li.newlines.tolist() and back.total_lines == li.total_lines and back.to_text() == text
    assert main(["-d", "--list", "--multistream", str(src)], engine=sim_engine) == 0
    assert capsys.readouterr().out == sim_engine.index(blob, True).to_text()   # --list is the block index, unchanged


# ---- 2. line reads ----
@pytest.fixture(scope="module")
def long_lines(oracle):
    """short lines, a line over three or more blocks, a line that starts exactly at a block boundary, no '\\n' at the end"""
    text = gen_text(9_000, 48).tobytes()
    body = text[:3000].rstrip(b"\n") + b"\n" + b"long " * 1800 + b"\n" + text[3000:]
    comp = make(oracle, body.rstrip(b"\n"), 2500)[0]
    return comp, body.rstrip(b"\n")


def test_first_last_boundary_and_long_lines(eng, oracle, long_lines):
    comp, data = long_lines
    li, _, lines = check_index(eng, oracle, comp, False)
    offs = block_starts(li)
    L = li.total_lines
    big = max(range(L), key=lambda i: len(lines[i]))
    starts = np.cumsum([0] + [len(x) for x in lines]).tolist()
    assert sum(1 for o in offs if starts[big] < o < starts[big + 1]) >= 2   # the long line spans three blocks or more
    check_reads(eng, comp, li, lines, [(0, 1), (L - 1, 1), (big, 1), (big - 1, 3), (L - 3, 3)])
    assert not data.endswith(b"\n") and lines[-1] == data[data.rindex(b"\n") + 1:]
    eng.decompressLines(comp, li, [(big, 1)])
    assert eng.stats().n_blocks >= 3


def test_empty_clipped_overlapping_and_all(eng, oracle, three):
    blob, _ = three
    li, data, lines = check_index(eng, oracle, blob, True, tiles=(0,))
    L = li.total_lines
    reqs = [(0, 0), (L, 0), (5, 0), (-5, 3), (-3, 10), (L - 2, 10), (L + 5, 3), (-L - 10, 4), (3, -1), (10, 20), (15, 20), (10, 20), (40, 5), (2, 3)]
    check_reads(eng, blob, li, lines, reqs)
    assert eng.decompressLines(blob, li, [(0, L)]) == [data]
    assert eng.decompressLines(blob, li, [(0, L)]) == [oracle.decompress(blob, True)] and eng.stats().n_blocks == len(li)
    assert eng.lineSpans(blob, li, [(0, 0), (L, 0)]).tolist() == [[0, 0], [len(data), 0]] and eng.stats().n_blocks == 0


def test_ten_thousand_random_lines(eng, oracle, three):
    blob, _ = three
    li, _, lines = check_index(eng, oracle, blob, True, tiles=(0,))
    rng = np.random.default_rng(49)
    reqs = [(int(f), 1) for f in rng.integers(0, li.total_lines, 10_000)]
    check_reads(eng, blob, li, lines, reqs)


def test_ranges_reuse_same_launches(eng, oracle):
    # the same input and requests as at the parent commit of the shared block decode: 21 launches there, with either kernel
    comp, _ = make(oracle, gen_text(30_000, 41).tobytes(), 2500)
    full = oracle.decompress(comp)
    ix = eng.index(comp)
    rs = [(100, 50), (7000, 6000), (29_000, 1000), (2500, 1), (0, 0)]
    assert eng.decompressRanges(comp, ix, rs) == [full[s:s + n] for s, n in rs]
    st = eng.stats()
    assert (len(ix), st.kernel_launches, st.n_blocks) == (12, 21, 6)


# ---- 3. errors ----
def c_lines(eng, comp, entries, newlines, total_lines, firsts, counts):
    a = np.frombuffer(comp, dtype=np.uint8)
    ent = np.ascontiguousarray(entries, dtype=INDEX_DTYPE)
    nl = np.ascontiguousarray(newlines, dtype=np.uint32)
    f, k = np.array(firsts, dtype=np.uint64), np.array(counts, dtype=np.uint64)
    out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
    rc = eng._L.bz2b200_decompress_lines(eng._ctx, a.ctypes.data, a.size, ent.ctypes.data, nl.ctypes.data, len(ent), total_lines, f.ctypes.data,
                                         k.ctypes.data, len(f), C.byref(out), C.byref(n), None)
    if rc == 0:
        eng._take(out, n.value)
    return rc, eng._L.bz2b200_last_error(eng._ctx).decode()


def err_code(fn):
    try:
        fn()
    except Bzip2Error as e:
        return e.errorCode
    return 0


def test_argument_errors(eng, oracle, long_lines):
    comp, data = long_lines
    li = eng.lineIndex(comp)
    e, nl, L = li.blocks.entries, li.newlines, li.total_lines
    assert c_lines(eng, comp, e, nl, L, [0, L - 1], [1, 1])[0] == 0
    bad = e.copy(); bad[[2, 3]] = bad[[3, 2]]
    rc, msg = c_lines(eng, comp, bad, nl, L, [0], [1])
    assert rc == _native.E_ARG and "index entry" in msg
    over = nl.copy(); over[1] = e["out_bytes"][1] + 1
    rc, msg = c_lines(eng, comp, e, over, L + int(over[1]) - int(nl[1]), [0], [1])
    assert rc == _native.E_ARG and "above the block's out_bytes" in msg
    for t in (L + 1, L - 2, 0):
        rc, msg = c_lines(eng, comp, e, nl, t, [0], [1])
        assert rc == _native.E_ARG and "total_lines" in msg
    rc, msg = c_lines(eng, comp, e[:0], nl[:0], 1, [0], [0])
    assert rc == _native.E_ARG and "total_lines" in msg
    for f, k in ((L, 1), (L + 1, 0), (L - 2, 3), (2 ** 63, 2 ** 63)):
        rc, msg = c_lines(eng, comp, e, nl, L, [f], [k])
        assert rc == _native.E_ARG and "outside the lines" in msg
    with pytest.raises(RuntimeError):
        eng.decompressLines(comp, Bzip2LineIndex(bad, nl, L), [(0, 1)])


def test_stale_line_index(eng, oracle):
    text = gen_text(20_000, 50).tobytes()
    k = 4
    comp = make(oracle, text, 2500)[0]
    li = eng.lineIndex(comp)
    o = block_starts(li)
    cut = text.index(b"\n", o[k])   # one '\n' fewer in block k, the same bytes per block
    other = text[:cut] + b" " + text[cut + 1:]
    theirs = eng.lineIndex(make(oracle, other, 2500)[0])
    assert theirs.blocks.entries["out_bytes"].tolist() == li.blocks.entries["out_bytes"].tolist()
    assert theirs.newlines.tolist() != li.newlines.tolist()
    stale = Bzip2LineIndex(li.blocks, theirs.newlines, theirs.total_lines)
    first = int(theirs.newlines[:k].sum()) + 1
    assert err_code(lambda: eng.decompressLines(comp, stale, [(first, 1)])) == Err.DATA_ERROR
    assert "index does not match the input" in eng._L.bz2b200_last_error(eng._ctx).decode()
    assert eng.decompressLines(comp, stale, [(0, 1)]) == [text[:text.index(b"\n") + 1]]   # block 0 agrees
    ends = text.endswith(b"\n")   # the last byte against total_lines
    wrong = Bzip2LineIndex(li.blocks, li.newlines, li.total_lines + (1 if ends else -1))
    assert err_code(lambda: eng.decompressLines(comp, wrong, [(0, 1), (wrong.total_lines - 1, 1)])) == Err.DATA_ERROR
    assert "index does not match the input" in eng._L.bz2b200_last_error(eng._ctx).decode()


@pytest.mark.parametrize("field", ["crc", "sel", "data"])
def test_damaged_block_gives_range_code(eng, oracle, field):
    text = gen_text(24_000, 51).tobytes()
    comp, pos = make(oracle, text, 2500)
    li = eng.lineIndex(comp)
    k = 5
    d = damage_field(oracle, comp, pos, k, field, np.random.default_rng(hash(field) & 0xffff))
    o = block_starts(li)
    code = err_code(lambda: eng.decompressRanges(d, li.blocks, [(o[k] + 10, 5)]))
    assert code != 0
    line = int(li.newlines[:k].sum()) + 1
    assert err_code(lambda: eng.decompressLines(d, li, [(line, 1)])) == code
    assert err_code(lambda: eng.lineIndex(d)) == err_code(lambda: eng.decompressFile(d))
    assert err_code(lambda: eng.lineIndex(d[:len(d) // 2])) == err_code(lambda: eng.decompressFile(d[:len(d) // 2])) != 0


# ---- 4. the command line and the text form ----
def test_command_line_lines(sim_engine, oracle, three, tmp_path, capsys):
    from compressjs_flattened_b200.__main__ import main
    blob, _ = three
    data = oracle.decompress(blob, True)
    lines = model_lines(data)
    src, out, lif, bif = tmp_path / "three.bz2", tmp_path / "out", tmp_path / "three.lines", tmp_path / "three.idx"
    src.write_bytes(blob)
    lif.write_text(sim_engine.lineIndex(blob, True).to_text())
    bif.write_text(sim_engine.index(blob, True).to_text())
    assert main(["-d", "--lines", "5:3", "--index", str(lif), str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == b"".join(lines[4:7])
    assert main(["-d", "--multistream", "--lines", f"{len(lines) - 1}:10", str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == b"".join(lines[-2:])
    assert main(["-d", "--lines", "1:2", str(src), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == b"".join(model_lines(oracle.decompress(blob))[:2])
    # the numbers --grep --line-number prints select the same lines
    assert main(["-d", "--multistream", "--grep", "the", "--line-number", str(src), str(out)], engine=sim_engine) == 0
    for row in out.read_bytes().split(b"\n")[:5]:
        no, text = row.split(b":", 1)
        assert main(["-d", "--lines", f"{int(no)}:1", "--index", str(lif), str(src), str(tmp_path / "one")], engine=sim_engine) == 0
        assert (tmp_path / "one").read_bytes() == text + b"\n"
    capsys.readouterr()
    for argv, msg in ((["-d", "--lines", "1:1", "--index", str(bif)], f"--lines needs a line index (--line-index output), and {bif} is a block index"),
                      (["-z", "--lines", "1:1"], "--lines can only be used without -z"), (["-z", "--line-index"], "--line-index can only be used without -z"),
                      (["-d", "--lines", "1:1", "-b", "32"], "--lines and --block can't be used together"),
                      (["-d", "--line-index", "-b", "32"], "--line-index and --block can't be used together"),
                      (["--lines", "1:1", "--recover"], "--lines and --recover can't be used together"),
                      (["--line-index", "--recover"], "--line-index and --recover can't be used together"),
                      (["-d", "--lines", "1:1", "-9"], "Compression level has no effect when reading lines."),
                      (["-d", "--line-index", "-3"], "Compression level has no effect when listing lines."),
                      (["-d", "--lines", "1:1", "--range", "0:1"], "--range and --lines can't be used together"),
                      (["-d", "--lines", "1:1", "--grep", "a"], "--grep and --lines can't be used together"),
                      (["-d", "--lines", "1:1", "--list"], "--list and --lines can't be used together"),
                      (["-d", "--line-index", "--list"], "--list and --line-index can't be used together"),
                      (["-d", "--line-index", "--lines", "1:1"], "--line-index and --lines can't be used together"),
                      (["-d", "--line-index", "--index", str(lif)], "--index can only be used with --range"),
                      (["-d", "--lines", "0:1"], "--lines takes FIRST:COUNT with FIRST from 1, not 0:1"),
                      (["-d", "--lines", "7"], "--lines takes FIRST:COUNT with FIRST from 1, not 7")):
        assert main(argv + [str(src), str(out)], engine=sim_engine) == 1
        assert capsys.readouterr().err.strip() == msg


def test_line_index_text_rejects_malformed():
    blocks = np.array([(32, 9000, 0, 2500, 0xdeadbeef, 0, 9), (9000, 17000, 2500, 2000, 0x1234, 0, 9)], dtype=INDEX_DTYPE)
    good = Bzip2LineIndex(blocks, [7, 3], 11)
    text = good.to_text()
    assert text.splitlines()[:3] == ["# bzip2 line index v1", "# lines 11", "0\t9\t32\t9000\t0\t2500\tdeadbeef\t7"]
    back = Bzip2LineIndex.from_text(text)
    equal_index(back.blocks, blocks)
    assert back.newlines.tolist() == [7, 3] and back.total_lines == 11 and back.total == 4500
    assert Bzip2LineIndex.from_text(text.replace("# lines 11", "# lines 10")).total_lines == 10
    empty = Bzip2LineIndex.from_text("# bzip2 line index v1\n# lines 0\n")
    assert (len(empty), empty.total_lines) == (0, 0)
    lines = text.splitlines()
    for bad in ("", Bzip2Index(blocks).to_text(), text.replace("v1", "v2"), text.replace("# lines 11", "# lines 12"),
                text.replace("# lines 11", "# lines 9"), text.replace("# lines 11", "# lines -1"), text.replace("# lines 11", "#lines 11"),
                "\n".join(lines[:1] + lines[2:]) + "\n", text.replace("\t7\n", "\t2501\n"), text.replace("\t7\n", "\t\n"),
                text.replace("\t7\n", "\t4294967296\n"), text.replace("\t7\n", "\n"), text + "1\t2\n", "# bzip2 line index v1\n# lines 1\n"):
        with pytest.raises(ValueError):
            Bzip2LineIndex.from_text(bad)


def test_debug_line_tile_limits(sim_engine):
    for bad in (100, 8192 + 256, 257):
        with pytest.raises(RuntimeError):
            sim_engine.debug_set_line_tile(bad)
    sim_engine.debug_set_line_tile(8192)
    sim_engine.debug_set_line_tile(0)


# ---- 5. GPU only: sizes a user reads ----
@pytest.mark.gpu
def test_bench_stream_lines(gpu_engine, oracle):
    g = json.load(open(os.path.join(HERE, "golden", "corpus_goldens.json")))["text:100000000:8:L9"]
    src = gen_text(100_000_000, 8).tobytes()
    comp = gpu_engine.compressFile(src, None, 9)
    assert hashlib.sha256(comp).hexdigest() == g["out_sha256"]
    li = gpu_engine.lineIndex(comp)
    lines = model_lines(src)
    assert li.total_lines == len(lines) and li.total == len(src) and len(li) == g["n_blocks"]
    offs = block_starts(li) + [len(src)]
    assert li.newlines.tolist() == [src.count(b"\n", a, b) for a, b in zip(offs, offs[1:])]
    rng = np.random.default_rng(52)
    reqs = [(int(f), 1) for f in rng.integers(0, len(lines), 4096)]
    check_reads(gpu_engine, comp, li, lines, reqs, tiles=(0,))


@pytest.mark.gpu
def test_fifty_megabyte_line(gpu_engine, oracle):
    body = gen_text(50_000_000, 52).tobytes().replace(b"\n", b" ")
    data = b"head\n" + body + b"\ntail"
    comp = gpu_engine.compressFile(data, None, 9)
    li = gpu_engine.lineIndex(comp)
    assert li.total_lines == 3 and len(li) >= 50
    lines = [b"head\n", body + b"\n", b"tail"]
    check_reads(gpu_engine, comp, li, lines, [(1, 1), (0, 1), (2, 1), (0, 3), (0, 2), (1, 2)], tiles=(0,))
