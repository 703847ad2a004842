"""Appending to a stream and its line index: Bzip2Engine.append, bz2b200_zstream_open_append and -z --append.

The model: S = oracle.compress(A, level) under the block cap the case sets (on the oracle and on the engine); appending B
must give S[:keep] + tail == oracle.compress(A + B, level), keep = the last block's bit_begin // 8, and the index
test_compress_index.expected gives for A + B, which the decoder's lineIndex of the result gives too.  The index passed in
is the model's index of S, never one from the code under test.  Every case runs on the simulator and on the GPU (-m gpu),
with both parse kernels, and each case that aims at a boundary asserts that it reaches it."""
import bz2
import ctypes as C
import hashlib
import io
import json
import os

import numpy as np
import pytest

from compressjs_flattened_b200 import _native
from compressjs_flattened_b200.bzip2 import INDEX_DTYPE, Bzip2Engine, Bzip2Error, Bzip2Index, Bzip2LineIndex
from compressjs_flattened_b200.corpus import gen_text
from test_compress_index import check_index, check_reads, expected
from test_lines import model_lines
from test_random_access import equal_index, expected_index

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_SO = os.environ.get("BZ2B200_SIM_LIB") or os.path.join(HERE, "sim", "libbz2b200_sim.so")
RUNLESS = b"abcdefghijklmno\n"   # no byte repeats: a block holds exactly `cap` input bytes

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
    yield e
    e.close()


# ---- the model ----
def model(oracle, data, level, cap):
    """(oracle stream of data, its Bzip2LineIndex, the block index rows)"""
    comp, ix, nl, total = expected(oracle, data, level, cap)
    return comp, Bzip2LineIndex(ix, np.array(nl, dtype=np.uint32), total), ix


def runless(n):
    return (RUNLESS * (n // len(RUNLESS) + 1))[:n]


def check(eng, oracle, A, B, level=9, cap=2500, decoder=True, reads=True, **kw):
    """append B to the oracle's stream of A with the model's index; asserts the result and the index against the model and
    returns (A's block index, the result's)"""
    S, li, ix = model(oracle, A, level, cap)
    want, wix, wnl, wtotal = expected(oracle, A + B, level, cap)
    eng.debug_set_block_cap(cap)
    try:
        keep, tail, got = eng.append(S, B, li, **kw)
    finally:
        eng.debug_set_block_cap(0)
    assert keep == (int(ix[-1]["bit_begin"]) // 8 if len(ix) else 4)
    assert S[:keep] + tail == want, (len(S), keep, len(tail), len(want))
    check_index(got, wix, wnl, wtotal)
    if decoder:
        check_index(eng.lineIndex(want), wix, wnl, wtotal, "decoder")
    if reads and A + B:
        check_reads(eng, want, got, A + B)
    return ix, wix


# ---- 1. levels and empty inputs ----
def test_levels(eng, oracle):
    A, B = gen_text(14_000, 81).tobytes(), gen_text(5_000, 82).tobytes()
    for level in (1, 5, 9):
        ix, wix = check(eng, oracle, A, B, level)
        assert len(ix) >= 5 and set(wix["level"].tolist()) == {level}
    check(eng, oracle, gen_text(130_000, 83).tobytes(), B, 1, cap=0, reads=False)   # the level's own block size


def test_empty_inputs(eng, oracle):
    A = gen_text(9_000, 84).tobytes()
    S, li, _ = model(oracle, A, 9, 2500)
    eng.debug_set_block_cap(2500)
    try:
        keep, tail, got = eng.append(S, b"", li)
    finally:
        eng.debug_set_block_cap(0)
    assert S[:keep] + tail == S                       # nothing appended: the stream itself
    check_index(got, *expected(oracle, A, 9, 2500)[1:])
    B = gen_text(6_000, 85).tobytes()
    for level in (1, 9):
        empty = oracle.compress(b"", level)
        assert len(empty) == 14
        keep, tail, got = eng.append(empty, B, Bzip2LineIndex(np.zeros(0, INDEX_DTYPE), [], 0))
        assert keep == 4 and empty[:4] + tail == oracle.compress(B, level)
        check_index(got, *expected(oracle, B, level)[1:])
        keep, tail, got = eng.append(empty, b"", Bzip2LineIndex(np.zeros(0, INDEX_DTYPE), [], 0))
        assert empty[:keep] + tail == empty and (len(got), got.total_lines) == (0, 0)
    check(eng, oracle, b"", B, 9, cap=2500)


# ---- 2. the cut at the old last block ----
def test_last_block_bit_phases(eng, oracle):
    A, B = gen_text(6_000, 86).tobytes(), gen_text(1_500, 87).tobytes()
    found = {}
    for cap in range(900, 1500, 3):   # the oracle alone finds a cap for every phase of the last block's start
        found.setdefault(int(expected(oracle, A, 9, cap)[1][-1]["bit_begin"]) % 8, cap)
    assert sorted(found) == list(range(8))
    for phase, cap in sorted(found.items()):
        ix, _ = check(eng, oracle, A, B, reads=phase == 3, cap=cap)
        assert int(ix[-1]["bit_begin"]) % 8 == phase


def test_last_block_lengths(eng, oracle):
    B = gen_text(3_000, 87).tobytes()
    for m in (1, 2, 3, 4, 5, 255, 256):
        ix, _ = check(eng, oracle, runless(2 * 2000 + m), B, cap=2000, decoder=m in (1, 256), reads=m == 5)
        assert len(ix) == 3 and int(ix[-1]["out_bytes"]) == m


def test_last_block_full(eng, oracle):
    A, B = runless(3 * 2000), gen_text(3_000, 88).tobytes()
    ix, wix = check(eng, oracle, A, B, cap=2000)
    assert int(ix[-1]["out_bytes"]) == 2000 and len(A) in wix["out_offset"].tolist()   # B starts a block of its own


def _run_cut(oracle, head, run, cap):
    """the first A = head[:k] + run whose last block starts inside the run"""
    for k in range(cap - 40, cap):
        A = head[:k] + run
        o = int(expected(oracle, A, 9, cap)[1][-1]["out_offset"])
        if k < o < len(A) and A[o - 1] == A[o] == run[0]:
            return A
    raise AssertionError("no cut inside the run")


def test_last_block_starts_in_a_run_that_b_continues(eng, oracle):
    A = _run_cut(oracle, runless(3000), b"x" * 600, 2000)
    tail = gen_text(1_000, 89).tobytes()
    for k in (1, 2, 3, 4, 5, 6, 250, 251, 252, 255, 256, 259, 300):
        check(eng, oracle, A, b"x" * k + tail, cap=2000, decoder=k in (1, 300), reads=k == 251)


def test_previous_block_cut_in_a_run(eng, oracle):
    A = _run_cut(oracle, runless(3000), b"\n" * 700, 2000) + gen_text(900, 90).tobytes()
    ix, _ = check(eng, oracle, A, gen_text(2_000, 91).tobytes(), cap=2000)
    o = int(ix[-1]["out_offset"])
    assert A[o - 1] == A[o] == ord("\n")


def test_run_block_as_last_block(eng, oracle):
    A = gen_text(3_000, 92).tobytes() + b"x" * 400_000
    ix = expected(oracle, A, 9, 2500)[1]
    big = int(np.argmax(ix["out_bytes"]))
    A = A[:int(ix[big]["out_offset"] + ix[big]["out_bytes"])]   # ends where a full run block ends
    ix, _ = check(eng, oracle, A, b"x" * 1000 + gen_text(2_000, 93).tobytes(), reads=False)
    assert int(ix[-1]["out_bytes"]) > 40 * 2500 and A[-1] == ord("x")   # the old last block spans many times the cap


# ---- 3. newlines ----
def test_newlines(eng, oracle):
    text = gen_text(8_000, 94).tobytes()
    A = text.rstrip(b"\n")
    for a, b in ((A + b"\n", b"next line\n" * 40), (A, b" continued\n" + text[:2000]), (A + b"\r", b"\n" + text[:3000]),
                 (A + b"\n", text[:3000].replace(b"\n", b" ")), (A, b"no newline here")):
        check(eng, oracle, a, b)


# ---- 4. pieces, steps and repeats ----
def test_pieces_and_steps(eng, oracle):
    A, B = gen_text(10_000, 95).tobytes(), gen_text(6_000, 96).tobytes()
    for piece in (1, 7, 4096):
        check(eng, oracle, A, B[:1500] if piece == 1 else B, piece_bytes=piece, decoder=piece == 7, reads=False)
    check(eng, oracle, A, gen_text(30_000, 97).tobytes(), chunk_bytes=4096, piece_bytes=1000)   # B spans many zstream steps
    sink = io.BytesIO()
    S, li, _ = model(oracle, A, 9, 2500)
    eng.debug_set_block_cap(2500)
    try:
        keep, got, _ = eng.append(S, io.BytesIO(B), li, sink=sink)
    finally:
        eng.debug_set_block_cap(0)
    assert got is sink and S[:keep] + sink.getvalue() == expected(oracle, A + B, 9, 2500)[0]


def test_five_appends_in_a_row(eng, oracle):
    parts = [gen_text(7_000, 98).tobytes()] + [gen_text(n, 99 + n).tobytes() for n in (1, 900, 2600, 40, 3100)]
    S, li, _ = model(oracle, parts[0], 9, 2500)
    eng.debug_set_block_cap(2500)
    try:
        for B in parts[1:]:
            keep, tail, li = eng.append(S, B, li)
            S = S[:keep] + tail
    finally:
        eng.debug_set_block_cap(0)
    data = b"".join(parts)
    want, wix, wnl, wtotal = expected(oracle, data, 9, 2500)
    assert S == want
    check_index(li, wix, wnl, wtotal)
    check_reads(eng, S, li, data)


# ---- 5. multistream and libbz2 ----
def test_multistream(eng, oracle):
    A1, A2, B = gen_text(6_000, 104).tobytes(), gen_text(5_000, 105).tobytes(), gen_text(4_000, 106).tobytes()
    oracle.set_block_cap(1500)
    try:
        s1, s2, s2b = oracle.compress(A1, 9), oracle.compress(A2, 1), oracle.compress(A2 + B, 1)
    finally:
        oracle.set_block_cap(0)

    def line_index(blob, streams, data):
        _, ix = expected_index(oracle, streams, True)
        nl = [data[o:o + n].count(b"\n") for o, n in zip(ix["out_offset"].tolist(), ix["out_bytes"].tolist())]
        return Bzip2LineIndex(ix, np.array(nl, dtype=np.uint32), len(model_lines(data)))

    li = line_index(s1 + s2, [(s1, 9), (s2, 1)], A1 + A2)
    want = line_index(s1 + s2b, [(s1, 9), (s2b, 1)], A1 + A2 + B)
    eng.debug_set_block_cap(1500)
    try:
        keep, tail, got = eng.append(s1 + s2, B, li)
    finally:
        eng.debug_set_block_cap(0)
    assert (s1 + s2)[:keep] + tail == s1 + s2b
    check_index(got, want.blocks.entries, want.newlines.tolist(), want.total_lines)
    new = got.blocks.entries[len(li) - 1:]
    assert len(new) >= 2 and set(new["stream"].tolist()) == {1} and set(new["level"].tolist()) == {1}
    check_index(eng.lineIndex(s1 + s2b, multistream=True), want.blocks.entries, want.newlines.tolist(), want.total_lines)


def test_libbz2_stream(eng, oracle):
    A, B = gen_text(230_000, 107).tobytes(), gen_text(20_000, 108).tobytes()
    S = bz2.compress(A, 1)
    _, ix = expected_index(oracle, [(S, 1)], False)
    assert len(ix) >= 3
    nl = [A[o:o + n].count(b"\n") for o, n in zip(ix["out_offset"].tolist(), ix["out_bytes"].tolist())]
    keep, tail, got = eng.append(S, B, Bzip2LineIndex(ix, np.array(nl, dtype=np.uint32), len(model_lines(A))))
    out = S[:keep] + tail
    assert keep == int(ix[-1]["bit_begin"]) // 8 and out[:keep] == S[:keep]
    assert bz2.decompress(out) == A + B == eng.decompressFile(out)
    _, wix = expected_index(oracle, [(out, 1)], False)
    wnl = [(A + B)[o:o + n].count(b"\n") for o, n in zip(wix["out_offset"].tolist(), wix["out_bytes"].tolist())]
    check_index(got, wix, wnl, len(model_lines(A + B)))
    assert got.blocks.entries[:len(ix) - 1].tolist() == ix[:len(ix) - 1].tolist()


# ---- 6. errors ----
def c_open(eng, blob, li, count=None, newlines=True):
    """bz2b200_zstream_open_append called directly: (rc, zstream handle or None, keep)"""
    a = np.frombuffer(blob, dtype=np.uint8)
    ix = np.ascontiguousarray(li.blocks.entries, dtype=INDEX_DTYPE)
    nl = np.ascontiguousarray(li.newlines, dtype=np.uint32)
    h, keep = C.c_void_p(), C.c_uint64(7)
    rc = eng._L.bz2b200_zstream_open_append(eng._ctx, a.ctypes.data, a.size, ix.ctypes.data, nl.ctypes.data if newlines else None,
                                            len(ix) if count is None else count, li.total_lines, 0, C.byref(h), C.byref(keep))
    if h:
        eng._L.bz2b200_zstream_close(h)
    return rc, h.value, keep.value


def expect_error(eng, blob, li, rc, text, **kw):
    got, h, keep = c_open(eng, blob, li, **kw)
    assert (got, h, keep) == (rc, None, 0)
    assert text in eng._L.bz2b200_last_error(eng._ctx).decode()


def test_errors(eng, oracle):
    A = gen_text(9_000, 109).tobytes()
    S, li, ix = model(oracle, A, 9, 2500)
    eng.debug_set_block_cap(2500)
    try:
        assert c_open(eng, S, li)[0] == 0

        def edited(field=None, k=-1, delta=1, nl_delta=0, lines_delta=0):
            e = li.blocks.entries.copy()
            if field:
                e[field][k] += delta
            nl = li.newlines.copy()
            nl[-1] = int(nl[-1]) + nl_delta
            return Bzip2LineIndex(e, nl, li.total_lines + lines_delta)
        stale = "index does not match the input"
        # a stale index: a wrong CRC (the last block's, or an earlier one's), a wrong bit_end, a wrong '\n' count
        expect_error(eng, S, edited("crc"), -5, stale)
        expect_error(eng, S, edited("crc", k=1), -5, stale)
        expect_error(eng, S, edited("bit_end"), -5, "no end-of-stream signature")
        assert li.newlines[-1] > 0
        expect_error(eng, S, edited(nl_delta=-1, lines_delta=-1), -5, "'\\n' bytes, the index gives")
        # a footer CRC that does not match its blocks
        bad, q = bytearray(S), int(ix[-1]["bit_end"]) + 48
        bad[q // 8] ^= 0x80 >> (q % 8)
        expect_error(eng, bytes(bad), li, -5, "the stream CRC")
        # bytes after the footer: trailing data, a second (empty) stream, a second stream the index does not cover
        for extra in (b"junk", oracle.compress(b"", 9), oracle.compress(b"more", 1)):
            expect_error(eng, S + extra, li, _native.E_ARG, f"{len(extra)} bytes follow the end")
        # a malformed index
        expect_error(eng, S, edited("out_offset", k=1), _native.E_ARG, "out_offset not contiguous")
        expect_error(eng, S, edited("level", delta=5), _native.E_ARG, "level outside 1..9")
        expect_error(eng, S, edited(lines_delta=2), _native.E_ARG, "total_lines")
        expect_error(eng, S, edited(nl_delta=100_000), _native.E_ARG, "above the block's out_bytes")
        # count == 0 on a non-empty stream, and newlines missing
        empty = Bzip2LineIndex(np.zeros(0, INDEX_DTYPE), [], 0)
        expect_error(eng, S, empty, _native.E_ARG, "an empty index describes only an empty stream")
        expect_error(eng, oracle.compress(b"", 9) + b"x", empty, _native.E_ARG, "an empty index describes only an empty stream")
        expect_error(eng, S, li, _native.E_ARG, "newlines is required", newlines=False)
    finally:
        eng.debug_set_block_cap(0)
    a = np.frombuffer(S, dtype=np.uint8)
    h, keep = C.c_void_p(), C.c_uint64()
    assert eng._L.bz2b200_zstream_open_append(None, a.ctypes.data, a.size, None, None, 0, 0, 0, C.byref(h), C.byref(keep)) == _native.E_ARG
    assert eng._L.bz2b200_zstream_open_append(eng._ctx, a.ctypes.data, a.size, None, None, 0, 0, 0, None, C.byref(keep)) == _native.E_ARG
    assert eng._L.bz2b200_zstream_open_append(eng._ctx, a.ctypes.data, a.size, None, None, 0, 0, 0, C.byref(h), None) == _native.E_ARG
    # in Python: a block index is refused, an argument error raises RuntimeError, a stale index Bzip2Error
    with pytest.raises(TypeError, match="needs a line index"):
        eng.append(S, b"x", li.blocks)
    with pytest.raises(RuntimeError, match="bytes follow the end"):
        eng.append(S + b"junk", b"x", li)
    with pytest.raises(Bzip2Error, match=stale) as e:
        eng.append(S, b"x", edited("crc"))
    assert e.value.errorCode == -5


def test_path_and_built_index(eng, oracle, tmp_path):
    A, B = gen_text(8_000, 110).tobytes(), gen_text(3_000, 111).tobytes()
    S = oracle.compress(A, 9)
    p = tmp_path / "a.bz2"
    p.write_bytes(S)
    keep, tail, got = eng.append(str(p), B)   # memory-mapped, and the index built by lineIndex
    want, wix, wnl, wtotal = expected(oracle, A + B, 9)
    assert S[:keep] + tail == want
    check_index(got, wix, wnl, wtotal)


# ---- 7. the command line ----
def test_command_line(sim_engine, oracle, tmp_path, capsys):
    from compressjs_flattened_b200.__main__ import main
    A, B1, B2 = gen_text(12_000, 112).tobytes(), gen_text(4_000, 113).tobytes(), gen_text(5_000, 114).tobytes()
    src, bz, lif, b1, b2 = (tmp_path / n for n in ("a.txt", "a.bz2", "a.lines", "b1.txt", "b2.txt"))
    src.write_bytes(A)
    b1.write_bytes(B1)
    b2.write_bytes(B2)
    assert main(["-z", "-9", "--index-out", str(lif), str(src), str(bz)], engine=sim_engine) == 0
    assert main(["-z", "--append", str(bz), str(b1)], engine=sim_engine) == 0   # without --index: built from the file
    assert bz.read_bytes() == oracle.compress(A + B1, 9)
    assert main(["-z", "--index-out", str(lif), "--append", str(bz), str(b1)], engine=sim_engine) == 0
    assert main(["-z", "--append", str(bz), "--index", str(lif), "--index-out", str(lif), str(b2)], engine=sim_engine) == 0
    data = A + B1 + B1 + B2
    comp = bz.read_bytes()
    assert comp == oracle.compress(data, 9)
    assert lif.read_text() == sim_engine.lineIndex(comp).to_text()
    check_index(Bzip2LineIndex.from_text(lif.read_text()), *expected(oracle, data, 9)[1:])
    assert sorted(os.listdir(tmp_path)) == ["a.bz2", "a.lines", "a.txt", "b1.txt", "b2.txt"]   # no temporary file left
    # refusals: exit status 1, FILE untouched
    capsys.readouterr()
    before = hashlib.sha256(bz.read_bytes()).hexdigest()
    bif = tmp_path / "a.idx"
    bif.write_text(Bzip2Index(sim_engine.lineIndex(comp).blocks.entries).to_text())
    for extra, msg in ((["-d"], "--append can only be used with -z, not with -d"), (["--list"], "not with --list"), (["--range", "0:1"], "not with --range"),
                       (["--grep", "a"], "not with --grep"), (["--line-index"], "not with --line-index"), (["--lines", "1:1"], "not with --lines"),
                       (["--recover"], "not with --recover"), (["-b", "32"], "not with -b"), (["-9"], "compression level has no effect"),
                       ([str(b1), str(tmp_path / "out")], "takes no outfile"), (["--index", str(bif), str(b1)], "needs a line index")):
        assert main(["-z", "--append", str(bz)] + extra, engine=sim_engine) == 1, extra
        assert msg in capsys.readouterr().err, extra
    assert not (tmp_path / "out").exists()
    # a failing append (a stale index) leaves FILE as it was
    stale = Bzip2LineIndex.from_text(lif.read_text())
    stale.blocks.entries["crc"][-1] ^= 1
    lif.write_text(stale.to_text())
    with pytest.raises(Bzip2Error, match="index does not match the input"):
        main(["-z", "--append", str(bz), "--index", str(lif), str(b1)], engine=sim_engine)
    assert hashlib.sha256(bz.read_bytes()).hexdigest() == before
    assert sorted(os.listdir(tmp_path)) == ["a.bz2", "a.idx", "a.lines", "a.txt", "b1.txt", "b2.txt"]


# ---- 8. GPU only: sizes a user appends ----
def _gpu_check(eng, out, li, data):
    """the result is compressFile(A + B) and the index counts the input's '\\n' bytes block by block"""
    assert out == eng.compressFile(data, None, 9)
    assert li.total == len(data) and li.total_lines == len(model_lines(data))
    offs = li.blocks.entries["out_offset"].tolist() + [len(data)]
    assert li.newlines.tolist() == [data.count(b"\n", a, b) for a, b in zip(offs, offs[1:])]
    ref = eng.lineIndex(out)
    equal_index(li.blocks, ref.blocks.entries)
    assert li.newlines.tolist() == ref.newlines.tolist()


@pytest.mark.gpu
def test_gpu_bench_stream(gpu_engine):
    g = json.load(open(os.path.join(HERE, "golden", "corpus_goldens.json")))["text:100000000:8:L9"]
    A = gen_text(100_000_000, 8).tobytes()
    S, li = gpu_engine.compressIndexed(A, 9)
    assert hashlib.sha256(S).hexdigest() == g["out_sha256"]
    for n, seed in ((1_000_000, 115), (100_000_000, 116)):
        B = gen_text(n, seed).tobytes()
        keep, tail, got = gpu_engine.append(S, B, li)
        assert keep == int(li.blocks.entries[-1]["bit_begin"]) // 8
        _gpu_check(gpu_engine, S[:keep] + tail, got, A + B)


@pytest.mark.gpu
def test_gpu_run_block_as_last_block(gpu_engine):
    _, li = gpu_engine.compressIndexed(bytes(60_000_000), 9)
    first = int(li.blocks.entries[0]["out_bytes"])   # a full block of zeros: ~46 MB of input
    assert first > 40_000_000
    A = bytes(first)
    S, li = gpu_engine.compressIndexed(A, 9)
    assert len(li) == 1
    B = bytes(1000) + gen_text(2_000_000, 117).tobytes()
    keep, tail, got = gpu_engine.append(S, B, li)
    _gpu_check(gpu_engine, S[:keep] + tail, got, A + B)
