"""The line index as a by-product of compression: Bzip2Engine.compressIndexed, Bzip2Pool.compressIndexed,
compressStream(..., index=True) and -z --index-out (bz2b200_compress_indexed, bz2b200_pool_compress_indexed,
bz2b200_zstream_open_indexed / bz2b200_zstream_index in include/bz2b200.h).

Expected values come from the oracle and the input, never from the code under test: the stream from oracle.compress
(under the block cap the case sets), the block index from test_random_access.expected_index, the '\\n' bytes of every
block from data[out_offset:out_offset + out_bytes].count(b"\\n") over the oracle's rows, total_lines from
test_lines.model_lines.  Every case also checks the plain call of the same entry point (same stream), the decoder's
lineIndex of the stream (same index, except for a D1 stream, which the reference's decoder rejects), and reads lines and
ranges with the returned index.  Each runs with the default and with 256-byte segments of the '\\n' count, on the
simulator and on the GPU (-m gpu)."""
import ctypes as C
import hashlib
import io
import json
import os

import numpy as np
import pytest

from compressjs_flattened_b200 import _native
from compressjs_flattened_b200.bzip2 import INDEX_DTYPE, Bzip2Engine, Bzip2Index, Bzip2LineIndex
from compressjs_flattened_b200.corpus import gen_text
from compressjs_flattened_b200.pool import Bzip2Pool
from test_compress_conformance import _rle1, _sections
from test_lines import model_lines
from test_random_access import equal_index, expected_index
from test_recover import footer_pos

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_SO = os.environ.get("BZ2B200_SIM_LIB") or os.path.join(HERE, "sim", "libbz2b200_sim.so")
SEGS = (0, 256)
B9 = 899_981


def _ngpu():
    import torch
    return torch.cuda.device_count()


@pytest.fixture(params=["sim", pytest.param("gpu", marks=pytest.mark.gpu)])
def eng(request):
    if request.param == "sim":
        request.getfixturevalue("sim_engine")   # builds the simulator library when it is stale
        e = Bzip2Engine(0, _native.Library(SIM_SO))
    else:
        e = Bzip2Engine(0)
    e.on_gpu = request.param == "gpu"
    yield e
    e.close()


# ---- the model ----
def expected(oracle, data, level=9, cap=0, with_d1=False):
    """(oracle stream, its block index, the '\\n' bytes of every block, total_lines[, whether the oracle reached D1])"""
    oracle.set_block_cap(cap)
    try:
        comp, st = oracle.compress(data, level, return_stats=True)
    finally:
        oracle.set_block_cap(0)
    _, ix = expected_index(oracle, [(comp, level)], False)
    nl = [data[o:o + n].count(b"\n") for o, n in zip(ix["out_offset"].tolist(), ix["out_bytes"].tolist())]
    return (comp, ix, nl, len(model_lines(data))) + ((bool(st.d1_triggered),) if with_d1 else ())


def check_index(li, ix, nl, total, label=""):
    assert isinstance(li, Bzip2LineIndex), label
    equal_index(li.blocks, ix)
    assert li.newlines.dtype == np.uint32 and li.newlines.tolist() == nl, label
    assert li.total_lines == total, label


def check_reads(eng, comp, li, data):
    """lines and ranges read with the returned index are the model's"""
    lines = model_lines(data)
    L = len(lines)
    reqs = [(0, 1), (L - 1, 1), (L // 2, 3), (0, L)] + [(i, 2) for i in range(0, L, max(1, L // 23))]
    assert eng.decompressLines(comp, li, reqs) == [b"".join(lines[f:f + k]) for f, k in reqs]
    n = len(data)
    rs = [(0, n), (n // 3, 1000), (max(0, n - 7), 7)] + [(int(o) - 3, 6) for o in li.blocks.entries["out_offset"][1:]]
    assert eng.decompressRanges(comp, li, rs) == [data[slice(s, s + k)] for s, k in rs]


def check(eng, oracle, data, level=9, cap=0, batch=0, reads=True, segs=SEGS):
    """compressIndexed against the model, the plain compressFile and (but for a D1 stream, which the reference's decoder
    rejects: a one-byte input is one) the decoder; returns the expectations"""
    comp, ix, nl, total, d1 = expected(oracle, data, level, cap, with_d1=True)
    eng.debug_set_block_cap(cap)
    eng.debug_set_batch_blocks(batch)
    try:
        for seg in segs:
            eng.debug_set_line_tile(seg)
            got, li = eng.compressIndexed(data, level)
            assert got == comp, (seg, len(got), len(comp))
            check_index(li, ix, nl, total, seg)
            flagged = eng.stats().d1_triggered
        eng.debug_set_line_tile(0)
        assert eng.compressFile(data, None, level) == comp and eng.stats().d1_triggered == flagged
    finally:
        eng.debug_set_line_tile(0)
        eng.debug_set_block_cap(0)
        eng.debug_set_batch_blocks(0)
    if not d1:
        check_index(eng.lineIndex(comp), ix, nl, total, "decoder")
        if reads and len(data):
            check_reads(eng, comp, li, data)
    return comp, ix, nl, total


# ---- 1. levels and small inputs ----
def test_levels(eng, oracle):
    text = gen_text(14_000, 61).tobytes()
    for level in (1, 5, 9):
        _, ix, _, _ = check(eng, oracle, text, level, cap=2500)
        assert len(ix) >= 5 and set(ix["level"].tolist()) == {level} and not ix["stream"].any()
    check(eng, oracle, gen_text(120_000, 62).tobytes(), 1)   # the level's own block size


def test_small_inputs(eng, oracle):
    text = gen_text(9_000, 63).tobytes()
    cases = [b"a", b"\n", b"\n\n", text.replace(b"\n", b" "), text.replace(b"\n", b"\r\n"), text.rstrip(b"\n") + b"\n",
             text.rstrip(b"\n") + b"tail"]
    for data in cases:
        _, ix, nl, total = check(eng, oracle, data, 9, cap=2500)
        assert total == data.count(b"\n") + (not data.endswith(b"\n"))
    comp, li = eng.compressIndexed(b"", 9)
    assert len(comp) == 14 and (len(li), li.total_lines, li.total) == (0, 0, 0)
    check(eng, oracle, b"", 9)
    assert check(eng, oracle, text.replace(b"\n", b" "), 9, cap=2500)[3] == 1


# ---- 2. block edges ----
def test_newline_at_block_edges(eng, oracle):
    # 10-byte lines, 2500-byte blocks: every block ends with '\n'; shifted by one, every block starts with one
    for shift in (0, 1):
        data = b"\n" * shift + b"abcdefghi\n" * 1500
        _, ix, _, _ = check(eng, oracle, data, 9, cap=2500)
        offs = ix["out_offset"].tolist()[1:]
        assert len(offs) >= 4
        assert all(data[o - 1 + shift] == ord("\n") for o in offs)


def test_aligned_and_unaligned_block_starts(eng, oracle):
    data = b"abcdefghijklmno\n" * 1200   # no runs: a block holds exactly `cap` input bytes
    starts = []
    for cap in (2048, 2500):
        starts += check(eng, oracle, data, 9, cap=cap)[1]["out_offset"].tolist()[1:]
    assert any(s % 16 == 0 for s in starts) and any(s % 16 for s in starts)


def test_newline_runs_across_cuts(eng, oracle):
    text = gen_text(6_000, 64).tobytes()
    data = text[:2000] + b"\n" * 100_000 + text[2000:] + b"\n" * 700
    _, ix, nl, _ = check(eng, oracle, data, 9, cap=2500)
    inside = [o for o in ix["out_offset"].tolist()[1:] if data[o - 1:o + 1] == b"\n\n"]
    assert inside   # a cut inside a run of '\n' longer than 4 + 255
    check(eng, oracle, b"\n" * 300_000, 9, cap=2500)


def test_run_heavy_block(eng, oracle):
    data = gen_text(3_000, 65).tobytes() + b"x" * 400_000 + b"\n" * 200_000 + gen_text(3_000, 66).tobytes()
    _, ix, nl, _ = check(eng, oracle, data, 9, cap=2500)
    assert int(ix["out_bytes"].max()) > 40 * 2500   # one block spans many times the cap (and many 256-byte segments)
    assert max(nl) > 40 * 2500


def test_batches(eng, oracle):
    data = gen_text(40_000, 67).tobytes()
    for batch in (1, 3):
        _, ix, _, _ = check(eng, oracle, data, 9, cap=2500, batch=batch, reads=batch == 3)
        assert len(ix) > 3 * batch


# ---- 3. the context's own two-lane pool ----
def test_own_pool_route(eng, oracle):
    data = gen_text(30_000, 68).tobytes()
    data = data[:9000] + b"\n" * 4000 + data[9000:]   # a shard boundary inside a run
    eng.debug_set_pool(min_bytes=1, shard_bytes=7000)
    try:
        _, ix, _, _ = check(eng, oracle, data, 9, cap=2500)
        check(eng, oracle, data, 1, cap=997, batch=2, reads=False)
        assert eng.stats().n_blocks == len(expected(oracle, data, 1, 997)[1])
    finally:
        eng.debug_set_pool()
    assert len(ix) > 6


# ---- 4. pools ----
POOLS = [pytest.param(("sim", (0, 0), 2), id="sim-2x2"), pytest.param(("sim", (0,), 3), id="sim-1x3"),
         pytest.param(("gpu", (0,), 2), id="gpu-1x2", marks=pytest.mark.gpu),
         pytest.param(("gpu", (0, 1), 2), id="gpu-2x2", marks=pytest.mark.gpu)]


@pytest.fixture(params=POOLS)
def pool(request):
    where, devices, lanes = request.param
    if where == "sim":
        request.getfixturevalue("sim_engine")
        lib = _native.Library(SIM_SO)
    else:
        if len(devices) > _ngpu():
            pytest.skip(f"needs {len(devices)} GPUs")
        lib = None
    p = Bzip2Pool(list(devices), lanes, library=lib)
    p.eng = Bzip2Engine(0, lib)
    yield p
    p.eng.close()
    p.close()


def test_pool_compress_indexed(pool, oracle):
    text = gen_text(36_000, 69).tobytes()
    data = text[:5000] + b"\n" * 3000 + text[5000:20_000] + b"z" * 9000 + text[20_000:]
    for cap, batch, shard in ((2500, 0, 4096), (1800, 3, 6000), (2500, 1, 0)):
        comp, ix, nl, total = expected(oracle, data, 9, cap)
        pool.debug(block_cap=cap, batch_blocks=batch)
        try:
            got, li = pool.compressIndexed(data, 9, shard_bytes=shard)
            assert got == comp == pool.compressFile(data, None, 9, shard_bytes=shard)
        finally:
            pool.debug()
        check_index(li, ix, nl, total, (cap, batch, shard))
        assert pool.stats().ms_stage[5] >= 0
        if shard:   # a shard whose first block starts inside a run
            offs = ix["out_offset"].tolist()
            firsts = [next(o for o in offs if o >= b) for b in range(shard, len(data), shard) if b < offs[-1]]
            assert any(0 < o < len(data) and data[o - 1] == data[o] and o % shard for o in firsts)
    check_index(pool.eng.lineIndex(comp), ix, nl, total)
    check_reads(pool.eng, comp, li, data)
    got, li = pool.compressIndexed(b"", 5)
    assert got == oracle.compress(b"", 5) and (len(li), li.total_lines) == (0, 0)
    with pytest.raises(ValueError):
        pool.compressIndexed(data, 10)


# ---- 5. the stream flavour ----
def test_zstream_indexed(eng, oracle):
    data = gen_text(20_000, 70).tobytes() + b"\n" * 3000 + gen_text(6_000, 71).tobytes().rstrip(b"\n")
    comp, ix, nl, total = expected(oracle, data, 9, 2500)
    eng.debug_set_block_cap(2500)
    try:
        for chunk, piece in ((4096, 1), (6000, 7), (9000, 4096), (1 << 20, 4096)):
            if piece == 1 and len(data) > 12_000 and not eng.on_gpu:
                src = data[:12_000]
                want = expected(oracle, src, 9, 2500)
            else:
                src, want = data, (comp, ix, nl, total)
            got, li = eng.compressStream(io.BytesIO(src), None, 9, chunk_bytes=chunk, piece_bytes=piece, index=True)
            assert got == want[0] == eng.compressStream(io.BytesIO(src), None, 9, chunk_bytes=chunk, piece_bytes=piece), (chunk, piece)
            check_index(li, *want[1:], (chunk, piece))
        sink = io.BytesIO()
        assert eng.compressStream(io.BytesIO(data), sink, 9, chunk_bytes=5000, index=True)[0] is sink and sink.getvalue() == comp
        got, li = eng.compressStream(b"", None, 9, index=True)
        assert got == oracle.compress(b"", 9) and (len(li), li.total_lines) == (0, 0)
    finally:
        eng.debug_set_block_cap(0)


def c_zindex(eng, h, null=None):
    outs = [C.POINTER(_native.BlockEntry)(), C.POINTER(C.c_uint32)(), C.c_size_t(), C.c_uint64()]
    args = [None if i == null else C.byref(o) for i, o in enumerate(outs)]
    rc = eng._L.bz2b200_zstream_index(h, *args)
    if rc == 0:
        eng._L.bz2b200_free(outs[0])
        eng._L.bz2b200_free(outs[1])
    return rc


def test_zstream_index_errors(eng):
    L = eng._L
    out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
    data = np.frombuffer(b"one\ntwo\n", dtype=np.uint8)
    for opener in (L.bz2b200_zstream_open, L.bz2b200_zstream_open_indexed):
        h = C.c_void_p()
        assert opener(eng._ctx, 9, 0, C.byref(h)) == 0
        try:
            assert L.bz2b200_zstream_feed(h, data.ctypes.data, data.size, C.byref(out), C.byref(n)) == 0
            eng._take(out, n.value)
            assert c_zindex(eng, h) == _native.E_ARG
            msg = L.bz2b200_last_error(eng._ctx).decode()
            assert ("after bz2b200_zstream_finish" if opener is L.bz2b200_zstream_open_indexed else "not opened with") in msg
            assert L.bz2b200_zstream_finish(h, C.byref(out), C.byref(n)) == 0
            eng._take(out, n.value)
            if opener is L.bz2b200_zstream_open:
                assert c_zindex(eng, h) == _native.E_ARG and "not opened with" in L.bz2b200_last_error(eng._ctx).decode()
            else:
                for k in range(4):
                    assert c_zindex(eng, h, null=k) == _native.E_ARG
                assert c_zindex(eng, h) == 0
        finally:
            L.bz2b200_zstream_close(h)
    assert L.bz2b200_zstream_open_indexed(eng._ctx, 0, 0, C.byref(C.c_void_p())) == _native.E_LEVEL
    assert L.bz2b200_zstream_open_indexed(eng._ctx, 9, 0, None) == _native.E_ARG
    assert L.bz2b200_zstream_index(None, None, None, None, None) == _native.E_ARG


# ---- 6. defect D1 ----
def test_d1_stream_and_input_index(eng, oracle):
    for seed in range(40):
        data = _sections(np.random.default_rng(2000 + seed), 2, 40, 120)
        st = oracle.block_stages(_rle1(oracle, data, B9)[0])
        if st["d1"] and st["alpha"] + 2 < st["n_groups"]:
            break
    else:
        raise AssertionError("no D1 case")
    comp, exp_st = oracle.compress(data, 9, return_stats=True)
    assert exp_st.d1_triggered
    starts, _, crcs = oracle.cut_points(np.frombuffer(data, np.uint8), 9)
    assert len(crcs) == 1   # one block: it starts after the header and ends at the end-of-stream signature
    ix = np.array([(32, footer_pos(comp), 0, len(data), int(crcs[0]), 0, 9)], dtype=INDEX_DTYPE)
    for seg in SEGS:
        eng.debug_set_line_tile(seg)
        got, li = eng.compressIndexed(data, 9)
        assert got == comp and eng.stats().d1_triggered
        check_index(li, ix, [data.count(b"\n")], len(model_lines(data)))
    eng.debug_set_line_tile(0)


# ---- 7. argument errors ----
def c_indexed(eng, data, level, null=None, pool=None):
    a = np.frombuffer(data, dtype=np.uint8)
    outs = [C.POINTER(C.c_uint8)(), C.c_size_t(), C.POINTER(_native.BlockEntry)(), C.POINTER(C.c_uint32)(), C.c_size_t(), C.c_uint64()]
    args = [None if i == null else C.byref(o) for i, o in enumerate(outs)]
    if pool is None:
        rc = eng._L.bz2b200_compress_indexed(eng._ctx, a.ctypes.data if a.size else None, a.size, level, *args)
    else:
        rc = pool._L.bz2b200_pool_compress_indexed(pool._p, a.ctypes.data if a.size else None, a.size, level, 0, *args)
    if rc == 0:
        for p in (outs[0], outs[2], outs[3]):
            eng._L.bz2b200_free(p)
    return rc, outs


def test_argument_errors(eng):
    data = b"abc\ndef\n"
    pool = Bzip2Pool([0], 2, library=eng._lib)
    try:
        for target in (None, pool):
            assert c_indexed(eng, data, 9, pool=target)[0] == 0
            for k in range(6):
                rc, outs = c_indexed(eng, data, 9, null=k, pool=target)
                assert rc == _native.E_ARG and not outs[0] and not outs[2] and not outs[3]
            for level in (0, 10, -1):
                rc, outs = c_indexed(eng, data, level, pool=target)
                assert rc == _native.E_LEVEL and not outs[0] and not outs[2]
        assert eng._L.bz2b200_compress_indexed(None, None, 0, 9, *([None] * 6)) == _native.E_ARG
        assert eng._L.bz2b200_pool_compress_indexed(None, None, 0, 9, 0, *([None] * 6)) == _native.E_ARG
        a = C.POINTER(C.c_uint8)()
        rc = eng._L.bz2b200_compress_indexed(eng._ctx, None, 5, 9, C.byref(a), C.byref(C.c_size_t()), C.byref(C.POINTER(_native.BlockEntry)()),
                                             C.byref(C.POINTER(C.c_uint32)()), C.byref(C.c_size_t()), C.byref(C.c_uint64()))
        assert rc == _native.E_ARG and not a
        for bad in (0, 10, 2.5, "9"):
            if isinstance(bad, str):
                assert eng.compressIndexed(data, bad)[0] == eng.compressFile(data, None, 9)   # props that are not a number: level 9
                continue
            for call in (lambda: eng.compressIndexed(data, bad), lambda: pool.compressIndexed(data, bad),
                         lambda: eng.compressStream(data, None, bad, index=True)):
                with pytest.raises(ValueError, match="Invalid block size multiplier"):
                    call()
    finally:
        pool.close()


# ---- 8. a line index where a block index is taken ----
def test_line_index_where_block_index_is_taken(eng, oracle):
    data = gen_text(12_000, 72).tobytes()
    eng.debug_set_block_cap(2500)
    try:
        comp, li = eng.compressIndexed(data, 9)
    finally:
        eng.debug_set_block_cap(0)
    assert eng.decompressRange(comp, li, 3000, 4000) == data[3000:7000] == eng.decompressRange(comp, li.blocks, 3000, 4000)
    f = eng.open(comp, index=li)
    f.seek(5000)
    assert f.read(3000) == data[5000:8000] and f.read() == data[8000:]


# ---- 9. the command line ----
def test_command_line_index_out(sim_engine, oracle, tmp_path, capsys):
    from compressjs_flattened_b200.__main__ import main
    data = gen_text(30_000, 73).tobytes().rstrip(b"\n") + b" end"
    src, bz, lif, out = tmp_path / "in.txt", tmp_path / "in.bz2", tmp_path / "in.lines", tmp_path / "out"
    src.write_bytes(data)
    for level in (1, 9):
        assert main(["-z", f"-{level}", "--index-out", str(lif), str(src), str(bz)], engine=sim_engine) == 0
        comp = bz.read_bytes()
        assert comp == oracle.compress(data, level)
        text = lif.read_text()
        li = Bzip2LineIndex.from_text(text)
        _, ix, nl, total = expected(oracle, data, level)
        check_index(li, ix, nl, total)
        assert text == sim_engine.lineIndex(comp).to_text()
    lines = model_lines(data)
    assert main(["-d", "--lines", "5:3", "--index", str(lif), str(bz), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == b"".join(lines[4:7])
    assert main(["-d", "--lines", f"{len(lines)}:1", "--index", str(lif), str(bz), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == lines[-1]
    assert main(["-d", "--range", "1000:5000", "--index", str(lif), str(bz), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == data[1000:6000]
    bif = tmp_path / "in.idx"
    bif.write_text(Bzip2Index(expected(oracle, data, 9)[1]).to_text())
    assert main(["-d", "--range", "7:9", "--index", str(bif), str(bz), str(out)], engine=sim_engine) == 0   # the block index still works
    assert out.read_bytes() == data[7:16]
    capsys.readouterr()
    for extra, flag in ((["-d"], "-d"), (["--list"], "--list"), (["--range", "0:1"], "--range"), (["--grep", "a"], "--grep"),
                        (["--line-index"], "--line-index"), (["--lines", "1:1"], "--lines"), (["--recover"], "--recover"),
                        (["-b", "32"], "-b"), (["-d", "-b", "32"], "-d")):
        assert main(["--index-out", str(tmp_path / "x")] + extra + [str(bz), str(out)], engine=sim_engine) == 1
        assert capsys.readouterr().err.strip() == f"--index-out can only be used with -z, not with {flag}"
    assert not (tmp_path / "x").exists()


# ---- 10. GPU only: sizes a user compresses ----
def _gpu_check(eng, comp, li, data, decoder=True):
    assert li.total == len(data) and li.total_lines == len(model_lines(data))
    offs = li.blocks.entries["out_offset"].tolist() + [len(data)]
    assert li.newlines.tolist() == [data.count(b"\n", a, b) for a, b in zip(offs, offs[1:])]
    if decoder:
        ref = eng.lineIndex(comp)
        equal_index(li.blocks, ref.blocks.entries)
        assert li.newlines.tolist() == ref.newlines.tolist() and li.total_lines == ref.total_lines


@pytest.mark.gpu
def test_gpu_bench_input(gpu_engine):
    g = json.load(open(os.path.join(HERE, "golden", "corpus_goldens.json")))["text:100000000:8:L9"]
    src = gen_text(100_000_000, 8).tobytes()
    comp, li = gpu_engine.compressIndexed(src, 9)
    assert hashlib.sha256(comp).hexdigest() == g["out_sha256"] and len(li) == g["n_blocks"]
    assert gpu_engine.stats().ms_stage[5] > 0
    _gpu_check(gpu_engine, comp, li, src)
    lines = model_lines(src)
    rng = np.random.default_rng(74)
    reqs = [(int(f), 1) for f in rng.integers(0, len(lines), 2048)]
    assert gpu_engine.decompressLines(comp, li, reqs) == [lines[f] for f, _ in reqs]


@pytest.mark.gpu
def test_gpu_one_gigabyte_own_pool(gpu_engine):
    src = np.tile(gen_text(100_000_000, 8), 10).tobytes()
    comp, li = gpu_engine.compressIndexed(src, 9)
    assert comp == gpu_engine.compressFile(src, None, 9)
    _gpu_check(gpu_engine, comp, li, src)


@pytest.mark.gpu
def test_gpu_pools(oracle):
    src = gen_text(60_000_000, 75).tobytes()
    ref = Bzip2Engine(0)
    comp, li = ref.compressIndexed(src, 9)
    pools = [Bzip2Pool([0], 2)] + ([Bzip2Pool(list(range(_ngpu())), 2)] if _ngpu() >= 2 else [])
    try:
        for p in pools:
            for shard in (0, 7_000_000):
                got, pli = p.compressIndexed(src, 9, shard_bytes=shard)
                assert got == comp
                equal_index(pli.blocks, li.blocks.entries)
                assert pli.newlines.tolist() == li.newlines.tolist() and pli.total_lines == li.total_lines
        _gpu_check(ref, comp, li, src)
    finally:
        for p in pools:
            p.close()
        ref.close()


@pytest.mark.gpu
def test_gpu_fifty_megabyte_line_and_zeros(gpu_engine):
    data = b"head\n" + gen_text(50_000_000, 76).tobytes().replace(b"\n", b" ") + b"\ntail"
    comp, li = gpu_engine.compressIndexed(data, 9)
    _gpu_check(gpu_engine, comp, li, data)
    assert li.total_lines == 3
    zeros = bytes(200_000_000)   # run blocks of ~46 MB of input each
    comp, li = gpu_engine.compressIndexed(zeros, 9)
    assert int(li.blocks.entries["out_bytes"].max()) > 40_000_000 and li.total_lines == 1
    _gpu_check(gpu_engine, comp, li, zeros)
    comp, li = gpu_engine.compressStream(io.BytesIO(data), None, 9, chunk_bytes=16 << 20, index=True)
    _gpu_check(gpu_engine, comp, li, data, decoder=False)
