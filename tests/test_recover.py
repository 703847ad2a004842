"""Recovery of damaged files (Bzip2Engine.recover, bz2b200_recover in include/bz2b200.h).

The expected outcome comes from the oracle, never from the code under test: an input is compressed by the oracle with a
small block cap (many blocks), its `table` gives the block positions p_i, then a copy is damaged.  Block i must be
  - if its 48 signature bits are intact: what oracle.decompress_block(d, p_i) gives (bytes, or an error status), where d
    is the damaged copy with its header replaced by BZh9 when it is no longer BZh1..BZh9;
  - if its signature is damaged: recovered (flagged NO_SIGNATURE) only when block i-1, or for i = 0 the header, was
    recovered, with the bytes the oracle decodes once the signature is restored; otherwise it has no region of its own.
Every case runs on the simulator (both parse kernels; the libbz2 level-9 case, six 900 kB blocks, only on the GPU) and on the
GPU (-m gpu, both parse kernels)."""
import bz2
import hashlib
import json
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from compressjs_flattened_b200 import _native
from compressjs_flattened_b200.bzip2 import (NO_SIGNATURE, REGION_BLOCK, REGION_END, REGION_HEADER, REGION_UNKNOWN, Bzip2Engine,
                                             Err)
from compressjs_flattened_b200.corpus import gen_text

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_SO = os.path.join(HERE, "sim", "libbz2b200_sim.so")
MAGIC_BLOCK, MAGIC_END = 0x314159265359, 0x177245385090

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


# ---- bit helpers and the oracle's expectation ----
def get_bits(blob, pos, n):
    b0, b1 = pos >> 3, (pos + n + 7) >> 3
    v = int.from_bytes(bytes(blob[b0:b1]).ljust(b1 - b0, b"\0"), "big")
    return (v >> (8 * (b1 - b0) - (pos - 8 * b0) - n)) & ((1 << n) - 1)


def flip(blob, *bits):
    b = bytearray(blob)
    for p in bits:
        b[p >> 3] ^= 0x80 >> (p & 7)
    return bytes(b)


def make(oracle, data, cap, level=9):
    """oracle stream with blocks of at most `cap` bytes, and its block positions"""
    oracle.set_block_cap(cap)
    try:
        comp = oracle.compress(data, level)
    finally:
        oracle.set_block_cap(0)
    return comp, [p for p, _ in oracle.table(comp)]


def footer_pos(comp):
    n = 8 * len(comp)
    return next(q for q in range(n - 87, n - 79) if get_bits(comp, q, 48) == MAGIC_END)


def block_fields(blob, p):
    """bit positions of a block's fields (BJ:1434-1520): stored CRC, origPtr, selectors, code lengths, symbol data"""
    q = p + 48 + 32 + 1 + 24
    used = get_bits(blob, q, 16)
    q += 16
    nsym = 0
    for i in range(16):
        if used >> (15 - i) & 1:
            nsym += bin(get_bits(blob, q, 16)).count("1")
            q += 16
    ng, nsel = get_bits(blob, q, 3), get_bits(blob, q + 3, 15)
    q += 18
    sel = q
    for _ in range(nsel):
        while get_bits(blob, q, 1):
            q += 1
        q += 1
    lens = q
    for _ in range(ng):
        q += 5
        for _ in range(nsym + 2):
            while get_bits(blob, q, 1):
                q += 2
            q += 1
    return dict(crc=(p + 48, p + 80), orig=(p + 81, p + 105), sel=(sel, lens), lens=(lens, q), data=(q, None))


def oracle_block(oracle, d, p):
    try:
        return "ok", oracle.decompress_block(d, p)
    except oracle.OracleError as e:
        return "err", e.errorCode


def expected(oracle, good, d, positions):
    """per block of `good` (at `positions`): (outcome, bytes or status, signature damaged, status comparable)"""
    hdr_ok = len(d) >= 4 and d[:3] == b"BZh" and 0x31 <= d[3] <= 0x39
    d9 = d if hdr_ok else b"BZh9" + d[4:]
    out, prev_ok = [], hdr_ok
    for p in positions:
        if p >= 8 * len(d):
            out.append(("gone", None, True, False))
        elif p + 48 <= 8 * len(d) and get_bits(d, p, 48) == MAGIC_BLOCK:
            out.append(oracle_block(oracle, d9, p) + (False, True))
        elif prev_ok:
            whole = p + 48 <= 8 * len(d)
            fixed = flip(d9, *[q for q in range(p, min(p + 48, 8 * len(d))) if get_bits(d9, q, 1) != get_bits(good, q, 1)])
            out.append(oracle_block(oracle, fixed, p) + (True, whole))
        else:
            out.append(("gone", None, True, False))
        prev_ok = out[-1][0] == "ok"
    return out


def check_tiling(regs, n, data):
    if n == 0:
        assert regs == []
        return
    assert regs[0].bit_begin == 0 and regs[-1].bit_end == 8 * n
    ends = 0
    off = 0
    for a, b in zip(regs, regs[1:]):
        assert a.bit_end == b.bit_begin
    for r in regs:
        assert r.bit_begin < r.bit_end
        assert r.out_offset == off and r.stream == ends
        assert r.out_bytes == 0 or (r.kind == REGION_BLOCK and r.status == 0)
        if r.kind == REGION_UNKNOWN:
            assert r.status == Err.NOT_BZIP_DATA
        if r.kind == REGION_END:
            ends += 1
        off += r.out_bytes
    assert off == len(data)


def check_recover(eng, oracle, good, d, positions):
    """recover(d) against the oracle's expectation; returns (data, regions, expectation)"""
    exp = expected(oracle, good, d, positions)
    data, regs = eng.recover(d)
    check_tiling(regs, len(d), data)
    blocks = {r.bit_begin: r for r in regs if r.kind == REGION_BLOCK}
    want = bytearray()
    for p, (what, val, nosig, comparable) in zip(positions, exp):
        flags = NO_SIGNATURE if nosig else 0
        if what == "ok":
            r = blocks[p]
            assert (r.status, r.flags) == (0, flags)
            assert data[r.out_offset:r.out_offset + r.out_bytes] == val
            want += val
        elif what == "err":
            r = blocks[p]
            assert r.flags == flags and r.status != 0 and r.out_bytes == 0
            if comparable:
                assert r.status == val
        else:
            assert p not in blocks
    assert data == bytes(want)
    assert sum(1 for r in regs if r.kind == REGION_BLOCK and r.status == 0) == sum(1 for e in exp if e[0] == "ok")
    st = eng.stats()
    assert (st.n_blocks, st.out_bytes) == (sum(1 for e in exp if e[0] == "ok"), len(data))
    return data, regs, exp


def damage_field(oracle, comp, positions, k, field, rng, tries=200):
    """a one-bit flip in `field` of block k that the oracle confirms is damage"""
    f = block_fields(comp, positions[k])[field]
    hi = f[1] if f[1] is not None else positions[k + 1] - 1
    for _ in range(tries):
        q = int(rng.integers(f[0], hi))
        d = flip(comp, q)
        if oracle_block(oracle, d, positions[k])[0] == "err":
            return d
    raise AssertionError(f"no damaging flip found in {field} of block {k}")


# ---- 1. intact inputs ----
def test_recover_intact_single_and_multistream(eng, oracle):
    one, _ = make(oracle, gen_text(30_000, 4).tobytes(), 2500)
    two, _ = make(oracle, gen_text(9_000, 5).tobytes(), 997, 3)
    for blob in (one, one + two, two + one):
        data, regs = eng.recover(blob)
        assert data == eng.decompressFile(blob, None, True)
        check_tiling(regs, len(blob), data)
        assert all(r.status == 0 and r.flags == 0 for r in regs)
        rows = []
        eng.table(blob, lambda p, s: rows.append((p, s)), True)
        assert [(r.bit_begin, r.out_bytes) for r in regs if r.kind == REGION_BLOCK] == rows
        kinds = [r.kind for r in regs]
        assert kinds.count(REGION_HEADER) == kinds.count(REGION_END) == (1 if blob is one else 2)
        assert eng.stats().n_blocks == len(rows)
    assert eng.recover(b"") == (b"", [])


@pytest.mark.gpu
def test_recover_intact_100mb_bench_stream(gpu_engine):
    """the text:100000000:8:L9 stream of corpus_goldens.json: the recovered bytes hash to the input's SHA-256"""
    g = json.load(open(os.path.join(HERE, "golden", "corpus_goldens.json")))["text:100000000:8:L9"]
    comp = gpu_engine.compressFile(gen_text(100_000_000, 8), None, 9)
    assert hashlib.sha256(comp).hexdigest() == g["out_sha256"]
    data, regs = gpu_engine.recover(comp)
    assert hashlib.sha256(data).hexdigest() == g["input_sha256"]
    assert all(r.status == 0 for r in regs) and sum(r.kind == REGION_BLOCK for r in regs) == g["n_blocks"]
    rows = []
    gpu_engine.table(comp, lambda p, s: rows.append((p, s)), True)
    assert [(r.bit_begin, r.out_bytes) for r in regs if r.kind == REGION_BLOCK] == rows


# ---- 2. damage inside one block ----
@pytest.mark.parametrize("field", ["sel", "lens", "data", "crc", "orig"])
def test_recover_one_damaged_block(eng, oracle, field):
    comp, pos = make(oracle, gen_text(24_000, 6).tobytes(), 2500)
    k = 4
    d = damage_field(oracle, comp, pos, k, field, np.random.default_rng(hash(field) & 0xffff))
    data, regs, exp = check_recover(eng, oracle, comp, d, pos)
    assert [e[0] for e in exp] == ["ok"] * k + ["err"] + ["ok"] * (len(pos) - k - 1)
    lost = next(r for r in regs if r.bit_begin == pos[k])
    assert lost.kind == REGION_BLOCK and lost.bit_end == pos[k + 1]
    assert [r.status for r in regs if r.kind == REGION_END] == [Err.DATA_ERROR]


# ---- 3. damaged signatures ----
@pytest.mark.parametrize("ks", [(0,), (5,), (6, 7)])
def test_recover_damaged_signature(eng, oracle, ks):
    comp, pos = make(oracle, gen_text(24_000, 7).tobytes(), 2500)
    d = flip(comp, *[pos[k] + 17 for k in ks])
    data, regs, exp = check_recover(eng, oracle, comp, d, pos)
    assert data == oracle.decompress(comp)
    for k in ks:
        r = next(r for r in regs if r.bit_begin == pos[k])
        assert (r.kind, r.status, r.flags) == (REGION_BLOCK, 0, NO_SIGNATURE)
    assert all(r.status == 0 for r in regs)


# ---- 4. damaged block followed by a damaged signature ----
def test_recover_damage_then_signature(eng, oracle):
    comp, pos = make(oracle, gen_text(24_000, 8).tobytes(), 2500)
    k = 3
    d = flip(damage_field(oracle, comp, pos, k, "data", np.random.default_rng(4)), pos[k + 1] + 30)
    data, regs, exp = check_recover(eng, oracle, comp, d, pos)
    assert [e[0] for e in exp[k:k + 3]] == ["err", "gone", "ok"]
    r = next(r for r in regs if r.bit_begin == pos[k])
    assert r.bit_end == pos[k + 2] and r.status != 0


# ---- 5. header and footer ----
def test_recover_header_and_footer_damage(eng, oracle):
    src = gen_text(20_000, 9).tobytes()
    comp, pos = make(oracle, src, 2500)
    f = footer_pos(comp)
    bad_hdr = comp[:3] + bytes([comp[3] ^ 0x40]) + comp[4:]
    data, regs, _ = check_recover(eng, oracle, comp, bad_hdr, pos)
    assert data == src
    assert (regs[0].kind, regs[0].status, regs[0].bit_end) == (REGION_HEADER, Err.NOT_BZIP_DATA, 32)
    assert regs[-1].kind == REGION_END and regs[-1].status == 0
    data, regs, _ = check_recover(eng, oracle, comp, flip(comp, f + 9), pos)
    assert data == src
    assert regs[-1].kind == REGION_BLOCK and regs[-1].flags == NO_SIGNATURE and regs[-1].status != 0 and regs[-1].bit_begin == f
    assert not any(r.kind == REGION_END for r in regs)
    data, regs, _ = check_recover(eng, oracle, comp, flip(comp, f + 60), pos)
    assert data == src
    assert (regs[-1].kind, regs[-1].status) == (REGION_END, Err.DATA_ERROR)


# ---- 6. truncation ----
def test_recover_truncated(eng, oracle):
    comp, pos = make(oracle, gen_text(24_000, 10).tobytes(), 2500)
    k = 6
    cut = (pos[k] + pos[k + 1]) // 16
    d = comp[:cut]
    data, regs, exp = check_recover(eng, oracle, comp, d, pos)
    assert [e[0] for e in exp[:k]] == ["ok"] * k
    last = regs[-1]
    assert (last.kind, last.bit_begin, last.bit_end) == (REGION_BLOCK, pos[k], 8 * cut)
    assert last.status == oracle_block(oracle, d, pos[k])[1] == Err.UNEXPECTED_INPUT_EOF


# ---- 7. garbage around and between streams ----
def test_recover_garbage_between_streams(eng, oracle):
    a, b = gen_text(15_000, 11).tobytes(), gen_text(8_000, 12).tobytes()
    s1, _ = make(oracle, a, 2500)
    s2, _ = make(oracle, b, 997, 2)
    rng = np.random.default_rng(5)
    g1, g2, g3 = (b"#" + rng.integers(0, 256, m, dtype=np.uint8).tobytes() for m in (36, 52, 28))
    blob = g1 + s1 + g2 + s2 + g3
    data, regs = eng.recover(blob)
    check_tiling(regs, len(blob), data)
    assert data == a + b
    unknown = [r for r in regs if r.kind == REGION_UNKNOWN]
    assert [r.bit_begin for r in unknown] == [0, 8 * (len(g1) + len(s1)), 8 * (len(g1) + len(s1) + len(g2) + len(s2))]
    assert unknown[-1].bit_end == 8 * len(blob)
    assert all(r.status == 0 for r in regs if r.kind in (REGION_BLOCK, REGION_END))
    assert [r.stream for r in regs if r.kind == REGION_END] == [0, 1]


# ---- 8. nothing to recover ----
def test_recover_no_signature(eng):
    blob = b"not a bzip2 file at all; " * 200
    data, regs = eng.recover(blob)
    assert data == b""
    assert [(r.kind, r.bit_begin, r.bit_end, r.status) for r in regs] == [(REGION_UNKNOWN, 0, 8 * len(blob), Err.NOT_BZIP_DATA)]


# ---- 9. damage at decode-batch boundaries ----
def test_recover_batch_boundaries(eng, oracle):
    comp, pos = make(oracle, gen_text(24_000, 13).tobytes(), 600)
    assert len(pos) == 40
    d = damage_field(oracle, comp, pos, 5, "data", np.random.default_rng(6))
    d = damage_field(oracle, d, pos, 14, "sel", np.random.default_rng(7))
    d = flip(d, pos[6] + 3, pos[9] + 40, pos[20] + 1, pos[21] + 47, pos[35] + 12)
    eng._L.bz2b200_debug_set_decode_batch(eng._ctx, None, 3)
    try:
        data, regs, exp = check_recover(eng, oracle, comp, d, pos)
    finally:
        eng._L.bz2b200_debug_set_decode_batch(eng._ctx, None, 0)
    assert [i for i, e in enumerate(exp) if e[0] != "ok"] == [5, 6, 14]   # 6: signature hit behind a lost block
    assert eng.recover(d) == (data, regs)


# ---- 10. randomized ----
def test_recover_randomized(eng, oracle):
    rng = np.random.default_rng(2024)
    for t in range(100):
        n = int(rng.integers(1_500, 12_000))
        src = gen_text(n, int(rng.integers(1, 1000))).tobytes()
        comp, pos = make(oracle, src, int(rng.choice([300, 997, 2500])), int(rng.integers(1, 10)))
        bits = [int(q) for q in rng.integers(0, 8 * len(comp), int(rng.integers(1, 5)))]
        d = flip(comp, *bits)
        if rng.random() < 0.3:
            d = d[:int(rng.integers(len(d) // 2, len(d)))]
        check_recover(eng, oracle, comp, d, pos)


# ---- 11. a libbz2-made stream, against bzip2recover ----
@pytest.mark.parametrize("level", [1, 9])
def test_recover_libbz2_stream_against_bzip2recover(eng, oracle, level):
    if level == 9 and not eng.on_gpu:
        pytest.skip("six 900 kB blocks: GPU only")
    src = gen_text(560_000 if level == 1 else 5_000_000, 14).tobytes()
    comp = bz2.compress(src, level)
    pos = [p for p, _ in oracle.table(comp)]
    assert len(pos) >= 6
    rng = np.random.default_rng(level)
    d = damage_field(oracle, comp, pos, 0, "data", rng)
    d = damage_field(oracle, d, pos, len(pos) - 1, "sel", rng)
    d_sig = flip(d, pos[3] + 20)   # and one block whose signature alone is hit
    data, regs, exp = check_recover(eng, oracle, comp, d_sig, pos)
    assert [e[0] for e in exp] == ["err"] + ["ok"] * (len(pos) - 2) + ["err"] and exp[3][2]
    if shutil.which("bzip2recover") is None:
        pytest.skip("bzip2recover is not on the PATH")
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "damaged.bz2")
        with open(path, "wb") as fh:
            fh.write(d_sig)
        subprocess.run(["bzip2recover", path], cwd=tmp, check=True, capture_output=True)
        pieces = []
        for name in sorted(f for f in os.listdir(tmp) if f.startswith("rec")):
            try:
                pieces.append(bz2.decompress(open(os.path.join(tmp, name), "rb").read()))
            except (OSError, ValueError):
                pass
    assert pieces
    at = 0
    for piece in pieces:   # every piece bzip2recover saved is in the recovered bytes, in order
        at = data.find(piece, at)
        assert at >= 0
        at += len(piece)
    assert len(data) > sum(len(p) for p in pieces)   # and the block behind the damaged signature as well


# ---- the command line ----
def test_recover_command_line(sim_engine, oracle, tmp_path, capsys):
    from compressjs_flattened_b200.__main__ import main
    src = gen_text(12_000, 15).tobytes()
    comp, pos = make(oracle, src, 2500)
    good, bad, out = tmp_path / "good.bz2", tmp_path / "bad.bz2", tmp_path / "out"
    good.write_bytes(comp)
    bad.write_bytes(damage_field(oracle, comp, pos, 1, "crc", np.random.default_rng(1)))
    assert main(["--recover", str(good), str(out)], engine=sim_engine) == 0
    assert out.read_bytes() == src and capsys.readouterr().err == ""
    assert main(["--recover", str(bad), str(out)], engine=sim_engine) == 2
    sizes = [sz for _, sz in oracle.table(comp)]
    assert out.read_bytes() == src[:sizes[0]] + src[sizes[0] + sizes[1]:]
    err = capsys.readouterr().err.splitlines()
    assert err == [f"bits {pos[1]}-{pos[2]}: BLOCK DATA_ERROR", f"bits {footer_pos(comp)}-{8 * len(comp)}: END DATA_ERROR"]
    for extra, msg in ((["-z"], "--recover can only be used without -z"), (["-b", "32"], "--recover and --block can't be used together"),
                       (["-9"], "Compression level has no effect when recovering.")):
        assert main(["--recover"] + extra + [str(good), str(out)], engine=sim_engine) == 1
        assert capsys.readouterr().err.strip() == msg
