"""Decoder conformance on hand-built bzip2 streams.

The compressor only writes a small part of what the format allows, and libbz2 a slightly larger one.  The streams here
come from a small writer that can express every choice the decoder must honour: the RLE1 content of a block, its
used-byte map, the number of tables, per-table code lengths (1..20 bits, complete or not), the selectors (with extra
ones, or raw MTF indices), origPtr and the block CRC, the level of each stream and several streams back to back.  The
writer takes the BWT from the oracle and writes MTF, RUNA/RUNB runs and canonical codes itself; it is checked against
oracle.compress byte for byte.

Every case goes through every decode entry point (decompressFile under each parse kernel, table, decompressBlock,
decompressStream, Bzip2Pool.decompressFile, recover).  A valid stream must decode to what the writer put in (the
oracle and, unless noted, libbz2 agree); an invalid one must fail with the oracle's error code.  The `not gpu` leg runs
the simulator build of the kernels on the small cases and the level-1 capacity cases; the `gpu` leg runs all of them."""
import bz2
import functools
import io
import os

import numpy as np
import pytest

import oracle_binding as O
from compressjs_flattened_b200 import _native
from compressjs_flattened_b200.bzip2 import REGION_BLOCK, Bzip2Engine, Bzip2Error, Err
from compressjs_flattened_b200.corpus import gen_text
from compressjs_flattened_b200.pool import Bzip2Pool

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_SO = os.path.join(HERE, "sim", "libbz2b200_sim.so")
MAGIC_BLOCK, MAGIC_END = 0x314159265359, 0x177245385090
GROUP = 50


# ---------------------------------------------------------------------------------------------------- the writer ----
def put(v, n):
    """n bits of v, most significant first, as an array of 0/1"""
    return np.array([(v >> (n - 1 - i)) & 1 for i in range(n)], dtype=np.uint8)


def mtf_rle2(L, used):
    """MTF over the used bytes, runs of index 0 as RUNA (0) / RUNB (1) digits, end-of-block = len(used) + 1"""
    lst, out, run = list(used), [], 0

    def flush():
        nonlocal run
        while run:
            if run & 1:
                out.append(0)
                run -= 1
            else:
                out.append(1)
                run -= 2
            run >>= 1
    for c in L:
        j = lst.index(c)
        if j == 0:
            run += 1
            continue
        flush()
        del lst[j]
        lst.insert(0, c)
        out.append(j + 1)
    flush()
    out.append(len(used) + 1)
    return out


def canonical(lens):
    """codes assigned in (length, symbol) order: what limit/base/permute decode"""
    code, c, prev = [0] * len(lens), 0, 0
    for s in sorted(range(len(lens)), key=lambda s: (lens[s], s)):
        c <<= lens[s] - prev
        code[s] = c
        c += 1
        prev = lens[s]
    return code


def ibwt(L, orig):
    """the reference's inverse BWT (BJ:1677-1690 and the walk of BJ:1716-1763) started at `orig`"""
    order = np.argsort(np.frombuffer(L, dtype=np.uint8), kind="stable").tolist()
    out, pos = bytearray(len(L)), order[orig]
    for i in range(len(L)):
        out[i] = L[pos]
        pos = order[pos]
    return bytes(out)


def rle1_expand(blk):
    """_read_bunzip (oracle bz2_oracle.c read_bunzip): the byte after four equal ones is a count"""
    out, current, run = bytearray(), -1, -1
    for b in blk:
        previous, current = current, b
        if run == 3:
            out += bytes([previous]) * current
            current = -1
        else:
            out.append(current)
        run += 1
        if current != previous:
            run = 0
    return bytes(out)


def sel_from_mtf(raw, ng):
    """the reference's selector MTF (BJ:1481-1496): a zeroed Uint8Array(256) with 0..ng-1 in front"""
    lst, out = list(range(ng)) + [0] * (256 - ng), []
    for j in raw:
        v = lst.pop(j)
        lst.insert(0, v)
        out.append(v)
    return out


def sel_to_mtf(tables, ng):
    lst, out = list(range(ng)), []
    for t in tables:
        j = lst.index(t)
        lst.insert(0, lst.pop(j))
        out.append(j)
    return out


@functools.lru_cache(maxsize=32)
def _transform(content, used):
    L, pidx = O.bwt(content)
    return L, pidx, mtf_rle2(L, used)


def huffman(A, S):
    return [int(x) for x in O.huff_lengths(np.bincount(A, minlength=S).astype(np.int32))]


def make_block(content, used=None, ntab=2, lens=None, sel=None, sel_mtf=None, nsel=None, orig_ptr=None, crc=None):
    """One block.  content: the RLE1 bytes; used: the byte map (default: the bytes present); lens: per-table code lengths,
    or f(A, S) -> lengths of every table; sel: the table of every group, or f(g); sel_mtf: raw selector MTF indices
    instead (at least one per group); nsel: selectors written, more than the groups (the extra ones cycle through the
    tables); orig_ptr / crc: stored values instead of the right ones.  Returns the bits, the stored CRC, the bytes the
    reference decodes (None: origPtr past the data), the symbols and the bit offset where each ends."""
    content = bytes(content)
    used = tuple(sorted(set(content) if used is None else set(used)))
    assert set(content) <= set(used) and used
    L, pidx, A = _transform(content, used)
    S, m = len(used) + 2, len(A)
    ngroups = (m + GROUP - 1) // GROUP
    if lens is None:
        lens = [huffman(A, S)] * ntab
    elif callable(lens):
        lens = lens(A, S)
    assert len(lens) == ntab and all(len(t) == S and min(t) >= 1 and max(t) <= 20 for t in lens)
    assert all(sum(2.0 ** -x for x in t) <= 1 for t in lens)    # codes that can be written
    if sel_mtf is not None:
        raw = list(sel_mtf)
        tables = sel_from_mtf(raw, ntab)[:ngroups]
    else:
        tables = [sel(g) if callable(sel) else sel[g] for g in range(ngroups)] if sel is not None else [g % ntab for g in range(ngroups)]
        raw = sel_to_mtf(tables + [g % ntab for g in range(ngroups, nsel or ngroups)], ntab)
    assert len(tables) == ngroups and 1 <= len(raw) < 1 << 15
    orig = pidx if orig_ptr is None else orig_ptr
    if orig < len(content):
        seq = content if orig == pidx else ibwt(L, orig)
        out = rle1_expand(seq)
    else:
        out = None                                              # origPtr past the data: a Data error
    if orig == pidx:
        assert ibwt(L, pidx) == content
    stored = O.crc32(out if out is not None else b"") if crc is None else crc
    bits, sym_end = write_block(A, used, orig, stored, lens, tables, raw)
    return dict(bits=bits, crc=stored, out=out, A=A, sym_end=sym_end, n=len(content), used=used,
                lens=lens, tables=tables, nsel=len(raw))


def write_block(A, used, orig, stored, lens, tables, raw):
    """The bits of one block: the symbols A (MTF/RLE2 over the byte map `used`, end-of-block last) coded with the code
    lengths lens[tables[g]] in group g, raw selector MTF indices, origPtr and the stored CRC.  Returns the bits and the bit
    offset where each symbol ends."""
    m = len(A)
    hdr = [put(MAGIC_BLOCK, 48), put(stored, 32), put(0, 1), put(orig, 24)]
    groups = [any(b >> 4 == i for b in used) for i in range(16)]
    hdr.append(np.array(groups, dtype=np.uint8))
    for i in range(16):
        if groups[i]:
            hdr.append(np.array([(i << 4 | j) in used for j in range(16)], dtype=np.uint8))
    hdr += [put(len(lens), 3), put(len(raw), 15)]
    r = np.array(raw, dtype=np.int64)
    sb = np.ones(int((r + 1).sum()), dtype=np.uint8)
    sb[np.cumsum(r + 1) - 1] = 0
    hdr.append(sb)
    for t in lens:
        bits, cur = [], t[0]
        for x in t:
            bits += ([1, 0] if cur < x else [1, 1]) * abs(x - cur) + [0]
            cur = x
        hdr += [put(t[0], 5), np.array(bits, dtype=np.uint8)]
    Aw = np.array(A, dtype=np.int64)
    tab = np.repeat(np.array(tables, dtype=np.int64), GROUP)[:m]
    codes = np.array([canonical(t) for t in lens], dtype=np.int64)[tab, Aw]
    ln = np.array(lens, dtype=np.int64)[tab, Aw]
    ends = np.cumsum(ln)
    k = np.arange(int(ends[-1])) - np.repeat(ends - ln, ln)
    data = ((np.repeat(codes, ln) >> (np.repeat(ln, ln) - 1 - k)) & 1).astype(np.uint8)
    head = np.concatenate(hdr)
    return np.concatenate([head, data]), len(head) + ends


def make_stream(level, blocks):
    """header, blocks, end-of-stream: (bit array, bit positions of the blocks)"""
    parts, pos, at, fold = [put(0x425A68, 24), put(0x30 + level, 8)], [], 32, 0
    for b in blocks:
        pos.append(at)
        parts.append(b["bits"])
        at += len(b["bits"])
        fold = (((fold << 1) | (fold >> 31)) & 0xFFFFFFFF) ^ b["crc"]
    parts += [put(MAGIC_END, 48), put(fold, 32)]
    return np.concatenate(parts), pos


def pack(bits):
    return np.packbits(bits).tobytes()


# ------------------------------------------------------------------------------------------- the writer's check ----
@pytest.mark.parametrize("n,cap,level", [(40_000, 0, 9), (23_000, 2500, 3)])
def test_writer_reproduces_oracle_compress(oracle, n, cap, level):
    """Given the oracle's own choices (cut points, selectors, code lengths), the writer makes oracle.compress's bytes."""
    data = gen_text(n, 11).tobytes()
    oracle.set_block_cap(cap)
    try:
        want = oracle.compress(data, level)
        starts, lens, crcs = oracle.cut_points(data, level)
        bcap = cap or 100_000 * level - 19
        blocks = []
        for k in range(len(lens)):
            blk, used, crc = oracle.rle1_block(data[starts[k]:], bcap)
            st = oracle.block_stages(blk.tobytes())
            assert (len(blk), crc) == (lens[k], crcs[k])
            b = make_block(blk.tobytes(), ntab=st["n_groups"], lens=[list(map(int, t)) for t in st["lens"]],
                           sel=[int(x) for x in st["sel"]])
            assert b["crc"] == crc and b["out"] == data[starts[k]:starts[k] + used]
            assert b["A"] == st["A"].tolist()
            blocks.append(b)
    finally:
        oracle.set_block_cap(0)
    assert len(blocks) == (1 if cap == 0 else 10)
    assert pack(make_stream(level, blocks)[0]) == want


def test_writer_pieces():
    assert rle1_expand(b"abbbb\x03c") == b"a" + b"b" * 7 + b"c"
    assert rle1_expand(b"aaaa") == b"aaaa" and rle1_expand(b"aaaa\x00aaaa") == b"aaaaaaaa"
    assert sel_from_mtf([0, 1, 2, 2], 2) == [0, 1, 0, 0]        # index 2 == nGroups: the zero behind the list
    assert canonical([1, 3, 3, 2]) == [0b0, 0b110, 0b111, 0b10]


# ---------------------------------------------------------------------------------------------------- the cases ----
def text(n, seed=3):
    return gen_text(n, seed).tobytes()


def no_runs_of_four(n, seed):
    a = np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8)
    while True:
        r = np.nonzero((a[3:] == a[2:-1]) & (a[3:] == a[1:-2]) & (a[3:] == a[:-3]))[0] + 3
        if not len(r):
            return a.tobytes()
        a[r] ^= 0x55


def fib_lengths(S):
    """oracle.huff_alloc on Fibonacci frequencies (ascending, above a floor of ones), limited to 20 bits: longest first"""
    f = [1, 1]
    while len(f) < min(S, 30):
        f.append(f[-1] + f[-2])
    return O.huff_alloc([1] * (S - len(f)) + [S * x for x in f], 20)


def by_frequency(A, S, lens_longest_first, longest_to_frequent):
    freq = np.bincount(A, minlength=S)
    order = np.argsort(-freq if longest_to_frequent else freq, kind="stable")
    out = [0] * S
    for rank, s in enumerate(order):
        out[int(s)] = int(lens_longest_first[rank])
    return out


def long_codes(A, S):      # the 18-20-bit codes on the most frequent symbols
    return by_frequency(A, S, fib_lengths(S), True)


def short_codes(A, S):     # the usual way round: a 1-bit code on the most frequent symbol
    return by_frequency(A, S, fib_lengths(S), False)


def min11_codes(A, S):     # no code of 10 bits or fewer: every code goes through the long-code walk
    return [min(20, x + 10) for x in long_codes(A, S)]


def equal_codes(A, S):     # all-equal, incomplete: the code of all one bits is missing
    return [max(2, int(np.ceil(np.log2(S))) + 1)] * S


def equal_tables(A, S):
    return [equal_codes(A, S)] * 2


def overflow_at(A, cap):
    """index of the symbol at which the reference's size checks (BJ:1647,1663) stop a block of capacity `cap`"""
    count, t_run, run_pos, eob = 0, 0, 0, max(A)
    for i, s in enumerate(A):
        if s <= 1:
            if not run_pos:
                run_pos, t_run = 1, 0
            t_run += run_pos << s
            run_pos <<= 1
            if t_run > cap:
                return i
            continue
        if run_pos:
            run_pos = 0
            if count + t_run > cap:
                return i
            count += t_run
        if s == eob:
            return None
        if count >= cap:
            return i
        count += 1
    return None


class Case:
    def __init__(self, name, streams, valid=True, err=None, cut=None, sim=True, libbz2=None, multistream=False, check=None):
        self.name, self.streams, self.valid, self.err, self.cut = name, streams, valid, err, cut
        self.sim, self.libbz2, self.multistream, self.check = sim, libbz2, multistream, check

    @functools.cached_property
    def built(self):
        """(stream bytes, expected output, global bit positions of the blocks, the blocks)"""
        blob, expect, pos, blocks = b"", b"", [], []
        for level, specs in self.streams:
            bl = [make_block(**s) for s in specs]
            bits, p = make_stream(level, bl)
            base = 8 * len(blob)
            if self.cut is not None:
                bits = self.cut(bits, p, bl)
            blob += pack(bits)
            pos += [base + q for q in p]
            blocks += bl
            expect += b"".join(b["out"] or b"" for b in bl)
        return blob, expect, pos, blocks


def cut_after(sym):
    """truncate a one-block stream right after symbol `sym(block)` of its block"""
    return lambda bits, p, bl: bits[:p[0] + int(bl[0]["sym_end"][sym(bl[0])])]


def bad_code_after(sym):
    """a one-block stream whose symbol `sym(block)` is followed by a code the (all-equal, incomplete) tables lack"""
    def f(bits, p, bl):
        e = p[0] + int(bl[0]["sym_end"][sym(bl[0])])
        return np.concatenate([bits[:e], np.ones(64, dtype=np.uint8), bits[e:e + 256]])
    return f


NO_RUNS = functools.lru_cache(maxsize=8)(no_runs_of_four)
RUN_BYTE = 0x41


def capacity_cases(level):
    cap, big = 100_000 * level, level > 1
    exact = lambda: NO_RUNS(cap, level)                                   # noqa: E731
    over = lambda: NO_RUNS(cap + 1, level)                                # noqa: E731
    at_over = lambda b: overflow_at(b["A"], cap)                          # noqa: E731
    cs = [
        Case(f"L{level}-exact", [(level, [dict(content=exact(), lens=equal_tables)])], sim=not big,
             check="exact"),
        Case(f"L{level}-plus1-literals", [(level, [dict(content=over(), lens=equal_tables)])], valid=False, err=Err.DATA_ERROR,
             sim=not big, check="literal"),
        Case(f"L{level}-plus1-run", [(level, [dict(content=bytes([RUN_BYTE]) * (cap + 1))])], valid=False, err=Err.DATA_ERROR,
             check="run"),
        Case(f"L{level}-plus1-literals-truncated", [(level, [dict(content=over(), lens=equal_tables)])], valid=False,
             err=Err.DATA_ERROR, cut=cut_after(at_over), sim=not big),
        Case(f"L{level}-plus1-run-truncated", [(level, [dict(content=bytes([RUN_BYTE]) * (cap + 1))])], valid=False,
             err=Err.DATA_ERROR, cut=cut_after(at_over)),
        Case(f"L{level}-plus1-literals-bad-code", [(level, [dict(content=over(), lens=equal_tables)])], valid=False,
             err=Err.DATA_ERROR, cut=bad_code_after(at_over), sim=not big),
        Case(f"L{level}-plus1-run-bad-code", [(level, [dict(content=bytes([RUN_BYTE]) * (cap + 1), lens=equal_tables)])],
             valid=False, err=Err.DATA_ERROR, cut=bad_code_after(at_over)),
    ]
    small = text(3000, level)
    n = len(small)
    cs += [
        Case(f"L{level}-origptr-0", [(level, [dict(content=small, orig_ptr=0)])]),
        Case(f"L{level}-origptr-count-1", [(level, [dict(content=small, orig_ptr=n - 1)])]),
        Case(f"L{level}-origptr-count", [(level, [dict(content=small, orig_ptr=n)])], valid=False, err=Err.DATA_ERROR),
        # origPtr is checked as soon as it is read: before the truncated tables are
        Case(f"L{level}-origptr-over-truncated", [(level, [dict(content=small, orig_ptr=cap + 1)])], valid=False,
             err=Err.DATA_ERROR, cut=lambda bits, p, bl: bits[:p[0] + 600]),
    ]
    return cs


def rle1_case(name, piece):
    return Case(name, [(9, [dict(content=text(700, 5) + piece + text(300, 6))])])


def three_to_four(g):
    return Case(f"tables-3-to-4-at-group-{g}",
                [(9, [dict(content=text(6000, 7), ntab=4, lens=lambda A, S: [long_codes(A, S), short_codes(A, S), min11_codes(A, S),
                                                                              long_codes(A, S)],
                           sel=lambda q: q % 3 if q < g else 3 if q == g else (q * 7) % 4)])])


def perms_of_256(k, seed):
    rng = np.random.default_rng(seed)
    return b"".join(rng.permutation(256).astype(np.uint8).tobytes() for _ in range(k))


def many_blocks():
    rng = np.random.default_rng(9)
    return [dict(content=text(int(rng.integers(20, 400)), int(s)).rstrip(b" "), ntab=int(rng.integers(2, 7))) for s in range(1, 41)]


# where libbz2's rules differ from the reference's, the case is not decoded with libbz2
NO_LIBBZ2_SEL = "libbz2 rejects a selector MTF index >= nGroups (it allows 0..nGroups-1)"
NO_LIBBZ2_TRAILING_RUN = "libbz2 rejects a block that ends in four equal bytes without a count byte"

CASES = [
    # long codes
    Case("codes-long-on-frequent", [(9, [dict(content=text(5000, 1), lens=lambda A, S: [long_codes(A, S), short_codes(A, S)])])],
         check="long"),
    Case("codes-min-11-bits", [(9, [dict(content=text(5000, 2), lens=lambda A, S: [min11_codes(A, S), min11_codes(A, S)])])],
         check="min11"),
    Case("codes-equal-incomplete-and-1-bit", [(9, [dict(content=text(5000, 3), lens=lambda A, S: [equal_codes(A, S), short_codes(A, S)])])],
         check="onebit"),
    # tables and selectors
    Case("tables-6-on-a-tiny-block", [(9, [dict(content=text(300, 4), ntab=6, sel=lambda g: (g * 5 + 1) % 6)])]),
    Case("tables-2-on-a-full-level-9-block", [(9, [dict(content=NO_RUNS(900_000, 9), ntab=2, sel=lambda g: (g // 3) % 2)])], sim=False),
    Case("tables-6-cycled-every-group-20-bit", [(9, [dict(content=text(20_000, 5), ntab=6,
                                                          lens=lambda A, S: [long_codes(A, S), min11_codes(A, S)] * 3,
                                                          sel=lambda g: g % 6)])], check="long"),
] + [three_to_four(g) for g in (5, 6, 7, 8, 16)] + [
    Case("selectors-32767", [(9, [dict(content=text(2000, 6), ntab=3, nsel=32767)])],
         check="sel32767"),
    Case("selector-mtf-index-equal-to-ngroups", [(9, [dict(content=text(2000, 8), ntab=3, sel_mtf=[0, 3, 1, 3, 3, 2] + [1] * 40)])],
         libbz2=NO_LIBBZ2_SEL),
    # alphabet
    Case("alphabet-all-256", [(9, [dict(content=perms_of_256(8, 1))])], check="mtf255"),
    Case("alphabet-one-byte", [(9, [dict(content=b"qqq")])]),
    Case("alphabet-unused-bytes-in-map", [(9, [dict(content=text(800, 9), used=set(text(800, 9)) | {0, 1, 0x80, 0xFF})])]),
    # RLE1 content no encoder writes
    rle1_case("rle1-count-0", b"zzzz\x00"),
    rle1_case("rle1-count-251", b"zzzz\xfb"),
    rle1_case("rle1-count-252", b"zzzz\xfc"),
    rle1_case("rle1-count-255", b"zzzz\xff"),
    rle1_case("rle1-count-equal-to-run-byte", b"zzzzz"),
    Case("rle1-trailing-run-without-count", [(9, [dict(content=text(500, 7) + b"zzzz")])], libbz2=NO_LIBBZ2_TRAILING_RUN),
    # layout
    Case("layout-many-small-blocks", [(4, many_blocks())], check="phases"),
    Case("layout-long-codes-over-many-ring-passes", [(9, [dict(content=text(40_000, 10), lens=lambda A, S: [long_codes(A, S)] * 2)])]),
    Case("layout-multistream-levels-1-9-4", [(1, [dict(content=text(900, 1)), dict(content=text(1300, 2))]),
                                             (9, [dict(content=text(700, 3), ntab=5)]),
                                             (4, [dict(content=b"qqq"), dict(content=text(2000, 4), ntab=6)])], multistream=True),
] + capacity_cases(1) + capacity_cases(5) + capacity_cases(9)

BY_NAME = {c.name: c for c in CASES}
assert len(BY_NAME) == len(CASES)


# ------------------------------------------------------------------------------------- what each case must show ----
def check_shape(case):
    """the property a case exists for is really in its stream"""
    blob, _, pos, blocks = case.built
    b = blocks[0]
    if case.check == "long":                                    # 18-20-bit codes on the most frequent symbol
        top = int(np.argmax(np.bincount(b["A"])))
        assert max(b["lens"][0]) == 20 and b["lens"][0][top] >= 18
    if case.check == "min11":
        assert min(min(t) for t in b["lens"]) >= 11
    if case.check == "onebit":
        assert len(set(b["lens"][0])) == 1 and sum(2.0 ** -x for x in b["lens"][0]) < 1 and 1 in b["lens"][1]
    if case.check == "exact":
        cap = 100_000 * int(case.streams[0][0])
        blk, used, _ = O.rle1_block(blocks[0]["out"], cap)
        assert b["n"] == cap and used == cap and blk.tobytes() == blocks[0]["out"]
    if case.check == "literal":
        cap = 100_000 * int(case.streams[0][0])
        assert b["A"][overflow_at(b["A"], cap)] >= 2            # the block outgrows its size at a literal
    if case.check == "run":
        cap = 100_000 * int(case.streams[0][0])
        assert b["A"][overflow_at(b["A"], cap)] <= 1            # ... at a RUNA/RUNB digit
    if case.check == "mtf255":
        assert max(b["A"][:-1]) == 256 and len(b["used"]) == 256
    if case.check == "phases":
        assert {p % 8 for p in pos} == set(range(8))
    if case.check == "sel32767":
        assert b["nsel"] == 32767 > len(b["tables"])


def outcome(fn):
    try:
        return ("ok", fn())
    except (Bzip2Error, O.OracleError) as e:
        return ("err", e.errorCode)


def oracle_block(blob, p):
    return outcome(lambda: O.decompress_block(blob, p))


# ------------------------------------------------------------------------------------------------------- engines ----
def _engines(library):
    engs = {}
    old = os.environ.get("BZ2B200_PARSE")
    try:
        for mode in ("1", "2", None):      # BZ2B200_PARSE is read when the context is created
            if mode is None:
                os.environ.pop("BZ2B200_PARSE", None)
            else:
                os.environ["BZ2B200_PARSE"] = mode
            engs[mode] = Bzip2Engine(0, library)
    finally:
        if old is None:
            os.environ.pop("BZ2B200_PARSE", None)
        else:
            os.environ["BZ2B200_PARSE"] = old
    return engs, Bzip2Pool([0], 2, library=library)


@pytest.fixture(scope="module")
def sim_engines(sim_engine):                       # sim_engine builds the simulator library when it is stale
    engs, pool = _engines(_native.Library(SIM_SO))
    yield engs, pool
    for e in engs.values():
        e.close()
    pool.close()


@pytest.fixture(scope="module")
def gpu_engines():
    engs, pool = _engines(None)
    yield engs, pool
    for e in engs.values():
        e.close()
    pool.close()


def run_case(case, engs, pool):
    blob, expect, pos, blocks = case.built
    ms = case.multistream
    check_shape(case)
    want = outcome(lambda: O.decompress(blob, ms))
    if case.valid:
        assert want == ("ok", expect)
        if case.libbz2 is None:
            assert bz2.decompress(blob) == expect
    else:
        assert want == ("err", case.err)
    # decompressFile under each parse kernel (1 = CTA per block, 2 = speculative window, unset = chosen per batch)
    for mode, eng in engs.items():
        assert outcome(lambda: eng.decompressFile(blob, None, ms)) == want, f"BZ2B200_PARSE={mode}"
    eng = engs[None]
    rows = []
    assert outcome(lambda: (eng.table(blob, lambda p, s: rows.append((p, s)), ms), rows)[1]) == outcome(lambda: O.table(blob, ms))
    for p in pos:
        assert outcome(lambda: eng.decompressBlock(blob, p)) == oracle_block(blob, p), f"block at bit {p}"
    assert outcome(lambda: eng.decompressStream(io.BytesIO(blob), None, ms, chunk_bytes=1 << 16, piece_bytes=5000)) == want
    assert outcome(lambda: pool.decompressFile(blob, None, ms, slice_bytes=16_000)) == want
    data, regs = eng.recover(blob)
    found = {r.bit_begin: r for r in regs if r.kind == REGION_BLOCK}
    if case.valid:
        assert data == expect and all(r.status == 0 for r in regs)
        assert sorted(found) == pos
    else:
        assert pos[0] in found
        for p in pos:
            if p in found:
                r, (what, val) = found[p], oracle_block(blob, p)
                if what == "ok":
                    assert r.status == 0 and data[r.out_offset:r.out_offset + r.out_bytes] == val
                else:
                    assert (r.status, r.out_bytes) == (val, 0)   # a block over its stream's size is dropped


SIM_CASES = [pytest.param(c.name, id=c.name) for c in CASES if c.sim]
GPU_CASES = [pytest.param(c.name, id=c.name) for c in CASES]


@pytest.mark.parametrize("name", SIM_CASES)
def test_conformance_sim(sim_engines, oracle, name):
    run_case(BY_NAME[name], *sim_engines)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_CASES)
def test_conformance_gpu(gpu_engines, oracle, name):
    run_case(BY_NAME[name], *gpu_engines)
