"""Decoder conformance stage by stage, on blocks built to reach each inverse kernel's internal limits.

test_decode_conformance.py covers what the parse kernels read (header, tables, selectors, code lengths).  This file
covers the rest of the decoder: the signature scan, the RLE2 inverse offsets, the inverse MTF, the T vector and the
inverse-BWT list ranking, the RLE1 inverse and the block CRC.  Blocks are written from a given symbol list or from a
given L column and origPtr (the writer of test_decode_conformance.py), so that a case can put a run digit, a rank, a
splitter or a strip end exactly where a kernel changes state.  A Python reference computes every stage; after a decode
the stage dumps of the last decode batch (Bzip2Engine.decode_stages / decode_inverted) are compared with it in order, and
the first stage that differs is reported with its block and index.  Every case asserts that it really reaches its target.

Every case runs under both parse kernels and both forced widths of the RLE1 inverse.  The signature cases also run every
entry point that scans for signatures (decompressFile, table, index, search, recover, decompressStream in small pieces,
Bzip2Pool.decompressFile in small slices) against the oracle and libbz2.  The `not gpu` leg runs the simulator build at
small sizes; the `gpu` leg runs every case at full size."""
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
from test_decode_conformance import MAGIC_BLOCK, MAGIC_END, SIM_SO, huffman, ibwt, make_stream, mtf_rle2, no_runs_of_four, pack, \
    rle1_expand, sel_to_mtf, write_block

SEG = 4096                 # IMTF_SEG, and the symbols of one k_sym_offsets chunk (1024 threads x 4)
TILE = 4096                # SORT_TILE
SPL = 64                   # IBWT_S
STRIP = {512: 8 * 512, 1024: 8 * 1024}   # RLE1 inverse strip bytes by CTA width
CRC_CHUNK = 1 << 16
ALL = tuple(range(256))


# --------------------------------------------------------------------------------------------- the references ----
def ref_offsets(A):
    """where each symbol's bytes start in the L column: exclusive sum of literal = 1, run digit k = (sym + 1) << k,
    end-of-block = 0; len(A) + 1 entries (Python ints: a run of many digits is larger than any block)"""
    off, o, k = [0] * (len(A) + 1), 0, 0
    for i, s in enumerate(A[:-1]):
        off[i] = o
        if s <= 1:
            o += (s + 1) << k
            k += 1
        else:
            o += 1
            k = 0
    off[len(A) - 1] = off[len(A)] = o
    return off


def ref_L(A, used):
    """the MTF inverse over the byte map: the L column"""
    lst, out, k = list(used), bytearray(), 0
    for s in A[:-1]:
        if s <= 1:
            out += bytes([lst[0]]) * ((s + 1) << k)
            k += 1
        else:
            c = lst.pop(s - 1)
            lst.insert(0, c)
            out.append(c)
            k = 0
    return bytes(out)


def _ends_in_run(seq):
    """four equal RLE1 bytes at the end, with no count byte after them (libbz2 rejects that, the reference does not)"""
    current, run = -1, -1
    for b in seq:
        previous, current = current, b
        if run == 3:
            current = -1
        run += 1
        if current != previous:
            run = 0
    return run == 3


def cycle_of(L, orig):
    """the slots of the T-vector cycle that holds origPtr"""
    order = np.argsort(np.frombuffer(L, dtype=np.uint8), kind="stable")
    cyc, p = [], int(order[orig])
    while True:
        cyc.append(p)
        p = int(order[p])
        if p == cyc[0]:
            return cyc


# ----------------------------------------------------------------------------------------------------- blocks ----
class Blk:
    """One block given by its symbols (A, used) or by its L column (L, used), origPtr and code lengths (None: Huffman of
    the symbols; an int: every symbol that many bits).  Computes every stage of the reference."""

    def __init__(self, A=None, L=None, used=None, orig=0, content=None, lens=None):
        if content is not None:
            L, orig = O.bwt(content)
        if L is not None:
            used = tuple(sorted(set(L))) if used is None else tuple(used)
            A = mtf_rle2(L, used)
        self.A, self.used, self.orig = list(A), tuple(used), orig
        self.offs = ref_offsets(self.A)
        self.n = self.offs[-1]
        self.L = self.seq = self.out = None               # a block larger than any level's: a Data error, no stages
        if self.n <= 900_000:
            self.L = ref_L(self.A, self.used) if L is None else L
            assert len(self.L) == self.n
            if orig < self.n:
                self.seq = ibwt(self.L, orig)               # the inverse-BWT output (RLE1 bytes)
                self.out = rle1_expand(self.seq)
        self.trailing_run = self.seq is not None and _ends_in_run(self.seq)
        self.crc = O.crc32(self.out or b"")
        S, m = len(self.used) + 2, len(self.A)
        ng = (m + 49) // 50
        if lens is None:
            tl = [huffman(self.A, S)] * 2
        else:
            tl = [[lens] * S] * 2
        tables = [g % 2 for g in range(ng)]
        self.bits, _ = write_block(self.A, self.used, orig, self.crc, tl, tables, sel_to_mtf(tables, 2))


def sym(rank):
    """the symbol of MTF rank 1..255"""
    return rank + 1


def run_digits(v):
    """RUNA/RUNB digits of a run of v bytes"""
    out = []
    while v:
        if v & 1:
            out.append(0)
            v -= 1
        else:
            out.append(1)
            v -= 2
        v >>= 1
    return out


class Case:
    def __init__(self, name, streams, multistream=False, scan=False, check=None, libbz2=True, sim=True, small=None):
        """streams: [(level, [Blk factory, ...])]; scan: run every entry point that scans for signatures; check(case):
        asserts the case reaches its target; small: a smaller version for the simulator leg"""
        self.name, self.streams, self.multistream, self.scan = name, streams, multistream, scan
        self.check, self.libbz2, self.sim, self.small = check, libbz2, sim, small

    @functools.cached_property
    def built(self):
        blob, pos, blocks = b"", [], []
        for level, specs in self.streams:
            bl = [f() for f in specs]
            bits, p = make_stream(level, [dict(bits=b.bits, crc=b.crc) for b in bl])
            pos += [8 * len(blob) + q for q in p]
            blob += pack(bits)
            blocks += bl
        return blob, pos, blocks

    @functools.cached_property
    def one_batch(self):
        """every signature candidate fits one decode batch (1 280), so the stage dumps show every block"""
        return len(signature_hits(self.built[0])) < 1280

    @functools.cached_property
    def expect(self):
        blob, _, _ = self.built
        try:
            return O.decompress(blob, self.multistream)
        except O.OracleError as e:
            return e.errorCode


def signature_hits(blob):
    """bit positions of every 48-bit block / end-of-stream signature"""
    bits = np.unpackbits(np.frombuffer(blob, dtype=np.uint8)).astype(np.uint64)
    if len(bits) < 48:
        return []
    w = np.zeros(len(bits) - 47, dtype=np.uint64)
    for i in range(48):
        w = (w << np.uint64(1)) | bits[i:len(bits) - 47 + i]
    return np.nonzero((w == MAGIC_BLOCK) | (w == MAGIC_END))[0].tolist()


# ------------------------------------------------------------------------------------------------- the families ----
BLOCK_SIG = [0x31, 0x41, 0x59, 0x26, 0x53, 0x59]
END_SIG = [0x17, 0x72, 0x45, 0x38, 0x50, 0x90]
DENSE_USED = tuple(range(1, 255))          # 254 bytes: 256 symbols, end-of-block = 255; with 8-bit codes a symbol is its byte


def dense(pattern, k, orig=0):
    """symbol data that spells `pattern` byte for byte, k times: a signature hit every 48 bits of coded data"""
    return lambda: Blk(A=pattern * k + [255], used=DENSE_USED, orig=orig, lens=8)


def dense_check(case):
    blob, pos, blocks = case.built
    hits = signature_hits(blob)
    assert len(hits) > len(blob) // 16 + 64          # more than the scan's candidate buffer of one window
    assert set(pos) <= set(hits)


def text(n, seed=3):
    return gen_text(n, seed).tobytes()


def sig_cases(full):
    k = 150_000 if full else 3000
    return [
        Case("sig-block-magic-1KB", [(9, [dense(BLOCK_SIG, 150)])], scan=True, check=dense_check),
        Case(f"sig-block-magic-{k}", [(9, [dense(BLOCK_SIG, k)])], scan=True, check=dense_check),
        Case("sig-end-magic", [(9, [dense(END_SIG, 700)])], scan=True, check=dense_check),
        Case("sig-both-magics", [(9, [dense(BLOCK_SIG + END_SIG, 400)])], scan=True, check=dense_check),
        Case("sig-multistream-false-hits-around-true-blocks",
             [(9, [dense(BLOCK_SIG, 300), lambda: Blk(content=text(3000, 1))]),
              (5, [lambda: Blk(content=text(2000, 2)), dense(END_SIG + BLOCK_SIG, 200, orig=17), lambda: Blk(content=text(500, 3))]),
              (9, [dense(END_SIG, 250)])], multistream=True, scan=True, check=dense_check),
    ]


def lits(n, seed, hi=4):
    """n literals of MTF ranks 1..hi-1"""
    return [sym(int(r)) for r in np.random.default_rng(seed).integers(1, hi, n)]


def offsets_cases(full):
    cs = []
    for j in (1, 2):
        for d in (1, 2, 3):           # the run's first digit d symbols before symbol 4096 j, the rest after it
            A = lits(SEG * j - d, d) + [0, 1, 0, 1, 1] + lits(300, 9) + [257]
            cs.append(Case(f"offsets-run-across-{SEG * j}-minus-{d}", [(9, [lambda A=A: Blk(A=A, used=ALL)])],
                           check=lambda c, i=SEG * j - d: _assert_run_at(c, i)))
    cs.append(Case("offsets-block-starts-with-a-run", [(9, [lambda: Blk(A=[1, 0, 1] + lits(5000, 1) + [257], used=ALL)])]))
    v19 = (1 << 19) - 1 + 300_000                       # a run of 19 digits
    assert len(run_digits(v19)) == 19
    cs.append(Case("offsets-run-of-19-digits", [(9, [lambda: Blk(A=lits(SEG - 7, 2) + run_digits(v19) + lits(50, 3) + [257], used=ALL)])],
                   sim=False))
    for nd in (20, 22):                                 # at least 2^20 - 1 bytes: a Data error
        cs.append(Case(f"offsets-run-of-{nd}-digits", [(9, [lambda nd=nd: Blk(A=lits(SEG - 9, 4) + [0] * nd + lits(5, 5) + [257], used=ALL)])],
                       check=lambda c: _assert(c.expect == Err.DATA_ERROR)))
    for e in (SEG * 2, SEG * 2 - 1):                   # end-of-block at symbol e
        cs.append(Case(f"offsets-end-of-block-at-{e}", [(9, [lambda e=e: Blk(A=lits(e - 3, 6) + [0, 1, 0] + [257], used=ALL)])],
                       check=lambda c, e=e: _assert(len(c.built[2][0].A) == e + 1)))
    return cs


def _assert(x):
    assert x


def _assert_run_at(case, i):
    A = case.built[2][0].A
    assert A[i - 1] >= 2 and A[i] <= 1 and A[i + 4] <= 1 and A[i + 5] >= 2


RANKS = (1, 31, 32, 33, 63, 64, 95, 96, 224, 255)


def imtf_cases(full):
    cs = []
    for where, at in (("lane-0", 32 * 5), ("lane-31", 32 * 5 + 31), ("segment-first", SEG), ("segment-last", 2 * SEG - 1)):
        # one block per rank, with the rank exactly at `at`; the filler ranks reach the cold rows too
        cs.append(Case(f"imtf-ranks-at-{where}",
                       [(9, [lambda r=r, at=at: Blk(A=lits(at, r, 70) + [sym(r)] + lits(300, r + 1, 70) + [257], used=ALL) for r in RANKS])],
                       check=lambda c, at=at: _assert([b.A[at] - 1 for b in c.built[2]] == list(RANKS))))
    cs.append(Case("imtf-segment-of-run-digits", [(9, [lambda: Blk(A=lits(SEG - 2, 1) + [0] * (SEG + 2) + lits(9, 2) + [257], used=ALL)])],
                   check=lambda c: _assert(c.expect == Err.DATA_ERROR)))
    cs.append(Case("imtf-run-split-over-two-segments",
                   [(9, [lambda: Blk(A=lits(SEG - 2, 3, 70) + run_digits(5000) + lits(2000, 4, 70) + [257], used=ALL)])],
                   check=lambda c: _assert(c.built[2][0].A[SEG - 3] >= 2 and c.built[2][0].A[SEG - 2] <= 1 and c.built[2][0].A[SEG] <= 1)))
    for nseg, n in (("1", 3000), ("2", 7000)) + ((("220", 899_000),) if full else ()):
        cs.append(Case(f"imtf-{nseg}-segments", [(9, [lambda n=n: Blk(content=no_runs_of_four(n, 11))])],
                       check=lambda c, nseg=nseg: _assert((len(c.built[2][0].A) + SEG - 1) // SEG == int(nseg))))
    for nu in (1, 2, 255, 256):
        used = ALL[:nu]
        content = bytes(np.random.default_rng(nu).choice(np.array(used, dtype=np.uint8), 6000 if nu > 1 else 3))
        cs.append(Case(f"imtf-used-map-{nu}", [(9, [lambda content=content, used=used: Blk(L=O.bwt(content)[0], used=used,
                                                                                             orig=O.bwt(content)[1])])],
                       check=lambda c, nu=nu: _assert(len(c.built[2][0].used) == nu)))
    return cs


def random_L(n, alpha, seed):
    return np.random.default_rng(seed).integers(0, alpha, n).astype(np.uint8).tobytes()


def ibwt_cases(full):
    cs = []
    counts = [1, 2, 63, 64, 65, 4032, 4033, 4096, 4097, TILE * 2 - 1, TILE * 2 + 1, 20_000] + ([TILE * 50, 900_000] if full else [])
    for n in counts:
        for alpha in (2, 256):
            L = random_L(n, alpha, n + alpha)
            cs.append(Case(f"ibwt-count-{n}-alpha-{alpha}", [(9, [lambda L=L, a=alpha: Blk(L=L, used=ALL[:a], orig=len(L) // 3)])],
                           libbz2=False, sim=n <= 20_000))
    # pos0 (the slot origPtr leads to) at 0, at a multiple of 64 and at the last slot
    L = random_L(8193, 26, 3)
    order = np.argsort(np.frombuffer(L, dtype=np.uint8), kind="stable")
    inv = np.argsort(order)
    for name, p0 in (("0", 0), ("64x", 64 * 70), ("last", 8192)):
        orig = int(inv[p0])
        cs.append(Case(f"ibwt-pos0-{name}", [(9, [lambda L=L, orig=orig: Blk(L=L, used=ALL[:26], orig=orig)])], libbz2=False,
                       check=lambda c, p0=p0: _assert(cycle_of(c.built[2][0].L, c.built[2][0].orig)[0] == p0)))
    # a start cycle shorter than n that does not divide it
    for n, alpha in ((5000, 2), (20_000, 26)):
        for seed in range(100):
            L = random_L(n, alpha, seed)
            c = len(cycle_of(L, 0))
            if c < n and n % c:
                break
        cs.append(Case(f"ibwt-start-cycle-{c}-of-{n}", [(9, [lambda L=L, a=alpha: Blk(L=L, used=ALL[:a], orig=0)])], libbz2=False,
                       check=lambda c, n=n: _assert(n % len(cycle_of(c.built[2][0].L, 0)) != 0)))
    # a start cycle that holds no splitter but pos0
    pick = None
    for seed in range(50):
        L = random_L(4097, 2, seed)
        order = np.argsort(np.frombuffer(L, dtype=np.uint8), kind="stable")
        inv = np.argsort(order)
        seen = set()
        for s in range(len(L)):
            if s in seen:
                continue
            cyc = cycle_of(L, int(inv[s]))
            seen |= set(cyc)
            if 1 < len(cyc) < len(L) and not any(x % SPL == 0 for x in cyc):
                pick = int(inv[s])
                break
        if pick is not None:
            break
    cs.append(Case("ibwt-start-cycle-without-splitters", [(9, [lambda L=L, pick=pick: Blk(L=L, used=(0, 1), orig=pick)])], libbz2=False,
                   check=lambda c: _assert(not any(x % SPL == 0 for x in cycle_of(c.built[2][0].L, c.built[2][0].orig)))))
    # periodic blocks
    for per in (1, 2, 63, 64, 65, "half"):
        n = 20_000 if full else 6000
        p = n // 2 if per == "half" else per
        unit = bytes(range(1, p + 1)) if p < 256 else no_runs_of_four(p, p)
        content = unit * (n // p)
        cs.append(Case(f"ibwt-period-{per}", [(9, [lambda content=content: Blk(content=content)])], libbz2=p > 1,
                       check=lambda c, p=p: _assert(len(cycle_of(c.built[2][0].L, c.built[2][0].orig)) == p)))
    return cs


def rle1_content(end, l, seed):
    """RLE1 bytes with a run of l 'z' whose last byte is at index `end`, no other run of four"""
    head, tail = bytearray(no_runs_of_four(end + 1 - l, seed)), bytearray(no_runs_of_four(300, seed + 1))
    head = head.replace(b"z", b"y")
    tail = tail.replace(b"z", b"y")
    return bytes(head + b"z" * l + tail)


def _run_ends_at(seq, e, l):
    assert seq[e - l + 1:e + 1] == b"z" * l and seq[e - l] != ord("z") and seq[e + 1] != ord("z")


def rle1_cases(full):
    cs = []
    for width, strip in STRIP.items():
        for l in range(5, 10):                               # l mod 5 = 0..4
            for where, end in (("thread", 8 * 37 - 1), ("strip", strip - 1), ("strip-2", 2 * strip - 1)):
                cs.append(Case(f"rle1-{width}-run-{l}-ends-{where}", [(9, [lambda e=end, l=l: Blk(content=rle1_content(e, l, l))])],
                               check=lambda c, e=end, l=l: _run_ends_at(c.built[2][0].seq, e, l)))
            tail = no_runs_of_four(strip * 2 - 1 - l, 3).replace(b"z", b"y")
            cs.append(Case(f"rle1-{width}-run-{l}-ends-block", [(9, [lambda t=tail, l=l: Blk(content=t + b"z" * l)])], libbz2=l % 5 != 4))
        cs.append(Case(f"rle1-{width}-count-byte-first-of-strip",
                       [(9, [lambda s=strip: Blk(content=rle1_content(s - 1, 4, 9)[:s] + b"\x05" + no_runs_of_four(700, 4))])],
                       check=lambda c, s=strip: _assert(c.built[2][0].seq[s - 4:s + 1] == b"zzzz\x05")))
    cs += [
        Case("rle1-run-longer-than-a-strip", [(9, [lambda: Blk(content=text(3000, 1) + b"z" * 20_003 + text(3000, 2))])]),
        Case("rle1-counts-0-and-255", [(9, [lambda: Blk(content=text(5000, 3) + b"zzzz\x00" + text(4500, 4) + b"yyyy\xff" + text(100, 5))])]),
        Case("rle1-trailing-run-without-count", [(9, [lambda: Blk(content=text(9000, 6) + b"zzzz")])], libbz2=False),
    ]
    return cs


def crc_cases(full):
    cs = []
    for j in ((1, 2, 13) if full else (1, 2)):
        for d in (-1, 0, 1):
            n = CRC_CHUNK * j + d
            cs.append(Case(f"crc-output-{j}x64KiB{d:+d}", [(9, [lambda n=n, j=j: Blk(content=no_runs_of_four(n, j))])],
                           check=lambda c, n=n: _assert(len(c.expect) == n), sim=n < 140_000))
    cs.append(Case("crc-blocks-at-odd-offsets", [(9, [lambda s=s, n=n: Blk(content=no_runs_of_four(n, s)) for s, n in
                                                      ((1, 70_001), (2, 65_537), (3, 3), (4, 131_071))])],
                   check=lambda c: _assert(all(len(b.out) % 2 for b in c.built[2]))))
    if full:
        cs.append(Case("crc-largest-block-output", [(9, [lambda: Blk(content=b"aaaa\xff" * 180_000)])],
                       check=lambda c: _assert(len(c.expect) == 180_000 * 259)))
    return cs


def families(full):
    return {"sig": sig_cases(full), "offsets": offsets_cases(full), "imtf": imtf_cases(full), "ibwt": ibwt_cases(full),
            "rle1": rle1_cases(full), "crc": crc_cases(full)}


SIM = {c.name: c for cs in families(False).values() for c in cs if c.sim}
GPU = {c.name: c for cs in families(True).values() for c in cs}


# ---------------------------------------------------------------------------------------------------- checking ----
def first_diff(stage, blk, got, want):
    got, want = np.asarray(got, dtype=np.int64), np.asarray(want, dtype=np.int64)
    if len(got) == len(want) and (got == want).all():
        return
    n = min(len(got), len(want))
    i = int(np.argmax(got[:n] != want[:n])) if n and (got[:n] != want[:n]).any() else n
    raise AssertionError(f"stage {stage}, block at bit {blk}, index {i}: got {got[i:i + 8].tolist()} want {want[i:i + 8].tolist()} "
                         f"(lengths {len(got)} / {len(want)})")


def check_stages(eng, case):
    """the stage dumps of the last decode batch against the reference, in stage order"""
    blob, pos, blocks = case.built
    by_pos = dict(zip(pos, blocks))
    cands = eng.decode_candidates()
    if case.one_batch and not any(c.bitpos in by_pos for c in cands):
        raise AssertionError(f"stage signatures: the last decode batch holds none of the blocks (candidates: {len(cands)})")
    seen = 0
    for k, c in enumerate(cands):
        b = by_pos.get(c.bitpos)
        if b is None or c.kind != 0:
            continue
        syms, offs, L = eng.decode_stages(k, len(b.A))
        first_diff("symbols", c.bitpos, syms, b.A)
        first_diff("offsets", c.bitpos, offs, b.offs)
        assert c.err == 0 and c.nsym == len(b.A), f"block at bit {c.bitpos}: error {c.err} after correct symbols and offsets"
        first_diff("L column", c.bitpos, np.frombuffer(L.tobytes(), dtype=np.uint8), np.frombuffer(b.L, dtype=np.uint8))
        seen += 1
    inv = eng.decode_inverted()
    for k, seq in inv:
        b = by_pos[cands[k].bitpos]
        first_diff("inverse BWT", cands[k].bitpos, np.frombuffer(seq, dtype=np.uint8), np.frombuffer(b.seq, dtype=np.uint8))
    return seen, len(inv)


def outcome(fn):
    try:
        return ("ok", fn())
    except (Bzip2Error, O.OracleError) as e:
        return ("err", e.errorCode)


def run_case(case, engs, pool, full):
    blob, pos, blocks = case.built
    ms = case.multistream
    if case.check:
        case.check(case)
    want = ("ok", case.expect) if isinstance(case.expect, bytes) else ("err", case.expect)
    if want[0] == "ok":
        assert want[1] == b"".join(b.out for b in blocks)
        if case.libbz2 and not any(b.trailing_run for b in blocks):
            assert bz2.decompress(blob) == want[1]
    for name, eng in engs.items():
        got = outcome(lambda: eng.decompressFile(blob, None, ms))
        if got != want and want[0] == "ok":         # name the first stage that differs (a wrong block fails its CRC)
            check_stages(eng, case)
            if got[0] == "ok":
                first_diff("output bytes", pos[0], np.frombuffer(got[1], dtype=np.uint8), np.frombuffer(want[1], dtype=np.uint8))
            raise AssertionError(f"stage output bytes / CRC: every stage up to the inverse BWT equals the reference, {name} failed with {got[1]}")
        assert got == want, name
        if want[0] == "ok":
            seen, inverted = check_stages(eng, case)
            if case.one_batch:                      # every block was checked
                assert seen == inverted == len(blocks), name
    if case.scan:
        check_scan(engs[next(iter(engs))], pool, blob, ms, want[1], pos)


def check_scan(eng, pool, blob, ms, out, pos):
    """every entry point that scans for signatures, against the oracle: table, index, search, recover, the stream
    decoder in small pieces and the pool in small slices"""
    rows = []
    eng.table(blob, lambda p, s: rows.append((p, s)), ms)
    assert rows == O.table(blob, ms) and [p for p, _ in rows] == pos
    ix = eng.index(blob, ms)
    assert [(int(e["bit_begin"]), int(e["out_bytes"])) for e in ix.entries] == rows
    pat, hits = out[len(out) // 2:len(out) // 2 + 4], []
    i = out.find(pat)
    while i >= 0:
        hits.append(i)
        i = out.find(pat, i + 1)
    assert eng.search(blob, pat, multistream=ms).matches["offset"].tolist() == hits
    data, regs = eng.recover(blob)
    assert data == out and all(r.status == 0 for r in regs)
    assert sorted(r.bit_begin for r in regs if r.kind == REGION_BLOCK) == pos
    piece = max(1 << 16, len(blob) // 64)
    assert eng.decompressStream(io.BytesIO(blob), None, ms, chunk_bytes=piece, piece_bytes=piece // 13) == out
    assert pool.decompressFile(blob, None, ms, slice_bytes=max(16_000, len(blob) // 64)) == out


# ------------------------------------------------------------------------------------------------------- engines ----
def _engines(library, widths_auto):
    """parse kernel x RLE1 inverse width: (1, 512) and (2, 1024) cover both of each"""
    engs = {}
    old = os.environ.get("BZ2B200_PARSE")
    try:
        for mode, width in (("1", 512), ("2", 1024)) + ((("0", 0),) if widths_auto else ()):
            os.environ["BZ2B200_PARSE"] = mode
            e = Bzip2Engine(0, library)
            e.debug_set_rle1_threads(width)
            engs[f"parse{mode}-rle1x{width}"] = e
    finally:
        if old is None:
            os.environ.pop("BZ2B200_PARSE", None)
        else:
            os.environ["BZ2B200_PARSE"] = old
    pool = Bzip2Pool([0], 2, library=library)
    pool.debug_rle1_threads(512)
    return engs, pool


@pytest.fixture(scope="module")
def sim_engines(sim_engine):
    engs, pool = _engines(_native.Library(SIM_SO), False)
    yield engs, pool
    for e in engs.values():
        e.close()
    pool.close()


@pytest.fixture(scope="module")
def gpu_engines():
    engs, pool = _engines(None, True)
    yield engs, pool
    for e in engs.values():
        e.close()
    pool.close()


@pytest.mark.parametrize("name", list(SIM))
def test_stages_sim(sim_engines, oracle, name):
    run_case(SIM[name], *sim_engines, False)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GPU))
def test_stages_gpu(gpu_engines, oracle, name):
    run_case(GPU[name], *gpu_engines, True)


# ---------------------------------------------------------------------------------------------------- batches ----
def mixed(full):
    """blocks of every family in one stream"""
    pick = ["sig-block-magic-1KB", "offsets-run-across-4096-minus-2", "offsets-end-of-block-at-8191", "imtf-ranks-at-lane-31",
            "imtf-run-split-over-two-segments", "ibwt-count-4097-alpha-2", "ibwt-pos0-64x", "ibwt-period-63", "rle1-512-run-8-ends-strip",
            "rle1-1024-count-byte-first-of-strip", "crc-output-1x64KiB+1"]
    src = GPU if full else SIM
    return Case("mixed", [(9, [f for n in pick for _, specs in src[n].streams for f in specs])], libbz2=False)


def run_batches(engs, full):
    case = mixed(full)
    blob, pos, blocks = case.built
    assert len(pos) > 12 and isinstance(case.expect, bytes)
    for name, eng in engs.items():
        eng.debug_set_decode_batch(3)           # neighbours fall in different batches
        try:
            got = eng.decompressFile(blob)
        finally:
            eng.debug_set_decode_batch(0)
        if got != case.expect:
            first_diff("output bytes", pos[0], np.frombuffer(got, dtype=np.uint8), np.frombuffer(case.expect, dtype=np.uint8))


def test_batches_sim(sim_engines, oracle):
    run_batches(sim_engines[0], False)


@pytest.mark.gpu
def test_batches_gpu(gpu_engines, oracle):
    run_batches(gpu_engines[0], True)


@pytest.mark.gpu
@pytest.mark.parametrize("nblocks", [140, 200])
def test_rle1_width_by_block_count_gpu(gpu_engines, oracle, nblocks):
    """no setter: 1024 threads for a batch of at most one block per SM (148 on a B200), 512 above"""
    eng = gpu_engines[0]["parse0-rle1x0"]
    blocks = [Blk(content=rle1_content(STRIP[512 << (k % 2)] - 1, 5 + k % 5, k)) for k in range(nblocks)]
    bits, pos = make_stream(9, [dict(bits=b.bits, crc=b.crc) for b in blocks])
    blob, want = pack(bits), b"".join(b.out for b in blocks)
    assert eng.decompressFile(blob) == want == O.decompress(blob)
    assert len(eng.decode_inverted()) == nblocks


@pytest.mark.gpu
@pytest.mark.parametrize("straddler", ["true", "false"])
def test_signature_across_scan_window_gpu(gpu_engines, oracle, straddler):
    """an input longer than one 64 MiB scan window with a true (or a false) signature across byte 64 MiB: a leading
    stream of computed length, then a stream dense with false signatures"""
    engs, pool = gpu_engines
    eng = engs["parse0-rle1x0"]
    W = 64 << 20
    dense_blk = dense(BLOCK_SIG, 3000)()
    d_bits, _ = make_stream(9, [dict(bits=dense_blk.bits, crc=dense_blk.crc)])
    d = pack(d_bits)
    hits = signature_hits(d)
    h = hits[len(hits) // 2] if straddler == "false" else 32      # bit of the straddling signature in the dense stream
    lo, hi = W - (h + 47) // 8, W - h // 8                         # lead lengths that put it across byte W (bit 8 W)
    rnd = np.random.default_rng(1).integers(0, 256, W + (1 << 20), dtype=np.uint8)
    n = W - (1 << 18)
    for _ in range(60):
        lead = eng.compressFile(rnd[:n].tobytes(), None, 9)
        if lo <= len(lead) <= hi and 8 * len(lead) + h < 8 * W < 8 * len(lead) + h + 48:
            break
        n += max(-(1 << 20), min(1 << 20, (lo + hi) // 2 - len(lead))) or 1
    else:
        pytest.fail("no lead length puts the signature across byte 64 MiB")
    blob = lead + d
    assert 8 * len(lead) + h - 8 * (W - 64) in signature_hits(blob[W - 64:W + 64])
    out = rnd[:n].tobytes() + dense_blk.out
    assert O.decompress(blob, True) == out and bz2.decompress(blob) == out
    for e in engs.values():
        assert e.decompressFile(blob, None, True) == out
    check_scan(eng, pool, blob, True, out, [p for p, _ in O.table(blob, True)])
