"""Compressor conformance: inputs built to reach each compress kernel's internal limits, compared with the oracle stage by stage.

Every case is compressed by the engine and by `oracle.compress`; the streams must be byte-identical.  When they differ,
`stage_diff` names the first stage and block that differ, in pipeline order: block table, RLE1 bytes, BWT (L column and
origPtr), MTF/RLE2 symbols, block shape (alphabet, m, tables, selectors count), selectors, code lengths, and last the
block's bit count (a function of the stages before it, so a difference there alone points at the emission).

Every generator asserts the structure it claims -- from the oracle's stages, from the data, or from the Python models
below of the round-0 code (`sym_code`, a copy of k_sym_tab's bisection) and of the prefix-doubling rounds
(`doubling_groups`) -- so a case cannot drift off its target without failing.

The simulator leg (`-m "not gpu"`) runs every family at small sizes (tiny blocks through the block-cap hook) and a few
full-size blocks; the GPU leg runs every family at level-9 and level-1 block size and one 40 MB input that mixes them.
"""
import os

import numpy as np
import pytest

B9, B1 = 899_981, 99_981
KEY_BITS, KEY_SLACK = 44, 2  # KEY_BITS and KEY_SLACK of csrc/bwt.cuh
CPUS = os.cpu_count() or 1


@pytest.fixture(params=["sim", pytest.param("gpu", marks=pytest.mark.gpu)])
def leg(request):
    """(engine, full): `full` is True on the GPU, where every family also runs at full block size"""
    if request.param == "sim":
        return request.getfixturevalue("sim_engine"), False
    return request.getfixturevalue("gpu_engine"), True


@pytest.fixture
def block_cap(leg, oracle):
    """set_cap(c) overrides the block capacity of both sides for the rest of the test (0 = the level's)"""
    eng = leg[0]

    def set_cap(cap):
        oracle.set_block_cap(cap)
        eng.debug_set_block_cap(cap)
    yield set_cap
    set_cap(0)


# ---------------------------------------------------------------------------------------------------------------------
# comparison

def _u8(data):
    return np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data


def _first_diff(a, b):
    a, b = np.asarray(a), np.asarray(b)
    n = min(a.size, b.size)
    d = np.flatnonzero(a[:n] != b[:n])
    return int(d[0]) if d.size else n


def stage_diff(engine, oracle, data, level, cap=0):
    """None if every stage of every block of the last compress call (one batch) equals the oracle's, else a message naming
    the first stage that differs, the block and the first differing index"""
    arr = _u8(data)
    B = cap or level * 100_000 - 19
    starts, lens, crcs = oracle.cut_points(arr, level)
    recs = engine.block_table()
    got, exp = [(r.s, r.n, r.crc) for r in recs], list(zip(starts[:-1], lens, crcs))
    if got != exp:
        i = _first_diff(np.array(got[:len(exp)] or [(0, 0, 0)]), np.array(exp[:len(got)] or [(0, 0, 0)]))
        return (f"stage 1 (block table): entry {i}: device {got[i] if i < len(got) else None} vs oracle "
                f"{exp[i] if i < len(exp) else None} ({len(got)} vs {len(exp)} blocks)")
    metas = engine.block_meta()
    for k, r in enumerate(recs):
        blk, _, _ = oracle.rle1_block(arr[r.s:], B)
        dev = engine.debug_fetch(1, k, r.n)
        if dev.tobytes() != blk.tobytes():
            return f"stage 2 (RLE1 bytes): block {k}, index {_first_diff(dev, blk)}"
        st = oracle.block_stages(blk)
        dev = engine.debug_fetch(2, k, r.n)
        if dev.tobytes() != st["U"].tobytes():
            return f"stage 3 (BWT L column): block {k}, index {_first_diff(dev, st['U'])}"
        if r.orig_ptr != st["orig_ptr"]:
            return f"stage 3 (BWT origPtr): block {k}: device {r.orig_ptr} vs oracle {st['orig_ptr']}"
        mt = metas[k]
        A = np.frombuffer(engine.debug_fetch(3, k, 2 * mt.m).tobytes(), dtype=np.uint16)
        if not np.array_equal(A, st["A"]):
            return f"stage 4 (MTF/RLE2 symbols): block {k}, index {_first_diff(A, st['A'])} ({A.size} vs {st['A'].size} symbols)"
        shape = ("alpha", "m", "n_groups", "n_sel")
        gs, es = tuple(getattr(mt, f) for f in shape), tuple(st[f] for f in shape)
        if gs != es:
            return f"stage 5 (block shape {shape}): block {k}: device {gs} vs oracle {es}"
        sel, L = engine.block_huffman(k)
        if not np.array_equal(sel, st["sel"]):
            return f"stage 6 (selectors): block {k}, group {_first_diff(sel, st['sel'])}"
        L = L[:mt.n_groups, :mt.alpha + 2]
        if not np.array_equal(L, st["lens"]):
            t, s = np.argwhere(L != st["lens"])[0]
            return f"stage 7 (code lengths): block {k}, table {t}, symbol {s}: device {L[t, s]} vs oracle {st['lens'][t, s]}"
        if mt.bits != st["bits"] + 80:
            return f"stage 8 (block bits): block {k}: device {mt.bits} vs oracle {st['bits'] + 80}"
    return None


def check(engine, oracle, data, level=9, cap=0, label=""):
    """byte-identical stream (else: the first stage that differs); the oracle's stream decodes back to the input unless
    the case reproduces defect D1 (a stream the reference's own decoder rejects).  Returns the oracle's stats."""
    exp, st = oracle.compress(data, level, threads=CPUS, return_stats=True)
    got = engine.compressFile(data, None, level)
    if got != exp:
        where = stage_diff(engine, oracle, data, level, cap) or "every stage matches: the stream's framing differs"
        pytest.fail(f"{label} L{level}: stream differs from the oracle at byte {_first_diff(np.frombuffer(got, np.uint8), np.frombuffer(exp, np.uint8))} "
                    f"({len(got)} vs {len(exp)} bytes); first difference: {where}")
    if not st.d1_triggered:
        assert oracle.decompress(exp, threads=CPUS) == bytes(data), label
    return st


# ---------------------------------------------------------------------------------------------------------------------
# models of the BWT's round 0 and doubling rounds

def sym_code(block):
    """k_sym_tab: (lens[256], vals[256], maxlen, L) of the order-preserving prefix-free code of a block's bytes"""
    cnt = np.bincount(_u8(block), minlength=256).astype(np.int64)
    used = np.flatnonzero(cnt)
    alpha = used.size
    P = np.concatenate([[0], np.cumsum(cnt[used])])
    lens, vals = np.zeros(256, np.int64), np.zeros(256, np.int64)
    if alpha == 1:
        lens[used[0]] = 1
    elif alpha > 1:
        lb = 1
        while (1 << lb) < alpha:
            lb += 1
        lmax = lb + (KEY_SLACK if alpha > 2 else 0)
        for r, c in enumerate(used):
            lo, hi, ln, val = 0, alpha, 0, 0
            while hi - lo > 1:
                cap = 1 << (lmax - ln - 1)
                mid2 = P[lo] + P[hi]
                a, z = lo + 1, hi - 1
                while a < z:
                    m = (a + z) >> 1
                    if 2 * P[m] < mid2:
                        a = m + 1
                    else:
                        z = m
                s = a
                if s > lo + 1 and 2 * P[s] >= mid2 and mid2 - 2 * P[s - 1] < 2 * P[s] - mid2:
                    s -= 1
                s = max(s, hi - cap if hi > cap + lo else lo + 1)
                s = min(s, lo + cap if lo + cap < hi - 1 else hi - 1)
                val <<= 1
                if r >= s:
                    val |= 1
                    lo = s
                else:
                    hi = s
                ln += 1
            lens[c], vals[c] = ln, val
    maxlen = max(1, int(lens.max()))
    return lens, vals, maxlen, KEY_BITS // maxlen


def round0_keys(block, lens, vals):
    """the 44-bit key of every rotation: the first 44 bits of its code string (the block read cyclically)"""
    b = _u8(block)
    n = b.size
    ext = np.resize(b, n + 44)
    ln, vl = lens[ext], vals[ext]
    cum = np.concatenate([[0], np.cumsum(ln)])
    total = int(cum[-1])
    sym = np.repeat(np.arange(ext.size), ln)
    pos = np.arange(total) - cum[sym]
    bits = ((vl[sym] >> (ln[sym] - 1 - pos)) & 1).astype(np.uint8)
    packed = np.concatenate([np.packbits(bits), np.zeros(8, np.uint8)])
    o = cum[:n]
    win = packed[(o >> 3)[:, None] + np.arange(7)].astype(np.uint64)
    w = np.zeros(n, np.uint64)
    for j in range(7):
        w = (w << np.uint64(8)) | win[:, j]
    w = (w << (o & 7).astype(np.uint64)) & np.uint64((1 << 56) - 1)
    return w >> np.uint64(56 - KEY_BITS)


def doubling_groups(block):
    """the prefix-doubling sort of bwt.cuh / refine.cuh on one block, as the kernels run it: round 0 ranks by the 44-bit
    key, round r >= 1 by (rank, rank of the rotation h = L << (r - 1) further on), and by descending index once h >= n.
    Returns (L, maxlen, rounds), rounds[r] = (sizes of the groups of > 1 rotation after round r in SA order, the group id
    of every rotation); the sort takes len(rounds) + 1 rounds (the last one leaves no group)."""
    lens, vals, maxlen, L = sym_code(block)
    n = len(block)
    _, rank = np.unique(round0_keys(block, lens, vals), return_inverse=True)
    rounds, r, idx = [], 0, np.arange(n, dtype=np.int64)
    while True:
        cnt = np.bincount(rank)
        if not (cnt > 1).any():
            return L, maxlen, rounds
        rounds.append((cnt[cnt > 1], rank))
        h = min(L << r, 1 << 24)
        key2 = (n - 1 - idx) if h >= n else rank[(idx + h) % n]
        _, rank = np.unique(rank.astype(np.int64) * (n + 1) + key2, return_inverse=True)
        r += 1


def _rle1(oracle, data, cap):
    blk, used, _ = oracle.rle1_block(_u8(data), cap)
    return blk, used


# ---------------------------------------------------------------------------------------------------------------------
# group sizes: k copies of a string S in filler -> a group of exactly k rotations that survives a chosen number of rounds

def groups_input(rng, k, slen, lead=0, n_fill=0):
    """`lead` copies of S0 = 00 00 .. and k copies of S = 00 01 .. in filler over bytes 2..255 (no byte 0 or 1 elsewhere):
    after round 0 the active list starts with the S0 group (`lead` slots) and then the S group (k slots)"""
    S0 = bytes([0, 0]) + rng.integers(2, 256, max(slen - 2, 1), dtype=np.uint8).tobytes()
    S = bytes([0, 1]) + rng.integers(2, 256, max(slen - 2, 1), dtype=np.uint8).tobytes()
    pieces = [S0] * lead + [S] * k
    order = rng.permutation(len(pieces))
    gaps = rng.integers(3, 9, len(pieces)) + (n_fill // max(len(pieces), 1))
    out = []
    for j, g in zip(order, gaps):
        f = rng.integers(2, 256, int(g), dtype=np.uint8)
        f[1:][f[1:] == f[:-1]] ^= 0x80   # no runs in the filler (RLE1 is the identity)
        out += [pieces[j], f.tobytes()]
    return b"".join(out), S, S0


def assert_group(block, S, k, lead, survive):
    """the S group has exactly k rotations, starts at offset `lead` of the active list and survives exactly `survive`
    doubling rounds (0 = it splits in round 1); returns the model's rounds"""
    b = bytes(block)
    assert b.count(S) == k
    L, maxlen, rounds = doubling_groups(block)
    first = b.find(S)
    whole = 0   # rounds (round 0 included) after which the group is still whole
    for r, (sizes, rank) in enumerate(rounds):
        g = rank[first]
        if int(np.count_nonzero(rank == g)) != k:
            break
        if r == 0:   # offset of the group in the list sorted by round 1: the groups of > 1 rotation before it
            cnt = np.bincount(rank)
            assert int(cnt[:g][cnt[:g] > 1].sum()) == lead
        whole = r + 1
    assert whole - 1 == survive, (whole - 1, survive, L, maxlen)
    return rounds


def group_case(rng, k, survive, lead=0, n_fill=0):
    """groups_input whose S group survives exactly `survive` doubling rounds: |S| grows from (2^survive - 1) L + 2 until
    the model says so (two copies stay tied in round r while the key at offset (2^r - 1) L lies inside S)"""
    for slen in range((2 ** survive - 1) * 4 + 2, (2 ** survive - 1) * 5 + 16):
        data, S, _ = groups_input(np.random.default_rng(rng.integers(1 << 30)), k, slen, lead, n_fill)
        try:
            return data, S, assert_group(np.frombuffer(data, np.uint8), S, k, lead, survive)
        except AssertionError:
            continue
    raise AssertionError(f"no |S| gives a group of {k} that survives {survive} rounds")


@pytest.mark.parametrize("k", [2, 32, 33, 256, 257, 1024, 1025, 2048, 2049, 5000])
def test_group_sizes(leg, oracle, k):
    """k rotations tied on S, for S long enough to survive 0, 1, 2 and 3 doubling rounds; at k > 1024 the group is a BIG
    group (k_group_bounds / k_big_*).  The filler over bytes 2..255 has no runs, so the block is the input itself."""
    eng, full = leg
    rng = np.random.default_rng(k)
    survives = (0, 1, 2, 3) if full else ((0, 3) if k <= 1025 else (1,) if k < 5000 else ())
    for surv in survives:
        n_fill = max(0, (B9 - 60_000) // k - 40) if full else 0
        data, S, rounds = group_case(rng, k, surv, 0, n_fill)
        blk, used = _rle1(oracle, data, B9)
        assert used == len(data) and blk.tobytes() == data   # the model ran on the block itself
        check(eng, oracle, data, 9, label=f"k={k} survive={surv}")
        assert eng.stats().sort_rounds == len(rounds) + 1


def test_big_groups_at_list_boundaries(leg, oracle, block_cap):
    """a big group that starts at, ends at and straddles a nominal 1024-slot boundary of the active list; many big groups
    in one round; big groups in several blocks of one batch"""
    eng, full = leg
    rng = np.random.default_rng(77)
    for lead, k, where in ((1024, 1100, "starts at"), (924, 1124, "ends at"), (500, 1025, "straddles"), (1023, 2050, "straddles")):
        data, S, S0 = groups_input(rng, k, 14, lead)
        blk, _ = _rle1(oracle, data, B9)
        rounds = assert_group(blk, S, k, lead, 1)
        lo, hi = lead, lead + k
        if where == "starts at":
            assert lo % 1024 == 0
        elif where == "ends at":
            assert hi % 1024 == 0
        else:
            assert lo // 1024 != (hi - 1) // 1024 and lo % 1024 and hi % 1024
        check(eng, oracle, data, 9, label=f"big group {where} a boundary: lead={lead} k={k}")
        assert eng.stats().sort_rounds == len(rounds) + 1
    # many big groups in one round: 24 strings, 1030..1300 copies each
    parts = []
    for j in range(24 if full else 6):
        S = bytes([2 + j]) + rng.integers(2, 256, 13, dtype=np.uint8).tobytes()
        parts += [S] * int(rng.integers(1030, 1300))
    rng.shuffle(parts)
    data = b"".join(p + rng.integers(2, 256, 5, dtype=np.uint8).tobytes() for p in parts)
    blk, used = _rle1(oracle, data, B9)
    sizes = doubling_groups(blk)[2][0][0]
    assert used == len(data) and np.count_nonzero(sizes > 1024) >= len(set(parts))
    check(eng, oracle, data, 9, label="many big groups")
    # big groups in several blocks of one batch
    cap = 300_000 if full else 60_000
    block_cap(cap)
    pieces = []
    for j in range(4):
        k = 1025 + 500 * j
        d, S, _ = groups_input(rng, k, 12, 0, max(cap - 20 * k, 0))
        pad = rng.integers(2, 256, max(cap - len(d), 0), dtype=np.uint8)
        pad[1:][pad[1:] == pad[:-1]] ^= 0x80
        pieces.append((d + pad.tobytes())[:cap])
    data = b"".join(pieces)
    starts = oracle.cut_points(data, 9)[0]
    assert len(starts) - 1 >= 4
    big_blocks = sum(1 for s, e in zip(starts[:-1], starts[1:]) if (doubling_groups(_rle1(oracle, data[s:e], cap)[0])[2][0][0] > 1024).any())
    assert big_blocks >= 3
    check(eng, oracle, data, 9, cap, label="big groups in several blocks")


# ---------------------------------------------------------------------------------------------------------------------
# round-0 code shapes

def _no_runs(x, alpha_vals):
    """break every run of 4 equal bytes (RLE1 stays the identity) by the next byte of the alphabet"""
    x = x.copy()
    while True:
        r = np.flatnonzero((x[3:] == x[2:-1]) & (x[2:-1] == x[1:-2]) & (x[1:-2] == x[:-3])) + 3
        if not r.size:
            return x
        pos = {v: i for i, v in enumerate(alpha_vals)}
        for i in r[::4]:
            x[i] = alpha_vals[(pos[int(x[i])] + 1) % len(alpha_vals)]


def shape_input(rng, alpha, dist, n):
    vals = np.sort(rng.permutation(256)[:alpha]).astype(np.uint8)
    if alpha == 1:
        return vals[:1].repeat(min(n, 3)).tobytes()
    w = {"uniform": np.ones(alpha), "geometric": 0.7 ** np.arange(alpha), "zipf": 1.0 / np.arange(1, alpha + 1) ** 1.5,
         "dominant": np.r_[1.0, np.full(alpha - 1, 0.02 / (alpha - 1))]}[dist]
    x = vals[rng.permutation(alpha)][rng.choice(alpha, n, p=w / w.sum())]
    x[:alpha] = vals[rng.permutation(alpha)]   # every byte occurs
    return _no_runs(x, vals).tobytes()


def test_round0_code_shapes(leg, oracle):
    """alphabets 1..256 (9 for a uniform 4-bit code) under uniform, geometric, Zipf and one-dominant frequencies: the longest code of the round-0 key
    (a copy of k_sym_tab's bisection) takes every value from 1 to 10, and L = 44 / maxlen with it"""
    eng, full = leg
    rng = np.random.default_rng(3)
    seen = set()
    for alpha in (1, 2, 3, 4, 5, 9, 17, 128, 255, 256):
        for dist in ("uniform", "geometric", "zipf", "dominant"):
            for level, n in (((9, B9), (1, B1)) if full else ((9, 6000),)):
                data = shape_input(rng, alpha, dist, n)
                blk, used = _rle1(oracle, data, level * 100_000 - 19)
                assert used == len(data) and len(np.unique(blk)) == alpha
                lens, _, maxlen, L = sym_code(blk)
                assert L == KEY_BITS // maxlen and lens.max() == maxlen or alpha == 1
                seen.add(maxlen)
                check(eng, oracle, data, level, label=f"alpha={alpha} {dist} maxlen={maxlen}")
    assert seen == set(range(1, 11)), sorted(seen)


def test_round0_key_edge_decides_order(leg, oracle):
    """8 equally frequent bytes: 3-bit codes, L = 14, and a key holds 14 symbols + the top 2 bits of the 15th.  Pairs of
    copies of a 14-symbol string followed by 'a' / 'b' (codes 000 / 001: equal keys) and then by 'h' / 'a': the 15th
    symbol decides the order, and a first doubling distance of 15 would order them by the 16th."""
    eng, full = leg
    rng = np.random.default_rng(44)
    abc = np.frombuffer(b"abcdefgh", np.uint8)
    parts = []
    for _ in range(3000 if full else 150):
        S = abc[rng.integers(0, 8, 14)].tobytes()
        parts += [S + b"ah", S + b"ba"]
        parts.append(abc[rng.integers(0, 8, int(rng.integers(20, 60 if not full else 250)))].tobytes())
    data = _no_runs(np.frombuffer(b"".join(parts), np.uint8), abc).tobytes()
    blk, used = _rle1(oracle, data, B9)
    assert used == len(data)
    lens, vals, maxlen, L = sym_code(blk)
    assert (lens[abc] == 3).all() and L == 14
    keys = round0_keys(blk, lens, vals)
    b = bytes(blk)
    i = b.find(parts[0])
    j = b.find(parts[1], i + 1)
    assert b[i:i + 14] == b[j:j + 14] and keys[i] == keys[j] and b[i + 14] != b[j + 14] and b[i + 15] > b[j + 15]
    check(eng, oracle, data, 9, label="key edge")


# ---------------------------------------------------------------------------------------------------------------------
# periodic and near-periodic blocks

def test_periodic_blocks(leg, oracle):
    """periods 1, 2, 3, 43, 44, 45, 4096, 4097 and n/2, as they are and with one byte changed near the end or at the
    first byte (the rotation that wraps): identical rotations sort by descending index once h >= n"""
    eng, full = leg
    rng = np.random.default_rng(9)
    sizes = ((9, B9), (1, B1)) if full else ((9, 9000),)
    for level, n in sizes:
        for p in (1, 2, 3, 43, 44, 45, 4096, 4097, n // 2):
            if p > n // 2:
                continue
            pat = rng.integers(0, 256, p, dtype=np.uint8)
            pat[1:][pat[1:] == pat[:-1]] ^= 0x55
            if p > 1 and pat[0] == pat[-1]:
                pat[0] ^= 0x0F
            base = np.resize(pat, n)
            for where in ("none", "end", "wrap"):
                x = base.copy()
                if where != "none":
                    i = n - 3 if where == "end" else 0
                    x[i] ^= 0xA5
                blk, used = _rle1(oracle, x, level * 100_000 - 19)
                if p > 1:
                    assert used == n and np.count_nonzero(blk != np.resize(pat, blk.size)) == (where != "none")
                else:
                    assert len(np.unique(blk[:-8])) <= 3    # one byte: RLE1 turns it into 'cccc' + count 251, repeated
                st = check(eng, oracle, x.tobytes(), level, label=f"period {p} change={where}")
                if where == "none" and p > 1 and n % p == 0:
                    rounds = doubling_groups(blk)[2]
                    assert eng.stats().sort_rounds == len(rounds) + 1 and len(rounds) >= 1


def test_tiny_blocks(leg, oracle, block_cap):
    """blocks of n = 1 .. 50 bytes (the whole input below 8 bytes, the block-cap hook above): keys that wrap around
    the block (k_keys_init stages bytes cyclically) and, for periodic blocks of n <= L, the tie rule applied in k_keys2"""
    eng, _ = leg
    rng = np.random.default_rng(50)
    for n in range(1, 51):
        block_cap(max(n, 8))
        for pat in (b"ab", b"abc", b"aab", b"zyx", rng.integers(0, 256, 7, dtype=np.uint8).tobytes()):
            data = (pat * (3 * n // len(pat) + 2))[:n if n < 8 else 3 * n]
            starts, lens, _ = oracle.cut_points(data, 9)
            assert set(lens[:-1]) <= {n} and lens[0] == n
            check(eng, oracle, data, 9, max(n, 8), label=f"n={n} pattern={pat!r}")
            if n <= KEY_BITS and pat == b"ab" and n % 2 == 0:
                assert sym_code(np.frombuffer(data[:n], np.uint8))[3] >= n   # h = L >= n already in round 1


# ---------------------------------------------------------------------------------------------------------------------
# blocks with a designed L column (inverse BWT)

def text_for_bwt(L, rng, keep=()):
    """a block whose BWT is L, up to a few swaps of adjacent distinct bytes that join the cycles of the LF mapping into
    one (a swap at i composes LF with the transposition (i i+1)).  Swaps avoid `keep`, runs and new equal neighbours.
    Returns (block, L actually used, origPtr)."""
    L = np.array(L, dtype=np.uint8)
    n = L.size
    LF = np.empty(n, np.int64)
    LF[np.argsort(L, kind="stable")] = np.arange(n)
    lab = np.full(n, -1, np.int64)
    nc = 0
    for s in range(n):
        if lab[s] < 0:
            i = s
            while lab[i] < 0:
                lab[i] = nc
                i = LF[i]
            nc += 1
    parent = list(range(nc))

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a
    banned = np.zeros(n + 2, bool)
    for k in keep:
        banned[max(k - 2, 0):k + 3] = True
    left = nc - 1
    for _ in range(4):   # a few passes: a merge elsewhere can make a pair eligible
        for i in rng.permutation(n - 1):
            if not left:
                break
            i = int(i)
            prev, nxt = int(L[i - 1]) if i else -1, int(L[i + 2]) if i + 2 < n else -2
            if banned[i] or banned[i + 1] or L[i] == L[i + 1] or prev in (L[i], L[i + 1]) or nxt in (L[i], L[i + 1]):
                continue
            a, b = find(lab[i]), find(lab[i + 1])
            if a == b:
                continue
            parent[a] = b
            L[i], L[i + 1] = L[i + 1], L[i]
            banned[max(i - 1, 0):i + 3] = True
            left -= 1
        banned[:] = False
        for k in keep:
            banned[max(k - 2, 0):k + 3] = True
    if left:   # e.g. a fixed point between two equal bytes: no swap joins it without making equal neighbours
        return None
    LF[np.argsort(L, kind="stable")] = np.arange(n)
    T = np.empty(n, np.uint8)
    i = 0
    for j in range(n - 1, -1, -1):
        T[j] = L[i]
        i = LF[i]
    return T, L, 0


def designed_block(oracle, rng, L, keep=()):
    """(block bytes, oracle stages, L column) for a designed L column (an array, or a function of rng that draws one);
    asserts that the oracle's BWT of the block is that L and that RLE1 leaves the block alone"""
    for _ in range(8):
        res = text_for_bwt(L(rng) if callable(L) else L, rng, keep)
        if res is None:
            continue
        T, Lu, optr = res
        blk, used = _rle1(oracle, T, B9)
        if used == T.size and blk.size == T.size:
            break
    else:
        raise AssertionError("no inverse without a run of 4 equal bytes and with one LF cycle")
    st = oracle.block_stages(blk)
    assert st["U"].tobytes() == Lu.tobytes() and st["orig_ptr"] == optr
    return T.tobytes(), st, Lu


def no_neighbours(rng, n, alpha, lo=0):
    """n bytes over [lo, lo + alpha) with no two equal neighbours (MTF gives no zero: m = n + 1)"""
    x = rng.integers(0, alpha - 1, n)
    step = rng.integers(1, alpha, n)
    out = (np.cumsum(step) + x[0]) % alpha   # consecutive values differ by a non-zero step
    return (out + lo).astype(np.uint8)


def test_mtf_rle2_segments(leg, oracle):
    """MTF over 8 KiB segments / 256-byte sub-segments and RLE2 over 8 KiB tiles: rank 255 at every segment and
    sub-segment start, a byte absent for several segments and then used again, block lengths 8192 k and 8192 k +- 1,
    zero runs at block position 0, at the block end, across tiles and of lengths 2^k - 1, 2^k, 2^k + 1"""
    eng, full = leg
    rng = np.random.default_rng(255)
    n = 8192 * (100 if full else 6)
    # rank 255: the 256 byte values in a fixed cyclic order -> every symbol from position 256 on has rank 255
    L = np.resize(rng.permutation(256).astype(np.uint8), n)
    keep = range(0, n, 256)
    data, st, Lu = designed_block(oracle, rng, L, keep)
    assert (st["A"][256:n:256] == 256).all() and st["m"] == n + 1
    check(eng, oracle, data, 9, label="rank 255 at segment starts")
    # a byte absent from segments 1..4 (and every other byte used), then used again
    def absent(r):
        L = no_neighbours(r, n, 200, lo=20)
        L[r.integers(0, 8192, 50)] = 7
        L[5 * 8192 + r.integers(0, 8192, 50)] = 7
        L[1:][L[1:] == L[:-1]] = 8
        return L
    data, st, Lu = designed_block(oracle, rng, absent)
    pos7 = np.flatnonzero(Lu == 7)
    assert pos7.size and not ((pos7 >= 8192) & (pos7 < 5 * 8192)).any() and (pos7 >= 5 * 8192).any()
    check(eng, oracle, data, 9, label="byte absent for 4 segments")
    # block lengths around multiples of 8192
    for ln in ((8192 * 109 - 1, 8192 * 109, 8192 * 109 + 1, 8192 - 1, 8192, 8193) if full else (8191, 8192, 8193, 16383, 16384, 16385)):
        data, st, _ = designed_block(oracle, rng, lambda r: no_neighbours(r, ln, 200, lo=40))
        assert st["n"] == ln
        check(eng, oracle, data, 9, label=f"n={ln}")
    # zero runs: r repeats of a short pattern make runs of r - 1 .. r + 1 equal bytes in L (zero runs of the MTF)
    parts = []
    for r in [2 ** k + d for k in range(1, 14 if full else 12) for d in (-1, 0, 1)] + [9000]:
        pat = rng.integers(0, 256, int(rng.integers(5, 12)), dtype=np.uint8)
        pat[1:][pat[1:] == pat[:-1]] ^= 0x33
        parts += [np.tile(pat, r), rng.integers(0, 256, 30, dtype=np.uint8)]
    data = np.concatenate(parts).tobytes()
    blk, used = _rle1(oracle, data, B9)
    U = oracle.block_stages(blk)["U"]
    runs = np.diff(np.r_[0, np.flatnonzero(np.diff(U.astype(np.int64))) + 1, U.size])
    assert used == len(data) and runs.max() > 8192   # a run longer than an RLE2 tile crosses one
    assert {2 ** k + d for k in range(1, 12) for d in (-1, 0, 1)} <= set(runs.tolist())
    check(eng, oracle, data, 9, label="zero runs")
    # one zero run that covers the whole block
    for d in (b"q", b"qq", b"qqq"):
        st = oracle.block_stages(np.frombuffer(d, np.uint8))
        assert st["alpha"] == 1 and list(st["A"][:-1]) == {1: [0], 2: [1], 3: [0, 0]}[len(d)]
        check(eng, oracle, d, 9, label=f"whole-block run {d!r}")


# ---------------------------------------------------------------------------------------------------------------------
# Huffman optimiser

def tie_share(st):
    """share of groups whose best cost is reached by two tables or more (k_huf_assign's strict '<' picks the first)"""
    A, lens = st["A"], st["lens"].astype(np.int64)
    m = A.size
    g = np.arange(m) // 50
    cost = np.stack([np.bincount(g, weights=lens[t][A]) for t in range(lens.shape[0])])
    return float(np.mean((cost == cost.min(0)).sum(0) >= 2))


def test_huffman_table_counts(leg, oracle):
    """m = 199/200, 599/600, 1199/1200, 2399/2400 (the table-count thresholds) and m mod 50 = 0, 1, 49: a designed L
    with no equal neighbours gives m = n + 1 exactly"""
    eng, _ = leg
    rng = np.random.default_rng(1200)
    target = {199: 2, 200: 3, 599: 3, 600: 4, 1199: 4, 1200: 5, 2399: 5, 2400: 6, 2401: 6, 2449: 6, 5000: 6, 5001: 6, 5049: 6}
    for m, ng in target.items():
        data, st, _ = designed_block(oracle, rng, lambda r: no_neighbours(r, m - 1, 30, lo=65))
        assert st["m"] == m and st["n_groups"] == ng and st["n_sel"] == (m + 49) // 50
        check(eng, oracle, data, 9, label=f"m={m}")


def _sections(rng, alpha, nsec, sec, lo=97):
    """sections of different symbol distributions over a small alphabet, runs of at most 3"""
    vals = np.arange(lo, lo + alpha, dtype=np.uint8)
    out = [vals]
    for _ in range(nsec):
        w = rng.dirichlet(np.full(alpha, 0.4))
        out.append(vals[rng.choice(alpha, sec, p=w)])
    return _no_runs(np.concatenate(out), vals).tobytes()


def test_huffman_ties_unused_tables_and_length_20(leg, oracle):
    """cost ties on >= 30 % of the groups (k_huf_assign's strict '<', k_huf_split's stable median split), a table no
    group selects, code length 20 reached in a real block, and defect D1 (alphabet + 2 < tables) at several m"""
    eng, full = leg
    rng = np.random.default_rng(20)
    # ties: three bytes, short sections
    found = 0
    for seed in range(40):
        data = _sections(np.random.default_rng(seed), 3, 30, 300, lo=120)
        blk, _ = _rle1(oracle, data, B9)
        st = oracle.block_stages(blk)
        if st["n_groups"] >= 3 and not st["d1"] and tie_share(st) >= 0.3:
            check(eng, oracle, data, 9, label=f"ties {tie_share(st):.2f}")
            found += 1
            if found == 3:
                break
    assert found == 3
    # a table that no group selects (alphabet large enough that D1 is not involved)
    found = 0
    for seed in range(60):
        data = _sections(np.random.default_rng(1000 + seed), 6, 40, 500)
        blk, _ = _rle1(oracle, data, B9)
        st = oracle.block_stages(blk)
        if not st["d1"] and len(np.unique(st["sel"])) < st["n_groups"]:
            check(eng, oracle, data, 9, label="unused table")
            found += 1
            break
    assert found
    # code length 20: bytes drawn with weights 1.55^-i, so the MTF symbol frequencies fall about like a Fibonacci sequence
    n = 400_000 if full else 120_000
    vals = np.arange(64, 112, dtype=np.uint8)
    w = 1.55 ** -np.arange(48.0)
    data = _no_runs(vals[np.random.default_rng(2).choice(48, n, p=w / w.sum())], vals).tobytes()
    st = oracle.block_stages(_rle1(oracle, data, B9)[0])
    assert st["lens"].max() == 20
    check(eng, oracle, data, 9, label="code length 20")
    # D1: fewer symbols than tables, at 5 and 6 tables
    for alpha, sec in ((2, 120), (3, 300)):
        for seed in range(40):
            data = _sections(np.random.default_rng(2000 + seed), alpha, 40, sec)
            st = oracle.block_stages(_rle1(oracle, data, B9)[0])
            if st["d1"] and st["alpha"] + 2 < st["n_groups"]:
                break
        else:
            raise AssertionError(f"no D1 case at alphabet {alpha}")
        assert check(eng, oracle, data, 9, label=f"D1 alphabet {alpha} m={st['m']}").d1_triggered


def test_18000_selectors(leg, oracle):
    """a full level-9 block whose L column has no equal neighbours: m = n + 1 = 899 982, 18 000 selectors (the most a
    level-9 block can have)"""
    eng, _ = leg
    rng = np.random.default_rng(18000)
    data, st, _ = designed_block(oracle, rng, lambda r: no_neighbours(r, B9, 256))
    assert st["n"] == B9 and st["m"] == B9 + 1 and st["n_sel"] == 18_000
    check(eng, oracle, data, 9, label="18000 selectors")


# ---------------------------------------------------------------------------------------------------------------------
# every structure in one batch

def mixed_input(oracle):
    """>= 45 level-9 blocks, each one generator's full-size output (padded with run-free filler to exactly one block)"""
    rng = np.random.default_rng(4545)
    pieces = []
    for k, surv in ((2, 0), (33, 1), (257, 2), (1025, 3), (2049, 0), (5000, 1), (1024, 2), (2048, 3), (256, 0), (32, 3)):
        pieces.append(group_case(rng, k, surv, 0, max(0, (B9 - 60_000) // k - 40))[0])
    for alpha in (2, 3, 4, 5, 9, 17, 128, 255, 256):
        for dist in ("uniform", "geometric", "zipf", "dominant"):
            pieces.append(shape_input(rng, alpha, dist, B9))
    for p in (2, 3, 45, 4097):
        pat = rng.integers(0, 256, p, dtype=np.uint8)
        pat[1:][pat[1:] == pat[:-1]] ^= 0x55
        pieces.append(np.resize(pat, B9).tobytes())
    pieces.append(designed_block(oracle, rng, lambda r: no_neighbours(r, B9, 256))[0])
    out, offs = [], []
    for d in pieces:
        if len(d) < B9:
            pad = rng.integers(2, 256, B9 - len(d), dtype=np.uint8)
            pad[1:][pad[1:] == pad[:-1]] ^= 0x80
            d += pad.tobytes()
        if out and out[-1][-1] == d[0]:   # a run across the seam would move the cut
            d = d[::-1]
        offs.append(sum(len(x) for x in out))
        out.append(d)
    data = b"".join(out)
    starts = oracle.cut_points(data, 9)[0]
    assert starts[:-1] == offs and len(offs) >= 45 and len(data) >= 40_000_000
    return data


@pytest.mark.gpu
def test_mixed_structures_one_batch(gpu_engine, oracle):
    """one 40 MB input whose blocks come from every family: through the two-lane pool (compressFile at this size), the
    single launch (with the per-block stage comparison) and forced batches of 7 blocks"""
    data = mixed_input(oracle)
    exp = oracle.compress(data, 9, threads=CPUS)
    assert gpu_engine.compressFile(data, None, 9) == exp, "two-lane pool path"
    gpu_engine.debug_set_pool(1 << 62)
    try:
        got = gpu_engine.compressFile(data, None, 9)
        assert stage_diff(gpu_engine, oracle, data, 9) is None
        assert got == exp, "single launch"
        gpu_engine.debug_set_batch_blocks(7)
        assert gpu_engine.compressFile(data, None, 9) == exp, "batches of 7 blocks"
    finally:
        gpu_engine.debug_set_batch_blocks(0)
        gpu_engine.debug_set_pool()
