// search.cuh -- fixed-string search over decoded bytes in HBM (bz2b200_search; included after decode.cuh).
//
// The decoded output is cut into TILES of `tile` bytes (a multiple of SEARCH_THREADS, at most SEARCH_TILE_MAX); thread i
// of a CTA owns the CH = tile / SEARCH_THREADS consecutive positions i*CH .. i*CH + CH - 1 of its tile, so that one
// 32-bit mask per thread describes its newlines and the positions where a match starts.  A match belongs to the tile
// where it starts; a tile reads up to 255 bytes past its end (the longest pattern), clamped at the output's end.
// The kernels work on a SLICE of the output (SearchSlice): `own` bytes at global offset `base`, followed in the buffer by
// what follows them, `avail` bytes in all.  Matches start and newlines count in the own bytes only; the verify may read
// all of them.  Every position the kernels write is global.  One context searches one slice: base 0, own = avail = n.
//   k_search_count  per tile: matches, newlines, first / last newline, the lines of its first and last match and the
//                   distinct lines its matches start in; per thread: (mask of match positions, match count)
//   k_search_scan   one CTA over the tiles: exclusive sums of matches and newlines, exclusive max of the last newline
//                   (line_begin), suffix min of the first newline (line_end), exclusive max of the last match line and
//                   from it the exclusive sum of lines that hold a first match (the rank of a line among those); the
//                   carries start at a seed (what the slices before and after hold), and the unseeded scan of a slice can
//                   write the slice's own summary, composed by the host over the slices as this kernel composes tiles
//   k_search_emit   per tile holding a match of rank < n_ret: the matches in (offset, pattern) order with their line
//                   fields, and for every returned FIRST_IN_LINE match the piece [line_begin, line_end] of its line
// The patterns come with a filter: a 65 536-bit table of the first two bytes of the patterns of two bytes or more and a
// 256-bit table of the one-byte patterns, both held in shared memory by the count pass; only positions that pass are
// verified against the candidate lists (CSR by the first two bytes / by the byte, ascending pattern index).
#define SEARCH_THREADS 256
#define SEARCH_TILE_MAX 8192u        // CH <= 32: one mask word per thread
#define SEARCH_TILE_DEFAULT 8192u
#define SEARCH_HALO 256u             // >= the longest pattern - 1, and a multiple of 16
#define SEARCH_MAX_PATTERNS 256u
#define SEARCH_MAX_LEN 256u

struct SearchPats {
  const u32 *bg_bits;   // bit (b0 << 8 | b1): some pattern of >= 2 bytes starts with the (folded) bytes b0 b1
  const u32 *one_bits;  // bit b: some one-byte pattern is b
  const u32 *bg_off;    // [65537] CSR offsets into bg_list by (b0 << 8 | b1)
  const u32 *bg_list;   // pattern indices, ascending within a key
  const u32 *one_off;   // [257] CSR offsets into one_list by byte
  const u32 *one_list;
  const u32 *pat_off, *pat_len;
  const u8 *pat;        // the patterns, folded when fold != 0
  u32 fold;             // ASCII A-Z compare equal to a-z
};
struct SearchTile {     // k_search_count -> k_search_scan
  u64 first_nl;         // first '\n' of the tile (global position), n if none
  i64 last_nl;          // last '\n' of the tile, -1 if none
  u32 matches, nl, lines, pad;  // lines: distinct lines (within the tile) in which a match of the tile starts
  i64 first_ml, last_ml;        // tile-local line (newlines of the tile before it) of the first / last match, -1 if none
};
struct SearchBase {     // k_search_scan -> k_search_emit
  u64 match0, nl0, line0;  // matches, newlines, lines holding a first match in the tiles before
  i64 prev_nl;             // last '\n' before the tile, -1 if none
  u64 next_nl;             // first '\n' after the tile, n if none
  i64 prev_ml;             // line of the last match before the tile, -1 if none
};
struct SearchTotals { u64 matches, lines, pieces, pad; };
struct SearchSlice {    // the bytes a launch searches: own bytes at global offset base, avail >= own readable, n = global output length
  u64 base, own, avail, n;
};
struct SearchSum {      // a slice as a SearchTile: global first / last newline, 64-bit counts, slice-local lines of its first / last match
  u64 first_nl;
  i64 last_nl;
  u64 matches, nl, lines;
  i64 first_ml, last_ml;
};
struct SearchMatch {    // bz2b200_match, field for field
  u64 offset, line, line_begin, line_end;
  u32 pattern, flags;
};

// ASCII A-Z -> a-z in each byte of a word; every other byte (also >= 0x80) unchanged
__host__ __device__ __forceinline__ u32 search_fold4(u32 x) {
  const u32 lo = x & 0x7f7f7f7fu;
  const u32 upper = (lo + 0x3f3f3f3fu) & ~(lo + 0x25252525u) & ~x & 0x80808080u;  // 0x41 <= b <= 0x5a
  return x | (upper >> 2);
}

// bytes [t0, min(t0 + tile + SEARCH_HALO, n)) of src into s (folded), as 16-byte words: the source must be readable 15
// bytes past n (a decode sink keeps 64 bytes of slack); what lies past n is never compared
__device__ __forceinline__ void search_stage(const u8 *__restrict__ src, u64 n, u64 t0, u32 tile, u32 fold, u8 *s) {
  const u64 want = n - t0 < (u64)tile + SEARCH_HALO ? n - t0 : (u64)tile + SEARCH_HALO;
  const u32 nw = (u32)((want + 15) >> 4);
  const uint4 *w = reinterpret_cast<const uint4 *>(src + t0);
  uint4 *d = reinterpret_cast<uint4 *>(s);
  for (u32 v = threadIdx.x; v < nw; v += SEARCH_THREADS) {
    uint4 x = w[v];
    if (fold) { x.x = search_fold4(x.x); x.y = search_fold4(x.y); x.z = search_fold4(x.z); x.w = search_fold4(x.w); }
    d[v] = x;
  }
  __syncthreads();
}

__device__ __forceinline__ bool search_equal(const u8 *a, const u8 *b, u32 len) {
  for (u32 k = 0; k < len; k++)
    if (a[k] != b[k]) return false;
  return true;
}
// pattern j (>= 2 bytes, its first two bytes already equal) at s[0..), with `room` bytes left before the output's end
__device__ __forceinline__ bool search_verify(const SearchPats &P, u32 j, const u8 *s, u64 room) {
  const u32 len = P.pat_len[j];
  return len <= room && search_equal(s + 2, P.pat + P.pat_off[j] + 2, len - 2);
}
__device__ __forceinline__ u32 search_line_of(u32 nlmask, u32 k) { return __popc(nlmask & ((1u << k) - 1u)); }

// persistent: every CTA loads the filter once and takes tiles blockIdx.x, + gridDim.x, ... (4 CTAs per SM fit 64 registers)
__global__ void __launch_bounds__(SEARCH_THREADS, 4) k_search_count(const u8 *__restrict__ src, SearchSlice S, u32 tile, u32 n_tiles, SearchPats P,
                                                                    SearchTile *__restrict__ tiles, uint2 *__restrict__ tsum) {
  __shared__ __align__(16) u8 s[SEARCH_TILE_MAX + SEARCH_HALO];
  __shared__ u32 bg[2048], one[8];
  __shared__ i64 ws[33];
  __shared__ u64 wsu[33];
  for (u32 i = threadIdx.x; i < 2048; i += SEARCH_THREADS) bg[i] = P.bg_bits[i];
  if (threadIdx.x < 8) one[threadIdx.x] = P.one_bits[threadIdx.x];
  const u32 CH = tile / SEARCH_THREADS;
  for (u32 t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const u64 t0 = (u64)t * tile;
    __syncthreads();  // the previous tile's text is no longer read (and the tables are in place)
    search_stage(src, S.avail, t0, tile, P.fold, s);
    const u32 k0 = threadIdx.x * CH;
    u32 nlmask = 0, mmask = 0, cnt = 0;
    for (u32 k = 0; k < CH; k++) {
      const u64 p = t0 + k0 + k;  // in the slice
      if (p >= S.own) break;
      const u32 c = s[k0 + k];
      if (c == '\n') nlmask |= 1u << k;
      u32 m = 0;
      if ((one[c >> 5] >> (c & 31)) & 1u) m += P.one_off[c + 1] - P.one_off[c];
      if (p + 1 < S.avail) {
        const u32 key = (c << 8) | s[k0 + k + 1];
        if ((bg[key >> 5] >> (key & 31)) & 1u)
          for (u32 q = P.bg_off[key], qe = P.bg_off[key + 1]; q < qe; q++) m += search_verify(P, P.bg_list[q], s + k0 + k, S.avail - p);
      }
      if (m) { mmask |= 1u << k; cnt += m; }
    }
    tsum[(u64)t * SEARCH_THREADS + threadIdx.x] = make_uint2(mmask, cnt);
    // tile-local lines: newlines of the tile before the thread's chunk, then within it
    u64 nl_tot;
    const u64 nl_before = block_excl_sum<u64>((u64)__popc(nlmask), nl_tot, wsu);
    const i64 first_ml = mmask ? (i64)(nl_before + search_line_of(nlmask, __ffs((int)mmask) - 1)) : -1;
    const i64 last_ml = mmask ? (i64)(nl_before + search_line_of(nlmask, 31 - __clz((int)mmask))) : -1;
    i64 ml_tot;
    const i64 prev_ml = block_excl_max<i64>(last_ml, (i64)-1, ml_tot, ws);
    u32 lines = 0;
    for (u32 mm = mmask, prev = (u32)-1; mm; mm &= mm - 1) {  // distinct lines of the chunk's matches
      const u32 ln = search_line_of(nlmask, __ffs((int)mm) - 1);
      lines += ln != prev;
      prev = ln;
    }
    if (first_ml >= 0 && first_ml == prev_ml) lines--;  // that line was counted by an earlier chunk of the tile
    const u64 m_tile = block_sum<u64>(cnt, wsu), l_tile = block_sum<u64>(lines, wsu);
    const i64 first_nl = nlmask ? (i64)(S.base + t0 + k0 + __ffs((int)nlmask) - 1) : (i64)S.n;
    const i64 last_nl = nlmask ? (i64)(S.base + t0 + k0 + 31 - __clz((int)nlmask)) : -1;
    const i64 fnl = block_min<i64>(first_nl, ws), lnl = block_max<i64>(last_nl, ws);
    const i64 fml = block_min<i64>(first_ml >= 0 ? first_ml : INT64_MAX, ws);
    if (threadIdx.x == 0) {
      SearchTile r;
      r.first_nl = (u64)fnl; r.last_nl = lnl; r.matches = (u32)m_tile; r.nl = (u32)nl_tot; r.lines = (u32)l_tile; r.pad = 0;
      r.first_ml = fml == INT64_MAX ? -1 : fml; r.last_ml = ml_tot;
      tiles[t] = r;
    }
  }
}

// one CTA of 1024 threads over the tiles, in rounds of 1024 with carries: forward for the prefix quantities, backward for
// the suffix min of the first newline.  The carries start at `seed` (nothing before: 0, 0, 0, -1, n, -1).  sum != nullptr
// (unseeded): the slice's summary; its lines are slice-local.  tot: the totals through the slice.
__global__ void __launch_bounds__(1024) k_search_scan(const SearchTile *__restrict__ tiles, u32 n_tiles, u64 n, SearchBase seed,
                                                      SearchBase *__restrict__ base, SearchTotals *__restrict__ tot, SearchSum *__restrict__ sum) {
  __shared__ u64 wsu[33];
  __shared__ i64 ws[33];
  u64 c_match = seed.match0, c_nl = seed.nl0, c_line = seed.line0;
  i64 c_prev_nl = seed.prev_nl, c_prev_ml = seed.prev_ml;
  for (u32 b = 0; b < n_tiles; b += blockDim.x) {
    const u32 t = b + threadIdx.x;
    const bool on = t < n_tiles;
    SearchTile r{};
    if (on) r = tiles[t];
    else { r.last_nl = -1; r.first_ml = -1; r.last_ml = -1; }
    u64 s_match, s_nl, s_line;
    i64 m_nl, m_ml;
    const u64 match0 = c_match + block_excl_sum<u64>(r.matches, s_match, wsu);
    const u64 nl0 = c_nl + block_excl_sum<u64>(r.nl, s_nl, wsu);
    i64 prev_nl = block_excl_max<i64>(r.last_nl, (i64)-1, m_nl, ws);
    prev_nl = prev_nl > c_prev_nl ? prev_nl : c_prev_nl;
    const i64 last_ml = r.last_ml >= 0 ? (i64)nl0 + r.last_ml : -1;
    i64 prev_ml = block_excl_max<i64>(last_ml, (i64)-1, m_ml, ws);
    prev_ml = prev_ml > c_prev_ml ? prev_ml : c_prev_ml;
    const u64 lines = r.lines - (r.first_ml >= 0 && (i64)nl0 + r.first_ml == prev_ml ? 1u : 0u);
    const u64 line0 = c_line + block_excl_sum<u64>(lines, s_line, wsu);
    if (sum && r.matches && match0 == seed.match0) sum->first_ml = (i64)nl0 + r.first_ml;  // the first tile with a match
    if (on) {
      SearchBase o;
      o.match0 = match0; o.nl0 = nl0; o.line0 = line0; o.prev_nl = prev_nl; o.next_nl = n; o.prev_ml = prev_ml;
      base[t] = o;
    }
    c_match += s_match; c_nl += s_nl; c_line += s_line;
    if (m_nl > c_prev_nl) c_prev_nl = m_nl;
    if (m_ml > c_prev_ml) c_prev_ml = m_ml;
  }
  __syncthreads();
  // suffix min as an exclusive max of the negated values with the tiles in descending order
  i64 c_next = -(i64)seed.next_nl;
  for (u32 b = 0; b < n_tiles; b += blockDim.x) {
    const bool on = b + threadIdx.x < n_tiles;
    const u32 t = on ? n_tiles - 1 - (b + threadIdx.x) : 0;
    const i64 v = on ? -(i64)tiles[t].first_nl : -(i64)n;
    i64 m;
    i64 e = block_excl_max<i64>(v, -(i64)n, m, ws);
    e = e > c_next ? e : c_next;
    if (on) base[t].next_nl = (u64)(-e);
    if (m > c_next) c_next = m;
  }
  if (threadIdx.x == 0) {
    tot->matches = c_match; tot->lines = c_line; tot->pieces = 0; tot->pad = 0;
    if (sum) {  // first_ml: written above when the slice has a match
      sum->first_nl = (u64)(-c_next); sum->last_nl = c_prev_nl; sum->matches = c_match; sum->nl = c_nl; sum->lines = c_line; sum->last_ml = c_prev_ml;
      if (!c_match) sum->first_ml = -1;
    }
  }
}

// Matches of rank < n_ret, match of rank r written at out[r - rank0]; with piece_src != nullptr also the line of every
// returned FIRST_IN_LINE match as piece (line rank lr at lr - lrank0), clipped to the own bytes: piece_src = its first
// byte in the slice, piece_len = through its '\n' (to n for a last line without one).
// tot->pieces = line rank of the match of rank n_ret - 1, plus one.
__global__ void __launch_bounds__(SEARCH_THREADS) k_search_emit(const u8 *__restrict__ src, SearchSlice S, u32 tile, u32 n_tiles, SearchPats P,
                                                                const SearchTile *__restrict__ tiles, const SearchBase *__restrict__ base,
                                                                const uint2 *__restrict__ tsum, u64 n_ret, u64 rank0, u64 lrank0,
                                                                SearchMatch *__restrict__ out, u64 *__restrict__ piece_src, u64 *__restrict__ piece_len,
                                                                SearchTotals *__restrict__ tot) {
  __shared__ __align__(16) u8 s[SEARCH_TILE_MAX + SEARCH_HALO];
  __shared__ i64 ws[33], nxt[SEARCH_THREADS];
  __shared__ u64 wsu[33];
  const u32 t = blockIdx.x;
  const SearchBase B = base[t];
  if (tiles[t].matches == 0 || B.match0 >= n_ret) return;
  const u32 CH = tile / SEARCH_THREADS;
  const u64 t0 = (u64)t * tile;
  search_stage(src, S.avail, t0, tile, P.fold, s);
  const u32 k0 = threadIdx.x * CH;
  u32 nlmask = 0;
  for (u32 k = 0; k < CH && t0 + k0 + k < S.own; k++)
    if (s[k0 + k] == '\n') nlmask |= 1u << k;
  const uint2 ts = tsum[(u64)t * SEARCH_THREADS + threadIdx.x];
  const u32 mmask = ts.x;
  const u64 pos0 = S.base + t0 + k0;
  // newlines around the chunk
  u64 nl_tot;
  const u64 line0 = B.nl0 + block_excl_sum<u64>((u64)__popc(nlmask), nl_tot, wsu);
  i64 m;
  i64 prev_nl = block_excl_max<i64>(nlmask ? (i64)(pos0 + 31 - __clz((int)nlmask)) : -1, (i64)-1, m, ws);
  if (B.prev_nl > prev_nl) prev_nl = B.prev_nl;
  {  // first newline after the chunk: suffix min over the later chunks, as an exclusive max in reversed thread order
    const i64 mine = nlmask ? (i64)(pos0 + __ffs((int)nlmask) - 1) : (i64)B.next_nl;
    nxt[threadIdx.x] = -mine;
    __syncthreads();
    const i64 e = block_excl_max<i64>(nxt[SEARCH_THREADS - 1 - threadIdx.x], -(i64)B.next_nl, m, ws);
    nxt[SEARCH_THREADS - 1 - threadIdx.x] = -e;
    __syncthreads();
  }
  const u64 next_nl = (u64)nxt[threadIdx.x];
  // ranks: of the chunk's first match, and of the first new line among its matches
  u64 m_tot;
  u64 rank = B.match0 + block_excl_sum<u64>(ts.y, m_tot, wsu);
  const i64 last_ml = mmask ? (i64)(line0 + search_line_of(nlmask, 31 - __clz((int)mmask))) : -1;
  i64 prev_ml = block_excl_max<i64>(last_ml, (i64)-1, m, ws);
  if (B.prev_ml > prev_ml) prev_ml = B.prev_ml;
  u32 new_lines = 0;
  for (u32 mm = mmask, prev = (u32)-1; mm; mm &= mm - 1) {
    const u32 l = search_line_of(nlmask, __ffs((int)mm) - 1);
    new_lines += l != prev && (i64)(line0 + l) != prev_ml;
    prev = l;
  }
  u64 l_tot;
  u64 lrank = B.line0 + block_excl_sum<u64>(new_lines, l_tot, wsu);
  // the walk
  for (u32 mm = mmask; mm && rank < n_ret; mm &= mm - 1) {
    const u32 k = __ffs((int)mm) - 1;
    const u64 p = pos0 + k;
    const u32 below = nlmask & ((1u << k) - 1u), above = nlmask >> k;
    SearchMatch r;
    r.offset = p;
    r.line = line0 + __popc(below);
    r.line_begin = (u64)((below ? (i64)(pos0 + 31 - __clz((int)below)) : prev_nl) + 1);
    r.line_end = above ? p + __ffs((int)above) - 1 : next_nl;
    const bool first = (i64)r.line != prev_ml;
    const u64 lr = first ? lrank : lrank - 1;  // rank of the match's line among the lines that hold a first match
    if (first && piece_src) {
      const u64 b = r.line_begin > S.base ? r.line_begin : S.base, e = r.line_end < S.n ? r.line_end + 1 : S.n;
      piece_src[lr - lrank0] = b - S.base;
      piece_len[lr - lrank0] = (e < S.base + S.own ? e : S.base + S.own) - b;
    }
    // the patterns at p in ascending index: merge the one-byte list and the list of the first two bytes
    const u8 *sp = s + k0 + k;
    const u32 c = sp[0];
    u32 q1 = P.one_off[c], e1 = P.one_off[c + 1], q2 = 0, e2 = 0;
    const u64 room = S.avail - (p - S.base);
    if (room > 1) { const u32 key = (c << 8) | sp[1]; q2 = P.bg_off[key]; e2 = P.bg_off[key + 1]; }
    u32 flags = first ? 1u : 0u;
    while (rank < n_ret) {
      u32 j;
      if (q1 < e1 && (q2 >= e2 || P.one_list[q1] < P.bg_list[q2])) j = P.one_list[q1++];
      else if (q2 < e2) {
        j = P.bg_list[q2++];
        if (!search_verify(P, j, sp, room)) continue;
      } else break;
      r.pattern = j;
      r.flags = flags;
      flags = 0;
      out[rank - rank0] = r;
      if (rank == n_ret - 1) tot->pieces = lr + 1;
      rank++;
    }
    if (first) { lrank++; prev_ml = (i64)r.line; }
  }
}

// In-place exclusive sum of a[0..n) (u64), a[n] = the total: SCAN64_ITEMS per CTA, partials scanned by one CTA
#define SCAN64_THREADS 1024
#define SCAN64_PER 4
#define SCAN64_ITEMS (SCAN64_THREADS * SCAN64_PER)
__global__ void __launch_bounds__(SCAN64_THREADS) k_scan64_reduce(const u64 *__restrict__ a, u64 n, u64 *__restrict__ part) {
  __shared__ u64 ws[33];
  const u64 i0 = (u64)blockIdx.x * SCAN64_ITEMS + (u64)threadIdx.x * SCAN64_PER;
  u64 v = 0;
  for (u32 k = 0; k < SCAN64_PER; k++) if (i0 + k < n) v += a[i0 + k];
  v = block_sum<u64>(v, ws);
  if (threadIdx.x == 0) part[blockIdx.x] = v;
}
__global__ void __launch_bounds__(SCAN64_THREADS) k_scan64_partials(u64 *__restrict__ part, u32 nb, u64 *__restrict__ a, u64 n) {
  __shared__ u64 ws[33];
  u64 carry = 0;
  for (u32 b = 0; b < nb; b += SCAN64_THREADS) {
    const u32 i = b + threadIdx.x;
    u64 tot;
    const u64 v = i < nb ? part[i] : 0;
    const u64 e = block_excl_sum<u64>(v, tot, ws);
    if (i < nb) part[i] = carry + e;
    carry += tot;
  }
  if (threadIdx.x == 0) a[n] = carry;
}
__global__ void __launch_bounds__(SCAN64_THREADS) k_scan64_apply(u64 *__restrict__ a, u64 n, const u64 *__restrict__ part) {
  __shared__ u64 ws[33];
  const u64 i0 = (u64)blockIdx.x * SCAN64_ITEMS + (u64)threadIdx.x * SCAN64_PER;
  u64 v[SCAN64_PER], sum = 0;
  for (u32 k = 0; k < SCAN64_PER; k++) { v[k] = i0 + k < n ? a[i0 + k] : 0; sum += v[k]; }
  u64 tot;
  u64 run = part[blockIdx.x] + block_excl_sum<u64>(sum, tot, ws);
  for (u32 k = 0; k < SCAN64_PER; k++)
    if (i0 + k < n) { a[i0 + k] = run; run += v[k]; }
}
