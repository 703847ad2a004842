// huff.cuh -- K-S4/K-S5: multi-table Huffman optimisation and bit emission for one block.
//
// Replaces StaticHuffman (BJ:1866-1951), HuffmanAllocator.allocateHuffmanCodeLengths
// (BJ:1135-1298), assignSelectors (BJ:1989-2004), optimizeHuffmanGroups (BJ:2005-2054) and
// the emission half of compressBlock (BJ:2059-2086, 2150-2194), iteration for iteration:
//   - tables start as {global histogram, flat}; while fewer than the target: assign selectors
//     (strict '<', lowest table wins ties), take the first most-used table, STABLE-sort its
//     groups by cost (done as a counting sort: costs <= 50*20), move the upper half
//     (positions >= len>>>1) to a new table, recount ALL histograms, rebuild ALL tables;
//   - code lengths: keys (freq<<9)|sym ascending through the in-place length-limited
//     allocator with limit 20; canonical codes by (length, symbol).
// The optimiser is a chain of small kernels so that the passes over the symbols run grid-wide:
//   k_huf_init    (per block)  first two tables {global histogram, flat}
//   k_huf_assign  (grid-wide)  cost of every group of 50 symbols under every table (all six lengths of a symbol
//                              packed in one u64, so one add per symbol), winner + its cost
//   k_huf_split   (per block)  most-used table, stable median split (counting sort over costs), new selector ids
//   k_huf_hist    (grid-wide)  histograms of all tables from the selectors
//   k_huf_build   (per block)  code lengths of all tables (the allocator is sequential: one thread per table)
//   k_huf_codes   (per block)  canonical codes, block header, selector + table bits, bit offset of every group
//   k_huf_emit    (grid-wide)  every thread packs one group of 50 symbols at its bit offset
// A block leaves the loop when it has its target number of tables (BJ:2150); the host launches the
// assign/split/hist/build round four times (2 -> 6 tables) and finished blocks skip.
#pragma once
#include "common.cuh"
#include "mtf.cuh"

#define HUF_LSTRIDE 260
#define HUF_GT 256                       // groups per CTA of the grid-wide kernels (one per thread)
#define HUF_GT_SYMS (HUF_GT * BZ_GROUP)  // symbols staged per CTA
#define HUF_BT 256                       // threads of the per-block kernels
#define HUF_CT 1024                      // threads of k_huf_codes

struct HufBlk {   // optimiser state of one block
  int ng, target, S, active;
  u32 m, nsel, pad0, pad1;
};
// per-block arrays in global memory (strides in elements)
struct HufArrays {
  u32 *freq;     // [nb][6][BZ_MAX_SYMS]
  u8 *lens;      // [nb][6][HUF_LSTRIDE]
  u64 *plen;     // [nb][BZ_MAX_SYMS]: the six lengths of a symbol, 10 bits each
  u32 *codes;    // [nb][6][BZ_MAX_SYMS]: length << 24 | canonical code
  u8 *sel;       // [nb][sel_stride]
  u16 *cost;     // [nb][sel_stride]: first the winning cost of the group, finally the selector MTF rank
  u32 *goff;     // [nb][sel_stride]: bit offset of the group inside the block's stream
  HufBlk *hb;    // [nb]
  i64 sel_stride;
};

// ---- in-place length-limited code-length allocation (BJ:1135-1298) -------------------------
__device__ __forceinline__ int ha_fls(u32 v) { return 32 - __clz((int)v); }
__device__ inline int ha_first(const int *a, int N, int i, int nodes_to_move) {
  int limit = i, k = N - 2;
  while (i >= nodes_to_move && (a[i] % N) > limit) {
    k = i;
    i -= (limit - i + 1);
  }
  if (i < nodes_to_move - 1) i = nodes_to_move - 1;
  while (k > i + 1) {
    int t = (i + k) >> 1;
    if ((a[t] % N) > limit) k = t; else i = t;
  }
  return k;
}
__device__ inline void ha_allocate(int *a, int N, int maxlen) {
  if (N == 2) a[1] = 1;
  if (N <= 2) { if (N >= 1) a[0] = 1; return; }
  a[0] += a[1];
  int head = 0, top = 2;
  for (int tail = 1; tail < N - 1; tail++) {
    int tmp;
    if (top >= N || a[head] < a[top]) { tmp = a[head]; a[head++] = tail; }
    else tmp = a[top++];
    if (top >= N || (head < tail && a[head] < a[top])) { tmp += a[head]; a[head++] = tail + N; }
    else tmp += a[top++];
    a[tail] = tmp;
  }
  int node = N - 2;
  for (int depth = 1; depth < maxlen - 1 && node > 1; depth++) node = ha_first(a, N, node - 1, 0);
  const int reloc = node;
  if ((a[0] % N) >= reloc) {
    int first_node = N - 2, next = N - 1;
    for (int depth = 1, avail = 2; avail > 0; depth++) {
      int last = first_node;
      first_node = ha_first(a, N, last - 1, 0);
      for (int i = avail - (last - first_node); i > 0; i--) a[next--] = depth;
      avail = (last - first_node) << 1;
    }
  } else {
    int insert_depth = maxlen - ha_fls((u32)(reloc - 1));
    int first_node = N - 2, next = N - 1;
    int depth = insert_depth == 1 ? 2 : 1;
    int left = insert_depth == 1 ? reloc - 2 : reloc;
    for (int avail = depth << 1; avail > 0; depth++) {
      int last = first_node;
      first_node = first_node <= reloc ? first_node : ha_first(a, N, last - 1, reloc);
      int off = 0;
      if (depth >= insert_depth) {
        off = 1 << (depth - insert_depth);
        if (left < off) off = left;
      } else if (depth == insert_depth - 1) {
        off = 1;
        if (a[first_node] == last) first_node++;
      }
      for (int i = avail - (last - first_node + off); i > 0; i--) a[next--] = depth;
      left -= off;
      avail = (last - first_node + off) << 1;
    }
  }
}

// tests/ only (bz2b200_debug_huffman_lengths): the allocator on the device over one array of ascending frequencies
__global__ void k_debug_ha_allocate(int *a, int N, int maxlen) {
  if (threadIdx.x == 0 && blockIdx.x == 0) ha_allocate(a, N, maxlen);
}

// rebuild tables [0, ng) from freq (StaticHuffman ctor, BJ:1866-1894); blockDim.x == HUF_BT
struct HufBuildSmem {
  u32 freq[BZ_MAX_GROUPS][BZ_MAX_SYMS];
  u32 keys[BZ_MAX_GROUPS][BZ_MAX_SYMS];
  int work[BZ_MAX_GROUPS][BZ_MAX_SYMS];
  u8 lens[BZ_MAX_GROUPS][HUF_LSTRIDE];
};
__device__ inline void huf_build(HufBuildSmem &sm, int ng, int S, u8 *__restrict__ lens_g, u64 *__restrict__ plen_g) {
  for (int x = threadIdx.x; x < ng * S; x += HUF_BT) {
    int t = x / S, i = x - t * S;
    u32 key = (sm.freq[t][i] << 9) | (u32)i;
    int rank = 0;
    for (int j = 0; j < S; j++) rank += ((sm.freq[t][j] << 9) | (u32)j) < key ? 1 : 0;
    sm.keys[t][rank] = key;
  }
  __syncthreads();
  for (int x = threadIdx.x; x < ng * S; x += HUF_BT) {
    int t = x / S, i = x - t * S;
    sm.work[t][i] = (int)(sm.keys[t][i] >> 9);
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0 && (int)(threadIdx.x >> 5) < ng) ha_allocate(sm.work[threadIdx.x >> 5], S, BZ_MAX_CODE);
  __syncthreads();
  for (int x = threadIdx.x; x < ng * S; x += HUF_BT) {
    int t = x / S, i = x - t * S;
    sm.lens[t][sm.keys[t][i] & 0x1ffu] = (u8)sm.work[t][i];
  }
  __syncthreads();
  for (int x = threadIdx.x; x < ng * S; x += HUF_BT) {
    int t = x / S, i = x - t * S;
    lens_g[t * HUF_LSTRIDE + i] = sm.lens[t][i];
  }
  for (int i = threadIdx.x; i < S; i += HUF_BT) {
    u64 v = 0;
    for (int t = 0; t < ng; t++) v |= (u64)sm.lens[t][i] << (10 * t);
    plen_g[i] = v;
  }
}

// initial tables: global histogram and flat (BJ:2155-2157)
__global__ void __launch_bounds__(HUF_BT) k_huf_init(HufArrays ha, const u32 *__restrict__ freq_in, const BlockMeta *__restrict__ meta) {
  DYN_SMEM(HufBuildSmem, smp);
  HufBuildSmem &sm = *smp;
  const u32 p = blockIdx.x;
  const u32 m = meta[p].m, alpha = meta[p].alpha;
  const int S = (int)alpha + 2;
  for (int i = threadIdx.x; i < S; i += HUF_BT) {
    sm.freq[0][i] = freq_in[(i64)p * BZ_MAX_SYMS + i];
    sm.freq[1][i] = 1;
  }
  if (threadIdx.x == 0) {
    HufBlk h;
    h.ng = 2;
    h.target = m >= 2400 ? 6 : m >= 1200 ? 5 : m >= 600 ? 4 : m >= 200 ? 3 : 2;  // BJ:2150
    h.S = S; h.active = 0; h.m = m; h.nsel = (m + BZ_GROUP - 1) / BZ_GROUP; h.pad0 = h.pad1 = 0;
    ha.hb[p] = h;
  }
  __syncthreads();
  huf_build(sm, 2, S, ha.lens + (i64)p * BZ_MAX_GROUPS * HUF_LSTRIDE, ha.plen + (i64)p * BZ_MAX_SYMS);
}

// BJ:1989-2004; also records each group's winning cost.  grid (ceil(max nsel / HUF_GT), nb)
__global__ void __launch_bounds__(HUF_GT) k_huf_assign(HufArrays ha, const u16 *__restrict__ A, i64 a_stride, int final_pass) {
  __align__(16) __shared__ u16 sy[HUF_GT_SYMS];
  __shared__ u64 pl[BZ_MAX_SYMS];
  const u32 p = blockIdx.y;
  const HufBlk h = ha.hb[p];
  if (!final_pass && h.ng >= h.target) return;
  const u32 g0 = blockIdx.x * HUF_GT;
  if (g0 >= h.nsel) return;
  const u16 *Ap = A + (i64)p * a_stride;
  const u32 i0 = g0 * BZ_GROUP, cnt = h.m - i0 < HUF_GT_SYMS ? h.m - i0 : (u32)HUF_GT_SYMS;
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(Ap + i0);  // 16-byte aligned: the stride and i0 are multiples of 8 symbols
    uint4 *dst = reinterpret_cast<uint4 *>(sy);
    for (u32 x = threadIdx.x; x < (cnt + 7) / 8; x += HUF_GT) dst[x] = src[x];
  }
  for (int i = threadIdx.x; i < h.S; i += HUF_GT) pl[i] = ha.plen[(i64)p * BZ_MAX_SYMS + i];
  __syncthreads();
  const u32 g = g0 + threadIdx.x;
  if (g >= h.nsel) return;
  const u32 j0 = threadIdx.x * BZ_GROUP, j1 = j0 + BZ_GROUP < cnt ? j0 + BZ_GROUP : cnt;
  u64 acc = 0;
  for (u32 j = j0; j < j1; j++) acc += pl[sy[j]];
  u32 best = 0, bc = (u32)(acc & 1023u);
#pragma unroll
  for (int t = 1; t < BZ_MAX_GROUPS; t++) {
    u32 ct = (u32)(acc >> (10 * t)) & 1023u;
    if (t < h.ng && ct < bc) { best = t; bc = ct; }
  }
  ha.sel[(i64)p * ha.sel_stride + g] = (u8)best;
  ha.cost[(i64)p * ha.sel_stride + g] = (u16)bc;
}

// BJ:2014-2036: first most-used table, stable median split; zeroes the histograms for k_huf_hist
__global__ void __launch_bounds__(HUF_BT) k_huf_split(HufArrays ha) {
  __shared__ u32 chist[1024];
  __shared__ u32 counts[8];
  __shared__ u32 bcast[2];
  __shared__ u32 ws[34];
  const u32 p = blockIdx.x;
  const HufBlk h = ha.hb[p];
  if (h.ng >= h.target) {
    if (threadIdx.x == 0 && h.active) ha.hb[p].active = 0;
    return;
  }
  u8 *sel = ha.sel + (i64)p * ha.sel_stride;
  const u16 *cost = ha.cost + (i64)p * ha.sel_stride;
  const u32 nsel = h.nsel;
  const int ng = h.ng;
  if (threadIdx.x < 8) counts[threadIdx.x] = 0;
  for (int i = threadIdx.x; i < 1024; i += HUF_BT) chist[i] = 0;
  __syncthreads();
  {
    u32 loc[BZ_MAX_GROUPS] = {0, 0, 0, 0, 0, 0};
    for (u32 g = threadIdx.x; g < nsel; g += HUF_BT) {
      u32 s = sel[g];
#pragma unroll
      for (int t = 0; t < BZ_MAX_GROUPS; t++) loc[t] += s == (u32)t ? 1u : 0u;
    }
#pragma unroll
    for (int t = 0; t < BZ_MAX_GROUPS; t++) {
      u32 v = warp_sum<u32>(loc[t]);
      if (lane_id() == 0 && v) atomicAdd(&counts[t], v);
    }
  }
  __syncthreads();
  int which = 0;
  for (int t = 1; t < ng; t++) if (counts[t] > counts[which]) which = t;  // first maximum (BJ:2019)
  for (u32 g = threadIdx.x; g < nsel; g += HUF_BT)
    if (sel[g] == which) atomicAdd(&chist[cost[g]], 1u);
  __syncthreads();
  const u32 len = counts[which], half = len >> 1;
  {  // cost bin that straddles the median position: the first bin whose inclusive prefix exceeds `half` (scan of the 1024 bins)
    constexpr int PER = 1024 / HUF_BT;
    u32 v[PER], mine = 0;
#pragma unroll
    for (int q = 0; q < PER; q++) { v[q] = chist[threadIdx.x * PER + q]; mine += v[q]; }
    u32 tot;
    u32 ex = block_excl_sum<u32>(mine, tot, ws);
    if (threadIdx.x == 0) { bcast[0] = 1024; bcast[1] = tot; }  // 1024 when len == 0 (cannot happen: the most-used table has a group)
    __syncthreads();
#pragma unroll
    for (int q = 0; q < PER; q++) {
      if (ex <= half && ex + v[q] > half) { bcast[0] = threadIdx.x * PER + q; bcast[1] = ex; }  // exactly one bin qualifies
      ex += v[q];
    }
  }
  __syncthreads();
  const u32 cstar = bcast[0], below = bcast[1];
  // stable split: among the groups of `which` with cost == cstar, those at position >= half (in group order) move up.
  // Every thread owns HS_E consecutive groups per round, so a round costs one block scan for HS_E * HUF_BT groups.
  constexpr int HS_E = 8;
  u32 carry = 0;
  for (u32 base = 0; base < nsel; base += HUF_BT * HS_E) {
    const u32 g0 = base + threadIdx.x * HS_E;
    u32 fl = 0, mn = 0, cnt = 0;
    u32 cgv[HS_E];
#pragma unroll
    for (int e = 0; e < HS_E; e++) {
      const u32 g = g0 + e;
      const bool mine = g < nsel && sel[g] == which;
      cgv[e] = mine ? cost[g] : 0;
      if (mine) mn |= 1u << e;
      if (mine && cgv[e] == cstar) { fl |= 1u << e; cnt++; }
    }
    u32 tot;
    u32 occ = carry + block_excl_sum<u32>(cnt, tot, ws);
#pragma unroll
    for (int e = 0; e < HS_E; e++) {
      if ((mn >> e) & 1u) {
        if (cgv[e] > cstar || (cgv[e] == cstar && below + occ >= half)) sel[g0 + e] = (u8)ng;
        occ += (fl >> e) & 1u;
      }
    }
    carry += tot;
  }
  u32 *fq = ha.freq + (i64)p * BZ_MAX_GROUPS * BZ_MAX_SYMS;
  for (int i = threadIdx.x; i < (ng + 1) * BZ_MAX_SYMS; i += HUF_BT) fq[i] = 0;
  if (threadIdx.x == 0) { ha.hb[p].ng = ng + 1; ha.hb[p].active = 1; }
}

// BJ:2037-2048: histograms of all tables.  grid (ceil(max nsel / HUF_GT), nb); one thread per group of 50 symbols
// (one table), RUNA / RUNB / rank 1 counted in registers
__global__ void __launch_bounds__(HUF_GT) k_huf_hist(HufArrays ha, const u16 *__restrict__ A, i64 a_stride) {
  __align__(16) __shared__ u16 sy[HUF_GT_SYMS];
  __shared__ u32 hs[BZ_MAX_GROUPS][BZ_MAX_SYMS];
  const u32 p = blockIdx.y;
  const HufBlk h = ha.hb[p];
  if (!h.active) return;
  const u32 g0 = blockIdx.x * HUF_GT;
  if (g0 >= h.nsel) return;
  const u16 *Ap = A + (i64)p * a_stride;
  const u32 i0 = g0 * BZ_GROUP, cnt = h.m - i0 < HUF_GT_SYMS ? h.m - i0 : (u32)HUF_GT_SYMS;
  for (int i = threadIdx.x; i < h.ng * BZ_MAX_SYMS; i += HUF_GT) (&hs[0][0])[i] = 0;
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(Ap + i0);
    uint4 *dst = reinterpret_cast<uint4 *>(sy);
    for (u32 x = threadIdx.x; x < (cnt + 7) / 8; x += HUF_GT) dst[x] = src[x];
  }
  __syncthreads();
  const u32 g = g0 + threadIdx.x;
  if (g < h.nsel) {
    const u32 j0 = threadIdx.x * BZ_GROUP, j1 = j0 + BZ_GROUP < cnt ? j0 + BZ_GROUP : cnt;
    u32 *ht = hs[ha.sel[(i64)p * ha.sel_stride + g]];
    u32 hot[3] = {0, 0, 0};
    for (u32 j = j0; j < j1; j++) {
      u32 sym = sy[j];
      if (sym < 3) { hot[0] += sym == 0; hot[1] += sym == 1; hot[2] += sym == 2; }
      else atomicAdd(&ht[sym], 1u);
    }
#pragma unroll
    for (int q = 0; q < 3; q++) if (hot[q]) atomicAdd(&ht[q], hot[q]);
  }
  __syncthreads();
  u32 *fq = ha.freq + (i64)p * BZ_MAX_GROUPS * BZ_MAX_SYMS;
  for (int x = threadIdx.x; x < h.ng * h.S; x += HUF_GT) {
    int t = x / h.S, i = x - t * h.S;
    u32 v = hs[t][i];
    if (v) atomicAdd(&fq[t * BZ_MAX_SYMS + i], v);
  }
}

// BJ:2050-2052: rebuild every table
__global__ void __launch_bounds__(HUF_BT) k_huf_build(HufArrays ha) {
  DYN_SMEM(HufBuildSmem, smp);
  HufBuildSmem &sm = *smp;
  const u32 p = blockIdx.x;
  const HufBlk h = ha.hb[p];
  if (!h.active) return;
  const u32 *fq = ha.freq + (i64)p * BZ_MAX_GROUPS * BZ_MAX_SYMS;
  for (int x = threadIdx.x; x < h.ng * h.S; x += HUF_BT) {
    int t = x / h.S, i = x - t * h.S;
    sm.freq[t][i] = fq[t * BZ_MAX_SYMS + i];
  }
  __syncthreads();
  huf_build(sm, h.ng, h.S, ha.lens + (i64)p * BZ_MAX_GROUPS * HUF_LSTRIDE, ha.plen + (i64)p * BZ_MAX_SYMS);
}

__device__ __forceinline__ void put_bits(u32 *W, u64 o, u64 val, u32 len) {
  while (len) {
    u32 bo = (u32)(o & 31), room = 32 - bo;
    u32 take = len < room ? len : room;
    u32 chunk = (u32)((val >> (len - take)) & ((1ULL << take) - 1));
    atomicOr(&W[o >> 5], chunk << (room - take));
    o += take;
    len -= take;
  }
}
// every thread contributes one (val,len) item in thread order; returns the advanced bit position
__device__ __forceinline__ u64 emit_items(u32 *W, u64 bitpos, u64 val, u32 len, u32 *ws) {
  u32 tot;
  u32 o = block_excl_sum<u32>(len, tot, ws);
  if (len) put_bits(W, bitpos + o, val, len);
  return bitpos + tot;
}

// canonical codes, block header, selectors, tables, bit offset of every group.  One CTA per block.
struct HufCodesSmem {
  u8 lens[BZ_MAX_GROUPS][HUF_LSTRIDE];
  int first[BZ_MAX_GROUPS][BZ_MAX_CODE + 2];
  u32 ws[34];
  u32 bcast[4];
};
__global__ void __launch_bounds__(HUF_CT) k_huf_codes(HufArrays ha, const BlockRec *__restrict__ recs, BlockMeta *__restrict__ meta,
                                                      u32 *__restrict__ W, i64 w_stride) {
  __shared__ HufCodesSmem sm;
  const u32 p = blockIdx.x;
  const HufBlk h = ha.hb[p];
  const int ng = h.ng, S = h.S;
  const u32 nsel = h.nsel, alpha = (u32)S - 2;
  u32 *Wp = W + (i64)p * w_stride;
  u8 *sel = ha.sel + (i64)p * ha.sel_stride;
  u16 *cost = ha.cost + (i64)p * ha.sel_stride;
  u32 *goff = ha.goff + (i64)p * ha.sel_stride;
  const u8 *lens_g = ha.lens + (i64)p * BZ_MAX_GROUPS * HUF_LSTRIDE;
  for (int x = threadIdx.x; x < ng * HUF_LSTRIDE; x += HUF_CT) (&sm.lens[0][0])[x] = lens_g[x];
  // total bits of the symbol data = sum of the winning costs; zero exactly the words this block will touch
  u32 data_bits = 0;
  for (u32 g = threadIdx.x; g < nsel; g += HUF_CT) data_bits += cost[g];
  {
    u32 tot;
    block_excl_sum<u32>(data_bits, tot, sm.ws);
    data_bits = tot;
  }
  {
    u64 maxbits = 80 + 25 + 16 + 256 + 18 + 7ull * nsel + 6ull * (5 + 258 * 39) + data_bits;
    u32 nw = (u32)((maxbits + 31) >> 5) + 2;
    if ((i64)nw > w_stride) nw = (u32)w_stride;
    for (u32 x = threadIdx.x; x < nw; x += HUF_CT) Wp[x] = 0;
  }
  __syncthreads();
  // canonical codes (BJ:1896-1916): first code of each length, then rank among equal lengths
  if ((threadIdx.x & 31) == 0 && (int)(threadIdx.x >> 5) < ng) {
    int t = threadIdx.x >> 5;
    u32 cnt[BZ_MAX_CODE + 2];
    for (int Lq = 0; Lq <= BZ_MAX_CODE + 1; Lq++) cnt[Lq] = 0;
    for (int i = 0; i < S; i++) cnt[sm.lens[t][i]]++;
    u32 code = 0;
    for (int Lq = 1; Lq <= BZ_MAX_CODE; Lq++) { sm.first[t][Lq] = (int)code; code = (code + cnt[Lq]) << 1; }
  }
  __syncthreads();
  u32 *codes = ha.codes + (i64)p * BZ_MAX_GROUPS * BZ_MAX_SYMS;
  for (int x = threadIdx.x; x < ng * S; x += HUF_CT) {
    int t = x / S, i = x - t * S, Lq = sm.lens[t][i], r = 0;
    for (int j = 0; j < i; j++) r += sm.lens[t][j] == Lq ? 1 : 0;
    codes[t * BZ_MAX_SYMS + i] = ((u32)Lq << 24) | ((u32)sm.first[t][Lq] + (u32)r);
  }
  // ---- header ----
  u64 bp = 0;
  if (threadIdx.x == 0) {
    put_bits(Wp, 0, BZ_MAGIC_BLOCK, 48);                 // BJ:2238
    put_bits(Wp, 48, recs[p].crc, 32);                   // BJ:2239
    put_bits(Wp, 80, 0, 1);                              // BJ:2061
    put_bits(Wp, 81, recs[p].orig_ptr, 24);              // BJ:2062
    u64 o = 105;
    u32 range = 0;
    for (int i = 0; i < 16; i++) {
      u32 wbits = (meta[p].used[i >> 1] >> (16 * (i & 1))) & 0xffffu;
      if (wbits) range |= 1u << (15 - i);
    }
    put_bits(Wp, o, range, 16); o += 16;                 // BJ:2071-2073
    for (int i = 0; i < 16; i++) {
      u32 wbits = (meta[p].used[i >> 1] >> (16 * (i & 1))) & 0xffffu;
      if (wbits) { put_bits(Wp, o, __brev(wbits) >> 16, 16); o += 16; }  // BJ:2074-2080
    }
    put_bits(Wp, o, (u32)ng, 3); o += 3;                 // BJ:2167
    put_bits(Wp, o, nsel, 15); o += 15;                  // BJ:2169
    sm.bcast[2] = (u32)o;
  }
  __syncthreads();
  bp = sm.bcast[2];
  // group bit offsets need the winning costs, which the selector ranks are about to overwrite: scan them first
  // (relative to the start of the symbol data; the base is added below)
  {
    u32 carry = 0;
    for (u32 base = 0; base < nsel; base += HUF_CT) {
      u32 g = base + threadIdx.x;
      u32 c = g < nsel ? cost[g] : 0, tot;
      u32 e = block_excl_sum<u32>(c, tot, sm.ws);
      if (g < nsel) goff[g] = carry + e;
      carry += tot;
    }
  }
  // selector MTF ranks (BJ:2170-2182) into cost[]: the rank of table s is the number of tables used more
  // recently than s; a table not used yet sits at its initial place (virtual last use -1-v).  Every thread
  // owns a contiguous run of groups; the last use of each table before the run comes from six max-scans.
  const bool d1 = (int)alpha < ng;
  if (!d1) {
    const u32 per = (nsel + HUF_CT - 1) / HUF_CT;
    const u32 gb = threadIdx.x * per < nsel ? threadIdx.x * per : nsel, ge = gb + per < nsel ? gb + per : nsel;
    const int NONE = -1000000;
    int last[BZ_MAX_GROUPS];
#pragma unroll
    for (int v = 0; v < BZ_MAX_GROUPS; v++) last[v] = NONE;
    for (u32 g = gb; g < ge; g++) {
      u32 sv = sel[g];
#pragma unroll
      for (int v = 0; v < BZ_MAX_GROUPS; v++) if (sv == (u32)v) last[v] = (int)g;
    }
    int cur[BZ_MAX_GROUPS];
#pragma unroll
    for (int v = 0; v < BZ_MAX_GROUPS; v++) {
      int tot;
      int e = block_excl_max<int>(last[v], NONE, tot, reinterpret_cast<int *>(sm.ws));
      cur[v] = e == NONE ? -1 - v : e;
    }
    for (u32 g = gb; g < ge; g++) {
      u32 sv = sel[g];
      int mine = 0;
#pragma unroll
      for (int v = 0; v < BZ_MAX_GROUPS; v++) if (sv == (u32)v) mine = cur[v];
      u32 j = 0;
#pragma unroll
      for (int v = 0; v < BZ_MAX_GROUPS; v++) {
        j += (v < ng && cur[v] > mine) ? 1u : 0u;
        if (sv == (u32)v) cur[v] = (int)g;
      }
      cost[g] = (u16)j;
    }
  } else if (threadIdx.x == 0) {
    // Reference defect D1 (SURVEY.md appendix E): the MTF list is a Uint8Array(alpha) shorter
    // than the table count; stores past its end vanish and loads past it never match.
    u8 ML[8];
    for (int i = 0; i < 8; i++) ML[i] = (u8)i;
    for (u32 g = 0; g < nsel; g++) {
      int s = sel[g], j;
      for (j = 0; j < ng; j++) if (j < (int)alpha && ML[j] == s) break;
      int src = j < (int)alpha ? ML[j] : 0;
      for (int q = j; q > 0; q--) if (q < (int)alpha) ML[q] = ML[q - 1];
      ML[0] = (u8)src;
      cost[g] = (u16)j;
    }
  }
  __syncthreads();
  for (u32 base = 0; base < nsel; base += HUF_CT) {
    u32 g = base + threadIdx.x;
    u32 j = g < nsel ? cost[g] : 0;
    bp = emit_items(Wp, bp, ((1ULL << j) - 1) << 1, g < nsel ? j + 1 : 0, sm.ws);
  }
  // tables (BJ:1926-1947)
  for (int t = 0; t < ng; t++) {
    int i = threadIdx.x;
    u64 val = 0;
    u32 len = 0;
    if (i < S) {
      int cur = sm.lens[t][i], prev = i ? sm.lens[t][i - 1] : cur;
      if (i == 0) { val = (u64)cur; len = 5; }
      int d = cur - prev;
      u64 two = d > 0 ? 2 : 3;
      int reps = d > 0 ? d : -d;
      for (int q = 0; q < reps; q++) { val = (val << 2) | two; len += 2; }
      val <<= 1;
      len += 1;
    }
    bp = emit_items(Wp, bp, val, len, sm.ws);
  }
  // the symbol data starts at bp
  for (u32 g = threadIdx.x; g < nsel; g += HUF_CT) goff[g] += (u32)bp;
  if (threadIdx.x == 0) {
    meta[p].n_groups = (u32)ng;
    meta[p].n_sel = nsel;
    meta[p].bits = bp + data_bits;
    meta[p].d1 = d1 ? 1u : 0u;
  }
}

// data (BJ:2189-2194): one thread per group of 50 symbols.  grid (ceil(max nsel / HUF_GT), nb)
__global__ void __launch_bounds__(HUF_GT) k_huf_emit(HufArrays ha, const u16 *__restrict__ A, i64 a_stride, u32 *__restrict__ W, i64 w_stride) {
  __align__(16) __shared__ u16 sy[HUF_GT_SYMS];
  __shared__ u32 cd[BZ_MAX_GROUPS][BZ_MAX_SYMS];
  const u32 p = blockIdx.y;
  const HufBlk h = ha.hb[p];
  const u32 g0 = blockIdx.x * HUF_GT;
  if (g0 >= h.nsel) return;
  const u16 *Ap = A + (i64)p * a_stride;
  u32 *Wp = W + (i64)p * w_stride;
  const u32 i0 = g0 * BZ_GROUP, cnt = h.m - i0 < HUF_GT_SYMS ? h.m - i0 : (u32)HUF_GT_SYMS;
  {
    const uint4 *src = reinterpret_cast<const uint4 *>(Ap + i0);
    uint4 *dst = reinterpret_cast<uint4 *>(sy);
    for (u32 x = threadIdx.x; x < (cnt + 7) / 8; x += HUF_GT) dst[x] = src[x];
  }
  {
    const u32 *codes = ha.codes + (i64)p * BZ_MAX_GROUPS * BZ_MAX_SYMS;
    for (int x = threadIdx.x; x < h.ng * BZ_MAX_SYMS; x += HUF_GT) (&cd[0][0])[x] = codes[x];
  }
  __syncthreads();
  const u32 g = g0 + threadIdx.x;
  if (g >= h.nsel) return;
  const u32 j0 = threadIdx.x * BZ_GROUP, j1 = j0 + BZ_GROUP < cnt ? j0 + BZ_GROUP : cnt;
  const u32 *tab = cd[ha.sel[(i64)p * ha.sel_stride + g]];
  const u32 o = ha.goff[(i64)p * ha.sel_stride + g];
  u32 wi = o >> 5, nbits = o & 31;  // nbits: bits already in the accumulator (the leading ones are not mine: zeros)
  u64 acc = 0;
  bool first = true;
  for (u32 j = j0; j < j1; j++) {
    u32 e = tab[sy[j]], len = e >> 24;
    acc = (acc << len) | (u64)(e & 0xffffffu);
    nbits += len;
    if (nbits >= 32) {
      nbits -= 32;
      u32 word = (u32)(acc >> nbits);
      if (first) { atomicOr(&Wp[wi], word); first = false; }  // shares its leading bits with the previous group
      else Wp[wi] = word;                                       // wholly mine
      wi++;
      acc &= (1ULL << nbits) - 1;
    }
  }
  if (nbits) atomicOr(&Wp[wi], (u32)(acc << (32 - nbits)));
}

// ---- K-S6: bit-granular concatenation of the per-block streams --------------------------
// Output bytes are produced as big-endian 32-bit words: bit 31 of word 0 is the first bit.
// offsets: header is 32 bits, block k starts at 32 + sum(bits[0..k)).
// A call in several batches passes the running bit offset as base_bits and the combined CRC of the earlier batches
// as crc_in; stream_crc is then the combined CRC of every block so far.
__global__ void __launch_bounds__(1024) k_stitch_offsets(const BlockMeta *__restrict__ meta, const BlockRec *__restrict__ recs, int nb,
                                                         u64 *__restrict__ bit_off, u32 *__restrict__ stream_crc, u64 base_bits, u32 crc_in) {
  __shared__ u64 ws[33];
  if (threadIdx.x == 0) {  // before the scan, so that crc_in does not hold a register through it
    u32 c = crc_in;
    for (int k = 0; k < nb; k++) c = ((c << 1) | (c >> 31)) ^ recs[k].crc;  // BJ:2237
    *stream_crc = c;
  }
  u64 carry = base_bits;  // 32 for a whole stream (after "BZh9"), the bit phase 0..7 for a shard segment
  for (int base = 0; base < nb; base += blockDim.x) {
    int k = base + threadIdx.x;
    u64 b = k < nb ? meta[k].bits : 0, tot;
    u64 e = block_excl_sum<u64>(b, tot, ws);
    if (k < nb) bit_off[k] = carry + e;
    carry += tot;
  }
  if (threadIdx.x == 0) bit_off[nb] = carry;
}
__device__ __forceinline__ u32 bswap32(u32 v) { return __byte_perm(v, 0, 0x0123); }
__global__ void __launch_bounds__(256) k_stitch(const u32 *__restrict__ W, i64 w_stride, const u64 *__restrict__ bit_off, u32 *__restrict__ out) {
  u32 k = blockIdx.y;
  u64 off = bit_off[k], bits = bit_off[k + 1] - off;
  u32 nwords = (u32)((bits + 31) >> 5);
  const u32 *Wp = W + (i64)k * w_stride;
  u32 sh = (u32)(off & 31);
  u64 w0 = off >> 5;
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += gridDim.x * blockDim.x) {
    u32 v = Wp[i];
    if (sh == 0) {
      atomicOr(&out[w0 + i], bswap32(v));
    } else {
      atomicOr(&out[w0 + i], bswap32(v >> sh));
      u32 lo = v << (32 - sh);
      if (lo) atomicOr(&out[w0 + i + 1], bswap32(lo));
    }
  }
}
// a shard's segment was stitched at bit phase 0; moved to its real phase (0..7) once the bit lengths of the earlier
// shards are known: dst[i] = src[i] >> phase | src[i-1] << (8 - phase), one byte more than the source
__global__ void __launch_bounds__(256) k_shift_bytes(const u8 *__restrict__ src, u64 nbytes, u32 phase, u8 *__restrict__ dst) {
  u64 i = (u64)blockIdx.x * 256 + threadIdx.x;
  if (i > nbytes) return;
  u32 cur = i < nbytes ? src[i] : 0u, prev = i ? src[i - 1] : 0u;
  dst[i] = (u8)((cur >> phase) | (prev << (8 - phase)));
}
// header, footer (BJ:2223-2226, 2245-2247) and the final length
__global__ void k_stream_ends(u32 *__restrict__ out, const u64 *__restrict__ bit_off, int nb, const u32 *__restrict__ stream_crc, int level,
                              u64 *__restrict__ out_len) {
  if (threadIdx.x || blockIdx.x) return;
  atomicOr(&out[0], bswap32(0x425A6830u + (u32)level));
  u64 o = bit_off[nb];
  u64 vals[2] = {BZ_MAGIC_END, (u64)*stream_crc};
  u32 lens[2] = {48, 32};
  for (int q = 0; q < 2; q++) {
    u64 val = vals[q];
    u32 len = lens[q];
    while (len) {
      u32 bo = (u32)(o & 31), room = 32 - bo, take = len < room ? len : room;
      u32 chunk = (u32)((val >> (len - take)) & ((1ULL << take) - 1));
      atomicOr(&out[o >> 5], bswap32(chunk << (room - take)));
      o += take;
      len -= take;
    }
  }
  *out_len = (o + 7) >> 3;
}
