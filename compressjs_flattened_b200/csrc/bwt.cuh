// bwt.cuh -- K-S2: cyclic-rotation BWT of every block by GPU prefix doubling.
//
// Replaces BWT.bwtransform2 (BJ:928-971) / SA_IS (BJ:730-857).  Semantics kept:
// rotations sorted lexicographically (unsigned bytes); equal rotations (periodic
// block) in DESCENDING start index (SURVEY.md appendix B, P5); U[j] = byte before
// the j-th rotation; origPtr = rank of rotation 0.
//
// Algorithm (Larsson-Sadakane doubling, all blocks of the batch at once):
//   ISA[i]  = current rank of rotation i = SA index (inside its block) of the first slot of its group
//   start   : key = (first L symbols of the rotation, dense codes, 44 bits) << 20 | i -> batched LSD radix sort of
//             bits 20..63 (5 passes of 9 bits, keys only); every block's slots are padded to a multiple of SORT_TILE so
//             a tile never straddles two blocks; tile_blk[] maps a tile to its block.  k_rank0 then finds
//             the groups, writes ISA and emits the ACTIVE LIST: the slots whose group has > 1 member, in
//             SA order over all blocks, as (gidx = block * stride + rotation, rank = block * stride + SA
//             index of the group's first slot).  The list is one global array: groups are contiguous runs
//             of equal rank, nothing else about blocks is needed (block = gidx / stride).
//   round h : key2 = ISA[(i+h) mod n] for every active slot (k_keys2), then every group is sorted by key2
//             (refine.cuh), new groups/ranks/ISA, singletons leave the list.  h = L, 2L, 4L, ... (per block)
//   h >= n  : remaining ties are identical rotations: key2 = n-1-i (descending index).
// Both list-producing kernels compact IN ORDER in a single pass (decoupled look-back, common.cuh).
#pragma once
#include "common.cuh"
#include "rle1.cuh"

#define SORT_TILE 4096
#ifndef SORT_THREADS
#define SORT_THREADS 512  // x 8 keys, warp-striped
#define SORT_E 8
#endif
#define SEG_THREADS 256   // x 16 slots, blocked
#define SEG_E 16
#define KEEP_BIT 0x80000000u

// ---- per-round bookkeeping: tiles of each block ------------------------------------------
// seg_tile0[p] = first tile of block p, seg_tile0[nb] = number of tiles; totals[0] = tiles,
// totals[1] = active slots (read back by the host each round).
__global__ void __launch_bounds__(1024) k_tilemap(const u32 *__restrict__ seg_cnt, int nb, u32 *__restrict__ seg_tile0,
                                                  u32 *__restrict__ tile_blk, u64 *__restrict__ totals) {
  __shared__ u32 ws[33];
  __shared__ u64 ws64[33];
  u32 carry = 0;
  u64 act = 0;
  for (int base = 0; base < nb; base += blockDim.x) {
    int p = base + threadIdx.x;
    u32 c = p < nb ? seg_cnt[p] : 0;
    u32 tiles = (c + SORT_TILE - 1) / SORT_TILE, tot;
    u32 t0 = carry + block_excl_sum<u32>(tiles, tot, ws);
    if (p < nb) {
      seg_tile0[p] = t0;
      for (u32 t = 0; t < tiles; t++) tile_blk[t0 + t] = (u32)p;
    }
    carry += tot;
    act += block_sum<u64>((u64)c, ws64);
  }
  if (threadIdx.x == 0) { seg_tile0[nb] = carry; totals[0] = carry; totals[1] = act; }
}

__global__ void k_seg_init(const BlockRec *__restrict__ recs, int nb, u32 *__restrict__ seg_cnt) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < nb) seg_cnt[p] = recs[p].n;
}

// ---- key construction ------------------------------------------------------------------------
#define KEY_BITS 44   // bits of the first sort key: 5 radix passes of 9 bits (36 bits, four passes, measured slower)
#define KEY_SLACK 2   // depth limit of the round-0 code tree above ceil(log2 alphabet)
// The first sort covers as many symbols as fit 44 bits.  Round 1 gave every symbol of a block the same number of bits
// (dense codes, b = ceil(log2 alphabet): 6 symbols of text).  Now the bytes get an ORDER-PRESERVING PREFIX-FREE code
// whose lengths follow the symbol frequencies (an alphabetic tree built by weight-balanced bisection, depth limited to
// ceil(log2 alphabet) + 2: measured 13.70 / 13.52 / 13.32 / 13.29 ms per step for + 0 / 1 / 2 / 3), and a key is the first 44 bits of the code string of the rotation: comparing such bit
// strings is comparing the rotations, frequent symbols take few bits, so a key of text covers ~8 symbols instead of 6
// and every key value is about equally likely -- fewer and smaller tie groups for the doubling rounds.  Keys that are
// equal agree on every symbol that lies wholly inside the 44 bits, at least L = 44 / (longest code) of them; L is the
// first doubling distance.  Finer-than-L ranks are harmless: a rank never contradicts the final order, and equal ranks
// still mean "equal on the first L symbols", which is all the doubling step needs.
struct BlkSort {
  u32 cnt[256];   // occurrences of every byte value in the block
  u32 L, maxlen;  // first doubling distance; longest code
  u32 pad[6];
  u8 clen[256];   // code length of a byte value (0: does not occur)
  u16 cval[256];  // code, right-aligned
};
// grid (32, nb): byte histogram of every block (warp-private counters in shared memory)
__global__ void __launch_bounds__(256) k_sym_used(const u8 *__restrict__ blk, i64 blk_stride, const BlockRec *__restrict__ recs,
                                                  BlkSort *__restrict__ bs) {
  __shared__ u32 h[8][256];
  const u32 p = blockIdx.y, n = recs[p].n;
  const u8 *T = blk + (i64)p * blk_stride;
  for (int i = threadIdx.x; i < 8 * 256; i += 256) (&h[0][0])[i] = 0;
  __syncthreads();
  u32 *hw = h[warp_id()];
  const u32 nv = n / 16;  // whole 16-byte vectors, then the tail byte by byte
  for (u32 x = blockIdx.x * 256 + threadIdx.x; x < nv; x += gridDim.x * 256) {
    uint4 v4 = reinterpret_cast<const uint4 *>(T)[x];
    u32 wv4[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
    for (int k = 0; k < 16; k++) atomicAdd(&hw[(wv4[k >> 2] >> (8 * (k & 3))) & 0xffu], 1u);
  }
  if (blockIdx.x == 0)
    for (u32 i = nv * 16 + threadIdx.x; i < n; i += 256) atomicAdd(&hw[T[i]], 1u);
  __syncthreads();
  u32 tot = 0;
#pragma unroll
  for (int w = 0; w < 8; w++) tot += h[w][threadIdx.x];
  if (tot) atomicAdd(&bs[p].cnt[threadIdx.x], tot);
}
// nb CTAs of 256 threads (thread = byte value): the code of every byte value, L
__global__ void __launch_bounds__(256) k_sym_tab(BlkSort *__restrict__ bs) {
  __shared__ u32 ws[33];
  __shared__ u32 P[257];     // P[r] = occurrences of the first r used symbols (by value)
  __shared__ u32 wmax[8];
  BlkSort &B = bs[blockIdx.x];
  const u32 c = threadIdx.x;
  const u32 f = B.cnt[c];
  u32 used = f ? 1u : 0u, alpha;
  const u32 r = block_excl_sum<u32>(used, alpha, ws);  // rank of this byte among the used ones
  u32 tot;
  const u32 pre = block_excl_sum<u32>(f, tot, ws);
  if (used) P[r] = pre;
  if (c == 0) P[alpha] = tot;
  __syncthreads();
  u32 len = 0, val = 0;
  if (used) {
    if (alpha == 1) { len = 1; val = 0; }
    else {
      u32 lb = 1;
      while ((1u << lb) < alpha) lb++;
      const u32 lmax = lb + (alpha > 2 ? KEY_SLACK : 0u);  // depth limit of the tree (at most 8 + 2 = 10 bits)
      u32 lo = 0, hi = alpha;                       // the node: used symbols [lo, hi)
      while (hi - lo > 1) {
        const u32 cap = 1u << (lmax - len - 1);     // leaves a child may still hold
        // split where the weights balance: first s with 2 * P[s] >= P[lo] + P[hi] ...
        const u64 mid2 = (u64)P[lo] + P[hi];
        u32 a = lo + 1, z = hi - 1;
        while (a < z) {
          const u32 m = (a + z) >> 1;
          if (2ull * P[m] < mid2) a = m + 1; else z = m;
        }
        u32 s = a;
        if (s > lo + 1 && 2ull * P[s] >= mid2 && mid2 - 2ull * P[s - 1] < 2ull * P[s] - mid2) s--;  // ... or the one before, whichever is closer
        // ... inside what the depth limit allows on either side
        const u32 smin = hi > cap + lo ? hi - cap : lo + 1, smax = lo + cap < hi - 1 ? lo + cap : hi - 1;
        if (s < smin) s = smin;
        if (s > smax) s = smax;
        val <<= 1;
        if (r >= s) { val |= 1u; lo = s; } else hi = s;
        len++;
      }
    }
  }
  B.clen[c] = (u8)len;
  B.cval[c] = (u16)val;
  u32 mx = warp_max<u32>(len);
  if (lane_id() == 0) wmax[warp_id()] = mx;
  __syncthreads();
  if (c == 0) {
    u32 m = 1;
    for (int w = 0; w < 8; w++) if (wmax[w] > m) m = wmax[w];
    B.maxlen = m;
    B.L = KEY_BITS / m;
  }
}
// the first KEY_BITS bits of the code string of each rotation, from bit 20 up; rotation
// index in the low 20 bits.  The tile's bytes (+ 43 more, cyclically: a key never needs more than 44 symbols) are staged
// in shared memory.  A thread owns 16 CONSECUTIVE rotations and slides a bit window over their code string (drop the
// first symbol's code, append codes at the end): ~2 table look-ups per rotation instead of one per covered symbol.  The
// keys go through shared memory so that the global stores are coalesced; the histogram of the first radix digit (bits
// 20..28) is counted on the way, so pass 0 needs no k_rs_hist.
__global__ void __launch_bounds__(SEG_THREADS) k_keys_init(const u8 *__restrict__ blk, i64 blk_stride, const BlockRec *__restrict__ recs,
                                                           const u32 *__restrict__ seg_tile0, const u32 *__restrict__ tile_blk,
                                                           const BlkSort *__restrict__ bs, u64 *__restrict__ keys, u32 *__restrict__ hist0) {
  __shared__ u32 cw[256];  // length << 16 | code
  __shared__ u8 sc[SORT_TILE + 48];
  __shared__ u32 h[512];
  __shared__ u64 sk[SORT_TILE];
  u32 tile = blockIdx.x, p = tile_blk[tile];
  u32 n = recs[p].n;
  cw[threadIdx.x] = ((u32)bs[p].clen[threadIdx.x] << 16) | bs[p].cval[threadIdx.x];
  for (int i = threadIdx.x; i < 512; i += SEG_THREADS) h[i] = 0;
  __syncthreads();
  const u8 *T = blk + (i64)p * blk_stride;
  u32 l0 = (tile - seg_tile0[p]) * SORT_TILE;
  u64 g0 = (u64)tile * SORT_TILE;
  const u32 m = n - l0 < SORT_TILE ? n - l0 : SORT_TILE;
  for (u32 j = threadIdx.x; j < m + 43; j += SEG_THREADS) {
    u32 x = l0 + j;
    if (x >= n) x %= n;
    sc[j] = T[x];
  }
  __syncthreads();
  {
    const u32 j0 = threadIdx.x * SEG_E;
    u64 buf = 0;       // code bits of symbols j .. kk-1, left-aligned
    u32 bits = 0, kk = j0;
    for (u32 e = 0; e < SEG_E; e++) {
      const u32 j = j0 + e;
      if (j >= m) break;
      while (bits < KEY_BITS) {  // at most 43 + 10 bits are ever held
        const u32 w = cw[sc[kk++]], l = w >> 16;
        buf |= (u64)(w & 0xffffu) << (64 - bits - l);
        bits += l;
      }
      const u64 key = ((buf >> (64 - KEY_BITS)) << 20) | (l0 + j);
      sk[j] = key;
      atomicAdd(&h[(u32)(key >> 20) & 511u], 1u);
      const u32 lj = cw[sc[j]] >> 16;  // the window moves on by the first symbol's code
      buf <<= lj;
      bits -= lj;
    }
  }
  __syncthreads();
  for (u32 j = threadIdx.x; j < m; j += SEG_THREADS) keys[g0 + j] = sk[j];
  for (int i = threadIdx.x; i < 512; i += SEG_THREADS) hist0[(u64)tile * 512 + i] = h[i];
}
// ---- one LSD radix pass (BITS-bit digit, 8 or 9), batched over blocks ---------------------------
// seg_base (optional): slot at which segment p starts; default = seg_tile0[p] * SORT_TILE (block layout)
template <int BITS>
__global__ void __launch_bounds__(SORT_THREADS) k_rs_hist(const u64 *__restrict__ keys, const u32 *__restrict__ seg_cnt,
                                                          const u32 *__restrict__ seg_tile0, const u32 *__restrict__ tile_blk, int shift,
                                                          u32 *__restrict__ hist, const u32 *__restrict__ seg_base) {
  constexpr int NB = 1 << BITS;
  __shared__ u32 h[NB];
  u32 tile = blockIdx.x, p = tile_blk[tile];
  u32 cnt = seg_cnt[p], l0 = (tile - seg_tile0[p]) * SORT_TILE;
  u64 g0 = seg_base ? (u64)seg_base[p] + l0 : (u64)tile * SORT_TILE;
  for (int i = threadIdx.x; i < NB; i += SORT_THREADS) h[i] = 0;
  __syncthreads();
  u64 k[SORT_E];
#pragma unroll
  for (int e = 0; e < SORT_E; e++) {  // all loads first
    u32 o = e * SORT_THREADS + threadIdx.x;
    k[e] = l0 + o < cnt ? keys[g0 + o] : 0;
  }
#pragma unroll
  for (int e = 0; e < SORT_E; e++) {
    u32 o = e * SORT_THREADS + threadIdx.x;
    if (l0 + o < cnt) atomicAdd(&h[(u32)(k[e] >> shift) & (NB - 1)], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < NB; i += SORT_THREADS) hist[(u64)tile * NB + i] = h[i];
}
// per block: column-wise exclusive prefix over its tiles (in place) and the digit totals.  grid (nb, NB / 32), 512
// threads: a CTA owns 32 digits (lane = digit), its 16 warps split the block's tiles into contiguous ranges: sum of
// the own range, exclusive scan over the warps in shared memory, then the prefixes of the own range.
#define RSS_WARPS 16
template <int BITS>
__global__ void __launch_bounds__(RSS_WARPS * 32) k_rs_scan(u32 *__restrict__ hist, const u32 *__restrict__ seg_tile0, u32 *__restrict__ digit_tot) {
  constexpr int NB = 1 << BITS;
  __shared__ u32 part[RSS_WARPS][32];
  const u32 p = blockIdx.x, d = blockIdx.y * 32 + lane_id();
  const int w = warp_id();
  const u32 t0 = seg_tile0[p], t1 = seg_tile0[p + 1], nt = t1 - t0;
  const u32 per = (nt + RSS_WARPS - 1) / RSS_WARPS;
  const u32 a = t0 + (u32)w * per < t1 ? t0 + (u32)w * per : t1, b = a + per < t1 ? a + per : t1;
  u32 sum = 0;
  for (u32 t = a; t < b; t++) sum += hist[(u64)t * NB + d];
  part[w][lane_id()] = sum;
  __syncthreads();
  u32 acc = 0;
  for (int ww = 0; ww < w; ww++) acc += part[ww][lane_id()];
  if (w == RSS_WARPS - 1) digit_tot[(u64)p * NB + d] = acc + sum;
  for (u32 t = a; t < b; t++) {
    u32 v = hist[(u64)t * NB + d];
    hist[(u64)t * NB + d] = acc;
    acc += v;
  }
}
template <int BITS>
__global__ void __launch_bounds__(SORT_THREADS, 3) k_rs_scatter(const u64 *__restrict__ keys_in, u64 *__restrict__ keys_out,
                                                             const u32 *__restrict__ seg_cnt, const u32 *__restrict__ seg_tile0,
                                                             const u32 *__restrict__ tile_blk, int shift, const u32 *__restrict__ hist,
                                                             const u32 *__restrict__ digit_tot, const u32 *__restrict__ seg_base) {
  constexpr int NB = 1 << BITS;
  __shared__ u16 wcnt[SORT_THREADS / 32][NB];  // a warp ranks 256 keys: counts fit 16 bits
  __shared__ u32 base[NB];
  u32 tile = blockIdx.x, p = tile_blk[tile];
  u32 cnt = seg_cnt[p], l0 = (tile - seg_tile0[p]) * SORT_TILE;
  u64 gp = seg_base ? (u64)seg_base[p] : (u64)seg_tile0[p] * SORT_TILE, g0 = gp + l0;
  int lane = lane_id(), w = warp_id();
  for (int i = threadIdx.x; i < (SORT_THREADS / 32) * NB / 2; i += SORT_THREADS) reinterpret_cast<u32 *>(&wcnt[0][0])[i] = 0;
  {  // base of digit d = keys of the block with a smaller digit (scan of the totals) + keys with digit d in earlier tiles
    static_assert(NB <= SORT_THREADS, "one digit per thread");
    __shared__ u32 ws[33];
    u32 tot_d = threadIdx.x < NB ? digit_tot[(u64)p * NB + threadIdx.x] : 0u, tot;
    u32 ex = block_excl_sum<u32>(tot_d, tot, ws);
    if (threadIdx.x < NB) base[threadIdx.x] = ex + hist[(u64)tile * NB + threadIdx.x];
  }
  __syncthreads();
  u64 key[SORT_E];
  u32 rk[SORT_E];
  u32 lt = (1u << lane) - 1;
#pragma unroll
  for (int e = 0; e < SORT_E; e++) {  // all loads first: eight independent requests in flight per thread
    u32 o = (u32)w * (32 * SORT_E) + e * 32 + lane;
    key[e] = l0 + o < cnt ? keys_in[g0 + o] : 0;
  }
#pragma unroll
  for (int e = 0; e < SORT_E; e++) {
    u32 o = (u32)w * (32 * SORT_E) + e * 32 + lane;
    bool ok = l0 + o < cnt;
    u32 d = ok ? ((u32)(key[e] >> shift) & (NB - 1)) : (u32)NB;
    u32 peers = __match_any_sync(FULL_MASK, d);
    int leader = __ffs((int)peers) - 1;
    u32 old = 0;
    if (lane == leader && ok) { old = wcnt[w][d]; wcnt[w][d] = (u16)(old + __popc(peers)); }
    old = __shfl_sync(FULL_MASK, old, leader);
    rk[e] = old + __popc(peers & lt);
    __syncwarp();
  }
  __syncthreads();
  for (int d = threadIdx.x; d < NB; d += SORT_THREADS) {  // exclusive prefix of each digit over the warps
    u32 acc = 0;
    for (int ww = 0; ww < SORT_THREADS / 32; ww++) { u32 t = wcnt[ww][d]; wcnt[ww][d] = (u16)acc; acc += t; }
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < SORT_E; e++) {
    u32 o = (u32)w * (32 * SORT_E) + e * 32 + lane;
    if (l0 + o < cnt) {
      u32 d = (u32)(key[e] >> shift) & (NB - 1);
      u64 dst = gp + base[d] + wcnt[w][d] + rk[e];
      keys_out[dst] = key[e];
    }
  }
}

// ---- regrouping after a sort ---------------------------------------------------------------
__device__ __forceinline__ void seg_load_flags(const u64 *__restrict__ keys, u64 g0, u32 l0, u32 cnt, int kshift, u64 k[SEG_E], u32 &flags, u32 &lbase) {
  lbase = l0 + threadIdx.x * SEG_E;
  u64 g = g0 + (u64)threadIdx.x * SEG_E;
  flags = 0;
  u64 prev = (lbase > 0 && lbase < cnt) ? keys[g - 1] : 0;
#pragma unroll
  for (int e = 0; e < SEG_E; e++) {
    if (lbase + e < cnt) {
      k[e] = keys[g + e];
      if (lbase + e == 0 || (k[e] >> kshift) != (prev >> kshift)) flags |= 1u << e;
      prev = k[e];
    }
  }
}
// last sub-group head (slot index within the block) of every tile, or -1
__global__ void __launch_bounds__(SEG_THREADS) k_sub_heads(const u64 *__restrict__ keys, const u32 *__restrict__ seg_cnt,
                                                           const u32 *__restrict__ seg_tile0, const u32 *__restrict__ tile_blk,
                                                           int *__restrict__ tile_last, const u32 *__restrict__ seg_base, int kshift) {
  __shared__ int ws[33];
  u32 tile = blockIdx.x, p = tile_blk[tile];
  u32 cnt = seg_cnt[p], l0 = (tile - seg_tile0[p]) * SORT_TILE;
  u64 k[SEG_E];
  u32 flags, lbase;
  seg_load_flags(keys, seg_base ? (u64)seg_base[p] + l0 : (u64)tile * SORT_TILE, l0, cnt, kshift, k, flags, lbase);
  int last = flags ? (int)(lbase + (31 - __clz((int)flags))) : -1;
  last = block_max<int>(last, ws);
  if (threadIdx.x == 0) tile_last[tile] = last;
}
// per block: exclusive max-scan (mode 0, int, identity -1) or exclusive sum-scan (mode 1, u32;
// also writes the block's new count) of a per-tile array over the block's tiles
__global__ void __launch_bounds__(256) k_seg_scan(const u32 *__restrict__ seg_tile0, int mode, const int *__restrict__ in, int *__restrict__ out,
                                                  u32 *__restrict__ seg_cnt_new) {
  __shared__ int ws[33];
  u32 p = blockIdx.x, t0 = seg_tile0[p], t1 = seg_tile0[p + 1];
  int carry = mode == 0 ? -1 : 0;
  for (u32 base = t0; base < t1; base += blockDim.x) {
    u32 t = base + threadIdx.x;
    int tot;
    if (mode == 0) {
      int v = t < t1 ? in[t] : -1;
      int e = block_excl_max<int>(v, -1, tot, ws);
      if (t < t1) out[t] = e > carry ? e : carry;
      if (tot > carry) carry = tot;
    } else {
      int v = t < t1 ? in[t] : 0;
      int e = block_excl_sum<int>(v, tot, ws);
      if (t < t1) out[t] = carry + e;
      carry += tot;
    }
  }
  if (mode == 1 && threadIdx.x == 0) seg_cnt_new[p] = (u32)carry;
}
// A rotation whose rank is final writes its byte of the L column (the byte before the rotation) and, for
// rotation 0, origPtr.  gidx = block base pb + rotation index; rank is global too (same stride everywhere).
__device__ __forceinline__ void bwt_emit_final(const u8 *__restrict__ T, u8 *__restrict__ L, BlockRec *__restrict__ recs, u32 p, u32 pb, u32 gidx,
                                               u32 rank) {
  if (gidx != pb) L[rank] = T[gidx - 1];
  else {
    L[rank] = T[pb + recs[p].n - 1];
    recs[p].orig_ptr = rank - pb;
  }
}

// ---- round 0 regroup: groups, ISA, active list (single pass, ordered) -------------------------------
#define R0_THREADS 512
#define R0_ROWS (SORT_TILE / R0_THREADS)  // rows of 32 slots per warp: warp w owns slots [w*256, w*256+256)
#define R0_NOKEY 0xffffffffffffffffull   // filler outside the block; the block's ends are tested explicitly
__global__ void __launch_bounds__(R0_THREADS) k_rank0(const u64 *__restrict__ keys, const u32 *__restrict__ seg_cnt,
                                                      const u32 *__restrict__ seg_tile0, const u32 *__restrict__ tile_blk,
                                                      u32 *__restrict__ isa, i64 stride, u32 *__restrict__ act_idx, u32 *__restrict__ act_rank,
                                                      u64 *__restrict__ status, u32 *__restrict__ ticket, u32 *__restrict__ n_act_out, u32 ntiles,
                                                      const u8 *__restrict__ T, u8 *__restrict__ L, BlockRec *__restrict__ recs) {
  __shared__ u64 sk[SORT_TILE + 2];  // sk[1 + i] = key of tile slot i; sk[0] / sk[m + 1] = the neighbours
  __shared__ int wlast[R0_THREADS / 32];
  __shared__ u32 wkeep[R0_THREADS / 32];
  __shared__ u32 sh_tile, sh_base;
  __shared__ int sh_carry;
  const int lane = lane_id(), w = warp_id();
  if (threadIdx.x == 0) sh_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const u32 tile = sh_tile, p = tile_blk[tile];
  const u32 cnt = seg_cnt[p], l0 = (tile - seg_tile0[p]) * SORT_TILE;
  const u64 gp = (u64)seg_tile0[p] * SORT_TILE;
  const u32 m = cnt - l0 < SORT_TILE ? cnt - l0 : SORT_TILE;
  for (u32 i = threadIdx.x; i < m + 2; i += R0_THREADS) {
    i64 j = (i64)l0 - 1 + i;
    sk[i] = (j >= 0 && j < (i64)cnt) ? keys[gp + (u64)j] : R0_NOKEY;
  }
  __syncthreads();
  // phase 1: head / keep ballots of this warp's rows
  u32 hb[R0_ROWS], kb[R0_ROWS];
  int wl = -1;
  u32 nkeep = 0;
#pragma unroll
  for (int e = 0; e < R0_ROWS; e++) {
    u32 i = (u32)w * (32 * R0_ROWS) + e * 32 + lane;
    bool valid = i < m, head = false, nh = false;
    if (valid) {
      u64 k = sk[i + 1] >> 20;
      head = l0 + i == 0 || k != (sk[i] >> 20);
      nh = l0 + i + 1 >= cnt || k != (sk[i + 2] >> 20);
    }
    hb[e] = __ballot_sync(FULL_MASK, head);
    kb[e] = __ballot_sync(FULL_MASK, valid && !(head && nh));
    if (hb[e]) wl = (int)(w * (32 * R0_ROWS) + e * 32 + (31 - __clz((int)hb[e])));
    nkeep += __popc(kb[e]);
  }
  if (lane == 0) { wlast[w] = wl; wkeep[w] = nkeep; }
  if (w == 0) {
    // head of the group that contains the tile's first slot when that slot is not a head itself
    int carry = (int)l0;
    if (l0 > 0 && (sk[1] >> 20) == (sk[0] >> 20)) {
      const u64 P5 = sk[1] >> 20;
      const u64 *K = keys + gp;
      i64 res = -1;
      for (u32 c0 = 0; c0 < 64 && res < 0; c0 += 32) {  // slot l0-1 has the prefix; test l0-2-c0-lane
        i64 j = (i64)l0 - 2 - c0 - lane;
        bool diff = j < 0 || (K[j] >> 20) != P5;
        u32 b = __ballot_sync(FULL_MASK, diff);
        if (b) res = (i64)l0 - 1 - c0 - (__ffs((int)b) - 1);
      }
      if (res < 0) {  // long group: first slot of the block with prefix >= P5
        u32 lo = 0, hi = l0 - 1;
        while (lo < hi) {
          u32 mid = (lo + hi) >> 1;
          if ((K[mid] >> 20) < P5) lo = mid + 1; else hi = mid;
        }
        res = lo;
      }
      carry = (int)res;
    }
    if (lane == 0) sh_carry = carry;
  }
  __syncthreads();
  int cur = sh_carry;  // block-local SA index of the last head before this warp's slots
  for (int ww = 0; ww < w; ww++) if (wlast[ww] >= 0) cur = (int)l0 + wlast[ww];
  // phase 2a: ranks + ISA (before the look-back, whose latency these scattered stores hide)
  const u32 pb = (u32)((u64)p * (u64)stride);
  const u32 le = lane == 31 ? 0xffffffffu : ((2u << lane) - 1);  // lanes <= mine
  const u32 lt = (1u << lane) - 1;
  u32 hpv[R0_ROWS];
#pragma unroll
  for (int e = 0; e < R0_ROWS; e++) {
    u32 i = (u32)w * (32 * R0_ROWS) + e * 32 + lane;
    u32 mk = hb[e] & le;
    int hp = mk ? (int)(l0 + w * (32 * R0_ROWS) + e * 32 + (31 - __clz((int)mk))) : cur;
    hpv[e] = (u32)hp;
    if (i < m) {
      const u32 gidx = pb + (u32)(sk[i + 1] & 0xFFFFFu);
      isa[gidx] = (u32)hp;
      if (!((kb[e] >> lane) & 1u)) bwt_emit_final(T, L, recs, p, pb, gidx, pb + (u32)hp);  // a singleton: final
    }
    if (hb[e]) cur = (int)(l0 + w * (32 * R0_ROWS) + e * 32 + (31 - __clz((int)hb[e])));
  }
  // ordered compaction base of this tile and of this warp
  if (w == 0) {
    u32 x = lane < R0_THREADS / 32 ? wkeep[lane] : 0;
    u32 inc = warp_incl_sum<u32>(x);
    u32 agg = __shfl_sync(FULL_MASK, inc, 31);
    u32 base = lookback_warp(status, tile, agg);
    if (lane < R0_THREADS / 32) wkeep[lane] = inc - x;
    if (lane == 0) {
      sh_base = base;
      if (tile == ntiles - 1) *n_act_out = base + agg;
    }
  }
  __syncthreads();
  // phase 2b: survivors
  u32 out = sh_base + wkeep[w];
#pragma unroll
  for (int e = 0; e < R0_ROWS; e++) {
    u32 i = (u32)w * (32 * R0_ROWS) + e * 32 + lane;
    if (i < m && ((kb[e] >> lane) & 1u)) {
      u32 o = out + __popc(kb[e] & lt);
      act_idx[o] = pb + (u32)(sk[i + 1] & 0xFFFFFu);
      act_rank[o] = pb + hpv[e];
    }
    out += __popc(kb[e]);
  }
}

