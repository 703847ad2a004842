// lines.cuh -- the newline directory over decoded bytes in HBM (bz2b200_line_index, bz2b200_decompress_lines; included
// after search.cuh, whose k_scan64_* turn the tile counts into their prefix).
//
// The bytes [0, n) are cut into TILES of `tile` bytes (a multiple of 256, at most LINE_TILE_MAX).  One warp per tile, or
// per query, reads 16-byte words and finds the '\n' bytes of a word with a SWAR compare, so no byte is looked at twice:
//   k_nl_tiles   '\n' bytes per tile -> counts[t]; k_scan64_* then make counts the exclusive prefix, counts[n_tiles] the total
//   k_nl_rank    byte position p (<= n) -> '\n' bytes before p: the prefix of its tile plus a count over the tile up to p
//   k_nl_select  rank k (< the total) -> position of the k-th '\n' (0-based): a binary search of the prefix for the tile,
//                then the warp walks the tile 512 bytes at a time (one word per lane, a warp scan of the counts) and the
//                lane that holds the k-th '\n' takes it from its word's 16-bit mask with __fns
// A word is read whole even where it runs past n (a decode sink keeps 64 bytes of slack after its bytes); what lies past
// n or past the tile is masked off and never counted.  k_index_rows (below) counts the input of the compressor's blocks
// with the same helpers.
#define LINE_TILE_DEFAULT 8192u
#define LINE_TILE_MAX 8192u
#define NL_THREADS 256              // 8 warps per CTA: 8 tiles or 8 queries
#define NL_WARPS (NL_THREADS / 32)

// 0x80 in every byte of w that is '\n', 0 in every other byte (exact: the add cannot carry from one byte into the next)
__host__ __device__ __forceinline__ u32 nl_marks(u32 w) {
  const u32 t = w ^ 0x0a0a0a0au;
  return ~(((t & 0x7f7f7f7fu) + 0x7f7f7f7fu) | t | 0x7f7f7f7fu);
}
// the bytes of word i (0..3) of a 16-byte word that lie among its first `valid` bytes
__device__ __forceinline__ u32 nl_keep(u32 valid, u32 i) {
  const u32 v = valid > 4 * i ? valid - 4 * i : 0;
  return v >= 4 ? 0xffffffffu : (1u << (8 * v)) - 1u;
}
// the marks of the first `valid` bytes of x (valid >= 16: all of them)
__device__ __forceinline__ uint4 nl_marks16(uint4 x, u32 valid) {
  uint4 m = make_uint4(nl_marks(x.x), nl_marks(x.y), nl_marks(x.z), nl_marks(x.w));
  if (valid < 16) { m.x &= nl_keep(valid, 0); m.y &= nl_keep(valid, 1); m.z &= nl_keep(valid, 2); m.w &= nl_keep(valid, 3); }
  return m;
}
__device__ __forceinline__ u32 nl_count16(uint4 m) { return __popc(m.x) + __popc(m.y) + __popc(m.z) + __popc(m.w); }
// bit j set: byte j of the word is a marked '\n'
__device__ __forceinline__ u32 nl_bits16(uint4 m) {
  u32 r = 0;
  const u32 w[4] = {m.x, m.y, m.z, m.w};
  for (int i = 0; i < 4; i++)
    r |= (((w[i] >> 7) & 1u) | ((w[i] >> 14) & 2u) | ((w[i] >> 21) & 4u) | ((w[i] >> 28) & 8u)) << (4 * i);
  return r;
}
__device__ __forceinline__ u64 nl_warp_sum(u64 v) {
  for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}
// '\n' bytes in [a, e) (a a multiple of 16, e - a at most a tile), summed over the warp
__device__ __forceinline__ u64 nl_warp_count(const u8 *__restrict__ src, u64 a, u64 e, u32 lane) {
  u32 cnt = 0;
#pragma unroll 4
  for (u64 b = a + 16 * (u64)lane; b < e; b += 16 * 32) {
    const uint4 x = *reinterpret_cast<const uint4 *>(src + b);
    cnt += nl_count16(nl_marks16(x, e - b < 16 ? (u32)(e - b) : 16u));
  }
  return nl_warp_sum(cnt);
}

__global__ void __launch_bounds__(NL_THREADS) k_nl_tiles(const u8 *__restrict__ src, u64 n, u32 tile, u32 n_tiles, u64 *__restrict__ counts) {
  const u32 t = blockIdx.x * NL_WARPS + threadIdx.x / 32, lane = threadIdx.x & 31;
  if (t >= n_tiles) return;
  const u64 t0 = (u64)t * tile, e = n - t0 < tile ? n : t0 + tile;
  const u64 c = nl_warp_count(src, t0, e, lane);
  if (lane == 0) counts[t] = c;
}

// prefix: n_tiles + 1 entries (the exclusive prefix of the tile counts, then the total); pos[q] <= n
__global__ void __launch_bounds__(NL_THREADS) k_nl_rank(const u8 *__restrict__ src, u32 tile, const u64 *__restrict__ prefix, const u64 *__restrict__ pos,
                                                        u32 nq, u64 *__restrict__ out) {
  const u32 q = blockIdx.x * NL_WARPS + threadIdx.x / 32, lane = threadIdx.x & 31;
  if (q >= nq) return;
  const u64 p = pos[q], t = p / tile;
  const u64 c = nl_warp_count(src, t * tile, p, lane);
  if (lane == 0) out[q] = prefix[t] + c;
}

// ks[q] < prefix[n_tiles]
__global__ void __launch_bounds__(NL_THREADS) k_nl_select(const u8 *__restrict__ src, u64 n, u32 tile, u32 n_tiles, const u64 *__restrict__ prefix,
                                                          const u64 *__restrict__ ks, u32 nq, u64 *__restrict__ out) {
  const u32 q = blockIdx.x * NL_WARPS + threadIdx.x / 32, lane = threadIdx.x & 31;
  if (q >= nq) return;
  const u64 k = ks[q];
  u32 lo = 0, hi = n_tiles;  // prefix[lo] <= k < prefix[hi]
  while (hi - lo > 1) {
    const u32 mid = (lo + hi) >> 1;
    if (prefix[mid] <= k) lo = mid; else hi = mid;
  }
  u64 r = k - prefix[lo];
  const u64 t0 = (u64)lo * tile, e = n - t0 < tile ? n : t0 + tile;
  for (u64 c = t0; c < e; c += 16 * 32) {
    const u64 b = c + 16 * (u64)lane;
    u32 bits = 0;
    if (b < e) bits = nl_bits16(nl_marks16(*reinterpret_cast<const uint4 *>(src + b), e - b < 16 ? (u32)(e - b) : 16u));
    const u32 cnt = __popc(bits);
    u32 incl = cnt;
    for (int d = 1; d < 32; d <<= 1) {
      const u32 v = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= (u32)d) incl += v;
    }
    const u32 total = __shfl_sync(0xffffffffu, incl, 31);
    if (r < total) {
      const u32 owner = __ffs((int)__ballot_sync(0xffffffffu, incl > r)) - 1;
      if (lane == owner) out[q] = b + __fns(bits, 0, (int)(r - (incl - cnt)) + 1);
      return;
    }
    r -= total;
  }
}

// ---- the line index of a compress call (bz2b200_compress_indexed and friends) ----------------------------------------
// Launched once per batch of the compressor, right after k_stitch_offsets.  For block b of the batch it writes the
// bz2b200_block_entry row rows[b] -- bits from bit_off (absolute for a whole stream, from 0 for a shard segment: the caller
// moves them), out_offset = the block's first input byte s (the caller adds the offset of the input buffer), out_bytes =
// p - s, since the block decodes to exactly the input bytes [s, p) -- and adds the '\n' bytes of [s, p) into counts[b]
// (zeroed by the caller).  A run-heavy block spans up to ~46 MB of input, so the grid is (segments, blocks): CTA (x, y)
// counts segment x -- `seg` bytes from the 16-byte word that holds s -- of blocks y, y + gridDim.y, ..., one atomicAdd per
// CTA.  Every word is loaded once with a 16-byte load (the word a block boundary cuts is loaded by both blocks); the bytes
// before s and from p on are masked off.  A word read past p stays inside the input buffer's 64 bytes of slack.
#define IX_THREADS 256
#define IX_SEG_DEFAULT 32768u  // bytes per segment (bz2b200_debug_set_line_tile sets it for tests)

// m without its first k bytes
__device__ __forceinline__ uint4 nl_drop16(uint4 m, u32 k) {
  m.x &= ~nl_keep(k, 0); m.y &= ~nl_keep(k, 1); m.z &= ~nl_keep(k, 2); m.w &= ~nl_keep(k, 3);
  return m;
}

__global__ void __launch_bounds__(IX_THREADS) k_index_rows(const u8 *__restrict__ in, const BlockRec *__restrict__ recs, const u64 *__restrict__ bit_off,
                                                           int nb, u32 seg, u32 level, bz2b200_block_entry *__restrict__ rows, u32 *__restrict__ counts) {
  __shared__ u32 part[IX_THREADS / 32];
  const u32 lane = threadIdx.x & 31, warp = threadIdx.x / 32;
  for (int b = blockIdx.y; b < nb; b += gridDim.y) {
    const u64 s = (u64)recs[b].s, p = (u64)recs[b].p;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      bz2b200_block_entry e;
      e.bit_begin = bit_off[b]; e.bit_end = bit_off[b + 1];
      e.out_offset = s; e.out_bytes = (u32)(p - s);
      e.crc = recs[b].crc; e.stream = 0; e.level = level;
      rows[b] = e;
    }
    const u64 a = (s & ~(u64)15) + (u64)blockIdx.x * seg;
    if (a >= p) continue;  // the same for the whole CTA
    const u64 e = p - a < seg ? p : a + seg;
    u32 cnt = 0;
#pragma unroll 4
    for (u64 w = a + 16 * (u64)threadIdx.x; w < e; w += 16 * IX_THREADS) {
      uint4 m = nl_marks16(*reinterpret_cast<const uint4 *>(in + w), e - w < 16 ? (u32)(e - w) : 16u);
      if (w < s) m = nl_drop16(m, (u32)(s - w));
      cnt += nl_count16(m);
    }
    cnt = (u32)nl_warp_sum(cnt);
    if (lane == 0) part[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
      u32 t = 0;
      for (int i = 0; i < IX_THREADS / 32; i++) t += part[i];
      if (t) atomicAdd(&counts[b], t);
    }
    __syncthreads();
  }
}
