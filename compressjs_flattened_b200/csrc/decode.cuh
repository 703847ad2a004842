// decode.cuh -- K-U1..U4: the decompress path.
//
// Replaces Bunzip (BJ:1393-1863): _get_next_block (BJ:1428-1709), _read_bunzip (BJ:1716-1763).
//   K-U1 k_magic_scan    : every bit offset is tested for the 48-bit block / end-of-stream magic
//                          (the reference has no search: it walks the stream sequentially; the host
//                          re-creates that walk over the candidates, so false hits are ignored)
//   K-U2   dec_header     : header fields, selectors (parallel: zero-bit ranks by a CTA scan, MTF moves composed
//                          as position maps), code lengths, limit/base/permute and a 10-bit LUT built by replaying
//                          the reference's walk (BJ:1434-1581)
//   K-U3a  k_huff_parse   : bits -> symbols (BJ:1597-1616), one CTA per candidate block; serial across the groups of
//                          50 symbols (table switch), parallel inside a group (pointer doubling over "next code")
//          k_huff_parse_win: the same for few blocks: a window of offsets decoded under every table of the next
//                          groups, one dependent chain of reads per group
//   K-U3b k_sym_offsets  : RLE2^-1 as a scan: the k-th RUNA/RUNB of a run = (sym+1)<<k copies of the front
//   K-U3c k_imtf_*       : MTF^-1 in parallel: every segment runs the MTF once from the identity list (list striped
//                          over a warp) and emits list positions + its permutation; permutations composed per
//                          block; positions mapped to bytes through the list at the segment start
//   K-U4a                : T-vector = one stable 8-bit radix pass (bwt.cuh kernels) of positions by byte, packed
//                          with the L byte like the reference's dbuf
//   K-U4b k_ibwt_*       : list ranking: splitters every IBWT_S slots walk to the next splitter, one CTA per
//                          block ranks the splitters (two levels, shared memory), second walk writes bytes
//   K-U4c k_rle1_inv     : RLE1^-1 in parallel: inside a maximal run of equal bytes every 5th byte
//                          is a count; whether a run's first byte is the previous run's count is a
//                          1-bit state propagated by a scan of functions {0,1}->{0,1}
//   CRC                  : k_crc_chunks / k_crc_fold (rle1.cuh) over each block's output range
#pragma once
#include "common.cuh"
#include "rle1.cuh"
#include "bwt.cuh"

#define DEC_LUT_BITS 10
#define DEC_LUT_BAD 0xffffu  // LUT entry of a prefix the reference's walk rejects; 0 = code longer than the LUT
#define DEC_MAX_SEL 32768
#define DEC_DBUF_MAX 900000
#define IBWT_S ibwt_s  // splitter spacing: a kernel parameter / host variable (power of two)

struct DecBlk {
  u64 bitpos;      // position of the 48-bit magic
  u64 endbit;      // first bit after the end-of-block symbol
  u32 target_crc;  // BJ:1440
  u32 orig_ptr;    // BJ:1448
  u32 count;       // dbufCount: bytes of the L column; with err: the symbols parsed before the error, then (k_sym_offsets)
                   // the most bytes a size check saw among them
  int err;         // 0 or a negative Err code
  u32 kind;        // 0 = block magic, 1 = end-of-stream magic (then target_crc = stream CRC)
  u32 nsym;        // symbols parsed, including end-of-block (0 with err)
};

// ---- K-U1 -----------------------------------------------------------------------------------
// bytes [b0, b1) of the buffer (n bytes readable): a range of a stream scans only its own bytes
__global__ void __launch_bounds__(256) k_magic_scan(const u8 *__restrict__ in, u64 n, u64 b0, u64 b1, u64 *__restrict__ cand, u32 cap,
                                                    u32 *__restrict__ ncand) {
  u64 i = b0 + (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b1 || i >= n) return;
  u64 w = 0;
  for (int k = 0; k < 8; k++) w = (w << 8) | (i + k < n ? in[i + k] : 0);
  for (int b = 0; b < 8; b++) {
    u64 v = (w >> (16 - b)) & 0xFFFFFFFFFFFFULL;
    if (v == BZ_MAGIC_BLOCK || v == BZ_MAGIC_END) {
      u32 slot = atomicAdd(ncand, 1u);
      if (slot < cap) cand[slot] = ((i * 8 + b) << 1) | (v == BZ_MAGIC_END ? 1u : 0u);
    }
  }
}

// ---- K-U2/3 ---------------------------------------------------------------------------------
struct BitRd {
  const u8 *p;
  u64 n, pos;  // next byte to load
  u64 buf;
  u32 avail;
  u32 overrun;  // a bit past EOF was needed (reads as 0, BJ:149-150)
};
__device__ __forceinline__ void br_init(BitRd &r, const u8 *p, u64 n, u64 bit) {
  r.p = p; r.n = n; r.pos = bit >> 3; r.buf = 0; r.avail = 0; r.overrun = 0;
  u32 skip = (u32)(bit & 7);
  if (skip) {
    r.buf = r.pos < n ? p[r.pos] : 0;
    if (r.pos >= n) r.overrun = 1;
    r.pos++;
    r.avail = 8 - skip;
    r.buf &= (1u << r.avail) - 1;
  }
}
__device__ __forceinline__ void br_fill(BitRd &r, u32 need) {
  while (r.avail < need) {
    u32 b = 0;
    if (r.pos < r.n) b = r.p[r.pos]; else r.overrun = 1;
    r.pos++;
    r.buf = (r.buf << 8) | b;
    r.avail += 8;
  }
}
__device__ __forceinline__ u32 br_get(BitRd &r, u32 nb) {  // nb <= 32
  if (nb == 0) return 0;
  br_fill(r, nb);
  u32 v = (u32)((r.buf >> (r.avail - nb)) & ((1ULL << nb) - 1));
  r.avail -= nb;
  return v;
}
__device__ __forceinline__ u32 br_peek(BitRd &r, u32 nb) {
  br_fill(r, nb);
  return (u32)((r.buf >> (r.avail - nb)) & ((1ULL << nb) - 1));
}
__device__ __forceinline__ u64 br_tell(const BitRd &r) { return r.pos * 8 - r.avail; }

#define DEC_RING 4096       // bytes of compressed input staged in shared memory per pass
// threads of k_huff_parse = bit offsets looked at per step (template parameter).  Measured on B200 per 100 MB: level 9
// (112 blocks) 128 -> 38.1 ms, 256 -> 29.7, 512 -> 31.6; level 1 (1000 blocks) 128 -> 17.5, 256 -> 16.8: 256 is used
#define DEC_LEVELS 6        // pointer-doubling levels: 2^6 > 50 codes of a group
#define DEC_SYM_STAGE 1024  // symbols staged per pass
#define DEC_SYM_STRIDE 900096  // u16 symbols per candidate (dbuf + end-of-block + slack)
#define IMTF_SEG 4096       // symbols per inverse-MTF segment

template <int PT>
struct DecSmem {
  int limit[BZ_MAX_GROUPS][BZ_MAX_CODE + 2];
  int base[BZ_MAX_GROUPS][BZ_MAX_CODE + 2];
  u16 permute[BZ_MAX_GROUPS][BZ_MAX_SYMS + 2];
  u16 lut[BZ_MAX_GROUPS][1 << DEC_LUT_BITS];
  u8 lens[BZ_MAX_GROUPS][BZ_MAX_SYMS + 2];
  int minl[BZ_MAX_GROUPS], maxl[BZ_MAX_GROUPS];
  u8 mtf[256];
  u8 sym2byte[256];
  __align__(16) u8 ring[DEC_RING + 16];
  u16 stage[DEC_SYM_STAGE];
  int hdr[8];  // err, ng, nsel, sym_total, overrun so far
  u32 scr[72];  // CTA scans of the header
  u64 sel_end;  // first bit after the selectors
  u64 bitpos_after_header;
  u16 J[DEC_LEVELS][PT];  // J[k][b]: bit offset reached from offset b after 2^k codes (>= DEC_PT: outside the step)
  u16 SY[PT];             // symbol decoded at offset b | 0x8000 if the code there is invalid
  u16 csym[64], cend[64];     // symbol and end offset of the r-th code of the chain
  u8 selbuf[256];             // selectors of the pass
  u32 ws[34];
  u32 first_eob, first_bad, first_eof, adv;
};

// a code the LUT does not hold: entry 0 = longer than DEC_LUT_BITS -> the reference's limit/base/permute walk
// (BJ:1605-1616) continued from there on a 32-bit window; DEC_LUT_BAD or a failed walk = invalid code, which comes back
// as length 1 with DEC_BAD set (it keeps the chain moving and only counts when it is ON the chain)
#define DEC_BAD (1u << 20)  // bit 15 of the symbol field: invalid code
#define DEC_BAD_CODE(bits_read) (DEC_BAD | ((u32)(bits_read) << 21) | 1u)
template <typename SM>
__device__ __forceinline__ u32 dec_long_code_inl(const SM &sm, int gi, u32 win, u32 entry) {
  // (an invalid code also reports how many bits the reference's walk read before it gave up, bits 21+: whether those
  // reach past the end of the input decides between "data error" and "unexpected EOF")
  int L = sm.minl[gi];
  if (entry != DEC_LUT_BAD && L < DEC_LUT_BITS + 1) L = DEC_LUT_BITS + 1;
  int j = (int)(win >> (32 - L));
  for (;; L++) {
    if (L > sm.maxl[gi]) return DEC_BAD_CODE(sm.maxl[gi] + 1);
    if (j <= sm.limit[gi][L]) break;
    j = (j << 1) | (int)((win >> (31 - L)) & 1u);
  }
  j -= sm.base[gi][L];
  if (j < 0 || j >= BZ_MAX_SYMS) return DEC_BAD_CODE(L);
  return ((u32)sm.permute[gi][j] << 5) | (u32)L;
}
template <typename SM>
__device__ __noinline__ u32 dec_long_code(const SM &sm, int gi, u32 win, u32 entry) { return dec_long_code_inl(sm, gi, win, entry); }

// 32 bits of the stream from bit position bp, first bit in bit 31; bits past EOF read as 0 (BJ:149-150)
__device__ __forceinline__ u32 dec_load32(const u8 *__restrict__ in, u64 n, u64 bp) {
  const u64 by = bp >> 3;
  u64 v = 0;
#pragma unroll
  for (int z = 0; z < 5; z++) v = (v << 8) | (by + z < n ? (u64)in[by + z] : 0ull);
  return (u32)(v >> (8 - (u32)(bp & 7)));
}
// selector MTF (BJ:1481-1496) as maps over the 7 list positions a selector can name (3 bits each): after the moves
// of map a, then those of map b, position q holds what position a[b[q]] held before
#define DEC_PERM_ID 06543210u
__device__ __forceinline__ u32 dec_perm_front(u32 p, u32 j) {  // move position j to the front
  const u32 v = (p >> (3 * j)) & 7u, lowmask = (1u << (3 * j)) - 1u;
  return (p & ~((lowmask << 3) | 7u)) | ((p & lowmask) << 3) | v;
}
__device__ __forceinline__ u32 dec_perm_compose(u32 a, u32 b) {
  u32 c = 0;
#pragma unroll
  for (int q = 0; q < 7; q++) c |= ((a >> (3 * ((b >> (3 * q)) & 7u))) & 7u) << (3 * q);
  return c;
}

// header (BJ:1434-1520), limit/base/permute (BJ:1521-1581) and the 10-bit LUT of one candidate block, shared by the two
// parse kernels.  Returns false when the candidate is not a block to parse (end-of-stream magic, header error): `out[k]`
// is written then.
template <int PT, typename SM>
__device__ __forceinline__ bool dec_header(SM &sm, const u8 *__restrict__ in, u64 n, const u64 *__restrict__ cand, u32 k, u32 dbuf_cap, int verify,
                                           DecBlk *__restrict__ out, u8 *__restrict__ sel, u8 *__restrict__ dmap, DecBlk &res) {
  const int lane = threadIdx.x;
  const u64 bitpos = cand[k] >> 1;
  u32 kind = (u32)(cand[k] & 1);
  if (verify) {  // candidate given by the caller (decompressBlock): read the 48-bit signature here (BJ:1434-1439)
    BitRd r0;
    br_init(r0, in, n, bitpos);
    u64 h = ((u64)br_get(r0, 24) << 24) | br_get(r0, 24);
    kind = h == BZ_MAGIC_END ? 1u : h == BZ_MAGIC_BLOCK ? 0u : 2u;
  }
  res.bitpos = bitpos; res.endbit = 0; res.target_crc = 0; res.orig_ptr = 0; res.count = 0; res.err = 0; res.kind = kind; res.nsym = 0;
  // ---- header (lane 0), BJ:1434-1520 ----
  if (lane == 0) {
    BitRd r;
    int err = kind == 2 ? BZ2B200_E_NOT_BZIP_DATA : 0, ng = 0, nsel = 0, sym_total = 0;
    br_init(r, in, n, bitpos + 48);
    res.target_crc = br_get(r, 32);
    if (kind == 0) {
      if (br_get(r, 1)) err = BZ2B200_E_OBSOLETE_INPUT;
      if (!err) {
        res.orig_ptr = br_get(r, 24);
        if (res.orig_ptr > dbuf_cap) err = BZ2B200_E_DATA_ERROR;
      }
      if (!err) {
        u32 map = br_get(r, 16);
        for (int i = 0; i < 16; i++)
          if (map & (1u << (15 - i))) {
            u32 kk = br_get(r, 16);
            for (int j = 0; j < 16; j++)
              if (kk & (1u << (15 - j))) sm.sym2byte[sym_total++] = (u8)(i * 16 + j);
          }
        ng = (int)br_get(r, 3);
        if (ng < 2 || ng > 6) err = BZ2B200_E_DATA_ERROR;
      }
      if (!err) {
        nsel = (int)br_get(r, 15);
        if (nsel == 0) err = BZ2B200_E_DATA_ERROR;
      }
    }
    sm.hdr[0] = err; sm.hdr[1] = ng; sm.hdr[2] = nsel; sm.hdr[3] = sym_total; sm.hdr[4] = (int)r.overrun;
    sm.sel_end = br_tell(r);
  }
  __syncthreads();
  // ---- selectors (BJ:1481-1496), all threads: selector i is the run of 1 bits before the i-th 0 bit, then an MTF move.
  // Every thread takes a 32-bit word of the stream: zeros are counted and ranked by a CTA scan, the run length of a
  // zero is its distance to the zero before it; the moves are composed by a scan of position maps.
  if (kind == 0 && sm.hdr[0] == 0) {
    const int ng = sm.hdr[1];
    const u32 nsel = (u32)sm.hdr[2];
    const u32 wid = (u32)lane >> 5, wl = (u32)lane & 31u, nw = PT / 32;
    u64 cur = sm.sel_end;
    u64 lastz = cur - 1;  // position of the zero before the run being measured
    u32 donez = 0;
    int perr = 0;
    __syncthreads();
    while (donez < nsel && !perr) {
      const u64 bp = cur + 32ull * (u32)lane;
      const u32 zm = ~dec_load32(in, n, bp);  // bit 31-k set: the k-th bit of the word is 0
      const u32 z = (u32)__popc(zm);
      const u32 lz = z ? 32u * (u32)lane + (32u - (u32)__ffs((int)zm)) + 1u : 0u;  // offset of the word's last zero, +1 (0: none)
      u32 zin = z, lin = lz;  // inclusive sum / max scans over the CTA
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const u32 a = __shfl_up_sync(FULL_MASK, zin, d), b = __shfl_up_sync(FULL_MASK, lin, d);
        if (wl >= (u32)d) { zin += a; lin = lin > b ? lin : b; }
      }
      if (wl == 31) { sm.scr[wid] = zin; sm.scr[32 + wid] = lin; }
      if (lane == 0) sm.scr[64] = 0;
      __syncthreads();
      u32 zbase = 0, lbase = 0, ztot = 0, lmax = 0;
      for (u32 w2 = 0; w2 < nw; w2++) {
        const u32 a = sm.scr[w2], b = sm.scr[32 + w2];
        if (w2 < wid) { zbase += a; lbase = lbase > b ? lbase : b; }
        ztot += a; lmax = lmax > b ? lmax : b;
      }
      u32 idx = donez + zbase + zin - z;
      u32 lprev = __shfl_up_sync(FULL_MASK, lin, 1);
      if (wl == 0) lprev = 0;
      lprev = lprev > lbase ? lprev : lbase;
      u64 prevpos = lprev ? cur + lprev - 1 : lastz;
      u32 m = zm;
      while (m && idx < nsel) {
        const u32 k2 = (u32)__clz((int)m);
        const u64 pos = bp + k2;
        const u64 j = pos - prevpos - 1;
        if (j > (u64)ng) perr = 1; else sel[idx] = (u8)j;  // BJ:1488-1490: the bound is tested on each 1 bit, so j == ng passes
        if (idx == nsel - 1) sm.sel_end = pos + 1;
        prevpos = pos;
        idx++;
        m &= ~(0x80000000u >> k2);
      }
      if (ztot == 0) perr = 1;  // a run of 1 bits longer than the whole chunk
      if (perr) sm.scr[64] = 1;
      __syncthreads();
      perr = (int)sm.scr[64];
      donez += ztot;
      if (lmax) lastz = cur + lmax - 1;
      cur += 32ull * PT;
      __syncthreads();
    }
    if (perr) {
      if (lane == 0) sm.hdr[0] = BZ2B200_E_DATA_ERROR;
    } else {
      // MTF: thread t owns selectors [t*C, (t+1)*C)
      const u32 C = (nsel + PT - 1) / PT, i0 = (u32)lane * C, i1 = i0 + C < nsel ? i0 + C : nsel;
      u32 p = DEC_PERM_ID;
      for (u32 i = i0; i < i1; i++) p = dec_perm_front(p, sel[i]);
      u32 pin = p;  // inclusive scan of the maps (earlier moves first)
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const u32 a = __shfl_up_sync(FULL_MASK, pin, d);
        if (wl >= (u32)d) pin = dec_perm_compose(a, pin);
      }
      if (wl == 31) sm.scr[wid] = pin;
      __syncthreads();
      u32 pre = DEC_PERM_ID;
      for (u32 w2 = 0; w2 < wid; w2++) pre = dec_perm_compose(pre, sm.scr[w2]);
      u32 pex = __shfl_up_sync(FULL_MASK, pin, 1);
      if (wl == 0) pex = DEC_PERM_ID;
      p = dec_perm_compose(pre, pex);
      for (u32 i = i0; i < i1; i++) {
        const u32 j = sel[i], v = (p >> (3 * j)) & 7u;
        sel[i] = (u8)(v < (u32)ng ? v : 0u);  // the list is a zeroed Uint8Array(256) with 0..ng-1 in front (BJ:1481-1483)
        p = dec_perm_front(p, j);
      }
    }
  }
  __syncthreads();
  // ---- code lengths (lane 0), BJ:1497-1520 ----
  if (lane == 0) {
    int err = sm.hdr[0];
    const int ng = sm.hdr[1], sym_total = sm.hdr[3];
    BitRd r;
    br_init(r, in, n, sm.sel_end);
    if (sm.hdr[4] || sm.sel_end > n * 8) r.overrun = 1;
    if (kind == 0) {
      if (!err) {
        int S = sym_total + 2;
        for (int t = 0; t < ng && !err; t++) {
          int cur = (int)br_get(r, 5);
          for (int i = 0; i < S && !err; i++) {
            for (;;) {
              if (cur < 1 || cur > BZ_MAX_CODE) { err = BZ2B200_E_DATA_ERROR; break; }
              if (!br_get(r, 1)) break;
              if (!br_get(r, 1)) cur++; else cur--;
            }
            sm.lens[t][i] = (u8)cur;
          }
        }
      }
      if (!err && r.overrun) err = BZ2B200_E_UNEXPECTED_INPUT_EOF;
    }
    sm.hdr[0] = err;
    sm.bitpos_after_header = br_tell(r);
  }
  __syncthreads();
  const int err0 = sm.hdr[0], ng = sm.hdr[1], nsel = sm.hdr[2], sym_total = sm.hdr[3];
  const int S = sym_total + 2;
  if (kind != 0 || err0) {
    if (lane == 0) {
      res.err = err0;
      res.endbit = sm.bitpos_after_header;
      out[k] = res;
    }
    return false;
  }
  for (int i = lane; i < 256; i += PT) dmap[(u64)k * 256 + i] = i < sym_total ? sm.sym2byte[i] : (u8)i;
  // ---- limit / base / permute per table (BJ:1521-1581), one lane per table ----
  if (lane < ng) {
    const int t = lane;
    int minl = sm.lens[t][0], maxl = sm.lens[t][0];
    for (int i = 1; i < S; i++) {
      int L = sm.lens[t][i];
      if (L > maxl) maxl = L; else if (L < minl) minl = L;
    }
    int cnt[BZ_MAX_CODE + 2];
    for (int L = 0; L < BZ_MAX_CODE + 2; L++) { cnt[L] = 0; sm.limit[t][L] = 0; sm.base[t][L] = 0; }
    int pp = 0;
    for (int L = minl; L <= maxl; L++)
      for (int s2 = 0; s2 < S; s2++)
        if (sm.lens[t][s2] == L) sm.permute[t][pp++] = (u16)s2;
    for (int i = 0; i < S; i++) cnt[sm.lens[t][i]]++;
    pp = 0;
    int tt = 0;
    for (int L = minl; L < maxl; L++) {
      pp += cnt[L];
      sm.limit[t][L] = pp - 1;
      pp <<= 1;
      tt += cnt[L];
      sm.base[t][L + 1] = pp - tt;
    }
    sm.limit[t][maxl] = pp + cnt[maxl] - 1;
    sm.base[t][minl] = 0;
    sm.minl[t] = minl;
    sm.maxl[t] = maxl;
  }
  __syncthreads();
  // ---- LUT: replay the reference's decode walk on every 10-bit prefix ----
  for (int x = lane; x < ng * (1 << DEC_LUT_BITS); x += PT) {
    int t = x >> DEC_LUT_BITS, prefix = x & ((1 << DEC_LUT_BITS) - 1);
    u16 e = 0;
    for (int L = sm.minl[t]; L <= DEC_LUT_BITS && L <= sm.maxl[t]; L++) {
      int j = prefix >> (DEC_LUT_BITS - L);
      if (j <= sm.limit[t][L]) {
        int idx = j - sm.base[t][L];
        e = idx >= 0 && idx < BZ_MAX_SYMS ? (u16)((sm.permute[t][idx] << 5) | L) : (u16)DEC_LUT_BAD;  // out-of-range index: an error
        break;
      }
    }
    sm.lut[t][prefix] = e;
  }
  __syncthreads();
  return true;
}

// ---- K-U2/3a: header + Huffman parse (bits -> symbols).  One CTA of DEC_PT threads per candidate block. -------
// Only this part of the decoder is serial across GROUPS (the coding table changes every 50 symbols, so the position
// of a group in the bit stream is unknown until everything before it is parsed); inside a group it is parallel:
// thread b decodes the code that WOULD start at bit P+b, pointer doubling over those "next code" links finds the
// codes that really start there (the chain from offset 0), a scan ranks them, the first `left` are the group.
template <int PT>
__global__ void __launch_bounds__(PT) k_huff_parse(const u8 *__restrict__ in, u64 n, const u64 *__restrict__ cand, u32 ncand, u32 dbuf_cap, int verify,
                                                   DecBlk *__restrict__ out, u16 *__restrict__ dsym, u8 *__restrict__ dsel, u8 *__restrict__ dmap) {
  __shared__ DecSmem<PT> sm;
  const u32 k = blockIdx.x;
  if (k >= ncand) return;
  const int lane = threadIdx.x;  // thread index in the CTA (the header code below predates the CTA-wide parse)
  u16 *Sk = dsym + (u64)k * DEC_SYM_STRIDE;
  u8 *sel = dsel + (u64)k * DEC_MAX_SEL;
  DecBlk res;
  if (!dec_header<PT>(sm, in, n, cand, k, dbuf_cap, verify, out, sel, dmap, res)) return;
  const int nsel = sm.hdr[2], sym_total = sm.hdr[3];
  // ---- symbols (BJ:1597-1616): parse passes ----
  // A pass stages DEC_RING bytes of the stream (byte-swapped words) and the selectors it can need.  A step looks at the
  // PT bit offsets from P: thread b decodes the code that would start at P+b with the group's table.
  const u32 eob = (u32)sym_total + 1;
  u64 cur_bit = sm.bitpos_after_header;  // absolute bit position (uniform across the CTA)
  u32 flushed = 0;
  int err = 0, done = 0, selector = 0;
  u32 left = 0;  // symbols left in the current group
  int gi = 0;
  u32 *ring32 = reinterpret_cast<u32 *>(sm.ring);
  const u32 RBITS = DEC_RING * 8;
  for (;;) {
    const u64 ring_base_w = (cur_bit >> 5) & ~(u64)3;  // 16-byte aligned word index
    for (u32 q = lane; q < DEC_RING / 16; q += PT) {
      u64 src = (ring_base_w + (u64)q * 4) * 4;
      u32 w[4] = {0, 0, 0, 0};
      if (src + 16 <= n) {
        uint4 v = *reinterpret_cast<const uint4 *>(in + src);
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
      } else {
        for (int z = 0; z < 16; z++) if (src + z < n) w[z >> 2] |= (u32)in[src + z] << (8 * (z & 3));  // bits past EOF read as 0
      }
      for (int z = 0; z < 4; z++) ring32[q * 4 + z] = __byte_perm(w[z], 0, 0x0123);
    }
    const int sel0 = selector;  // selectors sel0 .. sel0+255 are staged (a pass of 32768 bits holds fewer groups than that)
    for (int q = lane; q < 256; q += PT) sm.selbuf[q] = sel0 + q < nsel ? sel[sel0 + q] : 0;
    __syncthreads();
    u32 P = (u32)(cur_bit - ring_base_w * 32);  // bit offset inside the ring
    u32 staged = 0;
    while (!done && !err && staged + BZ_GROUP <= DEC_SYM_STAGE && P + PT + 64 <= RBITS && selector - sel0 < 255) {
      if (left == 0) {
        if (selector >= nsel) { err = BZ2B200_E_DATA_ERROR; break; }  // BJ:1601
        if (flushed + staged + BZ_GROUP >= DEC_SYM_STRIDE) { err = BZ2B200_E_DATA_ERROR; break; }  // more symbols than any valid block
        gi = sm.selbuf[selector - sel0];
        selector++;
        left = BZ_GROUP;
      }
      const u32 bp = P + (u32)lane;
      const u32 win = __funnelshift_l(ring32[(bp >> 5) + 1], ring32[bp >> 5], bp & 31u);  // 32 bits from bit P+lane
      u32 e = sm.lut[gi][win >> (32 - DEC_LUT_BITS)];  // (symbol << 5) | length, 0 = longer than the LUT
      if (e == 0 || e == DEC_LUT_BAD) e = dec_long_code_inl(sm, gi, win, e);  // sym 0x8000 = invalid code
      const u32 sym = e >> 5, nxt = (u32)lane + (e & 31u);
      sm.J[0][lane] = (u16)nxt;
      sm.SY[lane] = (u16)sym;
      if (lane == 0) { sm.first_eob = 0xffffffffu; sm.first_bad = 0xffffffffu; sm.first_eof = 0xffffffffu; sm.adv = 0; }
      __syncthreads();
#pragma unroll
      for (int q = 1; q < DEC_LEVELS; q++) {  // J[q] = J[q-1] o J[q-1]
        u32 v = sm.J[q - 1][lane];
        sm.J[q][lane] = v < PT ? sm.J[q - 1][v] : (u16)0xffff;
        __syncthreads();
      }
      // thread r < 64 finds the offset of the r-th code of the chain by composing the jumps of r's binary digits
      // (six dependent shared-memory reads, no barrier): it IS rank r
      if (lane < 64) {
        u32 pos = 0;
#pragma unroll
        for (int q = 0; q < DEC_LEVELS; q++)
          if (((u32)lane >> q) & 1u) pos = pos < PT ? sm.J[q][pos] : 0xffffu;
        const bool have = pos < PT;                       // the r-th code starts inside the step
        const u32 sy = have ? sm.SY[pos] : 0u;
        sm.csym[lane] = (u16)sy;
        sm.cend[lane] = have ? sm.J[0][pos] : (u16)0xffff;  // the bit after code r = where code r+1 starts
        // the first code whose bits reach past the end of the input is "unexpected EOF" (the oracle checks per code;
        // an invalid code read as many bits as the reference's walk did before giving up)
        bool over = false;
        if (have) {
          u32 bits = sm.J[0][pos] - pos;
          if (sy & 0x8000u) {
            const u32 bp2 = P + pos;
            const u32 w2 = __funnelshift_l(ring32[(bp2 >> 5) + 1], ring32[bp2 >> 5], bp2 & 31u);
            bits = dec_long_code_inl(sm, gi, w2, sm.lut[gi][w2 >> (32 - DEC_LUT_BITS)]) >> 21;
          }
          over = ring_base_w * 32 + P + pos + bits > n * 8;
        }
        const u32 hb = __ballot_sync(FULL_MASK, have), ob = __ballot_sync(FULL_MASK, over),
                  eb = __ballot_sync(FULL_MASK, have && !over && (sy & 0x7fffu) == eob), bb = __ballot_sync(FULL_MASK, have && !over && (sy & 0x8000u));
        if ((lane & 31) == 0) {  // `have` is monotone in r: the counts of the two warps add up
          atomicAdd(&sm.adv, (u32)__popc(hb));
          if (eb) atomicMin(&sm.first_eob, (u32)(lane + __ffs((int)eb) - 1));
          if (bb) atomicMin(&sm.first_bad, (u32)(lane + __ffs((int)bb) - 1));
          if (ob) atomicMin(&sm.first_eof, (u32)(lane + __ffs((int)ob) - 1));
        }
      }
      __syncthreads();
      const u32 total = sm.adv;  // codes of the chain that start inside the step (at most 64 are looked at)
      u32 take = left < total ? left : total;
      bool fin = false;
      if (sm.first_eob < take) { take = sm.first_eob + 1; fin = true; }
      if (sm.first_bad < take || sm.first_eof < take) {
        err = sm.first_eof < sm.first_bad ? BZ2B200_E_UNEXPECTED_INPUT_EOF : BZ2B200_E_DATA_ERROR;
        take = sm.first_eof < sm.first_bad ? sm.first_eof : sm.first_bad;  // the codes before it are kept (k_sym_offsets)
        if ((u32)lane < take) sm.stage[staged + lane] = (u16)(sm.csym[lane] & 0x7fffu);
        staged += take;
        break;
      }
      if ((u32)lane < take) sm.stage[staged + lane] = (u16)(sm.csym[lane] & 0x7fffu);
      const u32 advance = sm.cend[take - 1];
      __syncthreads();  // csym / cend / adv / first_* are rewritten in the next step
      staged += take;
      left -= take;
      P += advance;
      if (fin) done = 1;
    }
    cur_bit = ring_base_w * 32 + P;
    if (!err && cur_bit > n * 8) err = BZ2B200_E_UNEXPECTED_INPUT_EOF;  // reference: spins on zero bits (D3)
    __syncthreads();
    for (u32 q = lane; q < staged; q += PT) Sk[flushed + q] = sm.stage[q];
    flushed += staged;
    __syncthreads();
    if (err || done) break;
  }
  if (lane == 0) {
    res.err = err;
    res.count = err ? flushed : 0;  // with err the symbols before it; k_sym_offsets fills in the rest
    res.nsym = err ? 0 : flushed;
    res.endbit = cur_bit;
    out[k] = res;
  }
}

// ---- K-U2/3a, few blocks: the same parse with the serial part cut to three dependent reads per group -----------
// k_huff_parse above spends ~9 CTA barriers per group of 50 symbols; with fewer blocks than SMs that latency is the
// whole decode.  Here a window of W bit offsets is decoded speculatively under EVERY table the next groups use (the
// selectors are known up front): J_t[0][b] = b + length of the code that would start at b under table t, four
// pointer-doubling levels give J_t[k][b] = offset after 2^k codes, and then
//   * one thread walks the groups: the next group starts 16 + 16 + 16 + 2 codes on (four dependent reads);
//   * thread (q, r) composes the jumps of r's binary digits from group q's start and IS the r-th symbol of it.
// A window starts at a group start; a group is at most 50 * 20 = 1000 bits, so every window makes progress.  The price
// is work (up to 6 tables over every offset), so the host picks this kernel only when the blocks cannot fill the GPU.
#define DECW_PT 1024         // threads
#define DECW_WIN 2048        // widest window
#define DECW_ITEMS 6         // (table, offset) items per thread: 3 tables x 2048 offsets or 6 tables x 1024 offsets
#define DECW_LEVELS 5        // J1, J2, J4, J8, J16
#define DECW_JCAP (DECW_ITEMS * DECW_PT * DECW_LEVELS)
#define DECW_KMAX 16         // groups taken per window at most (16 * 50 symbols <= DECW_PT extraction threads)

struct DecWinSmem {
  int limit[BZ_MAX_GROUPS][BZ_MAX_CODE + 2];
  int base[BZ_MAX_GROUPS][BZ_MAX_CODE + 2];
  u16 permute[BZ_MAX_GROUPS][BZ_MAX_SYMS + 2];
  u16 lut[BZ_MAX_GROUPS][1 << DEC_LUT_BITS];
  u8 lens[BZ_MAX_GROUPS][BZ_MAX_SYMS + 2];
  int minl[BZ_MAX_GROUPS], maxl[BZ_MAX_GROUPS];
  u8 mtf[256];
  u8 sym2byte[256];
  __align__(16) u8 ring[DEC_RING + 16];
  int hdr[8];  // err, ng, nsel, sym_total, overrun so far
  u32 scr[72];  // CTA scans of the header
  u64 sel_end;  // first bit after the selectors
  u64 bitpos_after_header;
  // J[(s * 5 + k) * W + b]: offset reached from b after 2^k codes of table slot s; 0xffff when one of those codes would
  // start outside the window (a value in [W, W+20) is a valid end that cannot be continued)
  u16 J[DECW_JCAP];
  u8 selbuf[256];  // selectors of the pass
  u16 starts[DECW_KMAX];  // offset inside the window where the q-th group of the window starts
  u32 ngd, wend;          // groups that end inside the window, offset where the next one starts
  u32 first_eob, first_bad, first_eof, eob_end;
};

// plan of the window that starts at group `selector`, computed by every warp for itself (lane q looks at selector q):
// up to 3 distinct tables among the next groups -> 2048 offsets and as many groups as keep to those tables (<= 16);
// a 4th table within the next 6 groups -> 1024 offsets and all tables of the next 8 groups.  Table t sits in slot
// popc(mask below bit t).  Returns the table mask; kq = groups the walk may take.
__device__ __forceinline__ u32 decw_plan(const DecWinSmem &sm, int selector, int sel0, int nsel, u32 &W, u32 &kq) {
  const u32 wl = threadIdx.x & 31u;
  const bool valid = wl < DECW_KMAX && selector + (int)wl < nsel;
  u32 m = valid ? 1u << sm.selbuf[selector - sel0 + (int)(wl < DECW_KMAX ? wl : 0u)] : 0u;
#pragma unroll
  for (int d = 1; d < DECW_KMAX; d <<= 1) {
    const u32 o = __shfl_up_sync(FULL_MASK, m, d);
    if (wl >= (u32)d) m |= o;
  }
  const u32 nvalid = (u32)__popc(__ballot_sync(FULL_MASK, valid));
  kq = (u32)__popc(__ballot_sync(FULL_MASK, valid && __popc(m) <= 3));  // the count of tables grows with q
  W = DECW_WIN;
  if (kq < 6 && kq < nvalid) {
    W = DECW_WIN / 2;
    kq = nvalid < 8 ? nvalid : 8;
  }
  return __shfl_sync(FULL_MASK, m, (int)(kq ? kq - 1 : 0));
}

__global__ void __launch_bounds__(DECW_PT) k_huff_parse_win(const u8 *__restrict__ in, u64 n, const u64 *__restrict__ cand, u32 ncand, u32 dbuf_cap,
                                                            int verify, DecBlk *__restrict__ out, u16 *__restrict__ dsym, u8 *__restrict__ dsel,
                                                            u8 *__restrict__ dmap) {
  DYN_SMEM(DecWinSmem, smp);
  DecWinSmem &sm = *smp;
  const int PT = DECW_PT;
  const u32 k = blockIdx.x;
  if (k >= ncand) return;
  const int lane = threadIdx.x;
  u16 *Sk = dsym + (u64)k * DEC_SYM_STRIDE;
  u8 *sel = dsel + (u64)k * DEC_MAX_SEL;
  DecBlk res;
  if (!dec_header<PT>(sm, in, n, cand, k, dbuf_cap, verify, out, sel, dmap, res)) return;
  const int nsel = sm.hdr[2], sym_total = sm.hdr[3];
  const u32 eob = (u32)sym_total + 1;
  u64 cur_bit = sm.bitpos_after_header;  // absolute bit position (uniform across the CTA)
  u32 flushed = 0;
  int err = 0, done = 0, selector = 0;
  u32 *ring32 = reinterpret_cast<u32 *>(sm.ring);
  const u32 RBITS = DEC_RING * 8;
  for (;;) {
    const u64 ring_base_w = (cur_bit >> 5) & ~(u64)3;  // 16-byte aligned word index
    for (u32 q = lane; q < DEC_RING / 16; q += PT) {
      u64 src = (ring_base_w + (u64)q * 4) * 4;
      u32 w[4] = {0, 0, 0, 0};
      if (src + 16 <= n) {
        uint4 v = *reinterpret_cast<const uint4 *>(in + src);
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
      } else {
        for (int z = 0; z < 16; z++) if (src + z < n) w[z >> 2] |= (u32)in[src + z] << (8 * (z & 3));  // bits past EOF read as 0
      }
      for (int z = 0; z < 4; z++) ring32[q * 4 + z] = __byte_perm(w[z], 0, 0x0123);
    }
    const int sel0 = selector;  // selectors sel0 .. sel0+255 are staged
    for (int q = lane; q < 256; q += PT) sm.selbuf[q] = sel0 + q < nsel ? sel[sel0 + q] : 0;
    __syncthreads();
    u32 P = (u32)(cur_bit - ring_base_w * 32);  // bit offset inside the ring
    while (P + DECW_WIN + 64 <= RBITS && selector - sel0 + DECW_KMAX <= 256) {
      if (selector >= nsel) { err = BZ2B200_E_DATA_ERROR; break; }  // BJ:1601
      if (flushed + BZ_GROUP >= DEC_SYM_STRIDE) { err = BZ2B200_E_DATA_ERROR; break; }  // more symbols than any valid block
      u32 W, kq;
      const u32 tmask = decw_plan(sm, selector, sel0, nsel, W, kq);
      const u32 ntabs = (u32)__popc(tmask);
      u32 tabs = 0;  // nibble s: the table in slot s
      for (u32 t = 0, c = 0; t < BZ_MAX_GROUPS; t++)
        if ((tmask >> t) & 1u) { tabs |= t << (4 * c); c++; }
      const u32 opl = W / DECW_PT, nitems = ntabs * opl;  // (table slot, offset) items of this thread, all in flight together
      u64 slots = 0;  // warp 0: nibble q = table slot of the window's q-th group (for the walk below)
      if (lane < 32) {
        const u32 t = ((u32)lane < DECW_KMAX && selector + lane < nsel) ? sm.selbuf[selector - sel0 + lane] : 0u;
        const u32 sl = (u32)__popc(tmask & ((1u << t) - 1u));
        u32 lo = lane < 8 ? sl << (4 * lane) : 0u, hi = (lane >= 8 && lane < 16) ? sl << (4 * (lane - 8)) : 0u;
#pragma unroll
        for (int d = 16; d; d >>= 1) {
          lo |= __shfl_xor_sync(FULL_MASK, lo, d);
          hi |= __shfl_xor_sync(FULL_MASK, hi, d);
        }
        slots = ((u64)hi << 32) | lo;
      }
      // level 0: the code that would start at every offset, under every table of the window
      u32 nx[DECW_ITEMS];
      u16 *jr[DECW_ITEMS], *jw[DECW_ITEMS];  // J[slot][level][0] (gathers) and J[slot][level][own offset] (stores)
      {
        u32 wn[DECW_ITEMS], e[DECW_ITEMS];
        int tb[DECW_ITEMS];
#pragma unroll
        for (int i = 0; i < DECW_ITEMS; i++) {
          if ((u32)i >= nitems) break;
          const u32 s2 = (u32)i >> (opl - 1u), bo = (u32)lane + (((u32)i & (opl - 1u)) << 10);
          jr[i] = sm.J + s2 * DECW_LEVELS * W;
          jw[i] = jr[i] + bo;
          nx[i] = bo;
          tb[i] = (int)((tabs >> (4 * s2)) & 15u);
          const u32 bp = P + bo;
          wn[i] = __funnelshift_l(ring32[(bp >> 5) + 1], ring32[bp >> 5], bp & 31u);  // 32 bits from bit P+b
        }
#pragma unroll
        for (int i = 0; i < DECW_ITEMS; i++) {
          if ((u32)i >= nitems) break;
          e[i] = sm.lut[tb[i]][wn[i] >> (32 - DEC_LUT_BITS)];  // (symbol << 5) | length, 0 = longer than the LUT
        }
#pragma unroll
        for (int i = 0; i < DECW_ITEMS; i++) {
          if ((u32)i >= nitems) break;
          if (e[i] == 0 || e[i] == DEC_LUT_BAD) e[i] = dec_long_code(sm, tb[i], wn[i], e[i]);
          nx[i] += e[i] & 31u;
          *jw[i] = (u16)nx[i];
        }
      }
      __syncthreads();
      for (u32 q = 1; q < DECW_LEVELS; q++) {  // J[q] = J[q-1] o J[q-1]; a thread's own J[q-1] values stay in registers
#pragma unroll
        for (int i = 0; i < DECW_ITEMS; i++) {
          if ((u32)i >= nitems) break;
          const u32 v = jr[i][nx[i] < W ? nx[i] : 0u];
          nx[i] = nx[i] < W ? v : 0xffffu;
        }
#pragma unroll
        for (int i = 0; i < DECW_ITEMS; i++) {
          if ((u32)i >= nitems) break;
          jr[i] += W;
          jw[i] += W;
          *jw[i] = (u16)nx[i];
        }
        __syncthreads();
      }
      // the walk over the groups of the window (one thread): 50 = 16 + 16 + 16 + 2
      if (lane == 0) {
        u32 pos = 0, g = 0;
        u32 lim = (DEC_SYM_STRIDE - 1 - flushed) / BZ_GROUP;  // groups g with flushed + (g + 1) * 50 < DEC_SYM_STRIDE
        if (lim > kq) lim = kq;
        // Four dependent reads per group and nothing else on the chain: the table slot of every group was packed into
        // `slots` before the levels (a selector read here would sit between two groups' reads), the indices are clamped
        // into the window instead of tested (a clamped read returns some valid entry that is never used), and the tests
        // come behind the last read.
        while (g < lim && pos < W) {
          const u16 *Jb = sm.J + ((u32)(slots >> (4 * g)) & 15u) * DECW_LEVELS * W;
          const u16 *J16 = Jb + 4 * W;
          const u32 a = J16[pos];
          const u32 b2 = J16[min(a, W - 1u)];
          const u32 c2 = J16[min(b2, W - 1u)];
          const u32 d2 = Jb[W + min(c2, W - 1u)];
          if ((a >= W) | (b2 >= W) | (c2 >= W) | (d2 == 0xffffu)) break;
          sm.starts[g] = (u16)pos;
          pos = d2;
          g++;
        }
        sm.ngd = g; sm.wend = pos;
        sm.first_eob = 0xffffffffu; sm.first_bad = 0xffffffffu; sm.first_eof = 0xffffffffu;
      }
      __syncthreads();
      const u32 ngd = sm.ngd, total = ngd * BZ_GROUP;
      u32 my_end = 0;
      if ((u32)lane < total) {  // thread (q, r): the r-th code of the q-th group
        const u32 q = (u32)lane / BZ_GROUP, r = (u32)lane % BZ_GROUP;
        const int t = sm.selbuf[selector - sel0 + (int)q];
        const u32 s2 = (u32)__popc(tmask & ((1u << t) - 1u));
        const u16 *Jb = sm.J + (s2 * DECW_LEVELS) * W;
        u32 pos = sm.starts[q];
        for (u32 z = r >> 4; z; z--) pos = Jb[4 * W + pos];
#pragma unroll
        for (int z = 0; z < 4; z++)
          if ((r >> z) & 1u) pos = Jb[z * W + pos];
        const u32 bp = P + pos;
        const u32 wn = __funnelshift_l(ring32[(bp >> 5) + 1], ring32[bp >> 5], bp & 31u);
        u32 e = sm.lut[t][wn >> (32 - DEC_LUT_BITS)];
        if (e == 0 || e == DEC_LUT_BAD) e = dec_long_code(sm, t, wn, e);
        const u32 sy = e >> 5;
        my_end = pos + (e & 31u);
        Sk[flushed + lane] = (u16)(sy & 0x7fffu);
        // the first code whose bits reach past the end of the input is "unexpected EOF" (the oracle checks per code)
        if (ring_base_w * 32 + P + pos + ((sy & 0x8000u) ? e >> 21 : e & 31u) > n * 8) atomicMin(&sm.first_eof, (u32)lane);
        else if (sy & 0x8000u) atomicMin(&sm.first_bad, (u32)lane);
        else if (sy == eob) atomicMin(&sm.first_eob, (u32)lane);
      }
      __syncthreads();
      u32 take = total, advance = sm.wend;
      const u32 fe = sm.first_eob, fb = sm.first_bad, fo = sm.first_eof;
      if (fe < take) {  // the block ends here: the bit after the end-of-block code
        take = fe + 1;
        if ((u32)lane == fe) sm.eob_end = my_end;
        __syncthreads();
        advance = sm.eob_end;
        done = 1;
      }
      if (fb < take || fo < take) {
        err = fo < fb ? BZ2B200_E_UNEXPECTED_INPUT_EOF : BZ2B200_E_DATA_ERROR;
        flushed += fo < fb ? fo : fb;  // the codes before it are kept (k_sym_offsets)
        break;
      }
      flushed += take;
      P += advance;
      selector += (int)ngd;
      if (done) break;
    }
    cur_bit = ring_base_w * 32 + P;
    if (!err && cur_bit > n * 8) err = BZ2B200_E_UNEXPECTED_INPUT_EOF;  // reference: spins on zero bits (D3)
    __syncthreads();
    if (err || done) break;
  }
  if (lane == 0) {
    res.err = err;
    res.count = err ? flushed : 0;  // with err the symbols before it; k_sym_offsets fills in the rest
    res.nsym = err ? 0 : flushed;
    res.endbit = cur_bit;
    out[k] = res;
  }
}

// ---- K-U3b: RLE2^-1 offsets.  One CTA per candidate: the k-th RUNA/RUNB of a run stands for (sym+1) << k copies of
// the current list front (BJ:1621-1652), a literal for one byte; exclusive scan -> position of every symbol's output.
// A block whose parse failed gets the size the reference's checks saw before the failing code (count, see below): the
// reference checks the size at every symbol, so a block that outgrew its stream's block size first is a Data error.
__global__ void __launch_bounds__(1024) k_sym_offsets(DecBlk *__restrict__ blks, const u16 *__restrict__ dsym, u32 *__restrict__ doff, u32 dbuf_cap) {
  __shared__ int wsi[33];
  __shared__ u32 ws[33];
  const u32 k = blockIdx.x;
  const bool parsed = !blks[k].err;  // else: the m symbols before the parse error (the last one is no end-of-block)
  const u32 m = parsed ? blks[k].nsym : blks[k].count;
  if (blks[k].kind != 0 || m == 0) return;
  const u16 *Sk = dsym + (u64)k * DEC_SYM_STRIDE;
  u32 *Ok = doff + (u64)k * DEC_SYM_STRIDE;
  int carry_lit = -1;  // last non-run symbol so far
  u32 carry = 0;
  const u32 over = dbuf_cap + 1;
  for (u32 base = 0; base < m; base += 1024 * 4) {
    u32 i0 = base + threadIdx.x * 4;
    u32 sy[4];
    int my_lit = -1;
    for (int q = 0; q < 4; q++) { sy[q] = i0 + q < m ? Sk[i0 + q] : 2u; if (i0 + q < m && sy[q] >= 2) my_lit = (int)(i0 + q); }
    int tot_l;
    int lit = block_excl_max<int>(my_lit, -1, tot_l, wsi);
    if (carry_lit > lit) lit = carry_lit;
    u32 cp[4], mine = 0;
    {
      int cur = lit;
      for (int q = 0; q < 4; q++) {
        u32 i = i0 + q;
        cp[q] = 0;
        if (i >= m) continue;
        if (sy[q] >= 2) { cur = (int)i; cp[q] = i + 1 == m ? 0u : 1u; }  // the last symbol is end-of-block
        else {  // a run digit is clamped to dbuf_cap + 1 ("too large"), so no sum below can wrap: 4096 x 900 001 < 2^32
          u32 kk = i - (u32)(cur + 1), v = kk < 21 ? (sy[q] + 1) << kk : over;
          cp[q] = v < over ? v : over;
        }
        mine += cp[q];
      }
    }
    u32 tot;
    u32 o = carry + block_excl_sum<u32>(mine, tot, ws);
    for (int q = 0; q < 4; q++) if (i0 + q < m) { Ok[i0 + q] = o; o += cp[q]; }
    carry += tot;
    if (carry > over) carry = over;  // saturate at once (only "too large" matters): carry + a chunk's total stays below 2^32
    if (tot_l > carry_lit) carry_lit = tot_l;
  }
  if (!parsed) __syncthreads();  // Ok[] of every thread is read below
  if (threadIdx.x == 0) {
    Ok[m] = carry;
    if (!parsed) {
      // the sizes the reference checks before the failing code: t_run after every run digit (BJ:1647), the bytes before
      // every literal + 1 (BJ:1663); the largest is that of the last literal or of the run after it
      const u32 i0 = (u32)(carry_lit + 1);
      u32 lit = i0 == 0 ? 0u : i0 == m ? Ok[m - 1] + 1 : Ok[i0];  // (a last literal was counted as end-of-block above)
      lit = lit < over ? lit : over;
      u32 run = 0;
      for (u32 i = i0; i < m && run < over; i++) {  // at most 21 digits: (sym+1) << 20 > any block size
        const u32 kk = i - i0, v = kk < 21 ? ((u32)Sk[i] + 1) << kk : over;
        run = run + v < over ? run + v : over;
      }
      blks[k].count = lit > run ? lit : run;
      return;
    }
    // BJ:1647,1663 (dbuf overflow) and BJ:1677 (origPtr past the data) -> DATA_ERROR
    if (carry > dbuf_cap || blks[k].orig_ptr >= carry) { blks[k].err = BZ2B200_E_DATA_ERROR; blks[k].nsym = 0; carry = 0; }
    blks[k].count = carry;
  }
}

// ---- K-U3c: MTF^-1 in parallel.  The list is striped over the warp like in k_mtf_ranks. ----------------
// rank j < 32: one shuffle with a per-lane source (lane 0 takes list[j], lanes 1..j their left neighbour)
__device__ __forceinline__ void imtf_hot(u32 &hot, u32 j, int lane) {
  const int src = lane == 0 ? (int)j : lane - (lane <= (int)j ? 1 : 0);
  hot = __shfl_sync(FULL_MASK, hot, src);
}
// rank j >= 32 (rare): the target comes from a cold row, every row up to it shifts by one
__device__ __noinline__ void imtf_cold(u32 &hot, u64 &cold, u32 j, int lane) {
  int row = (int)(j >> 5), l = (int)(j & 31);
  u32 target = __shfl_sync(FULL_MASK, (u32)(cold >> (8 * (row - 1))) & 0xffu, l);
  u32 carry = target;
  {
    u32 last = __shfl_sync(FULL_MASK, hot, 31);
    u32 up = __shfl_up_sync(FULL_MASK, hot, 1);
    hot = lane == 0 ? carry : up;
    carry = last;
  }
  for (int r = 1; r <= row; r++) {
    u32 cur = (u32)(cold >> (8 * (r - 1))) & 0xffu;
    u32 last = __shfl_sync(FULL_MASK, cur, 31);
    u32 up = __shfl_up_sync(FULL_MASK, cur, 1);
    u32 nv = lane == 0 ? carry : up;
    if (r < row || lane <= l) cold = (cold & ~(0xffULL << (8 * (r - 1)))) | ((u64)nv << (8 * (r - 1)));
    carry = last;
  }
}
// one symbol: ranks 1..255 arrive as symbols 2..256 (0/1 = RUNA/RUNB, > 256 = end-of-block: no move)
__device__ __forceinline__ void imtf_sym(u32 &hot, u64 &cold, u32 sy, int lane) {
  const u32 j = sy - 1;
  if (j - 1 < 255u) {
    if (j < 32) imtf_hot(hot, j, lane); else imtf_cold(hot, cold, j, lane);
  }
}
// per candidate: the list at the start of every segment (in place over segperm)
__global__ void __launch_bounds__(32) k_imtf_scan(const DecBlk *__restrict__ blks, const u8 *__restrict__ dmap, u8 *__restrict__ segperm) {
  __shared__ u8 cur[256];
  const u32 k = blockIdx.x;
  const u32 m = blks[k].nsym;
  if (blks[k].kind != 0 || blks[k].err || m == 0) return;
  const int lane = threadIdx.x;
  for (int j = lane; j < 256; j += 32) cur[j] = dmap[(u64)k * 256 + j];
  __syncwarp();
  const u32 nseg = (m + IMTF_SEG - 1) / IMTF_SEG;
  for (u32 s2 = 0; s2 < nseg; s2++) {
    u8 *P = segperm + ((u64)k * (DEC_SYM_STRIDE / IMTF_SEG + 1) + s2) * 256;
    u8 nxt[8], old[8];
    for (int r = 0; r < 8; r++) { old[r] = cur[32 * r + lane]; nxt[r] = cur[P[32 * r + lane]]; }
    __syncwarp();
    for (int r = 0; r < 8; r++) { P[32 * r + lane] = old[r]; cur[32 * r + lane] = nxt[r]; }
    __syncwarp();
  }
}
// pass I (grid (segs/8, ncand), one warp per segment of IMTF_SEG symbols): the MTF of the segment run ONCE, from the
// identity list: what it emits are list POSITIONS at the segment start (written where the L bytes will be), what is left
// at the end is the permutation of positions the segment causes.  k_imtf_scan turns the permutations into the list at
// every segment start, k_imtf_map turns positions into bytes (a 256-byte table per segment) -- instead of one MTF pass
// for the permutations and a second one for the bytes.
__global__ void __launch_bounds__(256) k_imtf_index(const DecBlk *__restrict__ blks, const u16 *__restrict__ dsym, const u32 *__restrict__ doff,
                                                    u8 *__restrict__ segperm, u8 *__restrict__ dL, i64 l_stride) {
  const u32 k = blockIdx.y;
  const u32 m = blks[k].nsym;
  const int lane = lane_id();
  const u32 seg = blockIdx.x * 8 + warp_id();
  const u32 b0 = seg * IMTF_SEG;
  if (blks[k].kind != 0 || blks[k].err || b0 >= m) return;
  const u16 *Sk = dsym + (u64)k * DEC_SYM_STRIDE + b0;
  const u32 *Ok = doff + (u64)k * DEC_SYM_STRIDE + b0;
  u8 *Lk = dL + (i64)k * l_stride;
  u32 hot = (u32)lane;
  u64 cold = 0;
  for (int r = 7; r >= 1; r--) cold = (cold << 8) | (u64)(32 * r + lane);
  u32 lim = m - b0 < IMTF_SEG ? m - b0 : IMTF_SEG;
  for (u32 c0 = 0; c0 < lim; c0 += 32) {
    u32 mysym = c0 + lane < lim ? Sk[c0 + lane] : 0u;
    u32 myoff = c0 + lane <= lim ? Ok[c0 + lane] : 0u;   // Ok[m] exists: one entry past the last symbol
    u32 nxoff = c0 + lane + 1 <= lim ? Ok[c0 + lane + 1] : myoff;
    u32 mylen = c0 + lane < lim ? nxoff - myoff : 0u;
    // Only LITERALS (symbols 2..256) move the list; RUNA/RUNB digits and end-of-block leave it alone and only repeat the
    // byte at its front.  So the serial chain steps over the literals of the chunk alone (the source profile of the
    // step-every-symbol version had 80 % issue activity at 37 warp instructions per symbol), every lane remembers the
    // front after the last literal at or before it, and the bytes of the run digits are written afterwards.
    u32 front = __shfl_sync(FULL_MASK, hot, 0);  // the front the chunk starts with
    u32 lits = __ballot_sync(FULL_MASK, mysym - 2u < 255u);
    while (lits) {
      const int t = __ffs((int)lits) - 1;
      lits &= lits - 1;
      const u32 j = __shfl_sync(FULL_MASK, mysym, t) - 1;  // rank 1..255
      if (j < 32) imtf_hot(hot, j, lane); else imtf_cold(hot, cold, j, lane);
      const u32 f = __shfl_sync(FULL_MASK, hot, 0);
      if (lane >= t) front = f;
    }
    const u32 out_byte = front;
    u32 runs = __ballot_sync(FULL_MASK, mylen > 1);  // RUNA/RUNB digits that stand for several bytes: written by the whole warp
    while (runs) {
      const int t = __ffs((int)runs) - 1;
      runs &= runs - 1;
      const u32 len = __shfl_sync(FULL_MASK, mylen, t), o = __shfl_sync(FULL_MASK, myoff, t), byte = __shfl_sync(FULL_MASK, front, t);
      for (u32 q = lane; q < len; q += 32) Lk[o + q] = (u8)byte;
    }
    if (mylen == 1) Lk[myoff] = (u8)out_byte;
  }
  u8 *P = segperm + ((u64)k * (DEC_SYM_STRIDE / IMTF_SEG + 1) + seg) * 256;
  P[lane] = (u8)hot;
  for (int r = 1; r < 8; r++) P[32 * r + lane] = (u8)(cold >> (8 * (r - 1)));
}
// pass M (grid (segs, ncand)): list positions -> bytes through the list at the segment start
__global__ void __launch_bounds__(256) k_imtf_map(const DecBlk *__restrict__ blks, const u32 *__restrict__ doff, const u8 *__restrict__ segperm,
                                                  u8 *__restrict__ dL, i64 l_stride) {
  __shared__ u8 list[256];
  const u32 k = blockIdx.y, seg = blockIdx.x;
  const u32 m = blks[k].nsym, b0 = seg * IMTF_SEG;
  if (blks[k].kind != 0 || blks[k].err || b0 >= m) return;
  list[threadIdx.x] = segperm[((u64)k * (DEC_SYM_STRIDE / IMTF_SEG + 1) + seg) * 256 + threadIdx.x];
  __syncthreads();
  const u32 *Ok = doff + (u64)k * DEC_SYM_STRIDE;
  const u32 e = b0 + IMTF_SEG < m ? b0 + IMTF_SEG : m;
  u8 *Lk = dL + (i64)k * l_stride;
  for (u32 o = Ok[b0] + threadIdx.x, o1 = Ok[e]; o < o1; o += 256) Lk[o] = list[Lk[o]];
}

// ---- K-U4a helpers ----------------------------------------------------------------------------
__global__ void k_dec_seg_init(const DecBlk *__restrict__ blks, const u32 *__restrict__ order, int nb, u32 *__restrict__ seg_cnt) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < nb) seg_cnt[p] = blks[order[p]].count;
}
__global__ void __launch_bounds__(SEG_THREADS) k_dec_keys(const u8 *__restrict__ dL, i64 l_stride, const u32 *__restrict__ order,
                                                          const u32 *__restrict__ seg_cnt, const u32 *__restrict__ seg_tile0,
                                                          const u32 *__restrict__ tile_blk, u64 *__restrict__ keys) {
  u32 tile = blockIdx.x, p = tile_blk[tile];
  u32 cnt = seg_cnt[p], l0 = (tile - seg_tile0[p]) * SORT_TILE;
  const u8 *Lk = dL + (i64)order[p] * l_stride;
  u64 g0 = (u64)tile * SORT_TILE;
  for (int e = 0; e < SEG_E; e++) {
    u32 lj = l0 + e * SEG_THREADS + threadIdx.x;
    if (lj < cnt) keys[g0 + (lj - l0)] = ((u64)Lk[lj] << 20) | lj;
  }
}

// sorted keys -> T vector, packed like the reference's dbuf (BJ:1686-1690): (position of the slot's byte in the L
// column << 8) | the L byte AT this slot, so a hop of the walk is one random read instead of two
__global__ void __launch_bounds__(SEG_THREADS) k_dec_extract(const u64 *__restrict__ keys, const u8 *__restrict__ dL, i64 l_stride,
                                                             const u32 *__restrict__ order, const u32 *__restrict__ seg_cnt,
                                                             const u32 *__restrict__ seg_tile0, const u32 *__restrict__ tile_blk, u32 *__restrict__ tt) {
  u32 tile = blockIdx.x, p = tile_blk[tile];
  u32 cnt = seg_cnt[p], l0 = (tile - seg_tile0[p]) * SORT_TILE;
  const u8 *Lk = dL + (i64)order[p] * l_stride;
  u64 g0 = (u64)tile * SORT_TILE;
  for (int e = 0; e < SEG_E; e++) {
    u32 lj = l0 + e * SEG_THREADS + threadIdx.x;
    if (lj < cnt) tt[g0 + (lj - l0)] = ((u32)(keys[g0 + (lj - l0)] & 0xFFFFFu) << 8) | Lk[lj];
  }
}

// ---- K-U4b: list ranking ----------------------------------------------------------------------
// Splitters of block p: slots 0, S, 2S, ... plus one extra for the start slot pos0 = tt[origPtr].
// spl arrays are laid out per block at offset spl0[p]; W_p = ceil(n/S) + 1.
__device__ __forceinline__ bool ibwt_is_spl(u32 j, u32 pos0, u32 ibwt_s) { return (j & (IBWT_S - 1)) == 0 || j == pos0; }
__device__ __forceinline__ u32 ibwt_spl_index(u32 j, u32 pos0, u32 W, u32 ibwt_s) { return j == pos0 ? W - 1 : j / IBWT_S; }

__global__ void __launch_bounds__(256) k_ibwt_walk1(const u32 *__restrict__ tt, const DecBlk *__restrict__ blks, const u32 *__restrict__ order,
                                                    const u32 *__restrict__ seg_tile0, const u32 *__restrict__ spl0, int nb,
                                                    u32 *__restrict__ spl_next, u32 *__restrict__ spl_len, u32 p0, u32 ibwt_s) {
  u32 p = p0 + blockIdx.y;  // launched in batches of blocks whose T-vectors fit the L2 together
  const DecBlk &b = blks[order[p]];
  u32 n = b.count;
  if (n == 0) return;
  const u32 *T = tt + (u64)seg_tile0[p] * SORT_TILE;
  u32 W = (n + IBWT_S - 1) / IBWT_S + 1;
  u32 pos0 = T[b.orig_ptr] >> 8;
  for (u32 s = blockIdx.x * blockDim.x + threadIdx.x; s < W; s += gridDim.x * blockDim.x) {
    u32 start = s == W - 1 ? pos0 : s * IBWT_S;
    if (s != W - 1 && start == pos0) {  // duplicate of the extra splitter: unused
      spl_len[spl0[p] + s] = 0;
      spl_next[spl0[p] + s] = s;
      continue;
    }
    u32 cur = start, len = 0;
    do { cur = T[cur] >> 8; len++; } while (!ibwt_is_spl(cur, pos0, ibwt_s) && len < n);
    spl_next[spl0[p] + s] = ibwt_spl_index(cur, pos0, W, ibwt_s);
    spl_len[spl0[p] + s] = len;
  }
}
#define IBWT_R 64      // sub-splitter spacing of the splitter chase
#define IBWT_SUBS 256  // >= (900000 / 64 + 2) / IBWT_R + 2 sub-splitters
// one CTA per block: offsets of the splitters along the walk from pos0; period if the walk closes
// one CTA per block: the splitter links are staged in shared memory, one thread chases them there (a few dozen cycles
// per hop instead of a DRAM round trip), all threads write the offsets back.  Dynamic shared memory: 3 * W words.
// The walks between splitters are tail-bound (the longest chain is ~11x the spacing), so the spacing is small (64:
// walk1 + walk2 + rank = 0.64 + 1.29 + 0.85 ms per 100 MB; 128: 1.26 + 1.70 + 0.43; 256: 2.27 + 2.64 + 0.22).
__global__ void __launch_bounds__(256) k_ibwt_rank(const DecBlk *__restrict__ blks, const u32 *__restrict__ order, const u32 *__restrict__ spl0, int nb,
                                                   const u32 *__restrict__ spl_next, const u32 *__restrict__ spl_len, u32 *__restrict__ spl_off,
                                                   u32 *__restrict__ period, u32 ibwt_s) {
  DYN_SMEM(u32, sm);
  const int p = blockIdx.x;
  const u32 n = blks[order[p]].count;
  if (n == 0) { if (threadIdx.x == 0) period[p] = 0; return; }
  const u32 W = (n + IBWT_S - 1) / IBWT_S + 1, base = spl0[p];
  u64 *lk = reinterpret_cast<u64 *>(sm);  // (length << 32) | next splitter: one dependent read per hop
  u32 *of = sm + 2 * W;
  for (u32 s = threadIdx.x; s < W; s += blockDim.x) { lk[s] = ((u64)spl_len[base + s] << 32) | spl_next[base + s]; of[s] = 0xffffffffu; }
  __syncthreads();
  // the chase over W links is itself list ranking: every 64th link (and the start) is a sub-splitter, all threads walk
  // from theirs to the next one, one thread chases the few hundred sub-splitters, all threads walk again writing offsets
  __shared__ u32 sub_next[IBWT_SUBS], sub_len[IBWT_SUBS], sub_off[IBWT_SUBS];
  const u32 NS = (W + IBWT_R - 1) / IBWT_R + 1;  // the last one is the start link W-1
  for (u32 q = threadIdx.x; q < NS; q += blockDim.x) {
    const u32 s0 = q == NS - 1 ? W - 1 : q * IBWT_R;
    sub_off[q] = 0xffffffffu;
    sub_next[q] = q; sub_len[q] = 0;
    if (q != NS - 1 && s0 >= W - 1) continue;  // past the end, or the start link itself (its own sub-splitter)
    u32 cur = s0, acc = 0, hops = 0;
    do {
      const u64 e = lk[cur];
      acc += (u32)(e >> 32);
      cur = (u32)e;
      hops++;
    } while (cur != W - 1 && (cur % IBWT_R) != 0 && hops < W);  // (a cycle without sub-splitters is not on the path)
    sub_next[q] = cur == W - 1 ? NS - 1 : cur / IBWT_R;
    sub_len[q] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    u32 q = NS - 1, off = 0, per = 0;
    while (off < n) {
      if (sub_off[q] != 0xffffffffu) { per = off - sub_off[q]; break; }  // closed a cycle (periodic block)
      sub_off[q] = off;
      off += sub_len[q];
      q = sub_next[q];
    }
    period[p] = per;
  }
  __syncthreads();
  for (u32 q = threadIdx.x; q < NS; q += blockDim.x) {
    u32 off = sub_off[q];
    if (off == 0xffffffffu) continue;
    u32 cur = q == NS - 1 ? W - 1 : q * IBWT_R;
    do {
      const u64 e = lk[cur];
      of[cur] = off;
      off += (u32)(e >> 32);
      cur = (u32)e;
    } while (cur != W - 1 && (cur % IBWT_R) != 0);
  }
  __syncthreads();
  for (u32 s = threadIdx.x; s < W; s += blockDim.x) spl_off[base + s] = of[s];
}
__global__ void __launch_bounds__(256) k_ibwt_walk2(const u32 *__restrict__ tt, const u8 *__restrict__ dL, i64 l_stride,
                                                    const DecBlk *__restrict__ blks, const u32 *__restrict__ order,
                                                    const u32 *__restrict__ seg_tile0, const u32 *__restrict__ spl0, int nb,
                                                    const u32 *__restrict__ spl_len, const u32 *__restrict__ spl_off,
                                                    const u32 *__restrict__ period, u8 *__restrict__ blk_out, i64 b_stride, u32 p0, u32 ibwt_s) {
  u32 p = p0 + blockIdx.y;
  const DecBlk &b = blks[order[p]];
  u32 n = b.count;
  if (n == 0) return;
  const u32 *T = tt + (u64)seg_tile0[p] * SORT_TILE;
  u8 *out = blk_out + (i64)p * b_stride;
  u32 W = (n + IBWT_S - 1) / IBWT_S + 1;
  u32 pos0 = T[b.orig_ptr] >> 8, per = period[p];
  for (u32 s = blockIdx.x * blockDim.x + threadIdx.x; s < W; s += gridDim.x * blockDim.x) {
    u32 off = spl_off[spl0[p] + s], len = spl_len[spl0[p] + s];
    if (off == 0xffffffffu || len == 0) continue;
    u32 cur = s == W - 1 ? pos0 : s * IBWT_S;
    for (u32 t = 0; t < len; t++) {
      const u32 en = T[cur];
      const u8 byte = (u8)en;
      for (u64 o = (u64)off + t; o < n; o += per ? per : n) out[o] = byte;
      cur = en >> 8;
    }
  }
}

// ---- K-U4c: RLE1^-1 ---------------------------------------------------------------------------
// functions {0,1}->{0,1} packed as f(0) | f(1) << 1; compose(a, b) = b after a
__device__ __forceinline__ u32 fn_compose(u32 a, u32 b) { return ((b >> (a & 1)) & 1) | (((b >> ((a >> 1) & 1)) & 1) << 1); }
#define FN_ID 2u
__device__ __forceinline__ u32 block_excl_fn(u32 f, u32 &total, u32 *ws) {
  int lane = lane_id(), w = warp_id(), nw = blockDim.x >> 5;
  u32 inc = f;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    u32 t = __shfl_up_sync(FULL_MASK, inc, d);
    if (lane >= d) inc = fn_compose(t, inc);
  }
  u32 prev = __shfl_up_sync(FULL_MASK, inc, 1);
  if (lane == 0) prev = FN_ID;
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  if (w == 0) {
    u32 x = lane < nw ? ws[lane] : FN_ID, xi = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      u32 t = __shfl_up_sync(FULL_MASK, xi, d);
      if (lane >= d) xi = fn_compose(t, xi);
    }
    u32 xe = __shfl_up_sync(FULL_MASK, xi, 1);
    if (lane == 0) xe = FN_ID;
    ws[lane] = xe;
    if (lane == 31) ws[32] = xi;
  }
  __syncthreads();
  u32 res = fn_compose(ws[w], prev);
  total = ws[32];
  __syncthreads();
  return res;
}
#define RLI_K 8  // bytes per thread and strip
// threads: 1024 when every block has an SM to itself (latency), else 512 (62 registers: two CTAs per SM)
// mode 0: out_len[p] = decoded size of block p.  mode 1: write the bytes at out + out_off[p].
__global__ void __launch_bounds__(1024) k_rle1_inv(const u8 *__restrict__ blk, i64 b_stride, const DecBlk *__restrict__ blks,
                                                   const u32 *__restrict__ order, int mode, u64 *__restrict__ out_len,
                                                   const u64 *__restrict__ out_off, u8 *__restrict__ out) {
  __shared__ int wsi[33];
  __shared__ u32 ws[34];
  __shared__ u64 ws64[33];
  const u32 p = blockIdx.x;
  const u32 n = blks[order[p]].count;
  const u8 *E = blk + (i64)p * b_stride;
  u8 *O = mode ? out + out_off[p] : nullptr;
  int carry_head = 0;   // last run head seen so far
  u32 carry_fn = 0;     // composed carry function so far, applied to 0: constant -> store as value 0/1 in both bits
  u64 carry_out = 0;
  carry_fn = 0u;        // const 0 (c of the first run is 0)
  // a strip is RLI_K bytes per thread: the three CTA scans per strip are the cost (one CTA walks a block serially), so
  // the strip is wide
  for (u32 base = 0; base < n; base += blockDim.x * RLI_K) {
    u32 i0 = base + threadIdx.x * RLI_K;
    u8 e[RLI_K + 2];  // e[0] = byte before i0, e[1..RLI_K] = mine, e[RLI_K+1] = byte after
    if (i0 + RLI_K <= n) {  // (block buffers are 256-byte aligned and i0 is a multiple of 8)
      const uint2 v = *reinterpret_cast<const uint2 *>(E + i0);
#pragma unroll
      for (int k = 0; k < 4; k++) { e[1 + k] = (u8)(v.x >> (8 * k)); e[5 + k] = (u8)(v.y >> (8 * k)); }
    } else {
#pragma unroll
      for (int k = 0; k < RLI_K; k++) e[1 + k] = i0 + k < n ? E[i0 + k] : 0;
    }
    e[0] = i0 > 0 && i0 - 1 < n ? E[i0 - 1] : 0;
    e[RLI_K + 1] = i0 + RLI_K < n ? E[i0 + RLI_K] : 0;
    // run heads and ends among my positions
    int my_head = -1;
    u32 headm = 0, endm = 0;
#pragma unroll
    for (int k = 0; k < RLI_K; k++) {
      u32 i = i0 + k;
      const bool hd = i < n && (i == 0 || e[k + 1] != e[k]);
      const bool en = i < n && (i + 1 >= n || e[k + 2] != e[k + 1]);
      headm |= (u32)hd << k;
      endm |= (u32)en << k;
      if (hd) my_head = (int)i;
    }
    int tot_h;
    int hb = block_excl_max<int>(my_head, -1, tot_h, wsi);
    if (carry_head > hb) hb = carry_head;
    // carry function of my positions: at a run end of length l, f(c) = ((l - c) mod 5 == 4)
    u32 f = FN_ID;
    {
      int cur = hb;
#pragma unroll
      for (int k = 0; k < RLI_K; k++) {
        u32 i = i0 + k;
        if ((headm >> k) & 1u) cur = (int)i;
        if ((endm >> k) & 1u) {
          u32 l = i - (u32)cur + 1;
          u32 g = ((l % 5) == 4 ? 1u : 0u) | ((((l + 4) % 5) == 4) ? 2u : 0u);  // (l-1) mod 5 == 4  <=>  (l+4) mod 5 == 4
          f = fn_compose(f, g);
        }
      }
    }
    u32 tot_f;
    u32 fe = block_excl_fn(f, tot_f, ws);
    u32 c_in = (fn_compose(carry_fn, fe)) & 1u;  // carry_fn is constant: value in bit 0
    // counts
    u32 cnt = 0;
    u32 emit[RLI_K];
    {
      int cur = hb;
      u32 c = c_in;
#pragma unroll
      for (int k = 0; k < RLI_K; k++) {
        u32 i = i0 + k;
        emit[k] = 0;
        if (i < n) {
          if ((headm >> k) & 1u) cur = (int)i;
          int kk = (int)(i - (u32)cur) - (int)c;  // index among the run's own literals/counts
          if (kk < 0) emit[k] = 0x100u | e[k + 1];            // count byte of the previous run: e[k+1] copies of e[k]
          else if (kk % 5 == 4) emit[k] = 0x200u | e[k + 1];  // count byte of this run
          else emit[k] = 0x400u;                               // literal
          cnt += (emit[k] & 0x400u) ? 1u : (emit[k] & 0xffu);
          if ((endm >> k) & 1u) {
            u32 l = i - (u32)cur + 1;
            c = ((l - c) % 5 == 4) ? 1u : 0u;
          }
        }
      }
    }
    u64 tot_o;
    u64 o = carry_out + block_excl_sum<u64>((u64)cnt, tot_o, ws64);
    if (mode) {
#pragma unroll
      for (int k = 0; k < RLI_K; k++) {
        if (!emit[k]) continue;
        if (emit[k] & 0x400u) O[o++] = e[k + 1];
        else {
          u8 v = (emit[k] & 0x100u) ? e[k] : e[k + 1];
          u32 copies = emit[k] & 0xffu;
          for (u32 q = 0; q < copies; q++) O[o++] = v;
        }
      }
    }
    carry_out += tot_o;
    if (tot_h > carry_head) carry_head = tot_h;
    u32 cf = fn_compose(carry_fn, tot_f) & 1u;
    carry_fn = cf | (cf << 1);
  }
  if (mode == 0 && threadIdx.x == 0) out_len[p] = carry_out;
}

// BlockRec ranges for the CRC kernels: block p covers out[out_off[p], out_off[p+1])
__global__ void k_dec_crc_recs(const u64 *__restrict__ out_off, int nb, BlockRec *__restrict__ recs) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nb) return;
  BlockRec r;
  r.s = (i64)out_off[p]; r.p = (i64)out_off[p + 1]; r.e_true = 0; r.Ge = 0; r.outR = 0; r.n = 0; r.crc = 0; r.orig_ptr = 0;
  recs[p] = r;
}

// ---- range reads (bz2b200_decompress_ranges) --------------------------------------------------------------------------
// Packs pieces of the decoded blocks into one buffer: piece i = src[piece_src[i], +len) -> dst[piece_dst[i], +len), with
// piece_dst the exclusive scan of the lengths (piece_dst[n_pieces] = total, every piece at least one byte long).  The work
// is split by output bytes, GATHER_CHUNK per CTA: thread 0 finds the piece that holds the CTA's first byte by binary
// search, then the CTA copies every piece that meets its chunk together -- 16-byte stores on 16-byte-aligned destination
// addresses, the source read as aligned words and shifted into place when it is not aligned alike.  The source buffer
// must be readable for 4 bytes after a piece's end (a decode sink keeps 64 bytes of slack).
#define GATHER_CHUNK 8192u
#define GATHER_THREADS 256
__global__ void __launch_bounds__(GATHER_THREADS) k_gather_ranges(const u8 *__restrict__ src, const u64 *__restrict__ piece_src,
                                                                  const u64 *__restrict__ piece_dst, u32 n_pieces, u64 total, u8 *__restrict__ dst) {
  __shared__ u32 first;
  const u64 c0 = (u64)blockIdx.x * GATHER_CHUNK;
  const u64 c1 = c0 + GATHER_CHUNK < total ? c0 + GATHER_CHUNK : total;
  if (threadIdx.x == 0) {  // piece_dst[lo] <= c0 < piece_dst[hi]
    u32 lo = 0, hi = n_pieces;
    while (hi - lo > 1) {
      const u32 mid = (lo + hi) >> 1;
      if (piece_dst[mid] <= c0) lo = mid; else hi = mid;
    }
    first = lo;
  }
  __syncthreads();
  for (u32 p = first; p < n_pieces && piece_dst[p] < c1; p++) {
    const u64 a = piece_dst[p] > c0 ? piece_dst[p] : c0, e = piece_dst[p + 1] < c1 ? piece_dst[p + 1] : c1;
    const u8 *s = src + piece_src[p] + (a - piece_dst[p]);
    u8 *d = dst + a;
    const u32 len = (u32)(e - a);  // at most GATHER_CHUNK
    const u32 head = min((u32)((16u - ((uintptr_t)d & 15u)) & 15u), len);
    const u32 nvec = (len - head) >> 4;
    if (threadIdx.x < head) d[threadIdx.x] = s[threadIdx.x];
    const u8 *sv = s + head;
    uint4 *dv = reinterpret_cast<uint4 *>(d + head);
    if (((uintptr_t)sv & 15u) == 0) {
      for (u32 v = threadIdx.x; v < nvec; v += GATHER_THREADS) dv[v] = reinterpret_cast<const uint4 *>(sv)[v];
    } else {
      const u32 *w0 = reinterpret_cast<const u32 *>((uintptr_t)sv & ~(uintptr_t)3);
      const u32 sh = 8u * (u32)((uintptr_t)sv & 3u);
      for (u32 v = threadIdx.x; v < nvec; v += GATHER_THREADS) {
        const u32 *w = w0 + 4 * v;
        const u32 x0 = w[0], x1 = w[1], x2 = w[2], x3 = w[3], x4 = sh ? w[4] : 0u;
        dv[v] = make_uint4(__funnelshift_r(x0, x1, sh), __funnelshift_r(x1, x2, sh), __funnelshift_r(x2, x3, sh), __funnelshift_r(x3, x4, sh));
      }
    }
    const u32 t0 = head + 16 * nvec;
    if (threadIdx.x < len - t0) d[t0 + threadIdx.x] = s[t0 + threadIdx.x];
  }
}
