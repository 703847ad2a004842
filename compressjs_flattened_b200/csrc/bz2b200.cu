// bz2b200.cu -- host orchestration and the C ABI (include/bz2b200.h).
//
// Product build: nvcc -gencode arch=compute_100a,code=sm_100a -> libbz2b200.so (CUDA only; every
// entry point fails with BZ2B200_E_CUDA when no device is present -- there is no CPU path).
// Test build:    g++ -DBZ_SIM (cusim.h) -> tests/sim/libbz2b200_sim.so, kernel-logic tests only.
#include "../../include/bz2b200.h"
#include "common.cuh"
#include "rle1.cuh"
#include "bwt.cuh"
#include "refine.cuh"
#include "mtf.cuh"
#include "huff.cuh"
#include "decode.cuh"
#include "search.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <future>
#include <map>
#include <mutex>
#include <thread>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <fcntl.h>
#include <sched.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <string>
#include <utility>
#include <vector>

namespace {

// ---- bzip2 stream framing, host side (k_stream_ends writes the same header and footer on the device) ----------
// header: "BZh" and the level digit (BJ:2223-2226)
static void stream_header(u8 *h, int level) { h[0] = 'B'; h[1] = 'Z'; h[2] = 'h'; h[3] = (u8)('0' + level); }
// the 4 bytes at h start with "BZh", whatever the level digit
static bool stream_header_magic(const u8 *h) { return h[0] == 'B' && h[1] == 'Z' && h[2] == 'h'; }
// the level of the 4-byte header at h, 0 if it is not a header (BJ:1408-1427)
static int stream_header_level(const u8 *h) { return stream_header_magic(h) && h[3] >= '1' && h[3] <= '9' ? h[3] - '0' : 0; }
// the combined CRC after `blocks` more blocks whose own combined CRC, counted from 0, is `fold` (BJ:2237)
static u32 stream_crc_add(u32 crc, u32 blocks, u32 fold) {
  const u32 m = blocks & 31u;
  return (m ? (crc << m) | (crc >> (32 - m)) : crc) ^ fold;
}
// footer: the end-of-stream magic and the combined CRC, 80 bits ORed into dst from bit `bitpos` on (the caller clears
// those bytes); returns the bit after it (BJ:2245-2247)
static u64 stream_footer(u8 *dst, u64 bitpos, u32 crc) {
  const u64 vals[2] = {BZ_MAGIC_END, (u64)crc};
  const int lens[2] = {48, 32};
  for (int q = 0; q < 2; q++)
    for (int i = lens[q] - 1; i >= 0; i--, bitpos++)
      if ((vals[q] >> i) & 1) dst[bitpos >> 3] |= (u8)(0x80u >> (bitpos & 7));
  return bitpos;
}

// ---- results handed to the caller ------------------------------------------------------------
// Large results live in page-locked memory (the device-to-host copy then runs at PCIe speed instead of through
// the driver's pageable staging).  bz2b200_free() recognises them and keeps a few for reuse, so a caller that
// compresses in a loop does not pay cudaMallocHost every time.  Small results are plain malloc.
struct ResultPool {
  std::mutex mu;
  std::vector<std::pair<void *, size_t>> live, idle;  // (pointer, capacity)
  size_t idle_bytes = 0;
  static const size_t kMinPinned = 1 << 20, kMaxIdle = 48;  // a sharded call hands out one segment per shard
  static const size_t kMaxIdleBytes = (size_t)12 << 30;     // page-locked memory kept for reuse
  void *get(size_t bytes) {
    if (bytes < kMinPinned) return malloc(bytes ? bytes : 1);
    std::lock_guard<std::mutex> g(mu);
    size_t best = idle.size();
    for (size_t i = 0; i < idle.size(); i++)
      if (idle[i].second >= bytes && (best == idle.size() || idle[i].second < idle[best].second)) best = i;
    if (best < idle.size()) {
      auto e = idle[best];
      idle.erase(idle.begin() + (long)best);
      idle_bytes -= e.second;
      live.push_back(e);
      return e.first;
    }
    void *p = nullptr;
    size_t cap = bytes + bytes / 4 + 4096;
#ifndef BZ_SIM
    if (cudaMallocHost(&p, cap) != cudaSuccess) { cudaGetLastError(); p = nullptr; }
#endif
    if (!p) return malloc(bytes);  // page-locking failed: fall back to pageable memory
    live.push_back({p, cap});
    return p;
  }
  void put(void *p) {
    if (!p) return;
    {
      std::lock_guard<std::mutex> g(mu);
      for (size_t i = 0; i < live.size(); i++)
        if (live[i].first == p) {
          auto e = live[i];
          live.erase(live.begin() + (long)i);
          if (idle.size() < kMaxIdle && idle_bytes + e.second <= kMaxIdleBytes) { idle.push_back(e); idle_bytes += e.second; return; }
#ifndef BZ_SIM
          cudaFreeHost(p);
#endif
          return;
        }
    }
    free(p);
  }
};
ResultPool &result_pool() { static ResultPool rp; return rp; }

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
};

struct Ctx;
struct Pool;
void pool_delete(Pool *p);
struct Ctx {
  Pool *own_pool = nullptr;         // two lanes on this context's device: large host inputs of bz2b200_compress
  size_t pool_min_bytes = 32000000; // inputs of this size or more go through own_pool
  size_t pool_shard_bytes = 0, pool_halo0 = 0;
  bool pool_force_staging = false;
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  bz2b200_stats st{};
  std::vector<DevBuf *> pool;
  // compress-side buffers
  DevBuf in, tile_last, tile_first, head_carry, tile_emit, g_sub, h_sub, g_tile, recs, nblk, blk, crcpart, pow256;
  DevBuf isa, keysA, keysB, valsB, actI0, actI1, actR0, actR1, lb_status, lbm, hist, digit_base;
  DevBuf seg_cnt, seg_tile0, tile_blk, tile_i0, tile_i1, totals;
  DevBuf Lcol, ranks, lastocc, A, freq, meta, W, bit_off, scrc, out, out_len, used_bits;
  DevBuf gbounds;
  DevBuf key2, big_cnt, big_old, big_rank, big_tile0, big_tblk, totals2;
  DevBuf recs_cand, cand_first, out2, blksort, r2_status, hfreq, hlens, hplen, hcodes, hsel, hcost, hgoff, hblk;
  // decode-side buffers
  DevBuf d_in, cand, ncand, dmeta, dsyms, dL, dtt, dwalk, dblk, dout, dmisc, dsel, doff, dperm, dmap;
  DevBuf dpieces, dgather;  // range reads: the pieces and the packed bytes (search: the lines)
  DevBuf dspat, dstile, dsbase, dstsum, dsmatch, dspart, dstot;  // search: patterns and filter, per-tile and per-thread summaries, matches
  // last compress, for debug_fetch
  struct Pipe {
    const u8 *d_in = nullptr;
    i64 N = 0, T = 0, BS = 0, AS = 0, WS = 0;
    u32 B = 0;
    int level = 9, nb = 0;
    std::vector<BlockRec> hrecs;
  } pipe;
  bool trace = false;      // BZ2B200_TRACE
  int sms = 148;           // multiprocessors of the device
  int parse_mode = 0;      // BZ2B200_PARSE: 0 = by block count, 1 = k_huff_parse, 2 = k_huff_parse_win (development aid)
  std::vector<cudaEvent_t> trace_ev, trace_pool;
  std::vector<const char *> trace_names;
  void *rb_pin = nullptr;  // mapped page-locked scratch of rb_add / rb_sync (host address) and its device address
  void *rb_dev = nullptr;
  const void *rb_src[4];
  void *rb_dst[4];
  size_t rb_off[4], rb_len[4], rb_used = 0;
  int rb_n = 0;
  u32 rb_seq = 0;
  bool ignore_block_crc = false;  // tests only (bz2b200_debug_set_ignore_block_crc)
  u32 cap_override = 0;    // tests only
  u32 batch_override = 0;  // tests only: blocks per batch
  u32 dec_batch = 0;       // tests only: candidates per decode batch (0 = DEC_BATCH)
  u32 rle1_threads = 0;    // tests only: CTA width of k_rle1_inv, 512 or 1024 (0 = by block count)
  // the last decode batch, for the decode kinds of debug_fetch: candidates parsed, blocks inverted (indices into the
  // candidates, stream order) and the stride of their inverse-BWT outputs
  u32 dec_last_ncand = 0;
  std::vector<u32> dec_last_chain;
  i64 dec_last_bs = 0;
  u32 search_tile = 0;     // tests only: bytes per search tile (0 = SEARCH_TILE_DEFAULT)
  u64 shard_bits = 0;      // bit length of the last shard segment (phase 0 in `out`)
  int cand_n = 0, cand_max_blocks = 0, cand_nb[64];  // speculated cut walks of the last shard_cut_g
  i64 cand_s[64];
  int last_nb = 0;
  i64 last_bs = 0, last_as = 0, last_ss = 0;
  cudaEvent_t ev[10]{};
  bool ev_ok = false;
  std::vector<cudaEvent_t> dom_ev;  // start/stop pairs around the dominant kernel's launches
  size_t dom_used = 0;
  Ctx() {
    DevBuf *all[] = {&in, &tile_last, &tile_first, &head_carry, &tile_emit, &g_sub, &h_sub, &g_tile, &recs, &nblk, &blk, &crcpart, &pow256,
                     &isa, &keysA, &keysB, &valsB, &actI0, &actI1, &actR0, &actR1, &lb_status, &lbm, &hist, &digit_base,
                     &seg_cnt, &seg_tile0, &tile_blk, &tile_i0, &tile_i1, &totals,
                     &Lcol, &ranks, &lastocc, &A, &freq, &meta, &W, &bit_off, &scrc, &out, &out_len, &used_bits,
                     &gbounds, &key2, &big_cnt, &big_old, &big_rank, &big_tile0, &big_tblk, &totals2,
                     &recs_cand, &cand_first, &out2, &blksort, &r2_status, &hfreq, &hlens, &hplen, &hcodes, &hsel, &hcost, &hgoff, &hblk,
                     &d_in, &cand, &ncand, &dmeta, &dsyms, &dL, &dtt, &dwalk, &dblk, &dout, &dmisc, &dsel, &doff, &dperm, &dmap,
                     &dpieces, &dgather, &dspat, &dstile, &dsbase, &dstsum, &dsmatch, &dspart, &dstot};
    for (DevBuf *b : all) pool.push_back(b);
  }
};

#define CK(call)                                                                         \
  do {                                                                                   \
    cudaError_t _e = (call);                                                             \
    if (_e != cudaSuccess) {                                                             \
      c->err = std::string(#call) + ": " + cudaGetErrorString(_e);                       \
      return BZ2B200_E_CUDA;                                                             \
    }                                                                                    \
  } while (0)

// Small device -> host read-backs (block / slot counts): a one-warp kernel copies the pending words into a page of MAPPED
// host memory and writes a sequence number last; the host spins on that word.  Against cudaMemcpyAsync + cudaStreamSynchronize
// this saves the copy-engine command and the driver's wake-up per round trip (~20 round trips per compress call).
struct RbItem { const void *src; u32 off, bytes; };
__global__ void k_readback(RbItem i0, RbItem i1, RbItem i2, RbItem i3, int n, volatile u8 *host_page, u32 seq) {
  const RbItem it[4] = {i0, i1, i2, i3};
  for (int k = 0; k < n; k++)
    for (u32 b = threadIdx.x; b < it[k].bytes; b += blockDim.x) host_page[it[k].off + b] = reinterpret_cast<const u8 *>(it[k].src)[b];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) { *reinterpret_cast<volatile u32 *>(host_page + 1020) = seq; __threadfence_system(); }
}
int rb_add(Ctx *c, void *dst, const void *dev_src, size_t bytes) {
  if (!c->rb_pin) {
#ifndef BZ_SIM
    CK(cudaHostAlloc(&c->rb_pin, 1024, cudaHostAllocMapped));
    CK(cudaHostGetDevicePointer(&c->rb_dev, c->rb_pin, 0));
#else
    CK(cudaMallocHost(&c->rb_pin, 1024));
    c->rb_dev = c->rb_pin;
#endif
    memset(c->rb_pin, 0, 1024);
  }
  if (c->rb_n >= 4 || c->rb_used + bytes > 1000) { c->err = "internal: read-back scratch full"; return BZ2B200_E_CUDA; }
  c->rb_src[c->rb_n] = dev_src;
  c->rb_dst[c->rb_n] = dst; c->rb_off[c->rb_n] = c->rb_used; c->rb_len[c->rb_n] = bytes;
  c->rb_n++;
  c->rb_used += (bytes + 15) & ~(size_t)15;
  return 0;
}
int rb_sync(Ctx *c) {
  if (!c->rb_n) { CK(cudaStreamSynchronize(c->stream)); return 0; }
  RbItem it[4] = {};
  for (int i = 0; i < c->rb_n; i++) { it[i].src = c->rb_src[i]; it[i].off = (u32)c->rb_off[i]; it[i].bytes = (u32)c->rb_len[i]; }
  const u32 seq = ++c->rb_seq;
  KLAUNCH(k_readback, 1, 32, 0, c->stream, it[0], it[1], it[2], it[3], c->rb_n, (volatile u8 *)c->rb_dev, seq);
#ifndef BZ_SIM
  volatile u32 *flag = reinterpret_cast<volatile u32 *>((u8 *)c->rb_pin + 1020);
  for (unsigned spin = 0; *flag != seq; spin++) {
    if ((spin & 0xfffff) == 0xfffff && cudaStreamQuery(c->stream) != cudaErrorNotReady) {  // the kernel is gone: done, or a fault upstream
      if (*flag == seq) break;
      CK(cudaStreamSynchronize(c->stream));
      CK(cudaGetLastError());
      c->err = "internal: read-back kernel did not publish";
      return BZ2B200_E_CUDA;
    }
  }
  std::atomic_thread_fence(std::memory_order_acquire);
#endif
  for (int i = 0; i < c->rb_n; i++) memcpy(c->rb_dst[i], (char *)c->rb_pin + c->rb_off[i], c->rb_len[i]);
  c->rb_n = 0;
  c->rb_used = 0;
  return 0;
}
#define RC(call)               \
  do {                         \
    int _r = (call);           \
    if (_r) return _r;         \
  } while (0)

void trace_mark(Ctx *c, const char *name, bool begin) {
#ifndef BZ_SIM
  cudaEvent_t e;
  if (c->trace_pool.size() > c->trace_ev.size()) e = c->trace_pool[c->trace_ev.size()];
  else { if (cudaEventCreate(&e) != cudaSuccess) return; c->trace_pool.push_back(e); }
  cudaEventRecord(e, c->stream);
  c->trace_ev.push_back(e);
  if (begin) c->trace_names.push_back(name);
#else
  (void)c; (void)name; (void)begin;
#endif
}
void trace_report(Ctx *c) {
#ifndef BZ_SIM
  if (!c->trace || c->trace_ev.empty()) return;
  cudaStreamSynchronize(c->stream);
  std::vector<std::pair<std::string, std::pair<int, float>>> agg;
  float gaps = 0, total = 0;
  for (size_t i = 0; i + 1 < c->trace_ev.size(); i += 2) {
    float ms = 0;
    cudaEventElapsedTime(&ms, c->trace_ev[i], c->trace_ev[i + 1]);
    const std::string nm = c->trace_names[i / 2];
    size_t k = 0;
    for (; k < agg.size(); k++) if (agg[k].first == nm) break;
    if (k == agg.size()) agg.push_back({nm, {0, 0.f}});
    agg[k].second.first++;
    agg[k].second.second += ms;
    total += ms;
    if (i + 2 < c->trace_ev.size()) { float g = 0; cudaEventElapsedTime(&g, c->trace_ev[i + 1], c->trace_ev[i + 2]); gaps += g; }
  }
  std::sort(agg.begin(), agg.end(), [](const auto &a, const auto &b) { return a.second.second > b.second.second; });
  fprintf(stderr, "[bz2b200 trace] %zu launches, kernels %.3f ms, gaps between launches %.3f ms\n", c->trace_names.size(), total, gaps);
  for (auto &a : agg) fprintf(stderr, "[bz2b200 trace] %-28s x%-3d %8.3f ms\n", a.first.c_str(), a.second.first, a.second.second);
  c->trace_ev.clear();
  c->trace_names.clear();
#else
  (void)c;
#endif
}

int ensure(Ctx *c, DevBuf &b, size_t bytes) {
  if (bytes <= b.cap) return 0;
  if (b.p) CK(cudaFree(b.p));
  b.p = nullptr;
  b.cap = 0;
  size_t want = bytes + bytes / 8 + 4096;
  CK(cudaMalloc(&b.p, want));
  b.cap = want;
  return 0;
}
#define ENS(buf, bytes)                         \
  do {                                          \
    int _r = ensure(c, (buf), (size_t)(bytes)); \
    if (_r) return _r;                          \
  } while (0)
template <typename T> T *P(DevBuf &b) { return reinterpret_cast<T *>(b.p); }

// BZ2B200_TRACE=1 in the environment: CUDA events around every launch, per-kernel totals printed by trace_report()
// at the end of a compress call (development aid; the extra events serialise nothing but cost a few microseconds each)
#define LAUNCH(kern, grid, block, smem, ...)                        \
  do {                                                              \
    if (c->trace) trace_mark(c, #kern, true);                       \
    KLAUNCH(kern, grid, block, smem, c->stream, __VA_ARGS__);       \
    if (c->trace) trace_mark(c, #kern, false);                      \
    c->st.kernel_launches++;                                        \
  } while (0)

inline i64 round_up(i64 v, i64 a) { return (v + a - 1) / a * a; }

int mark(Ctx *c, int i) {
  if (c->ev_ok) CK(cudaEventRecord(c->ev[i], c->stream));
  return 0;
}

// ------------------------------------------------------------------------------ compress
// The pipeline is split so that a multi-GPU caller can interleave it with the two scalar exchanges of
// SURVEY section 8e: pipe_begin (tile summaries; independent of where the first block starts), pipe_cut
// (the sequential cut walk from a known first-block offset) and pipe_run (pipe_stages, everything per block, then the
// bit-granular stitch at a given bit offset, batch by batch).
int pipe_begin(Ctx *c, const u8 *d_in, size_t n_, int level) {
  if (level < 1 || level > 9) return BZ2B200_E_LEVEL;
  c->st = bz2b200_stats{};
  c->st.in_bytes = n_;
  c->err.clear();
  Ctx::Pipe &P_ = c->pipe;
  P_ = Ctx::Pipe{};
  P_.d_in = d_in; P_.N = (i64)n_; P_.level = level;
  P_.B = c->cap_override ? c->cap_override : (u32)level * 100000u - 19u;  // BJ:2212-2220
  P_.T = (P_.N + RLE_TILE - 1) / RLE_TILE;
  const i64 N = P_.N, T = P_.T;
  int rc;
  if ((rc = mark(c, 0))) return rc;
  if (N > 0) {
    ENS(c->tile_last, 8 * T); ENS(c->tile_first, 8 * T); ENS(c->head_carry, 8 * T);
    ENS(c->tile_emit, 4 * T); ENS(c->g_tile, 8 * (T + 1));
    LAUNCH(k_rle_heads, (unsigned)T, RLE_THREADS, 0, d_in, N, P<i64>(c->tile_last), P<i64>(c->tile_first));
    LAUNCH(k_scan_excl_max_i64, 1, 1024, 0, P<i64>(c->tile_last), P<i64>(c->head_carry), T);
    ENS(c->g_sub, 4 * (size_t)T * (RLE_THREADS / 32)); ENS(c->h_sub, 8 * (size_t)T * (RLE_THREADS / 32));
    LAUNCH(k_rle_count, (unsigned)T, RLE_THREADS, 0, d_in, N, P<i64>(c->head_carry), P<u32>(c->tile_emit), P<u32>(c->g_sub), P<i64>(c->h_sub));
    LAUNCH(k_scan_excl_sum_u32_u64, 1, 1024, 0, P<u32>(c->tile_emit), P<u64>(c->g_tile), T);
  }
  return BZ2B200_OK;
}

#define CUT_CANDIDATES 64  // speculative shard starts tried at once (phases g_start - 32 .. g_start + 31)
int pipe_cut(Ctx *c, i64 s_start, i64 own_end, i64 g_start = -1) {
  Ctx::Pipe &P_ = c->pipe;
  const i64 N = P_.N, T = P_.T;
  const u32 B = P_.B;
  const int max_blocks = (int)(N / ((i64)B * 4 / 5) + 2);
  const int ncand = g_start >= 0 ? CUT_CANDIDATES : 1;
  ENS(c->recs, sizeof(BlockRec) * (size_t)max_blocks);
  ENS(c->nblk, 64 + 4 * CUT_CANDIDATES);
  int nb = 0;
  P_.hrecs.clear();
  c->cand_n = 0;
  if (N > 0 && g_start >= 0) {
    // all candidates walk at once; the tables stay on the device until pipe_pick installs the right one
    ENS(c->recs_cand, sizeof(BlockRec) * (size_t)max_blocks * ncand);
    LAUNCH(k_rle_cut, ncand, CUT_THREADS, 0, P_.d_in, N, B, P<u32>(c->g_sub), P<i64>(c->h_sub), P<i64>(c->tile_first), P<u64>(c->g_tile), T,
           P<BlockRec>(c->recs_cand), max_blocks, P<int>(c->nblk) + 16, s_start, own_end, g_start);
    LAUNCH(k_cand_firsts, 1, CUT_CANDIDATES, 0, P<BlockRec>(c->recs_cand), max_blocks, P<int>(c->nblk) + 16, P<i64>(c->cand_first));
    RC(rb_add(c, c->cand_nb, P<int>(c->nblk) + 16, 4 * CUT_CANDIDATES));
    RC(rb_add(c, c->cand_s, c->cand_first.p, 8 * CUT_CANDIDATES));
    RC(rb_sync(c));
    c->cand_n = ncand;
    c->cand_max_blocks = max_blocks;
  } else if (N > 0 && s_start < N && s_start < own_end) {
    LAUNCH(k_rle_cut, 1, CUT_THREADS, 0, P_.d_in, N, B, P<u32>(c->g_sub), P<i64>(c->h_sub), P<i64>(c->tile_first), P<u64>(c->g_tile), T,
           P<BlockRec>(c->recs), max_blocks, P<int>(c->nblk), s_start, own_end, (i64)-1);
    RC(rb_add(c, &nb, c->nblk.p, sizeof(int)));
    RC(rb_sync(c));
    if (nb < 0) { c->err = "internal: block table overflow"; return BZ2B200_E_CUDA; }
    P_.hrecs.resize((size_t)nb);
    if (nb) CK(cudaMemcpy(P_.hrecs.data(), c->recs.p, sizeof(BlockRec) * (size_t)nb, cudaMemcpyDeviceToHost));
  }
  P_.nb = nb;
  c->st.n_blocks = (u32)nb;
  return BZ2B200_OK;
}
// install the speculated block table whose walk started at s_local (or the empty one when no block starts before
// own_end); false if no candidate matches
bool pipe_pick(Ctx *c, i64 s_local, i64 own_end, int &rc) {
  Ctx::Pipe &P_ = c->pipe;
  rc = BZ2B200_OK;
  if (!(s_local < P_.N && s_local < own_end)) {  // this shard owns no block whatever was speculated
    P_.hrecs.clear();
    P_.nb = 0;
    c->st.n_blocks = 0;
    return true;
  }
  for (int j = 0; j < c->cand_n; j++) {
    const int nbj = c->cand_nb[j];
    if (nbj <= 0 || c->cand_s[j] != s_local) continue;
    P_.hrecs.resize((size_t)nbj);
    const BlockRec *src = P<BlockRec>(c->recs_cand) + (size_t)j * c->cand_max_blocks;
    if (cudaMemcpyAsync(c->recs.p, src, sizeof(BlockRec) * (size_t)nbj, cudaMemcpyDeviceToDevice, c->stream) != cudaSuccess ||
        cudaMemcpy(P_.hrecs.data(), src, sizeof(BlockRec) * (size_t)nbj, cudaMemcpyDeviceToHost) != cudaSuccess) { rc = BZ2B200_E_CUDA; return false; }
    P_.nb = nbj;
    c->st.n_blocks = (u32)nbj;
    return true;
  }
  return false;
}

// the stages of blocks first .. first + nb - 1 of the block table
int pipe_stages(Ctx *c, int first, int nb) {
  Ctx::Pipe &P_ = c->pipe;
  const i64 N = P_.N, T = P_.T;
  const u32 B = P_.B;
  const u8 *d_in = P_.d_in;
  const BlockRec *hrecs = P_.hrecs.data() + first;
  BlockRec *recs = P<BlockRec>(c->recs) + first;
  int rc;
  const i64 BS = round_up((i64)B + 1, 256);  // per-block stride of byte arrays (block, L, ranks)
  const i64 AS = round_up((i64)B + 2, 128);  // per-block stride of the u16 symbol array
  P_.BS = BS; P_.AS = AS;
  c->last_nb = nb; c->last_bs = BS; c->last_as = AS;
  ENS(c->meta, sizeof(BlockMeta) * (size_t)(nb + 1));
  ENS(c->bit_off, 8 * (size_t)(nb + 2));
  ENS(c->scrc, 64);
  ENS(c->out_len, 64);
  i64 WS = 0;
  if (nb) {
    // ---- S1 emit + CRC ----
    ENS(c->blk, (size_t)nb * BS);
    const i64 t_first = hrecs[0].s / RLE_TILE, t_last = (hrecs[nb - 1].p + RLE_TILE - 1) / RLE_TILE;
    (void)T;
    LAUNCH(k_rle_emit, (unsigned)(t_last - t_first), RLE_THREADS, 0, d_in, N, B, P<i64>(c->head_carry), P<u64>(c->g_tile), recs, nb,
           P<u8>(c->blk), BS, t_first);
    i64 max_len = 0;
    for (int k = 0; k < nb; k++) { const BlockRec &r = hrecs[k]; if (r.p - r.s > max_len) max_len = r.p - r.s; c->st.rle1_bytes += r.n; }
    int max_chunks = (int)((max_len + CRC_CHUNK - 1) / CRC_CHUNK);
    ENS(c->crcpart, 4 * (size_t)nb * max_chunks);
    if (!c->pow256.p) {
      ENS(c->pow256, 1024);
      u32 h[256];
      for (int j = 0; j < 256; j++) h[j] = crc_xpow(8ull * 256 * (u64)j);
      CK(cudaMemcpy(c->pow256.p, h, sizeof h, cudaMemcpyHostToDevice));
    }
    LAUNCH(k_crc_chunks, dim3((unsigned)max_chunks, (unsigned)nb), 256, 0, d_in, recs, P<u32>(c->pow256), P<u32>(c->crcpart),
           max_chunks);
    LAUNCH(k_crc_fold, (unsigned)((nb + 127) / 128), 128, 0, recs, nb, P<u32>(c->crcpart), max_chunks,
           crc_xpow(8ull * CRC_CHUNK));
    if ((rc = mark(c, 1))) return rc;

    // ---- S2 BWT ----
    size_t slots = 0;
    for (int k = 0; k < nb; k++) slots += (size_t)round_up(hrecs[k].n, SORT_TILE);
    const size_t tiles0 = slots / SORT_TILE;
    if ((u64)nb * (u64)BS >= (1ull << 31)) { c->err = "too many bytes for one call (block table * stride must stay below 2^31)"; return BZ2B200_E_ARG; }
    const size_t big_tiles = 5 * tiles0 + 16;                // big groups have > RF_T0 slots each
    const u32 big_cap = (u32)(slots / RF_T0 + 16);
    const size_t lb_tiles = slots / RF_T0 + tiles0 + 16;
    ENS(c->isa, 4 * (size_t)nb * BS);
    ENS(c->Lcol, (size_t)nb * BS);  // written by whichever kernel makes a rotation's rank final
    ENS(c->keysA, 8 * slots); ENS(c->keysB, 8 * slots);
    ENS(c->actI0, 4 * slots); ENS(c->actI1, 4 * slots); ENS(c->actR0, 4 * slots); ENS(c->actR1, 4 * slots);
    ENS(c->key2, 4 * slots);
    ENS(c->hist, 4 * 512 * big_tiles); ENS(c->digit_base, 4 * 512 * (size_t)(big_cap > (u32)nb ? big_cap : (u32)nb));
    ENS(c->seg_cnt, 4 * (size_t)nb); ENS(c->seg_tile0, 4 * (size_t)(nb + 1)); ENS(c->tile_blk, 4 * tiles0);
    ENS(c->tile_i0, 4 * big_tiles); ENS(c->tile_i1, 4 * big_tiles);
    ENS(c->big_cnt, 4 * (size_t)big_cap); ENS(c->big_old, 4 * (size_t)big_cap);
    ENS(c->big_rank, 4 * (size_t)big_cap); ENS(c->big_tile0, 4 * ((size_t)big_cap + 1)); ENS(c->big_tblk, 4 * big_tiles);
    ENS(c->lb_status, 8 * lb_tiles); ENS(c->lbm, 64);
    ENS(c->totals, 64); ENS(c->totals2, 64);
    u32 *seg_cnt = P<u32>(c->seg_cnt), *tile0 = P<u32>(c->seg_tile0), *tblk = P<u32>(c->tile_blk);
    u64 *kA = P<u64>(c->keysA), *kB = P<u64>(c->keysB);
    u32 *actI[2] = {P<u32>(c->actI0), P<u32>(c->actI1)}, *actR[2] = {P<u32>(c->actR0), P<u32>(c->actR1)};
    u32 *lbm = P<u32>(c->lbm);  // [0] tile ticket, [1] length of the list being written, [2] big groups of the round
    u64 *status = P<u64>(c->lb_status);
    const u64 magic = ~0ull / (u64)BS + 1;  // gidx / BS == umul64hi(gidx, magic) for gidx < 2^32
    LAUNCH(k_seg_init, (unsigned)((nb + 255) / 256), 256, 0, recs, nb, seg_cnt);
    LAUNCH(k_tilemap, 1, 1024, 0, seg_cnt, nb, tile0, tblk, P<u64>(c->totals));
    const unsigned Ta = (unsigned)tiles0;
    ENS(c->blksort, sizeof(BlkSort) * (size_t)nb);
    CK(cudaMemsetAsync(c->blksort.p, 0, sizeof(BlkSort) * (size_t)nb, c->stream));
    LAUNCH(k_sym_used, dim3(32, (unsigned)nb), 256, 0, P<u8>(c->blk), BS, recs, P<BlkSort>(c->blksort));
    LAUNCH(k_sym_tab, (unsigned)nb, 256, 0, P<BlkSort>(c->blksort));
    u64 total_n = 0;
    for (int k = 0; k < nb; k++) total_n += hrecs[k].n;
    c->dom_used = 0;
    auto timed_scatter = [&](bool bits9, unsigned grid, const u64 *ki, u64 *ko, const u32 *scnt, const u32 *st0, const u32 *stb, int shift,
                             const u32 *sbase, u64 slots_now) -> int {
      if (c->ev_ok) {
        if (c->dom_used + 2 > c->dom_ev.size()) {
          cudaEvent_t a, b2;
          CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b2));
          c->dom_ev.push_back(a); c->dom_ev.push_back(b2);
        }
        CK(cudaEventRecord(c->dom_ev[c->dom_used], c->stream));
      }
      if (bits9) LAUNCH(k_rs_scatter<9>, grid, SORT_THREADS, 0, ki, ko, scnt, st0, stb, shift, P<u32>(c->hist), P<u32>(c->digit_base), sbase);
      else LAUNCH(k_rs_scatter<8>, grid, SORT_THREADS, 0, ki, ko, scnt, st0, stb, shift, P<u32>(c->hist), P<u32>(c->digit_base), sbase);
      if (c->ev_ok) { CK(cudaEventRecord(c->dom_ev[c->dom_used + 1], c->stream)); c->dom_used += 2; }
      c->st.dom_launches++;
      c->st.dom_bytes += 16ull * slots_now;
      return 0;
    };
    u32 hv[4] = {0, 0, 0, 0};
    // ---- round 0: first keys, batched global radix sort (5 passes), then groups + ISA + active list ----
    // All blocks of the batch are sorted at once (L2-sized groups of blocks were measured slower: profiles/r02_round0_l2_groups.log).
    {
      c->st.sort_rounds++;
      c->st.sort_slots += (u64)Ta * SORT_TILE;
      CK(cudaMemsetAsync(lbm, 0, 16, c->stream));
      CK(cudaMemsetAsync(status, 0, 8 * (size_t)Ta, c->stream));
      LAUNCH(k_keys_init, Ta, SEG_THREADS, 0, P<u8>(c->blk), BS, recs, tile0, tblk, P<BlkSort>(c->blksort), kA, P<u32>(c->hist));
      u64 *ki = kA, *ko = kB;
      for (int pass = 0; pass * 9 < KEY_BITS; pass++) {  // bits 20 .. 20 + KEY_BITS, 9 bits a pass
        if (pass) LAUNCH(k_rs_hist<9>, Ta, SORT_THREADS, 0, ki, seg_cnt, tile0, tblk, 20 + pass * 9, P<u32>(c->hist), (const u32 *)nullptr);  // pass 0: k_keys_init
        LAUNCH(k_rs_scan<9>, dim3((unsigned)nb, 512 / 32), RSS_WARPS * 32, 0, P<u32>(c->hist), tile0, P<u32>(c->digit_base));
        if ((rc = timed_scatter(true, Ta, ki, ko, seg_cnt, tile0, tblk, 20 + pass * 9, nullptr, total_n))) return rc;
        u64 *tk = ki; ki = ko; ko = tk;
      }
      LAUNCH(k_rank0, Ta, R0_THREADS, 0, ki, seg_cnt, tile0, tblk, P<u32>(c->isa), BS, actI[0], actR[0], status, lbm, lbm + 1, (u32)Ta, P<u8>(c->blk),
             P<u8>(c->Lcol), recs);
      RC(rb_add(c, hv, lbm, sizeof hv));
      RC(rb_sync(c));
    }
    // ---- rounds >= 1 (refine.cuh): list A (+ key2) -> sorted staging list B -> compacted list A ----
    u32 n_act = hv[1], round = 0;  // doubling round r compares h = L << r symbols further on (L per block)
    if (n_act) LAUNCH(k_keys2, (n_act + 255) / 256, 256, 0, actI[0], n_act, recs, P<u32>(c->isa), (u32)BS, magic, P<BlkSort>(c->blksort), round,
                      P<u32>(c->key2));
    while (n_act) {
      c->st.sort_rounds++;
      c->st.sort_slots += n_act;
      const u32 ntiles = (n_act + RF_T0 - 1) / RF_T0, ctiles = (n_act + CK_TILE - 1) / CK_TILE;
      CK(cudaMemsetAsync(lbm, 0, 16, c->stream));
      CK(cudaMemsetAsync(status, 0, 8 * (size_t)ctiles, c->stream));
      ENS(c->gbounds, 8 * ((size_t)ntiles + 2));
      u32 *gb_lo = P<u32>(c->gbounds), *gb_lo2 = gb_lo + ntiles + 1;
      LAUNCH(k_group_bounds, (ntiles + 1 + 7) / 8, 256, 0, actR[0], n_act, ntiles, gb_lo, gb_lo2, P<u32>(c->big_cnt), P<u32>(c->big_old), P<u32>(c->big_rank),
             lbm + 2, big_cap);
      LAUNCH(k_sort_groups, ntiles, RF_THREADS, sizeof(RfSmem), P<u32>(c->key2), actI[0], actR[0], n_act, P<u32>(c->isa), (u32)BS, magic, actI[1],
             actR[1], P<u32>(c->big_cnt), P<u32>(c->big_old), P<u32>(c->big_rank), lbm + 2, big_cap, P<u8>(c->blk), P<u8>(c->Lcol), recs,
             gb_lo, gb_lo2);
      RC(rb_add(c, hv, lbm, sizeof hv));
      RC(rb_sync(c));
      const u32 n_big = hv[2];
      if (n_big > big_cap) { c->err = "internal: big-group list overflow"; return BZ2B200_E_CUDA; }
      if (n_big) {  // groups of more than RF_T0 slots: the global radix sort
        u32 *bcnt = P<u32>(c->big_cnt), *bbase = P<u32>(c->big_old), *bt0 = P<u32>(c->big_tile0), *btb = P<u32>(c->big_tblk);
        u64 t2[2] = {0, 0};
        LAUNCH(k_tilemap, 1, 1024, 0, bcnt, (int)n_big, bt0, btb, P<u64>(c->totals2));
        RC(rb_add(c, t2, c->totals2.p, sizeof t2));
        RC(rb_sync(c));
        const unsigned Tb = (unsigned)t2[0];
        LAUNCH(k_big_keys, Tb, SEG_THREADS, 0, P<u32>(c->key2), actI[0], bcnt, bt0, btb, bbase, kA);
        u64 *ki = kA, *ko = kB;
        for (int pass = 0; pass < 3; pass++) {  // key2 < 2^20: bits 32..55
          LAUNCH(k_rs_hist<8>, Tb, SORT_THREADS, 0, ki, bcnt, bt0, btb, 32 + pass * 8, P<u32>(c->hist), bbase);
          LAUNCH(k_rs_scan<8>, dim3(n_big, 256 / 32), RSS_WARPS * 32, 0, P<u32>(c->hist), bt0, P<u32>(c->digit_base));
          if ((rc = timed_scatter(false, Tb, ki, ko, bcnt, bt0, btb, 32 + pass * 8, bbase, t2[1]))) return rc;
          u64 *tk = ki; ki = ko; ko = tk;
        }
        LAUNCH(k_sub_heads, Tb, SEG_THREADS, 0, ki, bcnt, bt0, btb, P<int>(c->tile_i0), bbase, 32);
        LAUNCH(k_seg_scan, n_big, 256, 0, bt0, 0, P<int>(c->tile_i0), P<int>(c->tile_i1), (u32 *)nullptr);
        LAUNCH(k_big_apply, Tb, SEG_THREADS, 0, ki, bcnt, bt0, btb, bbase, P<u32>(c->big_rank), P<int>(c->tile_i1), P<u32>(c->isa), (u32)BS, magic,
               actI[1], actR[1], P<u8>(c->blk), P<u8>(c->Lcol), recs);
      }
      round = round < 30 ? round + 1 : round;
      LAUNCH(k_compact_keys, ctiles, CK_THREADS, 0, actI[1], actR[1], n_act, recs, P<u32>(c->isa), (u32)BS, magic, P<BlkSort>(c->blksort), round,
             actI[0], actR[0],
             P<u32>(c->key2), status, lbm, lbm + 1, ctiles);
      RC(rb_add(c, hv, lbm, sizeof hv));
      RC(rb_sync(c));
      n_act = hv[1];
    }
    if ((rc = mark(c, 2))) return rc;

    // ---- S3 MTF + RLE2 ----
    const i64 nseg_max = (BS + MTF_SEG - 1) / MTF_SEG;
    ENS(c->ranks, (size_t)nb * BS);
    ENS(c->lastocc, 4 * 256 * (size_t)nseg_max * nb);
    ENS(c->A, 2 * (size_t)nb * AS);
    ENS(c->freq, 4 * BZ_MAX_SYMS * (size_t)nb);
    ENS(c->used_bits, 32 * (size_t)nb);
    CK(cudaMemsetAsync(c->used_bits.p, 0, 32 * (size_t)nb, c->stream));
    LAUNCH(k_mtf_lastocc, dim3((unsigned)((nseg_max + 7) / 8), (unsigned)nb), 256, 0, P<u8>(c->Lcol), BS, recs, P<int>(c->lastocc),
           nseg_max * 256, P<u32>(c->used_bits));
    LAUNCH(k_mtf_scan, (unsigned)nb, 256, 0, recs, P<int>(c->lastocc), nseg_max * 256, P<u32>(c->used_bits), P<BlockMeta>(c->meta));
    LAUNCH(k_mtf_ranks, dim3((unsigned)((nseg_max + MTR_WARPS - 1) / MTR_WARPS), (unsigned)nb), MTR_WARPS * 32, MTR_WARPS * sizeof(MtrSmem), P<u8>(c->Lcol),
           BS, recs, P<int>(c->lastocc), nseg_max * 256, P<u8>(c->ranks));
    {
      const i64 r2_tiles = (BS + R2_TILE - 1) / R2_TILE;
      ENS(c->r2_status, 8 * (size_t)nb * r2_tiles + 4 * (size_t)nb);
      CK(cudaMemsetAsync(c->r2_status.p, 0, 8 * (size_t)nb * r2_tiles + 4 * (size_t)nb, c->stream));
      CK(cudaMemsetAsync(c->freq.p, 0, 4 * BZ_MAX_SYMS * (size_t)nb, c->stream));
      LAUNCH(k_mtf_rle2, dim3((unsigned)r2_tiles, (unsigned)nb), R2_THREADS, 0, recs, P<u8>(c->ranks), BS, P<u16>(c->A), AS, P<u32>(c->freq),
             P<BlockMeta>(c->meta), P<u64>(c->r2_status), r2_tiles, reinterpret_cast<u32 *>(P<u64>(c->r2_status) + (size_t)nb * r2_tiles));
    }
    if ((rc = mark(c, 3))) return rc;

    // ---- S4/S5 Huffman + emission (huff.cuh) ----
    u64 maxbits = 80 + 25 + 16 + 256 + 18 + 7ull * ((B + 1 + 49) / 50) + 6ull * (5 + 258 * 39) + 20ull * (B + 1);
    WS = round_up((i64)((maxbits + 31) / 32) + 2, 64);
    ENS(c->W, 4 * (size_t)nb * WS);  // zeroed per block by k_huf_codes, only as far as the block's bits reach
    const u32 max_nsel = (B + 1 + BZ_GROUP - 1) / BZ_GROUP;
    HufArrays ha;
    ha.sel_stride = round_up((i64)max_nsel + 1, 16);
    c->last_ss = ha.sel_stride;
    ENS(c->hfreq, 4 * (size_t)nb * BZ_MAX_GROUPS * BZ_MAX_SYMS);
    ENS(c->hlens, (size_t)nb * BZ_MAX_GROUPS * HUF_LSTRIDE);
    ENS(c->hplen, 8 * (size_t)nb * BZ_MAX_SYMS);
    ENS(c->hcodes, 4 * (size_t)nb * BZ_MAX_GROUPS * BZ_MAX_SYMS);
    ENS(c->hsel, (size_t)nb * ha.sel_stride);
    ENS(c->hcost, 2 * (size_t)nb * ha.sel_stride);
    ENS(c->hgoff, 4 * (size_t)nb * ha.sel_stride);
    ENS(c->hblk, sizeof(HufBlk) * (size_t)nb);
    ha.freq = P<u32>(c->hfreq); ha.lens = P<u8>(c->hlens); ha.plen = P<u64>(c->hplen); ha.codes = P<u32>(c->hcodes);
    ha.sel = P<u8>(c->hsel); ha.cost = P<u16>(c->hcost); ha.goff = P<u32>(c->hgoff); ha.hb = P<HufBlk>(c->hblk);
    const dim3 ggrid((max_nsel + HUF_GT - 1) / HUF_GT, (unsigned)nb);
    LAUNCH(k_huf_init, (unsigned)nb, HUF_BT, sizeof(HufBuildSmem), ha, P<u32>(c->freq), P<BlockMeta>(c->meta));
    for (int it = 0; it < BZ_MAX_GROUPS - 2; it++) {  // 2 -> 6 tables; blocks at their target skip
      LAUNCH(k_huf_assign, ggrid, HUF_GT, 0, ha, P<u16>(c->A), AS, 0);
      LAUNCH(k_huf_split, (unsigned)nb, HUF_BT, 0, ha);
      LAUNCH(k_huf_hist, ggrid, HUF_GT, 0, ha, P<u16>(c->A), AS);
      LAUNCH(k_huf_build, (unsigned)nb, HUF_BT, sizeof(HufBuildSmem), ha);
    }
    LAUNCH(k_huf_assign, ggrid, HUF_GT, 0, ha, P<u16>(c->A), AS, 1);  // BJ:2163
    LAUNCH(k_huf_codes, (unsigned)nb, HUF_CT, 0, ha, recs, P<BlockMeta>(c->meta), P<u32>(c->W), WS);
    LAUNCH(k_huf_emit, ggrid, HUF_GT, 0, ha, P<u16>(c->A), AS, P<u32>(c->W), WS);
  } else {
    for (int i = 1; i <= 3; i++) if ((rc = mark(c, i))) return rc;
  }
  P_.WS = WS;
  if ((rc = mark(c, 4))) return rc;
  return BZ2B200_OK;
}

// ---- batches of blocks --------------------------------------------------------------------------
// The per-block state is ~45 bytes per input byte and global indices are 31 bits, so a call with more blocks than
// fit is run as consecutive batches of whole blocks: the stages see one batch at a time (a slice of the block table)
// and every batch is stitched behind the previous one at the running bit offset.
int batch_limit(Ctx *c) {
  if (c->batch_override) return (int)c->batch_override;
  const i64 BS = round_up((i64)c->pipe.B + 1, 256);
  const i64 by_index = ((1ll << 31) - 1) / BS;
  i64 by_mem = by_index;
#ifndef BZ_SIM
  // cudaMemGetInfo takes the driver lock and was seen to cost milliseconds: asked only when this call needs more
  // than the context already holds from earlier calls
  size_t pooled = 0;
  for (DevBuf *b : c->pool) pooled += b->cap;
  const size_t need = (size_t)c->pipe.nb * (size_t)BS * 52;
  if (need > pooled) {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) by_mem = (i64)((free_b + pooled) / 10 * 7 / (size_t)(BS * 52));
  }
#endif
  i64 lim = by_index < by_mem ? by_index : by_mem;
  return (int)(lim < 1 ? 1 : lim);
}

// stages + emission of every block in the table, batch by batch.  base_bits: 32 for a whole stream (then header and
// footer are written too), 0..7 for a shard segment.  The stats of the batches add up in c->st, which pipe_begin cleared.
int pipe_run(Ctx *c, u64 base_bits, bool whole, u32 *d_out, size_t out_cap, bool own_out, size_t *out_len, u64 *bits_out, u32 *crc_fold) {
  Ctx::Pipe &P_ = c->pipe;
  const int nb = P_.nb, maxb = batch_limit(c);
  const bool batched = nb > maxb;
  if (own_out && batched) {  // sized once: growing it later would drop the bits of the earlier batches
    out_cap = bz2b200_compress_bound((size_t)P_.N, P_.level) + 64;
    ENS(c->out, out_cap);
    d_out = P<u32>(c->out);
  }
  u64 end_bits = base_bits, olen = 0;
  u32 fold = 0;  // combined CRC of the blocks so far
  int rc, b0 = 0;
  do {
    const int bn = nb - b0 < maxb ? nb - b0 : maxb;
    if (b0) { if ((rc = mark(c, 0))) return rc; if ((rc = mark(c, 1))) return rc; }  // S1 of later batches: emit + CRC only, counted from here
    if ((rc = pipe_stages(c, b0, bn))) return rc;
    const u64 base = end_bits;
    LAUNCH(k_stitch_offsets, 1, 1024, 0, P<BlockMeta>(c->meta), P<BlockRec>(c->recs) + b0, bn, P<u64>(c->bit_off), P<u32>(c->scrc), base, fold);
    RC(rb_add(c, &end_bits, P<u64>(c->bit_off) + bn, 8));
    RC(rb_add(c, &fold, c->scrc.p, 4));
    RC(rb_sync(c));
    const size_t need = (size_t)((end_bits + (whole ? 80 : 0) + 7) / 8), need_w = round_up((i64)need, 4) + 8;
    if (own_out && !batched) {
      ENS(c->out, need_w);
      d_out = P<u32>(c->out);
    } else if (out_cap < need_w) {
      c->err = "output buffer too small";
      return BZ2B200_E_UNEXPECTED_OUTPUT_EOF;
    }
    // the words this batch touches are cleared; a later batch keeps the word that holds `base` (the earlier bits)
    const size_t w_first = b0 ? (size_t)(base >> 5) + 1 : 0;
    CK(cudaMemsetAsync(d_out + w_first, 0, need_w - 4 * w_first, c->stream));
    if (bn) LAUNCH(k_stitch, dim3(32, (unsigned)bn), 256, 0, P<u32>(c->W), P_.WS, P<u64>(c->bit_off), d_out);
    olen = need;
    if (whole && b0 + bn == nb) {
      LAUNCH(k_stream_ends, 1, 32, 0, d_out, P<u64>(c->bit_off), bn, P<u32>(c->scrc), P_.level, P<u64>(c->out_len));
      RC(rb_add(c, &olen, c->out_len.p, 8));
    }
    if ((rc = mark(c, 5))) return rc;
    RC(rb_sync(c));
    CK(cudaGetLastError());
    if (bn) {
      std::vector<BlockMeta> hm((size_t)bn);
      CK(cudaMemcpy(hm.data(), c->meta.p, sizeof(BlockMeta) * (size_t)bn, cudaMemcpyDeviceToHost));
      for (auto &m : hm) { c->st.mtf_syms += m.m; c->st.d1_triggered |= m.d1; }
    }
    if (c->ev_ok) {
      float t = 0;
      for (int i = 0; i < 5; i++) { CK(cudaEventElapsedTime(&t, c->ev[i], c->ev[i + 1])); c->st.ms_stage[i] += t; }
      CK(cudaEventElapsedTime(&t, c->ev[0], c->ev[5]));
      c->st.ms_total += t;
      for (size_t i = 0; i + 1 < c->dom_used; i += 2) { CK(cudaEventElapsedTime(&t, c->dom_ev[i], c->dom_ev[i + 1])); c->st.dom_ms += t; }
    }
    b0 += bn;
  } while (b0 < nb);
  if (bits_out) *bits_out = end_bits - base_bits;
  if (crc_fold) *crc_fold = fold;
  *out_len = (size_t)olen;
  c->st.out_bytes = olen;
  return BZ2B200_OK;
}

int compress_device(Ctx *c, const u8 *d_in, size_t n_, int level, u32 *d_out, size_t out_cap, size_t *out_len, bool own_out) {
  int rc;
  if ((rc = pipe_begin(c, d_in, n_, level))) return rc;
  if ((rc = pipe_cut(c, 0, (i64)n_))) return rc;
  rc = pipe_run(c, 32, true, d_out, out_cap, own_out, out_len, nullptr, nullptr);
  trace_report(c);
  return rc;
}

// the segment of `bits` bits that pipe_run left in c->out, moved to start at bit `phase` of its first byte (into
// c->out2 when phase > 0): *d_seg = its (phase + bits + 7) / 8 bytes on the device
int seg_shift(Ctx *c, u64 bits, u32 phase, const u8 **d_seg) {
  const u64 nsrc = (bits + 7) / 8;
  *d_seg = P<u8>(c->out);
  if (phase && bits) {
    ENS(c->out2, nsrc + 16);
    LAUNCH(k_shift_bytes, (unsigned)((nsrc + 256) / 256), 256, 0, P<u8>(c->out), nsrc, phase, P<u8>(c->out2));
    *d_seg = P<u8>(c->out2);
  }
  return 0;
}

#include "decode_host.inl"
#include "pool.inl"

// The opt-in for more than 48 KB of dynamic shared memory is a per-DEVICE function attribute: set for the current
// device by every bz2b200_create (contexts on several GPUs in one process each set their own).
cudaError_t set_kernel_attributes() {
#ifndef BZ_SIM
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(k_sort_groups, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RfSmem))) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_mtf_ranks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(MTR_WARPS * sizeof(MtrSmem)))) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_huf_init, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HufBuildSmem))) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_huf_build, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(HufBuildSmem))) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_huff_parse_win, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DecWinSmem))) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(k_ibwt_rank, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IBWT_RANK_SMEM)) != cudaSuccess) return e;
#endif
  return cudaSuccess;
}

int ctx_new(int device, Ctx **out) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return BZ2B200_E_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return BZ2B200_E_CUDA;
  Ctx *c = new Ctx();
  c->device = device;
  if (cudaStreamCreate(&c->stream) != cudaSuccess) { delete c; return BZ2B200_E_CUDA; }
  c->ev_ok = true;
  { const char *t = getenv("BZ2B200_TRACE"); c->trace = t && *t && *t != '0'; }
  { const char *t = getenv("BZ2B200_PARSE"); c->parse_mode = t ? atoi(t) : 0; }
  { int v = 0; if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) c->sms = v; }
  for (auto &e : c->ev) if (cudaEventCreate(&e) != cudaSuccess) c->ev_ok = false;
  if (set_kernel_attributes() != cudaSuccess) { ctx_delete(c); return BZ2B200_E_CUDA; }
  *out = c;
  return BZ2B200_OK;
}

void ctx_delete(Ctx *c) {
  if (!c) return;
  if (c->own_pool) pool_delete(c->own_pool);
  cudaSetDevice(c->device);
  for (DevBuf *b : c->pool) if (b->p) cudaFree(b->p);
  if (c->rb_pin) cudaFreeHost(c->rb_pin);
  for (auto &e : c->ev) if (e) cudaEventDestroy(e);
  for (auto &e : c->dom_ev) cudaEventDestroy(e);
  for (auto &e : c->trace_pool) cudaEventDestroy(e);
  cudaStreamDestroy(c->stream);
  delete c;
}

}  // namespace

// ------------------------------------------------------------------------------------ C ABI
extern "C" {

int bz2b200_create(int device, bz2b200_ctx **ctx) {
  if (!ctx) return BZ2B200_E_ARG;
  *ctx = nullptr;
  Ctx *c = nullptr;
  int rc = ctx_new(device, &c);
  if (rc) return rc;
  *ctx = reinterpret_cast<bz2b200_ctx *>(c);
  return BZ2B200_OK;
}

void bz2b200_destroy(bz2b200_ctx *ctx) { ctx_delete(reinterpret_cast<Ctx *>(ctx)); }

int bz2b200_compress_device(bz2b200_ctx *ctx, const void *d_in, size_t n, int level, void *d_out, size_t out_cap, size_t *out_len) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !out_len || (n && !d_in) || !d_out || ((uintptr_t)d_in & 15) || ((uintptr_t)d_out & 3)) return BZ2B200_E_ARG;
  CK(cudaSetDevice(c->device));
  return compress_device(c, (const u8 *)d_in, n, level, (u32 *)d_out, out_cap, out_len, false);
}

int bz2b200_compress(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level, uint8_t **out, size_t *out_len) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !out || !out_len || (n && !in)) return BZ2B200_E_ARG;
  if (level < 1 || level > 9) return BZ2B200_E_LEVEL;
  CK(cudaSetDevice(c->device));
  if (n >= c->pool_min_bytes) {
    // large input: shards over two lanes of this device, so that the copies in both directions hide under the kernels
    if (!c->own_pool) {
      const int dev = c->device;
      int prc = pool_new(&dev, 1, 2, &c->own_pool);
      if (prc) { c->err = "cannot create the lanes of the context's pool"; return prc; }
    }
    Pool *p = c->own_pool;
    p->cap_override = c->cap_override; p->batch_override = c->batch_override;
    p->halo0 = c->pool_halo0; p->force_staging = c->pool_force_staging;
    p->plan_first = n / 5 * 2 + 1;  // one device, two lanes: two shards of 40 / 60 % measured best (profiles/r02_pool_two_shard_plans_n1.log)
    p->plan_growth = 1000.0;
    int prc = pool_compress_whole(p, in, n, level, c->pool_shard_bytes, out, out_len);
    c->st = p->st;
    c->err = p->err;
    return prc;
  }
  ENS(c->in, n + 64);
  if (n) CK(cudaMemcpyAsync(c->in.p, in, n, cudaMemcpyHostToDevice, c->stream));
  size_t olen = 0;
  int rc = compress_device(c, P<u8>(c->in), n, level, nullptr, 0, &olen, true);
  if (rc) return rc;
  uint8_t *res = (uint8_t *)result_pool().get(olen);
  if (!res) return BZ2B200_E_OUT_OF_MEMORY;
  CK(cudaMemcpy(res, c->out.p, olen, cudaMemcpyDeviceToHost));
  *out = res;
  *out_len = olen;
  return BZ2B200_OK;
}

int bz2b200_shard_begin(bz2b200_ctx *ctx, const void *in, size_t n_avail, int on_device, int level) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || (n_avail && !in)) return BZ2B200_E_ARG;
  if (level < 1 || level > 9) return BZ2B200_E_LEVEL;
  CK(cudaSetDevice(c->device));
  const u8 *d_in = (const u8 *)in;
  if (!on_device) {
    ENS(c->in, n_avail + 64);
    if (n_avail) CK(cudaMemcpyAsync(c->in.p, in, n_avail, cudaMemcpyHostToDevice, c->stream));
    d_in = P<u8>(c->in);
  } else if ((uintptr_t)in & 15) return BZ2B200_E_ARG;
  return pipe_begin(c, d_in, n_avail, level);
}

static void shard_fill_info(Ctx *c, i64 s_start, int is_last, bz2b200_shard_info *info) {
  *info = bz2b200_shard_info{};
  const auto &h = c->pipe.hrecs;
  info->n_blocks = (uint32_t)h.size();
  info->next_start = h.empty() ? (uint64_t)(s_start < 0 ? 0 : s_start) : (uint64_t)h.back().p;
  info->complete = 1;
  if (!is_last && !h.empty() && h.back().p == c->pipe.N && h.back().n < c->pipe.B) info->complete = 0;  // halo too short
}

int bz2b200_shard_cut(bz2b200_ctx *ctx, uint64_t s_start, uint64_t own_len, int is_last, bz2b200_shard_info *info) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !info) return BZ2B200_E_ARG;
  CK(cudaSetDevice(c->device));
  if ((i64)own_len > c->pipe.N) own_len = (uint64_t)c->pipe.N;
  int rc = pipe_cut(c, (i64)s_start, (i64)own_len);
  if (rc) return rc;
  shard_fill_info(c, (i64)s_start, is_last, info);
  return BZ2B200_OK;
}

int bz2b200_shard_gtotal(bz2b200_ctx *ctx, uint64_t pos, uint64_t *g) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !g) return BZ2B200_E_ARG;
  CK(cudaSetDevice(c->device));
  const i64 N = c->pipe.N;
  *g = 0;
  if (N == 0) return BZ2B200_OK;
  ENS(c->nblk, 64 + 4 * CUT_CANDIDATES);
  LAUNCH(k_rle_gquery, 1, 32, 0, c->pipe.d_in, N, P<u32>(c->g_sub), P<i64>(c->h_sub), P<u64>(c->g_tile), c->pipe.T, (i64)(pos > (uint64_t)N ? (uint64_t)N : pos),
         P<u64>(c->nblk) + 1);
  u64 v = 0;
  RC(rb_add(c, &v, P<u64>(c->nblk) + 1, 8));
  RC(rb_sync(c));
  *g = v;
  return BZ2B200_OK;
}

int bz2b200_shard_cut_g(bz2b200_ctx *ctx, uint64_t g_before, uint64_t own_len) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c) return BZ2B200_E_ARG;
  CK(cudaSetDevice(c->device));
  c->cand_n = 0;
  if (c->pipe.N == 0) return BZ2B200_OK;
  if ((i64)own_len > c->pipe.N) own_len = (uint64_t)c->pipe.N;
  const u64 B = c->pipe.B, g_start = (B - g_before % B) % B;  // G still missing to the next multiple of B
  ENS(c->cand_first, 8 * CUT_CANDIDATES);
  return pipe_cut(c, 0, (i64)own_len, (i64)g_start);
}

int bz2b200_shard_cut_pick(bz2b200_ctx *ctx, uint64_t s_start, uint64_t own_len, int is_last, bz2b200_shard_info *info, int *found) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !info || !found) return BZ2B200_E_ARG;
  CK(cudaSetDevice(c->device));
  if ((i64)own_len > c->pipe.N) own_len = (uint64_t)c->pipe.N;
  int rc = BZ2B200_OK;
  *found = pipe_pick(c, (i64)s_start, (i64)own_len, rc) ? 1 : 0;
  if (rc) return rc;
  if (*found) shard_fill_info(c, (i64)s_start, is_last, info);
  return BZ2B200_OK;
}

int bz2b200_shard_compress(bz2b200_ctx *ctx, bz2b200_shard_info *info) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !info) return BZ2B200_E_ARG;
  CK(cudaSetDevice(c->device));
  // the segment is stitched at bit phase 0 now (in batches if need be); shard_emit moves it to its real phase
  size_t olen = 0;
  u64 bits = 0;
  u32 fold = 0;
  int rc = pipe_run(c, 0, false, nullptr, 0, true, &olen, &bits, &fold);
  if (rc) return rc;
  c->shard_bits = bits;
  info->bits = bits;
  info->crc_fold = fold;
  return BZ2B200_OK;
}

int bz2b200_shard_emit(bz2b200_ctx *ctx, int bit_phase, bz2b200_shard_info *info, uint8_t **seg, size_t *seg_bytes) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !info || !seg_bytes || bit_phase < 0 || bit_phase > 7) return BZ2B200_E_ARG;
  CK(cudaSetDevice(c->device));
  const u64 bits = c->shard_bits;
  const size_t olen = (size_t)(((u64)bit_phase + bits + 7) / 8);
  const u8 *d_seg = nullptr;
  RC(seg_shift(c, bits, (u32)bit_phase, &d_seg));
  CK(cudaStreamSynchronize(c->stream));
  info->bit_phase = (uint32_t)bit_phase;
  *seg_bytes = olen;
  if (!seg) return BZ2B200_OK;  // segment stays in HBM (device-resident timing)
  uint8_t *res = (uint8_t *)result_pool().get(olen);
  if (!res) return BZ2B200_E_OUT_OF_MEMORY;
  if (olen) CK(cudaMemcpy(res, d_seg, olen, cudaMemcpyDeviceToHost));
  *seg = res;
  *seg_bytes = olen;
  return BZ2B200_OK;
}

// Host-side assembly of the final stream (pure byte copies; the segments are already bit-aligned by shard_emit).
int bz2b200_stitch_shards(int level, int n_shards, const uint8_t *const *segs, const bz2b200_shard_info *infos, uint8_t **out, size_t *out_len) {
  if (level < 1 || level > 9) return BZ2B200_E_LEVEL;
  if (n_shards < 0 || !out || !out_len || (n_shards && (!segs || !infos))) return BZ2B200_E_ARG;
  u64 total_bits = 32;
  for (int r = 0; r < n_shards; r++) total_bits += infos[r].bits;
  size_t nbytes = (size_t)((total_bits + 80 + 7) / 8);
  uint8_t *o = (uint8_t *)calloc(nbytes + 8, 1);
  if (!o) return BZ2B200_E_OUT_OF_MEMORY;
  stream_header(o, level);
  u64 bitpos = 32;
  u32 crc = 0;
  for (int r = 0; r < n_shards; r++) {
    if (infos[r].bits) {
      if (infos[r].bit_phase != (u32)(bitpos & 7)) { free(o); return BZ2B200_E_ARG; }
      size_t off = (size_t)(bitpos >> 3), len = (size_t)((infos[r].bit_phase + infos[r].bits + 7) / 8);
      o[off] |= segs[r][0];
      if (len > 1) memcpy(o + off + 1, segs[r] + 1, len - 1);
      bitpos += infos[r].bits;
    }
    crc = stream_crc_add(crc, infos[r].n_blocks, infos[r].crc_fold);
  }
  bitpos = stream_footer(o, bitpos, crc);
  *out = o;
  *out_len = (size_t)((bitpos + 7) / 8);
  return BZ2B200_OK;
}

size_t bz2b200_compress_bound(size_t n, int level) {
  if (level < 1 || level > 9) level = 9;
  size_t B = (size_t)level * 100000 - 19;
  size_t nblocks = n / (B * 4 / 5) + 2;
  // RLE1 expands by at most 5/4 (a run of exactly four bytes becomes five), a block adds its end-of-block symbol, and a
  // table never costs more than 9 bits per symbol on the groups it was built from (a fixed 9-bit code is admissible for
  // <= 258 symbols and the allocator's lengths are optimal under the 20-bit limit; the final selector pass only lowers the
  // cost).  Per block: header 105 bits + maps 272 + 18 + selectors 18 002 x 6 bits + six tables of 5 + 258 x 39 bits.
  return (n + n / 4 + nblocks) / 8 * 9 + nblocks * 22000 + 1024;
}

void bz2b200_free(void *p) { result_pool().put(p); }

const char *bz2b200_strerror(int rc) {
  switch (rc) {  // messages of BJ:1376-1383
    case BZ2B200_OK: return "OK";
    case BZ2B200_E_LAST_BLOCK: return "Bad file checksum";
    case BZ2B200_E_NOT_BZIP_DATA: return "Not bzip data";
    case BZ2B200_E_UNEXPECTED_INPUT_EOF: return "Unexpected input EOF";
    case BZ2B200_E_UNEXPECTED_OUTPUT_EOF: return "Unexpected output EOF";
    case BZ2B200_E_DATA_ERROR: return "Data error";
    case BZ2B200_E_OUT_OF_MEMORY: return "Out of memory";
    case BZ2B200_E_OBSOLETE_INPUT: return "Obsolete (pre 0.9.5) bzip format not supported.";
    case BZ2B200_E_LEVEL: return "Invalid block size multiplier";
    case BZ2B200_E_CUDA: return "CUDA failure";
    case BZ2B200_E_ARG: return "bad argument";
    case BZ2B200_E_PEER: return "a peer of the shard group failed or timed out";
    default: return "unknown error";
  }
}

const char *bz2b200_last_error(bz2b200_ctx *ctx) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  return c ? c->err.c_str() : "no context";
}

int bz2b200_last_stats(bz2b200_ctx *ctx, bz2b200_stats *st) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !st) return BZ2B200_E_ARG;
  *st = c->st;
  return BZ2B200_OK;
}

long long bz2b200_debug_fetch(bz2b200_ctx *ctx, int what, int blk, void *dst, size_t cap) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !dst) return BZ2B200_E_ARG;
  const void *src = nullptr;
  size_t bytes = 0;
  int nb = c->last_nb;
  if (what >= 1 && what <= 6 && what != 4 && (blk < 0 || blk >= nb)) return BZ2B200_E_ARG;
  if (what >= 8 && what <= 10 && (blk < 0 || (u32)blk >= c->dec_last_ncand)) return BZ2B200_E_ARG;
  if (what == 11 && (blk < 0 || (size_t)blk >= c->dec_last_chain.size())) return BZ2B200_E_ARG;
  if (what == 12) {  // host copy
    bytes = 4 * c->dec_last_chain.size();
    if (bytes > cap) bytes = cap;
    if (bytes) memcpy(dst, c->dec_last_chain.data(), bytes);
    return (long long)bytes;
  }
  switch (what) {
    case 0: src = c->recs.p; bytes = sizeof(BlockRec) * (size_t)c->pipe.nb; break;
    case 1: src = P<u8>(c->blk) + (i64)blk * c->last_bs; bytes = (size_t)c->last_bs; break;
    case 2: src = P<u8>(c->Lcol) + (i64)blk * c->last_bs; bytes = (size_t)c->last_bs; break;
    case 3: src = P<u16>(c->A) + (i64)blk * c->last_as; bytes = 2 * (size_t)c->last_as; break;
    case 4: src = c->meta.p; bytes = sizeof(BlockMeta) * (size_t)nb; break;
    case 5: src = P<u8>(c->hsel) + (i64)blk * c->last_ss; bytes = (size_t)c->last_ss; break;
    case 6: src = P<u8>(c->hlens) + (i64)blk * BZ_MAX_GROUPS * HUF_LSTRIDE; bytes = BZ_MAX_GROUPS * HUF_LSTRIDE; break;
    case 7: src = c->dmeta.p; bytes = sizeof(DecBlk) * (size_t)c->dec_last_ncand; break;
    case 8: src = P<u16>(c->dsyms) + (i64)blk * DEC_SYM_STRIDE; bytes = 2 * (size_t)DEC_SYM_STRIDE; break;
    case 9: src = P<u32>(c->doff) + (i64)blk * DEC_SYM_STRIDE; bytes = 4 * (size_t)DEC_SYM_STRIDE; break;
    case 10: {
      const i64 LS = round_up(DEC_DBUF_MAX + 1024, 256);  // as in dec_parse
      src = P<u8>(c->dL) + (i64)blk * LS; bytes = (size_t)LS;
      break;
    }
    case 11: src = P<u8>(c->dblk) + (i64)blk * c->dec_last_bs; bytes = (size_t)c->dec_last_bs; break;
    default: return BZ2B200_E_ARG;
  }
  if (bytes > cap) bytes = cap;
  if (bytes && cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) return BZ2B200_E_CUDA;
  return (long long)bytes;
}

int bz2b200_debug_huffman_lengths(bz2b200_ctx *ctx, int32_t *a, int n, int maxlen) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || !a || n < 0 || n > 1 << 20 || maxlen < 1 || maxlen > 32) return BZ2B200_E_ARG;
  CK(cudaSetDevice(c->device));
  if (!n) return BZ2B200_OK;
  ENS(c->dmisc, 4 * (size_t)n + 64);
  CK(cudaMemcpyAsync(c->dmisc.p, a, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  LAUNCH(k_debug_ha_allocate, 1, 32, 0, P<int>(c->dmisc), n, maxlen);
  CK(cudaMemcpyAsync(a, c->dmisc.p, 4 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return BZ2B200_OK;
}

int bz2b200_debug_set_batch_blocks(bz2b200_ctx *ctx, uint32_t blocks) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c) return BZ2B200_E_ARG;
  c->batch_override = blocks;
  return BZ2B200_OK;
}

int bz2b200_debug_set_ignore_block_crc(bz2b200_ctx *ctx, int on) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c) return BZ2B200_E_ARG;
  c->ignore_block_crc = on != 0;
  return BZ2B200_OK;
}

int bz2b200_debug_set_block_cap(bz2b200_ctx *ctx, uint32_t cap) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || (cap && cap < 8) || cap > 899981) return BZ2B200_E_ARG;
  c->cap_override = cap;
  return BZ2B200_OK;
}

int bz2b200_debug_set_search_tile(bz2b200_ctx *ctx, uint32_t bytes) {
  Ctx *c = reinterpret_cast<Ctx *>(ctx);
  if (!c || bytes % SEARCH_THREADS || bytes > SEARCH_TILE_MAX) return BZ2B200_E_ARG;
  c->search_tile = bytes;
  return BZ2B200_OK;
}

#include "decode_abi.inl"
#include "pool_abi.inl"
#include "stream_abi.inl"

}  // extern "C"
