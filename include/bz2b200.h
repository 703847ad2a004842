/*
 * bz2b200.h -- C ABI of the B200-native bzip2 block compressor / decompressor.
 *
 * This is the drop-in boundary for the bzip2 path of compressjs
 * (BJ = /root/reference/Bzip2_joined_.js).  Every entry point is what an FFI for that
 * path binds (N-API addon for the JS shim, ctypes in this repo's tests); plain pointers
 * and sizes only.  Return value: 0 or the reference's negative Err codes (BJ:1365-1375),
 * BZ2B200_E_LEVEL for `Invalid block size multiplier` (BJ:2208), BZ2B200_E_CUDA for a
 * device failure.  No exceptions cross the ABI.  Calls are blocking, like the JS API.
 *
 *   replaces                               entry point
 *   Bzip2.compressFile   (BJ:2199-2249)    bz2b200_compress / bz2b200_compress_device
 *   Bzip2.decompressFile (BJ:1769-1796)    bz2b200_decompress / bz2b200_decompress_device
 *   Bzip2.decompressBlock(BJ:1797-1818)    bz2b200_decompress_block
 *   Bzip2.table          (BJ:1823-1863)    bz2b200_table
 *   Err / ErrorMessages  (BJ:1365-1383)    bz2b200_strerror
 *   (bzip2recover: no counterpart in BJ)   bz2b200_recover
 *   (random access: no counterpart in BJ)  bz2b200_index / bz2b200_decompress_ranges
 *   (bzgrep: no counterpart in BJ)         bz2b200_search
 *   (sed -n by line: no counterpart in BJ) bz2b200_line_index / bz2b200_decompress_lines
 *   (an index while compressing: none)     bz2b200_compress_indexed / bz2b200_pool_compress_indexed /
 *                                          bz2b200_zstream_open_indexed + bz2b200_zstream_index
 */
#ifndef BZ2B200_H
#define BZ2B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  BZ2B200_OK = 0,
  BZ2B200_E_LAST_BLOCK = -1,
  BZ2B200_E_NOT_BZIP_DATA = -2,
  BZ2B200_E_UNEXPECTED_INPUT_EOF = -3,
  BZ2B200_E_UNEXPECTED_OUTPUT_EOF = -4,
  BZ2B200_E_DATA_ERROR = -5,
  BZ2B200_E_OUT_OF_MEMORY = -6,
  BZ2B200_E_OBSOLETE_INPUT = -7,
  BZ2B200_E_END_OF_BLOCK = -8,
  BZ2B200_E_LEVEL = -100,   /* Error('Invalid block size multiplier') */
  BZ2B200_E_CUDA = -101,    /* CUDA runtime failure; see bz2b200_last_error */
  BZ2B200_E_ARG = -102,
  BZ2B200_E_PEER = -103     /* a peer of the shard group failed, or did not answer before the deadline */
};

typedef struct bz2b200_ctx bz2b200_ctx;

typedef struct {
  uint64_t in_bytes, out_bytes;
  uint32_t n_blocks;
  uint32_t sort_rounds;      /* prefix-doubling rounds of the last compress */
  uint64_t rle1_bytes;       /* sum of block lengths after RLE1 */
  uint64_t mtf_syms;         /* sum of nMTF */
  uint64_t sort_slots;       /* sum over rounds of slots sorted */
  uint32_t kernel_launches;  /* kernels launched by the last call */
  uint32_t d1_triggered;
  float ms_total;            /* device time of the last call (CUDA events) */
  float ms_stage[8];         /* compress: rle1, bwt, mtf, huff, stitch; decompress: scan, huff, ibwt, out */
  /* dominant kernel of the last compress (k_rs_scatter, the radix-sort scatter pass), timed live with
   * CUDA events on the launching stream; bytes = algorithmic bytes (16 B per sorted key per pass: 8 read + 8 written) */
  float dom_ms;
  uint32_t dom_launches;
  uint64_t dom_bytes;
} bz2b200_stats;

/* One context per calling thread / per GPU.  `device` = CUDA ordinal. */
int bz2b200_create(int device, bz2b200_ctx **ctx);
void bz2b200_destroy(bz2b200_ctx *ctx);

/* Host-buffer entry points (what the JS shim / ctypes call).  The input is caller-owned and
 * only read; *out is allocated by the library and released with bz2b200_free. */
int bz2b200_compress(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level, uint8_t **out, size_t *out_len);
int bz2b200_decompress(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int multistream, uint8_t **out, size_t *out_len);
int bz2b200_decompress_block(bz2b200_ctx *ctx, const uint8_t *in, size_t n, uint64_t bitpos, uint8_t **out, size_t *out_len);
int bz2b200_table(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int multistream, uint64_t **bitpos, uint32_t **sizes, size_t *count);
void bz2b200_free(void *p);

/* Recovery of a damaged file (what bzip2recover + bunzip2 of its pieces do, without stopping at damage).  The input is
 * read as a sequence of streams (like multistream = 1).  *out = the bytes of every RECOVERED block, in input order: a
 * block that decodes without error, fits its stream's block size (BZh<level>; 9 if that header is damaged) and whose CRC
 * equals the one in its header.  *regions tiles the input bits [0, 8n) in order:
 *   HEADER   the 4 header bytes (looked for at byte 0 and after a recognised footer)
 *   BLOCK    a block from its signature (or from where its predecessor ends) up to the next region
 *   END      end-of-stream signature, stream CRC, padding; status 0 only if every block of the stream was recovered and
 *            the stored CRC equals their fold
 *   UNKNOWN  bits nothing recognised claims (garbage, bits after a damaged header up to the first signature)
 * status = 0 or the BZ2B200_E_* code that condemned the region (a bad CRC or an oversized block: DATA_ERROR; UNKNOWN and
 * damaged headers: NOT_BZIP_DATA).  A block whose signature is damaged is still parsed where the region before it ends
 * if that region is a recovered block or an intact header: it is flagged BZ2B200_REGION_NO_SIGNATURE.  After a lost
 * block the walk goes on at the next signature.  Returns 0 whenever the call ran, whatever was lost; both arrays are
 * released with bz2b200_free.  bz2b200_last_stats: n_blocks = blocks recovered, out_bytes, ms_total. */
enum { BZ2B200_REGION_HEADER = 0, BZ2B200_REGION_BLOCK = 1, BZ2B200_REGION_END = 2, BZ2B200_REGION_UNKNOWN = 3 };
#define BZ2B200_REGION_NO_SIGNATURE 1u
typedef struct {
  uint64_t bit_begin, bit_end;   /* [bit_begin, bit_end) of the input */
  uint64_t out_offset;           /* where the region's bytes are (or would be) in *out */
  uint32_t out_bytes, crc;       /* bytes recovered from it; CRC stored in a BLOCK / END region */
  int32_t status;
  uint32_t kind, stream, flags;  /* stream = END regions before this one */
} bz2b200_region;
int bz2b200_recover(bz2b200_ctx *ctx, const uint8_t *in, size_t n, uint8_t **out, size_t *out_len, bz2b200_region **regions, size_t *n_regions);

/* Random access to the decompressed bytes.  bz2b200_index walks the input like bz2b200_table (same batches, same error
 * codes) and returns one entry per block in stream order; *entries is released with bz2b200_free.
 * bz2b200_decompress_ranges returns the bytes [starts[i], starts[i] + lens[i]) of the decompressed output (streams
 * concatenated), for every i, concatenated in request order: *out_len = sum of lens.  Ranges may overlap, repeat, come in
 * any order or be empty.  Only the blocks that cover a range are decoded, each once, and only their compressed bytes are
 * uploaded (one span per run of consecutive covering blocks, from byte bit_begin / 8 to byte (bit_end + 7) / 8); a block
 * of a later stream decodes at its entry's level.  BZ2B200_E_ARG: a range outside [0, total) (total = out_offset +
 * out_bytes of the last entry), entries not sorted by bit_begin or overlapping, out_offset not contiguous from 0, a
 * level outside 1..9, a bit_end not above bit_begin or past 8n.  Otherwise the first failing covering block in index
 * order decides: no signature at bit_begin -> NOT_BZIP_DATA (like decompress_block); a parse error or a block larger
 * than its level allows -> that code (also a stale index whose block runs on into the next uploaded span); a bad block
 * CRC -> DATA_ERROR; an end bit or size that differs from the entry, or a parse that runs past the uploaded bytes where
 * the input goes on -> DATA_ERROR "index does not match the input" (a stale index).  The stream CRC is NOT checked: a
 * partial read cannot see every block of a stream.  bz2b200_last_stats: n_blocks = blocks decoded, in_bytes = bytes
 * uploaded, out_bytes, ms_total (device time up to the packed result; its copy to the host is not included). */
typedef struct {
  uint64_t bit_begin;    /* first bit of the block signature (what bz2b200_table reports) */
  uint64_t bit_end;      /* first bit after the block (next signature or end-of-stream signature) */
  uint64_t out_offset;   /* first decoded byte of the block in the decompressed output (streams concatenated) */
  uint32_t out_bytes;    /* decoded bytes (bz2b200_table's size) */
  uint32_t crc;          /* stored block CRC */
  uint32_t stream;       /* 0-based stream the block belongs to */
  uint32_t level;        /* that stream's BZh level, 1..9 */
} bz2b200_block_entry;
int bz2b200_index(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int multistream, bz2b200_block_entry **entries, size_t *count);
int bz2b200_decompress_ranges(bz2b200_ctx *ctx, const uint8_t *in, size_t n, const bz2b200_block_entry *index, size_t count,
                              const uint64_t *starts, const uint64_t *lens, size_t n_ranges, uint8_t **out, size_t *out_len);

/* Lines by number.  Line i (0-based) of the decompressed output (streams concatenated) runs from just after the i-th '\n'
 * (or from byte 0) through the next '\n', or to the output's end for a last line without one; only '\n' ends a line.
 * total_lines = the '\n' bytes, plus 1 when the output is not empty and its last byte is not '\n' (0 for an empty output).
 * bz2b200_line_index decodes the input exactly as bz2b200_decompress(ctx, in, n, multistream) decodes it -- same walk,
 * block and stream CRC checks, error codes -- so the whole output must fit in device memory, as for bz2b200_search.  It
 * returns the block index (*entries equals bz2b200_index's for an intact input) and, in a parallel array, the '\n' bytes of
 * every block; *entries and *newlines are released with bz2b200_free.  The '\n' bytes are counted on the GPU where the
 * decode leaves the output, by a newline directory (per-tile counts and their prefix, rank and select queries).
 * bz2b200_decompress_lines returns the lines [firsts[i], firsts[i] + counts[i]) for every i, concatenated in request order,
 * byte for byte as they are in the output (no '\n' is added to a last line without one).  Requests may overlap, repeat,
 * come in any order, be empty or cover every line.  Only the blocks from the one that holds '\n' firsts[i] - 1 to the one
 * that holds '\n' firsts[i] + counts[i] - 1 are decoded, each once, as bz2b200_decompress_ranges decodes its covering
 * blocks (same uploads, checks and error codes).  out == NULL: nothing is gathered or returned (out_len may be NULL too).
 * spans (NULL: skipped): 2 * n_requests u64, the byte start and length of each request in the output -- what
 * bz2b200_decompress_ranges takes.  BZ2B200_E_ARG: an entry bz2b200_decompress_ranges rejects, a newlines[i] above
 * out_bytes, a total_lines other than the sum of newlines[] (or that sum + 1 for a non-empty output; 1 when the sum is 0),
 * a request past total_lines.  A covered block whose '\n' count differs from newlines[], or a last byte that disagrees with
 * total_lines, is DATA_ERROR "index does not match the input".  bz2b200_last_stats: n_blocks = blocks decoded, in_bytes =
 * bytes uploaded, out_bytes = bytes of the requested lines, ms_total as bz2b200_decompress_ranges, ms_stage[5] = device time
 * of the newline-directory kernels alone (also for bz2b200_line_index). */
int bz2b200_line_index(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int multistream, bz2b200_block_entry **entries, uint32_t **newlines,
                       size_t *count, uint64_t *total_lines);
int bz2b200_decompress_lines(bz2b200_ctx *ctx, const uint8_t *in, size_t n, const bz2b200_block_entry *index, const uint32_t *newlines, size_t count,
                             uint64_t total_lines, const uint64_t *firsts, const uint64_t *counts, size_t n_requests, uint8_t **out, size_t *out_len,
                             uint64_t *spans);
/* The line index as a by-product of compression, with no decode.  bz2b200_compress_indexed returns what
 * bz2b200_compress(ctx, in, n, level) returns -- the same stream bytes, return codes and errors, also through the two-lane
 * route of inputs of 32 MB or more -- and the line index of that stream: *entries, *newlines, *count and *total_lines equal
 * what bz2b200_line_index(stream, multistream = 0) returns for it (stream = 0 and the call's level in every entry).  The
 * compressor knows every field: block i decodes to exactly its input bytes [s, p), its bits are where the stitch puts
 * them and its CRC is the one it writes; the '\n' bytes of each block are counted on the GPU in the input it already holds
 * (k_index_rows, once per batch of blocks).  The index describes the input and the emitted bits: when a block reproduces
 * defect D1 (DESIGN.md section 2, a stream the reference's own decoder rejects) the stream is still the reference's and
 * the index is still the one computed from the input (stats d1_triggered set); nothing is decoded to check it.  An empty
 * input gives count 0 and total_lines 0.  The four index outputs are required (NULL: BZ2B200_E_ARG); they are released
 * with bz2b200_free.  On any error nothing is returned.  bz2b200_last_stats: as for bz2b200_compress, except that
 * kernel_launches also counts the index kernel (one launch per batch of blocks) and ms_stage[5] is its device time, summed
 * over the batches (and over the lanes for a pool).
 * bz2b200_pool_compress_indexed is bz2b200_pool_compress with the same index.  The stream flavour: a zstream opened with
 * bz2b200_zstream_open_indexed feeds and finishes exactly as one from bz2b200_zstream_open; once bz2b200_zstream_finish
 * has succeeded, bz2b200_zstream_index returns the index of the whole stream (BZ2B200_E_ARG, with a message in
 * bz2b200_last_error of the zstream's context, before that or on a zstream opened without an index).
 * Not indexed: bz2b200_compress_device, the ranked and group shard calls (bz2b200_pool_compress_shards, bz2b200_shard_*;
 * bz2b200_shard_result keeps its layout), and the JavaScript addon and shim. */
int bz2b200_compress_indexed(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level, uint8_t **out, size_t *out_len, bz2b200_block_entry **entries,
                             uint32_t **newlines, size_t *count, uint64_t *total_lines);

/* Fixed-string search of the decompressed output (what bzgrep -F does, without bringing the decoded bytes back).  The
 * input is decoded exactly as bz2b200_decompress(ctx, in, n, multistream) decodes it -- same walk, CRC checks and error
 * codes; on an error nothing is returned.  patterns: n_patterns byte strings packed one after the other, pattern_lens[i]
 * bytes each; any byte is allowed ('\n' and NUL too).  1 <= n_patterns <= 256 and 1 <= length <= 256, otherwise
 * BZ2B200_E_ARG (bz2b200_last_error says which).  flags: BZ2B200_SEARCH_IGNORE_CASE.
 * Every occurrence of every pattern is a match: overlapping ones, each occurrence of a pattern listed twice, and matches
 * across block or stream boundaries.  Matches are sorted by offset, then by pattern; *matches holds the first
 * min(total, max_matches) of them (max_matches = 0: counts only).  totals->matches counts all matches and totals->lines
 * the distinct lines in which a match starts, exact whatever max_matches is; totals->out_bytes is the decoded size.
 * lines (NULL: skipped): the distinct lines that hold the start of a returned match, in order, each followed by one '\n'
 * (for patterns without '\n', what grep -F prints, -i with IGNORE_CASE in the C locale).  *matches and *lines are
 * released with bz2b200_free.  bz2b200_last_stats: n_blocks, in_bytes and out_bytes as bz2b200_decompress; ms_total =
 * device time up to the packed results (their copy to the host is not included); ms_stage[5] = device time of the
 * search kernels and the line gather alone.
 * bz2b200_pool_search (with the shard scheduler below) searches one stream over every lane of a pool and returns what
 * bz2b200_search returns for the same arguments, byte for byte. */
#define BZ2B200_SEARCH_IGNORE_CASE 1u      /* ASCII: A-Z equal a-z; every other byte compares as it is */
#define BZ2B200_MATCH_FIRST_IN_LINE 1u     /* bz2b200_match.flags */
typedef struct {
  uint64_t offset;      /* first byte of the match in the decompressed output (streams concatenated) */
  uint64_t line;        /* '\n' bytes before offset: the 0-based line number */
  uint64_t line_begin;  /* first byte of that line */
  uint64_t line_end;    /* the '\n' that ends the line, or the output's length when the last line has none */
  uint32_t pattern;     /* index of the pattern in the request */
  uint32_t flags;       /* BZ2B200_MATCH_FIRST_IN_LINE: the first match of its line in the order above (no match starts
                           earlier in the line, and none at the same offset has a lower pattern index) */
} bz2b200_match;
typedef struct { uint64_t matches, lines, out_bytes; } bz2b200_search_totals;
int bz2b200_search(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int multistream, const uint8_t *patterns, const uint32_t *pattern_lens,
                   size_t n_patterns, unsigned flags, uint64_t max_matches, bz2b200_match **matches, size_t *n_matches,
                   bz2b200_search_totals *totals, uint8_t **lines, size_t *lines_len);

/* Device-resident entry points: input already in HBM (16-byte aligned), output written to a
 * caller-provided device buffer of out_cap bytes (multiple of 4).  Used for the roofline figure. */
int bz2b200_compress_device(bz2b200_ctx *ctx, const void *d_in, size_t n, int level, void *d_out, size_t out_cap, size_t *out_len);
int bz2b200_decompress_device(bz2b200_ctx *ctx, const void *d_in, size_t n, int multistream, void *d_out, size_t out_cap, size_t *out_len);
/* upper bound of the compressed size of n input bytes at `level` (for sizing d_out) */
size_t bz2b200_compress_bound(size_t n, int level);

/* ---- multi-GPU: block-range shards (SURVEY.md section 8e; one context = one GPU = one shard) ----
 * A shard is a slice of the input plus a halo after it.  The RLE1 automaton restarts at every block, so a
 * rank that knows where its first block starts can cut and compress its blocks alone.  Cross-rank data are
 * three scalars per rank: the first-block offset (a chain r -> r+1), the bit length (exclusive scan) and the
 * CRC fold.  There is no collective on the data path.
 *   shard_begin    tile summaries of in[0, n_avail) (does not depend on the first-block offset)
 *   shard_cut      cut walk from s_start; this shard owns the blocks that start in [s_start, own_len).
 *                  info->next_start = offset (in this buffer) of the first block of the next shard;
 *                  info->complete = 0 if the halo ended before the last owned block was full (not the last shard)
 *   shard_compress all per-block stages; fills info->bits and info->crc_fold
 *   shard_emit     the segment's bytes, pre-shifted so that its first bit sits at bit `bit_phase` (0..7) of
 *                  byte 0: the assembler only copies bytes and ORs one boundary byte (seg == NULL: keep it in HBM)
 *   stitch_shards  host-side assembly: "BZh<level>" + segments + end-of-stream magic + combined CRC */
typedef struct {
  uint64_t next_start;
  uint64_t bits;
  uint32_t n_blocks;
  uint32_t crc_fold;   /* fold of this shard's block CRCs starting from 0 (BJ:2237); shard folds compose by rotation */
  uint32_t complete;
  uint32_t bit_phase;  /* set by shard_emit */
} bz2b200_shard_info;
int bz2b200_shard_begin(bz2b200_ctx *ctx, const void *in, size_t n_avail, int on_device, int level);
int bz2b200_shard_cut(bz2b200_ctx *ctx, uint64_t s_start, uint64_t own_len, int is_last, bz2b200_shard_info *info);
/* Speculative start, so that the shards need not cut one after the other: when no cut falls inside a run, blocks
 * start where the run-length-coded byte count G reaches a multiple of B, and every cut inside a run upstream shifts
 * that phase by a few units.  shard_gtotal returns G(pos) of this buffer (pos = own_len: what this shard adds to G);
 * with g_before = sum over the earlier shards, shard_cut_g runs 64 cut walks at once, from the first positions whose
 * G reaches ceil(g_before / B) * B - g_before + d, d = -32..31.  Once the true offset of the shard's first block is
 * known (the previous shard's next_start), shard_cut_pick installs the walk that started there (*found = 1, info
 * filled) -- or reports *found = 0, and the caller falls back to shard_cut. */
int bz2b200_shard_gtotal(bz2b200_ctx *ctx, uint64_t pos, uint64_t *g);
int bz2b200_shard_cut_g(bz2b200_ctx *ctx, uint64_t g_before, uint64_t own_len);
int bz2b200_shard_cut_pick(bz2b200_ctx *ctx, uint64_t s_start, uint64_t own_len, int is_last, bz2b200_shard_info *info, int *found);
int bz2b200_shard_compress(bz2b200_ctx *ctx, bz2b200_shard_info *info);
int bz2b200_shard_emit(bz2b200_ctx *ctx, int bit_phase, bz2b200_shard_info *info, uint8_t **seg, size_t *seg_bytes);
int bz2b200_stitch_shards(int level, int n_shards, const uint8_t *const *segs, const bz2b200_shard_info *infos, uint8_t **out, size_t *out_len);

/* ---- the shard scheduler: one stream over several lanes, devices and processes (csrc/pool.inl) ----
 * A pool owns `lanes_per_device` contexts (each with its own stream) on every listed device.  A stream is cut into
 * shards; shard i goes to lane i mod lanes, lanes work at the same time, and the host<->device copies of one shard
 * run under the kernels of the others -- inside one blocking call.  bz2b200_compress() itself routes inputs of 32 MB
 * or more through a two-lane pool on its context's device; pageable input is staged through page-locked memory by a
 * helper thread (SURVEY.md 8b "may be pageable; the library stages through pinned memory").
 *   pool_compress    Bzip2.compressFile (BJ:2199-2249) on every device of the pool: the multi-GPU form of the
 *                    reference-facing call (SURVEY.md 8b `ngpus`).  shard_bytes = 0 picks a size.
 *   pool_decompress  Bzip2.decompressFile (BJ:1769-1796) of ONE stream, block ranges over the lanes (SURVEY.md 8e)
 * Ranks of one node (one process per GPU) join a GROUP: a page of POSIX shared memory that carries the per-shard
 * scalars (first-block offset, end bit, CRC fold) between processes.  Calls with a group are collective: every rank
 * makes the same sequence of calls; waits have a deadline (timeout_ms) and a failing rank wakes the others with
 * BZ2B200_E_PEER.  `name` must be unique per job (e.g. master port + launcher pid). */
typedef struct bz2b200_pool bz2b200_pool;
typedef struct bz2b200_group bz2b200_group;
int bz2b200_pool_create(const int *devices, int n_devices, int lanes_per_device, bz2b200_pool **pool);
void bz2b200_pool_destroy(bz2b200_pool *pool);
int bz2b200_pool_compress(bz2b200_pool *pool, const uint8_t *in, size_t n, int level, size_t shard_bytes, uint8_t **out, size_t *out_len);
/* pool_compress that also returns the stream's line index (see bz2b200_compress_indexed) */
int bz2b200_pool_compress_indexed(bz2b200_pool *pool, const uint8_t *in, size_t n, int level, size_t shard_bytes, uint8_t **out, size_t *out_len,
                                  bz2b200_block_entry **entries, uint32_t **newlines, size_t *count, uint64_t *total_lines);
/* shard plan of pool_compress when shard_bytes == 0: the first shard of every lane has first_bytes (0 = six blocks), every
 * following wave is `growth` times larger (0 = 2.5): only the first upload is exposed, large batches do most of the work */
int bz2b200_pool_set_plan(bz2b200_pool *pool, size_t first_bytes, double growth);
/* the plan itself (for callers that hand out shards to ranks): returns the number of shards, sizes[] filled */
int bz2b200_pool_plan(size_t n, int level, int lanes, size_t first_bytes, double growth, size_t *sizes, int cap);
/* Host placement.  Runs the CALLING thread on the CPUs of the NUMA node `device` is attached to (sysfs numa_node of its PCI
 * address), so that page-locked memory it allocates afterwards and the copies it issues stay on the device's socket; call it
 * once per feeding thread before allocating buffers (what `numactl --cpunodebind` does for a whole process).  Returns the node,
 * or -1 when the platform does not say (virtual machines often hide it), the node has none of the thread's CPUs, or
 * BZ2B200_NUMA=0: the thread is then left alone.  The library's own lane and upload threads do this by themselves. */
int bz2b200_bind_thread_to_device(int device);
int bz2b200_pool_last_stats(bz2b200_pool *pool, bz2b200_stats *st);
const char *bz2b200_pool_last_error(bz2b200_pool *pool);
int bz2b200_group_open(const char *name, int rank, int world, int timeout_ms, bz2b200_group **grp);
void bz2b200_group_close(bz2b200_group *grp);
/* This process's shards of a stream that spans the group (grp == NULL: this process holds all of them).
 * jobs[] in ascending `index`; shard `index` starts at input offset `base`, owns the blocks that start in
 * [base, base + own_len) and may read n_readable >= own_len bytes at src (the rest is its halo: the library starts
 * with 5/4 of a block and takes more when a run-heavy block needs it).  The last shard (index == total_shards - 1)
 * ends the stream.  results[i]: the segment of jobs[i], already shifted to its bit phase (seg == NULL with
 * keep_on_device), its bit offset in the stream and the running totals; bz2b200_stitch_shards assembles them. */
typedef struct {
  const void *src;
  size_t n_readable, own_len;
  uint64_t base;
  int32_t index, on_device;
} bz2b200_shard_job;
typedef struct {
  uint8_t *seg;               /* page-locked; release with bz2b200_free */
  size_t seg_bytes;
  bz2b200_shard_info info;    /* next_start in GLOBAL input coordinates here */
  uint64_t bit_offset;        /* of the segment's first bit in the stream */
  uint64_t end_bit, blocks_through;
  uint32_t crc_fold_through, pad;
} bz2b200_shard_result;
/* Decompression of ONE stream over the lanes: pool_decompress for a stream held by this process (size_hint = expected
 * output size, 0 = unknown: 6 x the input is reserved and a larger result is assembled by one more copy; slice_bytes
 * = 0 picks the slices); pool_decompress_shards for this process's byte slices of a stream that spans a group.
 * jobs[]: slice `index` = bytes [base, base + own_len) of the stream, n_readable >= own_len bytes readable at src (the
 * rest is the halo a block that starts in the slice may run into; the library takes what it needs).  results[i]:
 * the decoded bytes of the blocks whose signature starts in slice i, their offset in the output, and rc = the
 * slice's own status; the status of the stream is the first non-zero rc in slice order (what the reference's
 * sequential walk would have hit first). */
typedef struct {
  uint8_t *part;              /* page-locked; release with bz2b200_free (NULL with keep_on_device or 0 bytes) */
  uint64_t bytes, out_offset;
  int32_t rc;
  uint32_t n_blocks;
} bz2b200_range_result;
int bz2b200_pool_decompress(bz2b200_pool *pool, const uint8_t *in, size_t n, int multistream, size_t size_hint, size_t slice_bytes, uint8_t **out,
                            size_t *out_len);
int bz2b200_pool_decompress_shards(bz2b200_pool *pool, bz2b200_group *grp, const bz2b200_shard_job *jobs, int n_jobs, int total_shards,
                                   uint64_t total_n, int first_level, int multistream, int keep_on_device, bz2b200_range_result *results);
int bz2b200_pool_compress_shards(bz2b200_pool *pool, bz2b200_group *grp, const bz2b200_shard_job *jobs, int n_jobs, int total_shards, int level,
                                 int keep_on_device, bz2b200_shard_result *results);
/* bz2b200_search of ONE stream over the lanes: the slices of bz2b200_pool_decompress (slice_bytes = 0 picks them) are
 * decoded and searched on their lanes, and the host composes the per-slice counts into global ranks, line numbers and
 * lines.  Matches, totals, lines, return codes and argument-error texts (bz2b200_pool_last_error) equal bz2b200_search's
 * on one context; a damaged stream gives bz2b200_pool_decompress's error.  Each slice's decoded bytes stay on its lane's
 * device until the call ends, so a device holds its lanes' share of the output (all of it with one device).
 * bz2b200_pool_last_stats: n_blocks, in_bytes and out_bytes as bz2b200_pool_decompress, ms_total = host wall time of the
 * call, ms_stage[5] = device time of the search kernels and line gathers, summed over the lanes. */
int bz2b200_pool_search(bz2b200_pool *pool, const uint8_t *in, size_t n, int multistream, const uint8_t *patterns, const uint32_t *pattern_lens,
                        size_t n_patterns, unsigned flags, uint64_t max_matches, size_t slice_bytes, bz2b200_match **matches, size_t *n_matches,
                        bz2b200_search_totals *totals, uint8_t **lines, size_t *lines_len);
/* tests/ only: block capacity, blocks per batch, first halo (0 = defaults) and forced staging for every lane of a pool;
 * and for a context: inputs of min_bytes or more go through its own two-lane pool in shards of shard_bytes (0 = auto). */
int bz2b200_pool_debug(bz2b200_pool *pool, uint32_t block_cap, uint32_t batch_blocks, size_t first_halo, int force_staging);
/* tests/ only: candidates per decode batch (0 = 320) for a context / every lane of a pool */
int bz2b200_debug_set_decode_batch(bz2b200_ctx *ctx, bz2b200_pool *pool, uint32_t candidates);
/* tests/ only: threads per CTA of the RLE1 inverse, 512 or 1024 (0 = 1024 when the batch has no more blocks than the
 * device has SMs, else 512) for a context / every lane of a pool, so that one input reaches both strip widths */
int bz2b200_debug_set_rle1_threads(bz2b200_ctx *ctx, bz2b200_pool *pool, uint32_t threads);
/* tests/ only: bz2b200_debug_set_search_tile for every lane of a pool */
int bz2b200_debug_set_pool_search_tile(bz2b200_pool *pool, uint32_t bytes);
int bz2b200_debug_set_pool(bz2b200_ctx *ctx, size_t min_bytes, size_t shard_bytes, size_t first_halo, int force_staging);

/* ---- the stream flavour (SURVEY.md 8f N2; csrc/stream_abi.inl) ----
 * What Bzip2.compressFile / decompressFile do with {readByte} sources and {writeByte} sinks (BJ:178-272,
 * NPM/bin/compressjs:60-180), without holding input or output in full: feed pieces of any size; every call returns the
 * bytes that are complete (library-allocated, release with bz2b200_free; *out may be NULL with *out_len == 0).
 *   zstream  byte-identical to bz2b200_compress on the concatenated input; chunk_bytes (0 = 64 MiB) is how much input is
 *            collected before its blocks are cut (the second half of a chunk is the halo of the blocks of the first)
 *   dstream  decodes every block as soon as it is complete (chunk_bytes, 0 = 16 MiB of stream, between attempts); errors
 *            come out of the call that meets them, after the bytes of the blocks before */
typedef struct bz2b200_zstream bz2b200_zstream;
typedef struct bz2b200_dstream bz2b200_dstream;
int bz2b200_zstream_open(bz2b200_ctx *ctx, int level, size_t chunk_bytes, bz2b200_zstream **zs);
/* a zstream that also builds the stream's line index; bz2b200_zstream_index after finish (see bz2b200_compress_indexed) */
int bz2b200_zstream_open_indexed(bz2b200_ctx *ctx, int level, size_t chunk_bytes, bz2b200_zstream **zs);
int bz2b200_zstream_index(bz2b200_zstream *zs, bz2b200_block_entry **entries, uint32_t **newlines, size_t *count, uint64_t *total_lines);
/* Appending to a stream and its line index, without recompressing it.  Opens an indexed zstream that continues the LAST
 * stream of `in` (n bytes: caller-owned, only read, may be a memory map) whose line index is index / newlines / count /
 * total_lines (what bz2b200_compress_indexed, bz2b200_zstream_index or bz2b200_line_index return).  The new bytes then go
 * through bz2b200_zstream_feed and bz2b200_zstream_finish; the stream to keep is in[0, *keep) followed by every byte they
 * return, and bz2b200_zstream_index returns the line index of that whole stream.  For a stream the reference (or this
 * library) wrote from input A, appending B gives byte for byte bz2b200_compress(A + B) at the stream's level: every block
 * before the last keeps its bits, and the last block L is decoded and compressed again together with B (DESIGN.md
 * section 8, "Appending").  Any valid stream can be continued (one from libbz2 too); the result then decodes to A + B.  The call reads
 * only L's bytes, the footer after it and the byte at *keep = L.bit_begin / 8 (its bits before L are carried over).  Rows
 * the append writes carry L's stream and level.  Checks, before anything is returned: the index passes the checks of
 * bz2b200_decompress_lines (BZ2B200_E_ARG); the end-of-stream magic sits at L.bit_end and the stream CRC after it equals
 * the fold of the stored CRCs of L's stream's entries, L decodes (the verdicts of bz2b200_decompress_ranges) to
 * newlines[count - 1] '\n' bytes and ends as total_lines says (DATA_ERROR "index does not match the input" otherwise);
 * the stream ends the input, (L.bit_end + 87) / 8 == n (BZ2B200_E_ARG otherwise: the bytes after it, another stream or
 * trailing data, would be dropped).  count == 0 is accepted only for one empty stream (14 bytes; *keep = 4).  Blocks
 * before L are neither read nor checked, as range reads do not check the blocks they do not decode.  newlines is required.
 * bz2b200_last_stats after the call describes the decode of L, as bz2b200_decompress_lines would.  On error *zs is NULL. */
int bz2b200_zstream_open_append(bz2b200_ctx *ctx, const uint8_t *in, size_t n, const bz2b200_block_entry *index, const uint32_t *newlines, size_t count,
                                uint64_t total_lines, size_t chunk_bytes, bz2b200_zstream **zs, uint64_t *keep);
int bz2b200_zstream_feed(bz2b200_zstream *zs, const uint8_t *in, size_t n, uint8_t **out, size_t *out_len);
int bz2b200_zstream_finish(bz2b200_zstream *zs, uint8_t **out, size_t *out_len);
void bz2b200_zstream_close(bz2b200_zstream *zs);
int bz2b200_dstream_open(bz2b200_ctx *ctx, int multistream, size_t chunk_bytes, bz2b200_dstream **ds);
int bz2b200_dstream_feed(bz2b200_dstream *ds, const uint8_t *in, size_t n, uint8_t **out, size_t *out_len);
int bz2b200_dstream_finish(bz2b200_dstream *ds, uint8_t **out, size_t *out_len);
void bz2b200_dstream_close(bz2b200_dstream *ds);

const char *bz2b200_strerror(int rc);
const char *bz2b200_last_error(bz2b200_ctx *ctx);
int bz2b200_last_stats(bz2b200_ctx *ctx, bz2b200_stats *st);

/* Stage dumps for the parity tests (tests/ only): after a compress call, copy an intermediate
 * of block `blk` to host.  what: 0 = BlockRec table (all blocks), 1 = RLE1'd block bytes,
 * 2 = BWT L column, 3 = MTF/RLE2 symbols (u16), 4 = BlockMeta table (all blocks),
 * 5 = selectors: the table of every group of 50 symbols (u8 x n_sel), 6 = code lengths
 * (u8 [6][260]: table t, symbol s at t * 260 + s; n_groups tables of alphabet + 2 used).
 * Kinds 1-6 describe the last batch of the last compress call (see debug_set_batch_blocks).
 * Kinds 7-12 describe the last batch of the last decode call (see debug_set_decode_batch): 7 = the parsed candidates
 * (DecBlk of csrc/decode.cuh, one per candidate), 8 = the symbols of candidate blk (u16, nsym of them, end-of-block
 * last), 9 = its RLE2 inverse offsets (u32, nsym + 1: where each symbol's bytes start in the L column), 10 = its L
 * column after the inverse MTF (count bytes), 11 = the inverse-BWT output (RLE1 bytes) of the blk-th inverted block,
 * 12 = the inverted blocks as candidate indices (u32, stream order: entry blk is the candidate of kind 11's blk).
 * Returns the number of bytes written to dst (<= cap) or a negative error. */
long long bz2b200_debug_fetch(bz2b200_ctx *ctx, int what, int blk, void *dst, size_t cap);
/* tests/ only: override the block capacity B (0 = level*100000-19) to stress the cut-point logic. */
int bz2b200_debug_set_block_cap(bz2b200_ctx *ctx, uint32_t cap);
/* tests/ only: run the per-block stages in batches of at most `blocks` blocks (0 = as many as fit the
 * 31-bit index space and 70 % of the free device memory).  Stage dumps then show the last batch. */
int bz2b200_debug_set_batch_blocks(bz2b200_ctx *ctx, uint32_t blocks);
/* tests/ only: bytes per tile of the search kernels, a multiple of 256 up to 8192 (0 = 8192), so that small outputs
 * span many tiles. */
int bz2b200_debug_set_search_tile(bz2b200_ctx *ctx, uint32_t bytes);
/* tests/ only: bytes per newline-directory tile (a multiple of 256 up to 8192; 0 = the default, 8192), and per segment of the
 * indexed compress calls' '\n' count (0 = the default, 32768; a context's own two-lane pool takes it too) */
int bz2b200_debug_set_line_tile(bz2b200_ctx *ctx, uint32_t bytes);
/* tests/ only: skip the block-CRC comparison of the decoder (BJ:1756-1761), so that what a damaged stream decodes TO
 * can be compared with the oracle.  Not reachable from the environment. */
int bz2b200_debug_set_ignore_block_crc(bz2b200_ctx *ctx, int on);
/* tests/ only: the device copy of HuffmanAllocator.allocateHuffmanCodeLengths (BJ:1275-1298) on a[0..n): frequencies in
 * ascending order in, code lengths out (in place) -- pinned by the reference's own vectors, NPM/test/huffman.js:16-76 */
int bz2b200_debug_huffman_lengths(bz2b200_ctx *ctx, int32_t *a, int n, int maxlen);

#ifdef __cplusplus
}
#endif
#endif
