/* dcdf_cuda.h -- C-ABI of the B200-native Heuristic T-k^2-raster codec (libdcdf_cuda.so).
 *
 * This is the drop-in boundary for ONE hot path of Arbol-Project/dcdf: building Chunk / Superchunk
 * byte strings from (time, y, x) rasters and answering cell / window / value-range queries from
 * those bytes.  Plain pointers and sizes only; no torch / C++ types.  Every entry point cites the
 * reference interface it replaces (paths relative to dcdf/src in the reference tree).
 *
 * There is NO CPU fallback behind these symbols: every call runs sm_100a kernels on the context's
 * device and fails with DCDF_ERR_CUDA if that is impossible.
 *
 * Conventions
 *  - every function returns an int32_t status (DCDF_OK == 0); dcdf_last_error() gives the text.
 *    The reference panics on data errors (fixed.rs:40,51,66; superchunk.rs:105-110;
 *    mmarray.rs:218-229; block.rs:27-32); a Rust shim turns the DATA codes back into panic!().
 *  - arrays are described by base pointer + shape[3] + element strides[3] (an ndarray view,
 *    mmbuffer.rs:573-594); `mem` says where the pointer lives.  Inputs are borrowed for the call.
 *  - a dcdf_ctx owns one device, one stream and its scratch arenas; it is NOT re-entrant.  Built
 *    objects are immutable and may be queried from any context on the same device.
 */
#ifndef DCDF_CUDA_H
#define DCDF_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCDF_ABI_VERSION 1

/* status codes (errors.rs:9-18 + the reference's panics) */
enum {
  DCDF_OK = 0,
  DCDF_ERR_NONFINITE = 1,      /* fixed.rs:39-41   inf / -inf in the input            */
  DCDF_ERR_PRECISION_LOSS = 2, /* fixed.rs:51-57, mmbuffer.rs:606                     */
  DCDF_ERR_OVERFLOW = 3,       /* fixed.rs:66-69                                      */
  DCDF_ERR_BAD_LEVELS = 4,     /* superchunk.rs:105-110                               */
  DCDF_ERR_OUT_OF_BOUNDS = 5,  /* mmarray.rs:218-229                                  */
  DCDF_ERR_BAD_FORMAT = 6,     /* malformed serialized bytes (mmstruct.rs:45-59 ...)  */
  DCDF_ERR_CUDA = 7,           /* CUDA runtime failure / no device                    */
  DCDF_ERR_BAD_ARG = 8         /* NULL pointers, k != 2, 1x1 rasters (snapshot.rs:166)*/
};

/* MMEncoding  mmstruct.rs:36-43 */
enum { DCDF_ENC_I32 = 4, DCDF_ENC_I64 = 8, DCDF_ENC_F32 = 32, DCDF_ENC_F64 = 64 };

/* where a pointer lives */
enum { DCDF_MEM_HOST = 0, DCDF_MEM_DEVICE = 1 };

/* Reference kinds  superchunk.rs:827-831 (build never produces Local) */
enum { DCDF_REF_ELIDED = 0, DCDF_REF_LOCAL = 1, DCDF_REF_EXTERNAL = 2 };

typedef struct dcdf_ctx dcdf_ctx;
typedef struct dcdf_chunk dcdf_chunk;           /* one Chunk resident on the device           */
typedef struct dcdf_superchunk dcdf_superchunk; /* one Superchunk (or a run of them) + chunks */

/* ndarray ArrayView3 stand-in (mmbuffer.rs:255-260, 505-594) */
typedef struct dcdf_array3 {
  const void* base;
  int64_t shape[3];   /* instants, rows, cols */
  int64_t strides[3]; /* in ELEMENTS          */
  int32_t encoding;   /* DCDF_ENC_*           */
  int32_t mem;        /* DCDF_MEM_*           */
} dcdf_array3;

/* MMStruct3Build counters  mmstruct.rs:24-34.  `size` counts serialized Chunk bytes plus the
 * superchunk min/max DAC bytes (node / Links sizes carry CIDs and stay on the host side). */
typedef struct dcdf_build_stats {
  uint64_t size;
  uint32_t elided, local, external, snapshots, logs;
} dcdf_build_stats;

/* geom::Cube  geom.rs:72-120 -- bounds are re-ordered if swapped, exactly as Cube::new does */
typedef struct dcdf_cube {
  int64_t start, end, top, bottom, left, right;
} dcdf_cube;

/* ------------------------------------------------------------------ context */
int32_t dcdf_abi_version(void);
int32_t dcdf_ctx_create(int32_t device, dcdf_ctx** out);
int32_t dcdf_ctx_destroy(dcdf_ctx* ctx);
/* Borrow a caller-owned cudaStream_t (e.g. torch's current stream); NULL restores the private one. */
int32_t dcdf_ctx_set_stream(dcdf_ctx* ctx, void* cuda_stream);
/* Per-context knobs (the reference has no configuration system: all knobs are arguments, SURVEY section 5; these
 * select between code paths that produce identical bytes / results and exist for tests and A/B measurements):
 *   "stage_limit" <bytes>   encoder: structures larger than this are emitted straight into the arena (default 16384)
 *   "arena_hint"  <bytes>   first size of the encoder's output arena (grown and retried when it overflows)
 *   "no_fast_encode" 0|1    eligible full f32 tiles through the general encoder instead of the fast-path kernel
 *   "encode_tiles256" 0|1   full 64x64 tiles through the 256-thread tile encoder
 *   "fast_variant" 0|1|2    fast-path kernel launches for A/B runs: 1 = four tiles per CTA (255 registers), 2 = four tiles
 *                           per CTA with every instant's tile staged in shared memory by bulk copies behind an mbarrier
 *   "fast_sync_mask" <m>    fast-path kernel: the tiles of a CTA re-align every (m + 1) instants (default 3)
 *   "cell_tile_min" <n>     cell series: a tile that at least n series of a batch fall into is decoded once per instant by
 *                           the tile decoder instead of one root-to-leaf walk per (series, instant) (default 64, the measured break-even; 0 = never)
 *   "window_cells" 0|1      windows through the 4x4-block walker k_window_blocks (the path of trees larger than 64x64)
 *   "window_wide" 0|1       64-bit tile expansion even when every DAC code fits three bytes
 *   "search_share_min" <n>  value-range search: when the windows of a batch overlap (>= n windows per touched (time slice, tile)
 *                           on average; default 3, 0 = never) the counting pass decodes every touched tile once for all of them
 *   "search_dfs" 0|1        depth-first search kernel instead of the tile search
 *   "search_no_cache" 0|1   search's writing pass recomputes instead of reading the counting pass's findings
 *   "trace" 0|1             host-side phase times of the encode pipeline on stderr
 *   "time_stats_scratch" n  dcdf_superchunk_time_stats: bytes of partials per group of time slices (default 1 GiB,
 *                           <= 0 restores it; a group holds at least one slice); results do not depend on it
 * Unknown names return DCDF_ERR_BAD_ARG. */
int32_t dcdf_ctx_set_option(dcdf_ctx* ctx, const char* name, int64_t value);
/* Counters of the last build call: "encode_units_fast" (units encoded by the fast-path kernels), "encode_units_edge" (the
 * part of those with at most 32 rows or columns in the raster, one warp per tile), "encode_units_general",
 * "encode_units_wide" (64-bit values), "encode_units_clipped".  Of the last dcdf_superchunk_time_stats call:
 * "time_stats_groups" (groups of time slices, each one pass of its two kernels) and "time_stats_scratch_bytes" (partial
 * bytes of the largest group). */
int32_t dcdf_ctx_get_stat(const dcdf_ctx* ctx, const char* name, int64_t* value);
int32_t dcdf_ctx_synchronize(dcdf_ctx* ctx);
const char* dcdf_last_error(const dcdf_ctx* ctx);
/* Kernel launches issued by this context since creation (bench.py's gpu_launches). */
uint64_t dcdf_ctx_launch_count(const dcdf_ctx* ctx);
/* CUDA-event time (ms) of the dominant kernel(s) of the last build / query call, measured on the
 * context's stream.  which: 0 = encode kernel, 1 = stats kernel, 2 = gather, 3 = window decode,
 * 4 = cell decode, 5 = search, 6 = window statistics (both of its kernels), 7 = time statistics (all kernels of
 * the call, every group of slices). */
int32_t dcdf_ctx_last_kernel_ms(const dcdf_ctx* ctx, int32_t which, float* ms);

/* ------------------------------------------------------------------ a1 / a2 / a3 / a21 */
/* suggest_fraction  fixed.rs:96-159  (kind: 0 = Precise(bits), 1 = Round(bits)) */
int32_t dcdf_suggest_fraction(dcdf_ctx* ctx, const dcdf_array3* a, int32_t* kind, int32_t* bits);
/* MMBuffer3::min_max  mmbuffer.rs:366-395 (+ min_max_float :465-499): per-instant fixed (min,max) */
int32_t dcdf_min_max(dcdf_ctx* ctx, const dcdf_array3* a, int32_t fractional_bits, int32_t round,
                     int64_t* min_out, int64_t* max_out /* host, shape[0] entries each */);
/* to_fixed / from_fixed  fixed.rs:31-86 over flat arrays (host or device pointers per `mem`) */
int32_t dcdf_to_fixed(dcdf_ctx* ctx, const void* in, int32_t encoding, uint64_t n, int32_t fractional_bits,
                      int32_t round, int64_t* out, int32_t mem);
int32_t dcdf_from_fixed(dcdf_ctx* ctx, const int64_t* in, uint64_t n, int32_t fractional_bits, void* out,
                        int32_t encoding, int32_t mem);

/* ------------------------------------------------------------------ a10 / a11: Chunk */
/* Chunk::build  chunk.rs:42-96.  The array's fractional_bits / round are the MMBuffer3 fields
 * (mmbuffer.rs:318-341).  The returned chunk is resident on the device and immediately queryable;
 * its bytes are exactly Chunk::write_to (chunk.rs:235-243). */
int32_t dcdf_chunk_build(dcdf_ctx* ctx, const dcdf_array3* a, int32_t k, int32_t fractional_bits, int32_t round,
                         dcdf_chunk** out, dcdf_build_stats* stats);
/* Chunk::read_from  chunk.rs:247-266: upload + validate serialized bytes. */
int32_t dcdf_chunk_open(dcdf_ctx* ctx, const uint8_t* bytes, uint64_t len, int32_t mem, dcdf_chunk** out);
int32_t dcdf_chunk_free(dcdf_chunk* chunk);
/* Cacheable::size  chunk.rs:269-278 */
int32_t dcdf_chunk_size(const dcdf_chunk* chunk, uint64_t* len);
/* Chunk::write_to  chunk.rs:235-243 into caller memory (host or device per `mem`) */
int32_t dcdf_chunk_bytes(dcdf_ctx* ctx, const dcdf_chunk* chunk, uint8_t* dst, uint64_t cap, int32_t mem);
/* Chunk::shape chunk.rs:119-123, encoding / fractional_bits chunk.rs:36-40, blocks */
int32_t dcdf_chunk_info(const dcdf_chunk* chunk, int64_t shape[3], int32_t* encoding, int32_t* fractional_bits,
                        uint32_t* n_blocks);
/* instants per block (logs + 1), n_blocks entries -- the heuristic's decisions (chunk.rs:62) */
int32_t dcdf_chunk_block_instants(dcdf_ctx* ctx, const dcdf_chunk* chunk, uint32_t* out);

/* Queries.  `out_encoding` selects the element type written: DCDF_ENC_I64 = raw fixed-point i64
 * (what Chunk::get hands to MMBuffer0/1/3::set), or the chunk's own encoding (from_fixed applied,
 * mmbuffer.rs:561-563).  Out-of-bounds requests return DCDF_ERR_OUT_OF_BOUNDS (mmarray.rs:218-229). */
/* Chunk::get  chunk.rs:127-131, batched: irc = n x (instant,row,col) */
int32_t dcdf_chunk_get_batch(dcdf_ctx* ctx, const dcdf_chunk* chunk, uint64_t n, const int64_t* irc, void* out,
                             int32_t out_encoding, int32_t mem);
/* Chunk::fill_cell  chunk.rs:135-148, batched: q = n x (start,end,row,col); out_off[n+1] gives the
 * element offset of each series in `out` (exclusive prefix sum of end-start, computed by the caller).
 * q and out_off are host arrays; `mem` says where `out` lives (pinned host memory receives at the full PCIe rate). */
int32_t dcdf_chunk_cell_batch(dcdf_ctx* ctx, const dcdf_chunk* chunk, uint64_t n, const int64_t* q,
                              const uint64_t* out_off, void* out, int32_t out_encoding, int32_t mem);
/* Chunk::fill_window  chunk.rs:152-158: out is a dense [instants, rows, cols] array */
int32_t dcdf_chunk_window(dcdf_ctx* ctx, const dcdf_chunk* chunk, const dcdf_cube* bounds, void* out,
                          int32_t out_encoding, int32_t mem);
/* Chunk::iter_search  chunk.rs:213-228: (instant,row,col) triplets of cells with lower <= v <= upper
 * (fixed-point bounds, swapped if reversed), in the reference's traversal order.  Two-call protocol:
 * pass out == NULL to get *n_found, then a buffer of 3 * n_found int64. */
int32_t dcdf_chunk_search(dcdf_ctx* ctx, const dcdf_chunk* chunk, const dcdf_cube* bounds, int64_t lower,
                          int64_t upper, int64_t* out_irc, uint64_t cap, uint64_t* n_found, int32_t mem);

/* ------------------------------------------------------------------ a12 / a22: Superchunk */
/* Superchunk::build  superchunk.rs:88-270 (compute part: partition, min_max, elision, per-subchunk
 * compute_fractional_bits + Chunk::build, min/max DACs; CIDs / resolver.save stay on the host), run for
 * every `chunk_size`-instant slice of the array as Variable::append does (dataset.rs:834-851).
 *   chunk_size <= 0      : the whole array is ONE superchunk (plain Superchunk::build)
 *   compute_bits != 0    : buffer.compute_fractional_bits() per slice first (dataset.rs:842)
 * levels = k2_levels (sum must equal the levels needed, else DCDF_ERR_BAD_LEVELS). */
int32_t dcdf_superchunk_build(dcdf_ctx* ctx, const dcdf_array3* a, const uint32_t* levels, uint32_t n_levels,
                              int32_t k, int32_t fractional_bits, int32_t round, int32_t compute_bits,
                              int64_t chunk_size, dcdf_superchunk** out);
int32_t dcdf_superchunk_free(dcdf_superchunk* sc);

/* One entry per time slice. */
typedef struct dcdf_superchunk_info {
  int64_t shape[3];
  int64_t sidelen, chunks_sidelen, subsidelen; /* superchunk.rs:44-86 */
  uint32_t levels;
  int32_t encoding, fractional_bits;
  uint32_t n_refs;          /* subsidelen^2                                    */
  uint64_t max_dac_bytes;   /* Dac::size of the per-(instant,subchunk) max DAC */
  uint64_t min_dac_bytes;
  uint64_t chunk_bytes;     /* sum of stored subchunk sizes                    */
  dcdf_build_stats stats;
} dcdf_superchunk_info;
int32_t dcdf_superchunk_count(const dcdf_superchunk* sc, uint32_t* n_slices);
/* Nested superchunks (more than two k2_levels entries, superchunk.rs:171): the recursion's node tree is static
 * geometry shared by all slices.  Node 0 is the root; dcdf_superchunk_get_info / _refs / _bytes address node 0.
 * A node that is Elided in a slice has n_refs == 0 there. */
int32_t dcdf_superchunk_node_count(const dcdf_superchunk* sc, uint32_t* n_nodes);
int32_t dcdf_superchunk_node_info(const dcdf_superchunk* sc, uint32_t slice, uint32_t node, dcdf_superchunk_info* info);
/* As dcdf_superchunk_refs for any node; child_node[i] is the node index of a nested superchunk reference, -1 for
 * Chunk references and Elided slots. */
int32_t dcdf_superchunk_node_refs(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, uint32_t node, int32_t* kinds,
                                  int32_t* child_node, uint64_t* chunk_off, uint64_t* chunk_size, int32_t* chunk_bits);
/* which 1 = max Dac, 2 = min Dac of the node. */
int32_t dcdf_superchunk_node_bytes(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, uint32_t node, int32_t which,
                                   uint8_t* dst, uint64_t cap, int32_t mem);
int32_t dcdf_superchunk_get_info(const dcdf_superchunk* sc, uint32_t slice, dcdf_superchunk_info* info);
/* Reference kinds (DCDF_REF_*) per subchunk, row-major (superchunk.rs:127-181, 206-240) and, for
 * stored subchunks, [offset, offset+size) of its Chunk bytes inside the slice's chunk-byte blob and its
 * fractional bits.  All arrays are host, n_refs entries. */
int32_t dcdf_superchunk_refs(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, int32_t* kinds,
                             uint64_t* chunk_off, uint64_t* chunk_size, int32_t* chunk_bits);
/* Copy out bytes: which 0 = concatenated Chunk bytes of the slice, 1 = max Dac, 2 = min Dac. */
int32_t dcdf_superchunk_bytes(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, int32_t which, uint8_t* dst,
                              uint64_t cap, int32_t mem);
/* Total encoded bytes over all slices (chunk bytes + DACs) -- S_out of the roofline model. */
int32_t dcdf_superchunk_total_bytes(const dcdf_superchunk* sc, uint64_t* n);

/* Superchunk::get / fill_cell / fill_window / search  superchunk.rs:313-585, with the time axis routed
 * across slices as Span does (span.rs:121-279).  Semantics as the dcdf_chunk_* queries; values of
 * Elided subchunks come from the max DAC (superchunk.rs:325-330, 426-433, 541-559). */
int32_t dcdf_superchunk_get_batch(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const int64_t* irc, void* out,
                                  int32_t out_encoding, int32_t mem);
int32_t dcdf_superchunk_cell_batch(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const int64_t* q,
                                   const uint64_t* out_off, void* out, int32_t out_encoding, int32_t mem);
int32_t dcdf_superchunk_window(dcdf_ctx* ctx, const dcdf_superchunk* sc, const dcdf_cube* bounds, void* out,
                               int32_t out_encoding, int32_t mem);
/* Batched windows: n cubes, out_off[n+1] element offsets into `out`. */
int32_t dcdf_superchunk_window_batch(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                     const uint64_t* out_off, void* out, int32_t out_encoding, int32_t mem);
/* Per-instant statistics of n windows, reduced on the device from the encoded bytes (the reference has no counterpart:
 * there a window is decoded and reduced by the caller).  One record per (window, instant): window i has end - start
 * records, instants ascending, from record out_off[i] on (out_off[n+1] host array, the convention of
 * dcdf_superchunk_window_batch counted in records).  Record r is count[r], vmin / vmax[r], sum[r], sum_sq[r].
 *  - value of a cell: exactly what dcdf_superchunk_window writes for it in the superchunk's encoding -- from_fixed with
 *    its subchunk's own fractional bits; for an Elided slot at any nesting level the node's table value at the node's
 *    bits; the stored integer for i32 / i64.  NaN cells (code 0 of a float encoding) are skipped.
 *  - count (uint64): the number of non-NaN cells of the window at that instant, exact.
 *  - vmin / vmax: in the superchunk's encoding (float / double / int32_t / int64_t arrays), compared by value across
 *    subchunks, exact for i64.  count == 0: NaN for float encodings, 0 for integer ones.
 *  - sum / sum_sq (double): sum of the values and of their squares; 0 when count == 0.  Per (window, subchunk, instant)
 *    the values are summed exactly as integers and scaled once; partials are added in subchunk order (row-major), so
 *    the error is a few 2^-53 * sum|v| per subchunk the window touches.
 *  - determinism: a window's records are bitwise identical across calls, alone or inside any batch, with or without the
 *    context option "window_wide", for a built superchunk and the same one reopened with dcdf_superchunk_open.
 *  - reversed bounds are swapped (Cube::new); a zero-area window gives records with count 0; out-of-range windows
 *    return DCDF_ERR_OUT_OF_BOUNDS; out_off that does not match end - start, NULL pointers, or subchunks larger than
 *    64x64 (only possible for an opened superchunk) return DCDF_ERR_BAD_ARG.  `mem` says where all five outputs live. */
int32_t dcdf_superchunk_window_stats(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                     const uint64_t* out_off, uint64_t* count, void* vmin, void* vmax,
                                     double* sum, double* sum_sq, int32_t mem);
/* Per-cell statistics over time of n windows, reduced on the device from the encoded bytes (no reference counterpart).
 * One record per (window, cell): window i has (bottom - top) * (right - left) records, row-major, from record out_off[i]
 * on (out_off[n+1] host array, the convention of dcdf_superchunk_window_batch counted in records).  Record r is
 * count[r], n_band[r], vmin / vmax[r], sum[r], sum_sq[r].
 *  - value of a cell at an instant: as for dcdf_superchunk_window_stats, exactly what dcdf_superchunk_window writes.
 *    NaN values are skipped.
 *  - count (uint64): the number of non-NaN instants, exact.
 *  - n_band (uint64): the number of instants with lower[i] <= (double)v <= upper[i]; NaN never counts.  Reversed bounds
 *    are swapped, +-inf is allowed, a NaN bound returns DCDF_ERR_BAD_ARG.  lower and upper both NULL: no band, n_band
 *    may be NULL (when given, it receives count).
 *  - vmin / vmax: in the superchunk's encoding, compared by value.  count == 0: NaN for float encodings, 0 for integer ones.
 *  - sum / sum_sq (double), in a fixed order.  A piece is the window's instants inside one time slice.  Per piece,
 *    s_p = ((0 + v_0) + v_1) + ... in double, in time order, v the value converted to double (exact for f32 / f64 / i32,
 *    round-to-nearest for i64); sum_sq adds v * v rounded once.  The record's sum is ((0 + s_0) + s_1) + ... over the
 *    pieces in time order.
 *  - accumulate != 0: the outputs hold records of an earlier call for the same window shapes, and this call continues
 *    them as if its pieces followed the earlier ones: counts add, min / max fold by value, each piece is added to the
 *    running sums in order.  (A Variable's span groups end on slice boundaries, so a series of calls over consecutive
 *    instants equals one call.)
 *  - determinism: a window's records are bitwise identical alone or inside any batch, with or without "window_wide",
 *    for a built superchunk and the same one reopened, and for any "time_stats_scratch".
 *  - a zero-instant window gives records with count 0 (unchanged under accumulate); a zero-area window has no records.
 *    Out-of-range windows return DCDF_ERR_OUT_OF_BOUNDS; out_off that does not match the areas, NULL outputs, a NaN
 *    bound, or subchunks larger than 64x64 (only possible for an opened superchunk) return DCDF_ERR_BAD_ARG.  `mem`
 *    says where all six outputs live. */
int32_t dcdf_superchunk_time_stats(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                   const uint64_t* out_off, const double* lower, const double* upper,
                                   uint64_t* count, uint64_t* n_band, void* vmin, void* vmax,
                                   double* sum, double* sum_sq, int32_t accumulate, int32_t mem);
/* Batched value-range search over n windows (same fixed-point [lower, upper] semantics as
 * dcdf_chunk_search).  counts[n] (host) receives matches per window; out_irc (may be NULL) receives the
 * triplets window after window.  Order inside a window: subchunks row-major, then chunk order. */
int32_t dcdf_superchunk_search_batch(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                     const int64_t* lower, const int64_t* upper, uint64_t* counts, int64_t* out_irc,
                                     uint64_t cap, uint64_t* n_found, int32_t mem);
/* Value-range search in the array's own units (the decoded values dcdf_superchunk_window returns with the superchunk's
 * encoding): a cell matches iff lower <= value <= upper.  NaN cells never match.  Other semantics as
 * dcdf_superchunk_search_batch.
 *  - value: exactly what the window decoder writes for the cell -- from_fixed in the encoding's float type with the
 *    fractional bits of the cell's own subchunk; for an Elided slot, the table value of its node with the node's bits.
 *    A cell matches iff lower <= (double)value <= upper.  Integer encodings compare the stored integer itself (0 is the
 *    value 0 there, not NaN).
 *  - bounds: reversed bounds are swapped (chunk.rs:214); -inf / +inf are allowed; a NaN bound returns DCDF_ERR_BAD_ARG.
 *  - the hit set is exact, also where dcdf_superchunk_search_batch reproduces the reference's traversal (single-node
 *    Logs, Logs over a single-node Snapshot, SURVEY App. B #15).  The bounds are converted on the device, per subchunk,
 *    to the interval of codes whose value lies in [lower, upper] (from_fixed is monotone in the code).
 *  - order: windows in call order; inside a window subchunks row-major, then instants ascending, as
 *    dcdf_superchunk_search_batch; inside one (subchunk, instant) an order of the implementation's own, deterministic.
 *    counts[n] are exact per window.  Two-call protocol as dcdf_superchunk_search_batch (out_irc == NULL: counts and
 *    *n_found only). */
int32_t dcdf_superchunk_search_values(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                      const double* lower, const double* upper, uint64_t* counts, int64_t* out_irc,
                                      uint64_t cap, uint64_t* n_found, int32_t mem);

/* ------------------------------------------------------------------ storage side (SURVEY 8b / 8f1) */
/* Content address of a stored node as the reference's in-memory store computes it (testing.rs:172-183):
 * CIDv1 = version 0x01, codec 0x12, multihash { code 0x12 (sha2-256), length 0x20, 32 digest bytes }. */
#define DCDF_CID_BYTES 36
/* node types (node.rs:9-15) of the objects a saved superchunk consists of */
enum { DCDF_NODE_LINKS = 1, DCDF_NODE_SUBCHUNK = 4, DCDF_NODE_SUPERCHUNK = 5 };
typedef struct dcdf_saved dcdf_saved;

/* What Superchunk::build + Resolver::save store for one time slice (superchunk.rs:199-270, 678-710; links.rs:65-76;
 * resolver.rs:126-138; mmstruct.rs:199-222): every distinct subchunk node, the Links node(s), nested superchunk nodes
 * and, last, the superchunk node itself -- in the order of their first save.  Chunk nodes are hashed on the device
 * (SHA2-256 over bytes that never leave HBM); External references are de-duplicated by CID exactly as
 * superchunk.rs:222-232 does, so dcdf_saved_stats returns the reference's MMStruct3Build (size, elided, external =
 * DISTINCT subchunks, snapshots, logs).  `sc` must outlive the returned object. */
int32_t dcdf_superchunk_save(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, dcdf_saved** out);
int32_t dcdf_saved_free(dcdf_saved* saved);
int32_t dcdf_saved_count(const dcdf_saved* saved, uint32_t* n_nodes);
/* CID, node type (DCDF_NODE_*) and stored size of object i; the last object is the slice's superchunk node. */
int32_t dcdf_saved_node(const dcdf_saved* saved, uint32_t i, uint8_t* cid /* DCDF_CID_BYTES */, int32_t* node_type, uint64_t* size);
/* The stored bytes of object i (header included), into host or device memory. */
int32_t dcdf_saved_node_bytes(dcdf_ctx* ctx, const dcdf_saved* saved, uint32_t i, uint8_t* dst, uint64_t cap, int32_t mem);
/* Every object's stored bytes back to back in object order (what a StoreWrite loop would write, mapper.rs:19-38) with one
 * wait for all device-to-host transfers; offsets[i] .. offsets[i + 1] is object i (offsets has n_nodes + 1 entries).  dst == NULL only
 * fills offsets (offsets[n_nodes] = bytes needed). */
int32_t dcdf_saved_all_bytes(dcdf_ctx* ctx, const dcdf_saved* saved, uint8_t* dst, uint64_t cap, uint64_t* offsets);
int32_t dcdf_saved_stats(const dcdf_saved* saved, dcdf_build_stats* stats);

/* Mapper::load stand-in (mapper.rs:10-38): hand out the stored bytes of a node; they must stay valid until the call that
 * received the callback returns.  Return 0 on success. */
typedef int32_t (*dcdf_fetch_fn)(void* user, const uint8_t* cid /* DCDF_CID_BYTES */, const uint8_t** bytes, uint64_t* len);
/* Superchunk::load_from (superchunk.rs:713-768) + Resolver::get_mmstruct3 / get_links for every External reference, for
 * the n_slices superchunk nodes of consecutive time slices of one array (what a Span holds, span.rs:50-110): every
 * stored Chunk is uploaded once and validated like Chunk::read_from, the min / max Dacs are decoded into the tables the
 * Elided cells and the search pruning read, and the result answers every dcdf_superchunk_* query.  All slices but the
 * last must have the same number of instants. */
int32_t dcdf_superchunk_open(dcdf_ctx* ctx, uint32_t n_slices, const uint8_t* root_cids /* n_slices x DCDF_CID_BYTES */,
                             dcdf_fetch_fn fetch, void* user, dcdf_superchunk** out);

#ifdef __cplusplus
}
#endif
#endif /* DCDF_CUDA_H */
