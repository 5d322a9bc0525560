// api_encode.cu -- C-ABI entry points for the encode half of the path (context, a1/a2/a3, Chunk::build,
// Superchunk::build).  Host logic only orchestrates: every data pass is a kernel in encode_tile.cuh,
// stats.cuh, gather.cuh.  No CPU fallback exists: without a device every call returns DCDF_ERR_CUDA.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <mutex>

#include "encode_big.cuh"
#include "encode_v4.cuh"
#include "encode_v5.cuh"
#include "gather.cuh"
#include "host.hpp"
#include "tree_geo.hpp"
#include "stats.cuh"
#include "xfer.cuh"

using namespace dcdf;

namespace dcdf {
void free_chunk_meta(void* p);
void free_super_meta(void* p);
}  // namespace dcdf

namespace {

int32_t status_from_flags(u32 f, std::string& msg) {
  if (f & EF_NONFINITE) { msg = "cannot convert a non-finite value to fixed point (fixed.rs:39-41)"; return DCDF_ERR_NONFINITE; }
  if (f & EF_OVERFLOW) { msg = "overflow converting to fixed point (fixed.rs:66-69)"; return DCDF_ERR_OVERFLOW; }
  if (f & EF_PRECISION) { msg = "loss of precision converting to fixed point (fixed.rs:51-57)"; return DCDF_ERR_PRECISION_LOSS; }
  if (f & EF_BAD_LEVELS) { msg = "tree levels passed in do not match the levels a nested sub-array needs (superchunk.rs:105-110)"; return DCDF_ERR_BAD_LEVELS; }
  if (f & EF_REGION_EXACT) { msg = "nested region with negatives far below its positive range needs the exact fraction pass, which is not built for nested superchunks yet"; return DCDF_ERR_BAD_ARG; }
  if (f & EF_BAD_FORMAT) { msg = "internal consistency check failed in the encoder"; return DCDF_ERR_BAD_FORMAT; }
  if (f & EF_OUT_CAP) { msg = "output buffer too small"; return DCDF_ERR_BAD_ARG; }
  return DCDF_OK;
}

size_t elem_size(int enc) { return (enc == DCDF_ENC_I32 || enc == DCDF_ENC_F32) ? 4 : 8; }

template <typename Fn>
int32_t guarded(dcdf_ctx* ctx, Fn&& fn) {
  if (!ctx) return DCDF_ERR_BAD_ARG;
  try {
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) throw CudaFail{std::string("cudaSetDevice: ") + cudaGetErrorString(e)};
    fn();
    return DCDF_OK;
  } catch (const ApiFail& f) {
    ctx->last_error = f.msg;
    return f.code;
  } catch (const CudaFail& f) {
    ctx->last_error = f.msg;
    cudaGetLastError();
    return DCDF_ERR_CUDA;
  } catch (const std::bad_alloc&) {
    ctx->last_error = "host out of memory";
    return DCDF_ERR_BAD_ARG;
  } catch (const std::exception& e) {  // nothing may unwind across the C ABI
    ctx->last_error = std::string("unexpected exception: ") + e.what();
    return DCDF_ERR_BAD_ARG;
  } catch (...) {
    ctx->last_error = "unexpected exception";
    return DCDF_ERR_BAD_ARG;
  }
}

void validate_array(const dcdf_array3* a) {
  if (!a || !a->base) api_fail(DCDF_ERR_BAD_ARG, "null array");
  if (a->encoding != DCDF_ENC_I32 && a->encoding != DCDF_ENC_I64 && a->encoding != DCDF_ENC_F32 && a->encoding != DCDF_ENC_F64)
    api_fail(DCDF_ERR_BAD_ARG, "bad encoding %d", a->encoding);
  for (int i = 0; i < 3; i++) {
    if (a->shape[i] <= 0) api_fail(DCDF_ERR_BAD_ARG, "empty array axis %d", i);
  }
  if (a->mem != DCDF_MEM_HOST && a->mem != DCDF_MEM_DEVICE) api_fail(DCDF_ERR_BAD_ARG, "bad mem kind");
}

// Returns a device pointer for element [0, 0, 0] of the array (copying a host view's spanned extent if needed; strides
// may be negative, as in a reversed ndarray view: mmbuffer.rs:573-594).
const void* stage_input(dcdf_ctx* ctx, const dcdf_array3* a) {
  if (a->mem == DCDF_MEM_DEVICE) return a->base;
  int64_t lo = 0, hi = 0;  // lowest / highest element offset the view touches
  for (int i = 0; i < 3; i++) {
    const int64_t ext = (a->shape[i] - 1) * a->strides[i];
    if (ext < 0) lo += ext; else hi += ext;
  }
  const size_t es = elem_size(a->encoding);
  const size_t bytes = (size_t)(hi - lo + 1) * es;
  ctx->input_copy.reserve(bytes);
  // One host-to-device engine per GPU: uploads of different contexts are queued first come first served and each one
  // runs at the full link rate, so the kernels and downloads of one context overlap the upload of the next instead of
  // all contexts uploading (and then computing) in lockstep.
  static std::mutex upload_mutex[64];
  std::lock_guard<std::mutex> lock(upload_mutex[ctx->device & 63]);
  CK(cudaMemcpyAsync(ctx->input_copy.p, static_cast<const char*>(a->base) + lo * (int64_t)es, bytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return static_cast<const char*>(ctx->input_copy.p) - lo * (int64_t)es;
}

struct EncodeJob {
  const void* dev_data = nullptr;
  int encoding = 0;
  int64_t strides[3] = {0, 0, 0};
  std::vector<EncUnit> units;
  std::vector<SliceDesc> slices;
  std::vector<uint64_t> table_len;
  uint32_t n_slots = 1;
  uint32_t t_max = 1;
  int plain = 0, req_bits = 0, round = 0, compute_bits = 0;
  int64_t rows = 0, cols = 0;  // full raster (exact pass)
  size_t input_bytes = 0;
  TreeGeo* tree = nullptr;     // node tree for superchunk builds (null: plain Chunk::build units)
};

struct EncodeOut {
  std::vector<EncUnit> units;  // with bits / flags
  std::vector<UnitResult> results;
  std::vector<uint8_t> stored;
  std::vector<uint64_t> chunk_off;
  std::vector<SliceState> states;
  std::vector<Piece> dac_pieces;
  std::vector<Piece> pieces;  // only fetched on request
  uint8_t* blob = nullptr;
  uint64_t blob_size = 0;
  uint8_t* dac_blob = nullptr;
  uint64_t dac_blob_size = 0;
  std::vector<uint64_t> dac_off;  // [n_slices][n_nodes][2]
  std::vector<NodeState> nstate;  // [n_slices][n_nodes]
  int64_t* tbl_max = nullptr;
  int64_t* tbl_min = nullptr;
  uint64_t tbl_total = 0;
};

template <typename InT, typename V, bool FULL, int MINB>
void launch_encode_one(dcdf_ctx* ctx, const EncParams& P, u32 grid) {
  const size_t smem = sizeof(EncSmem<V>);
  CK(cudaFuncSetAttribute(k_encode_tiles<InT, V, FULL, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_encode_tiles<InT, V, FULL, MINB><<<grid, ENC_THREADS, smem, FULL ? ctx->stream : ctx->aux_stream>>>(P);
  CK(cudaGetLastError());
  ctx->launches++;
}
// Full 64x64 tiles with 31-bit values: 64-thread CTAs, 64 cells per thread (encode_v4.cuh).
// Option "stage_limit" lowers the size above which a structure is emitted straight into the arena (tests use it to
// cover that path).
template <typename InT, bool FULL>
void launch_encode_v4(dcdf_ctx* ctx, const EncParams& P, u32 grid) {
  constexpr int MINB = 4;
  const u32 stage_limit = std::min<u32>(ctx->opt.stage_limit, (u32)E4_POOL);
  const size_t smem = sizeof(E4Smem);
  CK(cudaFuncSetAttribute(k_encode_v4<InT, MINB, FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_encode_v4<InT, MINB, FULL><<<grid, E4_THREADS, smem, FULL ? ctx->stream : ctx->aux_stream>>>(P, stage_limit);
  CK(cudaGetLastError());
  ctx->launches++;
}
// Full f32 tiles that qualify for the small fast-path kernel (encode_v5.cuh; list 5, filled by k_finalize_tree).
template <bool FULL>
void launch_encode_v5(dcdf_ctx* ctx, const EncParams& P, u32 grid) {
  constexpr int G = 6;  // tiles per CTA, one CTA per SM
  const u32 stage_limit = std::min<u32>(ctx->opt.stage_limit, (u32)E5_POOL);
  const size_t smem = sizeof(E5Smem<FULL>) * G;
  CK(cudaFuncSetAttribute(k_encode_v5<G, FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_encode_v5<G, FULL><<<(grid + G - 1) / G, E5_THREADS * G, smem, FULL ? ctx->stream : ctx->aux_stream>>>(P, stage_limit, E5_SYNC_MASK);
  CK(cudaGetLastError());
  ctx->launches++;
}
// Clipped fast-path tiles with at most 32 rows or columns in the raster (list 7): one warp per tile, twelve tiles per
// CTA (384 threads, like the six two-warp tiles of k_encode_v5).  ptxas (sm_100a): 168 registers, 352 / 604 bytes of
// spill stores / loads; E5SmemEdge is 18,720 bytes, so twelve tiles take 224,640 of the 232,448 bytes an SM offers.
void launch_encode_v5_edge(dcdf_ctx* ctx, const EncParams& P, u32 grid) {
  constexpr int G = 12;
  const u32 stage_limit = std::min<u32>(ctx->opt.stage_limit, (u32)E5_POOL_EDGE);
  const size_t smem = sizeof(E5SmemEdge) * G;
  CK(cudaFuncSetAttribute(k_encode_v5_edge<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_encode_v5_edge<G><<<(grid + G - 1) / G, 32 * G, smem, ctx->aux_stream>>>(P, stage_limit, E5_SYNC_MASK);
  CK(cudaGetLastError());
  ctx->launches++;
}
// list = wide * 2 + clipped  (narrow kernels are compiled for two resident CTAs per SM); 4 = clipped 64-side trees,
// 5 = fast path, 6 = clipped fast path, 7 = clipped fast path with half the tree outside the raster
template <typename InT>
void launch_encode(dcdf_ctx* ctx, const EncParams& P, u32 grid, int list) {
  if (grid == 0) return;
  if (list >= 5) {
    if (sizeof(InT) == 4) {  // k_finalize_tree only fills these lists for f32 input
      if (list == 5) launch_encode_v5<true>(ctx, P, grid);
      else if (list == 6) launch_encode_v5<false>(ctx, P, grid);
      else launch_encode_v5_edge(ctx, P, grid);
    }
    return;
  }
  if (list == 0) { launch_encode_v4<InT, true>(ctx, P, grid); return; }
  if (list == 4) { launch_encode_v4<InT, false>(ctx, P, grid); return; }
  switch (list) {
    case 1: launch_encode_one<InT, int32_t, false, 2>(ctx, P, grid); break;
    case 2: launch_encode_one<InT, i64, true, 1>(ctx, P, grid); break;
    default: launch_encode_one<InT, i64, false, 1>(ctx, P, grid); break;
  }
}

template <typename InT, bool IS_FLOAT>
void launch_stats(dcdf_ctx* ctx, const StatParams& P) {
  k_unit_stats<InT, IS_FLOAT><<<P.n_units, STAT_THREADS, 0, ctx->stream>>>(P);
  CK(cudaGetLastError());
  ctx->launches++;
}

void time_begin(dcdf_ctx* ctx, int which) { CK(cudaEventRecord(ctx->ev[2 * which], ctx->stream)); }
void time_end(dcdf_ctx* ctx, int which) { CK(cudaEventRecord(ctx->ev[2 * which + 1], ctx->stream)); }
void time_collect(dcdf_ctx* ctx, int which) {
  float ms = 0;
  if (cudaEventElapsedTime(&ms, ctx->ev[2 * which], ctx->ev[2 * which + 1]) == cudaSuccess) ctx->kernel_ms[which] = ms;
  else cudaGetLastError();
}

// Option "trace" prints host-side phase times of run_encode to stderr (adds stream syncs).
struct Tracer {
  bool on;
  cudaStream_t st;
  std::chrono::steady_clock::time_point t0;
  Tracer(cudaStream_t s, bool on_) : on(on_), st(s), t0(std::chrono::steady_clock::now()) {}
  void mark(const char* what) {
    if (!on) return;
    cudaStreamSynchronize(st);
    auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[dcdf trace] %-28s %9.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

// The whole encode pipeline for a list of <=64x64 units grouped in slices.
void run_encode(dcdf_ctx* ctx, EncodeJob& job, EncodeOut& out, bool want_pieces) {
  cudaStream_t st = ctx->stream;
  Tracer tr(st, ctx->opt.trace != 0);
  const u32 n_units = (u32)job.units.size();
  const u32 n_slices = (u32)job.slices.size();
  if (n_units == 0) api_fail(DCDF_ERR_BAD_ARG, "nothing to encode");
  u64 n_pieces = 0;
  for (auto& u : job.units) { u.piece_base = (u32)n_pieces; n_pieces += (u64)u.instants; }
  if (n_pieces > 0xfffffff0ull) api_fail(DCDF_ERR_BAD_ARG, "too many (unit, instant) pairs for one call");
  u64 tbl_total = 0;
  const u32 n_nodes = job.tree ? (u32)job.tree->nodes.size() : 1u;
  const u32 n_tables = n_slices * n_nodes;
  std::vector<uint64_t> table_base(n_tables), table_len(n_tables);
  for (u32 s = 0; s < n_slices; s++) {
    job.slices[s].table_base = tbl_total;
    for (u32 n = 0; n < n_nodes; n++) {
      const u64 off = job.tree ? (u64)job.tree->nodes[n].tbl_off : 0, nch = job.tree ? (u64)job.tree->nodes[n].n_children : 0;
      table_base[(size_t)s * n_nodes + n] = tbl_total + off * (u64)job.slices[s].instants;
      table_len[(size_t)s * n_nodes + n] = job.plain ? 0 : nch * (u64)job.slices[s].instants;
    }
    tbl_total += job.plain ? 0 : job.table_len[s];
  }

  // ---- device scratch
  ctx->units.reserve(sizeof(EncUnit) * n_units);
  ctx->ustats.reserve(sizeof(UnitStats) * n_units);
  ctx->istats.reserve(sizeof(InstStats) * (size_t)n_units * job.t_max);
  ctx->slices.reserve(sizeof(SliceDesc) * n_slices + 2 * sizeof(u64) * n_tables);
  ctx->sstate.reserve(sizeof(SliceState) * n_slices);
  ctx->order.reserve(sizeof(u32) * (8 * (size_t)n_units + 8));
  ctx->pieces.reserve(sizeof(Piece) * (n_pieces + 2 * (size_t)n_tables));
  ctx->results.reserve(sizeof(UnitResult) * n_units);
  ctx->stored.reserve(n_units);
  ctx->chunk_off.reserve(sizeof(u64) * ((size_t)n_units + 1));
  ctx->small.reserve(256);
  if (!job.plain) ctx->tbl_scratch.reserve(sizeof(u64) * 4 * tbl_total);
  int64_t *d_tbl_max = nullptr, *d_tbl_min = nullptr;
  if (!job.plain && tbl_total) {
    d_tbl_max = static_cast<int64_t*>(pool_alloc(sizeof(i64) * tbl_total, st));
    d_tbl_min = static_cast<int64_t*>(pool_alloc(sizeof(i64) * tbl_total, st));
  }
  out.tbl_max = d_tbl_max;
  out.tbl_min = d_tbl_min;
  out.tbl_total = tbl_total;

  // small: [0] err (u32) | [8] arena_head (u64) | [16] order counts (8 x u32)
  u32* d_err = ctx->small.as<u32>();
  unsigned long long* d_head = reinterpret_cast<unsigned long long*>(ctx->small.as<u8>() + 8);
  u32* d_counts = reinterpret_cast<u32*>(ctx->small.as<u8>() + 16);

  ctx->pin.reserve(sizeof(EncUnit) * n_units + sizeof(SliceDesc) * n_slices + 2 * sizeof(u64) * n_tables + 64);
  EncUnit* h_units = ctx->pin.as<EncUnit>();
  memcpy(h_units, job.units.data(), sizeof(EncUnit) * n_units);
  SliceDesc* h_slices = reinterpret_cast<SliceDesc*>(h_units + n_units);
  memcpy(h_slices, job.slices.data(), sizeof(SliceDesc) * n_slices);
  u64* h_tb = reinterpret_cast<u64*>(h_slices + n_slices);
  for (u32 i = 0; i < n_tables; i++) { h_tb[i] = table_base[i]; h_tb[n_tables + i] = table_len[i]; }
  copy_by_kernel(ctx, ctx->units.p, h_units, sizeof(EncUnit) * n_units);  // ctx->pin is pinned: read in place
  copy_by_kernel(ctx, ctx->slices.p, h_slices, sizeof(SliceDesc) * n_slices + 2 * sizeof(u64) * n_tables);
  const u64* d_table_base = reinterpret_cast<const u64*>(ctx->slices.as<SliceDesc>() + n_slices);
  const u64* d_table_len = d_table_base + n_tables;
  // static node tree + per-(slice, node) state
  TreeNode* d_nodes = nullptr;
  TreeChild* d_children = nullptr;
  int32_t* d_leaf_unit = nullptr;
  NodeState* d_nstate = nullptr;
  if (job.tree) {
    const TreeGeo& G = *job.tree;
    const size_t b0 = sizeof(TreeNode) * G.nodes.size(), b1 = sizeof(TreeChild) * G.children.size(),
                 b2 = sizeof(int32_t) * G.leaf_unit.size(), b3 = sizeof(NodeState) * (size_t)n_tables;
    ctx->tree_buf.reserve(b0 + b1 + b2 + b3 + 1024);
    u8* tb = ctx->tree_buf.as<u8>();
    d_nodes = reinterpret_cast<TreeNode*>(tb);
    d_children = reinterpret_cast<TreeChild*>(tb + ((b0 + 255) & ~size_t(255)));
    d_leaf_unit = reinterpret_cast<int32_t*>(reinterpret_cast<u8*>(d_children) + ((b1 + 255) & ~size_t(255)));
    d_nstate = reinterpret_cast<NodeState*>(reinterpret_cast<u8*>(d_leaf_unit) + ((b2 + 255) & ~size_t(255)));
    upload_small(ctx, d_nodes, G.nodes.data(), b0);
    upload_small(ctx, d_children, G.children.data(), b1);
    upload_small(ctx, d_leaf_unit, G.leaf_unit.data(), b2);
  }

  tr.mark("scratch + uploads");
  // ---- K1: per-unit statistics
  StatParams SP;
  SP.data = job.dev_data;
  SP.stride_t = job.strides[0]; SP.stride_r = job.strides[1]; SP.stride_c = job.strides[2];
  SP.units = ctx->units.as<EncUnit>();
  SP.n_units = n_units;
  SP.t_max = job.t_max;
  SP.ustats = ctx->ustats.as<UnitStats>();
  SP.istats = ctx->istats.as<InstStats>();
  time_begin(ctx, KT_STATS);
  switch (job.encoding) {
    case DCDF_ENC_F32: launch_stats<float, true>(ctx, SP); break;
    case DCDF_ENC_F64: launch_stats<double, true>(ctx, SP); break;
    case DCDF_ENC_I32: launch_stats<int32_t, false>(ctx, SP); break;
    default: launch_stats<i64, false>(ctx, SP); break;
  }
  time_end(ctx, KT_STATS);
  tr.mark("k_unit_stats");

  // ---- K1b: slice finalisation
  FinalizeParams FP;
  FP.slices = ctx->slices.as<SliceDesc>();
  FP.state = ctx->sstate.as<SliceState>();
  FP.units_in = ctx->units.as<EncUnit>();
  FP.units = ctx->units.as<EncUnit>();
  FP.ustats = SP.ustats;
  FP.istats = SP.istats;
  FP.t_max = job.t_max;
  FP.n_slots = job.n_slots;
  FP.encoding = job.encoding;
  FP.req_bits = job.req_bits; FP.round = job.round; FP.compute_bits = job.compute_bits; FP.plain = job.plain;
  FP.tbl_min = d_tbl_min; FP.tbl_max = d_tbl_max;
  FP.order = ctx->order.as<u32>();
  FP.order_pitch = n_units;
  FP.order_counts = d_counts;
  FP.stored = ctx->stored.as<u8>();
  FP.err = d_err;
  CK(cudaMemsetAsync(ctx->small.p, 0, 64, st));
  k_finalize_phase1<<<n_slices, 256, 0, st>>>(FP, n_slices);
  CK(cudaGetLastError());
  ctx->launches++;
  const bool is_float = job.encoding == DCDF_ENC_F32 || job.encoding == DCDF_ENC_F64;
  if (is_float && job.compute_bits) {
    // Exact slice-level pass, needed only when a negative value may hit the saturating cast of
    // fixed.rs:150 (rare).  The flags are a few bytes per slice, read back once per call.
    SliceState* ss = ctx->sstate.as<SliceState>();
    std::vector<SliceState> hs(n_slices);
    read_small(ctx, hs.data(), ss, sizeof(SliceState) * n_slices);
    sync_reads(ctx);
    bool any = false;
    for (auto& s : hs) any = any || s.need_exact;
    if (any) {
      ctx->exact.reserve((sizeof(i64) + 5 * sizeof(int)) * n_slices + 64);
      std::vector<i64> t0(n_slices);
      std::vector<int> inst(n_slices);
      for (u32 s = 0; s < n_slices; s++) { t0[s] = job.slices[s].t0; inst[s] = job.slices[s].instants; }
      i64* d_t0 = ctx->exact.as<i64>();
      int* d_inst = reinterpret_cast<int*>(d_t0 + n_slices);
      upload_small(ctx, d_t0, t0.data(), sizeof(i64) * n_slices);
      upload_small(ctx, d_inst, inst.data(), sizeof(int) * n_slices);
      ExactParams XP;
      XP.data = job.dev_data;
      XP.stride_t = job.strides[0]; XP.stride_r = job.strides[1]; XP.stride_c = job.strides[2];
      XP.rows = job.rows; XP.cols = job.cols;
      XP.slice_t0 = d_t0; XP.slice_instants = d_inst;
      std::vector<int> need(n_slices), maxfb(n_slices);
      for (u32 s = 0; s < n_slices; s++) { need[s] = hs[s].need_exact; maxfb[s] = hs[s].maxfb; }
      int* d_need = d_inst + n_slices;
      int* d_maxfb = d_need + n_slices;
      int* d_f = d_maxfb + n_slices;
      int* d_round = d_f + n_slices;
      upload_small(ctx, d_need, need.data(), sizeof(int) * n_slices);
      upload_small(ctx, d_maxfb, maxfb.data(), sizeof(int) * n_slices);
      CK(cudaMemsetAsync(d_f, 0, 2 * sizeof(int) * n_slices, st));
      XP.slice_need = d_need; XP.slice_maxfb = d_maxfb; XP.slice_f = d_f; XP.slice_round = d_round;
      dim3 grid((unsigned)std::min<int64_t>(4 * ctx->sm_count, 65535), n_slices);
      if (job.encoding == DCDF_ENC_F32) k_fraction_exact<float><<<grid, 256, 0, st>>>(XP, n_slices);
      else k_fraction_exact<double><<<grid, 256, 0, st>>>(XP, n_slices);
      CK(cudaGetLastError());
      ctx->launches++;
      std::vector<int> f(n_slices), r(n_slices);
      read_small(ctx, f.data(), d_f, sizeof(int) * n_slices);
      read_small(ctx, r.data(), d_round, sizeof(int) * n_slices);
      sync_reads(ctx);
      for (u32 s = 0; s < n_slices; s++) { hs[s].f_exact = f[s]; hs[s].round_exact = r[s]; }
      upload_small(ctx, ss, hs.data(), sizeof(SliceState) * n_slices);
    }
  }
  if (job.tree) {
    const TreeGeo& G = *job.tree;
    TreeParams TP;
    TP.slices = FP.slices; TP.state = FP.state;
    TP.nodes = d_nodes; TP.children = d_children; TP.n_nodes = n_nodes;
    TP.leaf_unit = d_leaf_unit; TP.leaf_cols = G.leaf_cols; TP.leaf_side = G.leaf_side;
    TP.tbl_per_instant = G.tbl_per_instant;
    TP.nstate = d_nstate;
    TP.units = ctx->units.as<EncUnit>();
    TP.ustats = SP.ustats; TP.istats = SP.istats; TP.t_max = job.t_max;
    TP.encoding = job.encoding; TP.round = job.round; TP.req_bits = job.req_bits;
    TP.allow_fast = job.encoding == DCDF_ENC_F32 && !ctx->opt.no_fast_encode && job.strides[2] == 1;  // k_encode_v5 reads rows of four cells
    TP.tbl_min = d_tbl_min; TP.tbl_max = d_tbl_max;
    TP.order = FP.order; TP.order_pitch = FP.order_pitch; TP.order_counts = FP.order_counts;
    TP.stored = FP.stored; TP.err = d_err;
    k_finalize_tree<<<n_slices, 256, 0, st>>>(TP, n_slices);
  } else {
    k_finalize_phase2<<<n_slices, 256, 0, st>>>(FP, n_slices);
  }
  CK(cudaGetLastError());
  ctx->launches++;

  tr.mark("finalize");
  // ---- K_enc (+ table DACs), with arena growth on overflow
  if (ctx->arena_hint == 0) ctx->arena_hint = std::max<size_t>(job.input_bytes / 2 + (8u << 20), 16u << 20);
  std::vector<uint8_t> head_buf(64);
  u32 sticky = 0;  // flags raised before the emission (finalize / fraction passes) survive an arena retry
  for (int attempt = 0;; attempt++) {
    ctx->arena.reserve(ctx->arena_hint);
    const u64 arena_cap = ctx->arena.cap;
    CK(cudaMemsetAsync(d_head, 0, 8, st));
    EncParams EP;
    EP.data = job.dev_data;
    EP.stride_t = job.strides[0]; EP.stride_r = job.strides[1]; EP.stride_c = job.strides[2];
    EP.units = ctx->units.as<EncUnit>();
    EP.pieces = ctx->pieces.as<Piece>();
    EP.results = ctx->results.as<UnitResult>();
    EP.arena = ctx->arena.as<u8>();
    EP.arena_cap = arena_cap;
    EP.arena_head = d_head;
    EP.err = d_err;
    time_begin(ctx, KT_ENCODE);
    CK(cudaEventRecord(ctx->fork_ev, st));  // clipped-tile lists run on the auxiliary stream beside the full-tile lists
    CK(cudaStreamWaitEvent(ctx->aux_stream, ctx->fork_ev, 0));
    for (int list = 7; list >= 0; list--) {  // the fast-path lists (most units of a typical raster) go first
      EP.order = FP.order + (size_t)list * n_units;
      EP.order_count = d_counts + list;
      switch (job.encoding) {
        case DCDF_ENC_F32: launch_encode<float>(ctx, EP, n_units, list); break;
        case DCDF_ENC_F64: launch_encode<double>(ctx, EP, n_units, list); break;
        case DCDF_ENC_I32: launch_encode<int32_t>(ctx, EP, n_units, list); break;
        default: launch_encode<i64>(ctx, EP, n_units, list); break;
      }
    }
    CK(cudaEventRecord(ctx->join_ev, ctx->aux_stream));
    CK(cudaStreamWaitEvent(st, ctx->join_ev, 0));
    time_end(ctx, KT_ENCODE);
    tr.mark("k_encode_tiles");
    if (!job.plain) {
      TableDacParams TP;
      TP.tbl_min = d_tbl_min; TP.tbl_max = d_tbl_max;
      TP.table_base = d_table_base; TP.table_len = d_table_len;
      TP.alive = reinterpret_cast<const int*>(d_nstate);
      TP.scratch = ctx->tbl_scratch.as<u64>();
      TP.total = tbl_total;
      TP.pieces = ctx->pieces.as<Piece>() + n_pieces;
      TP.arena = ctx->arena.as<u8>(); TP.arena_cap = arena_cap; TP.arena_head = d_head; TP.err = d_err;
      k_table_dac<<<dim3(n_tables, 2), ENC_THREADS, 0, st>>>(TP);
      CK(cudaGetLastError());
      ctx->launches++;
    }
    tr.mark("k_table_dac");
    k_scan_units<<<1, 1024, 0, st>>>(ctx->results.as<UnitResult>(), ctx->stored.as<u8>(), n_units, ctx->chunk_off.as<u64>());
    CK(cudaGetLastError());
    ctx->launches++;
    read_small(ctx, head_buf.data(), ctx->small.p, 64);
    sync_reads(ctx);
    u32 flags;
    u64 head;
    memcpy(&flags, head_buf.data(), 4);
    memcpy(&head, head_buf.data() + 8, 8);
    memcpy(ctx->last_list_counts, head_buf.data() + 16, sizeof ctx->last_list_counts);
    sticky |= flags & ~(u32)EF_ARENA_FULL;
    std::string msg;
    if ((flags & EF_ARENA_FULL) && status_from_flags(sticky, msg) == DCDF_OK) {
      if (attempt >= 3) api_fail(DCDF_ERR_CUDA, "arena overflow persisted after growth");
      ctx->arena_hint = (size_t)head + (size_t)head / 16 + (1u << 20);
      CK(cudaMemsetAsync(d_err, 0, 4, st));
      // phase-2 outputs (order lists, unit bits) are still valid; only the emission is repeated
      continue;
    }
    flags = sticky;
    int32_t code = status_from_flags(flags, msg);
    if (code != DCDF_OK) {
      pool_free(d_tbl_max);
      pool_free(d_tbl_min);
      out.tbl_max = out.tbl_min = nullptr;
      throw ApiFail{code, msg};
    }
    break;
  }
  time_collect(ctx, KT_STATS);
  time_collect(ctx, KT_ENCODE);
  tr.mark("scan + flags readback");

  // ---- read back the small per-unit tables
  out.units.resize(n_units);
  out.results.resize(n_units);
  out.stored.resize(n_units);
  out.chunk_off.resize((size_t)n_units + 1);
  out.states.resize(n_slices);
  read_small(ctx, out.units.data(), ctx->units.p, sizeof(EncUnit) * n_units);
  read_small(ctx, out.results.data(), ctx->results.p, sizeof(UnitResult) * n_units);
  read_small(ctx, out.stored.data(), ctx->stored.p, n_units);
  read_small(ctx, out.chunk_off.data(), ctx->chunk_off.p, sizeof(u64) * ((size_t)n_units + 1));
  read_small(ctx, out.states.data(), ctx->sstate.p, sizeof(SliceState) * n_slices);
  if (!job.plain) {
    out.dac_pieces.resize(2 * (size_t)n_tables);
    read_small(ctx, out.dac_pieces.data(), ctx->pieces.as<Piece>() + n_pieces, sizeof(Piece) * 2 * n_tables);
    out.nstate.resize(n_tables);
    read_small(ctx, out.nstate.data(), d_nstate, sizeof(NodeState) * n_tables);
  }
  if (want_pieces) {
    out.pieces.resize(n_pieces);
    CK(cudaMemcpyAsync(out.pieces.data(), ctx->pieces.p, sizeof(Piece) * n_pieces, cudaMemcpyDeviceToHost, st));
  }
  sync_reads(ctx);

  tr.mark("tables readback");
  // ---- final blobs
  out.blob_size = out.chunk_off[n_units];
  out.blob = static_cast<uint8_t*>(pool_alloc(out.blob_size + 64, st));  // padding: decoders read aligned 16-byte blocks past the last byte
  CK(cudaMemsetAsync(out.blob + out.blob_size, 0, 64, st));
  GatherParams GP;
  GP.units = ctx->units.as<EncUnit>();
  GP.results = ctx->results.as<UnitResult>();
  GP.stored = ctx->stored.as<u8>();
  GP.pieces = ctx->pieces.as<Piece>();
  GP.chunk_off = ctx->chunk_off.as<u64>();
  GP.arena = ctx->arena.as<u8>();
  GP.out = out.blob;
  GP.out_cap = out.blob_size;
  GP.encoding = job.encoding;
  GP.n_units = n_units;
  GP.err = d_err;
  tr.mark("blob alloc");
  time_begin(ctx, KT_GATHER);
  k_gather_chunks<<<n_units, 256, 0, st>>>(GP);
  CK(cudaGetLastError());
  ctx->launches++;
  if (!job.plain) {
    out.dac_off.resize(2 * (size_t)n_tables);
    u64 off = 0;
    for (u32 i = 0; i < 2 * n_tables; i++) { out.dac_off[i] = off; off += out.dac_pieces[i].size; }
    out.dac_blob_size = off;
    out.dac_blob = static_cast<uint8_t*>(pool_alloc(off + 16, st));
    ctx->query_aux.reserve(sizeof(u64) * 2 * n_tables);
    upload_small(ctx, ctx->query_aux.p, out.dac_off.data(), sizeof(u64) * 2 * n_tables);
    GatherDacParams DP;
    DP.pieces = ctx->pieces.as<Piece>() + n_pieces;
    DP.dst_off = ctx->query_aux.as<u64>();
    DP.arena = ctx->arena.as<u8>();
    DP.out = out.dac_blob;
    k_gather_dacs<<<2 * n_tables, 256, 0, st>>>(DP);
    CK(cudaGetLastError());
    ctx->launches++;
  }
  time_end(ctx, KT_GATHER);
  read_small(ctx, head_buf.data(), ctx->small.p, 4);
  sync_reads(ctx);
  time_collect(ctx, KT_GATHER);
  tr.mark("gather");
  u32 flags;
  memcpy(&flags, head_buf.data(), 4);
  flags |= sticky;
  std::string msg;
  int32_t code = status_from_flags(flags, msg);
  if (code != DCDF_OK) throw ApiFail{code, msg};
}


// ===================================================================================== big Chunk::build
// Chunk::build for padded sides above 64 (encode_big.cuh).  Host-driven: one small counter readback per
// instant for the Snapshot-vs-Log decision (chunk.rs:62); every data pass is a kernel.
struct BigResult {
  uint8_t* blob = nullptr;
  uint64_t size = 0;
  uint32_t snapshots = 0, logs = 0;
  std::vector<uint32_t> block_instants;
};

struct BigScratch {
  dcdf_ctx* ctx;
  u8* base = nullptr;
  size_t used = 0, cap = 0;
  template <typename T>
  T* take(size_t n) {
    used = (used + 255) & ~size_t(255);
    T* p = reinterpret_cast<T*>(base + used);
    used += n * sizeof(T);
    return p;
  }
};

unsigned big_grid(dcdf_ctx* ctx, u64 n, int block = 256) {
  return (unsigned)std::max<u64>(1, std::min<u64>((n + block - 1) / block, (u64)ctx->sm_count * 16));
}

// out[i] = exclusive prefix of in[0..n)
void big_scan(dcdf_ctx* ctx, const u64* in, u64 n, u64* out, u64* block_sums) {
  if (n == 0) return;
  const unsigned nb = (unsigned)((n + SCAN_ITEMS - 1) / SCAN_ITEMS);
  kb_scan_blocks<<<nb, 1024, 0, ctx->stream>>>(in, n, out, block_sums);
  CK(cudaGetLastError());
  ctx->launches++;
  if (nb > 1) {
    kb_scan_top<<<1, 1024, 0, ctx->stream>>>(block_sums, nb);
    kb_scan_add<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(out, n, block_sums);
    CK(cudaGetLastError());
    ctx->launches += 2;
  }
}

u32 host_dac_size(const unsigned long long* h) {
  u32 c[8];
  for (int j = 0; j < 8; j++) c[j] = (u32)h[j];
  return dac_size_from_counts(c, 8);
}

template <typename InT>
void big_chunk_encode(dcdf_ctx* ctx, const void* dev_data, const int64_t* strides, int encoding, int64_t T, int64_t rows,
                      int64_t cols, int bits, int round, BigResult& R) {
  cudaStream_t st = ctx->stream;
  const int L = (int)levels_for(std::max(rows, cols), 2);
  if (L > 12) api_fail(DCDF_ERR_BAD_ARG, "rasters larger than 4096 x 4096 must be split into a superchunk");
  const u64 side = 1ull << L, N = (u64)big_lvl_off(L + 1), n_upper = (u64)big_lvl_off(L);
  const u64 n_blocks_scan = (N + SCAN_ITEMS - 1) / SCAN_ITEMS + 1;
  // ---- scratch
  size_t need = 5 * N * 8 + N + 5 * N * 8 + 2 * (n_upper + 64) + 2 * (N / 32 + 64) * 8 + n_blocks_scan * 8 + sizeof(BigCounts) + 64 * 1024;
  ctx->tbl_scratch.reserve(need);
  BigScratch S{ctx, ctx->tbl_scratch.as<u8>(), 0, ctx->tbl_scratch.cap};
  BigPyr P;
  P.tmax = S.take<i64>(N); P.tmin = S.take<i64>(N); P.smax = S.take<i64>(N); P.smin = S.take<i64>(N); P.diff = S.take<i64>(N);
  P.fl = S.take<u8>(N);
  P.L = L; P.N = N;
  u64* scan = S.take<u64>(N);
  u64* A = S.take<u64>(N);
  u64* B = S.take<u64>(N);
  u64* Cb = S.take<u64>(N);
  u64* more = S.take<u64>(N);
  u8* nmf = S.take<u8>(n_upper + 64);
  u8* eqf = S.take<u8>(n_upper + 64);
  u64* popc = S.take<u64>(N / 32 + 64);
  u64* popc_scan = S.take<u64>(N / 32 + 64);
  u64* block_sums = S.take<u64>(n_blocks_scan);
  BigCounts* d_counts = S.take<BigCounts>(1);
  ctx->small.reserve(256);
  u32* d_err = ctx->small.as<u32>();
  CK(cudaMemsetAsync(d_err, 0, 64, st));
  CK(cudaMemsetAsync(P.smax, 0, N * 8, st));
  // ---- arena (host-side bump allocation; grown by copy when it fills up)
  if (ctx->arena.cap < (64u << 20)) ctx->arena.reserve(64u << 20);
  u64 head = 0;
  std::vector<Piece> pieces((size_t)T);
  const InT* data = static_cast<const InT*>(dev_data);
  uint32_t n_logs = 0, run = 0;
  u64 total_bytes = 6;
  for (int64_t inst = 0; inst < T; inst++) {
    const bool first = inst == 0;
    kb_leaves<InT><<<big_grid(ctx, side * side), 256, 0, st>>>(data + inst * strides[0], strides[1], strides[2], (int)rows, (int)cols, bits,
                                                              round, P, d_err);
    for (int l = L - 1; l >= 0; l--) kb_reduce<<<big_grid(ctx, 1ull << (2 * l)), 256, 0, st>>>(P, l);
    CK(cudaMemsetAsync(d_counts, 0, sizeof(BigCounts), st));
    kb_classify<<<big_grid(ctx, N), 256, 0, st>>>(P, first ? 1 : 0, d_counts);
    CK(cudaGetLastError());
    ctx->launches += 2 + L;
    BigCounts hc;
    CK(cudaMemcpyAsync(&hc, d_counts, sizeof hc, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    // sizes (snapshot.rs:84-93, log.rs:92-98) and the heuristic (chunk.rs:62)
    const u32 snap_size = 13u + bitmap_size((u32)hc.n_upper[0]) + host_dac_size(hc.h[0][0]) + host_dac_size(hc.h[0][1]);
    const u32 log_size = 13u + bitmap_size((u32)hc.n_upper[1]) + bitmap_size((u32)(hc.n_upper[1] - hc.n_int[1])) +
                         host_dac_size(hc.h[1][0]) + host_dac_size(hc.h[1][1]);
    const bool snap = first || n_logs == 254u || snap_size <= log_size;
    const int cand = snap ? 0 : 1;
    const u32 size = snap ? snap_size : log_size;
    const u64 need_bytes = ((u64)size + 15ull) & ~15ull;
    if (head + need_bytes > ctx->arena.cap) {  // grow, keeping what was already emitted
      DevBuf bigger;
      bigger.reserve((size_t)std::max<u64>(2 * ctx->arena.cap, head + need_bytes + (64u << 20)));
      CK(cudaMemcpyAsync(bigger.p, ctx->arena.p, head, cudaMemcpyDeviceToDevice, st));
      CK(cudaStreamSynchronize(st));
      ctx->arena.release();
      ctx->arena = bigger;
    }
    u8* out = ctx->arena.as<u8>() + head;
    pieces[(size_t)inst] = Piece{head, size, snap ? 1u : 0u};
    head += need_bytes;
    // ---- emit the winner
    const u64 nm_len = hc.n_upper[cand], n_int = hc.n_int[cand];
    kb_scan_input<<<big_grid(ctx, N), 256, 0, st>>>(P, cand, more);
    big_scan(ctx, more, N, scan, block_sums);
    kb_scatter<<<big_grid(ctx, N), 256, 0, st>>>(P, cand, scan, A, B, nmf, eqf);
    kb_header<<<1, 1, 0, st>>>(out, (int)rows, (int)cols, (int)side);
    ctx->launches += 3;
    u64 off = 13;
    auto emit_bitmap = [&](const u8* flags, u64 length) {
      const u64 words = (length + 31) / 32, blocks = length / 128;
      kb_bitmap_words<<<(unsigned)std::max<u64>(1, (words * 32 + 255) / 256), 256, 0, st>>>(flags, length, out + off + 8 + 4 * blocks, popc);
      big_scan(ctx, popc, words, popc_scan, block_sums);
      kb_bitmap_index<<<(unsigned)std::max<u64>(1, (blocks + 255) / 256), 256, 0, st>>>(popc_scan, popc, length, out + off);
      ctx->launches += 2;
      off += 8 + 4 * blocks + 4 * words;
    };
    emit_bitmap(nmf, nm_len);
    if (!snap) emit_bitmap(eqf, nm_len - n_int);
    auto emit_dac = [&](u64* X, const unsigned long long* h) {
      int n_levels = 0;
      for (int j = 0; j < 8; j++) if (h[j] > 0) n_levels = j + 1;
      kb_byte<<<1, 1, 0, st>>>(out + off, (u8)n_levels);
      ctx->launches++;
      off += 1;
      u64* Y = Cb;
      for (int j = 0; j < n_levels; j++) {
        const u64 nj = h[j];
        const unsigned g = (unsigned)((nj + 255) / 256);
        kb_dac_more<<<g, 256, 0, st>>>(X, nj, more);
        big_scan(ctx, more, nj, scan, block_sums);
        kb_dac_level<<<g, 256, 0, st>>>(X, nj, scan, out + off, Y);
        ctx->launches += 2;
        off += 8 + 4 * (nj / 128) + 4 * ((nj + 31) / 32) + nj;
        std::swap(X, Y);
      }
    };
    emit_dac(A, hc.h[cand][0]);
    emit_dac(B, hc.h[cand][1]);
    CK(cudaGetLastError());
    if (off != size) api_fail(DCDF_ERR_BAD_FORMAT, "big chunk: emitted %llu bytes, predicted %u", (unsigned long long)off, size);
    if (snap) {
      kb_copy_ts<<<big_grid(ctx, N), 256, 0, st>>>(P);
      ctx->launches++;
      if (!first) R.block_instants.push_back(run);
      run = 0;
      R.snapshots++;
      n_logs = 0;
      total_bytes += 1;
    } else {
      n_logs++;
      R.logs++;
    }
    run++;
    total_bytes += size;
  }
  R.block_instants.push_back(run);
  u32 flags = 0;
  CK(cudaMemcpyAsync(&flags, d_err, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  std::string msg;
  int32_t code = status_from_flags(flags, msg);
  if (code != DCDF_OK) throw ApiFail{code, msg};
  // ---- frame the pieces as Chunk bytes (chunk.rs:235-243, block.rs:88-95)
  if ((u64)T > 0xfffffff0ull) api_fail(DCDF_ERR_BAD_ARG, "too many instants");
  ctx->pieces.reserve(sizeof(Piece) * (size_t)T);
  ctx->units.reserve(sizeof(EncUnit));
  ctx->results.reserve(sizeof(UnitResult));
  ctx->stored.reserve(16);
  ctx->chunk_off.reserve(16);
  EncUnit eu;
  memset(&eu, 0, sizeof eu);
  eu.rows = (int)rows; eu.cols = (int)cols; eu.instants = (int)T; eu.bits = bits; eu.piece_base = 0;
  UnitResult ur;
  ur.bytes = total_bytes; ur.snapshots = R.snapshots; ur.logs = R.logs;
  const u8 one = 1;
  const u64 zero = 0;
  CK(cudaMemcpyAsync(ctx->pieces.p, pieces.data(), sizeof(Piece) * (size_t)T, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->units.p, &eu, sizeof eu, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->results.p, &ur, sizeof ur, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->stored.p, &one, 1, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->chunk_off.p, &zero, 8, cudaMemcpyHostToDevice, st));
  R.size = total_bytes;
  R.blob = static_cast<uint8_t*>(pool_alloc(total_bytes + 64, st));
  CK(cudaMemsetAsync(R.blob + total_bytes, 0, 64, st));
  GatherParams GP;
  GP.units = ctx->units.as<EncUnit>();
  GP.results = ctx->results.as<UnitResult>();
  GP.stored = ctx->stored.as<u8>();
  GP.pieces = ctx->pieces.as<Piece>();
  GP.chunk_off = ctx->chunk_off.as<u64>();
  GP.arena = ctx->arena.as<u8>();
  GP.out = R.blob;
  GP.out_cap = total_bytes;
  GP.encoding = encoding;
  GP.n_units = 1;
  GP.err = d_err;
  k_gather_chunks<<<1, 256, 0, st>>>(GP);
  CK(cudaGetLastError());
  ctx->launches++;
  CK(cudaMemcpyAsync(&flags, d_err, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  code = status_from_flags(flags, msg);
  if (code != DCDF_OK) { pool_free(R.blob); R.blob = nullptr; throw ApiFail{code, msg}; }
}

void copy_out(dcdf_ctx* ctx, const uint8_t* dev_src, uint64_t n, uint8_t* dst, uint64_t cap, int32_t mem) {
  if (!dst) api_fail(DCDF_ERR_BAD_ARG, "null destination");
  if (cap < n) api_fail(DCDF_ERR_BAD_ARG, "destination too small: need %llu bytes", (unsigned long long)n);
  if (n == 0) return;
  CK(cudaMemcpyAsync(dst, dev_src, n, mem == DCDF_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
}

}  // namespace

// ===================================================================================== context
extern "C" {

int32_t dcdf_abi_version(void) { return DCDF_ABI_VERSION; }

int32_t dcdf_ctx_create(int32_t device, dcdf_ctx** out) {
  if (!out) return DCDF_ERR_BAD_ARG;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0 || device < 0 || device >= n) {
    cudaGetLastError();
    return DCDF_ERR_CUDA;  // no CPU fallback
  }
  dcdf_ctx* ctx = new dcdf_ctx();
  ctx->device = device;
  try {
    CK(cudaSetDevice(device));
    upload_log2_roundup_table();  // a1: floor(log2(max)) exactly as the host libm rounds it (fixed.rs:126)
    CK(cudaGetLastError());
    CK(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    for (auto& ev : ctx->ev) CK(cudaEventCreate(&ev));
    CK(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ctx->fork_ev, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->join_ev, cudaEventDisableTiming));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    cudaMemPool_t pool;
    CK(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t keep = UINT64_MAX;  // keep freed result buffers cached in the pool
    CK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
  } catch (const CudaFail&) {
    delete ctx;
    cudaGetLastError();
    return DCDF_ERR_CUDA;
  }
  *out = ctx;
  return DCDF_OK;
}

int32_t dcdf_ctx_destroy(dcdf_ctx* ctx) {
  if (!ctx) return DCDF_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  DevBuf* bufs[] = {&ctx->input_copy, &ctx->units, &ctx->ustats, &ctx->istats, &ctx->slices, &ctx->sstate, &ctx->tbl_scratch,
                    &ctx->order, &ctx->pieces, &ctx->results, &ctx->stored, &ctx->chunk_off, &ctx->arena, &ctx->small,
                    &ctx->exact, &ctx->query_in, &ctx->query_out, &ctx->query_aux, &ctx->query_aux2, &ctx->search_cache, &ctx->tree_buf};
  for (auto* b : bufs) b->release();
  ctx->pin.release();
  ctx->pin2.release();
  ctx->xfer_up.release();
  ctx->xfer_down.release();
  for (auto& ev : ctx->ev) if (ev) cudaEventDestroy(ev);
  if (ctx->fork_ev) cudaEventDestroy(ctx->fork_ev);
  if (ctx->join_ev) cudaEventDestroy(ctx->join_ev);
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
  return DCDF_OK;
}

int32_t dcdf_ctx_set_stream(dcdf_ctx* ctx, void* cuda_stream) {
  if (!ctx) return DCDF_ERR_BAD_ARG;
  ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
  return DCDF_OK;
}

int32_t dcdf_ctx_set_option(dcdf_ctx* ctx, const char* name, int64_t value) {
  if (!ctx || !name) return DCDF_ERR_BAD_ARG;
  const std::string n(name);
  if (n == "stage_limit") ctx->opt.stage_limit = value < 0 ? 0xffffffffu : (uint32_t)std::min<int64_t>(value, 0xffffffffll);
  else if (n == "arena_hint") ctx->arena_hint = value < 0 ? 0 : (size_t)value;
  else if (n == "no_fast_encode") ctx->opt.no_fast_encode = value != 0;
  else if (n == "search_share_min") ctx->opt.search_share_min = (uint32_t)std::max<int64_t>(value, 0);
  else if (n == "cell_tile_min") ctx->opt.cell_tile_min = (uint32_t)std::max<int64_t>(value, 0);
  else if (n == "window_cells") ctx->opt.window_cells = value != 0;
  else if (n == "window_wide") ctx->opt.window_wide = value != 0;
  else if (n == "search_dfs") ctx->opt.search_dfs = value != 0;
  else if (n == "search_no_cache") ctx->opt.search_no_cache = value != 0;
  else if (n == "trace") ctx->opt.trace = value != 0;
  else if (n == "time_stats_scratch") ctx->opt.time_stats_scratch = value <= 0 ? 1ull << 30 : (uint64_t)value;
  else {
    ctx->last_error = "unknown option " + n;
    return DCDF_ERR_BAD_ARG;
  }
  return DCDF_OK;
}

int32_t dcdf_ctx_get_stat(const dcdf_ctx* ctx, const char* name, int64_t* value) {
  if (!ctx || !name || !value) return DCDF_ERR_BAD_ARG;
  const std::string n(name);
  const uint32_t* c = ctx->last_list_counts;
  if (n == "encode_units_fast") *value = (int64_t)c[5] + c[6] + c[7];
  else if (n == "encode_units_edge") *value = (int64_t)c[7];
  else if (n == "encode_units_general") *value = (int64_t)c[0] + c[1] + c[2] + c[3] + c[4];
  else if (n == "encode_units_wide") *value = (int64_t)c[2] + c[3];
  else if (n == "encode_units_clipped") *value = (int64_t)c[1] + c[3] + c[4] + c[6] + c[7];
  else if (n == "time_stats_groups") *value = (int64_t)ctx->last_time_groups;
  else if (n == "time_stats_scratch_bytes") *value = (int64_t)ctx->last_time_scratch;
  else return DCDF_ERR_BAD_ARG;
  return DCDF_OK;
}

int32_t dcdf_ctx_synchronize(dcdf_ctx* ctx) {
  return guarded(ctx, [&] { CK(cudaStreamSynchronize(ctx->stream)); });
}

const char* dcdf_last_error(const dcdf_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
uint64_t dcdf_ctx_launch_count(const dcdf_ctx* ctx) { return ctx ? ctx->launches : 0; }
int32_t dcdf_ctx_last_kernel_ms(const dcdf_ctx* ctx, int32_t which, float* ms) {
  if (!ctx || !ms || which < 0 || which >= KT_COUNT) return DCDF_ERR_BAD_ARG;
  *ms = ctx->kernel_ms[which];
  return DCDF_OK;
}

// ===================================================================================== a1 / a2
// Tile an arbitrary [T,R,C] array into <=64x64 units that span all instants (statistics only).
static void tile_units(const dcdf_array3* a, std::vector<EncUnit>& units) {
  const int64_t rows = a->shape[1], cols = a->shape[2];
  for (int64_t top = 0; top < rows; top += 64)
    for (int64_t left = 0; left < cols; left += 64) {
      EncUnit u;
      memset(&u, 0, sizeof u);
      u.base = top * a->strides[1] + left * a->strides[2];
      u.rows = (int)std::min<int64_t>(64, rows - top);
      u.cols = (int)std::min<int64_t>(64, cols - left);
      u.instants = (int)a->shape[0];
      u.row0 = (int)top; u.col0 = (int)left;
      units.push_back(u);
    }
}

static void run_unit_stats(dcdf_ctx* ctx, const dcdf_array3* a, const void* dev, const std::vector<EncUnit>& units) {
  const u32 n_units = (u32)units.size();
  ctx->units.reserve(sizeof(EncUnit) * n_units);
  ctx->ustats.reserve(sizeof(UnitStats) * n_units);
  ctx->istats.reserve(sizeof(InstStats) * (size_t)n_units * (size_t)a->shape[0]);
  CK(cudaMemcpyAsync(ctx->units.p, units.data(), sizeof(EncUnit) * n_units, cudaMemcpyHostToDevice, ctx->stream));
  StatParams SP;
  SP.data = dev;
  SP.stride_t = a->strides[0]; SP.stride_r = a->strides[1]; SP.stride_c = a->strides[2];
  SP.units = ctx->units.as<EncUnit>();
  SP.n_units = n_units;
  SP.t_max = (u32)a->shape[0];
  SP.ustats = ctx->ustats.as<UnitStats>();
  SP.istats = ctx->istats.as<InstStats>();
  switch (a->encoding) {
    case DCDF_ENC_F32: launch_stats<float, true>(ctx, SP); break;
    case DCDF_ENC_F64: launch_stats<double, true>(ctx, SP); break;
    case DCDF_ENC_I32: launch_stats<int32_t, false>(ctx, SP); break;
    default: launch_stats<i64, false>(ctx, SP); break;
  }
}

int32_t dcdf_suggest_fraction(dcdf_ctx* ctx, const dcdf_array3* a, int32_t* kind, int32_t* bits) {
  return guarded(ctx, [&] {
    validate_array(a);
    if (!kind || !bits) api_fail(DCDF_ERR_BAD_ARG, "null out");
    if (a->encoding != DCDF_ENC_F32 && a->encoding != DCDF_ENC_F64) api_fail(DCDF_ERR_BAD_ARG, "suggest_fraction needs a float array");
    if (a->shape[0] > 0x7fffffff) api_fail(DCDF_ERR_BAD_ARG, "too many instants");
    cudaStream_t st = ctx->stream;
    const void* dev = stage_input(ctx, a);
    std::vector<EncUnit> units;
    tile_units(a, units);
    run_unit_stats(ctx, a, dev, units);
    const u32 n_units = (u32)units.size();
    ctx->slices.reserve(sizeof(SliceDesc));
    ctx->sstate.reserve(sizeof(SliceState));
    ctx->small.reserve(256);
    SliceDesc sd;
    memset(&sd, 0, sizeof sd);
    sd.instants = (int)a->shape[0]; sd.n_units = n_units;
    CK(cudaMemcpyAsync(ctx->slices.p, &sd, sizeof sd, cudaMemcpyHostToDevice, st));
    FinalizeParams FP;
    memset(&FP, 0, sizeof FP);
    FP.slices = ctx->slices.as<SliceDesc>();
    FP.state = ctx->sstate.as<SliceState>();
    FP.ustats = ctx->ustats.as<UnitStats>();
    FP.encoding = a->encoding;
    FP.compute_bits = 1;
    k_finalize_phase1<<<1, 256, 0, st>>>(FP, 1);
    CK(cudaGetLastError());
    ctx->launches++;
    SliceState hs;
    CK(cudaMemcpyAsync(&hs, ctx->sstate.p, sizeof hs, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (hs.err & EF_OVERFLOW) api_fail(DCDF_ERR_OVERFLOW, "value too large for fixed point (fixed.rs:130)");
    if (!hs.need_exact) { *kind = hs.sug_round; *bits = hs.sug_bits; return; }
    ctx->exact.reserve(64);
    i64 t0 = 0;
    int vals[5] = {(int)a->shape[0], 1, hs.maxfb, 0, 0};  // instants, need, maxfb, f, round
    i64* d_t0 = ctx->exact.as<i64>();
    int* d_vals = reinterpret_cast<int*>(d_t0 + 1);
    CK(cudaMemcpyAsync(d_t0, &t0, sizeof t0, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_vals, vals, sizeof vals, cudaMemcpyHostToDevice, st));
    ExactParams XP;
    XP.data = dev;
    XP.stride_t = a->strides[0]; XP.stride_r = a->strides[1]; XP.stride_c = a->strides[2];
    XP.rows = a->shape[1]; XP.cols = a->shape[2];
    XP.slice_t0 = d_t0; XP.slice_instants = d_vals; XP.slice_need = d_vals + 1; XP.slice_maxfb = d_vals + 2;
    XP.slice_f = d_vals + 3; XP.slice_round = d_vals + 4;
    dim3 grid((unsigned)(4 * ctx->sm_count), 1);
    if (a->encoding == DCDF_ENC_F32) k_fraction_exact<float><<<grid, 256, 0, st>>>(XP, 1);
    else k_fraction_exact<double><<<grid, 256, 0, st>>>(XP, 1);
    CK(cudaGetLastError());
    ctx->launches++;
    CK(cudaMemcpyAsync(vals, d_vals, sizeof vals, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *kind = vals[4] ? 1 : 0;
    *bits = vals[4] ? hs.maxfb : vals[3];
  });
}

int32_t dcdf_min_max(dcdf_ctx* ctx, const dcdf_array3* a, int32_t fractional_bits, int32_t round, int64_t* min_out,
                     int64_t* max_out) {
  return guarded(ctx, [&] {
    validate_array(a);
    if (!min_out || !max_out) api_fail(DCDF_ERR_BAD_ARG, "null out");
    if (a->shape[0] > 0x7fffffff) api_fail(DCDF_ERR_BAD_ARG, "too many instants");
    cudaStream_t st = ctx->stream;
    const void* dev = stage_input(ctx, a);
    std::vector<EncUnit> units;
    tile_units(a, units);
    run_unit_stats(ctx, a, dev, units);
    const int T = (int)a->shape[0];
    ctx->query_out.reserve(sizeof(i64) * 2 * (size_t)T);
    ctx->small.reserve(256);
    CK(cudaMemsetAsync(ctx->small.p, 0, 64, st));
    RegionMinMaxParams RP;
    RP.units = ctx->units.as<EncUnit>();
    RP.n_units = (u32)units.size();
    RP.istats = ctx->istats.as<InstStats>();
    RP.t_max = (u32)T;
    RP.region_cols = a->shape[2];
    RP.encoding = a->encoding; RP.bits = fractional_bits; RP.round = round;
    RP.instants = T;
    RP.out_min = ctx->query_out.as<i64>();
    RP.out_max = RP.out_min + T;
    RP.err = ctx->small.as<u32>();
    k_region_minmax<<<(T + 127) / 128, 128, 0, st>>>(RP);
    CK(cudaGetLastError());
    ctx->launches++;
    u32 flags = 0;
    CK(cudaMemcpyAsync(min_out, RP.out_min, sizeof(i64) * T, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(max_out, RP.out_max, sizeof(i64) * T, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&flags, RP.err, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    std::string msg;
    const int32_t code = status_from_flags(flags, msg);
    if (code != DCDF_OK) throw ApiFail{code, msg};
  });
}

// ===================================================================================== Chunk::build
int32_t dcdf_chunk_build(dcdf_ctx* ctx, const dcdf_array3* a, int32_t k, int32_t fractional_bits, int32_t round,
                         dcdf_chunk** out, dcdf_build_stats* stats) {
  return guarded(ctx, [&] {
    if (!out) api_fail(DCDF_ERR_BAD_ARG, "null out");
    *out = nullptr;
    validate_array(a);
    if (k != 2) api_fail(DCDF_ERR_BAD_ARG, "only k = 2 is supported (dataset.rs:848 hard-codes it)");
    if (fractional_bits < 0 || fractional_bits > 62) api_fail(DCDF_ERR_BAD_ARG, "fractional_bits out of range");
    const int64_t rows = a->shape[1], cols = a->shape[2];
    const int64_t longest = std::max(rows, cols);
    if (longest < 2) api_fail(DCDF_ERR_BAD_ARG, "1x1 rasters have an empty nodemap (snapshot.rs:166)");
    const uint32_t L = levels_for(longest, 2);
    if (L > 6) {
      // multi-level path: dense pyramid in global memory + device-wide scans (encode_big.cuh)
      const void* dev = stage_input(ctx, a);
      const bool is_float = a->encoding == DCDF_ENC_F32 || a->encoding == DCDF_ENC_F64;
      const int bits = is_float ? fractional_bits : 0;
      BigResult R;
      switch (a->encoding) {
        case DCDF_ENC_F32: big_chunk_encode<float>(ctx, dev, a->strides, a->encoding, a->shape[0], rows, cols, bits, round ? 1 : 0, R); break;
        case DCDF_ENC_F64: big_chunk_encode<double>(ctx, dev, a->strides, a->encoding, a->shape[0], rows, cols, bits, round ? 1 : 0, R); break;
        case DCDF_ENC_I32: big_chunk_encode<int32_t>(ctx, dev, a->strides, a->encoding, a->shape[0], rows, cols, bits, 0, R); break;
        default: big_chunk_encode<i64>(ctx, dev, a->strides, a->encoding, a->shape[0], rows, cols, bits, 0, R); break;
      }
      dcdf_chunk* c = new dcdf_chunk();
      c->device = ctx->device;
      c->bytes = R.blob; c->size = R.size; c->owner = true;
      for (int i = 0; i < 3; i++) c->shape[i] = a->shape[i];
      c->encoding = a->encoding;
      c->fractional_bits = bits;
      c->n_blocks = R.snapshots;
      c->block_instants = R.block_instants;
      if (stats) {
        stats->size = R.size; stats->elided = stats->local = stats->external = 0;
        stats->snapshots = R.snapshots; stats->logs = R.logs;
      }
      *out = c;
      return;
    }
    EncodeJob job;
    job.dev_data = stage_input(ctx, a);
    job.encoding = a->encoding;
    for (int i = 0; i < 3; i++) job.strides[i] = a->strides[i];
    job.rows = rows; job.cols = cols;
    job.plain = 1;
    job.req_bits = fractional_bits;
    job.round = round ? 1 : 0;
    job.t_max = (uint32_t)a->shape[0];
    job.input_bytes = (size_t)a->shape[0] * rows * cols * elem_size(a->encoding);
    EncUnit u;
    memset(&u, 0, sizeof u);
    u.base = 0; u.rows = (int)rows; u.cols = (int)cols; u.instants = (int)a->shape[0];
    u.lo = 6 - (int)L;
    job.units.push_back(u);
    SliceDesc sd;
    memset(&sd, 0, sizeof sd);
    sd.t0 = 0; sd.instants = (int)a->shape[0]; sd.unit_base = 0; sd.n_units = 1;
    job.slices.push_back(sd);
    job.table_len.push_back(0);
    EncodeOut eo;
    run_encode(ctx, job, eo, true);
    dcdf_chunk* c = new dcdf_chunk();
    c->device = ctx->device;
    c->bytes = eo.blob;
    c->size = eo.blob_size;
    c->owner = true;
    for (int i = 0; i < 3; i++) c->shape[i] = a->shape[i];
    c->encoding = a->encoding;
    c->fractional_bits = eo.units[0].bits;
    c->n_blocks = eo.results[0].snapshots;
    uint32_t run = 0;
    for (size_t i = 0; i < eo.pieces.size(); i++) {
      if (eo.pieces[i].kind == 1u && i > 0) { c->block_instants.push_back(run); run = 0; }
      run++;
    }
    c->block_instants.push_back(run);
    if (stats) {
      stats->size = eo.results[0].bytes;
      stats->elided = stats->local = stats->external = 0;
      stats->snapshots = eo.results[0].snapshots;
      stats->logs = eo.results[0].logs;
    }
    *out = c;
  });
}

int32_t dcdf_chunk_free(dcdf_chunk* c) {
  if (!c) return DCDF_OK;
  cudaSetDevice(c->device);
  if (c->dir) free_chunk_meta(c->dir);
  if (c->owner && c->bytes) pool_free(c->bytes);
  delete c;
  return DCDF_OK;
}

int32_t dcdf_chunk_size(const dcdf_chunk* c, uint64_t* len) {
  if (!c || !len) return DCDF_ERR_BAD_ARG;
  *len = c->size;
  return DCDF_OK;
}

int32_t dcdf_chunk_bytes(dcdf_ctx* ctx, const dcdf_chunk* c, uint8_t* dst, uint64_t cap, int32_t mem) {
  return guarded(ctx, [&] {
    if (!c) api_fail(DCDF_ERR_BAD_ARG, "null chunk");
    copy_out(ctx, c->bytes, c->size, dst, cap, mem);
  });
}

int32_t dcdf_chunk_info(const dcdf_chunk* c, int64_t shape[3], int32_t* encoding, int32_t* fractional_bits, uint32_t* n_blocks) {
  if (!c) return DCDF_ERR_BAD_ARG;
  if (shape) for (int i = 0; i < 3; i++) shape[i] = c->shape[i];
  if (encoding) *encoding = c->encoding;
  if (fractional_bits) *fractional_bits = c->fractional_bits;
  if (n_blocks) *n_blocks = c->n_blocks;
  return DCDF_OK;
}

int32_t dcdf_chunk_block_instants(dcdf_ctx* ctx, const dcdf_chunk* c, uint32_t* out) {
  return guarded(ctx, [&] {
    if (!c || !out) api_fail(DCDF_ERR_BAD_ARG, "null argument");
    if (c->block_instants.size() != c->n_blocks) api_fail(DCDF_ERR_BAD_FORMAT, "block table missing");
    for (size_t i = 0; i < c->block_instants.size(); i++) out[i] = c->block_instants[i];
  });
}

// ===================================================================================== Superchunk::build
int32_t dcdf_superchunk_build(dcdf_ctx* ctx, const dcdf_array3* a, const uint32_t* levels, uint32_t n_levels, int32_t k,
                              int32_t fractional_bits, int32_t round, int32_t compute_bits, int64_t chunk_size,
                              dcdf_superchunk** out) {
  return guarded(ctx, [&] {
    if (!out) api_fail(DCDF_ERR_BAD_ARG, "null out");
    *out = nullptr;
    validate_array(a);
    if (k != 2) api_fail(DCDF_ERR_BAD_ARG, "only k = 2 is supported (dataset.rs:848 hard-codes it)");
    if (!levels || n_levels < 2) api_fail(DCDF_ERR_BAD_LEVELS, "need at least two k2_levels entries");
    if (fractional_bits < 0 || fractional_bits > 62) api_fail(DCDF_ERR_BAD_ARG, "fractional_bits out of range");
    const int64_t T = a->shape[0], rows = a->shape[1], cols = a->shape[2];
    const uint32_t total_levels = levels_for(std::max(rows, cols), 2);
    uint32_t user_levels = 0;
    for (uint32_t i = 0; i < n_levels; i++) user_levels += levels[i];
    if (user_levels != total_levels)
      api_fail(DCDF_ERR_BAD_LEVELS, "Need %u tree levels to encode array, but %u levels passed in (superchunk.rs:105-110)", total_levels, user_levels);
    if (levels[n_levels - 1] > 6) api_fail(DCDF_ERR_BAD_ARG, "leaf subchunks larger than 64x64 are not built on the GPU yet");
    if (total_levels > 16) api_fail(DCDF_ERR_BAD_ARG, "raster side too large");
    const int64_t sidelen = (int64_t)1 << total_levels;
    const int64_t cs = chunk_size > 0 ? chunk_size : T;
    const uint32_t n_slices = (uint32_t)((T + cs - 1) / cs);

    TreeGeo G;
    build_tree(G, rows, cols, levels, n_levels);
    const uint32_t n_nodes = (uint32_t)G.nodes.size();
    const int ls = G.leaf_side;
    const uint32_t n_slots = (uint32_t)(G.leaf_grid * G.leaf_grid);
    const uint32_t units_per_slice = (uint32_t)(G.leaf_rows * G.leaf_cols);

    EncodeJob job;
    job.dev_data = stage_input(ctx, a);
    job.encoding = a->encoding;
    for (int i = 0; i < 3; i++) job.strides[i] = a->strides[i];
    job.rows = rows; job.cols = cols;
    job.plain = 0;
    job.req_bits = fractional_bits;
    job.round = round ? 1 : 0;
    job.compute_bits = compute_bits ? 1 : 0;
    job.n_slots = n_slots;
    job.t_max = (uint32_t)std::min<int64_t>(cs, T);
    job.input_bytes = (size_t)T * rows * cols * elem_size(a->encoding);
    job.tree = &G;
    std::vector<int32_t> slot_unit((size_t)n_slices * n_slots, -1);
    for (uint32_t s = 0; s < n_slices; s++) {
      const int64_t t0 = (int64_t)s * cs, t1 = std::min<int64_t>(t0 + cs, T);
      SliceDesc sd;
      memset(&sd, 0, sizeof sd);
      sd.t0 = t0; sd.instants = (int)(t1 - t0); sd.unit_base = (uint32_t)job.units.size();
      for (int gr = 0; gr < G.leaf_rows; gr++)
        for (int gc = 0; gc < G.leaf_cols; gc++) {
          const int64_t top = (int64_t)gr * ls, left = (int64_t)gc * ls;
          EncUnit u;
          memset(&u, 0, sizeof u);
          u.base = t0 * a->strides[0] + top * a->strides[1] + left * a->strides[2];
          u.rows = (int)std::min<int64_t>(ls, rows - top); u.cols = (int)std::min<int64_t>(ls, cols - left);
          u.instants = sd.instants;
          // each sub-array is built by Chunk::build from its OWN (clipped) shape: snapshot.rs:118-119
          u.lo = 6 - (int)levels_for(std::max<int64_t>(u.rows, u.cols), 2);
          u.slot = (uint32_t)((int64_t)gr * G.leaf_grid + gc);
          u.row0 = (int)top; u.col0 = (int)left;
          slot_unit[(size_t)s * n_slots + u.slot] = (int32_t)job.units.size();
          job.units.push_back(u);
        }
      sd.n_units = (uint32_t)job.units.size() - sd.unit_base;
      job.slices.push_back(sd);
      job.table_len.push_back((uint64_t)sd.instants * G.tbl_per_instant);
    }
    (void)units_per_slice;
    EncodeOut eo;
    run_encode(ctx, job, eo, false);

    dcdf_superchunk* sc = new dcdf_superchunk();
    sc->device = ctx->device;
    sc->encoding = a->encoding;
    for (int i = 0; i < 3; i++) sc->shape[i] = a->shape[i];
    sc->chunk_size = cs;
    sc->n_slots = n_slots;
    sc->units = std::move(eo.units);
    sc->stored = std::move(eo.stored);
    sc->chunk_off = std::move(eo.chunk_off);
    sc->results = std::move(eo.results);
    sc->slot_unit = std::move(slot_unit);
    sc->chunk_blob = eo.blob; sc->chunk_blob_size = eo.blob_size;
    sc->dac_blob = eo.dac_blob; sc->dac_blob_size = eo.dac_blob_size;
    sc->tbl_max = eo.tbl_max; sc->tbl_min = eo.tbl_min; sc->tbl_len = eo.tbl_total;
    sc->nodes = G.nodes; sc->children = G.children; sc->geom = G.geom; sc->leaf_unit = G.leaf_unit;
    sc->leaf_rows = G.leaf_rows; sc->leaf_cols = G.leaf_cols; sc->leaf_side = G.leaf_side; sc->leaf_grid = G.leaf_grid;
    sc->tbl_per_instant = G.tbl_per_instant;
    sc->nstate = std::move(eo.nstate);
    sc->node_dac_off.resize((size_t)n_slices * n_nodes * 2);
    sc->node_dac_size.resize((size_t)n_slices * n_nodes * 2);
    for (size_t i = 0; i < sc->node_dac_off.size(); i++) { sc->node_dac_off[i] = eo.dac_off[i]; sc->node_dac_size[i] = eo.dac_pieces[i].size; }
    for (uint32_t s = 0; s < n_slices; s++) {
      dcdf_superchunk::Slice sl;
      memset(&sl.info, 0, sizeof sl.info);
      const SliceDesc& sd = job.slices[s];
      sl.t0 = sd.t0; sl.unit_base = sd.unit_base; sl.n_units = sd.n_units;
      sl.table_base = sd.table_base;
      sl.chunk_blob_off = sc->chunk_off[sd.unit_base];
      sl.info.shape[0] = sd.instants;
      sl.info.chunk_bytes = sc->chunk_off[sd.unit_base + sd.n_units] - sc->chunk_off[sd.unit_base];
      sc->slices.push_back(sl);
    }
    (void)sidelen;
    *out = sc;
  });
}

namespace {
// MMStruct3Build counters of one node (recursive, superchunk.rs:200-269)
void node_stats(const dcdf_superchunk* sc, uint32_t slice, uint32_t node, dcdf_build_stats& bs, uint64_t& chunk_bytes) {
  const uint32_t n_nodes = (uint32_t)sc->nodes.size();
  const TreeNode& nd = sc->nodes[node];
  const auto& sl = sc->slices[slice];
  memset(&bs, 0, sizeof bs);
  chunk_bytes = 0;
  for (u32 c = 0; c < nd.n_children; c++) {
    const TreeChild& ch = sc->children[nd.first_child + c];
    if (ch.kind == 1) {
      const uint32_t u = sl.unit_base + (uint32_t)ch.index;
      if (sc->stored[u]) {
        bs.external++; bs.snapshots += sc->results[u].snapshots; bs.logs += sc->results[u].logs;
        chunk_bytes += sc->results[u].bytes;
        continue;
      }
    } else if (ch.kind == 2 && sc->nstate[(size_t)slice * n_nodes + ch.index].alive) {
      dcdf_build_stats cb;
      uint64_t cbytes;
      node_stats(sc, slice, (uint32_t)ch.index, cb, cbytes);
      bs.external++; bs.snapshots += cb.snapshots; bs.logs += cb.logs;
      bs.size += cb.size;
      continue;
    }
    bs.elided++;
  }
  const size_t di = ((size_t)slice * n_nodes + node) * 2;
  bs.size += chunk_bytes + sc->node_dac_size[di] + sc->node_dac_size[di + 1];
}

void fill_node_info(const dcdf_superchunk* sc, uint32_t slice, uint32_t node, dcdf_superchunk_info* info) {
  const uint32_t n_nodes = (uint32_t)sc->nodes.size();
  memset(info, 0, sizeof *info);
  const auto& g = sc->geom[node];
  const NodeState& st = sc->nstate[(size_t)slice * n_nodes + node];
  const bool is_float = sc->encoding == DCDF_ENC_F32 || sc->encoding == DCDF_ENC_F64;
  info->shape[0] = sc->slices[slice].info.shape[0]; info->shape[1] = g.rows; info->shape[2] = g.cols;
  info->sidelen = g.sidelen; info->chunks_sidelen = g.chunks_sidelen; info->subsidelen = g.subsidelen;
  info->levels = g.levels;
  info->encoding = sc->encoding;
  info->fractional_bits = is_float ? st.bits : 0;
  info->n_refs = st.alive ? sc->nodes[node].n_children : 0;
  const size_t di = ((size_t)slice * n_nodes + node) * 2;
  info->max_dac_bytes = sc->node_dac_size[di]; info->min_dac_bytes = sc->node_dac_size[di + 1];
  if (st.alive) node_stats(sc, slice, node, info->stats, info->chunk_bytes);
  if (node == 0) info->chunk_bytes = sc->slices[slice].info.chunk_bytes;  // the slice's whole chunk blob
}
}  // namespace

int32_t dcdf_superchunk_free(dcdf_superchunk* sc) {
  if (!sc) return DCDF_OK;
  cudaSetDevice(sc->device);
  pool_free(sc->chunk_blob);
  pool_free(sc->dac_blob);
  pool_free(sc->tbl_max);
  pool_free(sc->tbl_min);
  if (sc->dev_meta) free_super_meta(sc->dev_meta);
  pool_free(sc->dir);
  delete sc;
  return DCDF_OK;
}

int32_t dcdf_superchunk_count(const dcdf_superchunk* sc, uint32_t* n) {
  if (!sc || !n) return DCDF_ERR_BAD_ARG;
  *n = (uint32_t)sc->slices.size();
  return DCDF_OK;
}

int32_t dcdf_superchunk_node_count(const dcdf_superchunk* sc, uint32_t* n) {
  if (!sc || !n) return DCDF_ERR_BAD_ARG;
  *n = (uint32_t)sc->nodes.size();
  return DCDF_OK;
}

int32_t dcdf_superchunk_get_info(const dcdf_superchunk* sc, uint32_t slice, dcdf_superchunk_info* info) {
  if (!sc || !info || slice >= sc->slices.size()) return DCDF_ERR_BAD_ARG;
  fill_node_info(sc, slice, 0, info);
  return DCDF_OK;
}

int32_t dcdf_superchunk_node_info(const dcdf_superchunk* sc, uint32_t slice, uint32_t node, dcdf_superchunk_info* info) {
  if (!sc || !info || slice >= sc->slices.size() || node >= sc->nodes.size()) return DCDF_ERR_BAD_ARG;
  fill_node_info(sc, slice, node, info);
  return DCDF_OK;
}

int32_t dcdf_superchunk_node_refs(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, uint32_t node, int32_t* kinds,
                                  int32_t* child_node, uint64_t* chunk_off, uint64_t* chunk_size, int32_t* chunk_bits) {
  return guarded(ctx, [&] {
    if (!sc || slice >= sc->slices.size() || node >= sc->nodes.size()) api_fail(DCDF_ERR_BAD_ARG, "bad slice / node");
    const uint32_t n_nodes = (uint32_t)sc->nodes.size();
    const auto& sl = sc->slices[slice];
    const TreeNode& nd = sc->nodes[node];
    if (!sc->nstate[(size_t)slice * n_nodes + node].alive) api_fail(DCDF_ERR_BAD_ARG, "node %u is not built in slice %u (elided)", node, slice);
    for (u32 c = 0; c < nd.n_children; c++) {
      const TreeChild& ch = sc->children[nd.first_child + c];
      int32_t kind = DCDF_REF_ELIDED, cn = -1, bits = 0;
      uint64_t off = 0, size = 0;
      if (ch.kind == 1) {
        const uint32_t u = sl.unit_base + (uint32_t)ch.index;
        if (sc->stored[u]) { kind = DCDF_REF_EXTERNAL; off = sc->chunk_off[u] - sl.chunk_blob_off; size = sc->results[u].bytes; bits = sc->units[u].bits; }
      } else if (ch.kind == 2 && sc->nstate[(size_t)slice * n_nodes + ch.index].alive) {
        kind = DCDF_REF_EXTERNAL; cn = ch.index;
      }
      if (kinds) kinds[c] = kind;
      if (child_node) child_node[c] = cn;
      if (chunk_off) chunk_off[c] = off;
      if (chunk_size) chunk_size[c] = size;
      if (chunk_bits) chunk_bits[c] = bits;
    }
  });
}

int32_t dcdf_superchunk_refs(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, int32_t* kinds, uint64_t* chunk_off,
                             uint64_t* chunk_size, int32_t* chunk_bits) {
  return dcdf_superchunk_node_refs(ctx, sc, slice, 0, kinds, nullptr, chunk_off, chunk_size, chunk_bits);
}

int32_t dcdf_superchunk_node_bytes(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, uint32_t node, int32_t which,
                                   uint8_t* dst, uint64_t cap, int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc || slice >= sc->slices.size() || node >= sc->nodes.size() || which < 1 || which > 2) api_fail(DCDF_ERR_BAD_ARG, "bad slice / node / which");
    const size_t di = ((size_t)slice * sc->nodes.size() + node) * 2 + (size_t)(which - 1);
    copy_out(ctx, sc->dac_blob + sc->node_dac_off[di], sc->node_dac_size[di], dst, cap, mem);
  });
}

int32_t dcdf_superchunk_bytes(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint32_t slice, int32_t which, uint8_t* dst,
                              uint64_t cap, int32_t mem) {
  if (which == 0)
    return guarded(ctx, [&] {
      if (!sc || slice >= sc->slices.size()) api_fail(DCDF_ERR_BAD_ARG, "bad slice");
      const auto& sl = sc->slices[slice];
      copy_out(ctx, sc->chunk_blob + sl.chunk_blob_off, sl.info.chunk_bytes, dst, cap, mem);
    });
  return dcdf_superchunk_node_bytes(ctx, sc, slice, 0, which, dst, cap, mem);
}

int32_t dcdf_superchunk_total_bytes(const dcdf_superchunk* sc, uint64_t* n) {
  if (!sc || !n) return DCDF_ERR_BAD_ARG;
  *n = sc->chunk_blob_size + sc->dac_blob_size;
  return DCDF_OK;
}

}  // extern "C"
