// api_decode.cu -- C-ABI entry points for the query half of the path (Chunk::read_from, get / fill_cell /
// fill_window / iter_search at chunk and superchunk level, flat to_fixed / from_fixed).
#include <algorithm>
#include <cstdlib>
#include <mutex>

#include "decode.cuh"
#include "decode_tile4.cuh"
#include "decode_search4.cuh"
#include "host.hpp"

using namespace dcdf;

namespace {

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

size_t enc_size(int enc) { return (enc == DCDF_ENC_I32 || enc == DCDF_ENC_F32) ? 4 : 8; }

// Device-side metadata of a queryable object.
struct DevMeta {
  UnitMeta* units = nullptr;
  SliceMeta* slices = nullptr;
  int32_t* slot_unit = nullptr;
  SlotDesc* slot_desc = nullptr;
  u32* err = nullptr;
};

// Everything the query kernels need for one handle; owned by the handle (dev_meta / dir pointers).
struct MetaBlock {
  DevMeta d;
  QuerySet Q;
  u64 n_dir = 0;
  int max_sidelen = 0;  // tiles up to 64x64 take the level-synchronous window decoder
  int max_dac_levels = 0;  // <= 3: the window decoder can expand in 32-bit values
};

void check_err_word(dcdf_ctx* ctx, u32* d_err, const char* what) {
  u32 f = 0;
  CK(cudaMemcpyAsync(&f, d_err, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (f & EF_BAD_FORMAT) api_fail(DCDF_ERR_BAD_FORMAT, "%s: malformed chunk bytes", what);
  if (f & EF_OUT_OF_BOUNDS) {
    CK(cudaMemsetAsync(d_err, 0, 4, ctx->stream));
    api_fail(DCDF_ERR_OUT_OF_BOUNDS, "%s: query out of bounds", what);
  }
  if (f & EF_NONFINITE) api_fail(DCDF_ERR_NONFINITE, "%s: non-finite input", what);
  if (f & EF_OVERFLOW) api_fail(DCDF_ERR_OVERFLOW, "%s: overflow", what);
  if (f & EF_PRECISION) api_fail(DCDF_ERR_PRECISION_LOSS, "%s: loss of precision", what);
  if (f) api_fail(DCDF_ERR_CUDA, "%s: device error flags %u", what, f);
}

MetaBlock* make_meta(dcdf_ctx* ctx, const u8* blob, std::vector<UnitMeta>& units, const std::vector<SliceMeta>& slices,
                     const std::vector<int32_t>& slot_unit, const std::vector<SlotDesc>& slot_desc, u32 n_slots, i64 chunk_size, int chunks_sidelen, int subsidelen,
                     int encoding, const i64* shape, const i64* tbl_max, const i64* tbl_min, void** dir_out, bool count_first, bool validate) {
  cudaStream_t st = ctx->stream;
  MetaBlock* mb = new MetaBlock();
  *dir_out = nullptr;
  try {
    const size_t ub = sizeof(UnitMeta) * units.size(), sb = sizeof(SliceMeta) * slices.size(),
                 mbytes = (sizeof(int32_t) * slot_unit.size() + 15) & ~size_t(15), db = sizeof(SlotDesc) * slot_desc.size();
    u8* raw = nullptr;
    raw = static_cast<u8*>(pool_alloc(ub + sb + mbytes + db + 64, st));
    mb->d.units = reinterpret_cast<UnitMeta*>(raw);
    mb->d.slices = reinterpret_cast<SliceMeta*>(raw + ub);
    mb->d.slot_unit = reinterpret_cast<int32_t*>(raw + ub + sb);
    mb->d.slot_desc = reinterpret_cast<SlotDesc*>(raw + ub + sb + mbytes);
    mb->d.err = reinterpret_cast<u32*>(raw + ub + sb + mbytes + ((db + 15) & ~size_t(15)));
    CK(cudaMemcpyAsync(mb->d.slot_desc, slot_desc.data(), db, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(mb->d.err, 0, 16, st));
    CK(cudaMemcpyAsync(mb->d.units, units.data(), ub, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(mb->d.slices, slices.data(), sb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(mb->d.slot_unit, slot_unit.data(), sizeof(int32_t) * slot_unit.size(), cudaMemcpyHostToDevice, st));
    DirParams DP;
    DP.blob = blob;
    DP.units = mb->d.units;
    DP.dir = nullptr;
    DP.n_units = (u32)units.size();
    DP.validate = validate ? 1 : 0;
    DP.err = mb->d.err;
    const u32 grid = ((u32)units.size() + 63) / 64;
    if (count_first) {
      DP.count_only = 1;
      k_build_dir<<<grid, 64, 0, st>>>(DP);
      CK(cudaGetLastError());
      ctx->launches++;
      check_err_word(ctx, mb->d.err, "chunk open");
      CK(cudaMemcpyAsync(units.data(), mb->d.units, ub, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      u64 n = 0;
      for (auto& u : units) { u.dir_base = (u32)n; n += (u64)u.instants; }
      CK(cudaMemcpyAsync(mb->d.units, units.data(), ub, cudaMemcpyHostToDevice, st));
    }
    u64 n_dir = 0;
    for (auto& u : units) if (u.stored) n_dir = std::max<u64>(n_dir, (u64)u.dir_base + (u64)u.instants);
    InstDir* dir = nullptr;
    dir = static_cast<InstDir*>(pool_alloc(sizeof(InstDir) * std::max<u64>(n_dir, 1), st));
    *dir_out = dir;
    DP.dir = dir;
    DP.count_only = 0;
    k_build_dir<<<grid, 64, 0, st>>>(DP);
    CK(cudaGetLastError());
    ctx->launches++;
    check_err_word(ctx, mb->d.err, "chunk directory");
    CK(cudaMemcpyAsync(units.data(), mb->d.units, ub, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    mb->n_dir = n_dir;
    for (auto& u : units) if (u.stored) { mb->max_sidelen = std::max(mb->max_sidelen, u.sidelen); mb->max_dac_levels = std::max(mb->max_dac_levels, u.dac_levels); }
    QuerySet& Q = mb->Q;
    Q.blob = blob;
    Q.units = mb->d.units;
    Q.dir = dir;
    Q.slices = mb->d.slices;
    Q.slot_unit = mb->d.slot_unit;
    Q.slot_desc = mb->d.slot_desc;
    Q.tbl_max = tbl_max;
    Q.tbl_min = tbl_min;
    Q.n_slices = (u32)slices.size();
    Q.n_slots = n_slots;
    Q.chunk_size = chunk_size;
    Q.chunks_sidelen = chunks_sidelen;
    Q.subsidelen = subsidelen;
    Q.encoding = encoding;
    for (int i = 0; i < 3; i++) Q.shape[i] = shape[i];
    return mb;
  } catch (...) {
    cudaStreamSynchronize(st);
    pool_free(*dir_out);
    *dir_out = nullptr;
    pool_free(mb->d.units);
    delete mb;
    throw;
  }
}

// Built objects are immutable and may be queried from several contexts / host threads (dcdf_cuda.h): the lazily built
// device directory of a handle is created under this lock.
std::mutex g_meta_mutex;

// ---- handle -> MetaBlock (lazily for built objects)
MetaBlock* chunk_meta(dcdf_ctx* ctx, const dcdf_chunk* cc) {
  dcdf_chunk* c = const_cast<dcdf_chunk*>(cc);
  std::lock_guard<std::mutex> lock(g_meta_mutex);
  if (c->dir) return static_cast<MetaBlock*>(c->dir);
  std::vector<UnitMeta> units(1);
  memset(&units[0], 0, sizeof(UnitMeta));
  units[0].blob_off = 0; units[0].size = c->size; units[0].dir_base = 0; units[0].instants = (int)c->shape[0];
  units[0].stored = 1;
  std::vector<SliceMeta> slices(1);
  memset(&slices[0], 0, sizeof(SliceMeta));
  slices[0].t0 = 0; slices[0].instants = (int)c->shape[0]; slices[0].bits = c->fractional_bits;
  std::vector<int32_t> slot_unit(1, 0);
  std::vector<SlotDesc> slot_desc(1);
  memset(&slot_desc[0], 0, sizeof(SlotDesc));
  void* dir = nullptr;
  const bool count_first = c->shape[0] == 0;
  MetaBlock* mb = make_meta(ctx, c->bytes, units, slices, slot_unit, slot_desc, 1, 0, 1 << 30, 1, c->encoding, c->shape, nullptr, nullptr, &dir, count_first,
                            /*validate=*/count_first);  // opened from outside bytes
  if (count_first) {
    c->shape[0] = units[0].instants; c->shape[1] = units[0].rows; c->shape[2] = units[0].cols;
    c->fractional_bits = units[0].bits;
    c->encoding = units[0].enc;
    mb->Q.encoding = c->encoding;
    for (int i = 0; i < 3; i++) mb->Q.shape[i] = c->shape[i];
    slices[0].instants = (int)c->shape[0];  // now known: refresh the device copy
    slices[0].bits = c->fractional_bits;
    CK(cudaMemcpyAsync(mb->d.slices, slices.data(), sizeof(SliceMeta), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  mb->Q.chunk_size = std::max<i64>(c->shape[0], 1);
  c->dir = mb;
  return mb;
}

MetaBlock* super_meta(dcdf_ctx* ctx, const dcdf_superchunk* scc) {
  dcdf_superchunk* sc = const_cast<dcdf_superchunk*>(scc);
  std::lock_guard<std::mutex> lock(g_meta_mutex);
  if (sc->dev_meta) return static_cast<MetaBlock*>(sc->dev_meta);
  std::vector<UnitMeta> units(sc->units.size());
  for (size_t u = 0; u < units.size(); u++) {
    UnitMeta& m = units[u];
    memset(&m, 0, sizeof m);
    m.stored = sc->stored[u];
    m.blob_off = sc->chunk_off[u];
    m.size = m.stored ? sc->results[u].bytes : 0;
    m.dir_base = sc->units[u].piece_base;
    m.instants = sc->units[u].instants;
  }
  const uint32_t n_nodes = (uint32_t)sc->nodes.size();
  std::vector<SliceMeta> slices(sc->slices.size());
  std::vector<SlotDesc> slot_desc(sc->slot_unit.size());
  if (!slot_desc.empty()) memset(slot_desc.data(), 0, sizeof(SlotDesc) * slot_desc.size());
  for (size_t s = 0; s < slices.size(); s++) {
    SliceMeta& m = slices[s];
    memset(&m, 0, sizeof m);
    m.t0 = sc->slices[s].t0;
    m.instants = (int)sc->slices[s].info.shape[0];
    m.bits = sc->nstate[s * n_nodes].bits;
    m.table_base = sc->slices[s].table_base;
    m.slot_base = (u32)(s * sc->n_slots);
    // flatten the node tree: every in-bounds leaf slot either has a stored chunk or inherits the table entry of
    // the shallowest node that elided one of its ancestors (superchunk.rs:325-330 applied along the recursion)
    for (int gr = 0; gr < sc->leaf_rows; gr++)
      for (int gc = 0; gc < sc->leaf_cols; gc++) {
        const size_t slot = s * sc->n_slots + (size_t)gr * sc->leaf_grid + gc;
        const int64_t row = (int64_t)gr * sc->leaf_side, col = (int64_t)gc * sc->leaf_side;
        uint32_t node = 0;
        SlotDesc d;
        memset(&d, 0, sizeof d);
        for (;;) {
          const TreeNode& nd = sc->nodes[node];
          const auto& g = sc->geom[node];
          const int64_t cr = (row - g.top) / g.chunks_sidelen, cc = (col - g.left) / g.chunks_sidelen;
          const u32 c = (u32)(cr * g.subsidelen + cc);
          const TreeChild& ch = sc->children[nd.first_child + c];
          const u64 tbl0 = sc->slices[s].table_base + (u64)nd.tbl_off * (u64)m.instants + c;
          if (ch.kind == 2 && sc->nstate[s * n_nodes + ch.index].alive) {
            if (d.n_up >= 3) api_fail(DCDF_ERR_BAD_ARG, "superchunks nested more than four levels deep are not supported by the query kernels");
            d.up_tbl0[d.n_up] = tbl0; d.up_stride[d.n_up] = nd.n_children; d.up_bits[d.n_up] = sc->nstate[s * n_nodes + node].bits; d.n_up++;
            node = (uint32_t)ch.index;
            continue;
          }
          d.tbl0 = tbl0;
          d.stride = nd.n_children;
          d.bits = sc->nstate[s * n_nodes + node].bits;
          slot_desc[slot] = d;
          break;
        }
      }
  }
  void* dir = nullptr;
  MetaBlock* mb = make_meta(ctx, sc->chunk_blob, units, slices, sc->slot_unit, slot_desc, sc->n_slots, sc->chunk_size, sc->leaf_side,
                            (int)sc->leaf_grid, sc->encoding, sc->shape, sc->tbl_max, sc->tbl_min, &dir, false, sc->opened);
  sc->dir = dir;
  sc->dev_meta = mb;
  return mb;
}

void free_meta(void* p, bool free_dir) {
  MetaBlock* mb = static_cast<MetaBlock*>(p);
  if (!mb) return;
  if (free_dir && mb->Q.dir) pool_free(const_cast<InstDir*>(mb->Q.dir));
  pool_free(mb->d.units);
  delete mb;
}

// ---- query plumbing
struct OutSpec {
  int raw;        // 1 = fixed i64
  size_t esize;
};
OutSpec out_spec(int out_encoding, int obj_encoding) {
  if (out_encoding == DCDF_ENC_I64 && obj_encoding != DCDF_ENC_I64) return {1, 8};
  if (out_encoding == obj_encoding) return {obj_encoding == DCDF_ENC_I64 ? 1 : 0, enc_size(obj_encoding)};
  api_fail(DCDF_ERR_BAD_ARG, "out_encoding must be DCDF_ENC_I64 (raw fixed point) or the object's own encoding");
}

const void* to_device(dcdf_ctx* ctx, DevBuf& buf, const void* src, size_t bytes, int mem) {
  if (mem == DCDF_MEM_DEVICE) return src;
  buf.reserve(bytes);
  CK(cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  return buf.p;
}

struct OutTarget {
  void* dev;
  void* user;
  size_t bytes;
  int mem;
};
OutTarget out_begin(dcdf_ctx* ctx, void* user, size_t bytes, int mem) {
  if (!user && bytes) api_fail(DCDF_ERR_BAD_ARG, "null output");
  if (mem == DCDF_MEM_DEVICE) return {user, user, bytes, mem};
  ctx->query_out.reserve(bytes);
  return {ctx->query_out.p, user, bytes, mem};
}
void out_end(dcdf_ctx* ctx, const OutTarget& t) {
  if (t.mem != DCDF_MEM_DEVICE && t.bytes) CK(cudaMemcpyAsync(t.user, t.dev, t.bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
}

void tbegin(dcdf_ctx* ctx, int which) { CK(cudaEventRecord(ctx->ev[2 * which], ctx->stream)); }
void tend(dcdf_ctx* ctx, int which) { CK(cudaEventRecord(ctx->ev[2 * which + 1], ctx->stream)); }
void tcollect(dcdf_ctx* ctx, int which) {
  float ms = 0;
  if (cudaEventElapsedTime(&ms, ctx->ev[2 * which], ctx->ev[2 * which + 1]) == cudaSuccess) ctx->kernel_ms[which] = ms;
  else cudaGetLastError();
}

dcdf_cube order_cube(const dcdf_cube& c) {  // Cube::new re-orders swapped bounds (geom.rs:83-107)
  dcdf_cube o = c;
  if (o.start > o.end) std::swap(o.start, o.end);
  if (o.top > o.bottom) std::swap(o.top, o.bottom);
  if (o.left > o.right) std::swap(o.left, o.right);
  return o;
}
void check_cube(const dcdf_cube& c, const i64* shape) {  // mmarray.rs:218-229
  if (c.start < 0 || c.top < 0 || c.left < 0 || c.end > shape[0] || c.bottom > shape[1] || c.right > shape[2])
    api_fail(DCDF_ERR_OUT_OF_BOUNDS, "window [%lld:%lld, %lld:%lld, %lld:%lld] out of bounds for shape [%lld, %lld, %lld]",
             (long long)c.start, (long long)c.end, (long long)c.top, (long long)c.bottom, (long long)c.left, (long long)c.right,
             (long long)shape[0], (long long)shape[1], (long long)shape[2]);
}

void do_get_batch(dcdf_ctx* ctx, MetaBlock* mb, uint64_t n, const int64_t* irc, void* out, int32_t out_encoding, int32_t mem) {
  if (n == 0) return;
  if (!irc) api_fail(DCDF_ERR_BAD_ARG, "null queries");
  const OutSpec os = out_spec(out_encoding, mb->Q.encoding);
  if (mem == DCDF_MEM_HOST) {
    for (uint64_t i = 0; i < n; i++)
      for (int d = 0; d < 3; d++)
        if (irc[3 * i + d] < 0 || irc[3 * i + d] >= mb->Q.shape[d]) api_fail(DCDF_ERR_OUT_OF_BOUNDS, "cell query %llu out of bounds", (unsigned long long)i);
  }
  const i64* d_q = static_cast<const i64*>(to_device(ctx, ctx->query_in, irc, sizeof(i64) * 3 * n, mem));
  OutTarget ot = out_begin(ctx, out, os.esize * n, mem);
  tbegin(ctx, KT_CELL);
  k_get_batch<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(mb->Q, d_q, n, ot.dev, os.raw, mb->d.err);
  CK(cudaGetLastError());
  ctx->launches++;
  tend(ctx, KT_CELL);
  out_end(ctx, ot);
  tcollect(ctx, KT_CELL);
  if (mem == DCDF_MEM_DEVICE) check_err_word(ctx, mb->d.err, "get_batch");  // host queries were checked above
}

uint32_t spread1by1_host(uint32_t v) {  // common.cuh: spread1by1
  v &= 0x0000ffffu;
  v = (v | (v << 8)) & 0x00ff00ffu;
  v = (v | (v << 4)) & 0x0f0f0f0fu;
  v = (v | (v << 2)) & 0x33333333u;
  v = (v | (v << 1)) & 0x55555555u;
  return v;
}

void do_cell_batch(dcdf_ctx* ctx, MetaBlock* mb, uint64_t n, const int64_t* q, const uint64_t* out_off, void* out,
                   int32_t out_encoding, int32_t mem) {
  if (n == 0) return;
  if (!q || !out_off) api_fail(DCDF_ERR_BAD_ARG, "null queries");
  const OutSpec os = out_spec(out_encoding, mb->Q.encoding);
  std::vector<i64> qq(q, q + 4 * n);
  for (uint64_t i = 0; i < n; i++) {
    if (qq[4 * i] > qq[4 * i + 1]) std::swap(qq[4 * i], qq[4 * i + 1]);
    const i64 s = qq[4 * i], e = qq[4 * i + 1], r = qq[4 * i + 2], c = qq[4 * i + 3];
    if (s < 0 || e > mb->Q.shape[0] || r < 0 || r >= mb->Q.shape[1] || c < 0 || c >= mb->Q.shape[2])
      api_fail(DCDF_ERR_OUT_OF_BOUNDS, "cell series %llu out of bounds", (unsigned long long)i);
    if ((uint64_t)(e - s) != out_off[i + 1] - out_off[i]) api_fail(DCDF_ERR_BAD_ARG, "out_off does not match the series lengths");
  }
  const size_t total = out_off[n];
  // Series of one subchunk are walked next to each other (the kernel takes queries in array order): at any instant they
  // descend the same structure, so its upper levels are read from DRAM once and then from L2.  Only the order of the work
  // changes: every series still lands at its own out_off.
  std::vector<uint32_t> order(n);
  for (uint64_t i = 0; i < n; i++) order[i] = (uint32_t)i;
  if (n > 1 && n <= 0xffffffffull) {
    const i64 cs0 = mb->Q.chunks_sidelen;
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) {
      const i64 ra = qq[4 * a + 2], ca = qq[4 * a + 3], rb = qq[4 * b + 2], cb = qq[4 * b + 3];
      const i64 ta = (ra / cs0) * (i64)mb->Q.subsidelen + ca / cs0, tb = (rb / cs0) * (i64)mb->Q.subsidelen + cb / cs0;
      if (ta != tb) return ta < tb;
      if (ra != rb) return ra < rb;
      if (ca != cb) return ca < cb;
      return a < b;
    });
  }
  // Tiles that at least `cell_tile_min` series of the batch fall into are decoded once per instant by the tile decoder
  // (k_cell_tiles4) and hand out the asked-for cells; the other series take the per-cell walk.  A second series on a cell
  // that is already listed (same cell, other instants) also takes the walk.
  const i64 cs = mb->Q.chunks_sidelen;
  const uint32_t tile_min = ctx->opt.cell_tile_min;
  const bool tiles_ok = tile_min > 0 && mb->max_sidelen <= 64 && n <= 0xffffffffull;
  std::vector<i64> qs;                 // walker: queries in walk order
  std::vector<u64> bases;
  std::vector<uint16_t> masks;         // tile path: 256 entries per dense tile (asked-for cells of every 4x4 block)
  std::vector<CellRef> refs;
  std::vector<SeriesJob> jobs;
  qs.reserve(4 * n); bases.reserve(n + 1);
  i64 longest = 1;
  auto tile_of = [&](uint32_t i) { return (qq[4 * i + 2] / cs) * (i64)mb->Q.subsidelen + qq[4 * i + 3] / cs; };
  auto walk = [&](uint32_t i) {
    for (int k = 0; k < 4; k++) qs.push_back(qq[4 * i + k]);
    bases.push_back(out_off[i]);
    longest = std::max(longest, qq[4 * i + 1] - qq[4 * i]);
  };
  for (uint64_t j0 = 0; j0 < n;) {
    uint64_t j1 = j0 + 1;
    const i64 tile = tile_of(order[j0]);
    while (j1 < n && tile_of(order[j1]) == tile) j1++;
    if (!tiles_ok || j1 - j0 < tile_min) {
      for (uint64_t j = j0; j < j1; j++) walk(order[j]);
      j0 = j1;
      continue;
    }
    const uint32_t tile_idx = (uint32_t)(masks.size() / DT_THREADS);
    const uint32_t ref_first = (uint32_t)refs.size();
    masks.resize(masks.size() + DT_THREADS, 0);
    uint16_t* mk = masks.data() + (size_t)tile_idx * DT_THREADS;
    i64 t_min = INT64_MAX, t_max = INT64_MIN;
    i64 prev_r = -1, prev_c = -1;
    for (uint64_t j = j0; j < j1; j++) {
      const uint32_t i = order[j];
      const i64 s_ = qq[4 * i], e_ = qq[4 * i + 1], r = qq[4 * i + 2] % cs, c = qq[4 * i + 3] % cs;
      if (e_ <= s_) continue;                                  // empty series: nothing to write
      if (r == prev_r && c == prev_c) { walk(i); continue; }   // same cell again
      prev_r = r; prev_c = c;
      const uint32_t p = spread1by1_host((uint32_t)(c >> 2)) | (spread1by1_host((uint32_t)(r >> 2)) << 1);
      const uint32_t bit = 4u * (2u * (((uint32_t)r >> 1) & 1u) + (((uint32_t)c >> 1) & 1u)) + 2u * ((uint32_t)r & 1u) + ((uint32_t)c & 1u);
      mk[p] |= (uint16_t)(1u << bit);
      refs.push_back(CellRef{out_off[i], s_, e_, 16u * p + bit, 0u});
      t_min = std::min(t_min, s_); t_max = std::max(t_max, e_);
    }
    const uint32_t ref_count = (uint32_t)refs.size() - ref_first;
    if (ref_count) {
      const uint32_t slot = (uint32_t)tile;
      for (i64 sl = t_min / mb->Q.chunk_size; sl <= (t_max - 1) / mb->Q.chunk_size; sl++)
        jobs.push_back(SeriesJob{(uint32_t)sl, slot, tile_idx, ref_first, ref_count, 0u, t_min, t_max});
    }
    j0 = j1;
  }
  const uint64_t n_walk = bases.size();
  bases.push_back(out_off[n]);
  OutTarget ot = out_begin(ctx, out, os.esize * total, mem);
  // uploads first, then the timed kernels
  TileSeriesParams TP;
  if (!jobs.empty()) {
    const size_t b_masks = sizeof(uint16_t) * masks.size(), b_refs = sizeof(CellRef) * refs.size(), b_jobs = sizeof(SeriesJob) * jobs.size();
    ctx->query_aux.reserve(b_masks + 16);
    ctx->query_aux2.reserve(b_refs + b_jobs + 32);
    CellRef* d_refs = ctx->query_aux2.as<CellRef>();
    SeriesJob* d_jobs = reinterpret_cast<SeriesJob*>(ctx->query_aux2.as<u8>() + ((b_refs + 15) & ~size_t(15)));
    CK(cudaMemcpyAsync(ctx->query_aux.p, masks.data(), b_masks, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_refs, refs.data(), b_refs, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_jobs, jobs.data(), b_jobs, cudaMemcpyHostToDevice, ctx->stream));
    TP.Q = mb->Q; TP.jobs = d_jobs; TP.n_jobs = jobs.size(); TP.masks = ctx->query_aux.as<uint16_t>(); TP.refs = d_refs;
    TP.out = ot.dev; TP.raw = os.raw;
  }
  i64* d_q = nullptr;
  u64* d_off = nullptr;
  if (n_walk) {
    ctx->query_in.reserve(sizeof(i64) * 4 * n_walk + sizeof(u64) * (n_walk + 1));
    d_q = ctx->query_in.as<i64>();
    d_off = reinterpret_cast<u64*>(d_q + 4 * n_walk);
    CK(cudaMemcpyAsync(d_q, qs.data(), sizeof(i64) * 4 * n_walk, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_off, bases.data(), sizeof(u64) * (n_walk + 1), cudaMemcpyHostToDevice, ctx->stream));
  }
  tbegin(ctx, KT_CELL);
  if (!jobs.empty()) {
    const bool narrow = mb->max_dac_levels <= 3 && !ctx->opt.window_wide;
    if (narrow) CK(cudaFuncSetAttribute(k_cell_tiles4<int32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Series4Smem<int32_t>)));
    else CK(cudaFuncSetAttribute(k_cell_tiles4<i64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Series4Smem<i64>)));
    const unsigned grid = (unsigned)std::min<u64>(jobs.size(), (u64)ctx->sm_count * 64);
    if (narrow) k_cell_tiles4<int32_t><<<grid, DT_THREADS, sizeof(Series4Smem<int32_t>), ctx->stream>>>(TP);
    else k_cell_tiles4<i64><<<grid, DT_THREADS, sizeof(Series4Smem<i64>), ctx->stream>>>(TP);
    CK(cudaGetLastError());
    ctx->launches++;
  }
  if (n_walk) {
    dim3 grid((unsigned)std::min<i64>((longest + 127) / 128, 1024), (unsigned)std::min<uint64_t>(n_walk, 65535));
    k_cell_batch<<<grid, 128, 0, ctx->stream>>>(mb->Q, d_q, d_off, n_walk, ot.dev, os.raw);
    CK(cudaGetLastError());
    ctx->launches++;
  }
  tend(ctx, KT_CELL);
  out_end(ctx, ot);  // the host vectors stay alive until here
  tcollect(ctx, KT_CELL);
}

// Jobs of the tile window decoder (k_window_tiles4): one per (window, time slice, subchunk the window touches), window after
// window, slices ascending, subchunks row-major; job_base[i] is window i's first, job_base[n] the count.
u64 window_jobs(const MetaBlock* mb, const std::vector<CubeDev>& cubes, std::vector<u64>& job_base) {
  const uint64_t n = cubes.size();
  job_base.assign(n + 1, 0);
  u64 n_jobs = 0;
  const i64 cs = mb->Q.chunks_sidelen;
  for (uint64_t i = 0; i < n; i++) {
    const CubeDev& c = cubes[i];
    job_base[i] = n_jobs;
    if (c.end > c.start && c.bottom > c.top && c.right > c.left) {
      const u64 nsub = (u64)((c.bottom - 1) / cs - c.top / cs + 1) * (u64)((c.right - 1) / cs - c.left / cs + 1);
      const u64 nsl = (u64)((c.end - 1) / mb->Q.chunk_size - c.start / mb->Q.chunk_size + 1);
      n_jobs += nsub * nsl;
    }
  }
  job_base[n] = n_jobs;
  return n_jobs;
}

void do_window_batch(dcdf_ctx* ctx, MetaBlock* mb, uint64_t n, const dcdf_cube* bounds, const uint64_t* out_off, void* out,
                     int32_t out_encoding, int32_t mem) {
  if (n == 0) return;
  if (!bounds || !out_off) api_fail(DCDF_ERR_BAD_ARG, "null windows");
  const OutSpec os = out_spec(out_encoding, mb->Q.encoding);
  std::vector<CubeDev> cubes(n);
  i64 biggest = 1;
  for (uint64_t i = 0; i < n; i++) {
    const dcdf_cube c = order_cube(bounds[i]);
    check_cube(c, mb->Q.shape);
    cubes[i] = {c.start, c.end, c.top, c.bottom, c.left, c.right};
    const i64 cells = (c.end - c.start) * (c.bottom - c.top) * (c.right - c.left);
    if ((uint64_t)cells != out_off[i + 1] - out_off[i]) api_fail(DCDF_ERR_BAD_ARG, "out_off does not match the window sizes");
    biggest = std::max(biggest, cells);
  }
  const size_t total = out_off[n];
  ctx->query_in.reserve(sizeof(CubeDev) * n + sizeof(u64) * (n + 1));
  CubeDev* d_c = ctx->query_in.as<CubeDev>();
  u64* d_off = reinterpret_cast<u64*>(d_c + n);
  CK(cudaMemcpyAsync(d_c, cubes.data(), sizeof(CubeDev) * n, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(d_off, out_off, sizeof(u64) * (n + 1), cudaMemcpyHostToDevice, ctx->stream));
  OutTarget ot = out_begin(ctx, out, os.esize * total, mem);
  const bool tiles = mb->max_sidelen <= 64 && !ctx->opt.window_cells;
  if (tiles) {
    // one CTA per (window, slice, subchunk): per-thread walk with one block barrier per instant (decode_tile4.cuh)
    std::vector<u64> job_base;
    const u64 n_jobs = window_jobs(mb, cubes, job_base);
    ctx->query_aux.reserve(sizeof(u64) * (n + 1));
    CK(cudaMemcpyAsync(ctx->query_aux.p, job_base.data(), sizeof(u64) * (n + 1), cudaMemcpyHostToDevice, ctx->stream));
    TileWindowParams TP;
    TP.Q = mb->Q; TP.cubes = d_c; TP.out_off = d_off; TP.job_base = ctx->query_aux.as<u64>();
    TP.n_queries = n; TP.n_jobs = n_jobs; TP.out = ot.dev; TP.raw = os.raw;
    TP.part_base = nullptr; TP.part = nullptr;
    const bool narrow = mb->max_dac_levels <= 3 && !ctx->opt.window_wide;  // 32-bit expansion (4 CTAs / SM instead of 2)
    CK(cudaFuncSetAttribute(k_window_tiles4<i64, QuadOut>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Tile4Smem<i64>)));
    CK(cudaFuncSetAttribute(k_window_tiles4<int32_t, QuadOut>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Tile4Smem<int32_t>)));
    tbegin(ctx, KT_WINDOW);
    if (n_jobs) {
      const unsigned grid = (unsigned)std::min<u64>(n_jobs, (u64)ctx->sm_count * 64);
      if (narrow) k_window_tiles4<int32_t, QuadOut><<<grid, DT_THREADS, sizeof(Tile4Smem<int32_t>), ctx->stream>>>(TP);
      else k_window_tiles4<i64, QuadOut><<<grid, DT_THREADS, sizeof(Tile4Smem<i64>), ctx->stream>>>(TP);
      CK(cudaGetLastError());
      ctx->launches++;
    }
    tend(ctx, KT_WINDOW);
    out_end(ctx, ot);  // job_base stays alive until here
    tcollect(ctx, KT_WINDOW);
    return;
  }
  const unsigned gy = (unsigned)std::min<uint64_t>(n, 65535);
  const unsigned gx = (unsigned)std::max<i64>(1, std::min<i64>((biggest / 8 + 127) / 128, std::max<i64>(1, (i64)ctx->sm_count * 32 / gy)));
  tbegin(ctx, KT_WINDOW);
  k_window_blocks<<<dim3(gx, gy), 128, 0, ctx->stream>>>(mb->Q, d_c, d_off, n, ot.dev, os.raw);
  CK(cudaGetLastError());
  ctx->launches++;
  tend(ctx, KT_WINDOW);
  out_end(ctx, ot);
  tcollect(ctx, KT_WINDOW);
}

// Per-instant statistics of n windows (dcdf_superchunk_window_stats): k_window_tiles4<V, StatsOut<V>> writes one partial per
// (window, subchunk, instant), k_window_stats_combine folds them into the records.  Superchunk subchunks are at most 64x64
// (dcdf_superchunk_build refuses larger leaves); an opened superchunk with larger ones is refused here, there is no second
// reduction path.
void do_window_stats(dcdf_ctx* ctx, MetaBlock* mb, uint64_t n, const dcdf_cube* bounds, const uint64_t* out_off, uint64_t* count,
                     void* vmin, void* vmax, double* sum, double* sum_sq, int32_t mem) {
  if (n == 0) return;
  if (!bounds || !out_off || !count || !vmin || !vmax || !sum || !sum_sq) api_fail(DCDF_ERR_BAD_ARG, "null window statistics argument");
  if (mem != DCDF_MEM_HOST && mem != DCDF_MEM_DEVICE) api_fail(DCDF_ERR_BAD_ARG, "mem must be DCDF_MEM_HOST or DCDF_MEM_DEVICE");
  if (mb->max_sidelen > 64) api_fail(DCDF_ERR_BAD_ARG, "window statistics need subchunks of at most 64x64");
  std::vector<CubeDev> cubes(n);
  std::vector<u64> part_base(n);
  u64 n_part = 0;
  const i64 cs = mb->Q.chunks_sidelen;
  for (uint64_t i = 0; i < n; i++) {
    const dcdf_cube c = order_cube(bounds[i]);
    check_cube(c, mb->Q.shape);
    cubes[i] = {c.start, c.end, c.top, c.bottom, c.left, c.right};
    if (out_off[i + 1] < out_off[i] || (uint64_t)(c.end - c.start) != out_off[i + 1] - out_off[i])
      api_fail(DCDF_ERR_BAD_ARG, "out_off does not match the windows' instants");
    part_base[i] = n_part;
    if (c.bottom > c.top && c.right > c.left)
      n_part += (u64)((c.bottom - 1) / cs - c.top / cs + 1) * (u64)((c.right - 1) / cs - c.left / cs + 1) * (u64)(c.end - c.start);
  }
  const u64 rec0 = out_off[0], rec1 = out_off[n], n_rec = rec1 - rec0;
  std::vector<u64> job_base;
  const u64 n_jobs = window_jobs(mb, cubes, job_base);
  cudaStream_t st = ctx->stream;
  ctx->query_in.reserve(sizeof(CubeDev) * n + sizeof(u64) * (n + 1));
  CubeDev* d_c = ctx->query_in.as<CubeDev>();
  u64* d_off = reinterpret_cast<u64*>(d_c + n);
  CK(cudaMemcpyAsync(d_c, cubes.data(), sizeof(CubeDev) * n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_off, out_off, sizeof(u64) * (n + 1), cudaMemcpyHostToDevice, st));
  ctx->query_aux.reserve(sizeof(u64) * (2 * n + 1));
  u64* d_jb = ctx->query_aux.as<u64>();
  u64* d_pb = d_jb + n + 1;
  CK(cudaMemcpyAsync(d_jb, job_base.data(), sizeof(u64) * (n + 1), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_pb, part_base.data(), sizeof(u64) * n, cudaMemcpyHostToDevice, st));
  ctx->query_aux2.reserve(sizeof(StatsPartial) * std::max<u64>(n_part, 1));
  // outputs from record rec0 on: the caller's device arrays, or one staging block for the five host arrays
  const size_t es = enc_size(mb->Q.encoding);
  u64* o_count = count + rec0;
  void* o_min = static_cast<u8*>(vmin) + es * rec0;
  void* o_max = static_cast<u8*>(vmax) + es * rec0;
  double* o_sum = sum + rec0;
  double* o_sq = sum_sq + rec0;
  if (mem == DCDF_MEM_HOST) {
    const size_t a8 = (sizeof(u64) * n_rec + 15) & ~size_t(15), ae = (es * n_rec + 15) & ~size_t(15);
    ctx->query_out.reserve(3 * a8 + 2 * ae);
    u8* b = ctx->query_out.as<u8>();
    o_count = reinterpret_cast<u64*>(b);
    o_min = b + a8;
    o_max = b + a8 + ae;
    o_sum = reinterpret_cast<double*>(b + a8 + 2 * ae);
    o_sq = reinterpret_cast<double*>(b + 2 * a8 + 2 * ae);
  }
  TileWindowParams TP;
  TP.Q = mb->Q; TP.cubes = d_c; TP.out_off = d_off; TP.job_base = d_jb;
  TP.n_queries = n; TP.n_jobs = n_jobs; TP.out = nullptr; TP.raw = 0;
  TP.part_base = d_pb; TP.part = ctx->query_aux2.as<StatsPartial>();
  StatsCombineParams CP;
  CP.cubes = d_c; CP.out_off = d_off; CP.part_base = d_pb; CP.part = TP.part;
  CP.n_queries = n; CP.rec0 = rec0; CP.rec1 = rec1; CP.cs = cs; CP.encoding = mb->Q.encoding;
  CP.count = o_count; CP.vmin = o_min; CP.vmax = o_max; CP.sum = o_sum; CP.sum_sq = o_sq;
  const bool narrow = mb->max_dac_levels <= 3 && !ctx->opt.window_wide;
  const int smem32 = (int)(sizeof(Tile4Smem<int32_t>) + sizeof(StatsShared<int32_t>));
  const int smem64 = (int)(sizeof(Tile4Smem<i64>) + sizeof(StatsShared<i64>));
  if (narrow) CK(cudaFuncSetAttribute(k_window_tiles4<int32_t, StatsOut<int32_t>>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem32));
  else CK(cudaFuncSetAttribute(k_window_tiles4<i64, StatsOut<i64>>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem64));
  tbegin(ctx, KT_REDUCE);
  if (n_jobs) {
    const unsigned grid = (unsigned)std::min<u64>(n_jobs, (u64)ctx->sm_count * 64);
    if (narrow) k_window_tiles4<int32_t, StatsOut<int32_t>><<<grid, DT_THREADS, smem32, st>>>(TP);
    else k_window_tiles4<i64, StatsOut<i64>><<<grid, DT_THREADS, smem64, st>>>(TP);
    CK(cudaGetLastError());
    ctx->launches++;
  }
  if (n_rec) {
    k_window_stats_combine<<<(unsigned)((n_rec + 255) / 256), 256, 0, st>>>(CP);
    CK(cudaGetLastError());
    ctx->launches++;
  }
  tend(ctx, KT_REDUCE);
  if (mem == DCDF_MEM_HOST && n_rec) {
    CK(cudaMemcpyAsync(count + rec0, o_count, sizeof(u64) * n_rec, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(static_cast<u8*>(vmin) + es * rec0, o_min, es * n_rec, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(static_cast<u8*>(vmax) + es * rec0, o_max, es * n_rec, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(sum + rec0, o_sum, sizeof(double) * n_rec, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(sum_sq + rec0, o_sq, sizeof(double) * n_rec, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));  // job_base / part_base stay alive until here
  tcollect(ctx, KT_REDUCE);
}

// Per-cell statistics over time of n windows (dcdf_superchunk_time_stats).  The slices the windows touch are cut into
// groups whose partials (one TimePartial per (window, slice, cell)) fit the "time_stats_scratch" budget, at least one
// slice per group.  Per group, every window is clipped to the group's instants, k_window_tiles4<V, TimeStatsOut<V>> runs
// the group's jobs and k_time_stats_combine continues the records with the group's pieces in slice order; so the records
// do not depend on the grouping.  Subchunks larger than 64x64 are refused as in do_window_stats.
void do_time_stats(dcdf_ctx* ctx, MetaBlock* mb, uint64_t n, const dcdf_cube* bounds, const uint64_t* out_off, const double* lower,
                   const double* upper, uint64_t* count, uint64_t* n_band, void* vmin, void* vmax, double* sum, double* sum_sq,
                   int32_t accumulate, int32_t mem) {
  ctx->last_time_groups = 0;
  ctx->last_time_scratch = 0;
  if (n == 0) return;
  if (!bounds || !out_off || !count || !vmin || !vmax || !sum || !sum_sq) api_fail(DCDF_ERR_BAD_ARG, "null time statistics argument");
  if (!lower != !upper) api_fail(DCDF_ERR_BAD_ARG, "lower and upper must both be given or both be NULL");
  const bool band = lower != nullptr;
  if (band && !n_band) api_fail(DCDF_ERR_BAD_ARG, "a band needs n_band");
  if (mem != DCDF_MEM_HOST && mem != DCDF_MEM_DEVICE) api_fail(DCDF_ERR_BAD_ARG, "mem must be DCDF_MEM_HOST or DCDF_MEM_DEVICE");
  if (mb->max_sidelen > 64) api_fail(DCDF_ERR_BAD_ARG, "time statistics need subchunks of at most 64x64");
  std::vector<CubeDev> cubes(n);
  std::vector<double> bnd(band ? 2 * n : 0);
  const i64 csz = mb->Q.chunk_size, T = mb->Q.shape[0];
  const i64 n_sl = (T + csz - 1) / csz;
  std::vector<u64> cost(n_sl + 1, 0);  // cells of the windows that cover each slice (a difference array first)
  for (uint64_t i = 0; i < n; i++) {
    const dcdf_cube c = order_cube(bounds[i]);
    check_cube(c, mb->Q.shape);
    cubes[i] = {c.start, c.end, c.top, c.bottom, c.left, c.right};
    const u64 area = (u64)((c.bottom - c.top) * (c.right - c.left));
    if (out_off[i + 1] < out_off[i] || area != out_off[i + 1] - out_off[i]) api_fail(DCDF_ERR_BAD_ARG, "out_off does not match the windows' areas");
    if (band) {
      double lo = lower[i], hi = upper[i];
      if (std::isnan(lo) || std::isnan(hi)) api_fail(DCDF_ERR_BAD_ARG, "NaN band bound in window %llu", (unsigned long long)i);
      if (lo > hi) std::swap(lo, hi);
      bnd[2 * i] = lo; bnd[2 * i + 1] = hi;
    }
    if (area && c.end > c.start) {
      cost[c.start / csz] += area;
      cost[(c.end - 1) / csz + 1] -= area;
    }
  }
  for (i64 s = 1; s <= n_sl; s++) cost[s] += cost[s - 1];
  // groups of slices [g_lo, g_hi): greedy in slice order under the budget; slices no window covers are skipped
  const u64 budget = ctx->opt.time_stats_scratch;
  std::vector<std::pair<i64, i64>> groups;
  u64 g_bytes = 0, max_bytes = 0;
  for (i64 s = 0; s < n_sl; s++) {
    const u64 b = cost[s] * sizeof(TimePartial);
    if (!b) continue;
    if (groups.empty() || g_bytes + b > budget) {
      groups.push_back({s, s + 1});
      g_bytes = 0;
    }
    groups.back().second = s + 1;
    g_bytes += b;
    max_bytes = std::max(max_bytes, g_bytes);
  }
  const u64 rec0 = out_off[0], rec1 = out_off[n], n_rec = rec1 - rec0;
  const bool no_slices = groups.empty();
  if (no_slices) {
    if (accumulate || !n_rec) return;  // nothing to continue / no records
    groups.push_back({0, 0});          // zero-instant windows: the combine writes empty records
  }
  const size_t n_g = groups.size();
  // every group's clipped windows, job and partial offsets, uploaded before the timed kernels
  std::vector<CubeDev> gcubes(n_g * n);
  std::vector<u64> job_base(n_g * (n + 1)), part_base(n_g * n), n_jobs(n_g);
  for (size_t g = 0; g < n_g; g++) {
    const i64 t_lo = groups[g].first * csz, t_hi = std::min(groups[g].second * csz, T);
    CubeDev* gc = gcubes.data() + g * n;
    u64 np = 0;
    for (uint64_t i = 0; i < n; i++) {
      gc[i] = cubes[i];
      gc[i].start = std::min(std::max(cubes[i].start, t_lo), t_hi);
      gc[i].end = std::max(std::min(cubes[i].end, t_hi), gc[i].start);
      part_base[g * n + i] = np;
      if (gc[i].end > gc[i].start)
        np += (u64)((gc[i].bottom - gc[i].top) * (gc[i].right - gc[i].left)) * (u64)((gc[i].end - 1) / csz - gc[i].start / csz + 1);
    }
    std::vector<u64> jb;
    n_jobs[g] = window_jobs(mb, std::vector<CubeDev>(gc, gc + n), jb);
    std::copy(jb.begin(), jb.end(), job_base.begin() + g * (n + 1));
  }
  cudaStream_t st = ctx->stream;
  const size_t b_cubes = sizeof(CubeDev) * n_g * n, b_off = sizeof(u64) * (n + 1);
  ctx->query_in.reserve(b_cubes + b_off);
  CubeDev* d_c = ctx->query_in.as<CubeDev>();
  u64* d_off = reinterpret_cast<u64*>(d_c + n_g * n);
  CK(cudaMemcpyAsync(d_c, gcubes.data(), b_cubes, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_off, out_off, b_off, cudaMemcpyHostToDevice, st));
  ctx->query_aux.reserve(sizeof(u64) * (job_base.size() + part_base.size()) + sizeof(double) * bnd.size());
  u64* d_jb = ctx->query_aux.as<u64>();
  u64* d_pb = d_jb + job_base.size();
  double* d_band = reinterpret_cast<double*>(d_pb + part_base.size());
  CK(cudaMemcpyAsync(d_jb, job_base.data(), sizeof(u64) * job_base.size(), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_pb, part_base.data(), sizeof(u64) * part_base.size(), cudaMemcpyHostToDevice, st));
  if (band) CK(cudaMemcpyAsync(d_band, bnd.data(), sizeof(double) * bnd.size(), cudaMemcpyHostToDevice, st));
  ctx->query_aux2.reserve(std::max<u64>(max_bytes, 16));
  // outputs from record rec0 on: the caller's device arrays, or one staging block for the six host arrays (loaded with
  // the records to continue under accumulate)
  const size_t es = enc_size(mb->Q.encoding);
  u64* o_count = count + rec0;
  u64* o_band = n_band ? n_band + rec0 : nullptr;
  void* o_min = static_cast<u8*>(vmin) + es * rec0;
  void* o_max = static_cast<u8*>(vmax) + es * rec0;
  double* o_sum = sum + rec0;
  double* o_sq = sum_sq + rec0;
  if (mem == DCDF_MEM_HOST) {
    const size_t a8 = (sizeof(u64) * n_rec + 15) & ~size_t(15), ae = (es * n_rec + 15) & ~size_t(15);
    ctx->query_out.reserve(4 * a8 + 2 * ae);
    u8* b = ctx->query_out.as<u8>();
    u64* s_count = reinterpret_cast<u64*>(b);
    u64* s_band = reinterpret_cast<u64*>(b + a8);
    void* s_min = b + 2 * a8;
    void* s_max = b + 2 * a8 + ae;
    double* s_sum = reinterpret_cast<double*>(b + 2 * a8 + 2 * ae);
    double* s_sq = reinterpret_cast<double*>(b + 3 * a8 + 2 * ae);
    if (accumulate && n_rec) {
      CK(cudaMemcpyAsync(s_count, o_count, sizeof(u64) * n_rec, cudaMemcpyHostToDevice, st));
      if (o_band) CK(cudaMemcpyAsync(s_band, o_band, sizeof(u64) * n_rec, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(s_min, o_min, es * n_rec, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(s_max, o_max, es * n_rec, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(s_sum, o_sum, sizeof(double) * n_rec, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(s_sq, o_sq, sizeof(double) * n_rec, cudaMemcpyHostToDevice, st));
    }
    o_count = s_count; o_band = o_band ? s_band : nullptr; o_min = s_min; o_max = s_max; o_sum = s_sum; o_sq = s_sq;
  }
  TileWindowParams TP;
  TP.Q = mb->Q; TP.out_off = d_off; TP.n_queries = n; TP.out = nullptr; TP.raw = 0;
  TP.part = nullptr; TP.tpart = ctx->query_aux2.as<TimePartial>(); TP.band = band ? d_band : nullptr;
  TimeCombineParams CP;
  CP.out_off = d_off; CP.part = TP.tpart; CP.n_queries = n; CP.rec0 = rec0; CP.rec1 = rec1; CP.chunk_size = csz;
  CP.encoding = mb->Q.encoding;
  CP.count = o_count; CP.n_band = o_band; CP.vmin = o_min; CP.vmax = o_max; CP.sum = o_sum; CP.sum_sq = o_sq;
  const bool narrow = mb->max_dac_levels <= 3 && !ctx->opt.window_wide;
  const int smem32 = (int)(sizeof(Tile4Smem<int32_t>) + sizeof(TimeStatsShared<int32_t>));
  const int smem64 = (int)(sizeof(Tile4Smem<i64>) + sizeof(TimeStatsShared<i64>));
  if (narrow) CK(cudaFuncSetAttribute(k_window_tiles4<int32_t, TimeStatsOut<int32_t>>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem32));
  else CK(cudaFuncSetAttribute(k_window_tiles4<i64, TimeStatsOut<i64>>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem64));
  tbegin(ctx, KT_TIME_STATS);
  for (size_t g = 0; g < n_g; g++) {
    TP.cubes = CP.cubes = d_c + g * n;
    TP.job_base = d_jb + g * (n + 1);
    TP.part_base = CP.part_base = d_pb + g * n;
    TP.n_jobs = n_jobs[g];
    if (n_jobs[g]) {
      const unsigned grid = (unsigned)std::min<u64>(n_jobs[g], (u64)ctx->sm_count * 64);
      if (narrow) k_window_tiles4<int32_t, TimeStatsOut<int32_t>><<<grid, DT_THREADS, smem32, st>>>(TP);
      else k_window_tiles4<i64, TimeStatsOut<i64>><<<grid, DT_THREADS, smem64, st>>>(TP);
      CK(cudaGetLastError());
      ctx->launches++;
    }
    if (n_rec) {
      CP.init = g == 0 && !accumulate;
      k_time_stats_combine<<<(unsigned)((n_rec + 255) / 256), 256, 0, st>>>(CP);
      CK(cudaGetLastError());
      ctx->launches++;
    }
  }
  tend(ctx, KT_TIME_STATS);
  if (mem == DCDF_MEM_HOST && n_rec) {
    CK(cudaMemcpyAsync(count + rec0, o_count, sizeof(u64) * n_rec, cudaMemcpyDeviceToHost, st));
    if (o_band) CK(cudaMemcpyAsync(n_band + rec0, o_band, sizeof(u64) * n_rec, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(static_cast<u8*>(vmin) + es * rec0, o_min, es * n_rec, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(static_cast<u8*>(vmax) + es * rec0, o_max, es * n_rec, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(sum + rec0, o_sum, sizeof(double) * n_rec, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(sum_sq + rec0, o_sq, sizeof(double) * n_rec, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  tcollect(ctx, KT_TIME_STATS);
  ctx->last_time_groups = no_slices ? 0 : n_g;
  ctx->last_time_scratch = max_bytes;
}

// Fixed-point bounds (lower / upper), or, with strict, value bounds (vlower / vupper) that the kernels convert per subchunk
// with its own fractional bits, with the exact hit set (the strict kernels: k_search_tiles4 / k_count_tiles4 / k_search
// with ST = true).
void do_search_batch(dcdf_ctx* ctx, MetaBlock* mb, uint64_t n, const dcdf_cube* bounds, const int64_t* lower, const int64_t* upper,
                     uint64_t* counts, int64_t* out_irc, uint64_t cap, uint64_t* n_found, int32_t mem, bool strict = false,
                     const double* vlower = nullptr, const double* vupper = nullptr) {
  if (n_found) *n_found = 0;
  if (n == 0) return;
  if (!bounds || (strict ? !vlower || !vupper : !lower || !upper)) api_fail(DCDF_ERR_BAD_ARG, "null search arguments");
  std::vector<double> vlo, vhi;
  if (strict) {
    vlo.assign(vlower, vlower + n);
    vhi.assign(vupper, vupper + n);
    for (uint64_t i = 0; i < n; i++) {
      if (std::isnan(vlo[i]) || std::isnan(vhi[i])) api_fail(DCDF_ERR_BAD_ARG, "NaN search bound in window %llu", (unsigned long long)i);
      if (vlo[i] > vhi[i]) std::swap(vlo[i], vhi[i]);  // helpers.rs:7-16 via chunk.rs:214
    }
  }
  cudaStream_t st = ctx->stream;
  std::vector<CubeDev> cubes(n);
  std::vector<u64> job_base(n + 1);
  u64 n_jobs = 0;
  const i64 cs = mb->Q.chunks_sidelen;
  for (uint64_t i = 0; i < n; i++) {
    const dcdf_cube c = order_cube(bounds[i]);
    check_cube(c, mb->Q.shape);
    cubes[i] = {c.start, c.end, c.top, c.bottom, c.left, c.right};
    job_base[i] = n_jobs;
    if (c.end > c.start && c.bottom > c.top && c.right > c.left) {
      const u64 nsub = (u64)((c.bottom - 1) / cs - c.top / cs + 1) * (u64)((c.right - 1) / cs - c.left / cs + 1);
      n_jobs += nsub * (u64)(c.end - c.start);
    }
  }
  job_base[n] = n_jobs;
  if (n_jobs == 0) {
    if (counts) std::fill(counts, counts + n, 0);
    return;
  }
  const size_t in_bytes = sizeof(CubeDev) * n + sizeof(u64) * (n + 1) + 2 * sizeof(i64) * n;
  ctx->query_in.reserve(in_bytes);
  CubeDev* d_c = ctx->query_in.as<CubeDev>();
  u64* d_jb = reinterpret_cast<u64*>(d_c + n);
  i64* d_lo = reinterpret_cast<i64*>(d_jb + n + 1);
  i64* d_hi = d_lo + n;
  CK(cudaMemcpyAsync(d_c, cubes.data(), sizeof(CubeDev) * n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_jb, job_base.data(), sizeof(u64) * (n + 1), cudaMemcpyHostToDevice, st));
  // the strict search's value bounds take the place of the fixed ones (both 8 bytes a window)
  CK(cudaMemcpyAsync(d_lo, strict ? (const void*)vlo.data() : (const void*)lower, sizeof(i64) * n, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_hi, strict ? (const void*)vhi.data() : (const void*)upper, sizeof(i64) * n, cudaMemcpyHostToDevice, st));
  const double* d_vlo = reinterpret_cast<const double*>(d_lo);
  const double* d_vhi = reinterpret_cast<const double*>(d_hi);
  const u64 n_scan_chunks = (n_jobs + SCAN_CHUNK - 1) / SCAN_CHUNK;
  ctx->query_aux.reserve(sizeof(u64) * (2 * n_jobs + 2) + sizeof(u64) * (n + 1) + sizeof(u64) * (2 * n_scan_chunks + 2));
  u64* d_counts = ctx->query_aux.as<u64>();
  u64* d_offsets = d_counts + n_jobs;
  u64* d_pick = d_offsets + n_jobs + 1;
  u64* d_sums = d_pick + n + 1;
  u64* d_sum_off = d_sums + n_scan_chunks;
  SearchParams SP;
  SP.Q = mb->Q;
  SP.cubes = d_c; SP.job_base = d_jb; SP.n_queries = n; SP.n_jobs = n_jobs;
  SP.lower = d_lo; SP.upper = d_hi; SP.vlower = d_vlo; SP.vupper = d_vhi;
  SP.counts = d_counts; SP.offsets = d_offsets;
  SP.out = nullptr; SP.cap = 0;
  const unsigned grid = (unsigned)((n_jobs + 127) / 128);
  // default for trees up to 64x64: one CTA per (window, time slice, subchunk) with the per-thread walk (decode_search4.cuh);
  // option "search_dfs": one thread per (window, subchunk, instant) replaying the depth-first traversal (k_search)
  const bool tiles = mb->max_sidelen <= 64 && !ctx->opt.search_dfs;
  const bool narrow = mb->max_dac_levels <= 3 && !ctx->opt.window_wide;
  TileSearchParams TS;
  unsigned tgrid = 0;
  if (tiles) {
    std::vector<u64> tile_base(n + 1);
    u64 n_tiles = 0;
    for (uint64_t i = 0; i < n; i++) {
      const CubeDev& c = cubes[i];
      tile_base[i] = n_tiles;
      if (c.end > c.start && c.bottom > c.top && c.right > c.left) {
        const u64 nsub = (u64)((c.bottom - 1) / cs - c.top / cs + 1) * (u64)((c.right - 1) / cs - c.left / cs + 1);
        const u64 nsl = (u64)((c.end - 1) / mb->Q.chunk_size - c.start / mb->Q.chunk_size + 1);
        n_tiles += nsub * nsl;
      }
    }
    tile_base[n] = n_tiles;
    ctx->query_aux2.reserve(sizeof(u64) * (n + 1));
    CK(cudaMemcpyAsync(ctx->query_aux2.p, tile_base.data(), sizeof(u64) * (n + 1), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));  // tile_base is a local
    TS.Q = mb->Q; TS.cubes = d_c; TS.job_base = d_jb; TS.tile_base = ctx->query_aux2.as<u64>();
    TS.n_queries = n; TS.n_tiles = n_tiles; TS.lower = d_lo; TS.upper = d_hi; TS.vlower = d_vlo; TS.vupper = d_vhi;
    TS.counts = d_counts; TS.offsets = d_offsets; TS.out = nullptr; TS.cap = 0;
    // 1 KB per (window, subchunk, instant) keeps the counting pass's findings for the writing pass (up to 2 GB)
    TS.hit_cache = nullptr;
    if (out_irc && n_jobs * (u64)DT_THREADS * 4ull <= (2ull << 30) && !ctx->opt.search_no_cache) {
      ctx->search_cache.reserve(n_jobs * (size_t)DT_THREADS * 4);
      TS.hit_cache = ctx->search_cache.as<u32>();
    }
    tgrid = (unsigned)std::min<u64>(n_tiles, (u64)ctx->sm_count * 64);
    if (strict) {
      CK(cudaFuncSetAttribute(k_search_tiles4<i64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Search4Smem<i64>)));
      CK(cudaFuncSetAttribute(k_search_tiles4<int32_t, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Search4Smem<int32_t>)));
    } else {
      CK(cudaFuncSetAttribute(k_search_tiles4<i64, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Search4Smem<i64>)));
      CK(cudaFuncSetAttribute(k_search_tiles4<int32_t, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Search4Smem<int32_t>)));
    }
  }
  // Counting pass with shared decodes (k_count_tiles4) when the windows of the batch overlap: every (time slice, tile) some
  // window touches is decoded once for all of them.  Worth it from a few windows per touched tile on (ctx option
  // "search_share_min", default 3; the per-window kernel prunes by the window's own band, which a shared decode cannot).
  bool shared_count = false;
  TileCountParams TC;
  unsigned cgrid = 0;
  std::vector<CountEntry> entries;
  std::vector<CountJob> cjobs;
  // (a call that also wants the cells keeps the per-window counting pass: its cached findings make the writing pass cheap)
  if (tiles && (!out_irc || ctx->opt.search_share_min == 1) && ctx->opt.search_share_min > 0 && cs <= 64 && mb->Q.chunk_size <= 0xffff) {
    const i64 ct = mb->Q.chunk_size;
    const u64 n_slots = mb->Q.n_slots, n_keys = (u64)mb->Q.n_slices * n_slots;
    std::vector<uint32_t> key_count(n_keys + 1, 0);
    u64 n_ent = 0;
    auto for_each_entry = [&](auto&& fn) {
      for (uint64_t q = 0; q < n; q++) {
        const CubeDev& c = cubes[q];
        if (!(c.end > c.start && c.bottom > c.top && c.right > c.left)) continue;
        const i64 cr0 = c.top / cs, cc0 = c.left / cs, cr1 = (c.bottom - 1) / cs, cc1 = (c.right - 1) / cs;
        const i64 ncc = cc1 - cc0 + 1, T_all = c.end - c.start;
        for (i64 sl = c.start / ct; sl <= (c.end - 1) / ct; sl++)
          for (i64 cr = cr0; cr <= cr1; cr++)
            for (i64 cc = cc0; cc <= cc1; cc++) {
              const u64 key = (u64)sl * n_slots + (u64)(cr * mb->Q.subsidelen + cc);
              fn(q, c, sl, cr, cc, (cr - cr0) * ncc + (cc - cc0), T_all, key);
            }
      }
    };
    for_each_entry([&](uint64_t, const CubeDev&, i64, i64, i64, i64, i64, u64 key) { key_count[key + 1]++; n_ent++; });
    u64 touched = 0;
    for (u64 k = 0; k < n_keys; k++) touched += key_count[k + 1] ? 1 : 0;
    if (touched && n_ent >= (u64)ctx->opt.search_share_min * touched && n_ent <= 0xffffffffull) {
      shared_count = true;
      std::vector<u64> key_off(n_keys + 1, 0);
      for (u64 k = 0; k < n_keys; k++) key_off[k + 1] = key_off[k] + key_count[k + 1];
      entries.resize(n_ent);
      std::vector<u64> fill(key_off.begin(), key_off.end() - 1);
      for_each_entry([&](uint64_t q, const CubeDev& c, i64 sl, i64 cr, i64 cc, i64 sub, i64 T_all, u64 key) {
        CountEntry E;
        if (strict) {
          E.vlower = vlo[q]; E.vupper = vhi[q];
        } else {
          i64 lo = lower[q], hi = upper[q];
          if (lo > hi) std::swap(lo, hi);  // helpers.rs:7-16 via chunk.rs:214
          E.lower = lo; E.upper = hi;
        }
        const i64 s0 = sl * ct, t_lo = std::max(c.start, s0), t_hi = std::min(c.end, s0 + ct);
        E.t0 = (uint16_t)(t_lo - s0); E.t1 = (uint16_t)(t_hi - s0);
        E.cnt_base = (i64)job_base[q] + sub * T_all + (s0 - c.start);
        const i64 top = cr * cs, left = cc * cs;
        E.top = (uint8_t)(std::max(top, c.top) - top); E.bottom = (uint8_t)(std::min(top + cs, c.bottom) - top);
        E.left = (uint8_t)(std::max(left, c.left) - left); E.right = (uint8_t)(std::min(left + cs, c.right) - left);
        entries[fill[key]++] = E;
      });
      for (u64 k = 0; k < n_keys; k++)
        for (u64 e0 = key_off[k]; e0 < key_off[k + 1]; e0 += CT_MAX)
          cjobs.push_back(CountJob{(uint32_t)(k / n_slots), (uint32_t)(k % n_slots), (uint32_t)e0,
                                   (uint32_t)std::min<u64>(CT_MAX, key_off[k + 1] - e0)});
      const size_t b_ent = sizeof(CountEntry) * entries.size(), b_jobs = sizeof(CountJob) * cjobs.size();
      ctx->search_cache.reserve(b_ent + b_jobs + 32);
      CountEntry* d_ent = ctx->search_cache.as<CountEntry>();
      CountJob* d_cj = reinterpret_cast<CountJob*>(ctx->search_cache.as<u8>() + ((b_ent + 15) & ~size_t(15)));
      CK(cudaMemcpyAsync(d_ent, entries.data(), b_ent, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(d_cj, cjobs.data(), b_jobs, cudaMemcpyHostToDevice, st));
      TC.Q = mb->Q; TC.jobs = d_cj; TC.n_jobs = cjobs.size(); TC.entries = d_ent; TC.counts = d_counts;
      cgrid = (unsigned)std::min<u64>(cjobs.size(), (u64)ctx->sm_count * 64);
      const void* kc = narrow ? (strict ? (const void*)k_count_tiles4<int32_t, true> : (const void*)k_count_tiles4<int32_t, false>)
                              : (strict ? (const void*)k_count_tiles4<i64, true> : (const void*)k_count_tiles4<i64, false>);
      CK(cudaFuncSetAttribute(kc, cudaFuncAttributeMaxDynamicSharedMemorySize, narrow ? (int)sizeof(Count4Smem<int32_t>) : (int)sizeof(Count4Smem<i64>)));
      TS.hit_cache = nullptr;  // the shared counting pass keeps no per-thread findings; the buffer holds its entries
    }
  }
  auto launch_search = [&](int write) {
    if (tiles && !write && shared_count) {
      CK(cudaMemsetAsync(d_counts, 0, sizeof(u64) * n_jobs, st));
      if (narrow && strict) k_count_tiles4<int32_t, true><<<cgrid, DT_THREADS, sizeof(Count4Smem<int32_t>), st>>>(TC);
      else if (narrow) k_count_tiles4<int32_t, false><<<cgrid, DT_THREADS, sizeof(Count4Smem<int32_t>), st>>>(TC);
      else if (strict) k_count_tiles4<i64, true><<<cgrid, DT_THREADS, sizeof(Count4Smem<i64>), st>>>(TC);
      else k_count_tiles4<i64, false><<<cgrid, DT_THREADS, sizeof(Count4Smem<i64>), st>>>(TC);
    } else if (tiles) {
      if (!write) CK(cudaMemsetAsync(d_counts, 0, sizeof(u64) * n_jobs, st));  // the counting pass adds per warp
      if (narrow && strict) k_search_tiles4<int32_t, true><<<tgrid, DT_THREADS, sizeof(Search4Smem<int32_t>), st>>>(TS);
      else if (narrow) k_search_tiles4<int32_t, false><<<tgrid, DT_THREADS, sizeof(Search4Smem<int32_t>), st>>>(TS);
      else if (strict) k_search_tiles4<i64, true><<<tgrid, DT_THREADS, sizeof(Search4Smem<i64>), st>>>(TS);
      else k_search_tiles4<i64, false><<<tgrid, DT_THREADS, sizeof(Search4Smem<i64>), st>>>(TS);
    } else if (strict) {
      k_search<true><<<grid, 128, 0, st>>>(SP, write);
    } else {
      k_search<false><<<grid, 128, 0, st>>>(SP, write);
    }
  };
  tbegin(ctx, KT_SEARCH);
  launch_search(0);
  CK(cudaGetLastError());
  if (n_jobs <= 4u * SCAN_CHUNK) {
    k_scan_u64<<<1, 1024, 0, st>>>(d_counts, n_jobs, d_offsets);
  } else {
    const unsigned nb = (unsigned)((n_jobs + SCAN_CHUNK - 1) / SCAN_CHUNK);
    k_scan_sums<<<nb, 1024, 0, st>>>(d_counts, n_jobs, d_sums);
    k_scan_u64<<<1, 1024, 0, st>>>(d_sums, nb, d_sum_off);
    k_scan_apply<<<nb, 1024, 0, st>>>(d_counts, n_jobs, d_sum_off, d_offsets);
    ctx->launches += 2;
  }
  CK(cudaGetLastError());
  k_pick_u64<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(d_offsets, d_jb, n + 1, d_pick);
  CK(cudaGetLastError());
  ctx->launches += 3;
  tend(ctx, KT_SEARCH);  // the timer covers the kernels of both passes, not the host round trip / output allocation between them
  std::vector<u64> pick(n + 1);
  CK(cudaMemcpyAsync(pick.data(), d_pick, sizeof(u64) * (n + 1), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  tcollect(ctx, KT_SEARCH);
  const float ms_count = ctx->kernel_ms[KT_SEARCH];
  const u64 total = pick[n];
  if (n_found) *n_found = total;
  if (counts) for (uint64_t i = 0; i < n; i++) counts[i] = pick[i + 1] - pick[i];
  if (out_irc && total) {
    if (cap < total) api_fail(DCDF_ERR_BAD_ARG, "search output too small: need %llu triplets", (unsigned long long)total);
    OutTarget ot = out_begin(ctx, out_irc, sizeof(i64) * 3 * total, mem);
    SP.out = static_cast<i64*>(ot.dev);
    SP.cap = total;
    TS.out = SP.out; TS.cap = total;
    tbegin(ctx, KT_SEARCH);
    launch_search(1);
    CK(cudaGetLastError());
    ctx->launches++;
    tend(ctx, KT_SEARCH);
    out_end(ctx, ot);
    tcollect(ctx, KT_SEARCH);
    ctx->kernel_ms[KT_SEARCH] += ms_count;
  }
}

}  // namespace

namespace dcdf {
void build_super_meta(dcdf_ctx* ctx, const dcdf_superchunk* sc) { super_meta(ctx, sc); }
void free_chunk_meta(void* p) { free_meta(p, true); }
void free_super_meta(void* p) { free_meta(p, false); }
}  // namespace dcdf

extern "C" {

// ===================================================================================== Chunk::read_from
int32_t dcdf_chunk_open(dcdf_ctx* ctx, const uint8_t* bytes, uint64_t len, int32_t mem, dcdf_chunk** out) {
  return guarded(ctx, [&] {
    if (!out) api_fail(DCDF_ERR_BAD_ARG, "null out");
    *out = nullptr;
    if (!bytes || len < 6) api_fail(DCDF_ERR_BAD_FORMAT, "chunk bytes too short");
    if (len > 0xfffffff0ull) api_fail(DCDF_ERR_BAD_FORMAT, "a Chunk larger than 4 GiB cannot be addressed by the decode directory");
    dcdf_chunk* c = new dcdf_chunk();
    c->device = ctx->device;
    try {
      c->bytes = static_cast<uint8_t*>(pool_alloc(len + 64, ctx->stream));
      CK(cudaMemsetAsync(c->bytes + len, 0, 64, ctx->stream));
      CK(cudaMemcpyAsync(c->bytes, bytes, len, mem == DCDF_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
      c->size = len;
      c->owner = true;
      c->shape[0] = 0;  // unknown until the directory pass has counted the instants
      MetaBlock* mb = chunk_meta(ctx, c);
      // block table from the directory (snap indices)
      std::vector<InstDir> dir(c->shape[0]);
      CK(cudaMemcpyAsync(dir.data(), mb->Q.dir, sizeof(InstDir) * dir.size(), cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      uint32_t run = 0;
      for (size_t i = 0; i < dir.size(); i++) {
        if (dir[i].snap == i && i > 0) { c->block_instants.push_back(run); run = 0; }
        run++;
      }
      c->block_instants.push_back(run);
      c->n_blocks = (uint32_t)c->block_instants.size();
    } catch (...) {
      if (c->dir) free_chunk_meta(c->dir);
      c->dir = nullptr;
      pool_free(c->bytes);
      delete c;
      throw;
    }
    *out = c;
  });
}

int32_t dcdf_chunk_get_batch(dcdf_ctx* ctx, const dcdf_chunk* chunk, uint64_t n, const int64_t* irc, void* out,
                             int32_t out_encoding, int32_t mem) {
  return guarded(ctx, [&] {
    if (!chunk) api_fail(DCDF_ERR_BAD_ARG, "null chunk");
    do_get_batch(ctx, chunk_meta(ctx, chunk), n, irc, out, out_encoding, mem);
  });
}

int32_t dcdf_chunk_cell_batch(dcdf_ctx* ctx, const dcdf_chunk* chunk, uint64_t n, const int64_t* q, const uint64_t* out_off,
                              void* out, int32_t out_encoding, int32_t mem) {
  return guarded(ctx, [&] {
    if (!chunk) api_fail(DCDF_ERR_BAD_ARG, "null chunk");
    do_cell_batch(ctx, chunk_meta(ctx, chunk), n, q, out_off, out, out_encoding, mem);
  });
}

int32_t dcdf_chunk_window(dcdf_ctx* ctx, const dcdf_chunk* chunk, const dcdf_cube* bounds, void* out, int32_t out_encoding,
                          int32_t mem) {
  return guarded(ctx, [&] {
    if (!chunk || !bounds) api_fail(DCDF_ERR_BAD_ARG, "null argument");
    const dcdf_cube c = order_cube(*bounds);
    const uint64_t off[2] = {0, (uint64_t)((c.end - c.start) * (c.bottom - c.top) * (c.right - c.left))};
    do_window_batch(ctx, chunk_meta(ctx, chunk), 1, bounds, off, out, out_encoding, mem);
  });
}

int32_t dcdf_chunk_search(dcdf_ctx* ctx, const dcdf_chunk* chunk, const dcdf_cube* bounds, int64_t lower, int64_t upper,
                          int64_t* out_irc, uint64_t cap, uint64_t* n_found, int32_t mem) {
  return guarded(ctx, [&] {
    if (!chunk || !bounds) api_fail(DCDF_ERR_BAD_ARG, "null argument");
    do_search_batch(ctx, chunk_meta(ctx, chunk), 1, bounds, &lower, &upper, nullptr, out_irc, cap, n_found, mem);
  });
}

// ===================================================================================== Superchunk queries
int32_t dcdf_superchunk_get_batch(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const int64_t* irc, void* out,
                                  int32_t out_encoding, int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc) api_fail(DCDF_ERR_BAD_ARG, "null superchunk");
    do_get_batch(ctx, super_meta(ctx, sc), n, irc, out, out_encoding, mem);
  });
}

int32_t dcdf_superchunk_cell_batch(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const int64_t* q, const uint64_t* out_off,
                                   void* out, int32_t out_encoding, int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc) api_fail(DCDF_ERR_BAD_ARG, "null superchunk");
    do_cell_batch(ctx, super_meta(ctx, sc), n, q, out_off, out, out_encoding, mem);
  });
}

int32_t dcdf_superchunk_window(dcdf_ctx* ctx, const dcdf_superchunk* sc, const dcdf_cube* bounds, void* out, int32_t out_encoding,
                               int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc || !bounds) api_fail(DCDF_ERR_BAD_ARG, "null argument");
    const dcdf_cube c = order_cube(*bounds);
    const uint64_t off[2] = {0, (uint64_t)((c.end - c.start) * (c.bottom - c.top) * (c.right - c.left))};
    do_window_batch(ctx, super_meta(ctx, sc), 1, bounds, off, out, out_encoding, mem);
  });
}

int32_t dcdf_superchunk_window_batch(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                     const uint64_t* out_off, void* out, int32_t out_encoding, int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc) api_fail(DCDF_ERR_BAD_ARG, "null superchunk");
    do_window_batch(ctx, super_meta(ctx, sc), n, bounds, out_off, out, out_encoding, mem);
  });
}

int32_t dcdf_superchunk_window_stats(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                     const uint64_t* out_off, uint64_t* count, void* vmin, void* vmax, double* sum, double* sum_sq,
                                     int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc) api_fail(DCDF_ERR_BAD_ARG, "null superchunk");
    do_window_stats(ctx, super_meta(ctx, sc), n, bounds, out_off, count, vmin, vmax, sum, sum_sq, mem);
  });
}

int32_t dcdf_superchunk_time_stats(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                   const uint64_t* out_off, const double* lower, const double* upper, uint64_t* count,
                                   uint64_t* n_band, void* vmin, void* vmax, double* sum, double* sum_sq, int32_t accumulate,
                                   int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc) api_fail(DCDF_ERR_BAD_ARG, "null superchunk");
    do_time_stats(ctx, super_meta(ctx, sc), n, bounds, out_off, lower, upper, count, n_band, vmin, vmax, sum, sum_sq, accumulate, mem);
  });
}

int32_t dcdf_superchunk_search_batch(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                     const int64_t* lower, const int64_t* upper, uint64_t* counts, int64_t* out_irc, uint64_t cap,
                                     uint64_t* n_found, int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc) api_fail(DCDF_ERR_BAD_ARG, "null superchunk");
    do_search_batch(ctx, super_meta(ctx, sc), n, bounds, lower, upper, counts, out_irc, cap, n_found, mem);
  });
}

int32_t dcdf_superchunk_search_values(dcdf_ctx* ctx, const dcdf_superchunk* sc, uint64_t n, const dcdf_cube* bounds,
                                      const double* lower, const double* upper, uint64_t* counts, int64_t* out_irc,
                                      uint64_t cap, uint64_t* n_found, int32_t mem) {
  return guarded(ctx, [&] {
    if (!sc) api_fail(DCDF_ERR_BAD_ARG, "null superchunk");
    do_search_batch(ctx, super_meta(ctx, sc), n, bounds, nullptr, nullptr, counts, out_irc, cap, n_found, mem, true, lower, upper);
  });
}

// ===================================================================================== flat conversions
int32_t dcdf_to_fixed(dcdf_ctx* ctx, const void* in, int32_t encoding, uint64_t n, int32_t fractional_bits, int32_t round,
                      int64_t* out, int32_t mem) {
  return guarded(ctx, [&] {
    if (n == 0) return;
    if (!in || !out) api_fail(DCDF_ERR_BAD_ARG, "null argument");
    if (encoding != DCDF_ENC_F32 && encoding != DCDF_ENC_F64) api_fail(DCDF_ERR_BAD_ARG, "to_fixed needs a float encoding");
    const void* d_in = to_device(ctx, ctx->query_in, in, enc_size(encoding) * n, mem);
    OutTarget ot = out_begin(ctx, out, sizeof(i64) * n, mem);
    ctx->small.reserve(256);
    u32* d_err = ctx->small.as<u32>() + 32;
    CK(cudaMemsetAsync(d_err, 0, 4, ctx->stream));
    const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 32);
    if (encoding == DCDF_ENC_F32) k_to_fixed<float><<<grid, 256, 0, ctx->stream>>>(static_cast<const float*>(d_in), n, fractional_bits, round, static_cast<i64*>(ot.dev), d_err);
    else k_to_fixed<double><<<grid, 256, 0, ctx->stream>>>(static_cast<const double*>(d_in), n, fractional_bits, round, static_cast<i64*>(ot.dev), d_err);
    CK(cudaGetLastError());
    ctx->launches++;
    out_end(ctx, ot);
    check_err_word(ctx, d_err, "to_fixed");
  });
}

int32_t dcdf_from_fixed(dcdf_ctx* ctx, const int64_t* in, uint64_t n, int32_t fractional_bits, void* out, int32_t encoding,
                        int32_t mem) {
  return guarded(ctx, [&] {
    if (n == 0) return;
    if (!in || !out) api_fail(DCDF_ERR_BAD_ARG, "null argument");
    if (encoding != DCDF_ENC_F32 && encoding != DCDF_ENC_F64) api_fail(DCDF_ERR_BAD_ARG, "from_fixed needs a float encoding");
    const i64* d_in = static_cast<const i64*>(to_device(ctx, ctx->query_in, in, sizeof(i64) * n, mem));
    OutTarget ot = out_begin(ctx, out, enc_size(encoding) * n, mem);
    const unsigned grid = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)ctx->sm_count * 32);
    if (encoding == DCDF_ENC_F32) k_from_fixed<float><<<grid, 256, 0, ctx->stream>>>(d_in, n, fractional_bits, static_cast<float*>(ot.dev));
    else k_from_fixed<double><<<grid, 256, 0, ctx->stream>>>(d_in, n, fractional_bits, static_cast<double*>(ot.dev));
    CK(cudaGetLastError());
    ctx->launches++;
    out_end(ctx, ot);
  });
}

}  // extern "C"
