// host.hpp -- host-side plumbing shared by the C-ABI translation units (context, buffers, handles).
#pragma once
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/dcdf_cuda.h"
#include "common.cuh"
#include "encode_tile.cuh"
#include "tree_types.hpp"

namespace dcdf {

struct CudaFail {
  std::string msg;
};
struct ApiFail {
  int32_t code;
  std::string msg;
};

inline void cuda_check(cudaError_t e, const char* what, const char* file, int line) {
  if (e != cudaSuccess) {
    char buf[512];
    snprintf(buf, sizeof buf, "%s failed: %s (%s:%d)", what, cudaGetErrorString(e), file, line);
    throw CudaFail{buf};
  }
}
#define CK(x) ::dcdf::cuda_check((x), #x, __FILE__, __LINE__)
[[noreturn]] inline void api_fail(int32_t code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  throw ApiFail{code, buf};
}

// Grow-only device buffer owned by a context (scratch that survives between calls).
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  void reserve(size_t n) {
    if (n <= cap) return;
    if (p) CK(cudaFree(p));
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 256;
    CK(cudaMalloc(&p, want));
    cap = want;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

// Pinned host staging buffer.
struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  void reserve(size_t n) {
    if (n <= cap) return;
    if (p) CK(cudaFreeHost(p));
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 256;
    CK(cudaMallocHost(&p, want));
    cap = want;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

// Result buffers come from the device's stream-ordered pool (cudaMallocAsync) with an unlimited release
// threshold: cudaMalloc / cudaFree of multi-GB blobs cost hundreds of milliseconds per call on B200.
inline void* pool_alloc(size_t bytes, cudaStream_t st) {
  void* p = nullptr;
  CK(cudaMallocAsync(&p, bytes ? bytes : 16, st));
  return p;
}
inline void pool_free(void* p) {
  if (p) cudaFreeAsync(p, 0);  // callers have synchronized every stream that used p
}

enum { KT_ENCODE = 0, KT_STATS = 1, KT_GATHER = 2, KT_WINDOW = 3, KT_CELL = 4, KT_SEARCH = 5, KT_REDUCE = 6, KT_TIME_STATS = 7, KT_COUNT = 8 };

}  // namespace dcdf

struct dcdf_ctx {
  int device = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t aux_stream = nullptr;  // clipped-tile encode list runs beside the full-tile list
  cudaEvent_t fork_ev = nullptr, join_ev = nullptr;
  std::string last_error;
  uint64_t launches = 0;
  float kernel_ms[dcdf::KT_COUNT] = {0, 0, 0, 0, 0, 0, 0, 0};
  cudaEvent_t ev[2 * dcdf::KT_COUNT] = {};
  int sm_count = 148;
  // dcdf_ctx_set_option (include/dcdf_cuda.h)
  struct Options {
    uint32_t stage_limit = 0xffffffffu;  // encoder: structures above this many bytes are emitted straight into the arena
    int no_fast_encode = 0;              // keep eligible tiles away from the fast-path encoder (k_encode_v5)
    uint32_t cell_tile_min = 64;         // cell series: tiles with at least this many series of a batch are decoded by the tile decoder (0: never)
    int window_cells = 0;                // windows through the 4x4-block walker (the path of trees larger than 64x64)
    int window_wide = 0;                 // 64-bit expansion even when every DAC code fits three bytes
    uint32_t search_share_min = 3;       // value-range search: shared decodes for the counting pass from this many windows per touched (slice, tile) on (0: never)
    int search_dfs = 0;                  // depth-first search kernel instead of the tile search
    int search_no_cache = 0;             // the search's writing pass recomputes instead of reading cached findings
    int trace = 0;                       // host-side phase times of the encode pipeline on stderr (adds stream syncs)
    uint64_t time_stats_scratch = 1ull << 30;  // time statistics: partials per group of slices, in bytes (at least one slice per group)
  } opt;
  uint32_t last_list_counts[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // units per encoder work list of the last build (dcdf_ctx_get_stat)
  uint64_t last_time_groups = 0, last_time_scratch = 0;     // slice groups / partial bytes of the largest group, last time statistics call
  // scratch
  dcdf::DevBuf input_copy, units, ustats, istats, slices, sstate, tbl_scratch, order, pieces, results, stored, chunk_off,
      arena, small, exact, query_in, query_out, query_aux, query_aux2, search_cache, tree_buf;
  dcdf::PinBuf pin, pin2;
  size_t arena_hint = 0;
  // small transfers through mapped pinned memory (xfer.cuh)
  dcdf::PinBuf xfer_up, xfer_down;
  size_t up_off = 0, down_off = 0;
  struct PendingRead { void* dst; size_t off, n; };
  std::vector<PendingRead> reads;
};

// One Chunk resident on the device.  `bytes` may point into a superchunk's blob (owner == false).
struct dcdf_chunk {
  int device = 0;
  uint8_t* bytes = nullptr;
  uint64_t size = 0;
  bool owner = true;
  int64_t shape[3] = {0, 0, 0};
  int32_t encoding = 0, fractional_bits = 0;
  uint32_t n_blocks = 0;
  // decode directory (built lazily / at open): one entry per instant
  void* dir = nullptr;  // device: InstantDir[shape[0]]
  std::vector<uint32_t> block_instants;
};

struct dcdf_superchunk {
  int device = 0;
  int32_t encoding = 0;
  int64_t shape[3] = {0, 0, 0};  // whole array
  int64_t chunk_size = 0;
  struct Slice {
    dcdf_superchunk_info info;
    int64_t t0;
    uint32_t unit_base, n_units;
    uint64_t chunk_blob_off, dac_off[2], dac_size[2];
    uint64_t table_base;
  };
  std::vector<Slice> slices;
  uint32_t n_slots = 0;
  // host mirrors (small)
  std::vector<dcdf::EncUnit> units;
  std::vector<uint8_t> stored;
  std::vector<uint64_t> chunk_off;  // [n_units + 1] into chunk_blob
  std::vector<dcdf::UnitResult> results;
  std::vector<int32_t> slot_unit;   // [n_slices][n_slots] -> unit index or -1 (n_slots = padded leaf grid)
  // static node tree (same geometry for every slice) and per-slice node results
  struct NodeGeom { int64_t top, left, rows, cols, sidelen, chunks_sidelen, subsidelen; uint32_t levels; };
  std::vector<dcdf::TreeNode> nodes;
  std::vector<dcdf::TreeChild> children;
  std::vector<NodeGeom> geom;
  std::vector<dcdf::NodeState> nstate;           // [n_slices][n_nodes]
  std::vector<uint64_t> node_dac_off, node_dac_size;  // [n_slices][n_nodes][2] into dac_blob
  std::vector<int32_t> leaf_unit;                // [leaf_rows][leaf_cols] unit index inside a slice
  int leaf_rows = 0, leaf_cols = 0, leaf_side = 0;
  int64_t leaf_grid = 0;                         // padded leaf tiles per side
  uint64_t tbl_per_instant = 0;
  // device blobs
  uint8_t* chunk_blob = nullptr;
  uint64_t chunk_blob_size = 0;
  uint8_t* dac_blob = nullptr;
  uint64_t dac_blob_size = 0;
  int64_t* tbl_max = nullptr;  // fixed-point max table (values of elided subchunks), all slices
  int64_t* tbl_min = nullptr;
  uint64_t tbl_len = 0;
  void* dir = nullptr;         // device decode directory over all stored units
  void* dev_meta = nullptr;    // device copies of unit / slot tables for the query kernels
  bool opened = false;         // built from stored bytes by dcdf_superchunk_open (validated like Chunk::read_from)
  std::vector<uint8_t> unit_digests;  // SHA2-256 of every stored chunk node, 32 bytes per unit (dcdf_superchunk_save)
};
