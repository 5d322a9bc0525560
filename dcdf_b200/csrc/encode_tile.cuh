// encode_tile.cuh -- the Chunk::build kernel for tiles of side <= 64 (one CTA per Chunk).
//
// Replaces, per (subchunk x time slice) unit, the reference's
//   Chunk::build            chunk.rs:42-96      (heuristic: Snapshot vs Log per instant)
//   Snapshot::build         snapshot.rs:108-156 + K2TreeNode::_build  snapshot.rs:439-500
//   Log::build              log.rs:112-165      + K2PTreeNode::_build log.rs:725-817
//   BitMapBuilder::finish   bitmap.rs:66-113,   Dac::from dac.rs:96-132
//   and the Snapshot / Log / Dac / BitMap serializers (snapshot.rs:48-58, log.rs:53-64, dac.rs:37-44,
//   bitmap.rs:128-138).
//
// Layout of the work inside the CTA (256 threads, k = 2, tree of L <= 6 levels embedded in a 64x64
// frame; the tree root is the frame node at level lo = 6 - L, Morton index 0):
//   * thread t owns the level-4 frame node with Morton index t: a 4x4 block of cells kept in
//     registers in Morton order (cell m = quad (m>>2), child (m&3); row bit above column bit).
//   * levels 6 -> 5 -> 4 of the min/max/equal pyramid are reduced inside the thread, levels 3 and 2 with
//     warp shuffles, levels 1 and 0 through shared memory.
//   * node existence flows top-down (a node exists iff every ancestor is an internal node);
//     BFS output positions come from per-level ballot/popc ranks plus a cross-warp scan.
//   * DAC byte-length histograms of BOTH candidate encodings give their serialized sizes; only the
//     winner is emitted: values are staged in shared memory in BFS order and packed level by level
//     (byte, continuation bitmap, rank directory) with in-place compaction.
//   * each emitted Snapshot/Log is a "piece" in a bump-allocated arena; gather.cuh lays pieces out as
//     the final Chunk bytes.
#pragma once
#include "common.cuh"

namespace dcdf {

constexpr int ENC_THREADS = 256;
constexpr int ENC_WARPS = ENC_THREADS / 32;
constexpr int MAX_NODES = 5461;     // nodes of a 7-level (64x64) quadtree
constexpr int MAX_INTERNAL = 1365;  // nodes above the leaf level
constexpr int NM_WORDS = (MAX_INTERNAL + 31) / 32 + 1;
constexpr int STAGE_BYTES = 16 * 1024;  // structures up to this size are assembled in smem, then bulk-copied

struct EncUnit {
  i64 base;         // element offset of [t0, top, left] in the input array
  int rows, cols;   // in-bounds extent of the tile, 1..64
  int instants;     // 1..  (Block caps logs at 254, any length is fine)
  int bits;         // fractional bits written to the chunk header / used by to_fixed
  int flags;        // UF_*
  int lo;           // 6 - tree levels
  u32 piece_base;   // first entry of this unit in the piece table
  u32 slot;         // caller-defined (subchunk slot inside its slice)
  int row0, col0;   // origin of the tile inside its region (row-major order of the NaN quirk)
  int fmin;         // units of k_encode_v5: the smallest fixed code of the unit (k_finalize_tree); full tiles code cells relative to it
};
enum : int { UF_ROUND = 1, UF_NARROW = 2, UF_SKIP = 4, UF_FULL = 8 /* 64x64, all in bounds */,
              UF_EXACT = 16 /* float unit whose values all have <= bits fractional bits and are finite: to_fixed never rounds */ };

struct Piece {
  u64 off;   // byte offset in the arena (16-byte aligned)
  u32 size;  // serialized size of the Snapshot / Log
  u32 kind;  // 1 = Snapshot (starts a Block), 0 = Log
};

struct UnitResult {
  u64 bytes;       // Chunk::size()  (chunk.rs:269-278)
  u32 snapshots;   // == number of blocks
  u32 logs;
};

struct EncParams {
  const void* data;
  i64 stride_t, stride_r, stride_c;  // element strides
  const EncUnit* units;
  const u32* order;       // unit indices to process (one of the four narrow/wide x full/clipped lists)
  const u32* order_count; // number of valid entries in `order` (device scalar)
  Piece* pieces;
  UnitResult* results;
  u8* arena;
  u64 arena_cap;
  unsigned long long* arena_head;
  u32* err;               // EF_* bits
};

template <typename V>
struct VT;
template <>
struct VT<int32_t> {
  typedef u32 U;
  static constexpr int32_t NONE_MAX = INT32_MIN, NONE_MIN = INT32_MAX;
  static constexpr int MAXLEN = 4;
  static DCDF_DEVINL u32 zz(int32_t v) { return zigzag32(v); }
};
template <>
struct VT<i64> {
  typedef u64 U;
  static constexpr i64 NONE_MAX = INT64_MIN, NONE_MIN = INT64_MAX;
  static constexpr int MAXLEN = 8;
  static DCDF_DEVINL u64 zz(i64 v) { return zigzag64(v); }
};

template <typename V>
DCDF_DEVINL V vmax(V a, V b) { return a > b ? a : b; }
template <typename V>
DCDF_DEVINL V vmin(V a, V b) { return a < b ? a : b; }
template <typename V>
DCDF_DEVINL V shfl(V v, int src) { return __shfl_sync(0xffffffffu, v, src); }
template <typename V>
DCDF_DEVINL V shfl_xor(V v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }

// Upper-level node record shared through smem (levels 2, 1, 0 of the 64x64 frame).
template <typename V>
struct UpNode {
  V tmax, tmin;  // sentinels when None
  V diff;        // log: t - s of the first cell (log.rs:751,781)
  int eq;        // log: K2PTreeNode.equal
};

// Shared-memory plan of the encode CTA.
template <typename V>
struct EncSmem {
  // zigzag codes of `max` in BFS order live at A_raw + 3: BFS indices of sibling groups are 1 (mod 4), so every
  // group of four starts on a 16-byte boundary and is staged with one vector store
  __align__(16) typename VT<V>::U A_raw[MAX_NODES + 7];
  __align__(16) typename VT<V>::U C[MAX_NODES + 7];   // DAC compaction ping-pong partner of A / B
  typename VT<V>::U B[MAX_INTERNAL + 3];   // zigzag codes of `min`
  u8 nmf[MAX_INTERNAL + 3];                // nodemap flags (one byte per node above the leaf level)
  u8 eqf[MAX_INTERNAL + 3];                // equal flags (logs)
  u32 nm[NM_WORDS];                        // packed words, MSB first
  u32 eqw[NM_WORDS];
  UpNode<V> l2[16];
  UpNode<V> l1[4];
  UpNode<V> l0;
  V s_l1max[4], s_l1min[4], s_l0max, s_l0min;  // cached snapshot upper levels (per-thread regs hold l3,l2)
  u32 cntF[2][2][8];                       // fast pass : [candidate 0=snapshot,1=log][0=max,1=min][len > j]
  u32 cntX[2][2][8];                       // exact pass
  u32 strF[2][2];                          // fast pass : [candidate][0 = internal nodes on levels <= 4, 1 = internal quads]
  u32 strX[2][2];
  u32 bigF;                                // fast pass : some quad / leaf entry of the log needs more than 2 bytes
  u32 sel_max[8], sel_min[8];              // histogram of the winner (DAC layout)
  u32 my_size, as_snapshot, go_slow;
  u32 wtot[6][ENC_WARPS];                  // per-warp internal-node counts per level (scan input)
  u32 scan[ENC_WARPS];                     // scratch for the DAC compaction scan
  u64 piece_off;
  __align__(16) u8 stage[STAGE_BYTES];
};

// ---------------------------------------------------------------------------------------------------
// DAC emission (dac.rs:96-132 + dac.rs:37-44 + bitmap.rs:66-113,128-138), block-wide.
// `src` holds n zigzag codes (shared memory), n_j = cntgt[j] = number of codes longer than j bytes.
// Level j is dense: byte = code & 0xff, continuation bit = (code >> 8) != 0.  Each warp owns a contiguous
// run of the level (a multiple of 32 entries): pass 1 counts its survivors, one barrier turns the counts
// into offsets, pass 2 writes bytes / bitmap words / rank directory and compacts the survivors (order
// preserved) into `dst`, which becomes the next level.  Returns bytes written.  All threads must call.
template <typename U, int MAXLEN>
__device__ u32 block_dac_emit(U* src, U* dst, const u32* cntgt, u8* out, u32* scan) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int n_levels = 0;
  for (int j = 0; j < MAXLEN; j++)
    if (cntgt[j] > 0) n_levels = j + 1;
  if (tid == 0) out[0] = (u8)n_levels;
  u32 off = 1;
  for (int j = 0; j < n_levels; j++) {
    const u32 nj = cntgt[j];
    const u32 blocks = nj / 128u, words = (nj + 31u) / 32u;
    u8* p_len = out + off;
    u8* p_index = p_len + 8;
    u8* p_words = p_index + 4 * blocks;
    u8* p_bytes = p_words + 4 * words;
    if (tid == 0) {
      store_be32(p_len, nj);
      store_be32(p_len + 4, 4u);  // k = 4 (bitmap.rs:69)
    }
    const u32 seg = ((nj + 32u * ENC_WARPS - 1u) / (32u * ENC_WARPS)) * 32u;
    const u32 i_lo = min(nj, warp * seg), i_hi = min(nj, i_lo + seg);
    u32 cnt = 0;
    for (u32 i0 = i_lo; i0 < i_hi; i0 += 32u) {
      const u32 i = i0 + lane;
      cnt += __popc(__ballot_sync(0xffffffffu, i < nj && (src[i] >> 8) != 0));
    }
    if (lane == 0) scan[warp] = cnt;
    __syncthreads();
    u32 pre = 0;
#pragma unroll
    for (int w = 0; w < ENC_WARPS; w++) pre += w < warp ? scan[w] : 0u;
    for (u32 i0 = i_lo; i0 < i_hi; i0 += 32u) {
      const u32 i = i0 + lane;
      const U v = i < nj ? src[i] : (U)0;
      const bool more = (v >> 8) != 0;
      const u32 bal = __ballot_sync(0xffffffffu, more);
      if (i < nj) p_bytes[i] = (u8)(v & 0xff);
      if (more) dst[pre + __popc(bal & lanemask_lt())] = (U)(v >> 8);
      pre += __popc(bal);
      if (lane == 0) {
        store_be32(p_words + 4 * (i0 >> 5), __brev(bal));
        // rank directory: index[b] = ones in bits [0, 128(b+1))  (bitmap.rs:97-104)
        if (((i0 + 32u) & 127u) == 0 && (i0 + 32u) <= nj) store_be32(p_index + 4 * ((i0 + 32u) / 128u - 1u), pre);
      }
    }
    __syncthreads();  // next level complete in dst; scan[] reusable
    U* t = src; src = dst; dst = t;
    off += 8 + 4 * blocks + 4 * words + nj;
  }
  return off;
}

__host__ __device__ inline u32 dac_size_from_counts(const u32* cntgt, int maxlen) {
  u32 s = 1;
  for (int j = 0; j < maxlen; j++)
    if (cntgt[j] > 0) s += bitmap_size(cntgt[j]) + cntgt[j];
  return s;
}

// BitMap serialization (bitmap.rs:66-113,128-138) from one flag byte per bit; block-wide.  `words_smem`
// receives the MSB-first words (ballot + brev), from which the rank directory is summed.
__device__ inline u32 block_bitmap_emit(const u8* flags, u32* words_smem, u32 length, u8* out) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u32 blocks = length / 128u, words = (length + 31u) / 32u;
  for (u32 w = warp; w < words; w += ENC_WARPS) {
    const u32 i = 32u * w + lane;
    const u32 bal = __ballot_sync(0xffffffffu, i < length && flags[i] != 0);
    if (lane == 0) {
      const u32 word = __brev(bal);
      words_smem[w] = word;
      store_be32(out + 8 + 4 * blocks + 4 * w, word);
    }
  }
  if (tid == 0) {
    store_be32(out, length);
    store_be32(out + 4, 4u);
  }
  if (blocks) {
    __syncthreads();
    for (u32 b = tid; b < blocks; b += ENC_THREADS) {
      u32 c = 0;
      for (u32 w = 0; w < 4 * (b + 1); w++) c += __popc(words_smem[w]);
      store_be32(out + 8 + 4 * b, c);
    }
  }
  return 8 + 4 * blocks + 4 * words;
}

// ---------------------------------------------------------------------------------------------------
// Tile loader: thread t reads its 4x4 block (Morton order) of instant `p`.
template <typename InT>
DCDF_DEVINL void load_block(const InT* p, i64 sr, i64 sc, int rows, int cols, int r0, int c0, InT out[16], u32& inb) {
  inb = 0;
  const bool full = (r0 + 4 <= rows) && (c0 + 4 <= cols);
  if (full && sc == 1 && sizeof(InT) == 4 && ((((uintptr_t)(p + (i64)r0 * sr + c0)) | ((uintptr_t)(sr * (i64)sizeof(InT)))) & 15) == 0) {
    inb = 0xffffu;
#pragma unroll
    for (int rr = 0; rr < 4; rr++) {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(p + (i64)(r0 + rr) * sr + c0));
      const u32 w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int cc = 0; cc < 4; cc++) {
        const int m = ((rr >> 1) << 3) | ((cc >> 1) << 2) | ((rr & 1) << 1) | (cc & 1);
        out[m] = *reinterpret_cast<const InT*>(&w[cc]);
      }
    }
    return;
  }
#pragma unroll
  for (int rr = 0; rr < 4; rr++) {
#pragma unroll
    for (int cc = 0; cc < 4; cc++) {
      const int m = ((rr >> 1) << 3) | ((cc >> 1) << 2) | ((rr & 1) << 1) | (cc & 1);
      const bool in = (r0 + rr < rows) && (c0 + cc < cols);
      out[m] = in ? __ldg(p + (i64)(r0 + rr) * sr + (i64)(c0 + cc) * sc) : InT(0);
      inb |= in ? (1u << m) : 0u;
    }
  }
}

// Packed per-thread histogram: field j (8 bits) counts entries longer than j bytes.
template <typename V>
struct Hist;
template <>
struct Hist<int32_t> {
  u32 h = 0;
  DCDF_DEVINL void add(u32 zz) { h += 0x01010101u >> (32 - 8 * dac_len(zz)); }
  DCDF_DEVINL u32 field(int j) const { return (h >> (8 * j)) & 0xffu; }
};
template <>
struct Hist<i64> {
  u64 h = 0;
  DCDF_DEVINL void add(u64 zz) { h += 0x0101010101010101ull >> (64 - 8 * dac_len(zz)); }
  DCDF_DEVINL u32 field(int j) const { return (u32)(h >> (8 * j)) & 0xffu; }
};

// Block-reduce a histogram into smem counters cnt[0 .. MAXLEN) (two 16-bit fields per redux).
template <typename V>
DCDF_DEVINL void reduce_hist(const Hist<V>& h, u32* cnt) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < VT<V>::MAXLEN; j += 2) {
    u32 packed = h.field(j) | (h.field(j + 1) << 16);
    u32 r = __reduce_add_sync(0xffffffffu, packed);
    if (lane == 0 && r) {
      if (r & 0xffffu) atomicAdd(&cnt[j], r & 0xffffu);
      if (r >> 16) atomicAdd(&cnt[j + 1], r >> 16);
    }
  }
}

// Cheap exact accounting for entries known to be short: with m = v ^ (v >> sign) the zigzag code is 2m or
// 2m+1, so the code needs more than one byte iff m >= 128 and more than two iff m >= 32768.
template <typename V>
struct FastAcc {
  typedef typename VT<V>::U U;
  u32 c1 = 0;  // entries longer than one byte
  U big = 0;   // OR of all m (>= 32768 <=> some entry is longer than two bytes)
  DCDF_DEVINL void add(V v) {
    const U m = (U)(v ^ (v >> (8 * (int)sizeof(V) - 1)));
    c1 += m > (U)127 ? 1u : 0u;
    big |= m;
  }
};

// Snapshot / Log serialization from the staged smem arrays into `out` (smem stage or arena); block-wide.
template <typename V>
__device__ __forceinline__ u32 serialize_structure(EncSmem<V>& S, u8* out, const EncUnit& unit, int lo, bool as_snapshot,
                                                   u32 nm_len, u32 n_min) {
  typedef typename VT<V>::U U;
  if (threadIdx.x == 0) {
    out[0] = 2;  // k
    store_be32(out + 1, (u32)unit.rows);
    store_be32(out + 5, (u32)unit.cols);
    store_be32(out + 9, 64u >> lo);  // sidelen
  }
  u32 off = 13;
  off += block_bitmap_emit(S.nmf, S.nm, nm_len, out + off);
  if (!as_snapshot) off += block_bitmap_emit(S.eqf, S.eqw, nm_len - n_min, out + off);
  off += block_dac_emit<U, VT<V>::MAXLEN>(S.A_raw + 3, S.C, S.sel_max, out + off, S.scan);
  __syncthreads();  // C is reused by the min DAC
  off += block_dac_emit<U, VT<V>::MAXLEN>(S.B, S.C, S.sel_min, out + off, S.scan);
  return off;
}

// Conversion of one input cell to the kernel's value type.  The narrow (int32) path is only selected when
// the stats pass proved |fixed| < 2^30 and the unit has no +-inf, so range checks are dropped there.
template <typename InT, typename V>
struct CellConv {
  static DCDF_DEVINL V get(InT v, int bits, bool round, u32& err) { return (V)Conv<InT>::get(v, bits, round, err); }
};
template <>
struct CellConv<float, int32_t> {
  static DCDF_DEVINL int32_t get(float n, int bits, bool round, u32& err) {
    float shifted = n * (float)((i64)1 << bits);
    const float tr = truncf(shifted);
    if (shifted - tr > 0.0f) {  // fixed.rs:47
      if (round) shifted = roundf(shifted);
      else err |= EF_PRECISION;
    }
    const int32_t f = __float2int_rz(shifted * 2.0f) + 1;
    return n != n ? 0 : f;  // NaN -> 0 (fixed.rs:35-37)
  }
};

// ---------------------------------------------------------------------------------------------------
// MINB: min resident CTAs per SM the register allocator must allow.
template <typename InT, typename V, bool FULL, int MINB>
__global__ void __launch_bounds__(ENC_THREADS, MINB) k_encode_tiles(const EncParams P) {
  typedef typename VT<V>::U U;
  constexpr int MAXLEN = VT<V>::MAXLEN;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  EncSmem<V>& S = *reinterpret_cast<EncSmem<V>*>(smem_raw);

  if (blockIdx.x >= *P.order_count) return;
  const u32 unit_idx = P.order[blockIdx.x];
  const EncUnit unit = P.units[unit_idx];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lo = FULL ? 0 : unit.lo;
  const bool do_round = unit.flags & UF_ROUND;
  const int r0 = 4 * (int)morton_row(tid), c0 = 4 * (int)morton_col(tid);
  const InT* base = static_cast<const InT*>(P.data) + unit.base;

  // tree membership of this thread's frame nodes (tree root = frame node (lo, 0))
  const bool intree4 = FULL ? true : (lo <= 4 ? ((tid >> (8 - 2 * lo)) == 0) : (tid == 0));
  const u32 quad_mask = (FULL || lo <= 4) ? 0xfu : 0x1u;  // lo == 5: only quad 0 of thread 0 is in the tree
  const bool owner[5] = {tid == 0, (tid & 63) == 0, (tid & 15) == 0, (tid & 3) == 0, true};

  u32 err = 0;
  // cached snapshot (reference instant of the current block): leaves + own level-3 / level-2 ancestors
  V sv[16];
#pragma unroll
  for (int m = 0; m < 16; m++) sv[m] = 0;
  V s3max = 0, s3min = 0, s2max = 0, s2min = 0;
  u32 n_logs = 0, n_snap = 0, n_log_total = 0;
  u64 total_bytes = 0;

  InT raw[16];
  u32 inb;
  load_block<InT>(base, P.stride_r, P.stride_c, unit.rows, unit.cols, r0, c0, raw, inb);

  for (int inst = 0; inst < unit.instants; inst++) {
    // ---------------- convert (a3) and prefetch the next instant
    V tv[16];
#pragma unroll
    for (int m = 0; m < 16; m++) tv[m] = CellConv<InT, V>::get(raw[m], unit.bits, do_round, err);
    const u32 cur_inb = FULL ? 0xffffu : inb;
    if (inst + 1 < unit.instants)
      load_block<InT>(base + (i64)(inst + 1) * P.stride_t, P.stride_r, P.stride_c, unit.rows, unit.cols, r0, c0, raw, inb);
    const bool first = inst == 0;
#define CELL_IN(m) (FULL || ((cur_inb >> (m)) & 1u))

    // ---------------- bottom-up pyramid inside the thread: levels 6 -> 5 -> 4
    V t5max[4], t5min[4];
    V d0[4];        // diff of the first cell of each quad (log)
    u32 eq5 = 0;    // bit q: all four leaf diffs of quad q equal
#pragma unroll
    for (int q = 0; q < 4; q++) {
      V mx = VT<V>::NONE_MAX, mn = VT<V>::NONE_MIN;
      V dq[4];
#pragma unroll
      for (int c = 0; c < 4; c++) {
        const int m = 4 * q + c;
        const bool in = CELL_IN(m);
        if (in) { mx = vmax(mx, tv[m]); mn = vmin(mn, tv[m]); }
        dq[c] = (in && !first) ? (V)(tv[m] - sv[m]) : (V)0;  // OOB diff = 0 (log.rs:751)
      }
      t5max[q] = mx; t5min[q] = mn;
      d0[q] = dq[0];
      if (dq[1] == dq[0] && dq[2] == dq[0] && dq[3] == dq[0]) eq5 |= 1u << q;
    }
    const V t4max = vmax(vmax(t5max[0], t5max[1]), vmax(t5max[2], t5max[3]));
    const V t4min = vmin(vmin(t5min[0], t5min[1]), vmin(t5min[2], t5min[3]));
    const V diff4 = d0[0];
    const bool eq4 = eq5 == 0xfu && d0[1] == d0[0] && d0[2] == d0[0] && d0[3] == d0[0];

    // ---------------- levels 3 and 2 with shuffles (4 resp. 16 consecutive lanes)
    V t3max = vmax(t4max, shfl_xor(t4max, 1)); t3max = vmax(t3max, shfl_xor(t3max, 2));
    V t3min = vmin(t4min, shfl_xor(t4min, 1)); t3min = vmin(t3min, shfl_xor(t3min, 2));
    const V diff3 = shfl(diff4, lane & ~3);
    const u32 ok3 = __ballot_sync(0xffffffffu, eq4 && diff4 == diff3);
    const bool eq3 = ((ok3 >> (lane & ~3)) & 0xfu) == 0xfu;
    V t2max = vmax(t3max, shfl_xor(t3max, 4)); t2max = vmax(t2max, shfl_xor(t2max, 8));
    V t2min = vmin(t3min, shfl_xor(t3min, 4)); t2min = vmin(t2min, shfl_xor(t2min, 8));
    const V diff2 = shfl(diff3, lane & ~15);
    const u32 ok2 = __ballot_sync(0xffffffffu, eq3 && diff3 == diff2);
    const bool eq2 = ((ok2 >> (lane & ~15)) & 0xffffu) == 0xffffu;

    // ---------------- levels 1 and 0 through smem; counters and bit staging are reset meanwhile
    if ((lane & 15) == 0) {
      UpNode<V> n;
      n.tmax = t2max; n.tmin = t2min; n.diff = diff2; n.eq = eq2;
      S.l2[tid >> 4] = n;
    }
    if (tid < 32) { (&S.cntF[0][0][0])[tid] = 0; (&S.cntX[0][0][0])[tid] = 0; }
    if (tid < 4) { (&S.strF[0][0])[tid] = 0; (&S.strX[0][0])[tid] = 0; }
    if (tid == 0) S.bigF = 0;
    __syncthreads();
    if (tid < 4) {
      const UpNode<V> a = S.l2[4 * tid], b = S.l2[4 * tid + 1], c = S.l2[4 * tid + 2], d = S.l2[4 * tid + 3];
      UpNode<V> n;
      n.tmax = vmax(vmax(a.tmax, b.tmax), vmax(c.tmax, d.tmax));
      n.tmin = vmin(vmin(a.tmin, b.tmin), vmin(c.tmin, d.tmin));
      n.diff = a.diff;
      n.eq = a.eq && b.eq && c.eq && d.eq && b.diff == a.diff && c.diff == a.diff && d.diff == a.diff;
      S.l1[tid] = n;
    }
    __syncthreads();
    if (tid == 0) {
      const UpNode<V> a = S.l1[0], b = S.l1[1], c = S.l1[2], d = S.l1[3];
      UpNode<V> n;
      n.tmax = vmax(vmax(a.tmax, b.tmax), vmax(c.tmax, d.tmax));
      n.tmin = vmin(vmin(a.tmin, b.tmin), vmin(c.tmin, d.tmin));
      n.diff = a.diff;
      n.eq = a.eq && b.eq && c.eq && d.eq && b.diff == a.diff && c.diff == a.diff && d.diff == a.diff;
      S.l0 = n;
    }
    __syncthreads();
    const UpNode<V> N1 = S.l1[tid >> 6];
    const UpNode<V> N0 = S.l0;
    // snapshot upper levels (reference instant) for this thread's ancestors
    const V s1max = S.s_l1max[tid >> 6], s1min = S.s_l1min[tid >> 6], s0max = S.s_l0max, s0min = S.s_l0min;

    // ---------------- per-node classification for this thread's chain (levels 0..4) and its quads
    // U = "uniform in t" (min_t == max_t as Options; a None node is uniform)   snapshot.rs:133, log.rs:137
    auto uniform = [](V mx, V mn) { return mx == VT<V>::NONE_MAX || mx == mn; };
    const bool u0 = uniform(N0.tmax, N0.tmin), u1 = uniform(N1.tmax, N1.tmin), u2 = uniform(t2max, t2min),
               u3 = uniform(t3max, t3min), u4 = uniform(t4max, t4min);
    u32 u5 = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) u5 |= uniform(t5max[q], t5min[q]) ? (1u << q) : 0u;
    // internal flags: snapshot = !U ; log = !U && !equal
    const bool si[5] = {!u0, !u1, !u2, !u3, !u4};
    const bool li[5] = {!u0 && !N0.eq, !u1 && !N1.eq, !u2 && !eq2, !u3 && !eq3, !u4 && !eq4};
    const u32 si5 = ~u5 & 0xfu, li5 = ~u5 & ~eq5 & 0xfu;
    auto or0 = [](V v, V none) { return v == none ? (V)0 : v; };
    const V cmax[5] = {N0.tmax, N1.tmax, t2max, t3max, t4max};
    const V cmin[5] = {N0.tmin, N1.tmin, t2min, t3min, t4min};

    // snapshot pyramid levels 5/4 of the reference instant, recomputed from the cached leaves
    V s5max[4], s5min[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
      V mx = VT<V>::NONE_MAX, mn = VT<V>::NONE_MIN;
#pragma unroll
      for (int c = 0; c < 4; c++)
        if (CELL_IN(4 * q + c)) { mx = vmax(mx, sv[4 * q + c]); mn = vmin(mn, sv[4 * q + c]); }
      s5max[q] = mx; s5min[q] = mn;
    }
    const V s4max = vmax(vmax(s5max[0], s5max[1]), vmax(s5max[2], s5max[3]));
    const V s4min = vmin(vmin(s5min[0], s5min[1]), vmin(s5min[2], s5min[3]));
    const V csmax[5] = {s0max, s1max, s2max, s3max, s4max};
    const V csmin[5] = {s0min, s1min, s2min, s3min, s4min};

    // alive chains: al_s[l] / al_l[l] = this thread's level-l frame node exists in the snapshot / log tree
    bool al_s[6], al_l[6];
    {
      bool a = intree4 || lo == 5, b = a;
#pragma unroll
      for (int l = 0; l < 5; l++) {
        al_s[l] = l >= lo && a && intree4;
        al_l[l] = l >= lo && b && intree4;
        if (l >= lo) { a = a && si[l]; b = b && li[l]; }
      }
      al_s[5] = (!FULL && lo == 5) ? (tid == 0) : a;
      al_l[5] = (!FULL && lo == 5) ? (tid == 0) : b;
    }
    // structure counts: internal nodes owned on levels <= 4, internal quads
    u32 sup = 0, lup = 0;
#pragma unroll
    for (int l = 0; l < 5; l++) {
      sup += (owner[l] && al_s[l] && si[l]) ? 1u : 0u;
      lup += (owner[l] && al_l[l] && li[l]) ? 1u : 0u;
    }
    const u32 s5c = al_s[5] ? __popc(si5 & quad_mask) : 0u, l5c = al_l[5] ? __popc(li5 & quad_mask) : 0u;

    // ---------------- FAST pass: exact size of the Log, lower bound of the Snapshot (chunk.rs:62)
    bool slow = first || n_logs == 254u;
    if (!slow) {
      Hist<V> hmax, hmin;        // chain entries (levels lo..4): exact
      FastAcc<V> fmax, fmin;     // quads and leaves: short-entry accounting
#pragma unroll
      for (int l = 0; l < 5; l++) {
        if (l < lo || !(owner[l] && al_l[l])) continue;
        hmax.add(VT<V>::zz((V)(or0(cmax[l], VT<V>::NONE_MAX) - or0(csmax[l], VT<V>::NONE_MAX))));
        if (li[l]) hmin.add(VT<V>::zz((V)(cmin[l] - csmin[l])));
      }
      if (al_l[5]) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
          if (!FULL && !((quad_mask >> q) & 1u)) continue;
          fmax.add((V)(or0(t5max[q], VT<V>::NONE_MAX) - or0(s5max[q], VT<V>::NONE_MAX)));
          if ((li5 >> q) & 1u) {
            fmin.add((V)(t5min[q] - s5min[q]));
#pragma unroll
            for (int c = 0; c < 4; c++) {
              const int m = 4 * q + c;
              fmax.add(CELL_IN(m) ? (V)(tv[m] - sv[m]) : (V)0);
            }
          }
        }
      }
      // block reduction (16-bit fields; per-warp sums stay far below 65536)
      {
        u32 r = __reduce_add_sync(0xffffffffu, fmax.c1 | (fmin.c1 << 16));
        if (lane == 0 && r) {
          if (r & 0xffffu) atomicAdd(&S.cntF[1][0][1], r & 0xffffu);
          if (r >> 16) atomicAdd(&S.cntF[1][1][1], r >> 16);
        }
        r = __reduce_add_sync(0xffffffffu, lup | (l5c << 8) | (sup << 16) | (s5c << 24));  // <= 5 / 4 per thread
        if (lane == 0 && r) {
          atomicAdd(&S.strF[1][0], r & 0xffu);
          atomicAdd(&S.strF[1][1], (r >> 8) & 0xffu);
          atomicAdd(&S.strF[0][0], (r >> 16) & 0xffu);
          atomicAdd(&S.strF[0][1], r >> 24);
        }
        const u32 big = __reduce_or_sync(0xffffffffu, (u32)(((fmax.big | fmin.big) >> 15) != 0));
        if (lane == 0 && big) S.bigF = 1;
        if (__any_sync(0xffffffffu, (hmax.h | hmin.h) != 0)) {  // only owner lanes carry chain entries
          reduce_hist<V>(hmax, S.cntF[1][0]);
          reduce_hist<V>(hmin, S.cntF[1][1]);
        }
      }
      __syncthreads();
      if (tid == 0) {
        // n_min = internal nodes, nm_len = 1 + 4 * internal(levels <= 4), n_max = 1 + 4 * internal(all)
        const u32 l_int = S.strF[1][0] + S.strF[1][1], s_int = S.strF[0][0] + S.strF[0][1];
        const u32 l_nm = 1u + 4u * S.strF[1][0], s_nm = 1u + 4u * S.strF[0][0];
        const u32 l_nmax = 1u + 4u * l_int, s_nmax = 1u + 4u * s_int;
        u32 cm[8], cn[8];
#pragma unroll
        for (int j = 0; j < 8; j++) { cm[j] = S.cntF[1][0][j]; cn[j] = S.cntF[1][1][j]; }
        cm[0] = l_nmax; cn[0] = l_int;
        const u32 log_size = 13u + bitmap_size(l_nm) + bitmap_size(l_nm - l_int) + dac_size_from_counts(cm, 8) + dac_size_from_counts(cn, 8);
        // every snapshot entry takes at least one byte
        const u32 snap_lb = 13u + bitmap_size(s_nm) + 1u + bitmap_size(s_nmax) + s_nmax + (s_int ? 1u + bitmap_size(s_int) + s_int : 1u);
        const bool go_slow = S.bigF || snap_lb <= log_size;
        S.go_slow = go_slow;
        if (!go_slow) {
#pragma unroll
          for (int j = 0; j < 8; j++) { S.sel_max[j] = cm[j]; S.sel_min[j] = cn[j]; }
          S.my_size = log_size;
          S.as_snapshot = 0;
          const u64 need = ((u64)log_size + 15ull) & ~15ull;
          const u64 off = atomicAdd(P.arena_head, (unsigned long long)need);
          S.piece_off = off;
          Piece pc;
          pc.off = off; pc.size = log_size; pc.kind = 0u;
          P.pieces[unit.piece_base + inst] = pc;
        }
      }
      __syncthreads();
      slow = S.go_slow;
    }

    // ---------------- EXACT pass (first instant, 254-log cap, near ties, long entries): both candidates
    if (slow) {
      Hist<V> hsmax, hsmin, hlmax, hlmin;
#pragma unroll
      for (int l = 0; l < 5; l++) {
        if (l < lo || !owner[l]) continue;
        const V tm = or0(cmax[l], VT<V>::NONE_MAX);
        const V pmax = cmax[l > 0 ? l - 1 : 0], pmin = cmin[l > 0 ? l - 1 : 0];  // parent (unused at the root)
        if (al_s[l]) {
          hsmax.add(VT<V>::zz(l == lo ? tm : (V)(pmax - tm)));
          if (si[l]) hsmin.add(VT<V>::zz(l == lo ? cmin[l] : (V)(cmin[l] - pmin)));
        }
        if (!first && al_l[l]) {
          hlmax.add(VT<V>::zz((V)(tm - or0(csmax[l], VT<V>::NONE_MAX))));
          if (li[l]) hlmin.add(VT<V>::zz((V)(cmin[l] - csmin[l])));
        }
      }
#pragma unroll
      for (int q = 0; q < 4; q++) {
        if (!FULL && !((quad_mask >> q) & 1u)) continue;
        const V tm = or0(t5max[q], VT<V>::NONE_MAX);
        if (al_s[5]) {
          hsmax.add(VT<V>::zz((!FULL && lo == 5) ? tm : (V)(t4max - tm)));
          if ((si5 >> q) & 1u) {
            hsmin.add(VT<V>::zz((!FULL && lo == 5) ? t5min[q] : (V)(t5min[q] - t4min)));
#pragma unroll
            for (int c = 0; c < 4; c++) {
              const int m = 4 * q + c;
              hsmax.add(VT<V>::zz((V)(t5max[q] - (CELL_IN(m) ? tv[m] : (V)0))));
            }
          }
        }
        if (!first && al_l[5]) {
          hlmax.add(VT<V>::zz((V)(tm - or0(s5max[q], VT<V>::NONE_MAX))));
          if ((li5 >> q) & 1u) {
            hlmin.add(VT<V>::zz((V)(t5min[q] - s5min[q])));
#pragma unroll
            for (int c = 0; c < 4; c++) {
              const int m = 4 * q + c;
              hlmax.add(VT<V>::zz(CELL_IN(m) ? (V)(tv[m] - sv[m]) : (V)0));
            }
          }
        }
      }
      reduce_hist<V>(hsmax, S.cntX[0][0]);
      reduce_hist<V>(hsmin, S.cntX[0][1]);
      if (!first) {
        reduce_hist<V>(hlmax, S.cntX[1][0]);
        reduce_hist<V>(hlmin, S.cntX[1][1]);
      }
      {
        const u32 r = __reduce_add_sync(0xffffffffu, lup | (sup << 16));
        if (lane == 0 && r) {
          atomicAdd(&S.strX[1][0], r & 0xffffu);
          atomicAdd(&S.strX[0][0], r >> 16);
        }
      }
      __syncthreads();
      if (tid == 0) {
        u32 sm[8], sn[8], lm[8], ln[8];
#pragma unroll
        for (int j = 0; j < 8; j++) { sm[j] = S.cntX[0][0][j]; sn[j] = S.cntX[0][1][j]; lm[j] = S.cntX[1][0][j]; ln[j] = S.cntX[1][1][j]; }
        const u32 s_nm = 1u + 4u * S.strX[0][0], l_nm = 1u + 4u * S.strX[1][0];
        const u32 snap_size = 13u + bitmap_size(s_nm) + dac_size_from_counts(sm, 8) + dac_size_from_counts(sn, 8);
        const u32 log_size = 13u + bitmap_size(l_nm) + bitmap_size(l_nm - ln[0]) + dac_size_from_counts(lm, 8) + dac_size_from_counts(ln, 8);
        const bool snap = first || n_logs == 254u || snap_size <= log_size;  // chunk.rs:62
        const u32 size = snap ? snap_size : log_size;
#pragma unroll
        for (int j = 0; j < 8; j++) { S.sel_max[j] = snap ? sm[j] : lm[j]; S.sel_min[j] = snap ? sn[j] : ln[j]; }
        S.my_size = size;
        S.as_snapshot = snap;
        const u64 need = ((u64)size + 15ull) & ~15ull;
        const u64 off = atomicAdd(P.arena_head, (unsigned long long)need);
        S.piece_off = off;
        Piece pc;
        pc.off = off; pc.size = size; pc.kind = snap ? 1u : 0u;
        P.pieces[unit.piece_base + inst] = pc;
      }
      __syncthreads();
    }
    const bool as_snapshot = S.as_snapshot != 0;
    const u32 my_size = S.my_size;
    const u64 piece_off = S.piece_off;
    const bool fits = piece_off + (((u64)my_size + 15ull) & ~15ull) <= P.arena_cap;
    if (!fits) err |= EF_ARENA_FULL;

    // ---------------- BFS positions of the winner: per-level ranks of internal nodes
    bool in_[5], al[6];
#pragma unroll
    for (int l = 0; l < 5; l++) { in_[l] = as_snapshot ? si[l] : li[l]; al[l] = as_snapshot ? al_s[l] : al_l[l]; }
    al[5] = as_snapshot ? al_s[5] : al_l[5];
    const u32 in5 = as_snapshot ? si5 : li5;
    u32 rank_in_warp[5];
    rank_in_warp[0] = 0;
#pragma unroll
    for (int l = 1; l < 5; l++) {
      const bool f = owner[l] && al[l] && in_[l];
      const u32 b = __ballot_sync(0xffffffffu, f);
      rank_in_warp[l] = __popc(b & lanemask_lt());
      if (lane == 0) S.wtot[l][warp] = __popc(b);
    }
    u32 q_before = 0;
    {
      const u32 mine = al[5] ? (in5 & quad_mask) : 0u;
      u32 tot = 0;
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const u32 b = __ballot_sync(0xffffffffu, (mine >> q) & 1u);
        q_before += __popc(b & lanemask_lt());
        tot += __popc(b);
      }
      if (lane == 0) S.wtot[5][warp] = tot;
    }
    __syncthreads();
    u32 I[6], Rbase[6];  // I[l]: internal nodes at level l; Rbase[l]: internal nodes at level l in earlier warps
    I[0] = (lo == 0 && in_[0]) ? 1u : 0u;  // the root flag is uniform across the CTA
    Rbase[0] = 0;
#pragma unroll
    for (int l = 1; l < 6; l++) {
      u32 tot = 0, bs = 0;
#pragma unroll
      for (int w = 0; w < ENC_WARPS; w++) {
        const u32 x = S.wtot[l][w];
        if (w < warp) bs += x;
        tot += x;
      }
      I[l] = tot; Rbase[l] = bs;
    }
    // Pn[l]: BFS index of the first level-l node; Mn[l]: internal nodes on levels above l
    u32 Pn[8], Mn[8];
    {
      u32 p = 0, mm = 0, e = 1;  // e = nodes on the current level
#pragma unroll
      for (int l = 0; l <= 6; l++) {
        Pn[l] = p; Mn[l] = mm;
        if (l < lo) continue;
        p += e;
        const u32 il = l < 6 ? I[l] : 0u;
        mm += il;
        e = 4 * il;
      }
      Pn[7] = p; Mn[7] = mm;
    }
    const u32 n_min = Mn[6], nm_len = Pn[6];
    // rank (among internal nodes of its level) of each chain node, as seen by this thread
    u32 R[5];
    R[0] = 0;
    {
      u32 r1 = 0;  // level-1 owners are lane 0 of warps 0, 2, 4, 6
      for (int w = 0; w < (tid >> 6) * 2; w++) r1 += S.wtot[1][w];
      R[1] = r1;
      R[2] = shfl(Rbase[2] + rank_in_warp[2], lane & ~15);
      R[3] = shfl(Rbase[3] + rank_in_warp[3], lane & ~3);
      R[4] = Rbase[4] + rank_in_warp[4];
    }
    const u32 R5 = Rbase[5] + q_before;  // rank of this thread's first internal quad

    // ---------------- stage values / bits in BFS order
    U* const A = S.A_raw + 3;
#pragma unroll
    for (int l = 0; l < 5; l++) {
      if (l < lo || !(owner[l] && al[l])) continue;
      const u32 child = l == 0 ? 0u : ((u32)(tid >> (2 * (4 - l))) & 3u);
      const u32 pos = l == lo ? 0u : Pn[l] + 4u * R[l > 0 ? l - 1 : 0] + child;
      const V tm = or0(cmax[l], VT<V>::NONE_MAX);
      const V pmax = cmax[l > 0 ? l - 1 : 0], pmin = cmin[l > 0 ? l - 1 : 0];
      V e;
      if (as_snapshot) e = l == lo ? tm : (V)(pmax - tm);
      else e = (V)(tm - or0(csmax[l], VT<V>::NONE_MAX));
      A[pos] = VT<V>::zz(e);
      const u32 ones_before = Mn[l] + R[l];
      S.nmf[pos] = in_[l] ? 1 : 0;
      if (in_[l]) {
        V mv;
        if (as_snapshot) mv = l == lo ? cmin[l] : (V)(cmin[l] - pmin);
        else mv = (V)(cmin[l] - csmin[l]);
        S.B[ones_before] = VT<V>::zz(mv);
      } else if (!as_snapshot) {
        const bool eqf = l == 0 ? (bool)N0.eq : l == 1 ? (bool)N1.eq : l == 2 ? eq2 : l == 3 ? eq3 : eq4;
        const bool un = l == 0 ? u0 : l == 1 ? u1 : l == 2 ? u2 : l == 3 ? u3 : u4;
        S.eqf[pos - ones_before] = (!un && eqf) ? 1 : 0;
      }
    }
    if (al[5]) {
      u32 r5 = R5;
      const bool root5 = !FULL && lo == 5;
      U qe[4];  // the four level-5 entries of this thread (one sibling group)
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const V tm = or0(t5max[q], VT<V>::NONE_MAX);
        V e;
        if (as_snapshot) e = root5 ? tm : (V)(t4max - tm);
        else e = (V)(tm - or0(s5max[q], VT<V>::NONE_MAX));
        qe[q] = VT<V>::zz(e);
      }
      const u32 qpos = root5 ? 0u : Pn[5] + 4u * R[4];
      if (!root5) {
        if (sizeof(U) == 4) *reinterpret_cast<uint4*>(&A[qpos]) = make_uint4((u32)qe[0], (u32)qe[1], (u32)qe[2], (u32)qe[3]);
        else { A[qpos] = qe[0]; A[qpos + 1] = qe[1]; A[qpos + 2] = qe[2]; A[qpos + 3] = qe[3]; }
      } else {
        A[0] = qe[0];
      }
#pragma unroll
      for (int q = 0; q < 4; q++) {
        if (!FULL && !((quad_mask >> q) & 1u)) continue;
        const u32 pos = qpos + (u32)q;
        const u32 ones_before = Mn[5] + r5;
        const bool inq = (in5 >> q) & 1u;
        S.nmf[pos] = inq ? 1 : 0;
        if (inq) {
          V mv;
          if (as_snapshot) mv = root5 ? t5min[q] : (V)(t5min[q] - t4min);
          else mv = (V)(t5min[q] - s5min[q]);
          S.B[ones_before] = VT<V>::zz(mv);
          const u32 lpos = Pn[6] + 4u * r5;
          U le[4];
#pragma unroll
          for (int c = 0; c < 4; c++) {
            const int m = 4 * q + c;
            const bool in = CELL_IN(m);
            V x;
            if (as_snapshot) x = (V)(t5max[q] - (in ? tv[m] : (V)0));
            else x = in ? (V)(tv[m] - sv[m]) : (V)0;
            le[c] = VT<V>::zz(x);
          }
          if (sizeof(U) == 4) *reinterpret_cast<uint4*>(&A[lpos]) = make_uint4((u32)le[0], (u32)le[1], (u32)le[2], (u32)le[3]);
          else { A[lpos] = le[0]; A[lpos + 1] = le[1]; A[lpos + 2] = le[2]; A[lpos + 3] = le[3]; }
          r5++;
        } else if (!as_snapshot) {
          S.eqf[pos - ones_before] = (!((u5 >> q) & 1u) && ((eq5 >> q) & 1u)) ? 1 : 0;
        }
      }
    }
    __syncthreads();

    // ---------------- serialize (snapshot.rs:48-58 / log.rs:53-64)
    {
      const bool staged = my_size <= (u32)STAGE_BYTES;
      if (staged || fits) {
        u32 off;
        if (staged) off = serialize_structure<V>(S, S.stage, unit, lo, as_snapshot, nm_len, n_min);
        else off = serialize_structure<V>(S, P.arena + piece_off, unit, lo, as_snapshot, nm_len, n_min);
        if (off != my_size) err |= EF_BAD_FORMAT;  // internal consistency: emitted bytes == predicted size
        __syncthreads();
        if (staged && fits) {
          const uint4* src = reinterpret_cast<const uint4*>(S.stage);
          uint4* dst = reinterpret_cast<uint4*>(P.arena + piece_off);
          for (u32 i = tid; i < (my_size + 15u) / 16u; i += ENC_THREADS) dst[i] = src[i];
        }
      }
    }

    // ---------------- bookkeeping: start a new block or extend the current one
    if (as_snapshot) {
#pragma unroll
      for (int m = 0; m < 16; m++) sv[m] = tv[m];
      s3max = t3max; s3min = t3min; s2max = t2max; s2min = t2min;
      if (tid < 4) { S.s_l1max[tid] = S.l1[tid].tmax; S.s_l1min[tid] = S.l1[tid].tmin; }
      if (tid == 0) { S.s_l0max = N0.tmax; S.s_l0min = N0.tmin; }
      n_snap++;
      n_logs = 0;
      total_bytes += 1;  // Block's n_instants byte (block.rs:88-95)
    } else {
      n_logs++;
      n_log_total++;
    }
    total_bytes += my_size;
    __syncthreads();
#undef CELL_IN
  }

  if (tid == 0) {
    UnitResult r;
    r.bytes = total_bytes + 6;  // encoding + fractional_bits + n_blocks (chunk.rs:235-243)
    r.snapshots = n_snap;
    r.logs = n_log_total;
    P.results[unit_idx] = r;
  }
  err = __reduce_or_sync(0xffffffffu, err);  // one atomic per warp for the error bits
  if (lane == 0 && err) atomicOr(P.err, err);
}

}  // namespace dcdf
