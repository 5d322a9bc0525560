// encode_v5.cuh -- Chunk::build (chunk.rs:42-96) for the common case of a full 64x64 f32 tile whose to_fixed is exact
// (fixed.rs:47-57 never rounds), that holds no NaN, whose fixed-point values are below 2^22 in magnitude and lie within
// 32767 of each other over the whole unit (k_finalize_tree decides; everything else stays with k_encode_v4).  Under
// those conditions every DAC entry below the root takes at most two bytes, float -> fixed is one FFMA and one integer
// add, and the kernel can be small:
//   * same mapping as encode_v4.cuh (one 64-thread CTA per unit, thread t = level-3 node t in Morton order, 8x8 cells),
//     same masks / packed counters / BFS layout arithmetic, same bytes;
//   * ONE fused pass per Log instant: a thread reads its four level-4 nodes (4x4 cells each, four 128-bit loads)
//     straight from global memory, converts, and while the cells are in registers computes the differences to the
//     block's snapshot, the equal / uniform flags, the length classes AND the low bytes of every zigzag code, which
//     go to a 6 KB payload in shared memory.  The instant itself is never stored: emission copies payload words to
//     their scan-computed positions (the recomputation pass of v4 -- second read of both images, second min/max
//     pyramid, second zigzag -- is gone);
//   * entries longer than one byte (rare below the root) are re-derived at emission time from a second, L2-resident
//     read of just that level-4 node;
//   * a Snapshot is needed for one instant in several (first of a block): its exact size (only when the Log does not
//     already beat the one-byte-per-entry lower bound) and its emission each take their own pass over the tile from
//     L2; the emission pass also rewrites the snapshot image the following Logs refer to;
//   * the emission image is placed so that byte 1 of the max DAC's level 0 is 4-byte aligned: every sibling group
//     (BFS positions 1 + 4k .. 4 + 4k) is then one aligned 32-bit store; the copy to the arena re-aligns with funnel
//     shifts.
// 36 KB of shared memory per tile and <= 168 registers: six tiles per SM (v4: four).
// Reference functions restated: snapshot.rs:108-156 + 439-500, log.rs:112-165 + 725-817, bitmap.rs:66-113,
// dac.rs:96-132, chunk.rs:55-78, serializers snapshot.rs:48-58 / log.rs:53-64 / dac.rs:37-44 / bitmap.rs:128-138.
#pragma once
#include <type_traits>

#include "encode_v4.cuh"

namespace dcdf {

constexpr int E5_THREADS = 64;
constexpr int E5_POOL = 9 * 1024;
// Edge tiles (list 7): the raster covers at most the top or the left half of the tree, so one warp holds every
// level-3 node with cells; its structures are at most about half as large
constexpr int E5_POOL_EDGE = 5 * 1024;

// TT threads per tile (one per level-3 node that can hold cells), POOL bytes of emission image
template <int TT, int POOL>
struct E5SmemT {
  __align__(16) u8 pool[POOL + 16];  // emission image (+ room for the alignment shift)
  int4 cell[16][TT];                 // cells of the block's snapshot: [quad q][thread]
  int2 l4s[4][TT];                   // (max, min) of the snapshot's level-4 nodes
  int2 l4t[4][TT];                   // ... of the instant being encoded
  u32 leaf[16][TT];                  // Log payload: low bytes of the four leaf codes of quad q
  u32 qx[4][TT];                     // Log payload: low bytes of the four quad max codes of level-4 node a
  u32 qn[4][TT];                     // ... and of the four quad min codes
  int4 rec1[4];                      // level-1 nodes: tmax, tmin, first-cell diff, equal
  int2 ent1[4];                      // level-1 log entries
  u32 wt[2][2][4];                   // [warp][0 = snapshot, 1 = log][STRUCT, a1, b1, c1]
  u32 bm_off[12], bm_len[12];
  u32 n_bm;
  unsigned long long piece_off;
};
using E5Smem = E5SmemT<E5_THREADS, E5_POOL>;
using E5SmemEdge = E5SmemT<32, E5_POOL_EDGE>;

struct E5Cand {
  u32 in5, in4;        // internal flags: quad q = bit 15-q, level-4 node a = bit 3-a
  bool in3, in2, in1;
  u64 ml;              // leaves longer than one byte (cell m = bit 63-m)
  u32 mq;              // quads: max entries bits 15..0, min entries bits 31..16
  u32 mu;              // level 4 max (3..0) / min (7..4), level 3 max (8) / min (9), level 2 max (10) / min (11)
};

DCDF_DEVINL void e5_count(const E5Cand& C, bool owner2, u32* w /* [4] */) {
  const bool e2 = C.in1, e3 = e2 && C.in2, e4 = e3 && C.in3;
  const u32 ai4 = e4 ? C.in4 : 0u;
  const u32 X5 = e4_expand4(ai4);
  const u32 ai5 = C.in5 & X5;
  const u64 X6 = e4_expand16(ai5);
  const u32 mu = C.mu, mq = C.mq;
  w[0] = ((owner2 && e2 && C.in2) ? E4_F2 : 0u) + ((e3 && C.in3) ? E4_F3 : 0u) + (u32)__popc(ai4) * E4_F4 + (u32)__popc(ai5) * E4_F5;
  w[1] = ((owner2 && e2 && ((mu >> 10) & 1u)) ? E4_F2 : 0u) + ((e3 && ((mu >> 8) & 1u)) ? E4_F3 : 0u) +
         (e4 ? (u32)__popc(mu & 0xfu) : 0u) * E4_F4 + (u32)__popc(mq & 0xffffu & X5) * E4_F5;
  w[2] = (u32)__popcll(C.ml & X6);
  w[3] = ((owner2 && e2 && C.in2 && ((mu >> 11) & 1u)) ? E4_F2 : 0u) + ((e3 && C.in3 && ((mu >> 9) & 1u)) ? E4_F3 : 0u) +
         (u32)__popc((mu >> 4) & ai4) * E4_F4 + (u32)__popc((mq >> 16) & ai5) * E4_F5;
}

struct E5Tot {
  u32 tot[4];
  u32 I0, I1, nm_len, n_int;
};
// Block totals of one candidate (snapshot.rs:71-79, log.rs:77-86)
template <class Smem>
DCDF_DEVINL void e5_totals(E5Tot& T, const Smem& S, int cand, bool in0, u32 in1m) {
#pragma unroll
  for (int i = 0; i < 4; i++) T.tot[i] = in0 ? S.wt[0][cand][i] + S.wt[1][cand][i] : 0u;
  T.I0 = in0 ? 1u : 0u;
  T.I1 = in0 ? (u32)__popc(in1m) : 0u;
  const u32 upper = T.I0 + T.I1 + e4_f2(T.tot[0]) + e4_f3(T.tot[0]) + e4_f4(T.tot[0]);
  T.n_int = upper + e4_f5(T.tot[0]);
  T.nm_len = 1u + 4u * upper;
}

// The root's and the level-1 nodes' entries of a DAC are held one per lane: lane 0 = root, lane 1 + k = level-1 node k.
// They are the first entries of the DAC in BFS order, hence the first ones of every DAC level they reach (dac.rs:109-121).
// Byte length of such an entry (0: the entry does not exist)
DCDF_DEVINL int e5_len(bool valid, int e) {
  return valid ? 1 + (e4_longer<1>(e) ? 1 : 0) + (e4_longer<2>(e) ? 1 : 0) + (e4_longer<3>(e) ? 1 : 0) : 0;
}
// ... as nibbles 1..3 (nibble j set when the entry reaches DAC level j): a warp sum then counts the top entries per level
DCDF_DEVINL u32 e5_nib(int len) { return 0x1110u & ((1u << (4 * len)) - 1u); }
// an entry of the winner: zigzag code, length, position of its bytes on DAC levels 0 and 1 (levels 2 and 3: e5_top_long)
struct E5Top {
  u32 z;
  int len;
  u32 pos0, pos1;
};

// The stream items of a candidate, one per lane, in stream order (snapshot.rs:48-58 / log.rs:53-64, dac.rs:37-44):
// lane 0 = nodemap bitmap, 1 = `equal` bitmap (Logs only), 2 + j = level j of the max DAC, 6 + j = level j of the min
// DAC; the DAC's level-count byte goes with its level 0.  ntop: top entries per DAC level (e5_nib, min DAC << 16).
// cnt = the item's bits or entries; returns its size in bytes.  Below the level-1 nodes nothing is longer than two bytes,
// so DAC levels 2 and 3 only hold bytes of the root / level-1 entries.
DCDF_DEVINL u32 e5_item(u32& cnt, const E5Tot& T, bool as_log, u32 ntop, int lane) {
  const int j = (lane - 2) & 7, lev = j & 3;
  const bool mn = j >= 4;
  u32 c = (ntop >> (4 * j)) & 0xfu;
  if (lev == 0) c = mn ? T.n_int : 1u + 4u * T.n_int;
  else if (lev == 1) c += mn ? e4_fsum(T.tot[3]) : e4_fsum(T.tot[1]) + T.tot[2];
  if (lane == 0) c = T.nm_len;
  if (lane == 1) c = T.nm_len - T.n_int;
  cnt = lane < 10 ? c : 0u;
  if (lane < 2) return (lane == 0 || as_log) ? bitmap_size(c) : 0u;
  return lane >= 10 ? 0u : (c ? bitmap_size(c) + c : 0u) + (lev == 0 ? 1u : 0u);
}

// second byte of a two-byte code (DAC level 1): rare, out of line; returns the next position
__device__ __noinline__ u32 e5_hi(u8* b1, u32 z, u32 r1) {
  b1[r1] = (u8)(z >> 8);
  return r1 + 1u;
}

// OR a run of bits into a bit stream (e4_or_run): the 64-bit form is rare (leaf flags), out of line
__device__ __noinline__ void e5_or_run(u8* bytes, u32 bitpos, u64 V) { e4_or_run(bytes, bitpos, V); }
// ... a run of n <= 32 bits, right-aligned in `bits` (at most two containers)
DCDF_DEVINL void e5_or_bits(u8* bytes, u32 bitpos, u32 bits, int n) {
  if (n <= 0 || !bits) return;
  const u32 hi = bits << (32 - n);
  const uintptr_t A = (uintptr_t)bytes;
  const u32 g = bitpos + 8u * (u32)(A & 3u);
  const u32 sft = g & 31u;
  u32* w = reinterpret_cast<u32*>(A & ~(uintptr_t)3) + (g >> 5);
  const u32 w0 = hi >> sft, w1 = __funnelshift_r(0u, hi, sft);
  if (w0) e4_red_or(w, e4_bswap(w0));
  if (w1) e4_red_or(w + 1, e4_bswap(w1));
}
// ... one bit
DCDF_DEVINL void e5_or_bit(u8* bytes, u32 bitpos) {
  const uintptr_t A = (uintptr_t)bytes;
  const u32 g = bitpos + 8u * (u32)(A & 3u);
  e4_red_or(reinterpret_cast<u32*>(A & ~(uintptr_t)3) + (g >> 5), e4_bswap(0x80000000u >> (g & 31u)));
}
// Bytes 3 and 4 of the top entries (rare: the root of a Snapshot, or a jump of 2^15 or more): continuation bits on DAC
// levels 1 and 2 (phase A) or the bytes on levels 2 and 3 (phase B).  l0: lane of the DAC's level-0 item.  Warp-wide.
__device__ __noinline__ void e5_top_long(bool bytes, u8* out, const E5Top& t, int l0, u32 hdr, u32 cnt, u32 at) {
  const u32 lt = (1u << (threadIdx.x & 31u)) - 1u;
  const u32 p2 = (u32)__popc(__ballot_sync(0xffffffffu, t.len > 2) & lt);
  if (!bytes) {
    u8* const w1 = e4_words_of(out, __shfl_sync(0xffffffffu, hdr, l0 + 1), __shfl_sync(0xffffffffu, cnt, l0 + 1));
    u8* const w2 = e4_words_of(out, __shfl_sync(0xffffffffu, hdr, l0 + 2), __shfl_sync(0xffffffffu, cnt, l0 + 2));
    if (t.len > 2) e5_or_bit(w1, t.pos1);
    if (t.len > 3) e5_or_bit(w2, p2);
  } else {
    const u32 p3 = (u32)__popc(__ballot_sync(0xffffffffu, t.len > 3) & lt);
    u8* const b2 = out + __shfl_sync(0xffffffffu, at, l0 + 2);
    u8* const b3 = out + __shfl_sync(0xffffffffu, at, l0 + 3);
    if (t.len > 2) b2[p2] = (u8)(t.z >> 16);
    if (t.len > 3) b3[p3] = (u8)(t.z >> 24);
  }
}
// One level-4 node (4x4 cells at pn, row stride sr) as four quads (x, y = upper row; z, w = lower row).
// Clipped tiles (FULL == false): rl / cl = rows / columns of the node that lie inside the raster (may be <= 0); cells
// outside are not read and become None (E4_NONE, as in encode_v4.cuh: excluded from min / max, 0 in an entry).
template <bool FULL>
DCDF_DEVINL void e5_load_node(const float* pn, i64 sr, uint4 (&raw)[4], int rl, int cl, int vec) {
#pragma unroll
  for (int r = 0; r < 4; r++) {
    if (FULL || (r < rl && cl >= 4)) {
      const float* pr = pn + (i64)r * sr;
      if (vec == 2) {  // the instant's tile sits in shared memory (bulk-copy variant)
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(raw[r].x), "=r"(raw[r].y), "=r"(raw[r].z), "=r"(raw[r].w)
                     : "r"((u32)__cvta_generic_to_shared(pr)));
      } else if (vec) {
        raw[r] = __ldg(reinterpret_cast<const uint4*>(pr));
      } else {  // rows that are not 16-byte aligned (e.g. 1405 columns): four 32-bit loads
        raw[r] = make_uint4(__float_as_uint(__ldg(pr)), __float_as_uint(__ldg(pr + 1)), __float_as_uint(__ldg(pr + 2)), __float_as_uint(__ldg(pr + 3)));
      }
    } else {
      raw[r] = make_uint4(0, 0, 0, 0);
      if (r < rl) {
        const float* pr = pn + (i64)r * sr;
        if (cl > 0) raw[r].x = __float_as_uint(__ldg(pr));
        if (cl > 1) raw[r].y = __float_as_uint(__ldg(pr + 1));
        if (cl > 2) raw[r].z = __float_as_uint(__ldg(pr + 2));
      }
    }
  }
}
// to_fixed (a3) of an exact, finite, small value: n * 2^(bits+1) is an integer below 2^22, so adding 1.5 * 2^23
// leaves it in the low mantissa bits (fixed.rs:59-70: trunc(2 * shifted) + 1).  Without the NaN test: a NaN comes out as
// as_int(NaN) - (0x4B400000 - 1) > 2^29, far above any eligible value (e5_quads looks for it once per node).
DCDF_DEVINL int e5_conv_raw(float x, float scale2) { return __float_as_int(__fmaf_rn(x, scale2, 12582912.0f)) - (0x4B400000 - 1); }
DCDF_DEVINL int e5_nan0(u32 bits, int f) { return (bits & 0x7fffffffu) > 0x7f800000u ? 0 : f; }
template <bool FULL>
DCDF_DEVINL void e5_quads(const uint4 (&raw)[4], float scale2, int4 (&q)[4], int rl, int cl) {
#pragma unroll
  for (int h = 0; h < 2; h++) {
    const uint4 u = raw[2 * h], l = raw[2 * h + 1];
    q[2 * h] = make_int4(e5_conv_raw(__uint_as_float(u.x), scale2), e5_conv_raw(__uint_as_float(u.y), scale2),
                         e5_conv_raw(__uint_as_float(l.x), scale2), e5_conv_raw(__uint_as_float(l.y), scale2));
    q[2 * h + 1] = make_int4(e5_conv_raw(__uint_as_float(u.z), scale2), e5_conv_raw(__uint_as_float(u.w), scale2),
                             e5_conv_raw(__uint_as_float(l.z), scale2), e5_conv_raw(__uint_as_float(l.w), scale2));
  }
  // NaN -> 0 (fixed.rs:35-37), looked for once per node instead of once per cell: the largest of the sixteen values
  {
    const int m01 = max(max(max(q[0].x, q[0].y), max(q[0].z, q[0].w)), max(max(q[1].x, q[1].y), max(q[1].z, q[1].w)));
    const int m23 = max(max(max(q[2].x, q[2].y), max(q[2].z, q[2].w)), max(max(q[3].x, q[3].y), max(q[3].z, q[3].w)));
    if (max(m01, m23) > (1 << 28)) {
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const uint4 u = raw[2 * h], l = raw[2 * h + 1];
        q[2 * h] = make_int4(e5_nan0(u.x, q[2 * h].x), e5_nan0(u.y, q[2 * h].y), e5_nan0(l.x, q[2 * h].z), e5_nan0(l.y, q[2 * h].w));
        q[2 * h + 1] = make_int4(e5_nan0(u.z, q[2 * h + 1].x), e5_nan0(u.w, q[2 * h + 1].y), e5_nan0(l.z, q[2 * h + 1].z), e5_nan0(l.w, q[2 * h + 1].w));
      }
    }
  }
#pragma unroll
  for (int h = 0; h < 2; h++) {
    if (!FULL) {
      const bool ru = 2 * h < rl, rw = 2 * h + 1 < rl;
      if (!(ru && cl > 0)) q[2 * h].x = E4_NONE;
      if (!(ru && cl > 1)) q[2 * h].y = E4_NONE;
      if (!(rw && cl > 0)) q[2 * h].z = E4_NONE;
      if (!(rw && cl > 1)) q[2 * h].w = E4_NONE;
      if (!(ru && cl > 2)) q[2 * h + 1].x = E4_NONE;
      if (!(ru && cl > 3)) q[2 * h + 1].y = E4_NONE;
      if (!(rw && cl > 2)) q[2 * h + 1].z = E4_NONE;
      if (!(rw && cl > 3)) q[2 * h + 1].w = E4_NONE;
    }
  }
}
DCDF_DEVINL const float* e5_node_ptr(const float* pt, i64 sr, int a) { return pt + (i64)(4 * (a >> 1)) * sr + 4 * (a & 1); }
// differences that become DAC entries: a max of a node without cells counts as 0 (`None => 0`, snapshot.rs:122-130,
// log.rs:128-135); min entries only exist for internal nodes, whose min is a value
template <bool FULL>
DCDF_DEVINL int e5_dx(int a, int b) { return e4_sub(e4_o0<FULL>(a), e4_o0<FULL>(b)); }
DCDF_DEVINL int e5_dn(int a, int b) { return e4_sub(a, b); }

// low bytes of four values as one word, and the zigzag codes of four signed bytes at once (dac.rs:134-137 on values in
// -128..127: (b << 1) ^ (b >> 7) per byte; the carries of p + p land in the cleared low bits)
DCDF_DEVINL u32 e5_low4(int a, int b, int c, int d) { return __byte_perm(__byte_perm((u32)a, (u32)b, 0x0040), __byte_perm((u32)c, (u32)d, 0x0040), 0x5410); }
DCDF_DEVINL u32 e5_zz4(u32 p) { return ((p + p) & 0xfefefefeu) ^ (((p >> 7) & 0x01010101u) * 0xffu); }
DCDF_DEVINL u32 e5_pack4(u32 z0, u32 z1, u32 z2, u32 z3) { return (z0 & 0xffu) | ((z1 & 0xffu) << 8) | ((z2 & 0xffu) << 16) | (z3 << 24); }
// ALIGNED: the staged image is shifted so that every group of four sibling entries starts on a word (the caller knows)
template <bool ALIGNED = false>
DCDF_DEVINL void e5_store_word(u8* p, u32 w) {
  if (ALIGNED || (((uintptr_t)p) & 3u) == 0) *reinterpret_cast<u32*>(p) = w;
  else { p[0] = (u8)w; p[1] = (u8)(w >> 8); p[2] = (u8)(w >> 16); p[3] = (u8)(w >> 24); }
}

// Entries of one level-4 node that take two bytes (rare), re-derived from the node's cells: leaves of the internal
// quads, then the four quad max entries, then the min entries of the internal quads -- the order in which their second
// bytes sit in DAC level 1 (dac.rs:109-121).  Log: cells of the instant come from a second (L2-resident) read of the
// node, the snapshot's from shared memory.  Snapshot: the emission pass has just stored the cells in shared memory.
// scell: the node's quad 0 in E5SmemT::cell, whose quads lie TT apart
template <bool FULL, int TT = E5_THREADS>
__device__ __noinline__ void e5_long_node(bool as_snapshot, const float* pn, i64 sr, float scale2, const int4* scell, int2 n4, u32 in5a,
                                          u8* xb1, u8* nb1, u32* pos /* lx1, rx1, rn1 */, int rl, int cl, int vec) {
  int4 q[4];
  if (!as_snapshot) {
    uint4 raw[4];
    e5_load_node<FULL>(pn, sr, raw, rl, cl, vec);
    e5_quads<FULL>(raw, scale2, q, rl, cl);
  }
  u32 lx1 = pos[0], rx1 = pos[1], rn1 = pos[2];
  u32 zx[4], zn[4];
#pragma unroll
  for (int b = 0; b < 4; b++) {
    const int4 s = scell[b * TT];
    const int4 t = as_snapshot ? s : q[b];
    int qmax, qmin, sqmax, sqmin;
    e4_qmm<FULL>(t, qmax, qmin);
    e4_qmm<FULL>(s, sqmax, sqmin);
    zx[b] = zigzag32(as_snapshot ? e5_dx<FULL>(n4.x, qmax) : e5_dx<FULL>(qmax, sqmax));
    zn[b] = zigzag32(as_snapshot ? e5_dn(qmin, n4.y) : e5_dn(qmin, sqmin));
    if ((in5a >> (3 - b)) & 1u) {
      const u32 z0 = zigzag32(as_snapshot ? e5_dx<FULL>(qmax, t.x) : e4_sub(t.x, s.x)), z1 = zigzag32(as_snapshot ? e5_dx<FULL>(qmax, t.y) : e4_sub(t.y, s.y));
      const u32 z2 = zigzag32(as_snapshot ? e5_dx<FULL>(qmax, t.z) : e4_sub(t.z, s.z)), z3 = zigzag32(as_snapshot ? e5_dx<FULL>(qmax, t.w) : e4_sub(t.w, s.w));
      if (z0 > 0xffu) xb1[lx1++] = (u8)(z0 >> 8);
      if (z1 > 0xffu) xb1[lx1++] = (u8)(z1 >> 8);
      if (z2 > 0xffu) xb1[lx1++] = (u8)(z2 >> 8);
      if (z3 > 0xffu) xb1[lx1++] = (u8)(z3 >> 8);
    }
  }
#pragma unroll
  for (int b = 0; b < 4; b++)
    if (zx[b] > 0xffu) xb1[rx1++] = (u8)(zx[b] >> 8);
#pragma unroll
  for (int b = 0; b < 4; b++)
    if (((in5a >> (3 - b)) & 1u) && zn[b] > 0xffu) nb1[rn1++] = (u8)(zn[b] >> 8);
  pos[0] = lx1; pos[1] = rx1; pos[2] = rn1;
}

// mbarrier + bulk copy (the TMA unit's 1-D form) for the BULK variant of the kernel
DCDF_DEVINL u32 e5_smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
DCDF_DEVINL void e5_mbar_init(unsigned long long* b, u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(e5_smem_u32(b)), "r"(count) : "memory");
}
DCDF_DEVINL void e5_mbar_expect_tx(unsigned long long* b, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(e5_smem_u32(b)), "r"(bytes) : "memory");
}
DCDF_DEVINL void e5_mbar_wait(unsigned long long* b, u32 parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "E5_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra E5_DONE;\n\t"
      "bra E5_WAIT;\n\t"
      "E5_DONE:\n\t}" ::"r"(e5_smem_u32(b)), "r"(parity) : "memory");
}
DCDF_DEVINL void e5_bulk_g2s(void* smem, const void* g, u32 bytes, unsigned long long* b) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(e5_smem_u32(smem)),
               "l"(g), "r"(bytes), "r"(e5_smem_u32(b))
               : "memory");
}
// BULK variant: the instant's 64x64 f32 tile, row-major, filled by 64 bulk copies (one row each) behind an mbarrier
struct E5Bulk {
  __align__(16) float raw[64 * 64];
  __align__(8) unsigned long long mbar;
  unsigned long long pad_;
};

// barrier over the threads of one tile: named barrier 1 + tile slot for a two-warp tile (barrier 0 stays the CTA-wide
// one), the warp itself for a one-warp tile
template <int NW>
DCDF_DEVINL void e5_tile_sync(int slot) {
  if (NW == 1) __syncwarp();
  else asm volatile("bar.sync %0, 64;" ::"r"(slot + 1) : "memory");
}

// G tiles per CTA, one per group of NW warps.  The tiles are independent (own shared-memory slab, own named barrier);
// what they share is the instruction stream: one CTA-wide barrier per instant keeps all NW * G warps of the SM inside the
// same stretch of code, so instruction-cache lines fetched for one warp are hits for the others (with unsynchronised
// CTAs the kernel spent a quarter of its issue slots waiting for instruction fetches).
// NW = 2: thread t of a tile is level-3 node t.  NW = 1 (edge tiles, FULL == false only): the unit has at most 32 rows or
// at most 32 columns in the raster, so the level-3 nodes of the other half of the tree (rows 32-63: nodes 32-63;
// columns 32-63: nodes 16-31 and 48-63) hold no cell.  Lane l takes node l (top half) or node l, l + 16 (left half):
// each group of 16 lanes is still one level-1 node.  The missing half is two all-None level-1 nodes; what the NW = 2
// kernel computes for such a node is a constant: no internal node below it (all its counters are 0), record
// (None, INT32_MAX, diff 0, equal) and Log entries (0, 0), set once below.
template <int G, bool FULL, bool BULK, int NW = 2>
DCDF_DEVINL void e5_body(const EncParams& P, const u32 stage_limit, const int sync_mask);
template <int G, bool FULL, bool BULK = false>
__global__ void __launch_bounds__(E5_THREADS * G, 1) k_encode_v5(const EncParams P, const u32 stage_limit, const int sync_mask) {
  e5_body<G, FULL, BULK>(P, stage_limit, sync_mask);
}
template <int G>
__global__ void __launch_bounds__(32 * G, 1) k_encode_v5_edge(const EncParams P, const u32 stage_limit, const int sync_mask) {
  e5_body<G, false, false, 1>(P, stage_limit, sync_mask);
}
template <int G, bool FULL, bool BULK, int NW>
DCDF_DEVINL void e5_body(const EncParams& P, const u32 stage_limit, const int sync_mask) {
  static_assert(NW == 2 || (NW == 1 && !FULL && !BULK), "one-warp tiles are clipped edge tiles");
  constexpr int TT = 32 * NW;  // threads per tile
  using Smem = std::conditional_t<NW == 2, E5Smem, E5SmemEdge>;
  // every row of four cells is 16-byte aligned -> 128-bit loads; BULK (host checked the alignment): loads from the staged tile
  const int vec = BULK ? 2 : (((P.stride_r | P.stride_t) & 3) == 0 && (((uintptr_t)P.data) & 15) == 0) ? 1 : 0;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int slot = threadIdx.x / TT;
  constexpr size_t kSlab = sizeof(Smem) + (BULK ? sizeof(E5Bulk) : 0);
  Smem& S = *reinterpret_cast<Smem*>(smem_raw + (size_t)slot * kSlab);
  E5Bulk& SB = *reinterpret_cast<E5Bulk*>(smem_raw + (size_t)slot * kSlab + sizeof(Smem));  // only touched when BULK

  const u32 n_order = *P.order_count;
  if (blockIdx.x * (u32)G >= n_order) return;
  const u32 order_idx = blockIdx.x * (u32)G + (u32)slot;
  const bool tile_live = order_idx < n_order;
  const u32 unit_idx = P.order[tile_live ? order_idx : blockIdx.x * (u32)G];
  EncUnit unit = P.units[unit_idx];
  if (!tile_live) unit.instants = 0;
  // every tile of the CTA takes the CTA-wide barrier the same number of times
  int max_instants = 0;
  for (int g = 0; g < G; g++) {
    const u32 oi = blockIdx.x * (u32)G + (u32)g;
    if (oi < n_order) max_instants = max(max_instants, P.units[P.order[oi]].instants);
  }
  const int tid = threadIdx.x % TT, lane = tid & 31, warp = tid >> 5;
  // the thread's level-3 node (NW = 1: the top half of the tree when the unit has at most 32 rows, else the left half)
  const int node = NW == 2 ? tid : unit.rows <= 32 ? lane : lane < 16 ? lane : lane + 16;
  const float scale2 = (float)((i64)2 << unit.bits);
  const i64 sr = BULK ? 64 : P.stride_r;
  // the thread's 8x8 block
  const float* const base = BULK ? SB.raw + (8 * (int)morton_row(tid)) * 64 + 8 * (int)morton_col(tid)
                                 : static_cast<const float*>(P.data) + unit.base + (i64)(8 * (int)morton_row(node)) * sr + 8 * (int)morton_col(node);
  // BULK: thread r fetches row r of the tile (256 bytes) of one instant
  const float* const my_row = static_cast<const float*>(P.data) + unit.base + (i64)tid * P.stride_r;
  auto fetch_instant = [&](int t) {
    if (tid == 0) e5_mbar_expect_tx(&SB.mbar, 64u * 256u);
    e5_bulk_g2s(SB.raw + 64 * tid, my_row + (i64)t * P.stride_t, 256u, &SB.mbar);
  };
  if (BULK) {
    if (tid == 0) {
      e5_mbar_init(&SB.mbar, 1u);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    e5_tile_sync<NW>(slot);
    if (unit.instants > 0) fetch_instant(0);
  }
  const bool owner2 = (lane & 3) == 0;
  const bool is1 = (u32)(lane - 1) < 4u;  // lane 1 + k holds level-1 node k at the top of the tree
  const int k1 = node >> 4;  // own level-1 node
  // rows / columns of the raster left from the origin of the thread's level-4 node a (clipped tiles)
  const int rl8 = unit.rows - 8 * (int)morton_row(node), cl8 = unit.cols - 8 * (int)morton_col(node);
#define E5_RL(a) (rl8 - 4 * ((a) >> 1))
#define E5_CL(a) (cl8 - 4 * ((a) & 1))

  {  // the emission image starts out all zero; every copy-out re-zeroes what it used
    uint4* z = reinterpret_cast<uint4*>(S.pool);
    for (int i = tid; i < (int)(sizeof(S.pool) / 16); i += TT) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (!FULL) {  // cells outside the raster are None in the snapshot image from the start
    for (int q = 0; q < 16; q++) S.cell[q][tid] = make_int4(E4_NONE, E4_NONE, E4_NONE, E4_NONE);
    for (int a = 0; a < 4; a++) S.l4s[a][tid] = make_int2(E4_NONE, INT32_MAX);
  }
  if (NW == 1 && lane == 0) {  // the two level-1 nodes without threads (see above); never written again
    const u32 missing1 = unit.rows <= 32 ? 0xcu : 0xau;  // bit k: level-1 node k
    for (int k = 0; k < 4; k++) {
      if ((missing1 >> k) & 1u) {
        S.rec1[k] = make_int4(E4_NONE, INT32_MAX, 0, 1);
        S.ent1[k] = make_int2(0, 0);
      }
    }
    for (int c = 0; c < 2; c++)
      for (int i = 0; i < 4; i++) S.wt[1][c][i] = 0u;
  }

  u32 err = 0;
  int s3max = 0, s3min = 0, s2max = 0, s2min = 0, s1max = 0, s1min = 0, s0max = 0, s0min = 0;
  u32 n_logs = 0, n_snap = 0, n_log_total = 0;
  u64 total_bytes = 0;

#pragma unroll 1
  for (int inst = 0; inst < max_instants; inst++) {
    if ((inst & sync_mask) == 0) __syncthreads();  // all tiles of the CTA start the instant together (shared instruction stream)
    if (inst >= unit.instants) continue;
    const bool first = inst == 0;
    const float* const pt = BULK ? base : base + (i64)inst * P.stride_t;
    if (BULK) e5_mbar_wait(&SB.mbar, (u32)inst & 1u);  // the instant's tile has landed
    if (!BULK && inst + 1 < unit.instants) {  // the next instant's cells on their way into L2 (the tiles of a CTA all load at once)
#pragma unroll
      for (int r = 0; r < 8; r++)
        if (FULL || (r < rl8 && cl8 > 0)) asm volatile("prefetch.global.L2 [%0];" ::"l"(pt + P.stride_t + (i64)r * sr));
    }
    const bool forced = first || n_logs == 254u;  // chunk.rs:62 (Block caps logs at 254)

    u32 u5 = 0, eq5 = 0, u4 = 0, eq4 = 0;
    E5Cand L, C;
    L.ml = 0; L.mq = 0; L.mu = 0; L.in5 = 0; L.in4 = 0; L.in3 = L.in2 = L.in1 = false;
    C.ml = 0; C.mq = 0; C.mu = 0; C.in5 = 0; C.in4 = 0; C.in3 = C.in2 = C.in1 = false;
    int t3max = 0, t3min = 0, diff3 = 0;
    bool eq3 = false, u3 = false;
    int t2max = 0, t2min = 0, t1max = 0, t1min = 0, t0max = 0, t0min = 0;
    bool u2 = false, eq2 = false, u0 = false, eq0 = false;
    // lanes 1..4: level-1 node lane - 1 (record, flags, Log entries)
    int n1max = 0, n1min = 0, l_e1max = 0, l_e1min = 0;
    bool n1un = false, n1eq = false;
    u32 l_in1 = 0, s_in1 = 0;    // level-1 internal flags, node k = bit 3-k
    bool l_in0 = false, s_in0 = false;
    u32 wl[4] = {0, 0, 0, 0}, ws[4] = {0, 0, 0, 0};
    E5Tot T;
    u32 ntop = 0, item_cnt = 0, item_size = 0;  // the winner's top-entry counts and this lane's stream item (e5_item)
    bool as_snapshot = forced;
    u32 my_size = 0, log_size = 0;

    // Pass 0: the fused Log pass and the Log's exact size against a lower bound of the Snapshot's.  Pass 1 (first
    // instant of a block, the 254-log cap, or a Log that does not beat the bound): the Snapshot's exact size.
#pragma unroll 1
    for (int pass = forced ? 1 : 0; pass < 2; pass++) {
      t3max = INT32_MIN; t3min = INT32_MAX;
      u5 = 0; u4 = 0;
      uint4 raw[4];
      e5_load_node<FULL>(e5_node_ptr(pt, sr, 0), sr, raw, E5_RL(0), E5_CL(0), vec);
      if (pass == 0) {
        // ---------------- load, convert, differences, flags, length classes, payload
        eq3 = true;
#pragma unroll 1
        for (int a = 0; a < 4; a++) {
          int4 q[4];
          e5_quads<FULL>(raw, scale2, q, E5_RL(a), E5_CL(a));
          if (a < 3) e5_load_node<FULL>(e5_node_ptr(pt, sr, a + 1), sr, raw, E5_RL(a + 1), E5_CL(a + 1), vec);
          const int2 s4 = S.l4s[a][tid];
          int amax = INT32_MIN, amin = INT32_MAX, dfirst = 0;
          bool aeq = true;
          u32 leaf16 = 0, u5n = 0, e5n = 0, qx = 0, qn = 0;
          u32 exw = 0, enw = 0;          // low bytes of the four quad max / min entries
          u32 ovx = 0, ovn = 0, ovm = 0; // exact low bytes of the zigzag codes of entries outside -128..127
#pragma unroll
          for (int b = 0; b < 4; b++) {
            const int4 t = q[b], sq = S.cell[4 * a + b][tid];
            int qmax, qmin, sqmax, sqmin;
            e4_qmm<FULL>(t, qmax, qmin);
            e4_qmm<FULL>(sq, sqmax, sqmin);
            const int d0 = e4_sub(t.x, sq.x), d1 = e4_sub(t.y, sq.y), d2 = e4_sub(t.z, sq.z), d3 = e4_sub(t.w, sq.w);  // None - None = 0 (log.rs:751)
            const int ex = e5_dx<FULL>(qmax, sqmax), en = e5_dn(qmin, sqmin);
            const bool e5 = (((d1 ^ d0) | (d2 ^ d0) | (d3 ^ d0)) == 0);  // all four leaf diffs equal (log.rs:780-806)
            if (e4_unif<FULL>(qmax, qmin)) u5n |= 1u << (3 - b);
            if (e5) e5n |= 1u << (3 - b);
            u32 leafw = e5_zz4(e5_low4(d0, d1, d2, d3));
            exw = __byte_perm(exw, (u32)ex, b == 0 ? 0x3214 : b == 1 ? 0x3240 : b == 2 ? 0x3410 : 0x4210);
            enw = __byte_perm(enw, (u32)en, b == 0 ? 0x3214 : b == 1 ? 0x3240 : b == 2 ? 0x3410 : 0x4210);
            // one test for "some entry of this quad needs two bytes" (zigzag code above 255  <=>  value outside -128..127)
            if ((((u32)d0 + 128u) | ((u32)d1 + 128u) | ((u32)d2 + 128u) | ((u32)d3 + 128u) | ((u32)ex + 128u) | ((u32)en + 128u)) > 255u) {
              if (e4_longer<1>(d0)) leaf16 |= 1u << (15 - 4 * b);
              if (e4_longer<1>(d1)) leaf16 |= 1u << (14 - 4 * b);
              if (e4_longer<1>(d2)) leaf16 |= 1u << (13 - 4 * b);
              if (e4_longer<1>(d3)) leaf16 |= 1u << (12 - 4 * b);
              if (e4_longer<1>(ex)) qx |= 1u << (3 - b);
              if (e4_longer<1>(en)) qn |= 1u << (3 - b);
              if ((((u32)d0 + 32768u) | ((u32)d1 + 32768u) | ((u32)d2 + 32768u) | ((u32)d3 + 32768u)) > 65535u) err |= EF_BAD_FORMAT;  // not eligible
              leafw = e5_pack4(zigzag32(d0), zigzag32(d1), zigzag32(d2), zigzag32(d3));
              ovx |= (zigzag32(ex) & 0xffu) << (8 * b);
              ovn |= (zigzag32(en) & 0xffu) << (8 * b);
              ovm |= 0xffu << (8 * b);
            }
            S.leaf[4 * a + b][tid] = leafw;
            amax = max(amax, qmax); amin = min(amin, qmin);
            if (b == 0) dfirst = d0;
            aeq = aeq && e5 && d0 == dfirst;
          }
          const u32 zxw = (e5_zz4(exw) & ~ovm) | ovx, znw = (e5_zz4(enw) & ~ovm) | ovn;
          S.qx[a][tid] = zxw;
          S.qn[a][tid] = znw;
          S.l4t[a][tid] = make_int2(amax, amin);
          L.ml |= (u64)leaf16 << (48 - 16 * a);
          L.mq |= (qx << (12 - 4 * a)) | (qn << (28 - 4 * a));
          u5 |= u5n << (12 - 4 * a);
          eq5 |= e5n << (12 - 4 * a);
          if (e4_unif<FULL>(amax, amin)) u4 |= 1u << (3 - a);
          if (aeq) eq4 |= 1u << (3 - a);
          if (e4_longer<1>(e5_dx<FULL>(amax, s4.x))) L.mu |= 1u << (3 - a);
          if (e4_longer<1>(e5_dn(amin, s4.y))) L.mu |= 1u << (7 - a);
          t3max = max(t3max, amax); t3min = min(t3min, amin);
          if (a == 0) diff3 = dfirst;
          eq3 = eq3 && aeq && dfirst == diff3;
        }
        if (e4_longer<1>(e5_dx<FULL>(t3max, s3max))) L.mu |= 1u << 8;
        if (e4_longer<1>(e5_dn(t3min, s3min))) L.mu |= 1u << 9;
      } else {
        // ---------------- Snapshot entry masks of levels 6 and 5 (snapshot.rs:122-147: parent_max - child_max,
        // child_min - parent_min); the uniform flags and the level-4 records come out the same as in pass 0
        C.ml = 0; C.mq = 0;
#pragma unroll 1
        for (int a = 0; a < 4; a++) {
          int4 q[4];
          e5_quads<FULL>(raw, scale2, q, E5_RL(a), E5_CL(a));
          if (a < 3) e5_load_node<FULL>(e5_node_ptr(pt, sr, a + 1), sr, raw, E5_RL(a + 1), E5_CL(a + 1), vec);
          int qmax[4], qmin[4];
#pragma unroll
          for (int b = 0; b < 4; b++) e4_qmm<FULL>(q[b], qmax[b], qmin[b]);
          const int amax = max(max(qmax[0], qmax[1]), max(qmax[2], qmax[3])), amin = min(min(qmin[0], qmin[1]), min(qmin[2], qmin[3]));
          u32 leaf16 = 0, qx = 0, qn = 0, u5n = 0;
#pragma unroll
          for (int b = 0; b < 4; b++) {
            const int4 t = q[b];
            if (e4_unif<FULL>(qmax[b], qmin[b])) u5n |= 1u << (3 - b);
            // full tiles: every difference is >= 0 and below the quad's / node's range; clipped: a cell outside counts as 0
            if (!FULL || ((u32)(qmax[b] - qmin[b]) | (u32)(amax - qmax[b]) | (u32)(qmin[b] - amin)) > 127u) {
              if (e4_longer<1>(e5_dx<FULL>(qmax[b], t.x))) leaf16 |= 1u << (15 - 4 * b);
              if (e4_longer<1>(e5_dx<FULL>(qmax[b], t.y))) leaf16 |= 1u << (14 - 4 * b);
              if (e4_longer<1>(e5_dx<FULL>(qmax[b], t.z))) leaf16 |= 1u << (13 - 4 * b);
              if (e4_longer<1>(e5_dx<FULL>(qmax[b], t.w))) leaf16 |= 1u << (12 - 4 * b);
              if (e4_longer<1>(e5_dx<FULL>(amax, qmax[b]))) qx |= 1u << (3 - b);
              if (e4_longer<1>(e5_dn(qmin[b], amin))) qn |= 1u << (3 - b);
            }
          }
          S.l4t[a][tid] = make_int2(amax, amin);
          C.ml |= (u64)leaf16 << (48 - 16 * a);
          C.mq |= (qx << (12 - 4 * a)) | (qn << (28 - 4 * a));
          u5 |= u5n << (12 - 4 * a);
          if (e4_unif<FULL>(amax, amin)) u4 |= 1u << (3 - a);
          t3max = max(t3max, amax); t3min = min(t3min, amin);
        }
        if (t3max != E4_NONE && (u32)e4_sub(t3max, t3min) > 32767u) err |= EF_BAD_FORMAT;  // not eligible
      }
      u3 = e4_unif<FULL>(t3max, t3min);

      // ---------------- levels 2 and 1 with shuffles (4 resp. 16 consecutive lanes)
      t2max = max(t3max, shfl_xor(t3max, 1)); t2max = max(t2max, shfl_xor(t2max, 2));
      t2min = min(t3min, shfl_xor(t3min, 1)); t2min = min(t2min, shfl_xor(t2min, 2));
      const int diff2 = shfl(diff3, lane & ~3);
      const u32 ok3 = __ballot_sync(0xffffffffu, eq3 && diff3 == diff2);
      eq2 = ((ok3 >> (lane & ~3)) & 0xfu) == 0xfu;
      u2 = e4_unif<FULL>(t2max, t2min);
      t1max = max(t2max, shfl_xor(t2max, 4)); t1max = max(t1max, shfl_xor(t1max, 8));
      t1min = min(t2min, shfl_xor(t2min, 4)); t1min = min(t1min, shfl_xor(t1min, 8));
      const int diff1 = shfl(diff2, lane & ~15);
      const u32 ok2 = __ballot_sync(0xffffffffu, eq2 && diff2 == diff1);
      const bool eq1 = ((ok2 >> (lane & ~15)) & 0xffffu) == 0xffffu;
      const bool u1 = e4_unif<FULL>(t1max, t1min);

      // structure flags: snapshot internal = !uniform (snapshot.rs:133); log internal = !uniform && !equal (log.rs:137-152)
      C.in5 = ~u5 & 0xffffu; C.in4 = ~u4 & 0xfu; C.in3 = !u3; C.in2 = !u2; C.in1 = !u1;
      if (pass == 0) {
        if (e4_longer<1>(e5_dx<FULL>(t2max, s2max))) L.mu |= 1u << 10;
        if (e4_longer<1>(e5_dn(t2min, s2min))) L.mu |= 1u << 11;
        L.in5 = ~u5 & ~eq5 & 0xffffu; L.in4 = ~u4 & ~eq4 & 0xfu; L.in3 = !u3 && !eq3; L.in2 = !u2 && !eq2; L.in1 = !u1 && !eq1;
        e5_count(L, owner2, wl);
      } else {
        C.mu = 0;  // entry masks of the Snapshot above the quads
#pragma unroll
        for (int a = 0; a < 4; a++) {
          const int2 n4 = S.l4t[a][tid];
          if (e4_longer<1>(e5_dx<FULL>(t3max, n4.x))) C.mu |= 1u << (3 - a);
          if (e4_longer<1>(e5_dn(n4.y, t3min))) C.mu |= 1u << (7 - a);
        }
        if (e4_longer<1>(e5_dx<FULL>(t2max, t3max))) C.mu |= 1u << 8;
        if (e4_longer<1>(e5_dn(t3min, t2min))) C.mu |= 1u << 9;
        if (e4_longer<1>(e5_dx<FULL>(t1max, t2max))) C.mu |= 1u << 10;
        if (e4_longer<1>(e5_dn(t2min, t1min))) C.mu |= 1u << 11;
      }
      e5_count(C, owner2, ws);  // pass 0: structure only (the masks are still empty) -> the lower bound

      // ---------------- per-warp totals and the four level-1 records go through shared memory
      if (pass == 1 && !forced) e5_tile_sync<NW>(slot);  // the other warp may still be reading the totals of pass 0
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const u32 rs = __reduce_add_sync(0xffffffffu, ws[i]);
        if (lane == 0) S.wt[warp][0][i] = rs;
        if (pass == 0) {
          const u32 rl = __reduce_add_sync(0xffffffffu, wl[i]);
          if (lane == 0) S.wt[warp][1][i] = rl;
        }
      }
      if ((lane & 15) == 0) {
        S.rec1[k1] = make_int4(t1max, t1min, diff1, eq1 ? 1 : 0);
        if (pass == 0) S.ent1[k1] = make_int2(e5_dx<FULL>(t1max, s1max), e5_dn(t1min, s1min));
      }
      e5_tile_sync<NW>(slot);  // B1

      // ---------------- root from the level-1 records, one per lane (lane 1 + k: node k; the others hold neutral values)
      {
        const int4 r = S.rec1[(lane - 1) & 3];
        n1max = is1 ? r.x : INT32_MIN; n1min = is1 ? r.y : INT32_MAX;
        n1un = e4_unif<FULL>(r.x, r.y);
        n1eq = r.w != 0;
        t0max = __reduce_max_sync(0xffffffffu, n1max);
        t0min = __reduce_min_sync(0xffffffffu, n1min);
        const int dif0 = shfl(r.z, 1);
        eq0 = __ballot_sync(0xffffffffu, is1 && n1eq && r.z == dif0) == 0x1eu;
        // bit 1 + k of a ballot -> bit 3 - k
        s_in1 = __brev(__ballot_sync(0xffffffffu, is1 && !n1un)) >> 27;
        l_in1 = __brev(__ballot_sync(0xffffffffu, is1 && !n1un && !n1eq)) >> 27;
        if (pass == 0) { const int2 e = S.ent1[(lane - 1) & 3]; l_e1max = e.x; l_e1min = e.y; }
      }
      u0 = t0max == t0min;
      l_in0 = !u0 && !eq0; s_in0 = !u0;

      // ---------------- exact size of this pass's candidate (snapshot.rs:84-93, log.rs:92-98): one stream item per lane
      const bool as_log = pass == 0;
      E5Tot Tc;
      u32 c_ntop, c_cnt;
      {
        const bool c_in0 = as_log ? l_in0 : s_in0;
        const bool c_int1 = !n1un && !(as_log && n1eq);  // own level-1 node internal
        const int ex = lane == 0 ? (as_log ? t0max - s0max : t0max) : as_log ? l_e1max : e5_dx<FULL>(t0max, n1max);
        const int en = lane == 0 ? (as_log ? t0min - s0min : t0min) : as_log ? l_e1min : e5_dn(n1min, t0min);
        const int lx = e5_len(lane == 0 || (c_in0 && is1), ex), ln = e5_len(c_in0 && (lane == 0 || (is1 && c_int1)), en);
        c_ntop = __reduce_add_sync(0xffffffffu, e5_nib(lx) | (e5_nib(ln) << 16));
        e5_totals(Tc, S, as_log ? 1 : 0, c_in0, as_log ? l_in1 : s_in1);
      }
      const u32 c_size = e5_item(c_cnt, Tc, as_log, c_ntop, lane);
      const u32 size = 13u + __reduce_add_sync(0xffffffffu, c_size);
      if (as_log) {
        T = Tc;
        ntop = c_ntop; item_cnt = c_cnt; item_size = c_size;
        log_size = size; my_size = size;
        // lower bound of the Snapshot: every entry takes at least one byte
        const u32 st = s_in0 ? S.wt[0][0][0] + S.wt[1][0][0] : 0u;
        const u32 s_upper = (s_in0 ? 1u + (u32)__popc(s_in1) : 0u) + e4_f2(st) + e4_f3(st) + e4_f4(st);
        const u32 s_int = s_upper + e4_f5(st), s_nm = 1u + 4u * s_upper, s_nmax = 1u + 4u * s_int;
        const u32 snap_lb = 13u + bitmap_size(s_nm) + 1u + bitmap_size(s_nmax) + s_nmax + (s_int ? 1u + bitmap_size(s_int) + s_int : 1u);
        if (!(snap_lb <= log_size)) break;  // the Log wins without looking closer
      } else {
        as_snapshot = forced || size <= log_size;  // ties go to the snapshot (chunk.rs:62)
        if (as_snapshot) { T = Tc; ntop = c_ntop; item_cnt = c_cnt; item_size = c_size; my_size = size; }
      }
    }

    // ---------------- the winner, generic from here on
    E5Cand W;
    W.in5 = as_snapshot ? C.in5 : L.in5; W.in4 = as_snapshot ? C.in4 : L.in4;
    W.in3 = as_snapshot ? C.in3 : L.in3; W.in2 = as_snapshot ? C.in2 : L.in2; W.in1 = as_snapshot ? C.in1 : L.in1;
    W.ml = as_snapshot ? C.ml : L.ml; W.mq = as_snapshot ? C.mq : L.mq; W.mu = as_snapshot ? C.mu : L.mu;
    const int e1x = as_snapshot ? e5_dx<FULL>(t0max, n1max) : l_e1max, e1n = as_snapshot ? e5_dn(n1min, t0min) : l_e1min;
    const int e0x = as_snapshot ? t0max : t0max - s0max, e0n = as_snapshot ? t0min : t0min - s0min;
    const u32 nm_len = T.nm_len, n_int = T.n_int, I0 = T.I0, I1 = T.I1;
    const bool in0 = as_snapshot ? s_in0 : l_in0;
    const u32 in1m = as_snapshot ? s_in1 : l_in1;
    const int cand = as_snapshot ? 0 : 1;
    // this warp's share of the root / level-1 entries: warp 0 the max DAC, warp 1 the min DAC (lane j = entry j); the
    // warp of a one-warp tile takes both (top[0] max, top[1] min)
    constexpr int NTOP = 3 - NW;
    E5Top top[NTOP];
    const u32 lt = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < NTOP; r++) {
      const bool mn = NW == 2 ? warp == 1 : r == 1;
      const bool valid = mn ? (in0 && (lane == 0 || (is1 && !n1un && !(!as_snapshot && n1eq)))) : (lane == 0 || (in0 && is1));
      const int e = lane == 0 ? (mn ? e0n : e0x) : (mn ? e1n : e1x);
      top[r].z = zigzag32(e);
      top[r].len = e5_len(valid, e);
      top[r].pos0 = (u32)__popc(__ballot_sync(0xffffffffu, top[r].len > 0) & lt);
      top[r].pos1 = (u32)__popc(__ballot_sync(0xffffffffu, top[r].len > 1) & lt);
    }
    const bool staged = my_size <= stage_limit;
    // The piece's place in the arena: the atomic's round trip is long, so a staged structure only looks at the answer
    // when its image is complete (a warp stalls at the first instruction that needs a pending result).
    u64 my_off = 0;
    auto publish_piece = [&]() {
      S.piece_off = my_off;
      Piece pc;
      pc.off = my_off; pc.size = my_size; pc.kind = as_snapshot ? 1u : 0u;
      P.pieces[unit.piece_base + inst] = pc;
    };
    if (tid == 0) {
      const u64 need = ((u64)my_size + 15ull) & ~15ull;
      my_off = atomicAdd(P.arena_head, (unsigned long long)need);
      if (!staged) publish_piece();
    }
    // stream layout (snapshot.rs:48-58 / log.rs:53-64, dac.rs:37-44): where each lane's item (e5_item) starts; a DAC
    // level's bitmap header sits at item_hdr, its bytes at item_at
    const u32 item_hdr = 13u + e4_warp_excl(item_size, lane) + ((lane == 2 || lane == 6) ? 1u : 0u);
    const u32 item_at = item_hdr + (item_cnt ? bitmap_size(item_cnt) : 0u);
    const u32 eq_len = nm_len - n_int;
    const u32 nm_hdr = 13u;
    const u32 eq_hdr = nm_hdr + bitmap_size(nm_len);
    const u32 x_hdr0 = shfl(item_hdr, 2), x_at0 = shfl(item_at, 2), x_at1 = shfl(item_at, 3);
    const u32 n_hdr0 = shfl(item_hdr, 6), n_at0 = shfl(item_at, 6), n_at1 = shfl(item_at, 7);
    const u32 lv = __ballot_sync(0xffffffffu, item_cnt != 0u);
    const u32 x_levels = (u32)__popc(lv & 0x3cu), n_levels = (u32)__popc(lv & 0x3c0u);
    // the image starts `shift` bytes into the pool so that entry 1 of the max DAC's level 0 is 4-byte aligned
    const u32 shift = staged ? ((4u - ((x_at0 + 1u) & 3u)) & 3u) : 0u;
    if (!staged) e5_tile_sync<NW>(slot);
    u64 piece_off = 0;
    bool fits = true;
    if (!staged) {
      piece_off = S.piece_off;
      fits = piece_off + (((u64)my_size + 15ull) & ~15ull) <= P.arena_cap;
      if (!fits) err |= EF_ARENA_FULL;
      if (fits) {
        uint4* z = reinterpret_cast<uint4*>(P.arena + piece_off);
        for (u32 i = tid; i < (my_size + 15u) / 16u; i += TT) z[i] = make_uint4(0, 0, 0, 0);
      }
      e5_tile_sync<NW>(slot);
    }
    const bool emit = staged || fits;

    // Everything that touches the image, once for the shared-memory image (the compiler then knows the address space of
    // every pointer: 32-bit addressing, shared-memory reductions) and once for a structure too large for it, emitted
    // straight into its zeroed piece of the arena.
    auto emission = [&](auto in_shared) {
    u8* const out = decltype(in_shared)::value ? S.pool + shift : P.arena + piece_off;
    u8* const nm_words = e4_words_of(out, nm_hdr, nm_len);
    u8* const eq_words = e4_words_of(out, eq_hdr, eq_len);
    u8* const xw0 = e4_words_of(out, x_hdr0, 1u + 4u * n_int);  // continuation bits of DAC level 0
    u8* const nw0 = e4_words_of(out, n_hdr0, n_int);
    u8* const xb0 = out + x_at0;
    u8* const xb1 = out + x_at1;
    u8* const nb0 = out + n_at0;
    u8* const nb1 = out + n_at1;

    // block-wide positions
    const u32 T0 = T.tot[0];
    const u32 I2 = e4_f2(T0), I3 = e4_f3(T0), I4 = e4_f4(T0);
    const u32 Pn2 = 1u + 4u * I0, Pn3 = Pn2 + 4u * I1, Pn4 = Pn3 + 4u * I2, Pn5 = Pn4 + 4u * I3, Pn6 = Pn5 + 4u * I4;
    const u32 Mn2 = I0 + I1, Mn3 = Mn2 + I2, Mn4 = Mn3 + I3, Mn5 = Mn4 + I4;
    const u32 R1 = (u32)__popc(in1m >> (4 - k1));  // internal level-1 nodes before the own one
    const bool x2 = in0 && ((in1m >> (3 - k1)) & 1u);
    const bool x3 = x2 && W.in2, x4 = x3 && W.in3;
    const u32 ai4 = x4 ? W.in4 : 0u;
    const u32 X5 = e4_expand4(ai4);
    const u32 ai5 = W.in5 & X5;
    // prefix over earlier threads (Morton order) of the packed counters
    u32 pre[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      pre[i] = 0;
      if (i == 0 || T.tot[i] != 0)  // tile-uniform: without two-byte entries there is nothing to scan
        pre[i] = e4_warp_excl(as_snapshot ? ws[i] : wl[i], lane) + ((warp == 1 && in0) ? S.wt[0][cand][i] : 0u);
    }
    const u32 R2own = e4_f2(pre[0]);                       // internal level-2 nodes before the own group (valid on owner lanes)
    const u32 R2p = e4_f2(shfl(pre[0], lane & ~3));        // the same, seen by every lane of the group
    const u32 R3 = e4_f3(pre[0]), R4 = e4_f4(pre[0]), R5 = e4_f5(pre[0]);
    // positions of this thread's second bytes (DAC level 1) per tree level: entries longer than one byte before them
    const u32 tx = T.tot[1], tn = T.tot[3];
    const u32 bx2 = (ntop >> 4) & 0xfu, bx3 = bx2 + e4_f2(tx), bx4 = bx3 + e4_f3(tx), bx5 = bx4 + e4_f4(tx), bx6 = bx5 + e4_f5(tx);
    const u32 bn2 = (ntop >> 20) & 0xfu, bn3 = bn2 + e4_f2(tn), bn4 = bn3 + e4_f3(tn), bn5 = bn4 + e4_f4(tn);
    // log "equal" flags of nodes that are neither uniform nor internal
    const u32 eqb5 = ~u5 & eq5 & 0xffffu, eqb4 = ~u4 & eq4 & 0xfu;
    const bool eqb3 = !u3 && eq3, eqb2 = !u2 && eq2;

    if (emit) {
      // ================= phase A: every bitmap bit (OR of runs; no byte store is in flight) =================
      {  // quads and leaves
        const u32 mqn = (W.mq >> 16) & ai5;
        if ((W.ml != 0) | (mqn != 0)) {  // some leaf or quad-min entry takes two bytes: compress their flags
          u64 accL = 0; int nL = 0;
          u32 accM = 0; int nM = 0;
#pragma unroll 1
          for (int bit = 15; bit >= 0; bit--) {  // quad q = 15 - bit
            if ((ai5 >> bit) & 1u) {
              accL = (accL << 4) | ((W.ml >> (4 * bit)) & 0xfull); nL += 4;
              accM = (accM << 1) | ((mqn >> bit) & 1u); nM += 1;
            }
          }
          if (nL) e5_or_run(xw0, Pn6 + 4u * R5, accL << (64 - nL));
          e5_or_bits(nw0, Mn5 + R5, accM, nM);
        }
        if (!as_snapshot) {
          // `equal` flags of the quads that exist but are not internal, in quad order
          const u32 sel = X5 & ~ai5 & 0xffffu;
          u32 m = eqb5 & sel, accE = 0;
          const int nE = __popc(sel);
          while (m) {
            const int b = 31 - __clz((int)m);
            m ^= 1u << b;
            accE |= 1u << (nE - 1 - __popc(sel >> (b + 1)));
          }
          e5_or_bits(eq_words, (Pn5 - Mn5) + 4u * R4 - R5, accE, nE);
        }
        u32 accN = 0, accC = 0; int nN = 0;
#pragma unroll
        for (int a = 0; a < 4; a++) {
          if ((ai4 >> (3 - a)) & 1u) {
            accN = (accN << 4) | ((W.in5 >> (12 - 4 * a)) & 0xfu);
            accC = (accC << 4) | ((W.mq >> (12 - 4 * a)) & 0xfu);
            nN += 4;
          }
        }
        e5_or_bits(nm_words, Pn5 + 4u * R4, accN, nN);
        e5_or_bits(xw0, Pn5 + 4u * R4, accC, nN);
      }
      if (x4) {  // the four level-4 nodes
        e5_or_bits(nm_words, Pn4 + 4u * R3, W.in4, 4);
        e5_or_bits(xw0, Pn4 + 4u * R3, W.mu & 0xfu, 4);
        u32 accM = 0, accE = 0; int nM = 0, nE = 0;
#pragma unroll
        for (int a = 0; a < 4; a++) {
          if ((W.in4 >> (3 - a)) & 1u) { accM = (accM << 1) | ((W.mu >> (7 - a)) & 1u); nM++; }
          else { accE = (accE << 1) | ((eqb4 >> (3 - a)) & 1u); nE++; }
        }
        e5_or_bits(nw0, Mn4 + R4, accM, nM);
        if (!as_snapshot) e5_or_bits(eq_words, (Pn4 - Mn4) + 4u * R3 - R4, accE, nE);
      }
      if (x3) {  // own level-3 node
        const u32 pos = Pn3 + 4u * R2p + (u32)(node & 3);
        if (W.in3) {
          e5_or_bit(nm_words, pos);
          if ((W.mu >> 9) & 1u) e5_or_bit(nw0, Mn3 + R3);
        } else if (!as_snapshot && eqb3) {
          e5_or_bit(eq_words, pos - (Mn3 + R3));
        }
        if ((W.mu >> 8) & 1u) e5_or_bit(xw0, pos);
      }
      if (x2 && owner2) {  // level-2 node of the group
        const u32 pos = Pn2 + 4u * R1 + (u32)((node >> 2) & 3);
        if (W.in2) {
          e5_or_bit(nm_words, pos);
          if ((W.mu >> 11) & 1u) e5_or_bit(nw0, Mn2 + R2own);
        } else if (!as_snapshot && eqb2) {
          e5_or_bit(eq_words, pos - (Mn2 + R2own));
        }
        if ((W.mu >> 10) & 1u) e5_or_bit(xw0, pos);
      }
      // root and level-1 nodes, lane 0 = root, lane 1 + k = node k.  Continuation bits of their DAC entries: warp 0
      // takes the max DAC, warp 1 the min DAC
#pragma unroll
      for (int r = 0; r < NTOP; r++) {
        const bool mx = NW == 2 ? warp == 0 : r == 0;
        if (top[r].len > 1) e5_or_bit(mx ? xw0 : nw0, top[r].pos0);
        if (__any_sync(0xffffffffu, top[r].len > 2)) e5_top_long(false, out, top[r], mx ? 2 : 6, item_hdr, item_cnt, item_at);
      }
      // ... their nodemap and `equal` bits; a level-1 node's `equal` bit comes after those of the non-internal ones before it
      if (warp == NW - 1) {
        if (lane == 0) {
          if (in0) e5_or_bits(nm_words, 0, 0x10u | in1m, 5);
          else if (!as_snapshot && !u0 && eq0) e5_or_bit(eq_words, 0);
        } else if (is1 && in0 && !as_snapshot && !n1un && n1eq) {
          e5_or_bit(eq_words, (u32)(lane - 1 - __popc(in1m >> (5 - lane))));
        }
      }
    }
    e5_tile_sync<NW>(slot);  // B2a: all word-wide ORs done before the first byte store

    // ================= phase B: DAC bytes =================
    {
      u32 pos[3] = {bx6 + pre[2], bx5 + e4_f5(pre[1]), bn5 + e4_f5(pre[3])};  // lx1, rx1, rn1: second bytes of leaves / quad max / quad min
      u8* dst6 = xb0 + Pn6 + 4u * R5;
      u8* dst5 = xb0 + Pn5 + 4u * R4;
      u8* dmn = nb0 + Mn5 + R5;
      uint4 raw[4];
      if (as_snapshot) e5_load_node<FULL>(e5_node_ptr(pt, sr, 0), sr, raw, E5_RL(0), E5_CL(0), vec);
#pragma unroll 1
      for (int a = 0; a < 4; a++) {
        const int2 n4 = S.l4t[a][tid];
        const u32 in5a = (W.in5 >> (12 - 4 * a)) & 0xfu;
        const bool alive = emit && ((ai4 >> (3 - a)) & 1u);
        u32 zxw, znw;
        if (as_snapshot) {
          // quads and leaves of the Snapshot from a pass over the tile, which also installs the instant as the snapshot
          // image the following Logs are built against (even when nothing can be emitted: the sizes must stay exact)
          int4 q[4];
          e5_quads<FULL>(raw, scale2, q, E5_RL(a), E5_CL(a));
          if (a < 3) e5_load_node<FULL>(e5_node_ptr(pt, sr, a + 1), sr, raw, E5_RL(a + 1), E5_CL(a + 1), vec);
          S.l4s[a][tid] = n4;
          zxw = 0; znw = 0;
#pragma unroll
          for (int b = 0; b < 4; b++) {
            const int4 t = q[b];
            S.cell[4 * a + b][tid] = t;
            int qmax, qmin;
            e4_qmm<FULL>(t, qmax, qmin);
            zxw |= (zigzag32(e5_dx<FULL>(n4.x, qmax)) & 0xffu) << (8 * b);
            znw |= (zigzag32(e5_dn(qmin, n4.y)) & 0xffu) << (8 * b);
            if (alive && ((in5a >> (3 - b)) & 1u))
              e5_store_word<decltype(in_shared)::value>(dst6 + 4u * (u32)__popc(in5a >> (4 - b)),
                            e5_pack4(zigzag32(e5_dx<FULL>(qmax, t.x)), zigzag32(e5_dx<FULL>(qmax, t.y)), zigzag32(e5_dx<FULL>(qmax, t.z)),
                                     zigzag32(e5_dx<FULL>(qmax, t.w))));
          }
        } else {
          // quads and leaves of the Log from the payload of the fused pass
          zxw = S.qx[a][tid]; znw = S.qn[a][tid];
          if (alive) {
#pragma unroll
            for (int b = 0; b < 4; b++)
              if ((in5a >> (3 - b)) & 1u) e5_store_word<decltype(in_shared)::value>(dst6 + 4u * (u32)__popc(in5a >> (4 - b)), S.leaf[4 * a + b][tid]);
          }
        }
        if (!alive) continue;
        e5_store_word<decltype(in_shared)::value>(dst5, zxw);
        dst5 += 4;
        dst6 += 4u * (u32)__popc(in5a);
#pragma unroll
        for (int b = 0; b < 4; b++)
          if ((in5a >> (3 - b)) & 1u) *dmn++ = (u8)(znw >> (8 * b));
        const u32 ml16 = (u32)(W.ml >> (48 - 16 * a)) & 0xffffu;
        const u32 lq = ((W.mq >> (12 - 4 * a)) & 0xfu) | (((W.mq >> (28 - 4 * a)) & 0xfu) & in5a);
        if ((ml16 & (e4_expand4(in5a) & 0xffffu)) | lq)
          e5_long_node<FULL, TT>(as_snapshot, e5_node_ptr(pt, sr, a), sr, scale2, &S.cell[4 * a][tid], n4, in5a, xb1, nb1, pos, E5_RL(a), E5_CL(a), vec);
      }
    }
    if (emit) {
      if (x4) {  // ---- level-4 nodes
        u32 rx1 = bx4 + e4_f4(pre[1]), rn1 = bn4 + e4_f4(pre[3]);
        u32 zx[4], zn[4];
#pragma unroll
        for (int a = 0; a < 4; a++) {
          const int2 n4 = S.l4t[a][tid];
          // the Snapshot pass has already installed l4s = l4t, and a Snapshot's entries do not refer to it
          const int2 s4 = as_snapshot ? make_int2(0, 0) : S.l4s[a][tid];
          zx[a] = zigzag32(as_snapshot ? e5_dx<FULL>(t3max, n4.x) : e5_dx<FULL>(n4.x, s4.x));
          zn[a] = zigzag32(as_snapshot ? e5_dn(n4.y, t3min) : e5_dn(n4.y, s4.y));
        }
        e5_store_word<decltype(in_shared)::value>(xb0 + Pn4 + 4u * R3, e5_pack4(zx[0], zx[1], zx[2], zx[3]));
        u8* dmn = nb0 + Mn4 + R4;
        if (W.mu & 0xffu) {
#pragma unroll
          for (int a = 0; a < 4; a++)
            if (zx[a] > 0xffu) rx1 = e5_hi(xb1, zx[a], rx1);
        }
#pragma unroll
        for (int a = 0; a < 4; a++) {
          if ((W.in4 >> (3 - a)) & 1u) {
            *dmn++ = (u8)zn[a];
            if (zn[a] > 0xffu) rn1 = e5_hi(nb1, zn[a], rn1);
          }
        }
      }
      if (x3) {
        const u32 zx = zigzag32(as_snapshot ? e5_dx<FULL>(t2max, t3max) : e5_dx<FULL>(t3max, s3max));
        xb0[Pn3 + 4u * R2p + (u32)(node & 3)] = (u8)zx;
        if (zx > 0xffu) e5_hi(xb1, zx, bx3 + e4_f3(pre[1]));
        if (W.in3) {
          const u32 zn = zigzag32(as_snapshot ? e5_dn(t3min, t2min) : e5_dn(t3min, s3min));
          nb0[Mn3 + R3] = (u8)zn;
          if (zn > 0xffu) e5_hi(nb1, zn, bn3 + e4_f3(pre[3]));
        }
      }
      if (x2 && owner2) {
        const u32 zx = zigzag32(as_snapshot ? e5_dx<FULL>(t1max, t2max) : e5_dx<FULL>(t2max, s2max));
        xb0[Pn2 + 4u * R1 + (u32)((node >> 2) & 3)] = (u8)zx;
        if (zx > 0xffu) e5_hi(xb1, zx, bx2 + e4_f2(pre[1]));
        if (W.in2) {
          const u32 zn = zigzag32(as_snapshot ? e5_dn(t2min, t1min) : e5_dn(t2min, s2min));
          nb0[Mn2 + R2own] = (u8)zn;
          if (zn > 0xffu) e5_hi(nb1, zn, bn2 + e4_f2(pre[3]));
        }
      }
#pragma unroll
      for (int r = 0; r < NTOP; r++) {  // root and level-1 entries (any length): the same lanes as in phase A
        const bool mx = NW == 2 ? warp == 0 : r == 0;
        if (top[r].len > 0) (mx ? xb0 : nb0)[top[r].pos0] = (u8)top[r].z;
        if (top[r].len > 1) (mx ? xb1 : nb1)[top[r].pos1] = (u8)(top[r].z >> 8);
        if (__any_sync(0xffffffffu, top[r].len > 2)) e5_top_long(true, out, top[r], mx ? 2 : 6, item_hdr, item_cnt, item_at);
      }
      if ((NW == 1 || warp == 1) && lane >= 16) {  // structure header (snapshot.rs:48-52 / log.rs:53-58): k, shape, sidelen; DAC level counts
        const u32 i = lane - 16u;
        if (i < 13u) {
          const u32 word = i < 5u ? (u32)unit.rows : i < 9u ? (u32)unit.cols : 64u;
          out[i] = i == 0 ? (u8)2 : (u8)(word >> (8u * ((12u - i) & 3u)));
        } else if (i == 13u) {
          out[x_hdr0 - 1] = (u8)x_levels;
        } else if (i == 14u) {
          out[n_hdr0 - 1] = (u8)n_levels;
        }
      }
    }
    e5_tile_sync<NW>(slot);  // B2
    // BULK: nobody reads the staged tile any more -> the next instant's rows start coming in behind the rank directories
    if (BULK && inst + 1 < unit.instants) fetch_instant(inst + 1);

    if (emit) {
      // ================= bitmap headers and rank directories: index[b] = ones in bits [0, 128(b+1))  (bitmap.rs:97-104)
      // bitmaps in stream order: nodemap, equal (Logs), the levels of the max DAC, the levels of the min DAC
      const u32 n_fix = as_snapshot ? 1u : 2u;
      const u32 n_bm = n_fix + x_levels + n_levels;
#pragma unroll 1
      for (u32 i = warp; i < n_bm; i += NW) {
        // the lane that holds bitmap i: nodemap, `equal`, then the max DAC's levels from lane 2, the min DAC's from lane 6
        const int src = (int)(i < n_fix ? i : i < n_fix + x_levels ? 2u + (i - n_fix) : 6u + (i - n_fix - x_levels));
        const u32 hdr = shfl(item_hdr, src), len = shfl(item_cnt, src);
        if (lane == 0) {
          store_be32(out + hdr, len);
          store_be32(out + hdr + 4, 4u);  // k = 4 (bitmap.rs:69)
        }
        const u32 blocks = len >> 7;
        u8* const index = out + hdr + 8u;
        const u8* const words = index + 4u * blocks;
        u32 carry = 0;
#pragma unroll 1
        for (u32 b0 = 0; b0 < blocks; b0 += 32u) {
          const u32 b = b0 + lane;
          u32 c = b < blocks ? e4_popc_bytes16(words + 16u * b) : 0u;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const u32 n = __shfl_up_sync(0xffffffffu, c, d);
            if (lane >= d) c += n;
          }
          if (b < blocks) e4_store_be32(index + 4u * b, carry + c);
          carry += shfl(c, 31);
        }
      }
    }
    if (decltype(in_shared)::value && tid == 0) publish_piece();
    e5_tile_sync<NW>(slot);  // B3

    // ================= copy-out (re-aligning by `shift` bytes) and re-zero the image =================
    if constexpr (decltype(in_shared)::value) {
      piece_off = S.piece_off;
      fits = piece_off + (((u64)my_size + 15ull) & ~15ull) <= P.arena_cap;
      if (!fits) err |= EF_ARENA_FULL;
      u32* src = reinterpret_cast<u32*>(S.pool);
      uint4* dst = reinterpret_cast<uint4*>(P.arena + piece_off);
      const u32 sh = 8u * shift;
      const u32 n16 = (my_size + 15u) / 16u;
#pragma unroll 1
      for (u32 i = tid; i < n16; i += TT) {
        const uint4 v = *reinterpret_cast<const uint4*>(src + 4u * i);
        const u32 nx = src[4u * i + 4u];
        uint4 o;
        o.x = __funnelshift_r(v.x, v.y, sh); o.y = __funnelshift_r(v.y, v.z, sh);
        o.z = __funnelshift_r(v.z, v.w, sh); o.w = __funnelshift_r(v.w, nx, sh);
        if (fits) dst[i] = o;
      }
      e5_tile_sync<NW>(slot);  // every word has been read (a chunk's last word belongs to the next one's first)
#pragma unroll 1
      for (u32 i = tid; i < n16 + 1u; i += TT) *reinterpret_cast<uint4*>(src + 4u * i) = make_uint4(0, 0, 0, 0);
    }

    };
    if (staged) emission(std::true_type{});
    else emission(std::false_type{});

    // ---------------- bookkeeping: start a new block or extend the current one
    if (as_snapshot) {
      s3max = t3max; s3min = t3min; s2max = t2max; s2min = t2min; s1max = t1max; s1min = t1min; s0max = t0max; s0min = t0min;
      n_snap++;
      n_logs = 0;
      total_bytes += 1;  // Block's n_instants byte (block.rs:88-95)
    } else {
      n_logs++;
      n_log_total++;
    }
    total_bytes += my_size;
  }

  if (tid == 0 && tile_live) {
    UnitResult r;
    r.bytes = total_bytes + 6;  // encoding + fractional_bits + n_blocks (chunk.rs:235-243)
    r.snapshots = n_snap;
    r.logs = n_log_total;
    P.results[unit_idx] = r;
  }
  err = __reduce_or_sync(0xffffffffu, err);
  if (lane == 0 && err) atomicOr(P.err, err);
#undef E5_RL
#undef E5_CL
}

}  // namespace dcdf
