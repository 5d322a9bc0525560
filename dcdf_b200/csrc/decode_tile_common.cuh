// decode_tile_common.cuh -- pieces shared by the tile decoders (decode_tile4.cuh: windows, decode_search4.cuh:
// value-range search) for trees up to 64x64: constants, output conversion (from_fixed, fixed.rs:81-86), cp.async
// staging, four-entry DAC / bitmap fetches for the children of one node (their BFS indices are consecutive:
// 1 + 4 * rank(idx) .. + 3, snapshot.rs:177), the window-clipped quad writer.
#pragma once
#include <type_traits>

#include "decode.cuh"

namespace dcdf {

constexpr int DT_THREADS = 256;
constexpr int DT_WARPS = DT_THREADS / 32;
constexpr int DT_NODES = 5461;
constexpr int DT_UPPER = 1365;

DCDF_DEVINL u32 lvl_off(int k) { return (0x55555555u >> (32 - 2 * k)) & (k ? 0xffffffffu : 0u); }  // (4^k - 1) / 3

// Output of one cell: raw fixed point, or the chunk's own encoding with from_fixed applied to floats (fixed.rs:81-86;
// the divide by 2^(bits+1) is an exact scaling, done as a multiply by the exact reciprocal).
struct CellOut {
  void* out;
  int kind;  // 0: i64 (raw / ENC_I64), 1: i32, 2: f32, 3: f64
  float inv32;
  double inv64;
  DCDF_DEVINL void init(const QuerySet& Q, void* out_, int raw, int bits) {
    out = out_;
    kind = (raw || Q.encoding == 8) ? 0 : Q.encoding == 4 ? 1 : Q.encoding == 32 ? 2 : 3;
    inv32 = __int_as_float((126 - bits) << 23);                          // 2^-(bits+1)
    inv64 = __longlong_as_double((long long)(1022 - bits) << 52);
  }
  // 32-bit values (narrow expansion): the same conversions without 64-bit arithmetic
  DCDF_DEVINL void put(u64 i, int32_t fixed) const {
    if (kind == 2) static_cast<float*>(out)[i] = fixed == 0 ? __int_as_float(0x7fc00000) : __int2float_rn(fixed - 1) * inv32;
    else if (kind == 0) static_cast<i64*>(out)[i] = (i64)fixed;
    else if (kind == 1) static_cast<int32_t*>(out)[i] = fixed;
    else static_cast<double*>(out)[i] = fixed == 0 ? __longlong_as_double(0x7ff8000000000000ll) : __int2double_rn(fixed - 1) * inv64;
  }
  DCDF_DEVINL void put(u64 i, i64 fixed) const {
    if (kind == 2) static_cast<float*>(out)[i] = fixed == 0 ? __int_as_float(0x7fc00000) : __ll2float_rn(fixed - 1) * inv32;
    else if (kind == 0) static_cast<i64*>(out)[i] = fixed;
    else if (kind == 1) static_cast<int32_t*>(out)[i] = (int32_t)fixed;
    else static_cast<double*>(out)[i] = fixed == 0 ? __longlong_as_double(0x7ff8000000000000ll) : __ll2double_rn(fixed - 1) * inv64;
  }
};

// Window statistics (dcdf_superchunk_window_stats): the reduction of one (window, subchunk, instant).  min / max are codes
// at `bits` (from_fixed is monotone in the code at fixed bits, so they are compared as codes inside a tile and as values
// across tiles); sum / sum_sq are in the array's units.  count == 0: min / max are meaningless, the sums 0.
struct StatsPartial {
  u32 count;
  int bits;
  i64 min, max;
  double sum, sum_sq;
};
static_assert(sizeof(StatsPartial) == 40, "StatsPartial is 40 bytes");

// Per-cell statistics over time (dcdf_superchunk_time_stats): the reduction of one cell over one piece -- the window's
// instants inside one time slice.  min / max are values of the encoding (f for f32 / f64, i for i32 / i64; subchunk bits
// differ per slice, so codes could not be compared later); sum / sum_sq are ((0 + v_0) + v_1) + ... in double, in time
// order.  count == 0: min / max are meaningless, the sums 0.
union TimeVal {
  i64 i;
  double f;
};
struct TimePartial {
  u32 count, n_band;
  TimeVal min, max;
  double sum, sum_sq;
};
static_assert(sizeof(TimePartial) == 40, "TimePartial is 40 bytes");

struct TileWindowParams {
  QuerySet Q;
  const CubeDev* cubes;   // validated, ordered
  const u64* out_off;     // [n] element offsets
  const u64* job_base;    // [n + 1] prefix of (slices x subchunks) per window
  u64 n_queries, n_jobs;
  void* out;
  int raw;
  // window statistics: partial of (window q, subchunk sub, instant t) at part[part_base[q] + sub * (end - start) + t - start]
  const u64* part_base;
  StatsPartial* part;
  // time statistics: partial of (window q, k-th slice of the window, cell) at tpart[part_base[q] + k * area + cell], cells
  // row-major; band[2q], band[2q + 1]: the window's ordered band (nullptr: no band)
  TimePartial* tpart;
  const double* band;
};

// One job of k_window_tiles4: window q, one time slice [t_lo, t_hi), the subchunk `sub` (row-major among those the window
// touches) whose tile starts at (chunk_top, chunk_left); the window clipped to the tile in tile coordinates.
struct TileJob {
  CubeDev c;
  u64 q, sub;
  i64 chunk_top, chunk_left, t_lo, t_hi;
  int top, bottom, left, right;
};

constexpr u32 W3_NONE = 0xffffffffu;
constexpr int W3_UPPER = DT_UPPER + 3;  // levels above the cells, level k >= 1 at (4^k - 1) / 3 + 3 (16-byte aligned groups)
constexpr int W3_DIRW = (int)(sizeof(InstDir) / 4);

DCDF_DEVINL u32 off3(int k) { return k ? lvl_off(k) + 3u : 0u; }

DCDF_DEVINL void cp_async16(void* smem, const void* g) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((u32)__cvta_generic_to_shared(smem)), "l"(g) : "memory");
}
DCDF_DEVINL void cp_async4(void* smem, const void* g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((u32)__cvta_generic_to_shared(smem)), "l"(g) : "memory");
}
DCDF_DEVINL void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Level 0 of a DAC (bytes + continuation bits) with the general accessor for longer codes.
struct Dac4 {
  const u8* bytes0;
  const u8* more0;
  const u8* chunk;
  const DacDir* d;
  u32 len0;
};
DCDF_DEVINL Dac4 dac4_of(const u8* chunk, const DacDir* d) {
  const u32 len = d->len[0], base = d->base[0];
  const u32 words = base + 8u + 4u * (len / 128u);
  return Dac4{chunk + words + 4u * ((len + 31u) / 32u), chunk + words, chunk, d, d->n_levels ? len : 0u};
}
// codes longer than one byte: out of line, they are rare and the rank loop would be inlined a dozen times
__device__ __noinline__ i64 dac_slow_get(const u8* chunk, const DacDir* d, u32 idx) { return DacRef{chunk, d}.get(idx); }
template <typename V>
DCDF_DEVINL V unzz8(u32 b) { return (V)(int)((b >> 1) ^ (0u - (b & 1u))); }
template <typename V>
DCDF_DEVINL V dac_get1(const Dac4& m, u32 idx) {  // dac.rs:80-93
  if (idx >= m.len0) return (V)0;
  if (!((m.more0[idx >> 3] >> (7u - (idx & 7u))) & 1u)) return unzz8<V>(m.bytes0[idx]);
  return (V)dac_slow_get(m.chunk, m.d, idx);
}
// entries idx .. idx + 3 (the children of one node); anything but four one-byte codes goes out of line
template <typename V>
struct __align__(16) Quad { V c[4]; };
struct __align__(16) Quad32 { u32 c[4]; };
template <typename V>
__device__ __noinline__ Quad<V> dac_get4_slow(const u8* chunk, const DacDir* d, u32 idx) {
  Quad<V> q;
#pragma unroll 1
  for (int i = 0; i < 4; i++) {
    const V v = (V)DacRef{chunk, d}.get(idx + (u32)i);  // an empty DAC or an index past its end yields 0
    if (i == 0) q.c[0] = v; else if (i == 1) q.c[1] = v; else if (i == 2) q.c[2] = v; else q.c[3] = v;
  }
  return q;
}
// Four consecutive entries idx .. idx + 3 <= len0 of which some are longer than one byte (nib: continuation bits of
// level 0, bit 3 = entry idx).  The entries that continue sit next to each other on the next level as well, so every
// level costs ONE rank over the serialized directory (bitmap.rs:186-212) for the whole group, not one per entry
// (dac.rs:80-93 per entry would).
template <typename V>
__device__ __noinline__ Quad<V> dac_get4_multi(const u8* chunk, const DacDir* d, u32 idx, u32 nib) {
  u64 n0, n1, n2, n3;
  {
    const u32 len = d->len[0], words = d->base[0] + 8u + 4u * (len / 128u);
    const u8* b = chunk + words + 4u * ((len + 31u) / 32u) + idx;
    n0 = b[0]; n1 = b[1]; n2 = b[2]; n3 = b[3];
  }
  u32 cont = nib & 15u;  // bit 3 - i: entry i continues on the next level
  u32 p = idx;           // position of the group's first entry on the current level
  const u32 nl = d->n_levels;
#pragma unroll 1
  for (u32 j = 1; j < nl && cont; j++) {
    const BitMapRef up{chunk, d->len[j - 1], d->base[j - 1]};
    // the first continuing entry of the group sits at p + (entries before it that stopped); ones before it = ones before p
    // only if nothing between p and it is set, which holds: the entries in between did not continue
    const u32 r = up.rank(p);
    const u32 len = d->len[j], words = d->base[j] + 8u + 4u * (len / 128u);
    const u8* bytes = chunk + words + 4u * ((len + 31u) / 32u);
    const u8* more = chunk + words;
    const bool last = j + 1u >= nl;
    u32 next = 0, k = 0;
    const u32 sh = 8u * j;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if ((cont >> (3 - i)) & 1u) {
        const u32 pos = r + k;
        k++;
        if (pos < len) {  // malformed input guard
          const u64 byte = bytes[pos];
          if (i == 0) n0 |= byte << sh; else if (i == 1) n1 |= byte << sh; else if (i == 2) n2 |= byte << sh; else n3 |= byte << sh;
          if (!last && ((more[pos >> 3] >> (7u - (pos & 7u))) & 1u)) next |= 1u << (3 - i);
        }
      }
    }
    cont = next;
    p = r;
  }
  Quad<V> q;
  q.c[0] = (V)unzigzag64(n0); q.c[1] = (V)unzigzag64(n1); q.c[2] = (V)unzigzag64(n2); q.c[3] = (V)unzigzag64(n3);
  return q;
}
template <typename V>
DCDF_DEVINL void dac_get4(const Dac4& m, u32 idx, V (&d)[4]) {
  u32 nib = 1;
  if (idx + 4u <= m.len0) {
    const u32 by = idx >> 3;
    const u32 hw = ((u32)m.more0[by] << 8) | (u32)m.more0[by + 1];  // the byte after the bitmap is the DAC's first code
    nib = (hw >> (12u - (idx & 7u))) & 15u;
  }
  if (nib == 0) {
    const u8* b = m.bytes0 + idx;
#pragma unroll
    for (int i = 0; i < 4; i++) d[i] = unzz8<V>(b[i]);
  } else {
    const Quad<V> q = idx + 4u <= m.len0 ? dac_get4_multi<V>(m.chunk, m.d, idx, nib) : dac_get4_slow<V>(m.chunk, m.d, idx);
#pragma unroll
    for (int i = 0; i < 4; i++) d[i] = q.c[i];
  }
}
DCDF_DEVINL bool bit_at(const u8* bits, u32 i) { return (bits[i >> 3] >> (7u - (i & 7u))) & 1u; }
DCDF_DEVINL const u8* bitmap_bits(const u8* chunk, u32 len, u32 base) { return chunk + base + 8u + 4u * (len / 128u); }
// bits idx .. idx + 3 of an MSB-first bit stream as a mask (bit c = stream bit idx + c); positions >= len read as 0
DCDF_DEVINL u32 bits4(const u8* bits, u32 len, u32 idx) {
  const u32 by = idx >> 3;
  const u32 hw = ((u32)bits[by] << 8) | (u32)bits[by + 1];
  u32 nib = __brev((hw >> (12u - (idx & 7u))) & 15u) >> 28;
  if (idx + 4u > len) nib &= idx >= len ? 0u : (1u << (len - idx)) - 1u;
  return nib;
}

DCDF_DEVINL u32 below(u32 inb, int c) { return __popc(inb & ((1u << c) - 1u)); }

// Where the cells of the current (window, tile, instant) go.
struct QuadOut {
  static constexpr bool search_quirk = false;
  CellOut co;
  u64 base;       // element index of tile cell (0, 0) at this instant
  i64 pitch;      // window columns
  int top, bottom, left, right;  // window clipped to the tile, tile coordinates
  bool vec, vec4; // f32 output whose row pairs / row quadruples are 8 / 16-byte aligned
  // k_window_tiles4's hooks: a job starts (bits: the stored subchunk's), an Elided job, an instant starts (tbase: element
  // index of tile cell (0, 0) at that instant in a dense window output) / ends, a job ends
  DCDF_DEVINL void begin(const TileWindowParams& P, const TileJob& J, int bits, unsigned char*) {
    const i64 W_cols = J.c.right - J.c.left;
    const u64 obase = P.out_off[J.q];
    const i64 tile_org = (J.chunk_top - J.c.top) * W_cols + (J.chunk_left - J.c.left);  // element offset of tile cell (0, 0)
    co.init(P.Q, P.out, P.raw, bits);
    pitch = W_cols;
    top = J.top; bottom = J.bottom; left = J.left; right = J.right;
    vec = co.kind == 2 && !(W_cols & 1) && !((obase + (u64)tile_org) & 1ull) && !((uintptr_t)P.out & 7u);
    vec4 = co.kind == 2 && !(W_cols & 3) && !((obase + (u64)tile_org) & 3ull) && !((uintptr_t)P.out & 15u);
    base = 0;  // set per instant
  }
  // Elided: one value per instant from the max table, parent's fractional bits (superchunk.rs:426-433)
  DCDF_DEVINL void elided(const TileWindowParams& P, const TileJob& J, const SliceMeta& sm, const SlotDesc& sdsc) const {
    const int wr = bottom - top, wc = right - left;
    const i64 W_rows = J.c.bottom - J.c.top;
    const u64 org = P.out_off[J.q] + (u64)((J.chunk_top - J.c.top) * pitch + (J.chunk_left - J.c.left));
    for (i64 t = J.t_lo; t < J.t_hi; t++) {
      const i64 v = P.Q.tbl_max[sdsc.tbl0 + (u64)(t - sm.t0) * sdsc.stride];
      const u64 tb = org + (u64)((t - J.c.start) * W_rows * pitch);
      for (int i = threadIdx.x; i < wr * wc; i += DT_THREADS)
        emit(P.Q, P.out, tb + (u64)((i64)(top + i / wc) * pitch + (left + i % wc)), v, sdsc.bits, P.raw);
    }
  }
  DCDF_DEVINL void instant_begin(u32, u64 tbase) { base = tbase; }
  DCDF_DEVINL void instant_end(u32) {}
  DCDF_DEVINL void end(u32) {}
  template <typename V>
  DCDF_DEVINL float cvt(V v) const {  // from_fixed (fixed.rs:81-86): 0 -> NaN, else (v - 1) * 2^-(bits+1), exact scaling
    const float f = (sizeof(V) == 4 ? __int2float_rn((int)v - 1) : __ll2float_rn((i64)v - 1)) * co.inv32;
    return v == 0 ? __int_as_float(0x7fc00000) : f;
  }
  DCDF_DEVINL bool touches(int r0, int c0, int side) const { return r0 + side > top && r0 < bottom && c0 + side > left && c0 < right; }
  DCDF_DEVINL bool inside(int r0, int c0, int side) const { return r0 >= top && r0 + side <= bottom && c0 >= left && c0 + side <= right; }
  template <typename V>
  DCDF_DEVINL void put(int r0, int c0, const V (&v)[4]) const {  // one 2x2 quad
    if (!touches(r0, c0, 2)) return;
    const u64 i00 = base + (u64)((i64)r0 * pitch + c0);
    const bool in = inside(r0, c0, 2);
    if (in && vec) {
      float* o = static_cast<float*>(co.out) + i00;
      *reinterpret_cast<float2*>(o) = make_float2(cvt(v[0]), cvt(v[1]));
      *reinterpret_cast<float2*>(o + pitch) = make_float2(cvt(v[2]), cvt(v[3]));
      return;
    }
#pragma unroll
    for (int c = 0; c < 4; c++) {
      const int r = r0 + (c >> 1), col = c0 + (c & 1);
      if (!in && (r < top || r >= bottom || col < left || col >= right)) continue;
      co.put(i00 + (u64)((c >> 1) ? pitch : 0) + (u64)(c & 1), v[c]);
    }
  }
  // two quads side by side (a 2x4 strip at (r0, c0)); fast = the whole 4x4 block is inside the window and vec4 holds
  template <typename V>
  DCDF_DEVINL void put_pair(bool fast, int r0, int c0, const V (&a)[4], const V (&b)[4]) const {
    if (fast) {
      float* o = static_cast<float*>(co.out) + (base + (u64)((i64)r0 * pitch + c0));
      *reinterpret_cast<float4*>(o) = make_float4(cvt(a[0]), cvt(a[1]), cvt(b[0]), cvt(b[1]));
      *reinterpret_cast<float4*>(o + pitch) = make_float4(cvt(a[2]), cvt(a[3]), cvt(b[2]), cvt(b[3]));
      return;
    }
    put(r0, c0, a);
    put(r0, c0 + 2, b);
  }
};

// Cell series through the tile decoder (k_cell_tiles4): the cells of a tile that some series of the batch asks for.
struct CellRef {
  u64 base;        // output element of the series' first instant
  i64 start, end;  // the series covers instants [start, end)
  u32 cell;        // 16 * block + 4 * quad + cell: block = Morton index of the 4x4 block, quad = 2 * (row / 2) + col / 2 and
  u32 pad_;        // cell = 2 * (row & 1) + (col & 1) inside the block -- the order the block decoder produces values in
};
// Same interface as QuadOut towards the block decoder: the values of the blocks that hold an asked-for cell go to an image
// of the tile in shared memory (one instant), from which the CTA then serves every series of the tile.
template <typename V>
struct SeriesOut {
  static constexpr bool search_quirk = false;
  V* img;     // the thread's 16 cells: img[4 * quad + cell]
  u32 mask;   // asked-for cells of the block (bit 4 * quad + cell); 0: nothing to decode
  static constexpr bool vec4 = false;
  DCDF_DEVINL bool touches(int, int, int) const { return mask != 0; }
  DCDF_DEVINL bool inside(int, int, int) const { return false; }
  DCDF_DEVINL void put(int r0, int c0, const V (&v)[4]) const {  // the 2x2 quad at (r0, c0): only its place inside the block matters
    const u32 quad = 2u * (((u32)r0 >> 1) & 1u) + (((u32)c0 >> 1) & 1u);
    Quad<V> q;
#pragma unroll
    for (int i = 0; i < 4; i++) q.c[i] = v[i];
    reinterpret_cast<Quad<V>*>(img)[quad] = q;
  }
  DCDF_DEVINL void put_pair(bool, int r0, int c0, const V (&a)[4], const V (&b)[4]) const {
    if (!(mask & (0xffu << (8u * (((u32)r0 >> 1) & 1u))))) return;  // nothing asked for in this half of the block
    put(r0, c0, a);
    put(r0, c0 + 2, b);
  }
};

// Value-range COUNTS of many windows over one tile (k_count_tiles4): the windows of a batch that touch the tile in this time
// slice share one decode of every instant.  An entry = one (window, tile): its rectangle inside the tile, its band, the
// instants of the slice it covers and where its per-instant counts go.
struct CountEntry {
  i64 cnt_base;          // counts[cnt_base + t] for the slice-local instant t
  // the fixed band; for the strict search (k_count_tiles4<V, true>) the value bounds, converted to the tile's band when
  // the entry is loaded into shared memory
  union { i64 lower; double vlower; };
  union { i64 upper; double vupper; };
  uint16_t t0, t1;       // slice-local instants [t0, t1)
  u8 top, bottom, left, right;  // tile coordinates, exclusive ends (<= 64)
};
constexpr int CT_MAX = 64;  // entries per job (a tile touched by more windows is split into several jobs)
template <typename V>
struct CountShared {
  CountEntry ent[CT_MAX];
  V lo[CT_MAX], hi[CT_MAX];  // the entry's band in the expansion's value type (clamped; lo > hi: no value can match)
  u32 cnt[2][CT_MAX];   // hits of the instant being decoded / of the previous one (flushed while the next one is decoded)
  u32 keep[CT_MAX];     // 0: pruned by the superchunk's min / max tables (superchunk.rs:480-493); else bit 0 set, and
                        // bit 1 when code 0 (NaN) is no hit although it lies in the band (strict search)
  unsigned long long act[2];  // entries that cover the instant being decoded (by instant parity)
  V smin0, smax0;       // root of the block's snapshot
  u32 n;
};
// Same interface as QuadOut towards the block decoder: the values of one half of the thread's block are tested against
// every entry whose rectangle touches the block.  The hit SET of the reference's traversal (snapshot.rs:310-421,
// log.rs:519-702) is "value inside the band" because every node test uses exact bounds -- with one exception that is
// reproduced here: a Log's ROOT is tested with min = snapshot.min.get(0) + log.min.get(0) and max = snapshot.max.get(0) +
// log.max.get(0) (log.rs:527-548), and an empty min Dac yields 0 (dac.rs:80-93).  So a Log over a single-node Snapshot, and
// a Log that is a single node itself (SURVEY App. B #15), are tested against a wrong lower bound; a single-node Log is
// moreover read as "snapshot + root entry" whether or not its `equal` bit is set.  log4 builds those values
// (search_quirk); the root test is applied per entry below, to every Log instant (it changes nothing when it is exact).
// ST (strict, dcdf_superchunk_search_values): none of this -- the values are read as the window decoder reads them and the
// hit set is exact; code 0 is no hit for the entries whose keep bit 1 is set.
template <typename V, bool ST>
struct CountOut {
  static constexpr bool search_quirk = !ST;
  static constexpr bool vec4 = false;
  CountShared<V>* C;
  unsigned long long mine;  // entries whose rectangle touches the thread's block
  int R0, C0;               // the block's origin
  u32 t;                    // slice-local instant
  u32 buf;                  // counter set / activity mask of this instant
  bool is_log;              // the instant is a Log: the reference's root test applies
  V min_t, e_root;          // its root entries (min Dac: 0 when empty)
  DCDF_DEVINL bool touches(int, int, int) const { return mine != 0ull; }
  DCDF_DEVINL bool inside(int, int, int) const { return false; }
  DCDF_DEVINL void put_pair(bool, int r0, int c0, const V (&a)[4], const V (&b)[4]) const {
    unsigned long long m = mine & C->act[buf];
    if (!m) return;
    // the strip's own range first: most bands miss it or hold all of it
    const V vmin = min(min(min(a[0], a[1]), min(a[2], a[3])), min(min(b[0], b[1]), min(b[2], b[3])));
    const V vmax = max(max(max(a[0], a[1]), max(a[2], a[3])), max(max(b[0], b[1]), max(b[2], b[3])));
    while (m) {
      const int e = __ffsll((long long)m) - 1;
      m &= m - 1ull;
      const V lo = C->lo[e], hi = C->hi[e];
      bool all = false, none = false;
      const bool nz = ST && (C->keep[e] & 2u);
      if (!ST && is_log) {  // the traversal's root test (log.rs:527-548)
        const CountEntry& E = C->ent[e];
        const i64 mn = (i64)C->smin0 + (i64)min_t, mx = (i64)C->smax0 + (i64)e_root;
        all = mn >= E.lower && mx <= E.upper;
        none = !all && (mn > E.upper || mx < E.lower);
      }
      if (none || (!all && (vmax < lo || vmin > hi))) continue;
      // cells of this 2x4 strip inside the entry's rectangle: bits 0..3 = a, 4..7 = b (cell = 2 * (row & 1) + (col & 1))
      const uchar4 rc = *reinterpret_cast<const uchar4*>(&C->ent[e].top);  // top, bottom, left, right
      const u32 rowm = ((r0 >= (int)rc.x && r0 < (int)rc.y) ? 0x33u : 0u) | ((r0 + 1 >= (int)rc.x && r0 + 1 < (int)rc.y) ? 0xccu : 0u);
      const u32 colm = ((c0 >= (int)rc.z && c0 < (int)rc.w) ? 0x05u : 0u) | ((c0 + 1 >= (int)rc.z && c0 + 1 < (int)rc.w) ? 0x0au : 0u) |
                       ((c0 + 2 >= (int)rc.z && c0 + 2 < (int)rc.w) ? 0x50u : 0u) | ((c0 + 3 >= (int)rc.z && c0 + 3 < (int)rc.w) ? 0xa0u : 0u);
      const u32 in = rowm & colm;
      if (!in) continue;
      u32 hit = in;
      if (!all && !(vmin >= lo && vmax <= hi && !(nz && vmin <= 0 && vmax >= 0))) {
        hit = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
          if (a[i] >= lo && a[i] <= hi && !(nz && a[i] == 0)) hit |= 1u << i;
          if (b[i] >= lo && b[i] <= hi && !(nz && b[i] == 0)) hit |= 16u << i;
        }
        hit &= in;
      }
      if (hit) atomicAdd(&C->cnt[buf][e], (u32)__popc(hit));
    }
  }
  DCDF_DEVINL void put(int r0, int c0, const V (&v)[4]) const {  // trees of side 2: one quad at (0, 0)
    // the second quad of the strip lies outside every rectangle of a 2x2 tile (right <= 2); it repeats the first one so
    // that the strip's range is the quad's
    CountOut o = *this;
    o.put_pair(false, r0, c0, v, v);
  }
};

// Window statistics through the tile decoder (k_window_tiles4<V, StatsOut<V>>): every thread folds the cells of its block
// that lie inside the window into its own slot in shared memory (no atomics); after each instant the CTA reduces the slots
// in a fixed order and thread 0 writes the (window, subchunk, instant) partial.  The sum is exact: the decoded value of a
// code n is x * 2^-(bits+1) with x = float(n - 1) / double(n - 1) an integer (the code itself for integer encodings), and
// x is summed as an integer (64 bits for the 32-bit expansion, 128 for the 64-bit one), converted to double once and
// scaled.  sum_sq adds x * x in double and is scaled the same way.
template <typename V>
struct StatsSlot {
  using Sum = typename std::conditional<sizeof(V) == 4, i64, __int128>::type;
  Sum sum;
  double sq;
  V mn, mx;  // codes
  u32 n;
  DCDF_DEVINL void clear() {
    sum = 0; sq = 0.0; n = 0;
    mn = sizeof(V) == 4 ? (V)INT32_MAX : (V)INT64_MAX;
    mx = sizeof(V) == 4 ? (V)INT32_MIN : (V)INT64_MIN;
  }
  DCDF_DEVINL void fold(const StatsSlot& o) { sum += o.sum; sq += o.sq; n += o.n; mn = min(mn, o.mn); mx = max(mx, o.mx); }
};
template <typename V>
struct StatsShared {
  StatsSlot<V> slot[DT_THREADS];
  StatsSlot<V> warp[2][DT_WARPS];  // per-warp results of an instant, by instant parity (folded while the next one is decoded)
};
// An integer-valued float / double as the sum's type (exact: |x| <= 2^31 for the 32-bit expansion, <= 2^63 otherwise).
template <typename S, typename F>
DCDF_DEVINL S exact_int(F x) {
  if (sizeof(S) == 8) return (S)(i64)x;
  return fabs((double)x) < 0x1p62 ? (S)(i64)x : (S)x;
}
template <typename V>
struct StatsOut {
  using Sum = typename StatsSlot<V>::Sum;
  static constexpr bool search_quirk = false;
  static constexpr bool vec4 = false;
  StatsShared<V>* C;
  StatsPartial* rec;             // partial of the job's first instant; instant i at rec[i]
  int top, bottom, left, right;  // window clipped to the tile, tile coordinates
  int kind;                      // 0: integer encodings (the code is the value), 2: f32, 3: f64
  int bits;
  DCDF_DEVINL bool touches(int r0, int c0, int side) const { return r0 + side > top && r0 < bottom && c0 + side > left && c0 < right; }
  DCDF_DEVINL bool inside(int r0, int c0, int side) const { return r0 >= top && r0 + side <= bottom && c0 >= left && c0 + side <= right; }
  DCDF_DEVINL void add(StatsSlot<V>& s, V v) const {
    if (kind != 0 && v == 0) return;  // NaN
    s.n++;
    s.mn = min(s.mn, v);
    s.mx = max(s.mx, v);
    if (kind == 2) {
      const float x = sizeof(V) == 4 ? __int2float_rn((int)v - 1) : __ll2float_rn((i64)v - 1);
      s.sum += exact_int<Sum>(x);
      s.sq += (double)x * (double)x;
    } else if (kind == 3) {
      const double x = sizeof(V) == 4 ? __int2double_rn((int)v - 1) : __ll2double_rn((i64)v - 1);
      s.sum += exact_int<Sum>(x);
      s.sq += x * x;
    } else {
      s.sum += (Sum)v;
      s.sq += (double)v * (double)v;
    }
  }
  DCDF_DEVINL void put_pair(bool, int r0, int c0, const V (&a)[4], const V (&b)[4]) const {
    // cells of this 2x4 strip inside the window: bits 0..3 = a, 4..7 = b (cell = 2 * (row & 1) + (col & 1))
    const u32 rowm = ((r0 >= top && r0 < bottom) ? 0x33u : 0u) | ((r0 + 1 >= top && r0 + 1 < bottom) ? 0xccu : 0u);
    const u32 colm = ((c0 >= left && c0 < right) ? 0x05u : 0u) | ((c0 + 1 >= left && c0 + 1 < right) ? 0x0au : 0u) |
                     ((c0 + 2 >= left && c0 + 2 < right) ? 0x50u : 0u) | ((c0 + 3 >= left && c0 + 3 < right) ? 0xa0u : 0u);
    const u32 in = rowm & colm;
    if (!in) return;
    StatsSlot<V>& slot = C->slot[threadIdx.x];
    StatsSlot<V> s = slot;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if ((in >> i) & 1u) add(s, a[i]);
      if ((in >> (4 + i)) & 1u) add(s, b[i]);
    }
    slot = s;
  }
  DCDF_DEVINL void put(int r0, int c0, const V (&v)[4]) const {  // trees of side 2: one quad at (0, 0)
    put_pair(false, r0, c0, v, v);  // the second quad lies outside every rectangle of a 2x2 tile (right <= 2)
  }
  // k_window_tiles4's hooks
  DCDF_DEVINL void begin(const TileWindowParams& P, const TileJob& J, int bits_, unsigned char* smem) {
    C = reinterpret_cast<StatsShared<V>*>(smem);
    rec = P.part + P.part_base[J.q] + J.sub * (u64)(J.c.end - J.c.start) + (u64)(J.t_lo - J.c.start);
    top = J.top; bottom = J.bottom; left = J.left; right = J.right;
    kind = P.Q.encoding == 32 ? 2 : P.Q.encoding == 64 ? 3 : 0;
    bits = bits_;
    C->slot[threadIdx.x].clear();
  }
  DCDF_DEVINL double scale() const { return kind ? __longlong_as_double((long long)(1022 - bits) << 52) : 1.0; }  // 2^-(bits+1)
  // Elided: one value per instant from the max table at its node's bits (superchunk.rs:426-433); nothing to decode
  DCDF_DEVINL void elided(const TileWindowParams& P, const TileJob& J, const SliceMeta& sm, const SlotDesc& sdsc) {
    bits = sdsc.bits;
    const double sc = scale();
    const i64 area = (i64)(bottom - top) * (i64)(right - left);
    for (i64 t = J.t_lo + (i64)threadIdx.x; t < J.t_hi; t += DT_THREADS) {
      const i64 v = P.Q.tbl_max[sdsc.tbl0 + (u64)(t - sm.t0) * sdsc.stride];
      const bool nan = kind != 0 && v == 0;
      const double x = kind == 2 ? (double)__ll2float_rn(v - 1) : kind == 3 ? __ll2double_rn(v - 1) : (double)v;
      StatsPartial p;
      p.count = nan ? 0u : (u32)area;
      p.bits = bits;
      p.min = v; p.max = v;
      const __int128 xi = kind == 0 ? (__int128)v : exact_int<__int128>(x);
      p.sum = nan ? 0.0 : (double)(xi * (__int128)area) * sc;
      p.sum_sq = nan ? 0.0 : (double)area * (x * x) * sc * sc;
      rec[t - J.t_lo] = p;
    }
  }
  DCDF_DEVINL void instant_begin(u32 i, u64) const {
    if (i > 0) flush(i - 1u);
  }
  // the CTA's reduction of instant i: warp shuffles in a fixed tree, then (flush) the warps in index order
  DCDF_DEVINL void instant_end(u32 i) const {
    StatsSlot<V>& slot = C->slot[threadIdx.x];
    StatsSlot<V> s = slot;
    slot.clear();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      StatsSlot<V> x;
      x.n = __shfl_down_sync(0xffffffffu, s.n, o);
      x.mn = __shfl_down_sync(0xffffffffu, s.mn, o);
      x.mx = __shfl_down_sync(0xffffffffu, s.mx, o);
      x.sq = __shfl_down_sync(0xffffffffu, s.sq, o);
      if (sizeof(V) == 4) {
        x.sum = (Sum)__shfl_down_sync(0xffffffffu, (long long)s.sum, o);
      } else {
        const unsigned long long lo = __shfl_down_sync(0xffffffffu, (unsigned long long)s.sum, o);
        const long long hi = __shfl_down_sync(0xffffffffu, (long long)(s.sum >> 64), o);
        x.sum = (Sum)(((unsigned __int128)(u64)hi << 64) | lo);
      }
      s.fold(x);
    }
    if ((threadIdx.x & 31u) == 0) C->warp[i & 1u][threadIdx.x >> 5] = s;
  }
  DCDF_DEVINL void flush(u32 i) const {  // thread 0, after a barrier that follows instant i's instant_end
    if (threadIdx.x != 0) return;
    StatsSlot<V> s = C->warp[i & 1u][0];
    for (int w = 1; w < DT_WARPS; w++) s.fold(C->warp[i & 1u][w]);
    const double sc = scale();
    StatsPartial p;
    p.count = s.n;
    p.bits = bits;
    p.min = (i64)s.mn; p.max = (i64)s.mx;
    p.sum = (double)s.sum * sc;
    p.sum_sq = s.sq * sc * sc;
    rec[i] = p;
  }
  DCDF_DEVINL void end(u32 n_t) const {
    __syncthreads();
    flush(n_t - 1u);
  }
};

// Per-cell statistics over time through the tile decoder (k_window_tiles4<V, TimeStatsOut<V>>).  A thread owns its 4x4
// block for the whole job, so it folds every instant of its cells into their accumulators in shared memory with no
// barrier and no atomics; after the last instant the CTA writes one TimePartial per cell of the clipped rectangle,
// row-major (coalesced).  Cell k = 4 * quad + cell of block p sits at index k * DT_THREADS + p (a warp's accesses are
// consecutive).  The counters are 16 bits wide: every TS_SPAN instants each thread adds its cells' counters to their
// partials in global memory and restarts them, so a slice may hold any number of instants.
constexpr int TS_CELLS = 16 * DT_THREADS;
constexpr u32 TS_SPAN = 0xffffu;
template <typename V>
struct TimeStatsShared {
  double sum[TS_CELLS], sq[TS_CELLS];
  V mn[TS_CELLS], mx[TS_CELLS];  // codes at the subchunk's bits
  uint16_t n[TS_CELLS], nb[TS_CELLS];
};
DCDF_DEVINL u32 ts_index(int r, int c) {  // accumulator of tile cell (r, c)
  const u32 k = 4u * (2u * (((u32)r >> 1) & 1u) + (((u32)c >> 1) & 1u)) + 2u * ((u32)r & 1u) + ((u32)c & 1u);
  return k * DT_THREADS + morton_encode((u32)r >> 2, (u32)c >> 2);
}
// The value the window decoder writes for an i64 code, as a double (NaN: code 0 of a float encoding, tested apart).
DCDF_DEVINL double ts_value(i64 v, int kind, int bits) {
  return kind == 2 ? (double)from_fixed_dev<float>(v, bits) : kind == 3 ? from_fixed_dev<double>(v, bits) : __ll2double_rn(v);
}
template <typename V>
struct TimeStatsOut {
  static constexpr bool search_quirk = false;
  static constexpr bool vec4 = false;
  TimeStatsShared<V>* C;
  TimePartial* rec;              // partial of tile cell (top, left); cell (r, c) at rec[(r - top) * pitch + c - left]
  u32 pitch;                     // window columns
  int top, bottom, left, right;  // window clipped to the tile, tile coordinates
  int kind;                      // 0: integer encodings (the code is the value), 2: f32, 3: f64
  int bits;
  double lo, hi;                 // band (-inf, inf without one)
  DCDF_DEVINL bool touches(int r0, int c0, int side) const { return r0 + side > top && r0 < bottom && c0 + side > left && c0 < right; }
  DCDF_DEVINL bool inside(int r0, int c0, int side) const { return r0 >= top && r0 + side <= bottom && c0 >= left && c0 + side <= right; }
  // the value QuadOut writes for the code (its cvt / CellOut::put), as a double
  DCDF_DEVINL double value(V v) const {
    if (kind == 2) return (double)((sizeof(V) == 4 ? __int2float_rn((int)v - 1) : __ll2float_rn((i64)v - 1)) * __int_as_float((126 - bits) << 23));
    if (kind == 3) return (sizeof(V) == 4 ? __int2double_rn((int)v - 1) : __ll2double_rn((i64)v - 1)) * __longlong_as_double((long long)(1022 - bits) << 52);
    return sizeof(V) == 4 ? (double)(int)v : __ll2double_rn((i64)v);
  }
  DCDF_DEVINL void add(u32 idx, V v) const {
    if (kind != 0 && v == 0) return;  // NaN
    const double x = value(v);
    TimeStatsShared<V>& S = *C;
    S.n[idx] = (uint16_t)(S.n[idx] + 1u);
    if (x >= lo && x <= hi) S.nb[idx] = (uint16_t)(S.nb[idx] + 1u);
    S.mn[idx] = min(S.mn[idx], v);
    S.mx[idx] = max(S.mx[idx], v);
    S.sum[idx] = __dadd_rn(S.sum[idx], x);
    S.sq[idx] = __dadd_rn(S.sq[idx], __dmul_rn(x, x));
  }
  DCDF_DEVINL void put_pair(bool, int r0, int c0, const V (&a)[4], const V (&b)[4]) const {
    // cells of this 2x4 strip inside the window: bits 0..3 = a, 4..7 = b (cell = 2 * (row & 1) + (col & 1))
    const u32 rowm = ((r0 >= top && r0 < bottom) ? 0x33u : 0u) | ((r0 + 1 >= top && r0 + 1 < bottom) ? 0xccu : 0u);
    const u32 colm = ((c0 >= left && c0 < right) ? 0x05u : 0u) | ((c0 + 1 >= left && c0 + 1 < right) ? 0x0au : 0u) |
                     ((c0 + 2 >= left && c0 + 2 < right) ? 0x50u : 0u) | ((c0 + 3 >= left && c0 + 3 < right) ? 0xa0u : 0u);
    const u32 in = rowm & colm;
    if (!in) return;
    const u32 ka = (4u * 2u * (((u32)r0 >> 1) & 1u)) * DT_THREADS + threadIdx.x;  // quad a: 2 * (row / 2 & 1), c0 % 4 == 0
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if ((in >> i) & 1u) add(ka + (u32)i * DT_THREADS, a[i]);
      if ((in >> (4 + i)) & 1u) add(ka + (u32)(4 + i) * DT_THREADS, b[i]);
    }
  }
  DCDF_DEVINL void put(int r0, int c0, const V (&v)[4]) const {  // trees of side 2: one quad at (0, 0)
    put_pair(false, r0, c0, v, v);  // the second quad lies outside every rectangle of a 2x2 tile (right <= 2)
  }
  // k_window_tiles4's hooks
  DCDF_DEVINL void begin(const TileWindowParams& P, const TileJob& J, int bits_, unsigned char* smem) {
    C = reinterpret_cast<TimeStatsShared<V>*>(smem);
    const i64 W_cols = J.c.right - J.c.left, area = (J.c.bottom - J.c.top) * W_cols;
    const u64 k = (u64)(J.t_lo / P.Q.chunk_size - J.c.start / P.Q.chunk_size);
    top = J.top; bottom = J.bottom; left = J.left; right = J.right;
    pitch = (u32)W_cols;
    rec = P.tpart + P.part_base[J.q] + k * (u64)area + (u64)((J.chunk_top + top - J.c.top) * W_cols + (J.chunk_left + left - J.c.left));
    kind = P.Q.encoding == 32 ? 2 : P.Q.encoding == 64 ? 3 : 0;
    bits = bits_;
    lo = P.band ? P.band[2 * J.q] : -INFINITY;
    hi = P.band ? P.band[2 * J.q + 1] : INFINITY;
  }
  DCDF_DEVINL TimeVal to_val(i64 code, int b) const {
    TimeVal r;
    if (kind) r.f = ts_value(code, kind, b); else r.i = code;
    return r;
  }
  // Elided: every cell holds the node's table value at the node's bits (superchunk.rs:426-433); one partial, computed by
  // every thread, written to each cell of the rectangle
  DCDF_DEVINL void elided(const TileWindowParams& P, const TileJob& J, const SliceMeta& sm, const SlotDesc& sdsc) const {
    TimePartial x;
    x.count = 0; x.n_band = 0;
    i64 mn = INT64_MAX, mx = INT64_MIN;
    double s = 0.0, q = 0.0;
    for (i64 t = J.t_lo; t < J.t_hi; t++) {
      const i64 v = P.Q.tbl_max[sdsc.tbl0 + (u64)(t - sm.t0) * sdsc.stride];
      if (kind != 0 && v == 0) continue;
      const double f = ts_value(v, kind, sdsc.bits);
      x.count++;
      if (f >= lo && f <= hi) x.n_band++;
      mn = min(mn, v); mx = max(mx, v);
      s = __dadd_rn(s, f);
      q = __dadd_rn(q, __dmul_rn(f, f));
    }
    x.min = to_val(mn, sdsc.bits); x.max = to_val(mx, sdsc.bits);
    x.sum = s; x.sum_sq = q;
    const int wc = right - left;
    for (int i = threadIdx.x; i < (bottom - top) * wc; i += DT_THREADS) rec[(u64)(i / wc) * pitch + (u32)(i % wc)] = x;
  }
  // instant 0: the thread's own accumulators start (the previous job's end read them before a barrier this one passed)
  DCDF_DEVINL void instant_begin(u32 i, u64) const {
    if (i % TS_SPAN == 0) {
      const u32 p = threadIdx.x;
      const int R0 = 4 * (int)morton_row(p), C0 = 4 * (int)morton_col(p);
      TimeStatsShared<V>& S = *C;
#pragma unroll 1
      for (u32 k = 0; k < 16u; k++) {
        const u32 idx = k * DT_THREADS + p;
        if (i > 0) {  // counters of the last TS_SPAN instants to the cell's partial
          const int r = R0 + 2 * (int)(k >> 3) + (int)((k >> 1) & 1u), c = C0 + 2 * (int)((k >> 2) & 1u) + (int)(k & 1u);
          if (r >= top && r < bottom && c >= left && c < right) {
            TimePartial& g = rec[(u64)(r - top) * pitch + (u32)(c - left)];
            g.count = (i == TS_SPAN ? 0u : g.count) + S.n[idx];
            g.n_band = (i == TS_SPAN ? 0u : g.n_band) + S.nb[idx];
          }
        } else {
          S.sum[idx] = 0.0; S.sq[idx] = 0.0;
          S.mn[idx] = sizeof(V) == 4 ? (V)INT32_MAX : (V)INT64_MAX;
          S.mx[idx] = sizeof(V) == 4 ? (V)INT32_MIN : (V)INT64_MIN;
        }
        S.n[idx] = 0; S.nb[idx] = 0;
      }
    }
  }
  DCDF_DEVINL void instant_end(u32) const {}
  DCDF_DEVINL void end(u32 n_t) const {
    __syncthreads();  // every block's accumulators are final (and the counters spilled by their owners are visible)
    const TimeStatsShared<V>& S = *C;
    const int wc = right - left;
    for (int i = threadIdx.x; i < (bottom - top) * wc; i += DT_THREADS) {
      const int r = top + i / wc, c = left + i % wc;
      const u32 idx = ts_index(r, c);
      TimePartial& g = rec[(u64)(r - top) * pitch + (u32)(c - left)];
      TimePartial x;
      x.count = (n_t > TS_SPAN ? g.count : 0u) + S.n[idx];
      x.n_band = (n_t > TS_SPAN ? g.n_band : 0u) + S.nb[idx];
      x.min = to_val((i64)S.mn[idx], bits); x.max = to_val((i64)S.mx[idx], bits);
      x.sum = S.sum[idx]; x.sum_sq = S.sq[idx];
      g = x;
    }
  }
};

// The `equal` bits of the children that stop here are consecutive: child c's bit is at e0 + (non-internal children
// before c), e0 = idx0 - rank1(idx0) (rank0(idx + 1) - 1, log.rs:265).  Returns a 16-bit window starting at e0's byte.
DCDF_DEVINL u32 eq_window(const u8* eq, u32 e0) {
  const u32 by = e0 >> 3;
  return ((u32)eq[by] << 8) | (u32)eq[by + 1];
}
DCDF_DEVINL bool eq_bit(u32 win, u32 e0, u32 k) { return (win >> (15u - (e0 & 7u) - k)) & 1u; }

}  // namespace dcdf
