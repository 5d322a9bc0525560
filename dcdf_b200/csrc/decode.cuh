// decode.cuh -- batched queries straight from serialized Chunk bytes resident in HBM.
//
//   BitMap::{get,rank,rank0}  bitmap.rs:174-218      Dac::get              dac.rs:80-93
//   Snapshot::get             snapshot.rs:165-188    Log::get              log.rs:176-293
//   Snapshot::search_window   snapshot.rs:310-421    Log::search_window    log.rs:519-702
//   Block / Chunk dispatch    block.rs:42-81, chunk.rs:127-228
//   Superchunk routing        superchunk.rs:313-633 (Elided cells come from the max table)
//
// A per-(chunk, instant) directory (offsets of every bitmap / DAC level inside the byte string) is built
// once by k_build_dir -- the device-side equivalent of Chunk::read_from (chunk.rs:247-266), including
// its length validation.  Queries then run one thread per cell / per (window, instant).
#pragma once
#include "common.cuh"

namespace dcdf {

struct DacDir {
  u32 n_levels;
  u32 len[8];   // entries on level j
  u32 base[8];  // byte offset (from chunk start) of level j's BitMap
};
struct alignas(16) InstDir {  // 176 bytes: one entry is a 16-byte aligned bulk copy
  u32 off;      // structure start (from chunk start)
  u32 size;     // serialized bytes of the structure
  u32 snap;     // directory index (within the chunk) of the block's Snapshot; == own index for snapshots
  u32 nm_len, nm_base;
  u32 eq_len, eq_base;  // logs only (eq_base == 0 for snapshots)
  DacDir max, min;
  u32 pad_[3];
};
static_assert(sizeof(InstDir) == 176, "InstDir is copied with 16-byte bulk copies");
struct UnitMeta {
  u64 blob_off;   // chunk start inside the blob
  u64 size;       // chunk bytes
  u32 dir_base;   // first InstDir of this chunk
  int instants;
  int rows, cols, sidelen;
  int bits;       // fractional bits of this chunk
  int stored;     // 0 = elided (no bytes)
  int enc;
  int dac_levels; // most byte levels of any max DAC of the chunk (<= 3: every entry is below 2^23 in magnitude)
  int pad_;
};
struct SliceMeta {
  i64 t0;
  int instants;
  int bits;         // parent fractional bits (values of elided subchunks)
  u64 table_base;
  u32 slot_base;    // first entry of this slice in slot_unit
  u32 pad;
};
// Where the value of a cell of an Elided subchunk comes from: entry (instant * stride) of the max table of the
// superchunk node that elided it, decoded with that node's fractional bits (superchunk.rs:325-330).
struct SlotDesc {
  u64 tbl0;
  u32 stride;
  int bits;
  // the same entry coordinates in the tables of the superchunk nodes ABOVE that node (nested superchunks), root first:
  // Superchunk::search prunes a subchunk with its node's min / max Dacs at every level of the recursion
  u64 up_tbl0[3];
  u32 up_stride[3];
  int n_up;
  int up_bits[3];  // fractional bits of those nodes (their tables are at these bits)
};
struct QuerySet {
  const u8* blob;
  const UnitMeta* units;
  const InstDir* dir;
  const SliceMeta* slices;
  const int32_t* slot_unit;  // [n_slices][n_slots] unit index or -1
  const SlotDesc* slot_desc; // [n_slices][n_slots] source of elided values
  const i64* tbl_max;
  const i64* tbl_min;        // null for a plain Chunk
  u32 n_slices, n_slots;
  i64 chunk_size;            // instants per slice
  int chunks_sidelen, subsidelen;
  int encoding;
  i64 shape[3];
};

// ------------------------------------------------------------------ byte-stream accessors
// 4 big-endian bytes at an arbitrary offset, via two aligned 32-bit loads (blobs are padded by 16 bytes).
DCDF_DEVINL u32 be32_at(const u8* base, u32 off) {
  const uintptr_t a = (uintptr_t)(base + off);
  const u32* w = reinterpret_cast<const u32*>(a & ~(uintptr_t)3);
  const u32 sh = (u32)(a & 3) * 8u;
  const u32 lo = w[0];  // plain loads: `base` may point to a shared-memory copy of the structure
  const u32 le = sh ? __funnelshift_r(lo, w[1], sh) : lo;
  return __byte_perm(le, 0, 0x0123);
}

struct BitMapRef {
  const u8* chunk;
  u32 len, base;  // BitMap start: [len:4][k:4][index...][words...]
  DCDF_DEVINL u32 words_off() const { return base + 8u + 4u * (len / 128u); }
  DCDF_DEVINL bool get(u32 i) const {  // bitmap.rs:176-183
    const u32 w = be32_at(chunk, words_off() + 4u * (i >> 5));
    return (w >> (31u - (i & 31u))) & 1u;
  }
  // bitmap.rs:186-212: ones in [0, i).  The directory entry and the (up to four) words of i's 128-bit block are all
  // requested before the first of them is used -- a warp stalls at the first instruction that needs a pending load, so a
  // loop that adds one word at a time pays up to five memory round trips where this pays one.  `on` = false: no load, 0.
  DCDF_DEVINL u32 rank(u32 i, bool on = true) const {
    const u32 block = i >> 7, rel = i & 127u;
    const uintptr_t a = (uintptr_t)(chunk + words_off() + 16u * block);
    const u32* w = reinterpret_cast<const u32*>(a & ~(uintptr_t)3);
    const u32 sh = (u32)(a & 3) * 8u;
    const u32 nw = on ? (rel + 31u) >> 5 : 0u;            // words of the block with bits below i
    const u32 n_ld = nw + ((sh && nw) ? 1u : 0u);          // aligned words they lie in
    const uintptr_t ai = (uintptr_t)(chunk + base + 8u + 4u * (block - 1u));
    const u32* wi = reinterpret_cast<const u32*>(ai & ~(uintptr_t)3);
    const u32 shi = (u32)(ai & 3) * 8u;
    const bool want_idx = on && block > 0;
    u32 i0 = 0, i1 = 0, x0 = 0, x1 = 0, x2 = 0, x3 = 0, x4 = 0;
    if (want_idx) i0 = wi[0];
    if (want_idx && shi) i1 = wi[1];
    if (n_ld > 0) x0 = w[0];
    if (n_ld > 1) x1 = w[1];
    if (n_ld > 2) x2 = w[2];
    if (n_ld > 3) x3 = w[3];
    if (n_ld > 4) x4 = w[4];
    u32 count = __byte_perm(shi ? __funnelshift_r(i0, i1, shi) : i0, 0, 0x0123);
    const u32 b0 = __byte_perm(sh ? __funnelshift_r(x0, x1, sh) : x0, 0, 0x0123), b1 = __byte_perm(sh ? __funnelshift_r(x1, x2, sh) : x1, 0, 0x0123);
    const u32 b2 = __byte_perm(sh ? __funnelshift_r(x2, x3, sh) : x2, 0, 0x0123), b3 = __byte_perm(sh ? __funnelshift_r(x3, x4, sh) : x3, 0, 0x0123);
    // the first min(rel - 32k, 32) bits of word k
    const u32 r = on ? rel : 0u;
    count += __popc(b0 & (u32)(0xffffffff00000000ull >> min(r, 32u)));
    count += __popc(b1 & (u32)(0xffffffff00000000ull >> min(r > 32u ? r - 32u : 0u, 32u)));
    count += __popc(b2 & (u32)(0xffffffff00000000ull >> min(r > 64u ? r - 64u : 0u, 32u)));
    count += __popc(b3 & (u32)(0xffffffff00000000ull >> (r > 96u ? r - 96u : 0u)));
    return count;
  }
  DCDF_DEVINL u32 rank0(u32 i) const { return i - rank(i); }
};

struct DacRef {
  const u8* chunk;
  const DacDir* d;
  DCDF_DEVINL i64 get(u32 index) const {  // dac.rs:80-93 (an empty DAC yields 0)
    u64 n = 0;
    const u32 nl = d->n_levels;
    for (u32 j = 0; j < nl; j++) {
      const u32 len = d->len[j], base = d->base[j];
      if (index >= len) break;  // malformed input guard
      const u32 words = base + 8u + 4u * (len / 128u);
      const u32 bytes = words + 4u * ((len + 31u) / 32u);
      n |= (u64)chunk[bytes + index] << (8u * j);
      BitMapRef bm{chunk, len, base};
      if (bm.get(index)) index = bm.rank(index);
      else break;
    }
    return unzigzag64(n);
  }
};

// Fast accessors for dense expansion: the MSB-first word stream of a BitMap is a plain MSB-first byte stream,
// so a bit test is one byte load; most DAC entries are one byte long (no continuation bit).
struct BitsFast {
  const u8* bits;  // first byte of the bitmap words
  DCDF_DEVINL bool get(u32 i) const { return (bits[i >> 3] >> (7u - (i & 7u))) & 1u; }
};
DCDF_DEVINL BitsFast bits_fast(const u8* chunk, u32 len, u32 base) { return BitsFast{chunk + base + 8u + 4u * (len / 128u)}; }
struct DacFast {
  const u8* bytes0;
  BitsFast more0;
  DacRef slow;
  bool empty;  // no levels at all: every lookup yields 0 (dac.rs:80-93)
  // `on` = false: no load, 0.  The continuation bit and the byte are requested together.
  DCDF_DEVINL i64 get(u32 index, bool on = true) const {
    if (empty || !on) return 0;
    const u32 byte = bytes0[index];
    if (!more0.get(index)) return unzigzag64((u64)byte);
    return slow.get(index);
  }
  // Same lookup in the expansion's value type: a one-byte code decodes in 32-bit arithmetic.
  template <typename V>
  DCDF_DEVINL V getv(u32 index) const {
    if (empty) return (V)0;
    if (!more0.get(index)) {
      const int b = (int)bytes0[index];
      return (V)((b >> 1) ^ -(b & 1));
    }
    return (V)slow.get(index);
  }
};
DCDF_DEVINL DacFast dac_fast(const u8* chunk, const DacDir* d) {
  const u32 len = d->len[0], base = d->base[0];
  const u32 words = base + 8u + 4u * (len / 128u);
  return DacFast{chunk + words + 4u * ((len + 31u) / 32u), BitsFast{chunk + words}, DacRef{chunk, d}, d->n_levels == 0};
}

// ------------------------------------------------------------------ directory builder (Chunk::read_from)
struct DirParams {
  const u8* blob;
  UnitMeta* units;   // rows / cols / sidelen / bits / instants(out, when counting) are filled in
  InstDir* dir;      // may be null in counting mode
  u32 n_units;
  int count_only;    // 1: only walk and count instants (dcdf_chunk_open pass 1)
  int validate;      // 1: bytes come from outside (dcdf_chunk_open / dcdf_superchunk_open): check every count the walks rely on
  u32* err;
};

struct Cursor {
  const u8* p;
  u64 pos, end;
  bool ok;
  DCDF_DEVINL u32 u8_() {
    if (pos + 1 > end) { ok = false; return 0; }
    return p[pos++];
  }
  DCDF_DEVINL u32 u32_() {
    if (pos + 4 > end) { ok = false; return 0; }
    u32 v = load_be32(p + pos);
    pos += 4;
    return v;
  }
  DCDF_DEVINL void skip(u64 n) {
    if (pos + n > end) { ok = false; return; }
    pos += n;
  }
};
DCDF_DEVINL void parse_bitmap(Cursor& c, u32& len, u32& base) {
  base = (u32)c.pos;
  len = c.u32_();
  const u32 k = c.u32_();
  if (k != 4u) c.ok = false;  // BitMapBuilder::finish always writes k = 4 (bitmap.rs:69)
  if (!c.ok) return;
  c.skip(4ull * (len / 128u) + 4ull * ((len + 31u) / 32u));
}
DCDF_DEVINL void parse_dac(Cursor& c, DacDir& d) {
  d.n_levels = c.u8_();
  if (d.n_levels > 8) c.ok = false;
  for (u32 j = 0; j < 8; j++) { d.len[j] = 0; d.base[j] = 0; }
  for (u32 j = 0; j < d.n_levels && c.ok; j++) {
    parse_bitmap(c, d.len[j], d.base[j]);
    c.skip(d.len[j]);
    if (j > 0 && d.len[j] > d.len[j - 1]) c.ok = false;
  }
}

// Ones among the first `len` bits of a serialized BitMap, checking its rank directory on the way
// (index[b] == ones in words [0, 4(b+1)), bitmap.rs:97-104).  The walks trust both.
DCDF_DEVINL u32 checked_popcount(const u8* chunk, u32 len, u32 base, bool& ok) {
  const u32 blocks = len / 128u, words = (len + 31u) / 32u;
  const u32 wo = base + 8u + 4u * blocks;
  u32 ones = 0;
  for (u32 w = 0; w < words; w++) {
    u32 v = be32_at(chunk, wo + 4u * w);
    if (w == words - 1u && (len & 31u)) v &= ~(0xffffffffu >> (len & 31u));
    ones += __popc(v);
    if ((w & 3u) == 3u && (w >> 2) < blocks && be32_at(chunk, base + 8u + 4u * (w >> 2)) != ones) ok = false;
  }
  return ones;
}
// Dac::from invariants (dac.rs:96-132): level j + 1 holds one byte per continuation bit of level j.
DCDF_DEVINL void check_dac(const u8* chunk, const DacDir& d, u32 expect_len0, bool& ok) {
  if ((d.n_levels ? d.len[0] : 0u) != expect_len0) ok = false;
  for (u32 j = 0; j < d.n_levels && ok; j++) {
    const u32 ones = checked_popcount(chunk, d.len[j], d.base[j], ok);
    const u32 next = j + 1u < d.n_levels ? d.len[j + 1u] : 0u;
    if (ones != next) ok = false;
  }
}

__global__ void k_build_dir(const DirParams P) {
  const u32 u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= P.n_units) return;
  UnitMeta m = P.units[u];
  if (!m.stored) return;
  Cursor c{P.blob + m.blob_off, 0, m.size, true};
  const u32 enc = c.u8_();
  const u32 fb = c.u8_();
  const u32 n_blocks = c.u32_();
  if (!(enc == 4 || enc == 8 || enc == 32 || enc == 64) || n_blocks == 0) c.ok = false;
  u32 inst = 0, dac_levels = 0;
  int rows = 0, cols = 0, sidelen = 0;
  for (u32 b = 0; b < n_blocks && c.ok; b++) {
    const u32 n_inst = c.u8_();
    if (n_inst == 0) c.ok = false;
    const u32 snap_idx = inst;
    for (u32 i = 0; i < n_inst && c.ok; i++) {
      InstDir d;
      d.pad_[0] = d.pad_[1] = d.pad_[2] = 0;
      d.off = (u32)c.pos;
      d.snap = snap_idx;
      const u32 k = c.u8_();
      const u32 r = c.u32_(), cl = c.u32_(), sl = c.u32_();
      if (k != 2u || sl < 2u || (sl & (sl - 1u)) || r > sl || cl > sl || r == 0 || cl == 0) c.ok = false;
      if (inst == 0) { rows = (int)r; cols = (int)cl; sidelen = (int)sl; }
      else if ((int)r != rows || (int)cl != cols || (int)sl != sidelen) c.ok = false;
      parse_bitmap(c, d.nm_len, d.nm_base);
      d.eq_len = 0; d.eq_base = 0;
      if (i > 0) parse_bitmap(c, d.eq_len, d.eq_base);
      parse_dac(c, d.max);
      parse_dac(c, d.min);
      dac_levels = max(dac_levels, d.max.n_levels);
      d.size = (u32)c.pos - d.off;
      if (c.ok && d.nm_len == 0) c.ok = false;
      if (c.ok && P.validate && !P.count_only) {
        // one max entry for the root and four per internal node, one min entry per internal node, one `equal` bit per
        // node that is not internal (snapshot.rs:122-147, log.rs:128-158): the walks index with ranks of the nodemap
        bool ok = (d.nm_len & 3u) == 1u;
        const u32 ones = checked_popcount(c.p, d.nm_len, d.nm_base, ok);
        check_dac(c.p, d.max, 1u + 4u * ones, ok);
        check_dac(c.p, d.min, ones, ok);
        if (i > 0) {
          if (d.eq_len != d.nm_len - ones) ok = false;
          else checked_popcount(c.p, d.eq_len, d.eq_base, ok);
        }
        if (d.nm_len > 1u + 4u * ones) ok = false;
        if (!ok) c.ok = false;
      }
      if (c.ok && !P.count_only) {
        if (inst >= (u32)m.instants) c.ok = false;
        else P.dir[m.dir_base + inst] = d;
      }
      inst++;
    }
  }
  if (c.ok && c.pos != c.end) c.ok = false;  // trailing bytes
  if (c.ok && !P.count_only && inst != (u32)m.instants) c.ok = false;
  if (!c.ok) {
    atomicOr(P.err, (u32)EF_BAD_FORMAT);
    return;
  }
  m.rows = rows; m.cols = cols; m.sidelen = sidelen; m.bits = (int)fb; m.enc = (int)enc; m.dac_levels = (int)dac_levels;
  if (P.count_only) m.instants = (int)inst;
  P.units[u] = m;
  (void)n_blocks;
}

// ------------------------------------------------------------------ cell walks
struct ChunkView {
  const u8* chunk;
  const InstDir* dir;  // this chunk's directory
  int sidelen;
};

DCDF_DEVINL i64 snapshot_get(const ChunkView& cv, const InstDir& s, u32 row, u32 col) {  // snapshot.rs:165-188
  BitMapRef nm{cv.chunk, s.nm_len, s.nm_base};
  DacRef mx{cv.chunk, &s.max};
  i64 value = mx.get(0);
  if (!nm.get(0)) return value;
  u32 sl = (u32)cv.sidelen, index = 0;
  for (;;) {
    sl >>= 1;
    index = 1u + nm.rank(index) * 4u + (row / sl) * 2u + (col / sl);
    value -= mx.get(index);
    if (index >= s.nm_len || !nm.get(index)) return value;
    row %= sl; col %= sl;
  }
}

// `is_snap`: the instant is the block's Snapshot itself (l == s).  It takes the same walk as a Log whose tree ends at the
// root with offset 0 -- Snapshot::get (snapshot.rs:165-188) is exactly the snapshot half of this loop -- so that the lanes
// of a warp (consecutive instants of one cell series) stay on one code path instead of running snapshot_get and log_get
// one after the other.
DCDF_DEVINL i64 log_get(const ChunkView& cv, const InstDir& l, const InstDir& s, u32 row, u32 col, bool is_snap = false) {  // log.rs:176-293
  BitMapRef nm_t{cv.chunk, l.nm_len, l.nm_base}, nm_s{cv.chunk, s.nm_len, s.nm_base};
  BitMapRef eq{cv.chunk, l.eq_len, l.eq_base};
  // level 0 of both max DACs located once: a one-byte code is then a bit test and a byte load that do not wait for the
  // directory entry (DacRef re-reads its level table from global memory at every lookup)
  const DacFast mx_t = dac_fast(cv.chunk, &l.max), mx_s = dac_fast(cv.chunk, &s.max);
  i64 max_t = is_snap ? 0 : mx_t.get(0), max_s = mx_s.get(0);
  const bool single_t = is_snap || !nm_t.get(0), single_s = !nm_s.get(0);
  if (single_t && single_s) return max_t + max_s;
  if (!is_snap && single_t && !eq.get(0)) return max_t + max_s;
  bool has_t = !single_t, has_s = !single_s;
  u32 it = 0, is = 0, sl = (u32)cv.sidelen;
  for (;;) {
    sl >>= 1;
    if (sl == 0) return max_t + max_s;  // malformed input guard
    const u32 child = (row / sl) * 2u + (col / sl);
    // the two trees are descended side by side: both ranks in one round trip, then everything that hangs off the new
    // indices (entry, continuation bit, nodemap bit of either tree) in a second one
    const u32 rs = nm_s.rank(is, has_s), rt = nm_t.rank(it, has_t);
    if (has_s) is = 1u + rs * 4u + child;
    if (has_t) it = 1u + rt * 4u + child;
    const bool in_t = has_t && it < l.nm_len, in_s = has_s && is < s.nm_len;
    const bool bit_t = in_t ? nm_t.get(it) : false, bit_s = in_s ? nm_s.get(is) : false;
    const i64 es = mx_s.get(is, has_s), et = mx_t.get(it, has_t);
    max_s -= es;
    if (has_t) max_t = et;
    const bool leaf_t = !bit_t;
    const bool leaf_s = !bit_s;
    if (leaf_t && leaf_s) return max_t + max_s;
    if (leaf_s) {
      has_s = false;
    } else if (leaf_t) {
      if (has_t && it < l.nm_len) {
        if (!eq.get(nm_t.rank0(it + 1u) - 1u)) return max_t + max_s;
      }
      has_t = false;
    }
    row %= sl; col %= sl;
  }
}

// ---- block walks: one descent shared by the 4x4 cells below a node (Chunk::fill_window for trees the tile decoder does
// not take, snapshot.rs:238-301 / log.rs:324-508).  The state is log_get's; walk_child is one turn of its loop.
struct WalkTrees {
  BitMapRef nm_t, nm_s, eq;
  DacFast mx_t, mx_s;
  u32 len_t, len_s;
};
struct WalkState {
  i64 max_t, max_s;
  u32 it, is;
  bool has_t, has_s;
};
// Moves `st` from a node to its child `child`; rs / rt are the node's ranks in the two nodemaps (the same for its four
// children).  True when max_t + max_s is final for every cell below the child.
DCDF_DEVINL bool walk_child(const WalkTrees& W, WalkState& st, u32 rs, u32 rt, u32 child) {
  if (st.has_s) st.is = 1u + rs * 4u + child;
  if (st.has_t) st.it = 1u + rt * 4u + child;
  const bool in_t = st.has_t && st.it < W.len_t, in_s = st.has_s && st.is < W.len_s;
  const bool bit_t = in_t ? W.nm_t.get(st.it) : false, bit_s = in_s ? W.nm_s.get(st.is) : false;
  const i64 es = W.mx_s.get(st.is, st.has_s), et = W.mx_t.get(st.it, st.has_t);
  st.max_s -= es;
  if (st.has_t) st.max_t = et;
  if (!bit_t && !bit_s) return true;
  if (!bit_s) {
    st.has_s = false;
  } else if (!bit_t) {
    if (in_t && !W.eq.get(W.nm_t.rank0(st.it + 1u) - 1u)) return true;
    st.has_t = false;
  }
  return false;
}
DCDF_DEVINL void fill16(i64* v, i64 x) {
#pragma unroll
  for (int i = 0; i < 16; i++) v[i] = x;
}
// v[4 * dr + dc] = value of cell (row + dr, col + dc); row and col are multiples of min(4, sidelen) inside the tree.
// Trees of side 2 fill dr, dc < 2 only.
DCDF_DEVINL void log_get_block(const ChunkView& cv, const InstDir& l, const InstDir& s, u32 row, u32 col, bool is_snap, i64* v) {
  const WalkTrees W{BitMapRef{cv.chunk, l.nm_len, l.nm_base}, BitMapRef{cv.chunk, s.nm_len, s.nm_base},
                    BitMapRef{cv.chunk, l.eq_len, l.eq_base}, dac_fast(cv.chunk, &l.max), dac_fast(cv.chunk, &s.max), l.nm_len, s.nm_len};
  WalkState st;
  st.max_t = is_snap ? 0 : W.mx_t.get(0);
  st.max_s = W.mx_s.get(0);
  const bool single_t = is_snap || !W.nm_t.get(0), single_s = !W.nm_s.get(0);
  if ((single_t && single_s) || (!is_snap && single_t && !W.eq.get(0))) {
    fill16(v, st.max_t + st.max_s);
    return;
  }
  st.has_t = !single_t; st.has_s = !single_s;
  st.it = 0; st.is = 0;
  u32 sl = (u32)cv.sidelen;
  while (sl > 4u) {  // down to the node that covers the block
    sl >>= 1;
    const u32 rs = W.nm_s.rank(st.is, st.has_s), rt = W.nm_t.rank(st.it, st.has_t);
    if (walk_child(W, st, rs, rt, (row / sl) * 2u + (col / sl))) {
      fill16(v, st.max_t + st.max_s);
      return;
    }
    row %= sl; col %= sl;
  }
  const u32 rs = W.nm_s.rank(st.is, st.has_s), rt = W.nm_t.rank(st.it, st.has_t);
  if (sl == 2u) {    // the whole tree is one 2x2 node
#pragma unroll
    for (u32 c1 = 0; c1 < 4u; c1++) {
      WalkState s1 = st;
      walk_child(W, s1, rs, rt, c1);
      v[4u * (c1 >> 1) + (c1 & 1u)] = s1.max_t + s1.max_s;
    }
    return;
  }
#pragma unroll
  for (u32 c1 = 0; c1 < 4u; c1++) {
    WalkState s1 = st;
    const bool done = walk_child(W, s1, rs, rt, c1);
    const u32 r1 = 2u * (c1 >> 1), q1 = 2u * (c1 & 1u);
    u32 rs1 = 0, rt1 = 0;
    if (!done) { rs1 = W.nm_s.rank(s1.is, s1.has_s); rt1 = W.nm_t.rank(s1.it, s1.has_t); }
#pragma unroll
    for (u32 c2 = 0; c2 < 4u; c2++) {
      WalkState s2 = s1;
      if (!done) walk_child(W, s2, rs1, rt1, c2);
      v[4u * (r1 + (c2 >> 1)) + q1 + (c2 & 1u)] = s2.max_t + s2.max_s;
    }
  }
}

DCDF_DEVINL i64 chunk_get(const ChunkView& cv, u32 instant, u32 row, u32 col) {  // chunk.rs:127-131 + block.rs:42-47
  const InstDir& d = cv.dir[instant];
  return log_get(cv, d, cv.dir[d.snap], row, col, d.snap == instant);
}

// Route a global (instant,row,col) to (fixed value, fractional bits)  -- superchunk.rs:313-351 + span.rs:121-137
DCDF_DEVINL i64 set_get(const QuerySet& Q, i64 instant, i64 row, i64 col, int& bits) {
  const u32 s = (u32)(instant / Q.chunk_size);
  const SliceMeta sm = Q.slices[s];
  const u32 ti = (u32)(instant - sm.t0);
  const u32 cr = (u32)(row / Q.chunks_sidelen), cc = (u32)(col / Q.chunks_sidelen);
  const u32 slot = cr * (u32)Q.subsidelen + cc;
  const int32_t u = Q.slot_unit[sm.slot_base + slot];
  if (u >= 0) {
    const UnitMeta m = Q.units[u];
    if (m.stored) {
      bits = m.bits;
      ChunkView cv{Q.blob + m.blob_off, Q.dir + m.dir_base, m.sidelen};
      return chunk_get(cv, ti, (u32)(row % Q.chunks_sidelen), (u32)(col % Q.chunks_sidelen));
    }
  }
  const SlotDesc sdsc = Q.slot_desc[sm.slot_base + slot];
  bits = sdsc.bits;
  return Q.tbl_max[sdsc.tbl0 + (u64)ti * sdsc.stride];  // Elided: superchunk.rs:325-330
}

// set_get for the block of min(4, chunks_sidelen)^2 cells at (row, col) -- both multiples of that size, so the block
// lies inside one subchunk.
DCDF_DEVINL void set_get_block(const QuerySet& Q, i64 instant, i64 row, i64 col, int& bits, i64* v) {
  const u32 s = (u32)(instant / Q.chunk_size);
  const SliceMeta sm = Q.slices[s];
  const u32 ti = (u32)(instant - sm.t0);
  const u32 cr = (u32)(row / Q.chunks_sidelen), cc = (u32)(col / Q.chunks_sidelen);
  const u32 slot = cr * (u32)Q.subsidelen + cc;
  const int32_t u = Q.slot_unit[sm.slot_base + slot];
  if (u >= 0) {
    const UnitMeta m = Q.units[u];
    if (m.stored) {
      bits = m.bits;
      ChunkView cv{Q.blob + m.blob_off, Q.dir + m.dir_base, m.sidelen};
      const InstDir& d = cv.dir[ti];
      log_get_block(cv, d, cv.dir[d.snap], (u32)(row % Q.chunks_sidelen), (u32)(col % Q.chunks_sidelen), d.snap == ti, v);
      return;
    }
  }
  const SlotDesc sdsc = Q.slot_desc[sm.slot_base + slot];
  bits = sdsc.bits;
  fill16(v, Q.tbl_max[sdsc.tbl0 + (u64)ti * sdsc.stride]);
}

// Superchunk::search's has_cells (superchunk.rs:480-493): some instant of [t_lo, t_hi) -- slice-local indices -- has
// upper >= min && lower <= max in the subchunk's entry of the node's min / max tables; applied at every level of a
// nested superchunk.  Each caller tests the instants t_lo + first, t_lo + first + step, ... and ORs the results.
DCDF_DEVINL bool slot_has_cells_part(const QuerySet& Q, const SlotDesc& d, i64 t_lo, i64 t_hi, i64 lower, i64 upper, int first, int step,
                                     int level /* 0 .. n_up: n_up = the slot's own node */) {
  const u64 tbl0 = level < d.n_up ? d.up_tbl0[level] : d.tbl0;
  const u64 stride = level < d.n_up ? d.up_stride[level] : d.stride;
  bool any = false;
  for (i64 t = t_lo + first; t < t_hi; t += step) {
    const u64 idx = tbl0 + (u64)t * stride;
    any = any || (upper >= Q.tbl_min[idx] && lower <= Q.tbl_max[idx]);
  }
  return any;
}

// ------------------------------------------------------------------ value bounds (dcdf_superchunk_search_values)
// The value the window decoder writes for a code, as a double: from_fixed_dev in the encoding's float type, the stored
// integer itself for integer encodings.  Code 0 of a float encoding is NaN and never a hit; it is given the value 0 here,
// which lies between the values of codes -1 and 1, so that the map stays monotone non-decreasing in the code
// (fixed.rs:81-86) and the codes of any value interval form one interval.  INT64_MIN, where n - 1 would wrap, takes the
// value of INT64_MIN + 1.
DCDF_DEVINL double code_value(i64 n, int bits, int enc) {
  if (enc == 4 || enc == 8) return (double)n;
  if (n == 0) return 0.0;
  if (n == INT64_MIN) n++;
  return enc == 32 ? (double)from_fixed_dev<float>(n, bits) : from_fixed_dev<double>(n, bits);
}
// Fixed-point band of the value interval [lo, hi] at `bits` fractional bits: a code n is a hit iff lower <= n <= upper
// and not (nz && n == 0).  Both ends by binary search over all of i64 with code_value itself -- a closed form such as
// 2 ceil(lo 2^bits) + 1 misses when the float rounding of n - 1 maps many codes to one value (codes past 2^24 in f32).
struct FixedBand {
  i64 lower, upper;
  bool nz;
};
DCDF_DEVINL FixedBand value_band(double lo, double hi, int bits, int enc) {
  constexpr u64 SIGN = 1ull << 63;  // code = (i64)(offset ^ SIGN): offsets 0 .. 2^64 - 1 run over the codes in order
  FixedBand b{1, 0, false};         // empty
  if (!(code_value(INT64_MAX, bits, enc) >= lo) || !(code_value(INT64_MIN, bits, enc) <= hi)) return b;
  u64 a = 0, z = ~0ull;  // smallest code with value >= lo
  while (a < z) {
    const u64 mid = a + (z - a) / 2;
    if (code_value((i64)(mid ^ SIGN), bits, enc) >= lo) z = mid; else a = mid + 1;
  }
  b.lower = (i64)(a ^ SIGN);
  a = 0; z = ~0ull;      // largest code with value <= hi
  while (a < z) {
    const u64 mid = z - (z - a) / 2;
    if (code_value((i64)(mid ^ SIGN), bits, enc) <= hi) a = mid; else z = mid - 1;
  }
  b.upper = (i64)(a ^ SIGN);
  b.nz = (enc == 32 || enc == 64) && b.lower <= 0 && b.upper >= 0;
  return b;
}
// Hit tests against a band: one code / every code of [mn, mx] / no code of [mn, mx].  With nz false they are the plain
// interval tests of the fixed-bound search.
DCDF_DEVINL bool band_hit(i64 v, i64 lower, i64 upper, bool nz) { return lower <= v && v <= upper && !(nz && v == 0); }
DCDF_DEVINL bool band_all(i64 mn, i64 mx, i64 lower, i64 upper, bool nz) { return lower <= mn && mx <= upper && !(nz && mn <= 0 && mx >= 0); }
DCDF_DEVINL bool band_none(i64 mn, i64 mx, i64 lower, i64 upper, bool nz) { return mn > upper || mx < lower || (nz && mn == 0 && mx == 0); }

// slot_has_cells_part for value bounds [lo, hi].  A level's tables hold codes at that node's fractional bits nb
// (App. B #11), while a stored subchunk below encodes at its own bits: rounded (round = true) there, a value can lie
// outside the table's decoded bracket [from_fixed(min), from_fixed(max)] by less than one unit 2^-nb of the node's
// bits, and the decoded value carries one more rounding to the output type (at most one ulp, < 2^-22 |x| for f32).  So
// the bracket is widened by 2^-nb + 2^-22 |x| on each side before the test, and a table code 0 bounds nothing on its
// side (min_max_float stores a min of code 0 for an instant with NaN cells, App. B #10).  Integer tables are exact.
// Elided slots need no margin: their values are the table values, tested exactly by the caller.
DCDF_DEVINL bool slot_may_hold_part(const QuerySet& Q, const SlotDesc& d, i64 t_lo, i64 t_hi, double lo, double hi, int first, int step,
                                    int level) {
  const u64 tbl0 = level < d.n_up ? d.up_tbl0[level] : d.tbl0;
  const u64 stride = level < d.n_up ? d.up_stride[level] : d.stride;
  const int nb = level < d.n_up ? d.up_bits[level] : d.bits;
  const bool flt = Q.encoding == 32 || Q.encoding == 64;
  const double unit = flt ? ldexp(1.0, -nb) : 0.0, rel = flt ? 0x1p-22 : 0.0;
  bool any = false;
  for (i64 t = t_lo + first; t < t_hi && !any; t += step) {
    const u64 idx = tbl0 + (u64)t * stride;
    const i64 cmin = Q.tbl_min[idx], cmax = Q.tbl_max[idx];
    double vmin = -INFINITY, vmax = INFINITY;
    if (!flt || cmin != 0) { vmin = code_value(cmin, nb, Q.encoding); vmin -= unit + rel * fabs(vmin); }
    if (!flt || cmax != 0) { vmax = code_value(cmax, nb, Q.encoding); vmax += unit + rel * fabs(vmax); }
    any = hi >= vmin && lo <= vmax;
  }
  return any;
}

template <typename OutT>
DCDF_DEVINL void store_value(void* out, u64 i, i64 fixed, int bits, int out_enc) {
  if (out_enc == 8) static_cast<i64*>(out)[i] = fixed;
  else if (out_enc == 4) static_cast<int32_t*>(out)[i] = (int32_t)fixed;
  else if (out_enc == 32) static_cast<float*>(out)[i] = from_fixed_dev<float>(fixed, bits);
  else static_cast<double*>(out)[i] = from_fixed_dev<double>(fixed, bits);
}

// out_mode: 0 = raw fixed i64 ; otherwise the chunk's own encoding with from_fixed applied to floats
DCDF_DEVINL void emit(const QuerySet& Q, void* out, u64 i, i64 fixed, int bits, int raw) {
  if (raw) static_cast<i64*>(out)[i] = fixed;
  else store_value<void>(out, i, fixed, bits, Q.encoding);
}

// Chunk::get batched: one thread per (instant,row,col)
// Queries may live in device memory the host never saw: bounds are checked here (mmarray.rs:218-229); an offending
// query writes 0 and raises EF_OUT_OF_BOUNDS.
__global__ void k_get_batch(const QuerySet Q, const i64* irc, u64 n, void* out, int raw, u32* err) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int bits = 0;
  const i64 t = irc[3 * i], r = irc[3 * i + 1], c = irc[3 * i + 2];
  i64 v = 0;
  if (t < 0 || r < 0 || c < 0 || t >= Q.shape[0] || r >= Q.shape[1] || c >= Q.shape[2]) atomicOr(err, (u32)EF_OUT_OF_BOUNDS);
  else v = set_get(Q, t, r, c, bits);
  emit(Q, out, i, v, bits, raw);
}

// Chunk::fill_cell batched: queries (start,end,row,col); one thread per (query, instant), grid.y = query
__global__ void __launch_bounds__(128, 9) k_cell_batch(const QuerySet Q, const i64* q, const u64* out_off, u64 n, void* out, int raw) {
  for (u64 qi = blockIdx.y; qi < n; qi += gridDim.y) {
    const i64 start = q[4 * qi], end = q[4 * qi + 1], row = q[4 * qi + 2], col = q[4 * qi + 3];
    const u64 base = out_off[qi];
    for (i64 t = start + (i64)blockIdx.x * blockDim.x + threadIdx.x; t < end; t += (i64)gridDim.x * blockDim.x) {
      int bits;
      const i64 v = set_get(Q, t, row, col, bits);
      emit(Q, out, base + (u64)(t - start), v, bits, raw);
    }
  }
}

struct CubeDev { i64 start, end, top, bottom, left, right; };
// Chunk::fill_window batched, trees larger than 64x64 (and ctx option `window_cells`): one thread per 4x4 block of the
// window's aligned block grid; the descent to the block's ancestor is shared by its 16 cells (C1, one 100x256x256 Chunk: 1.03 ms with one walk per
// cell -> 0.20 ms).
__global__ void k_window_blocks(const QuerySet Q, const CubeDev* cubes, const u64* out_off, u64 n, void* out, int raw) {
  const i64 B = Q.chunks_sidelen < 4 ? Q.chunks_sidelen : 4;
  for (u64 qi = blockIdx.y; qi < n; qi += gridDim.y) {
    const CubeDev c = cubes[qi];
    const i64 rows = c.bottom - c.top, cols = c.right - c.left, T = c.end - c.start;
    if (rows <= 0 || cols <= 0 || T <= 0) continue;
    const i64 br0 = c.top / B, nbr = (c.bottom - 1) / B + 1 - br0, bc0 = c.left / B, nbc = (c.right - 1) / B + 1 - bc0;
    const i64 blocks = T * nbr * nbc;
    const u64 base = out_off[qi];
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < blocks; i += (i64)gridDim.x * blockDim.x) {
      const i64 t = i / (nbr * nbc), rem = i - t * nbr * nbc;
      const i64 r0 = (br0 + rem / nbc) * B, c0 = (bc0 + rem % nbc) * B;
      i64 v[16];
      int bits;
      set_get_block(Q, c.start + t, r0, c0, bits, v);
#pragma unroll
      for (int dr = 0; dr < 4; dr++) {
        const i64 r = r0 + dr;
        if (dr >= B || r < c.top || r >= c.bottom) continue;
#pragma unroll
        for (int dc = 0; dc < 4; dc++) {
          const i64 cc = c0 + dc;
          if (dc >= B || cc < c.left || cc >= c.right) continue;
          emit(Q, out, base + (u64)((t * rows + (r - c.top)) * cols + (cc - c.left)), v[4 * dr + dc], bits, raw);
        }
      }
    }
  }
}

// ------------------------------------------------------------------ value-range search
// One thread per (window, slice-instant, subchunk) job replays the reference's depth-first traversal with
// an explicit stack so that results come out in the reference's order.  Pass 1 (out == null) counts,
// pass 2 writes at the scanned offsets.
struct Sink {
  i64* out;       // null while counting
  u64 n;
  i64 instant;
  int row0, col0;
  DCDF_DEVINL void push(u32 row, u32 col) {
    if (out) {
      out[3 * n] = instant;
      out[3 * n + 1] = (i64)row + row0;
      out[3 * n + 2] = (i64)col + col0;
    }
    n++;
  }
  DCDF_DEVINL void push_rect(u32 top, u32 bottom, u32 left, u32 right, u32 top_off, u32 left_off) {  // inclusive bounds
    for (u32 r = top; r <= bottom; r++)
      for (u32 c = left; c <= right; c++) push(top_off + r, left_off + c);
  }
};

constexpr int SEARCH_DEPTH = 14;

// nz: code 0 is no hit (the value bounds of a float encoding, see value_band); the tests are exact either way
DCDF_DEVINL void snapshot_search(const ChunkView& cv, const InstDir& s, u32 top, u32 bottom, u32 left, u32 right, i64 lower,
                                 i64 upper, Sink& sink, bool nz = false) {  // snapshot.rs:310-421; bounds inclusive here
  BitMapRef nm{cv.chunk, s.nm_len, s.nm_base};
  DacRef mx{cv.chunk, &s.max}, mn{cv.chunk, &s.min};
  if (!nm.get(0)) {
    const i64 v = mx.get(0);
    if (band_hit(v, lower, upper, nz)) sink.push_rect(top, bottom, left, right, 0, 0);
    return;
  }
  struct Frame {
    u32 sl, top, bottom, left, right, index, top_off, left_off, i, j;
    i64 minv, maxv;
  } st[SEARCH_DEPTH];
  int sp = 0;
  {
    Frame& f = st[0];
    f.sl = (u32)cv.sidelen >> 1;
    f.top = top; f.bottom = bottom; f.left = left; f.right = right;
    f.index = 1u + nm.rank(0) * 4u;
    f.top_off = 0; f.left_off = 0;
    f.minv = mn.get(0); f.maxv = mx.get(0);
    f.i = top / f.sl; f.j = left / f.sl;
  }
  while (sp >= 0) {
    Frame& f = st[sp];
    if (f.i > f.bottom / f.sl) { sp--; continue; }
    if (f.j > f.right / f.sl) { f.i++; f.j = f.left / f.sl; continue; }
    const u32 i = f.i, j = f.j;
    f.j++;
    const u32 sl = f.sl;
    const u32 top_ = f.top > i * sl ? f.top - i * sl : 0u;
    const u32 bottom_ = min(sl - 1u, f.bottom - i * sl);
    const u32 left_ = f.left > j * sl ? f.left - j * sl : 0u;
    const u32 right_ = min(sl - 1u, f.right - j * sl);
    const u32 top_off_ = f.top_off + i * sl, left_off_ = f.left_off + j * sl;
    const u32 index_ = f.index + i * 2u + j;
    const i64 maxv_ = f.maxv - mx.get(index_);
    if (index_ >= s.nm_len || !nm.get(index_)) {
      if (band_hit(maxv_, lower, upper, nz)) sink.push_rect(top_, bottom_, left_, right_, top_off_, left_off_);
    } else {
      const u32 rk = nm.rank(index_);
      const i64 minv_ = f.minv + mn.get(rk);
      if (band_all(f.minv, maxv_, lower, upper, nz)) {  // snapshot.rs:392 uses the parent's min (sic)
        sink.push_rect(top_, bottom_, left_, right_, top_off_, left_off_);
      } else if (upper >= minv_ && lower <= maxv_) {
        if (sp + 1 >= SEARCH_DEPTH || sl < 2u) continue;  // malformed input guard
        Frame& g = st[++sp];
        g.sl = sl >> 1;
        g.top = top_; g.bottom = bottom_; g.left = left_; g.right = right_;
        g.index = 1u + rk * 4u;
        g.top_off = top_off_; g.left_off = left_off_;
        g.minv = minv_; g.maxv = maxv_;
        g.i = top_ / g.sl; g.j = left_ / g.sl;
      }
    }
  }
}

// strict: the root is read as Log::get reads it (log.rs:180-186) instead of the reference's root test (SURVEY App. B #15),
// so that the hit set is exact; nz as snapshot_search
DCDF_DEVINL void log_search(const ChunkView& cv, const InstDir& l, const InstDir& s, u32 top, u32 bottom, u32 left, u32 right,
                            i64 lower, i64 upper, Sink& sink, bool strict = false, bool nz = false) {  // log.rs:519-702 (reference behaviour incl. SURVEY B#15)
  BitMapRef nm_t{cv.chunk, l.nm_len, l.nm_base}, nm_s{cv.chunk, s.nm_len, s.nm_base};
  BitMapRef eq{cv.chunk, l.eq_len, l.eq_base};
  DacRef mx_t{cv.chunk, &l.max}, mx_s{cv.chunk, &s.max}, mn_t{cv.chunk, &l.min}, mn_s{cv.chunk, &s.min};
  struct Frame {
    u32 sl, top, bottom, left, right, it, is, top_off, left_off, i, j;
    u32 flags;  // bit0 has_t, bit1 has_s, bit2 expanded
    i64 min_t, min_s, max_t, max_s;
  } st[SEARCH_DEPTH];
  int sp = 0;
  {
    Frame& f = st[0];
    f.sl = (u32)cv.sidelen;
    f.top = top; f.bottom = bottom; f.left = left; f.right = right;
    f.it = 0; f.is = 0;
    f.flags = (nm_t.get(0) ? 1u : 0u) | (nm_s.get(0) ? 2u : 0u);
    f.top_off = 0; f.left_off = 0;
    f.min_t = mn_t.get(0); f.min_s = mn_s.get(0); f.max_t = mx_t.get(0); f.max_s = mx_s.get(0);
    f.i = 0; f.j = 0;
    if (strict) {
      if (!(f.flags & 2u)) f.min_s = f.max_s;  // a single-node Snapshot has no min Dac: its one value is the max entry
      if (!(f.flags & 1u)) {
        if (!(f.flags & 2u) || !eq.get(0)) {  // a uniform single-node Log: every cell is max_s + max_t
          if (band_hit(f.max_s + f.max_t, lower, upper, nz)) sink.push_rect(top, bottom, left, right, 0, 0);
          return;
        }
        f.min_t = f.max_t;  // the snapshot plus a constant
      }
    }
  }
  while (sp >= 0) {
    Frame& f = st[sp];
    if (!(f.flags & 4u)) {
      // entry of _search_window (log.rs:576-591)
      const i64 maxv = f.max_s + f.max_t, minv = f.min_s + f.min_t;
      if (band_all(minv, maxv, lower, upper, nz)) {
        sink.push_rect(f.top, f.bottom, f.left, f.right, f.top_off, f.left_off);
        sp--;
        continue;
      } else if (band_none(minv, maxv, lower, upper, nz)) {
        sp--;
        continue;
      }
      f.sl >>= 1;
      if (f.sl == 0) { sp--; continue; }  // malformed input guard
      if (f.flags & 1u) f.it = 1u + nm_t.rank(f.it) * 4u;
      if (f.flags & 2u) f.is = 1u + nm_s.rank(f.is) * 4u;
      f.flags |= 4u;
      f.i = f.top / f.sl; f.j = f.left / f.sl;
    }
    if (f.i > f.bottom / f.sl) { sp--; continue; }
    if (f.j > f.right / f.sl) { f.i++; f.j = f.left / f.sl; continue; }
    const u32 i = f.i, j = f.j;
    f.j++;
    const u32 sl = f.sl;
    const u32 top_ = f.top > i * sl ? f.top - i * sl : 0u;
    const u32 bottom_ = min(sl - 1u, f.bottom - i * sl);
    const u32 left_ = f.left > j * sl ? f.left - j * sl : 0u;
    const u32 right_ = min(sl - 1u, f.right - j * sl);
    const bool has_t = f.flags & 1u, has_s = f.flags & 2u;
    const u32 it_ = f.it + i * 2u + j, is_ = f.is + i * 2u + j;
    const i64 max_t_ = has_t ? mx_t.get(it_) : f.max_t;
    const i64 max_s_ = has_s ? f.max_s - mx_s.get(is_) : f.max_s;
    const bool leaf_t = has_t ? (it_ >= l.nm_len || !nm_t.get(it_)) : true;
    const bool leaf_s = has_s ? (is_ >= s.nm_len || !nm_s.get(is_)) : true;
    i64 min_t_ = has_t ? (leaf_t ? f.min_t : mn_t.get(nm_t.rank(it_))) : f.min_t;
    i64 min_s_ = has_s ? (leaf_s ? f.min_s : f.min_s + mn_s.get(nm_s.rank(is_))) : f.min_s;
    u32 nflags = 0;
    if (leaf_s) min_s_ = max_s_; else nflags |= 2u;
    if (leaf_t) {
      min_t_ = max_t_;
      if (has_t && it_ < l.nm_len && !eq.get(nm_t.rank0(it_ + 1u) - 1u)) min_t_ = max_s_ + max_t_ - min_s_;
    } else {
      nflags |= 1u;
    }
    if (sp + 1 >= SEARCH_DEPTH) continue;
    Frame& g = st[++sp];
    g.sl = sl;
    g.top = top_; g.bottom = bottom_; g.left = left_; g.right = right_;
    g.it = it_; g.is = is_;
    g.flags = nflags;
    g.top_off = st[sp - 1].top_off + i * sl; g.left_off = st[sp - 1].left_off + j * sl;
    g.min_t = min_t_; g.min_s = min_s_; g.max_t = max_t_; g.max_s = max_s_;
    g.i = 0; g.j = 0;
  }
}

struct SearchParams {
  QuerySet Q;
  const CubeDev* cubes;   // [n_queries] (already re-ordered / validated on the host)
  const u64* job_base;    // [n_queries + 1] prefix of jobs per query: subchunks x instants
  u64 n_queries, n_jobs;
  const i64* lower;       // per query
  const i64* upper;
  const double* vlower;   // per query, value bounds of the strict search (dcdf_superchunk_search_values)
  const double* vupper;
  u64* counts;            // [n_jobs]  pass 1 out
  const u64* offsets;     // [n_jobs]  pass 2 in
  i64* out;               // triplets
  u64 cap;                // in triplets
};

// Job order inside a query: overlapped subchunks row-major (superchunk.rs:589-633), then instants ascending,
// then the Snapshot / Log traversal order (chunk.rs:336-383).  STRICT: value bounds, converted per job with the
// subchunk's own fractional bits (value_band), and the exact hit set (log_search's strict root, code 0 never a hit).
template <bool STRICT>
__global__ void k_search(const SearchParams P, int write) {
  const u64 ji = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (ji >= P.n_jobs) return;
  // locate the query: largest q with job_base[q] <= ji
  u64 lo = 0, hi = P.n_queries;
  while (hi - lo > 1) {
    const u64 mid = (lo + hi) >> 1;
    if (P.job_base[mid] <= ji) lo = mid; else hi = mid;
  }
  const u64 q = lo;
  const CubeDev c = P.cubes[q];
  const u64 local = ji - P.job_base[q];
  const u64 T = (u64)(c.end - c.start);
  const u64 sub = local / T;
  const i64 instant = c.start + (i64)(local - sub * T);
  const QuerySet& Q = P.Q;
  const i64 cs = Q.chunks_sidelen;
  const i64 cr0 = c.top / cs, cc0 = c.left / cs, cc1 = (c.right - 1) / cs;
  const i64 ncc = cc1 - cc0 + 1;
  const i64 cr = cr0 + (i64)(sub / (u64)ncc), cc = cc0 + (i64)(sub % (u64)ncc);
  const i64 chunk_top = cr * cs, chunk_left = cc * cs;
  const i64 wt = max(chunk_top, c.top), wb = min(chunk_top + cs, c.bottom);
  const i64 wl = max(chunk_left, c.left), wr = min(chunk_left + cs, c.right);
  const u32 top = (u32)(wt - chunk_top), bottom = (u32)(wb - chunk_top - 1);
  const u32 left = (u32)(wl - chunk_left), right = (u32)(wr - chunk_left - 1);
  i64 lower = 0, upper = 0;
  if (!STRICT) {
    lower = P.lower[q]; upper = P.upper[q];
    if (lower > upper) { const i64 t = lower; lower = upper; upper = t; }  // helpers.rs:7-16 via chunk.rs:214
  }
  bool nz = false;
  Sink sink;
  sink.n = 0;
  sink.instant = instant;
  sink.row0 = (int)chunk_top; sink.col0 = (int)chunk_left;
  sink.out = nullptr;
  if (write) {
    const u64 off = P.offsets[ji];
    const u64 cnt = P.offsets[ji + 1] - off;
    if (off + cnt > P.cap) return;
    sink.out = P.out + 3 * off;
  }
  const u32 s = (u32)(instant / Q.chunk_size);
  const SliceMeta sm = Q.slices[s];
  const u32 ti = (u32)(instant - sm.t0);
  const u32 slot = (u32)(cr * Q.subsidelen + cc);
  const int32_t u = Q.slot_unit[sm.slot_base + slot];
  if (STRICT) {
    const bool stored = u >= 0 && Q.units[u].stored;
    const FixedBand b = value_band(P.vlower[q], P.vupper[q], stored ? Q.units[u].bits : Q.slot_desc[sm.slot_base + slot].bits, Q.encoding);
    lower = b.lower; upper = b.upper; nz = b.nz;
  }
  if (Q.tbl_min) {  // superchunk.rs:480-493: the subchunk is searched only if some instant of the window can have cells in range
    const SlotDesc sd = Q.slot_desc[sm.slot_base + slot];
    const i64 t_lo = max(c.start, sm.t0) - sm.t0, t_hi = min(c.end, sm.t0 + (i64)sm.instants) - sm.t0;
    for (int lv = 0; lv <= sd.n_up; lv++)
      if (STRICT ? !slot_may_hold_part(Q, sd, t_lo, t_hi, P.vlower[q], P.vupper[q], 0, 1, lv)
                 : !slot_has_cells_part(Q, sd, t_lo, t_hi, lower, upper, 0, 1, lv)) {
        if (!write) P.counts[ji] = 0;
        return;
      }
  }
  bool done = false;
  if (u >= 0) {
    const UnitMeta m = Q.units[u];
    if (m.stored) {
      ChunkView cv{Q.blob + m.blob_off, Q.dir + m.dir_base, m.sidelen};
      const InstDir& d = cv.dir[ti];
      if (d.snap == ti) snapshot_search(cv, d, top, bottom, left, right, lower, upper, sink, nz);
      else log_search(cv, d, cv.dir[d.snap], top, bottom, left, right, lower, upper, sink, STRICT, nz);
      done = true;
    }
  }
  if (!done) {
    // Elided subchunk: one value per instant from the max table (superchunk.rs:541-559)
    const SlotDesc sdsc = Q.slot_desc[sm.slot_base + slot];
    const i64 v = Q.tbl_max[sdsc.tbl0 + (u64)ti * sdsc.stride];
    if (band_hit(v, lower, upper, nz)) sink.push_rect(top, bottom, left, right, 0, 0);
  }
  if (!write) P.counts[ji] = sink.n;
}

__global__ void k_pick_u64(const u64* offsets, const u64* idx, u64 n, u64* out) {
  const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = offsets[idx[i]];
}

// exclusive scan of u64 counts (single CTA) -- offsets[n] = total
__global__ void __launch_bounds__(1024) k_scan_u64(const u64* in, u64 n, u64* out) {
  __shared__ u64 wsum[32];
  __shared__ u64 carry_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (u64 base = 0; base < n; base += 1024u) {
    const u64 i = base + tid;
    const u64 v = i < n ? in[i] : 0ull;
    u64 x = v;
    for (int o = 1; o < 32; o <<= 1) {
      u64 y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      u64 w = wsum[lane], xs = w;
      for (int o = 1; o < 32; o <<= 1) {
        u64 y = __shfl_up_sync(0xffffffffu, xs, o);
        if (lane >= o) xs += y;
      }
      wsum[lane] = xs - w;
    }
    __syncthreads();
    const u64 carry = carry_s;
    if (i < n) out[i] = carry + wsum[warp] + x - v;
    __syncthreads();
    if (tid == 1023) carry_s = carry + wsum[warp] + x;
    __syncthreads();
  }
  if (tid == 0) out[n] = carry_s;
}

// The same scan over many CTAs for long inputs (a search batch has one count per (window, subchunk, instant)): sums of
// 8192-element chunks -> k_scan_u64 over the sums -> every chunk scanned from its offset.
constexpr int SCAN_CHUNK = 8192;
__global__ void __launch_bounds__(1024) k_scan_sums(const u64* in, u64 n, u64* sums) {
  __shared__ u64 wsum[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u64 base = (u64)blockIdx.x * SCAN_CHUNK;
  u64 s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_CHUNK / 1024; k++) {
    const u64 i = base + (u64)k * 1024u + (u64)tid;
    if (i < n) s += in[i];
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if (lane == 0) wsum[warp] = s;
  __syncthreads();
  if (warp == 0) {
    u64 w = wsum[lane];
    for (int o = 16; o > 0; o >>= 1) w += __shfl_down_sync(0xffffffffu, w, o);
    if (lane == 0) sums[blockIdx.x] = w;
  }
}
__global__ void __launch_bounds__(1024) k_scan_apply(const u64* in, u64 n, const u64* chunk_off, u64* out) {
  __shared__ u64 wsum[32];
  __shared__ u64 carry_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry_s = chunk_off[blockIdx.x];
  __syncthreads();
  const u64 base0 = (u64)blockIdx.x * SCAN_CHUNK;
  for (int k = 0; k < SCAN_CHUNK / 1024; k++) {
    const u64 i = base0 + (u64)k * 1024u + (u64)tid;
    const u64 v = i < n ? in[i] : 0ull;
    u64 x = v;
    for (int o = 1; o < 32; o <<= 1) {
      u64 y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      u64 w = wsum[lane], xs = w;
      for (int o = 1; o < 32; o <<= 1) {
        u64 y = __shfl_up_sync(0xffffffffu, xs, o);
        if (lane >= o) xs += y;
      }
      wsum[lane] = xs - w;
    }
    __syncthreads();
    const u64 carry = carry_s;
    if (i < n) out[i] = carry + wsum[warp] + x - v;
    __syncthreads();
    if (tid == 1023) carry_s = carry + wsum[warp] + x;
    __syncthreads();
  }
  if (blockIdx.x == gridDim.x - 1 && tid == 0) out[n] = chunk_off[gridDim.x];
}

// flat to_fixed / from_fixed (fixed.rs:31-86)
template <typename F>
__global__ void k_to_fixed(const F* in, u64 n, int bits, int round, i64* out, u32* err) {
  u32 e = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
    out[i] = to_fixed_dev<F>(in[i], bits, round != 0, e);
  if (e) atomicOr(err, e);
}
template <typename F>
__global__ void k_from_fixed(const i64* in, u64 n, int bits, F* out) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
    out[i] = from_fixed_dev<F>(in[i], bits);
}

}  // namespace dcdf
