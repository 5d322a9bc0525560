// decode_search4.cuh -- batched value-range search over whole <=64x64 tiles with the per-thread walk of decode_tile4.cuh.
//
// Snapshot::search_window (snapshot.rs:310-421), Log::search_window (log.rs:519-702), Chunk::iter_search
// (chunk.rs:213-228,336-383), Superchunk::search (superchunk.rs:464-585).  k_search (decode.cuh) replays the reference's
// depth-first traversal with one thread per (window, subchunk, instant): correct, but its lanes diverge completely
// (3 of 32 active per instruction).  Here one CTA handles a (window, time slice, subchunk) and one thread owns a 4x4
// block of cells: per instant it walks root -> block with exactly the state the reference recursion carries down that
// path (index_t / min_t / max_t of the Log, min_s / max_s of the Snapshot from the expanded pyramid), applies the
// reference's tests at every node, then classifies its four quads and sixteen cells.  The result SET is what the
// traversal finds; the result ORDER is reproduced as well: the reference pushes the cells of a node that passes the
// "all inside" test (or of a leaf node) row-major over the node's clipped rectangle, and nodes in child order.  So a cell
// found below such a node E (level <= L-2) goes to base(E) + its row-major offset in E's rectangle, base(E) being the
// number of hits before E's first block in Morton order (one block-wide scan of the per-thread counts); inside a 4x4
// block the traversal order is the Morton order of the hits.  Two launches as before: count, (host scan), write.
#pragma once
#include "decode_tile4.cuh"

namespace dcdf {

struct SearchJob {
  i64 lower, upper;
  int top, bottom, left, right;  // window clipped to the tile, tile coordinates, exclusive ends
  i64 row0, col0;                // raster coordinates of the tile's origin
  bool nz;                       // strict search: code 0 (NaN) is no hit although it lies in [lower, upper]
};
// per thread: its 4x4 block / some block of its warp touches the window -- the others never need their part of any
// pyramid (a thread only reads what it wrote itself)
struct SearchAct {
  bool act, warp_act;
};

template <typename V>
struct Search4Smem {
  static constexpr int BUF = sizeof(V) == 4 ? 10 * 1024 : 16 * 1024;
  static constexpr bool PRIVATE_TOP = false;
  __align__(16) V cells[4096];
  __align__(16) V sup[W3_UPPER];   // snapshot max of every node above the cells
  __align__(16) V smin[W3_UPPER];  // snapshot min as the Log recursion sees it: accumulated for internal nodes, = max below
                                   // a leaf (log.rs:651-654), the literal min.get(0) at the root
  RankTab tab[DT_WARPS];
  V suptop[DT_WARPS][8];
  u32 single[DT_WARPS];
  u32 base[DT_THREADS];            // exclusive prefix of the per-thread hit counts of the current instant
  u32 wsum[DT_WARPS];
  SearchJob job;                   // the CTA's current job (uniform; kept here instead of in every thread's registers)
  FixedBand band;                  // strict search: the job's band, converted once by thread 0
  __align__(16) InstDir dir[3];
  __align__(16) u8 stage[2][BUF + 32];
};


// what a thread found for its 4x4 block: e_lvl >= 0: an ancestor of level e_lvl (or the block itself) emits its whole
// rectangle; otherwise m16 = hits in Morton order (bit 4 * quad + cell)
struct Hit {
  int e_lvl;
  u32 m16;
};

// ST (strict, dcdf_superchunk_search_values): the band is the job's converted value bounds and the hit set is exact.  The
// fixed-bound search compiles without the code-0 tests.
template <bool ST, typename V>
DCDF_DEVINL bool in_band(V v, const SearchJob& J) { return band_hit((i64)v, J.lower, J.upper, ST && J.nz); }

// Snapshot: expansion of the pyramid (max, min, cells) and, with `search`, the tests of snapshot.rs:371-413 on the way.
template <typename V, typename S_, bool ST>
DCDF_DEVINL Hit snapshot4s(const u8* chunk, const InstDir& d, int L, S_& S, bool search, const SearchJob& J, const SearchAct A) {
  const u32 p = threadIdx.x;
  RankTab& T = S.tab[threadIdx.x >> 5];
  const u32 nm_len = d.nm_len;
  const u8* nmb = bitmap_bits(chunk, nm_len, d.nm_base);
  const Dac4 mx = dac4_of(chunk, &d.max), mn = dac4_of(chunk, &d.min);
  bool has = bit_at(nmb, 0);
  V val = dac_get1<V>(mx, 0), mnv = dac_get1<V>(mn, 0);  // an empty min DAC yields 0 (dac.rs:80-93)
  u32 r = 0;
  if (p == 0) { S.sup[0] = val; S.smin[0] = mnv; S.single[0] = has ? 0u : 1u; }
  if (!A.warp_act) return Hit{-1, 0u};
  build_rank(nmb, nm_len, T);
  Hit h{-1, 0u};
  bool live = search;  // still descending
  if (search && !has) {  // single node (snapshot.rs:318-326)
    live = false;
    h.e_lvl = in_band<ST>(val, J) ? 0 : -1;
  }
  const int lvp = L - 2;
  if (p >= (1u << (2 * lvp)) || !A.act) return Hit{-1, 0u};
  for (int k = 1; k <= lvp; k++) {
    const u32 pk = p >> (2 * (lvp - k));
    if (has) {
      const V pmin = mnv;
      const u32 cidx = 1u + 4u * r + (pk & 3u);
      val -= dac_get1<V>(mx, cidx);
      has = cidx < nm_len && tab_bit(T, cidx);
      if (has) { r = tab_rank(T, cidx); mnv = pmin + dac_get1<V>(mn, r); } else mnv = val;
      if (live) {
        if (!has) { live = false; if (in_band<ST>(val, J)) h.e_lvl = k; }                                  // leaf node
        else if (band_all((i64)pmin, (i64)val, J.lower, J.upper, ST && J.nz)) { live = false; h.e_lvl = k; }  // parent's min (sic, :392)
        else if (!(J.upper >= (i64)mnv && J.lower <= (i64)val)) live = false;                            // pruned
      }
    } else {
      mnv = val;
    }
    sup_at(S, k, pk) = val;
    S.smin[off3(k) + pk] = mnv;
  }
  // the quads and the cells
  V dq[4] = {0, 0, 0, 0};
  u32 inb = 0, rq = 0;
  if (has) {
    const u32 idx0 = 1u + 4u * r;
    dac_get4<V>(mx, idx0, dq);
    if (idx0 < nm_len) { inb = tab_bits4(T, idx0); rq = tab_rank(T, idx0); }
  }
  Quad<V> qv, qm;
#pragma unroll
  for (int c = 0; c < 4; c++) {
    qv.c[c] = val - dq[c];
    qm.c[c] = (inb >> c) & 1u ? mnv + dac_get1<V>(mn, rq + below(inb, c)) : qv.c[c];
  }
  *reinterpret_cast<Quad<V>*>(&S.sup[off3(L - 1) + 4u * p]) = qv;
  *reinterpret_cast<Quad<V>*>(&S.smin[off3(L - 1) + 4u * p]) = qm;
#pragma unroll
  for (int c = 0; c < 4; c++) {
    V dd[4] = {0, 0, 0, 0};
    const bool qin = (inb >> c) & 1u;
    if (qin) dac_get4<V>(mx, 1u + 4u * (rq + below(inb, c)), dd);
    Quad<V> q;
#pragma unroll
    for (int i = 0; i < 4; i++) q.c[i] = qv.c[c] - dd[i];
    reinterpret_cast<Quad<V>*>(S.cells)[4u * p + (u32)c] = q;
    if (live && has) {  // the block's node is a branch that was entered: its children are the quads
      if (!qin) { if (in_band<ST>(qv.c[c], J)) h.m16 |= 15u << (4 * c); }
      else if (band_all((i64)mnv, (i64)qv.c[c], J.lower, J.upper, ST && J.nz)) h.m16 |= 15u << (4 * c);
      else if (J.upper >= (i64)qm.c[c] && J.lower <= (i64)qv.c[c]) {
#pragma unroll
        for (int i = 0; i < 4; i++)
          if (in_band<ST>(q.c[i], J)) h.m16 |= 1u << (4 * c + i);
      }
    }
  }
  return h;
}

// One entry test of Log::_search_window (log.rs:576-591): +1 all inside, -1 disjoint, 0 descend
template <bool ST, typename V>
DCDF_DEVINL int log_test(V min_s, V min_t, V max_s, V max_t, const SearchJob& J) {
  const i64 mn = (i64)min_s + (i64)min_t, mx = (i64)max_s + (i64)max_t;
  if (band_all(mn, mx, J.lower, J.upper, ST && J.nz)) return 1;
  if (band_none(mn, mx, J.lower, J.upper, ST && J.nz)) return -1;
  return 0;
}

// Log: the recursion's state down the thread's path, against the snapshot pyramid in S (log.rs:593-700).
template <typename V, typename S_, bool ST>
DCDF_DEVINL Hit log4s(const u8* chunk, const InstDir& d, int L, S_& S, const SearchJob& J, const SearchAct A) {
  const u32 p = threadIdx.x;
  RankTab& T = S.tab[threadIdx.x >> 5];
  const u32 nm_len = d.nm_len;
  const u8* nmb = bitmap_bits(chunk, nm_len, d.nm_base);
  const u8* eq = bitmap_bits(chunk, d.eq_len, d.eq_base);
  const Dac4 mx = dac4_of(chunk, &d.max), mn = dac4_of(chunk, &d.min);
  // the root's test is the same for every thread: a disjoint root ends the instant for the whole CTA (e_lvl = -2)
  // before the rank table is built
  V max_t = dac_get1<V>(mx, 0), min_t = dac_get1<V>(mn, 0);
  V min_s0 = S.smin[0];
  if (ST) {
    // the root as Log::get / the window decoder read it (log4), not the reference's root test (SURVEY App. B #15)
    if (S.single[0]) min_s0 = S.sup[0];  // a single-node Snapshot has no min Dac: its one value is the max entry
    if (!bit_at(nmb, 0)) {
      if (S.single[0] || !bit_at(eq, 0)) return in_band<ST>((V)(S.sup[0] + max_t), J) ? Hit{0, 0u} : Hit{-2, 0u};  // uniform
      min_t = max_t;  // the snapshot plus a constant
    }
  }
  int st = log_test<ST, V>(min_s0, min_t, S.sup[0], max_t, J);
  if (st < 0) return Hit{-2, 0u};
  if (!A.warp_act) return Hit{-1, 0u};
  build_rank(nmb, nm_len, T);
  const int lvp = L - 2;
  if (p >= (1u << (2 * lvp)) || !A.act) return Hit{-1, 0u};
  bool has_t = T.W[0] >> 31;  // index_t is Some
  u32 r = 0;                  // rank1 of the current log node (its children start at 1 + 4r)
  Hit h{-1, 0u};
  if (st > 0) h.e_lvl = 0;
  // one step of the children loop: node with BFS index cidx (when the parent is internal) over snapshot (min_s, max_s)
  auto step = [&](u32 c, V min_s, V max_s) {
    if (has_t) {
      const u32 cidx = 1u + 4u * r + c;
      max_t = dac_get1<V>(mx, cidx);
      const bool known = cidx < nm_len;
      const u32 rc = known ? tab_rank(T, cidx) : 0u;
      if (known && tab_bit(T, cidx)) {
        r = rc;
        min_t = dac_get1<V>(mn, rc);  // replaced, like max_t (log.rs:634)
      } else {
        min_t = max_t;
        if (known && !(cidx - rc < d.eq_len && bit_at(eq, cidx - rc))) min_t = max_s + max_t - min_s;  // log.rs:661-667
        has_t = false;
      }
    } else {
      min_t = max_t;  // leaf_t with index None (log.rs:658-660)
    }
  };
  for (int k = 1; k <= lvp && st == 0; k++) {
    const u32 pk = p >> (2 * (lvp - k));
    const V max_s = sup_at(S, k, pk), min_s = S.smin[off3(k) + pk];
    step(pk & 3u, min_s, max_s);
    st = log_test<ST, V>(min_s, min_t, max_s, max_t, J);
    if (st > 0) h.e_lvl = k;
  }
  if (st != 0) return h;
  // quads and cells below the block's node
  const Quad<V> qs = *reinterpret_cast<const Quad<V>*>(&S.sup[off3(L - 1) + 4u * p]);
  const Quad<V> qn = *reinterpret_cast<const Quad<V>*>(&S.smin[off3(L - 1) + 4u * p]);
  const bool b_has = has_t;
  const u32 b_r = r;
  const V b_max = max_t;
#pragma unroll
  for (int c = 0; c < 4; c++) {
    has_t = b_has; r = b_r; max_t = b_max;
    step((u32)c, qn.c[c], qs.c[c]);
    const int sq = log_test<ST, V>(qn.c[c], min_t, qs.c[c], max_t, J);
    if (sq > 0) h.m16 |= 15u << (4 * c);
    if (sq != 0) continue;
    const Quad<V> q = reinterpret_cast<const Quad<V>*>(S.cells)[4u * p + (u32)c];
    V dd[4];
    if (has_t) dac_get4<V>(mx, 1u + 4u * r, dd);  // leaves: max_t replaced by the cell's entry, no nodemap bit below
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const V mt = has_t ? dd[i] : max_t;
      if (in_band<ST>((V)(q.c[i] + mt), J)) h.m16 |= 1u << (4 * c + i);
    }
  }
  return h;
}

// Counts (pass 0) or writes (pass 1) the hits of one instant in the reference's order.
template <typename V, typename S_>
DCDF_DEVINL void emit_hits(const Hit h, int L, S_& S, const SearchJob& J, i64 instant, u64* count_out, i64* out, u64 off, u64 cap) {
  const u32 p = threadIdx.x, lane = p & 31u, warp = p >> 5;
  const int lvp = L - 2;
  const bool valid = p < (1u << (2 * lvp));
  const int R0 = 4 * (int)morton_row(p), C0 = 4 * (int)morton_col(p);
  u32 w16 = 0;  // cells of the block inside the window
  if (valid) {
#pragma unroll
    for (int b = 0; b < 16; b++) {
      const int rr = R0 + 2 * ((b >> 3) & 1) + ((b >> 1) & 1), cc = C0 + 2 * ((b >> 2) & 1) + (b & 1);
      if (rr >= J.top && rr < J.bottom && cc >= J.left && cc < J.right) w16 |= 1u << b;
    }
  }
  const u32 mine = h.e_lvl >= 0 ? w16 : (h.m16 & w16);
  const u32 n = __popc(mine);
  if (!out) {
    // counting pass: the instant's total is all that is needed -- one atomic per warp into the zeroed count, no barrier
    const u32 wt = __reduce_add_sync(0xffffffffu, n);
    if (lane == 0 && wt) atomicAdd(reinterpret_cast<unsigned long long*>(count_out), (unsigned long long)wt);
    return;
  }
  u32 inc = n;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 y = __shfl_up_sync(0xffffffffu, inc, o);
    if ((int)lane >= o) inc += y;
  }
  if (lane == 31) S.wsum[warp] = inc;
  __syncthreads();
  u32 before = 0, total = 0;
#pragma unroll
  for (int w = 0; w < DT_WARPS; w++) {
    const u32 x = S.wsum[w];
    if (w < (int)warp) before += x;
    total += x;
  }
  const u32 base = before + inc - n;
  S.base[p] = base;
  __syncthreads();
  if (!mine || off + total > cap) return;
  i64* o3 = out + 3 * off;
  if (h.e_lvl >= 0) {
    const int side = 1 << (L - h.e_lvl);
    const int Er = R0 & ~(side - 1), Ec = C0 & ~(side - 1);
    const u32 span = 1u << (2 * (lvp - h.e_lvl));  // blocks below the emitting node
    const u32 bE = S.base[p & ~(span - 1u)];
    const int rt = max(Er, J.top), cl = max(Ec, J.left), cr = min(Ec + side, J.right);
    const int width = cr - cl;
#pragma unroll 1
    for (int b = 0; b < 16; b++) {
      if (!((mine >> b) & 1u)) continue;
      const int rr = R0 + 2 * ((b >> 3) & 1) + ((b >> 1) & 1), cc = C0 + 2 * ((b >> 2) & 1) + (b & 1);
      const u64 pos = (u64)bE + (u64)((rr - rt) * width + (cc - cl));
      o3[3 * pos] = instant; o3[3 * pos + 1] = J.row0 + rr; o3[3 * pos + 2] = J.col0 + cc;
    }
  } else {
    u64 pos = base;
#pragma unroll 1
    for (int b = 0; b < 16; b++) {
      if (!((mine >> b) & 1u)) continue;
      const int rr = R0 + 2 * ((b >> 3) & 1) + ((b >> 1) & 1), cc = C0 + 2 * ((b >> 2) & 1) + (b & 1);
      o3[3 * pos] = instant; o3[3 * pos + 1] = J.row0 + rr; o3[3 * pos + 2] = J.col0 + cc;
      pos++;
    }
  }
}

template <typename V, typename S_, bool ST>
DCDF_DEVINL Hit instant4s(const u8* base, const InstDir& d, bool is_snap, bool search, int L, S_& S, const SearchJob& J, const SearchAct A) {
  return is_snap ? snapshot4s<V, S_, ST>(base, d, L, S, search, J, A) : log4s<V, S_, ST>(base, d, L, S, J, A);
}
// structures that do not fit the staging buffer are read from global memory by an out-of-line copy of the same code
template <typename V, typename S_, bool ST>
__device__ __noinline__ void instant4s_global(const u8* chunk, const InstDir* d, bool is_snap, bool search, int L, S_* S, int act, Hit* h) {
  *h = instant4s<V, S_, ST>(chunk, *d, is_snap, search, L, *S, S->job, SearchAct{(act & 1) != 0, (act & 2) != 0});
}

struct TileSearchParams {
  QuerySet Q;
  const CubeDev* cubes;
  const u64* job_base;       // [n + 1] prefix of (subchunk, instant) jobs per query -- the index space of counts / offsets
  const u64* tile_base;      // [n + 1] prefix of (time slice, subchunk) CTAs jobs per query
  u64 n_queries, n_tiles;
  const i64* lower;
  const i64* upper;
  const double* vlower;      // value bounds of the strict search (k_search_tiles4<V, true>)
  const double* vupper;
  u64* counts;
  const u64* offsets;
  i64* out;                  // null in the counting pass
  u64 cap;
  u32* hit_cache;            // [n_jobs][256] what every thread found in the counting pass ((e_lvl + 1) << 16 | m16), or null:
                             // the writing pass then places the hits without staging or expanding anything again
};

template <typename V, bool ST>
__global__ void __launch_bounds__(DT_THREADS, sizeof(V) == 4 ? 4 : 2) k_search_tiles4(const TileSearchParams P) {
  extern __shared__ __align__(16) unsigned char ds4_smem_raw[];
  typedef Search4Smem<V> SM;
  SM& S = *reinterpret_cast<SM*>(ds4_smem_raw);
  const QuerySet& Q = P.Q;
  const int tid = threadIdx.x;
  for (u64 ji = blockIdx.x; ji < P.n_tiles; ji += gridDim.x) {
    u64 lo_q = 0, hi_q = P.n_queries;
    while (hi_q - lo_q > 1) {
      const u64 mid = (lo_q + hi_q) >> 1;
      if (P.tile_base[mid] <= ji) lo_q = mid; else hi_q = mid;
    }
    const u64 q = lo_q;
    const CubeDev c = P.cubes[q];
    const u64 local = ji - P.tile_base[q];
    const i64 cs = Q.chunks_sidelen;
    const i64 cr0 = c.top / cs, cc0 = c.left / cs;
    const i64 ncr = (c.bottom - 1) / cs - cr0 + 1, ncc = (c.right - 1) / cs - cc0 + 1;
    const u64 nsub = (u64)(ncr * ncc);
    const u32 s = (u32)(c.start / Q.chunk_size) + (u32)(local / nsub);
    const u64 sub = local % nsub;
    const i64 cr = cr0 + (i64)(sub / (u64)ncc), cc = cc0 + (i64)(sub % (u64)ncc);
    const SliceMeta sm = Q.slices[s];
    const i64 t_lo = max(c.start, sm.t0), t_hi = min(c.end, sm.t0 + (i64)sm.instants);
    if (t_hi <= t_lo) continue;
    const i64 chunk_top = cr * cs, chunk_left = cc * cs;
    const u32 slot = (u32)(cr * Q.subsidelen + cc);
    const int32_t u = Q.slot_unit[sm.slot_base + slot];
    const UnitMeta m = u >= 0 ? Q.units[u] : UnitMeta{};
    const bool stored = u >= 0 && m.stored;
    SearchJob J;  // local copy: the elided / tiny-tile paths use it, the walk reads the CTA's copy in shared memory
    if (ST) {
      // the band of this subchunk's own fractional bits (an Elided slot: its node's); the binary search runs once per job
      __syncthreads();  // everyone has read the previous job's band
      if (tid == 0) S.band = value_band(P.vlower[q], P.vupper[q], stored ? m.bits : Q.slot_desc[sm.slot_base + slot].bits, Q.encoding);
      __syncthreads();
      J.lower = S.band.lower; J.upper = S.band.upper; J.nz = S.band.nz;
    } else {
      J.lower = P.lower[q]; J.upper = P.upper[q]; J.nz = false;
      if (J.lower > J.upper) { const i64 t = J.lower; J.lower = J.upper; J.upper = t; }  // helpers.rs:7-16 via chunk.rs:214
    }
    J.top = (int)(max(chunk_top, c.top) - chunk_top); J.bottom = (int)(min(chunk_top + cs, c.bottom) - chunk_top);
    J.left = (int)(max(chunk_left, c.left) - chunk_left); J.right = (int)(min(chunk_left + cs, c.right) - chunk_left);
    J.row0 = chunk_top; J.col0 = chunk_left;
    SearchAct A;
    {
      const int R0 = 4 * (int)morton_row((u32)tid), C0 = 4 * (int)morton_col((u32)tid);
      A.act = R0 + 4 > J.top && R0 < J.bottom && C0 + 4 > J.left && C0 < J.right;
      A.warp_act = __any_sync(0xffffffffu, A.act);
    }
    const int act_bits = (A.act ? 1 : 0) | (A.warp_act ? 2 : 0);
    const u64 T_all = (u64)(c.end - c.start);
    const u64 job0 = P.job_base[q] + sub * T_all;  // + (t - c.start)
    if (Q.tbl_min) {
      // Superchunk::search only looks into subchunks whose min / max entries say that some instant of the window can have
      // cells in range (superchunk.rs:480-493), at every level of a nested superchunk; the counts of a pruned job stay 0
      const SlotDesc sd = Q.slot_desc[sm.slot_base + slot];
      bool pruned = false;
      for (int lv = 0; lv <= sd.n_up; lv++)
        if (!__syncthreads_or((ST ? slot_may_hold_part(Q, sd, t_lo - sm.t0, t_hi - sm.t0, P.vlower[q], P.vupper[q], tid, DT_THREADS, lv)
                                  : slot_has_cells_part(Q, sd, t_lo - sm.t0, t_hi - sm.t0, J.lower, J.upper, tid, DT_THREADS, lv)) ? 1 : 0))
          pruned = true;
      if (pruned) continue;
    }
    const int L = stored ? 31 - __clz(m.sidelen) : 0;
    if (!stored) {
      // Elided subchunk: one value per instant from the max table (superchunk.rs:541-559); the window's cells row-major
      const SlotDesc sdsc = Q.slot_desc[sm.slot_base + slot];
      const int wc = J.right - J.left;
      const u64 area = (u64)(J.bottom - J.top) * (u64)wc;
      for (i64 t = t_lo; t < t_hi; t++) {
        const u64 jb = job0 + (u64)(t - c.start);
        const i64 v = Q.tbl_max[sdsc.tbl0 + (u64)(t - sm.t0) * sdsc.stride];
        const bool hit = band_hit(v, J.lower, J.upper, ST && J.nz);
        if (!P.out) {
          if (tid == 0) P.counts[jb] = hit ? area : 0ull;
        } else if (hit) {
          const u64 off = P.offsets[jb];
          if (off + area > P.cap) continue;
          for (u64 i = tid; i < area; i += DT_THREADS) {
            i64* o3 = P.out + 3 * (off + i);
            o3[0] = t; o3[1] = chunk_top + J.top + (i64)(i / (u64)wc); o3[2] = chunk_left + J.left + (i64)(i % (u64)wc);
          }
        }
      }
      continue;
    }
    if (L < 2) {
      // 2x2 tiles: the depth-first kernel's code, thread 0
      if (tid == 0) {
        for (i64 t = t_lo; t < t_hi; t++) {
          const u64 jb = job0 + (u64)(t - c.start);
          Sink sink;
          sink.n = 0; sink.instant = t; sink.row0 = (int)chunk_top; sink.col0 = (int)chunk_left; sink.out = nullptr;
          if (P.out) {
            const u64 off = P.offsets[jb];
            if (off + (P.offsets[jb + 1] - off) > P.cap) continue;
            sink.out = P.out + 3 * off;
          }
          const u32 ti = (u32)(t - sm.t0);
          ChunkView cv{Q.blob + m.blob_off, Q.dir + m.dir_base, m.sidelen};
          const InstDir& dd = cv.dir[ti];
          if (dd.snap == ti) snapshot_search(cv, dd, (u32)J.top, (u32)(J.bottom - 1), (u32)J.left, (u32)(J.right - 1), J.lower, J.upper, sink, ST && J.nz);
          else log_search(cv, dd, cv.dir[dd.snap], (u32)J.top, (u32)(J.bottom - 1), (u32)J.left, (u32)(J.right - 1), J.lower, J.upper, sink, ST, ST && J.nz);
          if (!P.out) P.counts[jb] = sink.n;
        }
      }
      continue;
    }
    const u8* chunk = Q.blob + m.blob_off;
    const InstDir* dir = Q.dir + m.dir_base;
    const u32 ti0 = (u32)(t_lo - sm.t0), n_t = (u32)(t_hi - t_lo);
    __syncthreads();  // the previous job's readers are done with the staging buffers and the job description
    if (tid == 0) S.job = J;
    __syncthreads();
    const SearchJob& JS = S.job;
    if (P.out && P.hit_cache) {
      for (u32 i = 0; i < n_t; i++) {
        const u64 jb = job0 + (u64)(t_lo + i - c.start);
        if (P.offsets[jb + 1] == P.offsets[jb]) continue;  // uniform
        const u32 pk = P.hit_cache[jb * DT_THREADS + (u64)tid];
        const Hit h{(int)(pk >> 16) - 1, pk & 0xffffu};
        emit_hits<V, SM>(h, L, S, JS, t_lo + (i64)i, P.counts + jb, P.out, P.offsets[jb], P.cap);
        __syncthreads();  // wsum / base are reused by the next instant
      }
      continue;
    }
    const u32 snap0 = dir[ti0].snap;
    if (snap0 != ti0) {
      // the window starts inside a block: expand the block's snapshot first
      prefetch_dir4<V, SM>(dir + snap0, S, 2);
      prefetch4<V, SM>(chunk, dir[snap0].off, dir[snap0].size, S, 1);
      cp_async_wait_all();
      __syncthreads();
      u32 delta;
      Hit hg;
      if (staged4<V>(chunk, S.dir[2], delta)) instant4s<V, SM, ST>(S.stage[1] + (int32_t)delta, S.dir[2], true, false, L, S, JS, A);
      else instant4s_global<V, SM, ST>(chunk, &S.dir[2], true, false, L, &S, act_bits, &hg);
      __syncthreads();
    }
    prefetch_dir4<V, SM>(dir + ti0, S, 0);
    prefetch4<V, SM>(chunk, dir[ti0].off, dir[ti0].size, S, 0);
    if (n_t > 1) prefetch_dir4<V, SM>(dir + ti0 + 1, S, 1);
    u32 rs = 0;  // i % 3
    for (u32 i = 0; i < n_t; i++) {
      const int b = (int)(i & 1u);
      const u32 ti = ti0 + i;
      const u32 slot1 = rs == 2 ? 0u : rs + 1u, slot2 = slot1 == 2 ? 0u : slot1 + 1u;
      cp_async_wait_all();
      __syncthreads();  // structure i and directory entry i+1 have landed; everyone is done with instant i-1
      if (i + 1 < n_t) {
        prefetch4<V, SM>(chunk, S.dir[slot1].off, S.dir[slot1].size, S, b ^ 1);
        if (i + 2 < n_t) prefetch_dir4<V, SM>(dir + ti + 2, S, slot2);
      }
      const InstDir& D = S.dir[rs];
      rs = slot1;
      const u64 jb = job0 + (u64)(t_lo + i - c.start);
      const bool is_snap = D.snap == ti;
      // writing pass: an instant the counting pass found empty is skipped (a Snapshot is still expanded for its Logs)
      const bool want = !P.out || P.offsets[jb + 1] != P.offsets[jb];
      if (!want && !is_snap) continue;
      u32 delta;
      Hit h;
      if (staged4<V>(chunk, D, delta)) h = instant4s<V, SM, ST>(S.stage[b] + (int32_t)delta, D, is_snap, want, L, S, JS, A);
      else instant4s_global<V, SM, ST>(chunk, &D, is_snap, want, L, &S, act_bits, &h);
      if (!want) continue;
      if (h.e_lvl == -2) continue;  // CTA-uniform: nothing of this instant is inside the band (its count stays 0)
      if (!P.out && P.hit_cache) P.hit_cache[jb * DT_THREADS + (u64)tid] = ((u32)(h.e_lvl + 1) << 16) | (h.m16 & 0xffffu);
      emit_hits<V, SM>(h, L, S, JS, t_lo + (i64)i, P.counts + jb, P.out, P.out ? P.offsets[jb] : 0ull, P.cap);
    }
  }
}

}  // namespace dcdf
