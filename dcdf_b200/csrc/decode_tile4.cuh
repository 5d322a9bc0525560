// decode_tile4.cuh -- window decode of whole <=64x64 tiles, barrier-free expansion.
//
// Same contract as k_window_tiles / k_window_tiles3 (Snapshot::fill_window snapshot.rs:204-301, Log::fill_window
// log.rs:311-508, Chunk::fill_window chunk.rs:152-158, Superchunk::fill_window superchunk.rs:402-457).
//
// One thread owns one 4x4 block of cells (a node of level L-2) for the whole job.  Per instant it walks from the root to
// that node the way Snapshot::get / Log::get do (snapshot.rs:165-188, log.rs:207-293: child = 1 + rank(idx) * k^2 + c),
// then decodes the node's four quads and sixteen cells with 4-entry fetches (decode_tile3.cuh).  Threads of a warp
// share their ancestors, so the walk's loads are broadcasts; nothing a thread reads was written by another thread
// (snapshot values of its ancestors and cells are rewritten, identically, by every thread below them), hence no
// barrier inside an instant.  rank() comes from a per-warp table over the staged nodemap (ones before each 32-bit
// word + the word itself, MSB first): two shared-memory loads and a popcount instead of the byte-order-dependent walk
// over the serialized rank directory (bitmap.rs:186-212).  The only block barrier per instant publishes the bytes
// that cp.async brought in while the previous instant was being decoded.
#pragma once
#include "decode_tile_common.cuh"

namespace dcdf {

constexpr int W4_TABW = 48;  // nodemap words of a 64x64 tree: ceil(1365 / 32) = 43

struct RankTab {
  u32 R[W4_TABW];  // ones before word j
  u32 W[W4_TABW];  // word j, bit i of the stream at position 31 - (i % 32)
};

template <typename V>
struct Tile4Smem {
  static constexpr int BUF = sizeof(V) == 4 ? 10 * 1024 : 16 * 1024;
  static constexpr bool PRIVATE_TOP = false;  // one block barrier per instant: warps share levels 0 and 1 of `sup`
  __align__(16) V cells[4096];     // snapshot values of the cells, Morton order (quad q = cells[4q .. 4q+3])
  __align__(16) V sup[W3_UPPER];   // snapshot max values of the levels above the cells (off3 layout)
  RankTab tab[DT_WARPS];
  V suptop[DT_WARPS][8];           // per-warp copies of the snapshot values of levels 0 and 1 (nodes shared between warps)
  u32 single[DT_WARPS];            // per warp: the block's snapshot is a single node
  __align__(16) InstDir dir[3];    // ring of directory entries: instant i in dir[i % 3], fetched two instants ahead
  __align__(16) u8 stage[2][BUF + 32];
};

// Per warp: rank table of the nodemap whose words start at byte pointer `bits` (any alignment).
DCDF_DEVINL void build_rank(const u8* bits, u32 nm_len, RankTab& T) {
  const u32 lane = threadIdx.x & 31u;
  const u32 nw = min((nm_len + 31u) / 32u, (u32)(W4_TABW - 2));
  const u32 j = 2u * lane;
  // big-endian words at any byte alignment from three aligned loads (the misalignment is the same for every word)
  const uintptr_t a = (uintptr_t)bits + 8u * lane;
  const u32* al = reinterpret_cast<const u32*>(a & ~(uintptr_t)3);
  const u32 mis = (u32)(a & 3u);
  const u32 sel = (mis + 3u) | ((mis + 2u) << 4) | ((mis + 1u) << 8) | (mis << 12);
  u32 w0 = 0, w1 = 0;
  if (j < nw) {
    const u32 x0 = al[0], x1 = al[1], x2 = al[2];  // x2 may lie past the bitmap, inside the staged structure
    w0 = __byte_perm(x0, x1, sel);
    if (j + 1u < nw) w1 = __byte_perm(x1, x2, sel);
  }
  const u32 c0 = __popc(w0), s = c0 + __popc(w1);
  u32 inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const u32 y = __shfl_up_sync(0xffffffffu, inc, o);
    if ((int)lane >= o) inc += y;
  }
  __syncwarp();  // the previous instant's readers of this table are done
  if (j < (u32)W4_TABW) {
    T.W[j] = w0; T.R[j] = inc - s;
    T.W[j + 1u] = w1; T.R[j + 1u] = inc - s + c0;
  }
  __syncwarp();
}
DCDF_DEVINL u32 tab_word(u32 idx) { return min(idx >> 5, (u32)(W4_TABW - 2)); }
DCDF_DEVINL u32 tab_rank(const RankTab& T, u32 idx) {  // ones in [0, idx)  (bitmap.rs:186-212)
  const u32 w = tab_word(idx);
  return T.R[w] + __popc(T.W[w] & ~(0xffffffffu >> (idx & 31u)));
}
DCDF_DEVINL bool tab_bit(const RankTab& T, u32 idx) { return (T.W[tab_word(idx)] >> (31u - (idx & 31u))) & 1u; }
DCDF_DEVINL u32 tab_bits4(const RankTab& T, u32 idx) {  // bits idx .. idx+3 as a mask, bit c = stream bit idx + c
  const u32 w = tab_word(idx);
  return __brev(__funnelshift_l(T.W[w + 1u], T.W[w], idx & 31u)) & 15u;
}

// Snapshot value of node pk of level k.  Levels 0 and 1 are shared between warps; a layout with PRIVATE_TOP keeps a copy
// per warp so that no warp ever reads what another one wrote (needed by a decoder whose warps drift apart by more than one
// instant -- the bulk-copy ring measured in round 1, DESIGN section 6; every shipped layout has PRIVATE_TOP = false).
template <typename S_>
DCDF_DEVINL auto& sup_at(S_& S, int k, u32 pk) {
  if (!S_::PRIVATE_TOP) return S.sup[off3(k) + pk];
  const u32 warp = threadIdx.x >> 5;
  return k <= 1 ? S.suptop[warp][k ? 1u + (pk & 3u) : 0u] : S.sup[off3(k) + pk];
}
template <typename S_>
DCDF_DEVINL u32 top_slot() { return S_::PRIVATE_TOP ? threadIdx.x >> 5 : 0u; }

// Cells of this thread's 4x4 block for one instant, given the state of its level L-2 node: mode 0 internal (r = rank1 of
// the node, its quads start at BFS index 1 + 4r), 1 uniform (value = pay), 2 equal (value = pay + snapshot cell).
template <typename V, typename S_, typename OUT>
DCDF_DEVINL void block4(const Dac4& mx, const u8* eq, u32 eq_len, const RankTab& T, u32 nm_len, u32 mode, V pay, u32 r, u32 p, u32 oQ,
                       const S_& S, const OUT& O) {
  const int R0 = 4 * (int)morton_row(p), C0 = 4 * (int)morton_col(p);
  if (!O.touches(R0, C0, 4)) return;
  const bool fast = O.vec4 && O.inside(R0, C0, 4);
  V dq[4] = {0, 0, 0, 0};
  u32 inb = 0, rq = 0, idx0 = 0, win = 0, e0 = 0;
  Quad<V> sn;
#pragma unroll
  for (int c = 0; c < 4; c++) sn.c[c] = 0;
  if (mode == 0) {
    idx0 = 1u + 4u * r;
    dac_get4<V>(mx, idx0, dq);
    if (idx0 < nm_len) { inb = tab_bits4(T, idx0); rq = tab_rank(T, idx0); }
    if (inb != 15u) {
      sn = *reinterpret_cast<const Quad<V>*>(&S.sup[oQ + 4u * p]);
      e0 = idx0 - rq;  // rank0(idx + 1) - 1 of the first quad that stops here (log.rs:265)
      win = e0 < eq_len ? eq_window(eq, e0) : 0u;  // malformed input guard: a bit past the bitmap reads as 0
    }
  }
#pragma unroll
  for (int h = 0; h < 2; h++) {
    V v[2][4];
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const int c = 2 * h + j;
      u32 m = mode;
      V py = pay;
      const u32 bl = below(inb, c);
      if (mode == 0 && !((inb >> c) & 1u)) {
        const bool e = e0 + ((u32)c - bl) < eq_len && eq_bit(win, e0, (u32)c - bl);
        m = e ? 2u : 1u;
        py = e ? dq[c] : dq[c] + sn.c[c];  // uniform: max_t + max_s of the quad (log.rs:266-268)
      }
      if (m == 1) {
#pragma unroll
        for (int i = 0; i < 4; i++) v[j][i] = py;
      } else {
        const Quad<V> q = reinterpret_cast<const Quad<V>*>(S.cells)[4u * p + (u32)c];
        if (m == 2) {
#pragma unroll
          for (int i = 0; i < 4; i++) v[j][i] = py + q.c[i];
        } else {
          V dd[4];
          dac_get4<V>(mx, 1u + 4u * (rq + bl), dd);  // leaves: max_t + max_s (log.rs:233,246)
#pragma unroll
          for (int i = 0; i < 4; i++) v[j][i] = dd[i] + q.c[i];
        }
      }
    }
    O.put_pair(fast, R0 + 2 * h, C0, v[0], v[1]);
  }
}

// Snapshot at `chunk + d.off`: every thread walks to its level L-2 node, writes the snapshot values of its ancestors,
// of its four quads and of its sixteen cells; with `emit` the cells also go to the window (the instant is the snapshot).
template <typename V, typename S_, typename OUT>
DCDF_DEVINL void snapshot4(const u8* chunk, const InstDir& d, int L, S_& S, bool emit, const OUT& O) {
  const u32 p = threadIdx.x;
  RankTab& T = S.tab[threadIdx.x >> 5];
  const u32 nm_len = d.nm_len;
  build_rank(bitmap_bits(chunk, nm_len, d.nm_base), nm_len, T);
  const Dac4 mx = dac4_of(chunk, &d.max);
  bool has = T.W[0] >> 31;
  V val = dac_get1<V>(mx, 0);
  u32 r = 0;
  if (S_::PRIVATE_TOP ? (p & 31u) == 0 : p == 0) { sup_at(S, 0, 0) = val; S.single[top_slot<S_>()] = has ? 0u : 1u; }
  if (L == 1) {
    if (p == 0) {
      V dd[4] = {0, 0, 0, 0};
      if (has) dac_get4<V>(mx, 1u, dd);
      Quad<V> q;
#pragma unroll
      for (int i = 0; i < 4; i++) q.c[i] = val - dd[i];
      reinterpret_cast<Quad<V>*>(S.cells)[0] = q;
      if (emit) O.put(0, 0, q.c);
    }
    return;
  }
  const int lvp = L - 2;
  if (p >= (1u << (2 * lvp))) return;
  for (int k = 1; k <= lvp; k++) {
    const u32 pk = p >> (2 * (lvp - k));
    if (has) {
      const u32 cidx = 1u + 4u * r + (pk & 3u);
      val -= dac_get1<V>(mx, cidx);  // snapshot.rs:179
      has = cidx < nm_len && tab_bit(T, cidx);
      if (has) r = tab_rank(T, cidx);
    }
    sup_at(S, k, pk) = val;
  }
  V dq[4] = {0, 0, 0, 0};
  u32 inb = 0, rq = 0;
  if (has) {
    const u32 idx0 = 1u + 4u * r;
    dac_get4<V>(mx, idx0, dq);
    if (idx0 < nm_len) { inb = tab_bits4(T, idx0); rq = tab_rank(T, idx0); }
  }
  Quad<V> qv;
#pragma unroll
  for (int c = 0; c < 4; c++) qv.c[c] = val - dq[c];
  *reinterpret_cast<Quad<V>*>(&S.sup[off3(L - 1) + 4u * p]) = qv;
#pragma unroll
  for (int c = 0; c < 4; c++) {
    V dd[4] = {0, 0, 0, 0};
    if ((inb >> c) & 1u) dac_get4<V>(mx, 1u + 4u * (rq + below(inb, c)), dd);
    Quad<V> q;
#pragma unroll
    for (int i = 0; i < 4; i++) q.c[i] = qv.c[c] - dd[i];
    reinterpret_cast<Quad<V>*>(S.cells)[4u * p + (u32)c] = q;
  }
  if (emit) block4<V, S_, OUT>(mx, chunk, 0u, T, nm_len, 2u, (V)0, 0u, p, off3(L - 1), S, O);  // "equal to the snapshot, offset 0"
}

// Log at `chunk + d.off` against the snapshot pyramid in S: walk to the level L-2 node, then the block's cells.
template <typename V, typename S_, typename OUT>
DCDF_DEVINL void log4(const u8* chunk, const InstDir& d, int L, S_& S, const OUT& O) {
  const u32 p = threadIdx.x;
  RankTab& T = S.tab[threadIdx.x >> 5];
  const u32 nm_len = d.nm_len;
  build_rank(bitmap_bits(chunk, nm_len, d.nm_base), nm_len, T);
  const u8* eq = bitmap_bits(chunk, d.eq_len, d.eq_base);
  const Dac4 mx = dac4_of(chunk, &d.max);
  u32 mode = 0, r = 0;
  V pay = dac_get1<V>(mx, 0);
  if (!(T.W[0] >> 31)) {
    // log.rs:180-186: a single-node log is uniform unless its equal bit says "snapshot + constant"
    const bool uniform = S.single[top_slot<S_>()] || (!OUT::search_quirk && !bit_at(eq, 0));
    mode = uniform ? 1u : 2u;
    if (uniform) pay += sup_at(S, 0, 0);
  }
  if (L == 1) {
    if (p == 0) {
      const Quad<V> q = reinterpret_cast<const Quad<V>*>(S.cells)[0];
      V v[4], dd[4] = {0, 0, 0, 0};
      if (mode == 0) dac_get4<V>(mx, 1u, dd);
#pragma unroll
      for (int i = 0; i < 4; i++) v[i] = mode == 1 ? pay : mode == 2 ? pay + q.c[i] : dd[i] + q.c[i];
      O.put(0, 0, v);
    }
    return;
  }
  const int lvp = L - 2;
  if (p >= (1u << (2 * lvp))) return;
  for (int k = 1; k <= lvp; k++) {
    if (mode == 0) {
      const u32 pk = p >> (2 * (lvp - k));
      const u32 cidx = 1u + 4u * r + (pk & 3u);
      pay = dac_get1<V>(mx, cidx);  // max_t is replaced, not accumulated (log.rs:233)
      const bool known = cidx < nm_len;
      const u32 rc = known ? tab_rank(T, cidx) : 0u;
      if (known && tab_bit(T, cidx)) {
        r = rc;
      } else {
        const bool e = cidx - rc < d.eq_len && bit_at(eq, cidx - rc);  // rank0(idx + 1) - 1 (log.rs:265)
        mode = e ? 2u : 1u;
        if (!e) pay += sup_at(S, k, pk);       // uniform: max_t + max_s of this node (log.rs:266-268)
      }
    }
  }
  block4<V, S_, OUT>(mx, eq, d.eq_len, T, nm_len, mode, pay, r, p, off3(L - 1), S, O);
}

template <typename V, typename S_, typename OUT>
DCDF_DEVINL void instant4(const u8* chunk, const InstDir& d, bool is_snap, bool emit, int L, S_& S, const OUT& O) {
  if (is_snap) snapshot4<V, S_, OUT>(chunk, d, L, S, emit, O);
  else log4<V, S_, OUT>(chunk, d, L, S, O);
}
template <typename V, typename S_, typename OUT>
__device__ __noinline__ void instant4_global(const u8* chunk, const InstDir* d, bool is_snap, bool emit, int L, S_* S, const OUT* O) {
  instant4<V, S_, OUT>(chunk, *d, is_snap, emit, L, *S, *O);
}

// Start the copy of a structure and of its directory entry into staging half b.
template <typename V, typename S_>
DCDF_DEVINL void prefetch_dir4(const InstDir* dg, S_& S, u32 slot) {
  const int tid = threadIdx.x;
  if (tid < W3_DIRW) cp_async4(reinterpret_cast<u32*>(&S.dir[slot]) + tid, reinterpret_cast<const u32*>(dg) + tid);
}
template <typename V, typename S_>
DCDF_DEVINL void prefetch4(const u8* chunk, u32 off, u32 size, S_& S, int b) {
  const int tid = threadIdx.x;
  const u8* src = chunk + off;
  const u32 mis = (u32)((uintptr_t)src & 15u);
  if (size + mis + 4u > (u32)S_::BUF + 32u) return;
  const u8* g = src - mis;
  const u32 n16 = (size + mis + 4u + 15u) / 16u;  // +4: a few bytes past the end may be read
  for (u32 i = tid; i < n16; i += DT_THREADS) cp_async16(S.stage[b] + 16u * i, g + 16u * i);
}
template <typename V>
DCDF_DEVINL bool staged4(const u8* chunk, const InstDir& d, u32& delta) {
  const u32 mis = (u32)((uintptr_t)(chunk + d.off) & 15u);
  delta = mis - d.off;
  return d.size + mis + 4u <= (u32)Tile4Smem<V>::BUF + 32u;
}

// CTAs per SM k_window_tiles4 is built for: TimeStatsOut's accumulators take most of an SM's shared memory, so it gets one
// CTA and the registers of the whole SM.
template <typename V, typename OUT>
constexpr int tiles4_min_blocks() { return std::is_same<OUT, TimeStatsOut<V>>::value ? 1 : sizeof(V) == 4 ? 4 : 2; }

// One CTA per (window, time slice, subchunk) job.  OUT receives the cells: QuadOut writes the window, StatsOut<V> reduces
// it per instant (dcdf_superchunk_window_stats), TimeStatsOut<V> per cell over the job's instants
// (dcdf_superchunk_time_stats); their hooks (begin / elided / instant_begin / instant_end / end) are all that differs.
template <typename V, typename OUT>
__global__ void __launch_bounds__(DT_THREADS, (tiles4_min_blocks<V, OUT>())) k_window_tiles4(const TileWindowParams P) {
  extern __shared__ __align__(16) unsigned char dt4_smem_raw[];
  Tile4Smem<V>& S = *reinterpret_cast<Tile4Smem<V>*>(dt4_smem_raw);
  const QuerySet& Q = P.Q;
  for (u64 ji = blockIdx.x; ji < P.n_jobs; ji += gridDim.x) {
    u64 lo_q = 0, hi_q = P.n_queries;
    while (hi_q - lo_q > 1) {
      const u64 mid = (lo_q + hi_q) >> 1;
      if (P.job_base[mid] <= ji) lo_q = mid; else hi_q = mid;
    }
    TileJob J;
    J.q = lo_q;
    J.c = P.cubes[J.q];
    const CubeDev& c = J.c;
    const u64 local = ji - P.job_base[J.q];
    const i64 cs = Q.chunks_sidelen;
    const i64 cr0 = c.top / cs, cc0 = c.left / cs;
    const i64 ncr = (c.bottom - 1) / cs - cr0 + 1, ncc = (c.right - 1) / cs - cc0 + 1;
    const u64 nsub = (u64)(ncr * ncc);
    const u32 s = (u32)(c.start / Q.chunk_size) + (u32)(local / nsub);
    J.sub = local % nsub;
    const i64 cr = cr0 + (i64)(J.sub / (u64)ncc), cc = cc0 + (i64)(J.sub % (u64)ncc);
    const SliceMeta sm = Q.slices[s];
    J.t_lo = max(c.start, sm.t0); J.t_hi = min(c.end, sm.t0 + (i64)sm.instants);
    const i64 t_lo = J.t_lo, t_hi = J.t_hi;
    const i64 chunk_top = cr * cs, chunk_left = cc * cs;
    J.chunk_top = chunk_top; J.chunk_left = chunk_left;
    // a dense window output: element offset of the window's first cell and of tile cell (0, 0) inside an instant
    const i64 W_rows = c.bottom - c.top, W_cols = c.right - c.left;
    const u64 obase = P.out_off[J.q];
    const i64 tile_org = (chunk_top - c.top) * W_cols + (chunk_left - c.left);
    J.top = (int)(max(chunk_top, c.top) - chunk_top); J.bottom = (int)(min(chunk_top + cs, c.bottom) - chunk_top);
    J.left = (int)(max(chunk_left, c.left) - chunk_left); J.right = (int)(min(chunk_left + cs, c.right) - chunk_left);
    const u32 slot = (u32)(cr * Q.subsidelen + cc);
    const int32_t u = Q.slot_unit[sm.slot_base + slot];
    const UnitMeta m = u >= 0 ? Q.units[u] : UnitMeta{};
    const bool stored = u >= 0 && m.stored;
    OUT O;
    O.begin(P, J, m.bits, dt4_smem_raw + sizeof(Tile4Smem<V>));
    if (!stored) {
      O.elided(P, J, sm, Q.slot_desc[sm.slot_base + slot]);
      continue;
    }
    const u8* chunk = Q.blob + m.blob_off;
    const InstDir* dir = Q.dir + m.dir_base;
    const int L = 31 - __clz(m.sidelen);
    if (t_hi <= t_lo) continue;
    const u32 ti0 = (u32)(t_lo - sm.t0), n_t = (u32)(t_hi - t_lo);
    __syncthreads();  // the previous job's readers are done with the staging buffers
    const u32 snap0 = dir[ti0].snap;
    if (snap0 != ti0) {
      // the window starts inside a block: expand the block's snapshot first
      prefetch_dir4<V, Tile4Smem<V>>(dir + snap0, S, 2);
      prefetch4<V, Tile4Smem<V>>(chunk, dir[snap0].off, dir[snap0].size, S, 1);
      cp_async_wait_all();
      __syncthreads();
      {  // once per job at most: through the out-of-line copy of the decoder (it accepts staged bytes as well), so that the
         // kernel holds ONE inlined copy of it
        u32 delta;
        const bool st = staged4<V>(chunk, S.dir[2], delta);
        const OUT O2 = O;
        instant4_global<V, Tile4Smem<V>, OUT>(st ? S.stage[1] + (int32_t)delta : chunk, &S.dir[2], true, false, L, &S, &O2);
      }
      __syncthreads();
    }
    prefetch_dir4<V, Tile4Smem<V>>(dir + ti0, S, 0);
    prefetch4<V, Tile4Smem<V>>(chunk, dir[ti0].off, dir[ti0].size, S, 0);
    if (n_t > 1) prefetch_dir4<V, Tile4Smem<V>>(dir + ti0 + 1, S, 1);
    const u64 t_stride = (u64)(W_rows * W_cols);
    u64 tbase = obase + (u64)((t_lo - c.start) * W_rows * W_cols + tile_org);
    u32 rs = 0;  // i % 3
    for (u32 i = 0; i < n_t; i++, tbase += t_stride) {
      const int b = (int)(i & 1u);
      const u32 ti = ti0 + i;
      const u32 slot1 = rs == 2 ? 0u : rs + 1u, slot2 = slot1 == 2 ? 0u : slot1 + 1u;
      cp_async_wait_all();
      __syncthreads();  // structure i and directory entry i+1 have landed; everyone is done with instant i-1
      if (i + 1 < n_t) {
        prefetch4<V, Tile4Smem<V>>(chunk, S.dir[slot1].off, S.dir[slot1].size, S, b ^ 1);
        if (i + 2 < n_t) prefetch_dir4<V, Tile4Smem<V>>(dir + ti + 2, S, slot2);
      }
      O.instant_begin(i, tbase);
      const InstDir& D = S.dir[rs];
      rs = slot1;
      const bool is_snap = D.snap == ti;
      u32 delta;
      if (staged4<V>(chunk, D, delta)) {
        instant4<V, Tile4Smem<V>, OUT>(S.stage[b] + (int32_t)delta, D, is_snap, true, L, S, O);
      } else {
        const OUT O2 = O;  // only the copy has its address taken
        instant4_global<V, Tile4Smem<V>, OUT>(chunk, &D, is_snap, true, L, &S, &O2);
      }
      O.instant_end(i);
    }
    O.end(n_t);
  }
}

// Window statistics, second pass: one thread per (window, instant) record folds the window's partials of that instant in
// subchunk order (row-major) -- a fixed order, so a window's records do not depend on the batch around it.  min / max are
// compared as values in the encoding's type (subchunks may have different fractional bits).
struct StatsCombineParams {
  const CubeDev* cubes;
  const u64* out_off;    // [n + 1] record offsets
  const u64* part_base;  // [n]
  const StatsPartial* part;
  u64 n_queries, rec0, rec1;  // records [rec0, rec1) = [out_off[0], out_off[n]); record g is written at index g - rec0
  i64 cs;
  int encoding;
  u64* count;
  void* vmin;
  void* vmax;
  double* sum;
  double* sum_sq;
};
template <typename T>
DCDF_DEVINL T stats_value(i64 code, int bits) {
  if constexpr (std::is_integral<T>::value) return (T)code;
  else return from_fixed_dev<T>(code, bits);
}
template <typename T>
DCDF_DEVINL void stats_fold(const StatsCombineParams& P, u64 r, const StatsPartial* p, u64 nsub, u64 T_all) {
  u64 n = 0;
  T mn = 0, mx = 0;
  double sum = 0.0, sq = 0.0;
  for (u64 k = 0; k < nsub; k++) {
    const StatsPartial x = p[k * T_all];
    if (x.count) {
      const T a = stats_value<T>(x.min, x.bits), b = stats_value<T>(x.max, x.bits);
      mn = n == 0 || a < mn ? a : mn;
      mx = n == 0 || b > mx ? b : mx;
    }
    n += x.count;
    sum += x.sum;
    sq += x.sum_sq;
  }
  if (n == 0) mn = mx = stats_value<T>(0, 0);  // NaN for floats (code 0), 0 for integers
  P.count[r] = n;
  static_cast<T*>(P.vmin)[r] = mn;
  static_cast<T*>(P.vmax)[r] = mx;
  P.sum[r] = sum;
  P.sum_sq[r] = sq;
}
__global__ void k_window_stats_combine(const StatsCombineParams P) {
  const u64 g = P.rec0 + (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.rec1) return;
  u64 lo = 0, hi = P.n_queries;  // the window of record g: the last one whose records start at or before g
  while (hi - lo > 1) {
    const u64 mid = (lo + hi) >> 1;
    if (P.out_off[mid] <= g) lo = mid; else hi = mid;
  }
  const CubeDev c = P.cubes[lo];
  const u64 T_all = (u64)(c.end - c.start), t = g - P.out_off[lo];
  const u64 nsub = c.bottom > c.top && c.right > c.left
                       ? (u64)((c.bottom - 1) / P.cs - c.top / P.cs + 1) * (u64)((c.right - 1) / P.cs - c.left / P.cs + 1) : 0u;
  const StatsPartial* p = P.part + P.part_base[lo] + t;
  const u64 r = g - P.rec0;
  if (P.encoding == 32) stats_fold<float>(P, r, p, nsub, T_all);
  else if (P.encoding == 64) stats_fold<double>(P, r, p, nsub, T_all);
  else if (P.encoding == 4) stats_fold<int32_t>(P, r, p, nsub, T_all);
  else stats_fold<i64>(P, r, p, nsub, T_all);
}

// Time statistics, second pass: one thread per (window, cell) record folds the record's partials of this scratch group in
// slice order into the outputs -- starting from empty records (init) or continuing the ones there.  A fixed order, so a
// record does not depend on the batch around it nor on how the slices were grouped.
struct TimeCombineParams {
  const CubeDev* cubes;   // the windows with their instants clipped to the group
  const u64* out_off;     // [n + 1] record offsets
  const u64* part_base;   // [n]
  const TimePartial* part;
  u64 n_queries, rec0, rec1;  // records [rec0, rec1) = [out_off[0], out_off[n]); record g is written at index g - rec0
  i64 chunk_size;
  int encoding, init;
  u64* count;
  u64* n_band;            // may be nullptr
  void* vmin;
  void* vmax;
  double* sum;
  double* sum_sq;
};
template <typename T>
DCDF_DEVINL T time_value(TimeVal v) {
  if constexpr (std::is_integral<T>::value) return (T)v.i;
  else return (T)v.f;
}
template <typename T>
DCDF_DEVINL void time_fold(const TimeCombineParams& P, u64 r, const TimePartial* p, u64 nsl, u64 area) {
  u64 n = 0, nb = 0;
  T mn = 0, mx = 0;
  double sum = 0.0, sq = 0.0;
  if (!P.init) {
    n = P.count[r];
    nb = P.n_band ? P.n_band[r] : 0u;
    mn = static_cast<const T*>(P.vmin)[r];
    mx = static_cast<const T*>(P.vmax)[r];
    sum = P.sum[r];
    sq = P.sum_sq[r];
  }
  for (u64 k = 0; k < nsl; k++) {
    const TimePartial x = p[k * area];
    if (x.count) {
      const T a = time_value<T>(x.min), b = time_value<T>(x.max);
      mn = n == 0 || a < mn ? a : mn;
      mx = n == 0 || b > mx ? b : mx;
    }
    n += x.count;
    nb += x.n_band;
    sum = __dadd_rn(sum, x.sum);
    sq = __dadd_rn(sq, x.sum_sq);
  }
  if (n == 0) mn = mx = stats_value<T>(0, 0);  // NaN for floats (code 0), 0 for integers
  P.count[r] = n;
  if (P.n_band) P.n_band[r] = nb;
  static_cast<T*>(P.vmin)[r] = mn;
  static_cast<T*>(P.vmax)[r] = mx;
  P.sum[r] = sum;
  P.sum_sq[r] = sq;
}
__global__ void k_time_stats_combine(const TimeCombineParams P) {
  const u64 g = P.rec0 + (u64)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.rec1) return;
  u64 lo = 0, hi = P.n_queries;  // the window of record g: the last one whose records start at or before g
  while (hi - lo > 1) {
    const u64 mid = (lo + hi) >> 1;
    if (P.out_off[mid] <= g) lo = mid; else hi = mid;
  }
  const CubeDev c = P.cubes[lo];
  const u64 area = (u64)((c.bottom - c.top) * (c.right - c.left));
  const u64 nsl = c.end > c.start ? (u64)((c.end - 1) / P.chunk_size - c.start / P.chunk_size + 1) : 0u;
  const TimePartial* p = P.part + P.part_base[lo] + (g - P.out_off[lo]);
  const u64 r = g - P.rec0;
  if (P.encoding == 32) time_fold<float>(P, r, p, nsl, area);
  else if (P.encoding == 64) time_fold<double>(P, r, p, nsl, area);
  else if (P.encoding == 4) time_fold<int32_t>(P, r, p, nsl, area);
  else time_fold<i64>(P, r, p, nsl, area);
}

// ---------------------------------------------------------------------------------------------------------------
// Cell series of a tile that many series of one batch fall into (Chunk::fill_cell chunk.rs:133-150, superchunk.rs:353-400):
// decode the tile's instants once with the window decoder's per-thread walk into an image of the tile in shared memory,
// then let the CTA hand every asked-for cell to its series.  A root-to-leaf walk per (series, instant) reads the same
// structure once per series; from some dozens of series per tile on, expanding it once is cheaper.  One CTA per (time
// slice, tile); blocks of the tile without an asked-for cell are not decoded.
struct SeriesJob {
  u32 slice, slot;
  u32 tile;          // index into `masks` (256 entries per tile)
  u32 ref_first, ref_count;
  u32 pad_;
  i64 t_min, t_max;  // union of the instants the tile's series cover
};
struct TileSeriesParams {
  QuerySet Q;
  const SeriesJob* jobs;
  u64 n_jobs;
  const uint16_t* masks;
  const CellRef* refs;
  void* out;
  int raw;
};
template <typename V>
struct Series4Smem {
  Tile4Smem<V> T;
  __align__(16) V img[4096];  // the instant being served, Morton order (img[16 * block + 4 * quad + cell])
};

template <typename V>
__global__ void __launch_bounds__(DT_THREADS, sizeof(V) == 4 ? 3 : 2) k_cell_tiles4(const TileSeriesParams P) {
  extern __shared__ __align__(16) unsigned char dt4_smem_raw[];
  Series4Smem<V>& SS = *reinterpret_cast<Series4Smem<V>*>(dt4_smem_raw);
  Tile4Smem<V>& S = SS.T;
  const QuerySet& Q = P.Q;
  const int tid = threadIdx.x;
  for (u64 ji = blockIdx.x; ji < P.n_jobs; ji += gridDim.x) {
    const SeriesJob J = P.jobs[ji];
    const SliceMeta sm = Q.slices[J.slice];
    const i64 t_lo = max(J.t_min, sm.t0), t_hi = min(J.t_max, sm.t0 + (i64)sm.instants);
    if (t_hi <= t_lo) continue;
    const int32_t u = Q.slot_unit[sm.slot_base + J.slot];
    const UnitMeta m = u >= 0 ? Q.units[u] : UnitMeta{};
    const bool stored = u >= 0 && m.stored;
    const CellRef* refs = P.refs + J.ref_first;
    // the thread's first reference stays in registers for the whole job (tiles with up to 256 series need no other)
    const bool have0 = (u32)tid < J.ref_count;
    const CellRef r0 = have0 ? refs[tid] : CellRef{0, 0, 0, 0, 0};
    CellOut co;
    if (!stored) {
      // Elided: one value per instant from the max table, parent's fractional bits (superchunk.rs:325-330)
      const SlotDesc sdsc = Q.slot_desc[sm.slot_base + J.slot];
      co.init(Q, P.out, P.raw, sdsc.bits);
      for (u32 k = (u32)tid; k < J.ref_count; k += DT_THREADS) {
        const CellRef r = k == (u32)tid ? r0 : refs[k];
        for (i64 t = max(t_lo, r.start); t < min(t_hi, r.end); t++)
          co.put(r.base + (u64)(t - r.start), (i64)Q.tbl_max[sdsc.tbl0 + (u64)(t - sm.t0) * sdsc.stride]);
      }
      continue;
    }
    co.init(Q, P.out, P.raw, m.bits);
    SeriesOut<V> O;
    O.img = SS.img + 16 * tid;
    O.mask = P.masks[(u64)J.tile * DT_THREADS + (u64)tid];
    const u8* chunk = Q.blob + m.blob_off;
    const InstDir* dir = Q.dir + m.dir_base;
    const int L = 31 - __clz(m.sidelen);
    const u32 ti0 = (u32)(t_lo - sm.t0), n_t = (u32)(t_hi - t_lo);
    __syncthreads();  // the previous job's readers are done with the staging buffers and the image
    const u32 snap0 = dir[ti0].snap;
    if (snap0 != ti0) {
      // the series start inside a block: expand the block's snapshot first
      prefetch_dir4<V, Tile4Smem<V>>(dir + snap0, S, 2);
      prefetch4<V, Tile4Smem<V>>(chunk, dir[snap0].off, dir[snap0].size, S, 1);
      cp_async_wait_all();
      __syncthreads();
      {  // once per job at most: through the out-of-line copy of the decoder (it accepts staged bytes as well)
        u32 delta;
        const bool st = staged4<V>(chunk, S.dir[2], delta);
        const SeriesOut<V> O2 = O;
        instant4_global<V, Tile4Smem<V>, SeriesOut<V>>(st ? S.stage[1] + (int32_t)delta : chunk, &S.dir[2], true, false, L, &S, &O2);
      }
      __syncthreads();
    }
    prefetch_dir4<V, Tile4Smem<V>>(dir + ti0, S, 0);
    prefetch4<V, Tile4Smem<V>>(chunk, dir[ti0].off, dir[ti0].size, S, 0);
    if (n_t > 1) prefetch_dir4<V, Tile4Smem<V>>(dir + ti0 + 1, S, 1);
    u32 rs = 0;  // i % 3
    for (u32 i = 0; i < n_t; i++) {
      const int b = (int)(i & 1u);
      const u32 ti = ti0 + i;
      const u32 slot1 = rs == 2 ? 0u : rs + 1u, slot2 = slot1 == 2 ? 0u : slot1 + 1u;
      cp_async_wait_all();
      __syncthreads();  // structure i and directory entry i+1 have landed; everyone is done with instant i-1 and its image
      if (i + 1 < n_t) {
        prefetch4<V, Tile4Smem<V>>(chunk, S.dir[slot1].off, S.dir[slot1].size, S, b ^ 1);
        if (i + 2 < n_t) prefetch_dir4<V, Tile4Smem<V>>(dir + ti + 2, S, slot2);
      }
      const InstDir& D = S.dir[rs];
      rs = slot1;
      const bool is_snap = D.snap == ti;
      u32 delta;
      if (staged4<V>(chunk, D, delta)) {
        instant4<V, Tile4Smem<V>, SeriesOut<V>>(S.stage[b] + (int32_t)delta, D, is_snap, true, L, S, O);
      } else {
        const SeriesOut<V> O2 = O;  // only the copy has its address taken
        instant4_global<V, Tile4Smem<V>, SeriesOut<V>>(chunk, &D, is_snap, true, L, &S, &O2);
      }
      __syncthreads();  // the image of instant i is complete
      const i64 t = t_lo + (i64)i;
      for (u32 k = (u32)tid; k < J.ref_count; k += DT_THREADS) {
        const CellRef r = k == (u32)tid ? r0 : refs[k];
        if (t >= r.start && t < r.end) co.put(r.base + (u64)(t - r.start), SS.img[r.cell]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Counting pass of a value-range search batch whose windows overlap (Chunk::iter_search / Superchunk::search counts,
// chunk.rs:213-228, superchunk.rs:464-585): one CTA per (time slice, tile) decodes every instant ONCE and counts the hits
// of every window that touches the tile there, instead of one decode per (window, tile).  counts[] has one slot per
// (window, subchunk, instant), exactly as the per-window kernel fills it; each slot belongs to one CTA (plain stores).
struct CountJob {
  u32 slice, slot;
  u32 ent_first, ent_count;  // ent_count <= CT_MAX
};
struct TileCountParams {
  QuerySet Q;
  const CountJob* jobs;
  u64 n_jobs;
  const CountEntry* entries;
  u64* counts;               // zeroed by the caller
};
template <typename V>
struct Count4Smem {
  Tile4Smem<V> T;
  CountShared<V> C;
};

template <typename V, bool ST>
__global__ void __launch_bounds__(DT_THREADS, sizeof(V) == 4 ? 4 : 2) k_count_tiles4(const TileCountParams P) {
  extern __shared__ __align__(16) unsigned char dt4_smem_raw[];
  Count4Smem<V>& SS = *reinterpret_cast<Count4Smem<V>*>(dt4_smem_raw);
  Tile4Smem<V>& S = SS.T;
  CountShared<V>& C = SS.C;
  const QuerySet& Q = P.Q;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (u64 ji = blockIdx.x; ji < P.n_jobs; ji += gridDim.x) {
    const CountJob J = P.jobs[ji];
    const SliceMeta sm = Q.slices[J.slice];
    const int32_t u = Q.slot_unit[sm.slot_base + J.slot];
    const UnitMeta m = u >= 0 ? Q.units[u] : UnitMeta{};
    const bool stored = u >= 0 && m.stored;
    __syncthreads();  // the previous job is done with the entries, the counters and the staging buffers
    if (tid < (int)J.ent_count) {
      CountEntry E = P.entries[J.ent_first + (u32)tid];
      bool nz = false;
      if (ST) {  // the band of this subchunk's own fractional bits (an Elided slot: its node's)
        const FixedBand fb = value_band(E.vlower, E.vupper, stored ? m.bits : Q.slot_desc[sm.slot_base + J.slot].bits, Q.encoding);
        E.lower = fb.lower; E.upper = fb.upper; nz = fb.nz;
      }
      C.ent[tid] = E;
      C.cnt[0][tid] = 0; C.cnt[1][tid] = 0;
      C.keep[tid] = nz ? 3u : 1u;
      // the band in the expansion's type: values outside V's range cannot occur
      const i64 vlo = sizeof(V) == 4 ? (i64)INT32_MIN : INT64_MIN, vhi = sizeof(V) == 4 ? (i64)INT32_MAX : INT64_MAX;
      const bool empty = E.lower > vhi || E.upper < vlo || E.lower > E.upper;
      C.lo[tid] = empty ? (V)1 : (V)max(E.lower, vlo);
      C.hi[tid] = empty ? (V)0 : (V)min(E.upper, vhi);
    }
    if (tid == 0) C.n = J.ent_count;
    __syncthreads();
    if (Q.tbl_min) {
      // Superchunk::search only looks into a subchunk when its min / max entries say that some instant of the window can
      // have cells in range (superchunk.rs:480-493), at every level of a nested superchunk: one warp per entry
      const SlotDesc sd = Q.slot_desc[sm.slot_base + J.slot];
      for (u32 e = (u32)warp; e < J.ent_count; e += DT_WARPS) {
        const CountEntry& E = C.ent[e];
        i64 lo = E.lower, hi = E.upper;
        if (lo > hi) { const i64 x = lo; lo = hi; hi = x; }
        const CountEntry& G = P.entries[J.ent_first + e];  // the strict search prunes with the value bounds
        bool ok = true;
        for (int lv = 0; lv <= sd.n_up; lv++)
          ok = ok && __any_sync(0xffffffffu, ST ? slot_may_hold_part(Q, sd, (i64)E.t0, (i64)E.t1, G.vlower, G.vupper, lane, 32, lv)
                                                : slot_has_cells_part(Q, sd, (i64)E.t0, (i64)E.t1, lo, hi, lane, 32, lv));
        if (lane == 0 && !ok) C.keep[e] = 0;
      }
      __syncthreads();
    }
    // slice-local instants any kept entry covers
    u32 t_lo = 0xffffffffu, t_hi = 0;
    unsigned long long mine = 0ull;
    const int R0 = 4 * (int)morton_row((u32)tid), C0 = 4 * (int)morton_col((u32)tid);
    for (u32 e = 0; e < J.ent_count; e++) {
      if (!C.keep[e]) continue;
      const CountEntry& E = C.ent[e];
      t_lo = min(t_lo, (u32)E.t0); t_hi = max(t_hi, (u32)E.t1);
      if (R0 + 4 > (int)E.top && R0 < (int)E.bottom && C0 + 4 > (int)E.left && C0 < (int)E.right) mine |= 1ull << e;
    }
    if (t_hi <= t_lo) continue;  // CTA-uniform
    if (!stored) {
      // Elided subchunk: one value per instant from the max table (superchunk.rs:541-559)
      const SlotDesc sdsc = Q.slot_desc[sm.slot_base + J.slot];
      for (u32 e = (u32)tid; e < J.ent_count; e += DT_THREADS) {
        if (!C.keep[e]) continue;
        const CountEntry E = C.ent[e];
        const u64 area = (u64)(E.bottom - E.top) * (u64)(E.right - E.left);
        for (u32 t = E.t0; t < E.t1; t++) {
          const i64 v = Q.tbl_max[sdsc.tbl0 + (u64)t * sdsc.stride];
          if (band_hit(v, E.lower, E.upper, ST && (C.keep[e] & 2u))) P.counts[E.cnt_base + (i64)t] = area;
        }
      }
      continue;
    }
    const u8* chunk = Q.blob + m.blob_off;
    const InstDir* dir = Q.dir + m.dir_base;
    const int L = 31 - __clz(m.sidelen);
    CountOut<V, ST> O;
    O.C = &C; O.mine = mine; O.R0 = R0; O.C0 = C0; O.t = t_lo; O.buf = 0; O.is_log = false; O.min_t = 0; O.e_root = 0;
    const u32 ti0 = t_lo, n_t = t_hi - t_lo;
    const u32 snap0 = dir[ti0].snap;
    // the block's snapshot is expanded first when the first instant is a Log; every Snapshot on the way leaves its root's
    // min / max for the single-node-Log rule
    auto snapshot_root = [&](const u8* base, const InstDir& D) {
      if (tid == 0) {
        const Dac4 mx = dac4_of(base, &D.max), mn = dac4_of(base, &D.min);
        const V vmax = dac_get1<V>(mx, 0);
        C.smax0 = vmax;
        C.smin0 = dac_get1<V>(mn, 0);  // the root's min entry is the absolute minimum (snapshot.rs:139-141); a single-node
                                       // Snapshot has no min Dac and the reference reads 0 from it (dac.rs:80-93)
      }
    };
    if (snap0 != ti0) {
      prefetch_dir4<V, Tile4Smem<V>>(dir + snap0, S, 2);
      prefetch4<V, Tile4Smem<V>>(chunk, dir[snap0].off, dir[snap0].size, S, 1);
      cp_async_wait_all();
      __syncthreads();
      {
        u32 delta;
        const bool st = staged4<V>(chunk, S.dir[2], delta);
        const u8* base = st ? S.stage[1] + (int32_t)delta : chunk;
        snapshot_root(base, S.dir[2]);
        const CountOut<V, ST> O2 = O;
        instant4_global<V, Tile4Smem<V>, CountOut<V, ST>>(base, &S.dir[2], true, false, L, &S, &O2);
      }
      __syncthreads();
    }
    prefetch_dir4<V, Tile4Smem<V>>(dir + ti0, S, 0);
    prefetch4<V, Tile4Smem<V>>(chunk, dir[ti0].off, dir[ti0].size, S, 0);
    if (n_t > 1) prefetch_dir4<V, Tile4Smem<V>>(dir + ti0 + 1, S, 1);
    u32 rs = 0;  // i % 3
    // entries that cover an instant: one bit per entry, built one instant ahead by the first two warps (read after the
    // barrier at the top of that instant)
    auto mark_active = [&](u32 t_next, u32 parity) {
      if (tid < CT_MAX) {
        const bool on = tid < (int)J.ent_count && C.keep[tid] && t_next >= (u32)C.ent[tid].t0 && t_next < (u32)C.ent[tid].t1;
        const u32 w = __ballot_sync(0xffffffffu, on);
        if (lane == 0) reinterpret_cast<u32*>(&C.act[parity])[warp] = w;
      }
    };
    mark_active(ti0, 0u);
    // counters of instant i - 1 go to counts[] while instant i is decoded (nobody adds to them any more)
    auto flush = [&](u32 t_done, u32 b) {
      if (tid < (int)J.ent_count) {
        const u32 c = C.cnt[b][tid];
        if (c) {
          const CountEntry& E = C.ent[tid];
          P.counts[E.cnt_base + (i64)t_done] = (u64)c;
          C.cnt[b][tid] = 0;
        }
      }
    };
    for (u32 i = 0; i < n_t; i++) {
      const int b = (int)(i & 1u);
      const u32 ti = ti0 + i;
      const u32 slot1 = rs == 2 ? 0u : rs + 1u, slot2 = slot1 == 2 ? 0u : slot1 + 1u;
      cp_async_wait_all();
      __syncthreads();  // structure i and directory entry i+1 have landed; everyone is done with instant i-1
      if (i + 1 < n_t) {
        prefetch4<V, Tile4Smem<V>>(chunk, S.dir[slot1].off, S.dir[slot1].size, S, b ^ 1);
        if (i + 2 < n_t) prefetch_dir4<V, Tile4Smem<V>>(dir + ti + 2, S, slot2);
      }
      if (i > 0) flush(ti - 1u, (u32)(b ^ 1));
      if (i + 1 < n_t) mark_active(ti + 1u, (u32)(b ^ 1));
      const InstDir& D = S.dir[rs];
      rs = slot1;
      const bool is_snap = D.snap == ti;
      u32 delta;
      const bool st = staged4<V>(chunk, D, delta);
      const u8* base = st ? S.stage[b] + (int32_t)delta : chunk;
      O.t = ti; O.buf = (u32)b;
      O.is_log = !is_snap;
      if (is_snap) {
        // written by thread 0 now, read by Logs after the next barrier; this instant itself does not use it
        snapshot_root(base, D);
      } else {
        O.e_root = dac_get1<V>(dac4_of(base, &D.max), 0);
        O.min_t = dac_get1<V>(dac4_of(base, &D.min), 0);
      }
      if (st) {
        instant4<V, Tile4Smem<V>, CountOut<V, ST>>(base, D, is_snap, true, L, S, O);
      } else {
        const CountOut<V, ST> O2 = O;  // only the copy has its address taken
        instant4_global<V, Tile4Smem<V>, CountOut<V, ST>>(chunk, &D, is_snap, true, L, &S, &O2);
      }
    }
    __syncthreads();
    flush(ti0 + n_t - 1u, (u32)((n_t - 1u) & 1u));
  }
}

}  // namespace dcdf