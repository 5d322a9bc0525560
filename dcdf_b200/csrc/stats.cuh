// stats.cuh -- the scan passes that precede encoding (one CTA per subchunk x time-slice unit):
//   suggest_fraction                      fixed.rs:96-159
//   MMBuffer3F32::compute_fractional_bits mmbuffer.rs:596-613
//   MMBuffer3::min_max / min_max_float    mmbuffer.rs:366-395, 434-499
// and the per-slice finalisation of Superchunk::build (superchunk.rs:127-198): parent/sub fractional
// bits, fixed-point (min,max) tables in instant-major order, elision flags, narrow/wide work lists.
#pragma once
#include <cmath>

#include "common.cuh"
#include "encode_tile.cuh"
#include "tree_types.hpp"

namespace dcdf {

constexpr int STAT_THREADS = 256;

struct UnitStats {
  double vmax;      // max over non-NaN values (floats) -- suggest_fraction uses max, not max-abs
  double vneg;      // most negative value (<= 0), 0 if none
  i64 imax, imin;   // integer encodings: exact extrema over the unit
  int has_value;    // any non-NaN value
  int frac_nonneg;  // max fractional bits over values >= 0
  int frac_neg;     // max fractional bits over values < 0
  int nonfinite;    // saw +-inf
  int sug_round;    // unit-level suggest_fraction: 1 = Round(bits), 0 = Precise(bits)
  int sug_bits;
  int sug_err;      // EF_* raised while computing the suggestion (whole part too large)
};

// per (unit, instant): raw extrema as 64-bit patterns (double for float inputs, i64 for integers)
struct InstStats {
  u64 mn, mx;
  u32 first;  // tile-local row-major index (r * cols + c) of the first non-NaN cell, 0xffffffff if none
  u32 last;   // 1 + index of the last NaN cell, 0 if none
  // all NaN  <=> first == 0xffffffff ; NaN quirk (mmbuffer.rs:485-487: a NaN after the first non-NaN makes
  // min NaN) <=> last > first
  DCDF_DEVINL u32 flags() const {
    const bool all_nan = first == 0xffffffffu;
    return (all_nan ? 1u : 0u) | ((!all_nan && last > first) ? 2u : 0u);
  }
};

template <typename T>
struct FloatBits;
template <>
struct FloatBits<int32_t> {
  static DCDF_DEVINL int fast(int32_t) { return 0; }
  static DCDF_DEVINL int fracbits(int32_t) { return 0; }
};
template <>
struct FloatBits<i64> {
  static DCDF_DEVINL int fast(i64) { return 0; }
  static DCDF_DEVINL int fracbits(i64) { return 0; }
};
template <>
struct FloatBits<float> {
  // branch-free: NaN / inf give 0 (E = 255), zero gives 0
  static DCDF_DEVINL int fast(float v) {
    const u32 b = __float_as_uint(v);
    const int E = (b >> 23) & 0xff;
    const u32 M = (b & 0x7fffffu) | (E ? 0x800000u : 0u);
    const int fb = 150 - (E ? E : 1) - (__ffs((int)M) - 1);
    return (M != 0 && fb > 0) ? fb : 0;
  }
  static DCDF_DEVINL int fracbits(float v) {
    u32 b = __float_as_uint(v);
    int E = (b >> 23) & 0xff;
    u32 M = b & 0x7fffffu;
    int e_odd;
    if (E == 0) {
      if (M == 0) return 0;
      e_odd = -149 + (__ffs((int)M) - 1);
    } else {
      e_odd = E - 150 + (__ffs((int)(M | 0x800000u)) - 1);
    }
    return e_odd < 0 ? -e_odd : 0;
  }
};
template <>
struct FloatBits<double> {
  static DCDF_DEVINL int fast(double v) {
    const u64 b = (u64)__double_as_longlong(v);
    const int E = (int)((b >> 52) & 0x7ff);
    const u64 M = (b & 0xfffffffffffffull) | (E ? (1ull << 52) : 0ull);
    const int fb = 1075 - (E ? E : 1) - (__ffsll((long long)M) - 1);
    return (M != 0 && fb > 0) ? fb : 0;
  }
  static DCDF_DEVINL int fracbits(double v) {
    u64 b = (u64)__double_as_longlong(v);
    int E = (int)((b >> 52) & 0x7ff);
    u64 M = b & 0xfffffffffffffull;
    int e_odd;
    if (E == 0) {
      if (M == 0) return 0;
      e_odd = -1074 + (__ffsll((long long)M) - 1);
    } else {
      e_odd = E - 1075 + (__ffsll((long long)(M | (1ull << 52))) - 1);
    }
    return e_odd < 0 ? -e_odd : 0;
  }
};

// Running maximum of FloatBits::fast over the values fed to add().  For f32 the per-value work avoids the bit scan:
// the lowest set bit of |v| as a float is |v| - (|v| with that mantissa bit cleared) -- exact, a power of two
// 2^(E' - 150 + tz(M)) -- and the most fractional bits belong to the smallest such power.
// Bit patterns of positive floats order like the values, so one unsigned min over (bits - 1) keeps it; zeros wrap to
// 0xffffffff and inf / NaN stay above every finite value, so none of them needs a branch.
template <typename T>
struct FracAcc {
  int fb = 0;
  DCDF_DEVINL void add(T v) { fb = max(fb, FloatBits<T>::fast(v)); }
  DCDF_DEVINL int result() const { return fb; }
};
template <>
struct FracAcc<float> {
  u32 acc = 0xffffffffu;
  DCDF_DEVINL void add(float v) {
    const u32 b = __float_as_uint(v) & 0x7fffffffu;
    const u32 c = (b & 0x7fffffu) ? (b & (b - 1u)) : 0u;  // mantissa field != 0: b - 1 only borrows inside it
    const float l = __uint_as_float(b) - __uint_as_float(c);
    acc = min(acc, __float_as_uint(l) - 1u);
  }
  DCDF_DEVINL int result() const {
    const u32 lb = acc + 1u;                   // bits of the smallest lowest-set-bit value: 2^e
    if (lb == 0u || lb >= 0x7f800000u) return 0;  // nothing finite and non-zero
    const int E = (int)(lb >> 23);
    const int e = E ? E - 127 : (31 - __clz((int)(lb & 0x7fffffu))) - 149;
    return e < 0 ? -e : 0;
  }
};

// whole_bits = 1 + (floor(log2(max)) as usize)  (fixed.rs:126; `as` saturates: NaN / negatives -> 0).
// The reference takes log2 with the host's libm, whose result ROUNDS UP to the integer k for the last few doubles below
// 2^k (8 - 2^-50 -> log2 == 3.0), so floor(log2(x)) is not ilogb(x) there.  c_log2_roundup[k] has bit j-1 set when
// floor(std::log2(2^k - j * 2^(k-53))) == k on THIS host (filled by dcdf_ctx_create with std::log2, the libm call
// behind Rust's f64::log2); only f64 inputs can come that close to a power of two.
__constant__ u64 c_log2_roundup[64];
DCDF_DEVINL int whole_bits_of(double vmax) {
  if (!(vmax > 0.0)) return 1;
  int e = ilogb(vmax);
  if (e >= 0 && e < 63) {
    const double j = (ldexp(1.0, e + 1) - vmax) * ldexp(1.0, 52 - e);  // exact: vmax is the j-th double below 2^(e+1)
    if (j <= 64.0 && ((c_log2_roundup[e + 1] >> ((int)j - 1)) & 1ull)) e += 1;
  }
  return 1 + (e > 0 ? e : 0);
}
inline void upload_log2_roundup_table() {
  u64 tab[64];
  for (int k = 0; k < 64; k++) {
    tab[k] = 0;
    for (int j = 1; j <= 64 && k >= 1; j++) {
      const double x = std::ldexp(1.0, k) - (double)j * std::ldexp(1.0, k - 53);
      if (std::floor(std::log2(x)) == (double)k) tab[k] |= 1ull << (j - 1);
    }
  }
  cudaMemcpyToSymbol(c_log2_roundup, tab, sizeof tab);
}

// Evaluate suggest_fraction from a (max, frac_nonneg, frac_neg, most-negative) summary.
// Returns false when negatives may hit the saturating cast (fixed.rs:150) and an exact pass is needed.
DCDF_DEVINL bool suggest_from_summary(bool has_value, double vmax, double vneg, int frac_nonneg, int frac_neg, int& round_,
                                      int& bits, int& err) {
  err = 0;
  if (!has_value) { round_ = 0; bits = 0; return true; }  // all NaN -> Precise(0)  (fixed.rs:121-124)
  // max == +inf: log2 is inf, the `as usize` cast saturates and 1 + usize::MAX wraps to 0 in a release build, so
  // max_fraction_bits = 62; inf.fract() is NaN != 0.0 -> Round(62)  (fixed.rs:126-148)
  if (isinf(vmax)) { round_ = 1; bits = 62; return true; }
  int whole = whole_bits_of(vmax);
  if (whole > 62) { err = EF_OVERFLOW; round_ = 0; bits = 0; return true; }
  int maxfb = 62 - whole;
  if (vneg < 0.0 && -vneg >= ldexp(1.0, 63 - maxfb)) return false;  // some negative saturates `as i64`
  int f = frac_nonneg > frac_neg ? frac_nonneg : frac_neg;
  if (f > maxfb) { round_ = 1; bits = maxfb; }  // fixed.rs:146-148
  else { round_ = 0; bits = f; }
  return true;
}

struct StatParams {
  const void* data;
  i64 stride_t, stride_r, stride_c;
  const EncUnit* units;
  u32 n_units;
  u32 t_max;  // row pitch of the per-instant tables
  UnitStats* ustats;
  InstStats* istats;  // [n_units][t_max]
};

// warp-wide min / max: one redux for 32-bit types (floats through an order-preserving key), shuffles otherwise
DCDF_DEVINL u32 fkey(float f) { const u32 b = __float_as_uint(f); return b ^ ((u32)((int32_t)b >> 31) | 0x80000000u); }
DCDF_DEVINL float funkey(u32 k) { return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu)); }
DCDF_DEVINL float warp_min(float v) { return funkey(__reduce_min_sync(0xffffffffu, fkey(v))); }
DCDF_DEVINL float warp_max(float v) { return funkey(__reduce_max_sync(0xffffffffu, fkey(v))); }
DCDF_DEVINL int32_t warp_min(int32_t v) { return __reduce_min_sync(0xffffffffu, v); }
DCDF_DEVINL int32_t warp_max(int32_t v) { return __reduce_max_sync(0xffffffffu, v); }
DCDF_DEVINL u32 warp_min(u32 v) { return __reduce_min_sync(0xffffffffu, v); }
DCDF_DEVINL u32 warp_max(u32 v) { return __reduce_max_sync(0xffffffffu, v); }
DCDF_DEVINL double warp_min(double v) {
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
DCDF_DEVINL double warp_max(double v) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
DCDF_DEVINL i64 warp_min(i64 v) {
  for (int o = 16; o > 0; o >>= 1) { const i64 x = __shfl_xor_sync(0xffffffffu, v, o); v = x < v ? x : v; }
  return v;
}
DCDF_DEVINL i64 warp_max(i64 v) {
  for (int o = 16; o > 0; o >>= 1) { const i64 x = __shfl_xor_sync(0xffffffffu, v, o); v = x > v ? x : v; }
  return v;
}
template <typename T> struct Lim;
template <> struct Lim<float> { static DCDF_DEVINL float hi() { return INFINITY; } static DCDF_DEVINL float lo() { return -INFINITY; } };
template <> struct Lim<double> { static DCDF_DEVINL double hi() { return INFINITY; } static DCDF_DEVINL double lo() { return -INFINITY; } };
template <> struct Lim<int32_t> { static DCDF_DEVINL int32_t hi() { return INT32_MAX; } static DCDF_DEVINL int32_t lo() { return INT32_MIN; } };
template <> struct Lim<i64> { static DCDF_DEVINL i64 hi() { return INT64_MAX; } static DCDF_DEVINL i64 lo() { return INT64_MIN; } };
template <typename T> DCDF_DEVINL u64 raw64(T v);
template <> DCDF_DEVINL u64 raw64<float>(float v) { return (u64)__double_as_longlong((double)v); }
template <> DCDF_DEVINL u64 raw64<double>(double v) { return (u64)__double_as_longlong(v); }
template <> DCDF_DEVINL u64 raw64<int32_t>(int32_t v) { return (u64)(i64)v; }
template <> DCDF_DEVINL u64 raw64<i64>(i64 v) { return (u64)v; }

constexpr int STAT_BATCH = 32;  // instants whose per-warp partials are kept in smem before one finalisation

// min / max that ignore NaN operands (IEEE minNum / maxNum); integer overloads only keep the templates well formed
DCDF_DEVINL float stat_fmin(float a, float b) { return fminf(a, b); }
DCDF_DEVINL float stat_fmax(float a, float b) { return fmaxf(a, b); }
DCDF_DEVINL double stat_fmin(double a, double b) { return fmin(a, b); }
DCDF_DEVINL double stat_fmax(double a, double b) { return fmax(a, b); }
DCDF_DEVINL int32_t stat_fmin(int32_t a, int32_t b) { return a < b ? a : b; }
DCDF_DEVINL int32_t stat_fmax(int32_t a, int32_t b) { return a > b ? a : b; }
DCDF_DEVINL i64 stat_fmin(i64 a, i64 b) { return a < b ? a : b; }
DCDF_DEVINL i64 stat_fmax(i64 a, i64 b) { return a > b ? a : b; }

template <typename InT, bool IS_FLOAT>
__global__ void __launch_bounds__(STAT_THREADS, 3) k_unit_stats(const StatParams P) {
  const u32 u = blockIdx.x;
  if (u >= P.n_units) return;
  const EncUnit unit = P.units[u];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const InT* base = static_cast<const InT*>(P.data) + unit.base;
  const int cols = unit.cols;
  const int cells = unit.rows * cols;
  __shared__ InT p_mn[STAT_BATCH][8], p_mx[STAT_BATCH][8];
  __shared__ u32 p_first[STAT_BATCH][8], p_last[STAT_BATCH][8];
  __shared__ double s_d[8][2];
  __shared__ i64 s_l[8][2];
  __shared__ int s_i[8][4];
  __shared__ int s_redo, s_maxfb;

  // row-major walk without divisions: thread t visits cells t, t + 256, ...
  const int r_init = tid / cols, c_init = tid - r_init * cols;
  const int step_r = STAT_THREADS / cols, step_c = STAT_THREADS - step_r * cols;
  const i64 q_step = (i64)step_r * P.stride_r + (i64)step_c * P.stride_c;  // pointer step for 256 cells ahead
  const i64 q_wrap = P.stride_r - (i64)cols * P.stride_c;                  // extra step when the column wraps
  const bool vec4 = sizeof(InT) == 4 && cols == 64 && P.stride_c == 1 && ((P.stride_r * 4) & 15) == 0 && ((P.stride_t * 4) & 15) == 0 &&
                    (((uintptr_t)base) & 15) == 0;

  InT umax = Lim<InT>::lo(), umin = Lim<InT>::hi();  // unit extrema over non-NaN values
  InT uneg = (InT)0;                                 // most negative value
  int has = 0, fnn = 0, fng = 0, nonfinite = 0;
  FracAcc<InT> facc;  // fractional bits: only max(frac_nonneg, frac_neg) is ever used, so one accumulator serves both

  // vec4 path: the next instant's four 128-bit loads are in flight while the current one is reduced
  uint4 nxt[4];
  auto fetch4 = [&](int inst) {
    const InT* p = base + (i64)inst * P.stride_t;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int row = (tid >> 4) + 16 * j;
      nxt[j] = row < unit.rows ? __ldg(reinterpret_cast<const uint4*>(p + (i64)row * P.stride_r + 4 * (tid & 15))) : make_uint4(0, 0, 0, 0);
    }
  };
  if (vec4) fetch4(0);

  for (int i0 = 0; i0 < unit.instants; i0 += STAT_BATCH) {
    const int nb = min(STAT_BATCH, unit.instants - i0);
    for (int bi = 0; bi < nb; bi++) {
      const InT* p = base + (i64)(i0 + bi) * P.stride_t;
      InT mn = Lim<InT>::hi(), mx = Lim<InT>::lo();
      u32 first = 0xffffffffu, last = 0;  // row-major position (+1 for last) of first non-NaN / last NaN
      if (vec4) {
        // full 64-column tile with 16-byte aligned rows: four 128-bit loads per thread and instant
        uint4 qv[4];
#pragma unroll
        for (int j = 0; j < 4; j++) qv[j] = nxt[j];
        if (i0 + bi + 1 < unit.instants) fetch4(i0 + bi + 1);
        bool anynan = false;
        u32 nanacc = 0;  // f32: largest |bits| seen; a NaN is anything above the infinity pattern
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const int row = (tid >> 4) + 16 * j;
          if (row >= unit.rows) break;
          const u32 wv[4] = {qv[j].x, qv[j].y, qv[j].z, qv[j].w};
#pragma unroll
          for (int e = 0; e < 4; e++) {
            const InT v = *reinterpret_cast<const InT*>(&wv[e]);
            if (IS_FLOAT) {
              // fmin / fmax skip NaN operands, which is what the reference's comparisons do (mmbuffer.rs:465-499);
              // the NaN positions are only worked out (below) for warps that saw one; the most negative value of the
              // unit follows from the per-instant minima
              if (sizeof(InT) == 4) nanacc = max(nanacc, wv[e] & 0x7fffffffu);
              else anynan = anynan || v != v;
              mn = stat_fmin(mn, v);
              mx = stat_fmax(mx, v);
              facc.add(v);
            } else {
              mn = v < mn ? v : mn;
              mx = v > mx ? v : mx;
            }
          }
        }
        if (IS_FLOAT) {
          if (sizeof(InT) == 4) anynan = nanacc > 0x7f800000u;
          if (__any_sync(0xffffffffu, anynan)) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
              const int row = (tid >> 4) + 16 * j;
              if (row >= unit.rows) break;
              const u32 wv[4] = {qv[j].x, qv[j].y, qv[j].z, qv[j].w};
#pragma unroll
              for (int e = 0; e < 4; e++) {
                const int idx = row * 64 + 4 * (tid & 15) + e;
                const InT v = *reinterpret_cast<const InT*>(&wv[e]);
                const bool isn = v != v;
                last = isn ? (u32)idx + 1u : last;
                first = min(first, isn ? 0xffffffffu : (u32)idx);
              }
            }
          } else if ((tid >> 4) < unit.rows) {
            first = (u32)((tid >> 4) * 64 + 4 * (tid & 15));  // no NaN in this warp: the thread's first cell
          }
        }
      } else {
      // all loads of the instant are issued before any value is consumed (16 per thread for a full tile);
        // the pointer walks the tile row-major without divisions
        const InT* q = p + (i64)r_init * P.stride_r + (i64)c_init * P.stride_c;
        int c = c_init;
        for (int idx0 = tid; idx0 < cells; idx0 += 16 * STAT_THREADS) {
          InT vals[16];
#pragma unroll
          for (int j = 0; j < 16; j++) {
            const int idx = idx0 + j * STAT_THREADS;
            vals[j] = idx < cells ? __ldg(q) : (InT)0;
            c += step_c;
            q += q_step;
            if (c >= cols) { c -= cols; q += q_wrap; }
          }
#pragma unroll
          for (int j = 0; j < 16; j++) {
            const int idx = idx0 + j * STAT_THREADS;
            if (idx >= cells) break;
            const InT v = vals[j];
            if (IS_FLOAT) {
              const bool isn = v != v;
              last = isn ? (u32)idx + 1u : last;           // idx ascends within a thread
              first = min(first, isn ? 0xffffffffu : (u32)idx);
              mn = (isn || v > mn) ? mn : v;
              mx = (isn || v < mx) ? mx : v;
              facc.add(v);
            } else {
              mn = v < mn ? v : mn;
              mx = v > mx ? v : mx;
            }
          }
        }
      }
      mn = warp_min(mn); mx = warp_max(mx);
      if (IS_FLOAT) { first = warp_min(first); last = warp_max(last); }
      if (lane == 0) { p_mn[bi][warp] = mn; p_mx[bi][warp] = mx; p_first[bi][warp] = first; p_last[bi][warp] = last; }
    }
    __syncthreads();
    if (tid < nb) {
      InT mn = p_mn[tid][0], mx = p_mx[tid][0];
      u32 first = p_first[tid][0], last = p_last[tid][0];
      for (int w = 1; w < 8; w++) {
        mn = p_mn[tid][w] < mn ? p_mn[tid][w] : mn;
        mx = p_mx[tid][w] > mx ? p_mx[tid][w] : mx;
        first = min(first, p_first[tid][w]); last = max(last, p_last[tid][w]);
      }
      InstStats st;
      st.mn = raw64<InT>(mn); st.mx = raw64<InT>(mx);
      if (IS_FLOAT) {
        st.first = first; st.last = last;
        if (first != 0xffffffffu) {
          has = 1;
          umax = mx > umax ? mx : umax;
          uneg = mn < uneg ? mn : uneg;  // most negative value of the unit (mn skips NaN)
          if (mx - mx != (InT)0 || mn - mn != (InT)0) nonfinite = 1;  // +-inf among the extrema
        }
      } else {
        st.first = 0; st.last = 0;
        has = 1;
        umax = mx > umax ? mx : umax;
        umin = mn < umin ? mn : umin;
      }
      P.istats[(size_t)u * P.t_max + i0 + tid] = st;
    }
    __syncthreads();
  }

  // unit-level reductions of the thread-local accumulators
  umax = warp_max(umax); umin = warp_min(umin); uneg = warp_min(uneg);
  fnn = facc.result();
  for (int o = 16; o > 0; o >>= 1) {
    fnn = max(fnn, __shfl_xor_sync(0xffffffffu, fnn, o));
    fng = max(fng, __shfl_xor_sync(0xffffffffu, fng, o));
    nonfinite |= __shfl_xor_sync(0xffffffffu, nonfinite, o);
    has |= __shfl_xor_sync(0xffffffffu, has, o);
  }
  if (lane == 0) {
    s_i[warp][0] = fnn; s_i[warp][1] = fng; s_i[warp][2] = nonfinite; s_i[warp][3] = has;
    if (IS_FLOAT) { s_d[warp][0] = (double)umax; s_d[warp][1] = (double)uneg; }
    else { s_l[warp][0] = (i64)umax; s_l[warp][1] = (i64)umin; }
  }
  __syncthreads();
  if (tid == 0) {
    double vmax = -INFINITY, vneg = 0.0;
    i64 imax = INT64_MIN, imin = INT64_MAX;
    fnn = 0; fng = 0; nonfinite = 0; has = 0;
    for (int w = 0; w < 8; w++) {
      fnn = max(fnn, s_i[w][0]); fng = max(fng, s_i[w][1]); nonfinite |= s_i[w][2]; has |= s_i[w][3];
      if (IS_FLOAT) { vmax = fmax(vmax, s_d[w][0]); vneg = fmin(vneg, s_d[w][1]); }
      else { imax = s_l[w][0] > imax ? s_l[w][0] : imax; imin = s_l[w][1] < imin ? s_l[w][1] : imin; }
    }
    UnitStats us;
    us.vmax = vmax; us.vneg = vneg; us.imax = imax; us.imin = imin;
    us.has_value = has; us.frac_nonneg = fnn; us.frac_neg = fng; us.nonfinite = nonfinite;
    us.sug_round = 0; us.sug_bits = 0; us.sug_err = 0;
    int redo = 0;
    if (IS_FLOAT) {
      if (!suggest_from_summary(has, vmax, vneg, fnn, fng, us.sug_round, us.sug_bits, us.sug_err)) redo = 1;
    }
    P.ustats[u] = us;
    s_redo = redo;
    s_maxfb = 62 - whole_bits_of(vmax);
  }
  __syncthreads();
  if (IS_FLOAT && s_redo) {
    // Exact second pass (rare): some negative value saturates the `as i64` cast of fixed.rs:150, so its
    // contribution is maxfb - 63 -> 0 bits instead of its own fractional bits.
    const int maxfb = s_maxfb;
    const double sat = ldexp(1.0, 63 - maxfb);
    int f = 0, rnd = 0;
    for (int inst = 0; inst < unit.instants; inst++) {
      const InT* p = base + (i64)inst * P.stride_t;
      for (int idx = tid; idx < cells; idx += STAT_THREADS) {
        const int r = idx / cols, c = idx - r * cols;
        const InT v = __ldg(p + (i64)r * P.stride_r + (i64)c * P.stride_c);
        const double d = (double)v;
        if (d != d) continue;
        const int fb = FloatBits<InT>::fracbits(v);
        if (fb > maxfb) rnd = 1;
        if (!(d < 0.0 && -d >= sat)) f = fb > f ? fb : f;
      }
    }
    for (int o = 16; o > 0; o >>= 1) {
      f = max(f, __shfl_xor_sync(0xffffffffu, f, o));
      rnd |= __shfl_xor_sync(0xffffffffu, rnd, o);
    }
    if (lane == 0) { s_i[warp][0] = f; s_i[warp][1] = rnd; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < 8; w++) { f = max(f, s_i[w][0]); rnd |= s_i[w][1]; }
      P.ustats[u].sug_round = rnd;
      P.ustats[u].sug_bits = rnd ? maxfb : f;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// Exact region-level suggest_fraction pass with a known maxfb, launched only when needed (device flag).
struct ExactParams {
  const void* data;
  i64 stride_t, stride_r, stride_c;
  i64 rows, cols;
  const i64* slice_t0;       // [n_slices] first instant
  const int* slice_instants; // [n_slices]
  const int* slice_need;     // [n_slices] 1 = run
  const int* slice_maxfb;    // [n_slices]
  int* slice_f;              // [n_slices] out: max bits (atomicMax)
  int* slice_round;          // [n_slices] out: any fractional overflow (atomicOr)
};
template <typename InT>
__global__ void __launch_bounds__(256) k_fraction_exact(const ExactParams P, u32 n_slices) {
  const u32 s = blockIdx.y;
  if (s >= n_slices || !P.slice_need[s]) return;
  const int maxfb = P.slice_maxfb[s];
  const double sat = ldexp(1.0, 63 - maxfb);
  const i64 n = (i64)P.slice_instants[s] * P.rows * P.cols;
  const InT* base = static_cast<const InT*>(P.data) + P.slice_t0[s] * P.stride_t;
  int f = 0, rnd = 0;
  for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
    const i64 t = i / (P.rows * P.cols), rem = i - t * P.rows * P.cols;
    const i64 r = rem / P.cols, c = rem - r * P.cols;
    const InT v = __ldg(base + t * P.stride_t + r * P.stride_r + c * P.stride_c);
    const double d = (double)v;
    if (d != d) continue;
    const int fb = FloatBits<InT>::fracbits(v);
    if (fb > maxfb) rnd = 1;
    if (!(d < 0.0 && -d >= sat)) f = fb > f ? fb : f;
  }
  for (int o = 16; o > 0; o >>= 1) {
    f = max(f, __shfl_xor_sync(0xffffffffu, f, o));
    rnd |= __shfl_xor_sync(0xffffffffu, rnd, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&P.slice_f[s], f);
    if (rnd) atomicOr(&P.slice_round[s], 1);
  }
}

// ---------------------------------------------------------------------------------------------------
// Per-slice finalisation (one CTA per slice) for a two-level superchunk: subsidelen^2 slots, in-bounds
// slots have a unit.  Phase 1 aggregates the slice-level suggestion; phase 2 assigns per-unit bits,
// fills the (instant-major, slot-minor) fixed-point min/max tables, elision flags and work lists.
struct SliceDesc {
  i64 t0;
  int instants;
  u32 unit_base;   // first unit of the slice
  u32 n_units;
  u64 table_base;  // offset of this slice's tables in tbl_min / tbl_max (instants * n_slots entries)
};
struct SliceState {
  int bits;        // parent fractional bits (after compute_fractional_bits, if requested)
  int need_exact;  // phase 1 -> exact pass
  int maxfb;
  int f_exact, round_exact;
  int sug_round, sug_bits;  // raw slice-level suggest_fraction result (valid when !need_exact)
  u32 err;         // EF_*
  u32 n_elided, n_stored;
};
struct FinalizeParams {
  const SliceDesc* slices;
  SliceState* state;
  const EncUnit* units_in;
  EncUnit* units;          // bits / flags written here
  const UnitStats* ustats;
  const InstStats* istats;
  u32 t_max;
  u32 n_slots;             // subsidelen^2
  int encoding;            // DCDF_ENC_*
  int req_bits, round, compute_bits;
  int plain;               // 1 = plain Chunk::build units: caller's bits, no tables, no elision
  i64* tbl_min;
  i64* tbl_max;
  u32* order;              // four work lists of n_units_total entries each: index = wide * 2 + clipped
  u32 order_pitch;
  u32* order_counts;       // [4]
  u8* stored;              // [n_units_total] 1 = Chunk is built and stored (not elided)
  u32* err;
};

__global__ void k_finalize_phase1(const FinalizeParams P, u32 n_slices) {
  const u32 s = blockIdx.x;
  if (s >= n_slices) return;
  const SliceDesc sd = P.slices[s];
  __shared__ double s_vmax[8], s_vneg[8];
  __shared__ int s_f[8][4];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double vmax = -INFINITY, vneg = 0.0;
  int has = 0, fnn = 0, fng = 0;
  for (u32 i = tid; i < sd.n_units; i += blockDim.x) {
    const UnitStats us = P.ustats[sd.unit_base + i];
    if (us.has_value) { has = 1; vmax = fmax(vmax, us.vmax); }
    vneg = fmin(vneg, us.vneg);
    fnn = max(fnn, us.frac_nonneg);
    fng = max(fng, us.frac_neg);
  }
  for (int o = 16; o > 0; o >>= 1) {
    vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    vneg = fmin(vneg, __shfl_xor_sync(0xffffffffu, vneg, o));
    has |= __shfl_xor_sync(0xffffffffu, has, o);
    fnn = max(fnn, __shfl_xor_sync(0xffffffffu, fnn, o));
    fng = max(fng, __shfl_xor_sync(0xffffffffu, fng, o));
  }
  if (lane == 0) { s_vmax[warp] = vmax; s_vneg[warp] = vneg; s_f[warp][0] = has; s_f[warp][1] = fnn; s_f[warp][2] = fng; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) {
      vmax = fmax(vmax, s_vmax[w]); vneg = fmin(vneg, s_vneg[w]);
      has |= s_f[w][0]; fnn = max(fnn, s_f[w][1]); fng = max(fng, s_f[w][2]);
    }
    SliceState st;
    st.bits = P.req_bits; st.need_exact = 0; st.maxfb = 0; st.f_exact = 0; st.round_exact = 0; st.err = 0;
    st.n_elided = 0; st.n_stored = 0; st.sug_round = 0; st.sug_bits = 0;
    const bool is_float = P.encoding == 32 || P.encoding == 64;
    if (is_float && P.compute_bits) {
      int rnd, bits, e;
      if (suggest_from_summary(has, vmax, vneg, fnn, fng, rnd, bits, e)) {
        st.err |= (u32)e;
        st.sug_round = rnd; st.sug_bits = bits;
        if (P.round) st.bits = min(bits, P.req_bits);       // mmbuffer.rs:602-603
        else { if (rnd) st.err |= EF_PRECISION; st.bits = bits; }  // mmbuffer.rs:605-609
      } else {
        st.need_exact = 1;
        st.maxfb = 62 - whole_bits_of(vmax);
      }
    }
    if (!is_float) st.bits = 0;
    P.state[s] = st;
  }
}

template <typename F>
DCDF_DEVINL i64 fixed_of_raw(u64 raw, int bits, bool round, u32& err) {
  return to_fixed_dev<F>((F)__longlong_as_double((long long)raw), bits, round, err);
}

__global__ void k_finalize_phase2(const FinalizeParams P, u32 n_slices) {
  const u32 s = blockIdx.x;
  if (s >= n_slices) return;
  const SliceDesc sd = P.slices[s];
  const int tid = threadIdx.x;
  __shared__ int s_bits;
  __shared__ u32 s_err;
  const bool is_float = P.encoding == 32 || P.encoding == 64;
  if (tid == 0) {
    SliceState st = P.state[s];
    if (st.need_exact) {
      const int rnd = st.round_exact, bits = rnd ? st.maxfb : st.f_exact;
      if (P.round) st.bits = min(bits, P.req_bits);
      else { if (rnd) st.err |= EF_PRECISION; st.bits = bits; }
      P.state[s].bits = st.bits;
    }
    s_bits = st.bits;
    s_err = st.err;
  }
  __syncthreads();
  const int pbits = s_bits;
  const bool round = P.round != 0;
  u32 err = 0;
  // tables default to (0,0): out-of-bounds slots are Elided with (0,0) per instant (superchunk.rs:134-139)
  i64* tmin = P.plain ? nullptr : P.tbl_min + sd.table_base;
  i64* tmax = P.plain ? nullptr : P.tbl_max + sd.table_base;
  const u64 n_tbl = P.plain ? 0 : (u64)sd.instants * P.n_slots;
  for (u64 i = tid; i < n_tbl; i += blockDim.x) { tmin[i] = 0; tmax[i] = 0; }
  __syncthreads();
  u32 n_el = 0, n_st = 0;
  for (u32 i = tid; i < sd.n_units; i += blockDim.x) {
    const u32 u = sd.unit_base + i;
    EncUnit unit = P.units_in[u];
    const UnitStats us = P.ustats[u];
    bool can_elide = !P.plain;
    for (int t = 0; t < sd.instants && !P.plain; t++) {
      const InstStats is = P.istats[(size_t)u * P.t_max + t];
      i64 fmn, fmx;
      if (P.encoding == 32) {
        // min_max_float NaN quirk: min becomes NaN (-> fixed 0) when a NaN follows the first non-NaN
        fmn = (is.flags() & 3u) ? 0 : fixed_of_raw<float>(is.mn, pbits, round, err);
        fmx = (is.flags() & 1u) ? 0 : fixed_of_raw<float>(is.mx, pbits, round, err);
      } else if (P.encoding == 64) {
        fmn = (is.flags() & 3u) ? 0 : fixed_of_raw<double>(is.mn, pbits, round, err);
        fmx = (is.flags() & 1u) ? 0 : fixed_of_raw<double>(is.mx, pbits, round, err);
      } else {
        fmn = (i64)is.mn; fmx = (i64)is.mx;
      }
      tmin[(u64)t * P.n_slots + unit.slot] = fmn;
      tmax[(u64)t * P.n_slots + unit.slot] = fmx;
      can_elide = can_elide && fmn == fmx;  // superchunk.rs:145-147
    }
    int flags = P.round ? UF_ROUND : 0;
    int bits = 0;
    bool narrow = false;
    if (can_elide) {
      flags |= UF_SKIP;
      n_el++;
    } else {
      n_st++;
      if (is_float) {
        // sub_buffer.compute_fractional_bits() with the parent's bits as the request (superchunk.rs:167)
        if (us.nonfinite) err |= EF_NONFINITE;
        if (P.plain) {
          bits = pbits;  // Chunk::build uses the buffer's bits as they are (chunk.rs:50,84)
        } else {
          err |= (u32)us.sug_err;
          if (P.round) bits = min(us.sug_bits, pbits);
          else { if (us.sug_round) err |= EF_PRECISION; bits = us.sug_bits; }
        }
        if (us.has_value) {
          const double lim = ldexp(1.0, 29 - bits);  // |fixed| = 2|v| 2^bits + 1 < 2^30
          narrow = fabs(us.vmax) < lim && fabs(us.vneg) < lim;
        } else narrow = true;
      } else {
        narrow = us.imax < (i64)0x3fffffff && us.imin > -(i64)0x3fffffff;
      }
      if (narrow) flags |= UF_NARROW;
      if (is_float && !us.nonfinite && max(us.frac_nonneg, us.frac_neg) <= bits) flags |= UF_EXACT;
    }
    if (unit.rows == 64 && unit.cols == 64 && unit.lo == 0) flags |= UF_FULL;
    unit.bits = bits;
    unit.flags = flags;
    P.units[u] = unit;
    P.stored[u] = can_elide ? 0 : 1;
    if (!can_elide) {
      const bool full = unit.rows == 64 && unit.cols == 64 && unit.lo == 0;
      u32 list = (narrow ? 0u : 2u) + (full ? 0u : 1u);
      if (narrow && !full && unit.lo == 0) list = 4u;  // clipped, but still a 64-side tree: k_encode_v4<.., false>
      P.order[(size_t)list * P.order_pitch + atomicAdd(&P.order_counts[list], 1u)] = u;
    }
  }
  if (n_el) atomicAdd(&P.state[s].n_elided, n_el);
  if (n_st) atomicAdd(&P.state[s].n_stored, n_st);
  // a panic of the slice-level compute_fractional_bits (dataset.rs:842) comes before anything Superchunk::build raises
  const bool slice_failed = P.state[s].err != 0;
  __syncthreads();
  if (err && !slice_failed) atomicOr(&s_err, err);
  __syncthreads();
  if (tid == 0 && s_err) { P.state[s].err = s_err; atomicOr(P.err, s_err); }
}

// ---------------------------------------------------------------------------------------------------
// MMBuffer3::min_max over a whole region tiled into units (mmbuffer.rs:366-395): one thread per instant
// combines the per-tile extrema; the NaN quirk is decided on region row-major positions.
struct RegionMinMaxParams {
  const EncUnit* units;
  u32 n_units;
  const InstStats* istats;
  u32 t_max;
  i64 region_cols;
  int encoding, bits, round;
  int instants;
  i64* out_min;
  i64* out_max;
  u32* err;
};
__global__ void k_region_minmax(const RegionMinMaxParams P) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= P.instants) return;
  const bool is_float = P.encoding == 32 || P.encoding == 64;
  double mn = INFINITY, mx = -INFINITY;
  i64 imn = INT64_MAX, imx = INT64_MIN;
  u64 first = ~0ull, last = 0;
  for (u32 u = 0; u < P.n_units; u++) {
    const EncUnit unit = P.units[u];
    const InstStats is = P.istats[(size_t)u * P.t_max + t];
    if (is_float) {
      if (is.first != 0xffffffffu) {
        mn = fmin(mn, __longlong_as_double((long long)is.mn));
        mx = fmax(mx, __longlong_as_double((long long)is.mx));
        const u64 r = is.first / (u32)unit.cols, c = is.first % (u32)unit.cols;
        const u64 key = ((u64)unit.row0 + r) * (u64)P.region_cols + (u64)unit.col0 + c;
        first = key < first ? key : first;
      }
      if (is.last) {
        const u32 idx = is.last - 1u;
        const u64 r = idx / (u32)unit.cols, c = idx % (u32)unit.cols;
        const u64 key = ((u64)unit.row0 + r) * (u64)P.region_cols + (u64)unit.col0 + c + 1ull;
        last = key > last ? key : last;
      }
    } else {
      imn = (i64)is.mn < imn ? (i64)is.mn : imn;
      imx = (i64)is.mx > imx ? (i64)is.mx : imx;
    }
  }
  u32 err = 0;
  i64 fmn, fmx;
  if (is_float) {
    const bool all_nan = first == ~0ull;
    const bool quirk = !all_nan && last > first;
    if (P.encoding == 32) {
      fmn = (all_nan || quirk) ? 0 : to_fixed_dev<float>((float)mn, P.bits, P.round != 0, err);
      fmx = all_nan ? 0 : to_fixed_dev<float>((float)mx, P.bits, P.round != 0, err);
    } else {
      fmn = (all_nan || quirk) ? 0 : to_fixed_dev<double>(mn, P.bits, P.round != 0, err);
      fmx = all_nan ? 0 : to_fixed_dev<double>(mx, P.bits, P.round != 0, err);
    }
  } else {
    fmn = imn; fmx = imx;
  }
  P.out_min[t] = fmn;
  P.out_max[t] = fmx;
  if (err) atomicOr(P.err, err);
}

// ---------------------------------------------------------------------------------------------------
// Multi-level Superchunk::build finalisation (superchunk.rs:88-270 including its recursion :171).
// The node tree is static geometry (same for every slice): node 0 is the root superchunk, further nodes are
// the in-bounds regions that recurse.  Every child of a node is out of bounds, a leaf unit (Chunk) or
// another node; its statistics are the combination of the leaf tiles it covers.
struct TreeParams {
  const SliceDesc* slices;
  SliceState* state;         // root bits come from phase 1
  const TreeNode* nodes;
  const TreeChild* children;
  u32 n_nodes;
  const int32_t* leaf_unit;  // [leaf_rows * leaf_cols] unit index inside the slice or -1
  int leaf_cols;             // leaf tiles per row of the in-bounds leaf grid
  int leaf_side;
  u64 tbl_per_instant;       // sum of n_children over all nodes
  NodeState* nstate;         // [n_slices][n_nodes]
  EncUnit* units;
  const UnitStats* ustats;
  const InstStats* istats;
  u32 t_max;
  int encoding, round, req_bits;
  int allow_fast;            // the input layout allows k_encode_v5's 128-bit loads
  i64* tbl_min;
  i64* tbl_max;
  u32* order;
  u32 order_pitch;
  u32* order_counts;
  u8* stored;
  u32* err;
};

// order-preserving map of a double onto unsigned integers (shared-memory atomicMin / atomicMax over raw extrema)
DCDF_DEVINL unsigned long long dbl_key(double v) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
DCDF_DEVINL double key_dbl(unsigned long long k) {
  const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

// one CTA per slice; nodes in index order (parents first).  Per node: the per-instant table entries are computed by one
// thread per (child, instant) -- a child of the root of a deep tree covers hundreds of leaf tiles -- and folded per child
// through shared memory; then one thread per child classifies it.
constexpr int kTreeBatch = 1024;  // children of one node handled per round
__global__ void __launch_bounds__(256) k_finalize_tree(const TreeParams P, u32 n_slices) {
  const u32 s = blockIdx.x;
  if (s >= n_slices) return;
  const SliceDesc sd = P.slices[s];
  const int tid = threadIdx.x;
  const bool is_float = P.encoding == 32 || P.encoding == 64;
  const bool round = P.round != 0;
  NodeState* ns = P.nstate + (size_t)s * P.n_nodes;
  u32 err = 0;
  u32 n_el = 0, n_st = 0;
  __shared__ int s_slice_failed;
  __shared__ unsigned long long s_rmin[kTreeBatch], s_rmax[kTreeBatch];
  __shared__ u8 s_keep[kTreeBatch], s_nan[kTreeBatch];  // some instant has min != max; some cell is NaN
  if (tid == 0) {
    // slice-level compute_fractional_bits (dataset.rs:842): resolve the exact pass and surface its panic, which comes
    // before anything Superchunk::build raises
    SliceState st = P.state[s];
    if (st.need_exact) {
      const int rnd = st.round_exact, bits = rnd ? st.maxfb : st.f_exact;
      if (round) st.bits = min(bits, P.req_bits);              // mmbuffer.rs:602-603
      else { if (rnd) st.err |= EF_PRECISION; st.bits = bits; }  // mmbuffer.rs:605-609
      P.state[s].bits = st.bits;
      P.state[s].err = st.err;
    }
    s_slice_failed = st.err != 0;
    if (st.err) atomicOr(P.err, st.err);
    ns[0].alive = 1;
    ns[0].bits = st.bits;
    for (u32 n = 1; n < P.n_nodes; n++) { ns[n].alive = 0; ns[n].bits = 0; }
  }
  __syncthreads();
  const bool slice_failed = s_slice_failed != 0;
  for (u32 n = 0; n < P.n_nodes; n++) {
    const TreeNode nd = P.nodes[n];
    const bool alive = ns[n].alive != 0;
    const int nbits = ns[n].bits;
    i64* tmin = P.tbl_min + sd.table_base + (u64)nd.tbl_off * (u64)sd.instants;
    i64* tmax = P.tbl_max + sd.table_base + (u64)nd.tbl_off * (u64)sd.instants;
    if (alive && !nd.levels_ok) err |= EF_BAD_LEVELS;
   for (u32 c_base = 0; c_base < nd.n_children; c_base += kTreeBatch) {
    const u32 c_end = min(nd.n_children, c_base + (u32)kTreeBatch);
    for (u32 i = tid; i < c_end - c_base; i += blockDim.x) {
      s_rmin[i] = dbl_key(INFINITY); s_rmax[i] = dbl_key(-INFINITY);
      s_keep[i] = 0; s_nan[i] = 0;
    }
    __syncthreads();
    // ---- per (child, instant): table entries (superchunk.rs:140-151,192-198)
    if (alive) {
      const u32 n_items = (c_end - c_base) * (u32)sd.instants;
      for (u32 item = tid; item < n_items; item += blockDim.x) {
        const u32 ci = item % (c_end - c_base), c = c_base + ci;
        const int t = (int)(item / (c_end - c_base));
        const TreeChild ch = P.children[nd.first_child + c];
        if (ch.kind == 0) {  // entirely outside the raster: Elided with (0,0) per instant (superchunk.rs:134-139)
          tmin[(u64)t * nd.n_children + c] = 0; tmax[(u64)t * nd.n_children + c] = 0;
          continue;
        }
        const i64 region_cols = (i64)(ch.gc1 - ch.gc0) * P.leaf_side;
        double mn = INFINITY, mx = -INFINITY;
        i64 lmn = INT64_MAX, lmx = INT64_MIN;
        u64 first = ~0ull, last = 0;
        for (int gr = ch.gr0; gr < ch.gr1; gr++)
          for (int gc = ch.gc0; gc < ch.gc1; gc++) {
            const int32_t lu = P.leaf_unit[gr * P.leaf_cols + gc];
            if (lu < 0) continue;
            const u32 u = sd.unit_base + (u32)lu;
            const InstStats is = P.istats[(size_t)u * P.t_max + t];
            if (is_float) {
              const int ucols = P.units[u].cols;
              const u64 r_off = (u64)(gr - ch.gr0) * P.leaf_side, c_off = (u64)(gc - ch.gc0) * P.leaf_side;
              if (is.first != 0xffffffffu) {
                mn = fmin(mn, __longlong_as_double((long long)is.mn));
                mx = fmax(mx, __longlong_as_double((long long)is.mx));
                const u64 key = (r_off + is.first / (u32)ucols) * (u64)region_cols + c_off + is.first % (u32)ucols;
                first = key < first ? key : first;
              }
              if (is.last) {
                const u32 idx = is.last - 1u;
                const u64 key = (r_off + idx / (u32)ucols) * (u64)region_cols + c_off + idx % (u32)ucols + 1ull;
                last = key > last ? key : last;
              }
            } else {
              lmn = (i64)is.mn < lmn ? (i64)is.mn : lmn;
              lmx = (i64)is.mx > lmx ? (i64)is.mx : lmx;
            }
          }
        i64 fmn, fmx;
        if (is_float) {
          const bool all_nan = first == ~0ull;
          if (all_nan || last != 0) s_nan[ci] = 1;
          if (!all_nan) { atomicMin(&s_rmin[ci], dbl_key(mn)); atomicMax(&s_rmax[ci], dbl_key(mx)); }
          const bool quirk = !all_nan && last > first;  // mmbuffer.rs:485-487
          if (P.encoding == 32) {
            fmn = (all_nan || quirk) ? 0 : to_fixed_dev<float>((float)mn, nbits, round, err);
            fmx = all_nan ? 0 : to_fixed_dev<float>((float)mx, nbits, round, err);
          } else {
            fmn = (all_nan || quirk) ? 0 : to_fixed_dev<double>(mn, nbits, round, err);
            fmx = all_nan ? 0 : to_fixed_dev<double>(mx, nbits, round, err);
          }
        } else {
          fmn = lmn; fmx = lmx;
        }
        tmin[(u64)t * nd.n_children + c] = fmn;
        tmax[(u64)t * nd.n_children + c] = fmx;
        if (fmn != fmx) s_keep[ci] = 1;  // superchunk.rs:145-147
      }
    }
    __syncthreads();
    // ---- per child: classification
    for (u32 c = c_base + tid; c < c_end; c += blockDim.x) {
      const TreeChild ch = P.children[nd.first_child + c];
      if (!alive) {
        if (ch.kind == 1) {
          const u32 u = sd.unit_base + (u32)ch.index;
          EncUnit unit = P.units[u];
          unit.flags |= UF_SKIP;
          P.units[u] = unit;
          P.stored[u] = 0;
        }
        continue;
      }
      if (ch.kind == 0) continue;
      bool has = false, nonfinite = false;
      double vmax = -INFINITY, vneg = 0.0;
      int fnn = 0, fng = 0;
      i64 imax = INT64_MIN, imin = INT64_MAX;
      const bool can_elide = s_keep[c - c_base] == 0;
      const bool any_nan = s_nan[c - c_base] != 0;  // some cell of some instant is NaN
      const double rmin = key_dbl(s_rmin[c - c_base]), rmax = key_dbl(s_rmax[c - c_base]);  // raw extrema over every instant (fast-path eligibility)
      // unit-level summaries over the covered tiles (for compute_fractional_bits of the child, :167)
      for (int gr = ch.gr0; gr < ch.gr1; gr++)
        for (int gc = ch.gc0; gc < ch.gc1; gc++) {
          const int32_t lu = P.leaf_unit[gr * P.leaf_cols + gc];
          if (lu < 0) continue;
          const UnitStats us = P.ustats[sd.unit_base + (u32)lu];
          if (us.has_value) { has = true; vmax = fmax(vmax, us.vmax); }
          vneg = fmin(vneg, us.vneg);
          fnn = max(fnn, us.frac_nonneg); fng = max(fng, us.frac_neg);
          nonfinite = nonfinite || us.nonfinite;
          imax = us.imax > imax ? us.imax : imax;
          imin = us.imin < imin ? us.imin : imin;
        }
      int cbits = 0;
      if (!can_elide && is_float) {
        int sug_round = 0, sug_bits = 0, sug_err = 0;
        if (ch.kind == 1) {
          const UnitStats us = P.ustats[sd.unit_base + (u32)ch.index];
          sug_round = us.sug_round; sug_bits = us.sug_bits; sug_err = us.sug_err;  // exact (second pass inside k_unit_stats)
        } else if (!suggest_from_summary(has, vmax, vneg, fnn, fng, sug_round, sug_bits, sug_err)) {
          err |= EF_REGION_EXACT;
        }
        err |= (u32)sug_err;
        if (nonfinite) err |= EF_NONFINITE;
        if (round) cbits = min(sug_bits, nbits);               // mmbuffer.rs:602-603
        else { if (sug_round) err |= EF_PRECISION; cbits = sug_bits; }
      }
      if (ch.kind == 2) {
        ns[ch.index].alive = can_elide ? 0 : 1;
        ns[ch.index].bits = cbits;
      } else {
        const u32 u = sd.unit_base + (u32)ch.index;
        EncUnit unit = P.units[u];
        int flags = round ? UF_ROUND : 0;
        bool narrow = false;
        if (can_elide) {
          flags |= UF_SKIP;
          n_el++;
        } else {
          n_st++;
          if (is_float) {
            if (has) {
              const double lim = ldexp(1.0, 29 - cbits);  // |fixed| = 2|v| 2^bits + 1 < 2^30
              narrow = fabs(vmax) < lim && fabs(vneg) < lim;
            } else narrow = true;
          } else {
            narrow = imax < (i64)0x3fffffff && imin > -(i64)0x3fffffff;
          }
          if (narrow) flags |= UF_NARROW;
          if (is_float && !nonfinite && max(fnn, fng) <= cbits) flags |= UF_EXACT;  // a leaf child covers exactly its own unit
        }
        const bool full = unit.rows == 64 && unit.cols == 64 && unit.lo == 0;
        if (full) flags |= UF_FULL;
        // k_encode_v5 (encode_v5.cuh): f32 tiles with a 64-side tree whose to_fixed is exact, every fixed value below
        // 2^22 in magnitude and all of them within 32767 of each other -> every entry below the root takes <= 2 bytes
        bool fast = false;
        if (P.allow_fast && !can_elide && unit.lo == 0 && narrow && P.encoding == 32 && (flags & UF_EXACT) && has) {
          const double sc = ldexp(1.0, cbits + 1);
          // fixed = 2 v 2^bits + 1 for values, 0 for NaN: every code of the unit within 32767 of every other one
          double lo = rmin * sc + 1.0, hi = rmax * sc + 1.0;
          if (any_nan) { lo = fmin(lo, 0.0); hi = fmax(hi, 0.0); }
          fast = hi - lo <= 32767.0 && fabs(hi) < 4194303.0 && fabs(lo) < 4194303.0;
          // clipped tiles: an entry next to a cell outside the raster is the max itself (snapshot.rs:122-130 with None => 0)
          if (!full) fast = fast && fabs(hi) <= 32767.0 && fabs(lo) <= 32767.0;
        }
        unit.bits = cbits;
        unit.flags = flags;
        P.units[u] = unit;
        P.stored[u] = can_elide ? 0 : 1;
        if (!can_elide) {
          u32 list = (narrow ? 0u : 2u) + (full ? 0u : 1u);
          if (narrow && !full && unit.lo == 0) list = 4u;  // clipped, but still a 64-side tree: k_encode_v4<.., false>
          if (fast) list = full ? 5u : 6u;                  // k_encode_v5<.., true / false>
          // ... at most 32 rows or columns in the raster: half of the tree holds no cell -> one warp per tile
          if (fast && !full && min(unit.rows, unit.cols) <= 32) list = 7u;  // k_encode_v5_edge
          P.order[(size_t)list * P.order_pitch + atomicAdd(&P.order_counts[list], 1u)] = u;
        }
      }
    }
    __syncthreads();  // node states written by this node's children are read by later nodes; the shared accumulators are reused
   }
  }
  if (n_el) atomicAdd(&P.state[s].n_elided, n_el);
  if (n_st) atomicAdd(&P.state[s].n_stored, n_st);
  if (err && !slice_failed) { atomicOr(&P.state[s].err, err); atomicOr(P.err, err); }
}

}  // namespace dcdf
