// numerics.cuh - the float32 recipe of the projection, shared by every kernel that
// quantizes (and compiled for the host by tests/hostcheck to pin it against the oracle).
//
// Follows source/quantization.py:69-144 of the reference operation by operation:
// IEEE float32 multiply / divide / subtract with round-to-nearest-even and no FMA
// contraction, `torch.round` = rint (half to even), `torch.linspace` = FMA form
// (SURVEY App. A.3).  Nothing here may be compiled with --use_fast_math.
#pragma once
#include <cstdint>
#include <cmath>
#include <cstring>

#if defined(__CUDACC__)
#define ADMMQ_HD __host__ __device__ __forceinline__
#else
#define ADMMQ_HD inline
#endif

namespace admmq {

// --- explicitly rounded float32 primitives (no contraction on either side) ------------
ADMMQ_HD float mul_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fmul_rn(a, b);
#else
  volatile float r = a * b;
  return r;
#endif
}
ADMMQ_HD float add_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fadd_rn(a, b);
#else
  volatile float r = a + b;
  return r;
#endif
}
ADMMQ_HD float sub_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fsub_rn(a, b);
#else
  volatile float r = a - b;
  return r;
#endif
}
ADMMQ_HD float div_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
  return __fdiv_rn(a, b);
#else
  volatile float r = a / b;
  return r;
#endif
}
ADMMQ_HD float fma_rn(float a, float b, float c) {
#if defined(__CUDA_ARCH__)
  return __fmaf_rn(a, b, c);
#else
  return fmaf(a, b, c);
#endif
}
ADMMQ_HD float rint_rn(float a) {
#if defined(__CUDA_ARCH__)
  return rintf(a);
#else
  return nearbyintf(a);
#endif
}

// --- quantizer description -------------------------------------------------------------
struct Levels {
  float lo;     // -q            (source/quantization.py:88: q = 2**(bits-1))
  float hi;     //  q-1
  float denom;  //  2q-1         (:89 scale_denom)
  float fast_lo, fast_hi, fast_thr;  // fast-path clamp window and "too close to .5" threshold
  int fmt;      // the FP8 / FP6 format of the clip search (kFmtE4M3 .. kFmtE2M3), 0 on every other grid
};

ADMMQ_HD Levels make_levels(int bits, int fmt = 0) {
  Levels L;
  L.fmt = fmt;
  const float q = (float)(1 << (bits - 1));
  L.lo = -q;
  L.hi = q - 1.0f;
  L.denom = 2.0f * q - 1.0f;
  L.fast_lo = -q - 0.25f;
  L.fast_hi = q - 0.75f;
  // |x*rcp(s) - x/s| <= |t| * 2^-23 (two roundings) and |fl(x/s) - x/s| <= |t| * 2^-24;
  // (q + 2) * 2^-21 leaves a >2.5x margin for every quotient |t| <= q + 1.5 whose rounding can matter (larger ones
  // clamp to the same code either way).
  L.fast_thr = 0.5f - (q + 2.0f) * 4.76837158203125e-07f;
  return L;
}

// --- candidate grid of quantize_tensor_mse (source/quantization.py:129-131) ----------
struct ClipGrid {
  float start, end, step;
  int n;
};

ADMMQ_HD ClipGrid make_clip_grid(float absmax, int n) {
  ClipGrid g;
  g.n = n;
  g.start = (float)(0.2 * (double)absmax);
  g.end = (float)(1.2 * (double)absmax);
  g.step = n > 1 ? div_rn(sub_rn(g.end, g.start), (float)(n - 1)) : 0.0f;
  return g;
}

ADMMQ_HD float clip_candidate(const ClipGrid& g, int i) {
  if (g.n == 1) return g.start;
  return (i < g.n / 2) ? fma_rn(g.step, (float)i, g.start) : fma_rn(-g.step, (float)(g.n - 1 - i), g.end);
}

// scale = 2 * tmax / scale_denom  (source/quantization.py:125)
ADMMQ_HD float scale_of(float clip, const Levels& L) { return div_rn(mul_rn(2.0f, clip), L.denom); }

// clamp(round(x / scale), -q, q-1)  (source/quantization.py:127) - the exact form
ADMMQ_HD float code_exact(float x, float scale, const Levels& L) {
  float k = rint_rn(div_rn(x, scale));
  k = fminf(fmaxf(k, L.lo), L.hi);
  return k;
}

// (x - code*scale)^2 with every intermediate rounded to float32 (:127, :138)
ADMMQ_HD float sqerr_exact(float x, float scale, const Levels& L) {
  const float d = sub_rn(x, mul_rn(code_exact(x, scale, L), scale));
  return mul_rn(d, d);
}

// Deviation (x - code*scale) with every intermediate rounded to float32 (:127, :138) - exact form.
ADMMQ_HD float dev_exact(float x, float scale, const Levels& L) {
  return sub_rn(x, mul_rn(code_exact(x, scale, L), scale));
}

// Fast path used inside the 200-candidate search: the code is obtained from x * (1/scale)
// (no division); `frac` returns |t - k| so that the caller can detect the rare inputs whose
// quotient lies too close to a rounding boundary for the shortcut to be provably equal to
// code_exact() and redo them with dev_exact().  MAGIC rounding = round-half-even for |t| < 2^22
// (|t| <= 37.5 here: |x| <= absmax and scale >= 0.2 * absmax * 2 / denom).
ADMMQ_HD float dev_fast(float x, float scale, float rcp_scale, const Levels& L, float& frac) {
  const float MAGIC = 12582912.0f;  // 1.5 * 2^23
  float t = mul_rn(x, rcp_scale);
  t = fminf(fmaxf(t, L.fast_lo), L.fast_hi);
  const float k = sub_rn(add_rn(t, MAGIC), MAGIC);
  frac = fabsf(sub_rn(t, k));
  return sub_rn(x, mul_rn(k, scale));
}
// An alternative form (not used by the kernels, see search.cuh eval_pair; kept pinned by the host tests): round the EXACT product x * rcp_scale (one FMA with the magic
// constant), take its rounding residual r with a second FMA, clamp the integer afterwards.  rint(x / scale) can differ
// from the rounded product only when the quotient lies within |x/s| * 2^-23 of a half integer, and only matters while
// the integer is inside [-q - 1, q]; |r| <= fast_thr = 0.5 - q * 2^-21 excludes both, everything else is redone exactly.
ADMMQ_HD float dev_fast2(float x, float scale, float rcp_scale, const Levels& L, float& frac) {
  const float MAGIC = 12582912.0f;  // 1.5 * 2^23
  const float ku = sub_rn(fma_rn(x, rcp_scale, MAGIC), MAGIC);
  frac = fabsf(fma_rn(x, rcp_scale, -ku));
  const float k = fminf(fmaxf(ku, L.lo), L.hi);
  return sub_rn(x, mul_rn(k, scale));
}
ADMMQ_HD float sqerr_fast(float x, float scale, float rcp_scale, const Levels& L, float& frac) {
  const float d = dev_fast(x, scale, rcp_scale, L, frac);
  return mul_rn(d, d);
}

// --- the summation recipe of the clip search ---------------------------------------------
// The reference takes `mean((x - xq)**2)` in float32 with ATen's reduction order, which no other
// implementation can reproduce bit for bit.  The kernels define the per-candidate sum as follows
// (tests/hostcheck pins this definition against the reference's argmin on the golden vectors):
//   * elements are taken in aligned groups of 8 (kSumGroup); missing tail elements count as x = 0,
//     which contributes exactly 0;
//   * within a group two float32 FMA chains accumulate d*d, one over the even and one over the odd
//     positions (the two lanes of a packed f32x2 FMA), and are added in float32;
//   * the 8 group sums of an aligned block of 64 elements (kSumBlock) are added in float32 in order (the float32 ->
//     float64 conversion runs on the quarter-rate conversion pipe: once per 64 elements instead of once per 8 it
//     costs ~2 % instead of ~14 % of the search);
//   * block sums are added in float64 in element order, the CTA/chunk totals in 64-bit fixed point.
// Blocks are aligned to the ABSOLUTE element index (chunk starts, stage sizes and warp slices are multiples of 64), so
// the result does not depend on the grid size or on how the elements are split over CTAs and warps.
constexpr int kSumGroup = 8;
constexpr int kSumBlock = 64;
ADMMQ_HD float group_sum8(const float d[kSumGroup]) {
  float even = 0.0f, odd = 0.0f;
  for (int i = 0; i < kSumGroup; i += 2) {
    even = fma_rn(d[i], d[i], even);
    odd = fma_rn(d[i + 1], d[i + 1], odd);
  }
  return add_rn(even, odd);
}

// --- fixed-point accumulation of the per-candidate squared-error sums --------------------
// Every element contributes d^2 <= 16 * absmax^2, so sum <= 16 * N * absmax^2 which is mapped to
// 2^62.  Integer addition is associative: the total does not depend on how many CTAs or in which
// order the partial sums arrive, and it resolves ~3e-15 of a typical total.
ADMMQ_HD double fixed_point_unit_inv(double n_elems, float absmax) {
  const double bound = n_elems * (double)absmax * (double)absmax;  // * 16 folded into 2^58
  return 288230376151711744.0 /* 2^58 */ / bound;
}
ADMMQ_HD double fixed_point_unit(double n_elems, float absmax) {
  const double bound = n_elems * (double)absmax * (double)absmax;
  return bound / 288230376151711744.0;
}

// mean as the reference forms it (:138 `.mean`): float32 total divided by float32 count, where
// the total is the correctly rounded sum of the float32 squares.
ADMMQ_HD float mse_from_fixed(long long fixed_sum, double unit, float n_elems_f) {
  const float total = (float)((double)fixed_sum * unit);
  return div_rn(total, n_elems_f);
}

// --- the threshold ("binned") form of the clip search ----------------------------------------
// For one candidate scale s the quantizer k(x) = clamp(rint(x / s), -q, q-1) is a monotone step function of x, so
// it is fully described by its 2q-1 thresholds: theta_j = the SMALLEST float32 x with rint(fl(x / s)) >= -q + j + 1
// (found by stepping through neighbouring floats with the exact division, so ties-to-even and the rounding of the
// quotient are captured exactly).  With C_j = #{x < theta_j}, P_j = sum{x < theta_j} x, the grid values
// y_j = fl32((-q + j) * s) (source/quantization.py:127 rounds `codes * scale` to float32) and summation by parts,
//     sum_e (x_e - y_k(e))^2 = sum_e x_e^2 + sum_{j=0}^{2q-2} [ C_j (y_j^2 - y_{j+1}^2) - 2 P_j (y_j - y_{j+1}) ]
//                                           + n y_top^2 - 2 P_tot y_top,
// which needs C and P at (2q-1) * num_attempts thresholds instead of num_attempts evaluations per element.  C is an
// integer, P is accumulated in 64-bit fixed point (x rounded to 2^-41 of the power of two above absmax), the bracket is
// evaluated in float64 and converted to the fixed-point unit of the per-candidate accumulators, so the result is
// independent of arrival order (bit-reproducible) and depends on the chunking only through the fixed-point rounding
// of the per-chunk terms (~1e-13 relative).  It is the exact real-number value of the reference's
// sum((x - xq)**2) up to ~1e-12 relative; the reference's own float32 evaluation of that sum carries ~1e-7.
ADMMQ_HD unsigned int f32_bits(float f) {
#if defined(__CUDA_ARCH__)
  return __float_as_uint(f);
#else
  unsigned int u;
  std::memcpy(&u, &f, 4);
  return u;
#endif
}
ADMMQ_HD float bits_f32(unsigned int u) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(u);
#else
  float f;
  std::memcpy(&f, &u, 4);
  return f;
#endif
}
// order-preserving map float -> uint32 (larger float <=> larger key); NaN maps above +inf
ADMMQ_HD unsigned int ordered_key(float f) {
  const unsigned int b = f32_bits(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
ADMMQ_HD float ordered_float(unsigned int k) { return bits_f32((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// smallest float32 x with rint(fl(x / scale)) >= level + 1   (level = -q .. q-2), in closed form:
//   rint(y) >= T  <=>  y >= y*,  y* = T - 0.5 if T is even (the tie rounds up to T), else the next float above it;
//   fl(z) >= y*   <=>  z > mid or (z == mid and the mantissa of y* is even),  mid = midpoint of pred(y*) and y*;
//   mid * scale is exact in float64 (25 x 24 significant bits), so theta is the first float above that product
//   (or the product itself when it is a float and the tie goes to y*).
// tests/hostcheck pins theta and its predecessor against the exact division for every level of random scales.
// The level-only part (mid, parity of y*) and the scale-dependent part are separate so that the clip search forms the
// former once per level instead of once per (candidate, level) pair.
struct ThresholdMid {
  double mid;   // midpoint of pred(y*) and y* (25 significant bits, never zero)
  bool odd;     // mantissa of y* is odd: a product that lands exactly on mid rounds away from y*
};
ADMMQ_HD ThresholdMid threshold_mid(float level) {
  const float target = level + 1.0f;
  const float b = target - 0.5f;
  const bool t_even = (((int)target) & 1) == 0;
  const float ystar = t_even ? b : ordered_float(ordered_key(b) + 1u);
  const float pred = ordered_float(ordered_key(ystar) - 1u);
  ThresholdMid m;
  m.mid = 0.5 * ((double)pred + (double)ystar);
  m.odd = (f32_bits(ystar) & 1u) != 0u;
  return m;
}
ADMMQ_HD float code_threshold_from_mid(float scale, double mid, bool odd) {
  const double P = mid * (double)scale;                 // exact; scale > 0, so P != 0 and has the sign of mid
  float x = (float)P;                                   // round to nearest
  const double xd = (double)x;
  // first float above P, or P itself when it is a float and the tie goes to y*: one step towards +inf
  if (xd < P || (xd == P && odd)) x = bits_f32(f32_bits(x) + (x > 0.0f ? 1u : 0xffffffffu));
  return x;
}
ADMMQ_HD float code_threshold(float scale, float level) {
  const ThresholdMid m = threshold_mid(level);
  return code_threshold_from_mid(scale, m.mid, m.odd);
}

// the same threshold by stepping through neighbouring floats with the exact division (reference implementation of the
// definition; used by the host tests)
ADMMQ_HD float code_threshold_search(float scale, float level) {
  const float target = level + 1.0f;
  unsigned int key = ordered_key(mul_rn(level + 0.5f, scale));
  if (rint_rn(div_rn(ordered_float(key), scale)) >= target) {
    for (int it = 0; it < 64 && rint_rn(div_rn(ordered_float(key - 1u), scale)) >= target; ++it) --key;
  } else {
    for (int it = 0; it < 64; ++it) {
      ++key;
      if (rint_rn(div_rn(ordered_float(key), scale)) >= target) break;
    }
  }
  return ordered_float(key);
}

// 64-bit fixed point of the elements: unit = 2^-41 of the power of two above absmax.  The threshold form is used for
// absmax in [2^-40, 2^40] (float32 squares neither overflow nor vanish); outside, the kernels fall back to the direct
// per-element evaluation.
struct FixX {
  float p2a;     // 2^a with 2^20 <= absmax * 2^a < 2^21
  double unit;   // value of one fixed-point step = 2^-(a + 20)
};
constexpr float kBinnedMinAbs = 9.094947017729282e-13f;  // 2^-40
constexpr float kBinnedMaxAbs = 1099511627776.0f;        // 2^40
ADMMQ_HD bool binned_range_ok(float absmax) { return absmax >= kBinnedMinAbs && absmax <= kBinnedMaxAbs; }
ADMMQ_HD FixX make_fix_x(float absmax) {
  const int e = (int)((f32_bits(absmax) >> 23) & 0xffu) - 127;  // absmax = 1.m * 2^e
  FixX f;
  f.p2a = bits_f32((unsigned int)(20 - e + 127) << 23);
  // 2^-(a + 20) = 2^(e - 40) as a double
  unsigned long long db = (unsigned long long)(e - 40 + 1023) << 52;
#if defined(__CUDA_ARCH__)
  f.unit = __longlong_as_double((long long)db);
#else
  std::memcpy(&f.unit, &db, 8);
#endif
  return f;
}
// x -> rne(x * 2^(a + 20)) without the conversion pipe: two magic-number roundings (|x * 2^a| < 2^21)
ADMMQ_HD long long fix_x(float x, const FixX& f) {
  const float MAGIC = 12582912.0f;  // 1.5 * 2^23, bits 0x4B400000
  const float xs = mul_rn(x, f.p2a);                 // exact (power of two)
  const float hb = add_rn(xs, MAGIC);                // integer part (rne) in the low mantissa bits
  const float r = sub_rn(xs, sub_rn(hb, MAGIC));     // exact, |r| <= 0.5
  const float lb = fma_rn(r, 1048576.0f, MAGIC);     // rne(r * 2^20)
  const long long th = (long long)((int)f32_bits(hb) - 0x4B400000);
  const long long tl = (long long)((int)f32_bits(lb) - 0x4B400000);
  return th * 1048576ll + tl;
}

// sum of squares of four consecutive elements as the kernels form it (float32 FMA chain, then float64)
ADMMQ_HD float sumsq4(float a, float b, float c, float d) {
  return fma_rn(d, d, fma_rn(c, c, fma_rn(b, b, mul_rn(a, a))));
}

// contribution of threshold j of one candidate to the per-candidate sum, in float64:
//   C (y_lo^2 - y_hi^2) - 2 P unit (y_lo - y_hi),   y_lo = fl32(lo_level * s), y_hi = fl32(hi_level * s)
// for the two neighbouring levels of the grid that the threshold separates
ADMMQ_HD double threshold_term(float scale, float lo_level, float hi_level, long long count, long long psum, double xunit) {
  const double ylo = (double)mul_rn(lo_level, scale), yhi = (double)mul_rn(hi_level, scale);
  const double d1 = ylo - yhi;
  return (double)count * (d1 * (ylo + yhi)) - 2.0 * ((double)psum * xunit) * d1;
}
// the integer grid: levels `level` and `level + 1`
ADMMQ_HD double threshold_term(float scale, float level, long long count, long long psum, double xunit) {
  return threshold_term(scale, level, level + 1.0f, count, psum, xunit);
}
// closing term n y_top^2 - 2 P_tot unit y_top, y_top = fl32((q - 1) * s)
ADMMQ_HD double closing_term(float scale, float top_level, long long n, long long ptot, double xunit) {
  const double y = (double)mul_rn(top_level, scale);
  return (double)n * (y * y) - 2.0 * ((double)ptot * xunit) * y;
}

// --- the FP4 E2M1 grid (tensor_mseminmax_e2m1, ADMMQ_Q_MSEMINMAX_E2M1) ---------------------------
// The reference has no such scheme; this is its definition (DESIGN.md 2b).  bits = 4 only.
//   candidates  the clip grid of quantize_tensor_mse, make_clip_grid(absmax, num_attempts); scale s_c = fl(clip_c / 6)
//   element     t = fl(x / s); the level is t rounded to the nearest of +-{0, 0.5, 1, 1.5, 2, 3, 4, 6}, ties to the
//               even mantissa, saturating at +-6 - what cvt.rn.satfinite.e2m1x2.f32 does to t; the value is
//               fl(level * s), -0 for a small negative t
//   code        the 4-bit E2M1 encoding 0 .. 15: bit 3 sign, bits 2-1 exponent, bit 0 mantissa
//   choice      the first minimum of the candidate MSEs, with the sums of the uniform search (fixed point, same argmin)
// The 15 distinct values -6 .. 6 have 14 boundaries; their thresholds come in closed form (e2m1_threshold_mid).
constexpr float kE2M1Magnitude[8] = {0.0f, 0.5f, 1.0f, 1.5f, 2.0f, 3.0f, 4.0f, 6.0f};   // by code & 7
constexpr int kE2M1Thresholds = 14;
constexpr float kE2M1Max = 6.0f;

// value of a code, from its bits (no table lookup on the device): magnitude 2^(e-1) (1 + m/2) for e > 0, m/2 for e = 0
ADMMQ_HD float e2m1_value(unsigned int code) {
  const unsigned int i = code & 7u;
  const unsigned int mag = i == 0u ? 0u : (i + (i == 1u ? 251u : 252u)) << 22;
  return bits_f32(mag | ((code & 8u) << 28));
}

// round-to-nearest-even onto E2M1 with saturation, in software (the host's form of the hardware conversion; t not NaN)
ADMMQ_HD unsigned int e2m1_round_sw(float t) {
  const float a = fabsf(t);
  // the boundaries are midpoints of neighbouring magnitudes; a tie goes to the even mantissa (even index)
  unsigned int i;
  if (a <= 0.25f) i = 0u;
  else if (a < 0.75f) i = 1u;
  else if (a <= 1.25f) i = 2u;
  else if (a < 1.75f) i = 3u;
  else if (a <= 2.5f) i = 4u;
  else if (a < 3.5f) i = 5u;
  else if (a <= 5.0f) i = 6u;
  else i = 7u;
  return i | ((f32_bits(t) >> 28) & 8u);
}

// code of a quotient t: cvt.rn.satfinite.e2m1x2.f32 on the device, e2m1_round_sw on the host
ADMMQ_HD unsigned int e2m1_code(float t) {
#if defined(__CUDA_ARCH__)
  unsigned int r;
  asm("{\n\t.reg .b8 b;\n\tcvt.rn.satfinite.e2m1x2.f32 b, %1, %1;\n\tmov.b32 %0, {b, b, b, b};\n\t}" : "=r"(r) : "f"(t));
  return r & 15u;
#else
  return e2m1_round_sw(t);
#endif
}

ADMMQ_HD float e2m1_scale_of(float clip) { return div_rn(clip, kE2M1Max); }

// the element step of the definition: code and value of x on the grid of scale s (exact division)
ADMMQ_HD float e2m1_quantize(float x, float scale, float& code) {
  const unsigned int c = e2m1_code(div_rn(x, scale));
  code = (float)c;
  return mul_rn(e2m1_value(c), scale);
}
ADMMQ_HD float e2m1_dev(float x, float scale) {
  float code;
  return sub_rn(x, e2m1_quantize(x, scale, code));
}

// the 15 distinct values in ascending order, j = 0 .. 14 (-6 .. 6; j = 7 is +0), and the code of each
ADMMQ_HD unsigned int e2m1_grid_code(int j) { return j < 7 ? (unsigned int)(15 - j) : (unsigned int)(j - 7); }
ADMMQ_HD float e2m1_grid_level(int j) { return e2m1_value(e2m1_grid_code(j)); }

// threshold j (j = 0 .. 13) separates grid values j and j + 1: the smallest float32 x with level(fl(x / s)) >= value
// j + 1.  The boundary b = (value j + value j+1) / 2 is exact in float32; rounding onto E2M1 reaches value j + 1 for
// t >= y*, y* = b when the tie goes up (value j + 1 has the even mantissa), else the next float above b.  From y* the
// midpoint machinery of the integer grid applies unchanged (code_threshold_from_mid).
ADMMQ_HD ThresholdMid e2m1_threshold_mid(int j) {
  const float b = mul_rn(0.5f, add_rn(e2m1_grid_level(j), e2m1_grid_level(j + 1)));
  const bool tie_up = (e2m1_grid_code(j + 1) & 1u) == 0u;
  const float ystar = tie_up ? b : ordered_float(ordered_key(b) + 1u);
  const float pred = ordered_float(ordered_key(ystar) - 1u);
  ThresholdMid m;
  m.mid = 0.5 * ((double)pred + (double)ystar);
  m.odd = (f32_bits(ystar) & 1u) != 0u;
  return m;
}
ADMMQ_HD float e2m1_threshold(float scale, int j) {
  const ThresholdMid m = e2m1_threshold_mid(j);
  return code_threshold_from_mid(scale, m.mid, m.odd);
}
// the same threshold by stepping through neighbouring floats with the exact division (reference of the definition;
// used by the host tests)
ADMMQ_HD bool e2m1_reaches(float x, float scale, float level) { return e2m1_value(e2m1_code(div_rn(x, scale))) >= level; }
ADMMQ_HD float e2m1_threshold_search(float scale, int j) {
  const float target = e2m1_grid_level(j + 1);
  const float b = mul_rn(0.5f, add_rn(e2m1_grid_level(j), target));
  unsigned int key = ordered_key(mul_rn(b, scale));
  if (e2m1_reaches(ordered_float(key), scale, target)) {
    for (int it = 0; it < 64 && e2m1_reaches(ordered_float(key - 1u), scale, target); ++it) --key;
  } else {
    for (int it = 0; it < 64; ++it) {
      ++key;
      if (e2m1_reaches(ordered_float(key), scale, target)) break;
    }
  }
  return ordered_float(key);
}

// --- the FP8 (E4M3, E5M2) and FP6 (E3M2, E2M3) grids (tensor_mseminmax_e4m3 / _e5m2 / _e3m2 / _e2m3) ----------------
// The reference has no such schemes; this is their definition (DESIGN.md 2c), the E2M1 definition with another value set:
//   candidates  make_clip_grid(absmax, num_attempts); scale s_c = fl(clip_c / max)
//   element     t = fl(x / s); the level is t rounded to the nearest value of the format, ties to the even mantissa,
//               saturating at +-max, subnormals included - what cvt.rn.satfinite.<fmt>x2.f32 does to t; the value is
//               fl(level * s), -0 for a small negative t
//   code        the format's encoding: for FP8 the byte itself (int8 storage of float8_e4m3fn / float8_e5m2), for FP6
//               0 .. 63 (bit 5 sign, then the exponent bits, then the mantissa bits)
//   choice      the first minimum of the candidate MSEs, with the sums of the uniform search (fixed point, same argmin)
// A non-finite abs-max takes the NONFINITE path first, as on the integer grid; a NaN element that still reaches the
// element step takes -max, as on the integer grid (fp_quantize).
// The format is a run-time value (the scheme id): one instantiation of every kernel serves all four.
constexpr int kFmtE4M3 = 6, kFmtE5M2 = 7, kFmtE3M2 = 8, kFmtE2M3 = 9;   // = ADMMQ_Q_MSEMINMAX_E4M3 .. _E2M3
ADMMQ_HD bool fp_format_id(int fmt) { return fmt >= kFmtE4M3 && fmt <= kFmtE2M3; }

struct FpFormat {
  int bits, ebits, mbits, bias;
  bool nan_top;   // the all-ones magnitude is NaN and the one below it is max (E4M3); otherwise max is the all-ones
                  // magnitude (FP6) or the last one below the IEEE infinities and NaNs (E5M2)
  int top;        // magnitude code of max: the magnitudes 0 .. top ascend with their codes
  float max;
};
ADMMQ_HD FpFormat fp_format(int fmt) {
  switch (fmt) {
    case kFmtE4M3: return {8, 4, 3, 7, true, 126, 448.0f};
    case kFmtE5M2: return {8, 5, 2, 15, false, 123, 57344.0f};
    case kFmtE3M2: return {6, 3, 2, 3, false, 31, 28.0f};
    default: return {6, 2, 3, 1, false, 31, 7.5f};   // kFmtE2M3
  }
}
// distinct values -max .. max (+-0 merged into one) and the thresholds between them: 2 top + 1 and 2 top
ADMMQ_HD int fp_thresholds(int fmt) { return 2 * fp_format(fmt).top; }

// value of a finite code from its bits: subnormal m 2^(1 - bias - mbits), normal (2^mbits + m) 2^(e - bias - mbits);
// both exact in float32
ADMMQ_HD float fp_value(int fmt, unsigned int code) {
  const FpFormat f = fp_format(fmt);
  const unsigned int sign = 1u << (f.bits - 1), k = code & (sign - 1u);
  const unsigned int e = k >> f.mbits, m = k & ((1u << f.mbits) - 1u);
  const float ulp = bits_f32((unsigned int)(127 + (e != 0u ? (int)e : 1) - f.bias - f.mbits) << 23);
  const float mag = mul_rn((float)(e != 0u ? (m | (1u << f.mbits)) : m), ulp);
  return bits_f32(f32_bits(mag) | ((code & sign) != 0u ? 0x80000000u : 0u));
}

// round-to-nearest-even onto the format with saturation, in software: the definition, and the host's form of the
// hardware conversion (t not NaN).  Between neighbouring magnitudes the boundary is their midpoint (exact in float32);
// a tie goes to the even mantissa, which is the even magnitude code.
ADMMQ_HD unsigned int fp_round_sw(int fmt, float t) {
  const FpFormat f = fp_format(fmt);
  const float a = fabsf(t);
  unsigned int lo = 0u, hi = (unsigned int)f.top;
  if (a >= f.max) {
    lo = hi;   // saturation, +-inf included
  } else {     // value(lo) <= a < value(hi)
    while (hi - lo > 1u) {
      const unsigned int mid = (lo + hi) >> 1;
      if (fp_value(fmt, mid) <= a) lo = mid;
      else hi = mid;
    }
    const float b = mul_rn(0.5f, add_rn(fp_value(fmt, lo), fp_value(fmt, hi)));
    if (a > b || (a == b && (hi & 1u) == 0u)) lo = hi;
  }
  return lo | ((f32_bits(t) >> 31) << (f.bits - 1));
}

#if defined(__CUDA_ARCH__)
// code and value of a quotient t by the hardware: cvt.rn.satfinite.<fmt>x2.f32, and back by cvt.rn.f16x2.<fmt>x2
// (exact: every value of the four formats is a float16).  fmt is uniform, so the switch does not diverge.
__device__ __forceinline__ unsigned int fp_code_hw(int fmt, float t, float& value) {
  unsigned short h;
  unsigned int v;
  switch (fmt) {
    case kFmtE4M3:
      asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %1;" : "=h"(h) : "f"(t));
      asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(v) : "h"(h));
      break;
    case kFmtE5M2:
      asm("cvt.rn.satfinite.e5m2x2.f32 %0, %1, %1;" : "=h"(h) : "f"(t));
      asm("cvt.rn.f16x2.e5m2x2 %0, %1;" : "=r"(v) : "h"(h));
      break;
    case kFmtE3M2:
      asm("cvt.rn.satfinite.e3m2x2.f32 %0, %1, %1;" : "=h"(h) : "f"(t));
      asm("cvt.rn.f16x2.e3m2x2 %0, %1;" : "=r"(v) : "h"(h));
      break;
    default:   // kFmtE2M3
      asm("cvt.rn.satfinite.e2m3x2.f32 %0, %1, %1;" : "=h"(h) : "f"(t));
      asm("cvt.rn.f16x2.e2m3x2 %0, %1;" : "=r"(v) : "h"(h));
      break;
  }
  asm("cvt.f32.f16 %0, %1;" : "=f"(value) : "h"((unsigned short)(v & 0xffffu)));
  return (unsigned int)h & 0xffu;   // FP6: the 6-bit code in the low bits of its byte, the two above it zero
}
#endif

// code of a quotient t: the hardware conversion on the device, fp_round_sw on the host
ADMMQ_HD unsigned int fp_code(int fmt, float t) {
#if defined(__CUDA_ARCH__)
  float value;
  return fp_code_hw(fmt, t, value);
#else
  return fp_round_sw(fmt, t);
#endif
}

ADMMQ_HD float fp_scale_of(float clip, int fmt) { return div_rn(clip, fp_format(fmt).max); }

// the element step of the definition: code and value of x on the grid of scale s (exact division).  The code is kept
// as the signed value of its byte, so that the int8 store of the kernels writes the byte.  The quotient is clamped to
// +-max first: for a finite or infinite t that is what the saturating conversion does anyway, and a NaN quotient becomes
// -max, the level the integer grid's clamp gives it (code_exact).  A NaN that reaches the element step without making
// the abs-max NaN (a NaN in the loop's input H does) so ends up in the same places on every grid, and the conversion of
// a NaN, NaN for FP8 and some finite code for FP6, decides nothing.
ADMMQ_HD float fp_quantize(float x, float scale, int fmt, float& code) {
  const float max = fp_format(fmt).max;
  const float t = fminf(fmaxf(div_rn(x, scale), -max), max);
#if defined(__CUDA_ARCH__)
  float level;
  const unsigned int c = fp_code_hw(fmt, t, level);
#else
  const unsigned int c = fp_round_sw(fmt, t);
  const float level = fp_value(fmt, c);
#endif
  code = (float)(int)(signed char)c;
  return mul_rn(level, scale);
}
ADMMQ_HD float fp_dev(float x, float scale, int fmt) {
  float code;
  return sub_rn(x, fp_quantize(x, scale, fmt, code));
}

// the 2 top + 1 distinct values in ascending order, j = 0 .. 2 top (j = top is +0), and the code of each
ADMMQ_HD unsigned int fp_grid_code(int fmt, int j) {
  const FpFormat f = fp_format(fmt);
  return j < f.top ? (1u << (f.bits - 1)) | (unsigned int)(f.top - j) : (unsigned int)(j - f.top);
}
ADMMQ_HD float fp_grid_level(int fmt, int j) { return fp_value(fmt, fp_grid_code(fmt, j)); }

// threshold j (j = 0 .. 2 top - 1) separates grid values j and j + 1, exactly as for E2M1 (e2m1_threshold_mid): the
// boundary b is their midpoint, exact in float32 (at most 3 mantissa bits); rounding reaches value j + 1 from y* = b
// when the tie goes up (value j + 1 has the even mantissa, also across a binade, and 0 against the smallest
// subnormal), else from the next float above b.
ADMMQ_HD ThresholdMid fp_threshold_mid(int fmt, int j) {
  const float b = mul_rn(0.5f, add_rn(fp_grid_level(fmt, j), fp_grid_level(fmt, j + 1)));
  const bool tie_up = (fp_grid_code(fmt, j + 1) & 1u) == 0u;
  const float ystar = tie_up ? b : ordered_float(ordered_key(b) + 1u);
  const float pred = ordered_float(ordered_key(ystar) - 1u);
  ThresholdMid m;
  m.mid = 0.5 * ((double)pred + (double)ystar);
  m.odd = (f32_bits(ystar) & 1u) != 0u;
  return m;
}
ADMMQ_HD float fp_threshold(float scale, int fmt, int j) {
  const ThresholdMid m = fp_threshold_mid(fmt, j);
  return code_threshold_from_mid(scale, m.mid, m.odd);
}
// the same threshold by stepping through neighbouring floats with the exact division (reference of the definition;
// used by the host tests)
ADMMQ_HD bool fp_reaches(float x, float scale, int fmt, float level) {
  return fp_value(fmt, fp_code(fmt, div_rn(x, scale))) >= level;
}
ADMMQ_HD float fp_threshold_search(float scale, int fmt, int j) {
  const float target = fp_grid_level(fmt, j + 1);
  const float b = mul_rn(0.5f, add_rn(fp_grid_level(fmt, j), target));
  unsigned int key = ordered_key(mul_rn(b, scale));
  if (fp_reaches(ordered_float(key), scale, fmt, target)) {
    for (int it = 0; it < 64 && fp_reaches(ordered_float(key - 1u), scale, fmt, target); ++it) --key;
  } else {
    for (int it = 0; it < 64; ++it) {
      ++key;
      if (fp_reaches(ordered_float(key), scale, fmt, target)) break;
    }
  }
  return ordered_float(key);
}

// --- the grid of a clip search, a compile-time choice: the integer grid of quantize_tensor_mse, E2M1, or the FP8 / FP6
// grids (the format in Levels::fmt).  Threshold j separates grid levels j and j + 1; the last level closes the sum by
// parts.
// The parameter is an int so that false / true still name the integer and the E2M1 grid.
enum Grid : int { kGridInt = 0, kGridE2M1 = 1, kGridFP = 2 };
template <int G> struct SearchGrid;
template <> struct SearchGrid<kGridInt> {
  static ADMMQ_HD float scale(float clip, const Levels& L) { return scale_of(clip, L); }
  static ADMMQ_HD int thresholds(int bits, const Levels&) { return (1 << bits) - 1; }
  static ADMMQ_HD ThresholdMid mid(int j, const Levels& L) { return threshold_mid(L.lo + (float)j); }
  static ADMMQ_HD float threshold(float scale, int j, const Levels& L) { return code_threshold(scale, L.lo + (float)j); }
  static ADMMQ_HD double term(float scale, int j, const Levels& L, long long count, long long psum, double xunit) {
    return threshold_term(scale, L.lo + (float)j, count, psum, xunit);
  }
  static ADMMQ_HD float top(const Levels& L) { return L.hi; }
  static ADMMQ_HD float dev(float x, float scale, const Levels& L) { return dev_exact(x, scale, L); }
};
template <> struct SearchGrid<kGridE2M1> {
  static ADMMQ_HD float scale(float clip, const Levels&) { return e2m1_scale_of(clip); }
  static ADMMQ_HD int thresholds(int, const Levels&) { return kE2M1Thresholds; }
  static ADMMQ_HD ThresholdMid mid(int j, const Levels&) { return e2m1_threshold_mid(j); }
  static ADMMQ_HD float threshold(float scale, int j, const Levels&) { return e2m1_threshold(scale, j); }
  static ADMMQ_HD double term(float scale, int j, const Levels&, long long count, long long psum, double xunit) {
    return threshold_term(scale, e2m1_grid_level(j), e2m1_grid_level(j + 1), count, psum, xunit);
  }
  static ADMMQ_HD float top(const Levels&) { return kE2M1Max; }
  static ADMMQ_HD float dev(float x, float scale, const Levels&) { return e2m1_dev(x, scale); }
};
template <> struct SearchGrid<kGridFP> {
  static ADMMQ_HD float scale(float clip, const Levels& L) { return fp_scale_of(clip, L.fmt); }
  static ADMMQ_HD int thresholds(int, const Levels& L) { return fp_thresholds(L.fmt); }
  static ADMMQ_HD ThresholdMid mid(int j, const Levels& L) { return fp_threshold_mid(L.fmt, j); }
  static ADMMQ_HD float threshold(float scale, int j, const Levels& L) { return fp_threshold(scale, L.fmt, j); }
  static ADMMQ_HD double term(float scale, int j, const Levels& L, long long count, long long psum, double xunit) {
    return threshold_term(scale, fp_grid_level(L.fmt, j), fp_grid_level(L.fmt, j + 1), count, psum, xunit);
  }
  static ADMMQ_HD float top(const Levels& L) { return fp_format(L.fmt).max; }
  static ADMMQ_HD float dev(float x, float scale, const Levels& L) { return fp_dev(x, scale, L.fmt); }
};

// --- the other tensor_* schemes ---------------------------------------------------------
struct QParams {
  int scheme;   // ADMMQ_Q_*
  float scale;  // mse/symmetric/affine: grid scale; minmax: (max - min)
  float aux;    // affine: zero point; minmax: min
  float n;      // minmax: 2^bits - 1
  int bits;
};

// min_max_quantize, source/quantization.py:48-66
ADMMQ_HD float minmax_value(float x, const QParams& p, float& level) {
  if (p.bits == 1) {
    const float sgn = (x > 0.0f ? 1.0f : 0.0f) - (x < 0.0f ? 1.0f : 0.0f);  // torch.sign = (0<x)-(x<0)
    level = sgn;
    return sub_rn(sgn, 1.0f);
  }
  const float unit = div_rn(sub_rn(x, p.aux), p.scale);
  const float k = floorf(add_rn(mul_rn(unit, p.n), 0.5f));
  level = k;
  return add_rn(div_rn(mul_rn(k, p.scale), p.n), p.aux);
}

// tensor_affine, source/quantization.py:97-106
ADMMQ_HD float affine_value(float x, const QParams& p, const Levels& L, float& code) {
  float k = add_rn(rint_rn(div_rn(x, p.scale)), p.aux);
  k = add_rn(fminf(fmaxf(k, L.lo), L.hi), 0.0f);  // `.to(int)` (:105) has no negative zero
  code = k;
  return mul_rn(sub_rn(k, p.aux), p.scale);
}

// zero point of tensor_affine (:102-103): clamp(int(-q - int(tmin/scale)), -q, q-1), `.int()` truncates
ADMMQ_HD float affine_zero_point(float tmin, float scale, const Levels& L) {
  const float t = truncf(div_rn(tmin, scale));
  float zp = truncf(sub_rn(L.lo, t));
  zp = fminf(fmaxf(zp, L.lo), L.hi);
  return zp;
}

}  // namespace admmq
