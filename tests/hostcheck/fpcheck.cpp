// fpcheck.cpp - the FP8 / FP6 grids of csrc/numerics.cuh (tensor_mseminmax_e4m3 / _e5m2 / _e3m2 / _e2m3) compiled for
// the HOST, for the CPU part of tests/test_fp_grids.py: software rounding, values of codes, closed-form thresholds,
// threshold-form and direct candidate sums.  fmt is the scheme id (6 .. 9).
// TEST INFRASTRUCTURE: never linked into libadmmq.so.
// Build: g++ -O2 -ffp-contract=off -shared -fPIC (tests/test_fp_grids.py does it).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <vector>
#include "../../admm-quantization_b200/csrc/numerics.cuh"

using namespace admmq;

extern "C" {

// {bits, ebits, mbits, bias, top, nan_top} and max of a format
void hc_fp_format(int fmt, int* ints, float* max) {
  const FpFormat f = fp_format(fmt);
  ints[0] = f.bits;
  ints[1] = f.ebits;
  ints[2] = f.mbits;
  ints[3] = f.bias;
  ints[4] = f.top;
  ints[5] = f.nan_top ? 1 : 0;
  *max = f.max;
}

void hc_fp_round(int fmt, const float* t, long long n, signed char* codes) {
  for (long long i = 0; i < n; ++i) codes[i] = (signed char)fp_round_sw(fmt, t[i]);
}

// fp_value of `n` codes
void hc_fp_value(int fmt, const int* codes, int n, float* values) {
  for (int i = 0; i < n; ++i) values[i] = fp_value(fmt, (unsigned int)codes[i]);
}

// the ascending grid: levels j = 0 .. 2 top and their codes; returns the number of levels
int hc_fp_grid(int fmt, float* levels, int* codes) {
  const int n = fp_thresholds(fmt) + 1;
  for (int j = 0; j < n; ++j) {
    levels[j] = fp_grid_level(fmt, j);
    codes[j] = (int)fp_grid_code(fmt, j);
  }
  return n;
}

// closed-form thresholds of one scale: theta[j] (j = 0 .. 2 top - 1) and the number of violations of the definition
// (theta reaches level j + 1, its predecessor does not, theta equals the neighbour-float search)
int hc_fp_thresholds(int fmt, float scale, float* theta) {
  int bad = 0;
  for (int j = 0; j < fp_thresholds(fmt); ++j) {
    theta[j] = fp_threshold(scale, fmt, j);
    const float target = fp_grid_level(fmt, j + 1);
    const float below = ordered_float(ordered_key(theta[j]) - 1u);
    if (!fp_reaches(theta[j], scale, fmt, target)) ++bad;
    if (fp_reaches(below, scale, fmt, target)) ++bad;
    if (theta[j] != fp_threshold_search(scale, fmt, j)) ++bad;
  }
  return bad;
}

void hc_fp_scales(int fmt, float absmax, int nc, float* scale) {
  const Levels L = make_levels(fp_format(fmt).bits, fmt);
  const ClipGrid g = make_clip_grid(absmax, nc);
  for (int c = 0; c < nc; ++c) scale[c] = SearchGrid<kGridFP>::scale(clip_candidate(g, c), L);
}

// per-candidate sums on an FP grid as float64, in the two forms the kernels use (as e2m1check.cpp hc_e2m1_sums):
//   direct      every element with the exact division, the group recipe of numerics.cuh, fixed point
//   thresholds  exact thresholds, counts and fixed-point prefix sums below each (from a sorted copy), summation by parts
// and the argmin of the threshold form.
void hc_fp_sums(int fmt, const float* x, long long n, float absmax, int nc, double* direct, double* thresholds, int* best) {
  const Levels L = make_levels(fp_format(fmt).bits, fmt);
  using G = SearchGrid<kGridFP>;
  const int nthr = G::thresholds(fp_format(fmt).bits, L);
  const ClipGrid g = make_clip_grid(absmax, nc);
  const double unit_inv = fixed_point_unit_inv((double)n, absmax), unit = fixed_point_unit((double)n, absmax);
  const FixX fx = make_fix_x(absmax);
  std::vector<float> xs(x, x + n);
  std::sort(xs.begin(), xs.end());
  std::vector<long long> pre(n + 1, 0);
  for (long long i = 0; i < n; ++i) pre[i + 1] = pre[i] + fix_x(xs[i], fx);
  double x2 = 0.0;
  for (long long i = 0; i < n; ++i) x2 += (double)x[i] * (double)x[i];
  const long long x2f = llrint(x2 * unit_inv);
  int arg = 0;
  float best_mse = 0.0f;
  for (int c = 0; c < nc; ++c) {
    const float s = G::scale(clip_candidate(g, c), L);
    double tot = 0.0;
    float block = 0.0f;
    for (long long b = 0; b < n; b += kSumGroup) {
      float d[kSumGroup];
      for (int i = 0; i < kSumGroup; ++i) d[i] = G::dev((b + i < n) ? x[b + i] : 0.0f, s, L);
      block = add_rn(block, group_sum8(d));
      if ((b + kSumGroup) % kSumBlock == 0 || b + kSumGroup >= n) {
        tot += (double)block;
        block = 0.0f;
      }
    }
    direct[c] = (double)llrint(tot * unit_inv) * unit;
    long long acc = 0;
    for (int j = 0; j < nthr; ++j) {
      const float theta = G::threshold(s, j, L);
      const long long cnt = std::lower_bound(xs.begin(), xs.end(), theta) - xs.begin();  // #{x < theta}
      double term = G::term(s, j, L, cnt, pre[cnt], fx.unit);
      if (j == nthr - 1) term += closing_term(s, G::top(L), n, pre[n], fx.unit);
      acc += llrint(term * unit_inv);
    }
    const long long f = std::max(acc + x2f, 0ll);
    thresholds[c] = (double)f * unit;
    const float mse = mse_from_fixed(f, unit, (float)n);
    if (c == 0 || mse < best_mse) {
      best_mse = mse;
      arg = c;
    }
  }
  *best = arg;
}
}
