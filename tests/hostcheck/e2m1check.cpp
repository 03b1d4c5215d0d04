// e2m1check.cpp - the E2M1 grid of csrc/numerics.cuh (tensor_mseminmax_e2m1) compiled for the HOST, for the CPU part of
// tests/test_e2m1.py: software rounding, closed-form thresholds, threshold-form and direct candidate sums.
// TEST INFRASTRUCTURE: never linked into libadmmq.so.
// Build: g++ -O2 -ffp-contract=off -shared -fPIC (tests/test_e2m1.py does it).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <vector>
#include "../../admm-quantization_b200/csrc/numerics.cuh"

using namespace admmq;

extern "C" {

void hc_e2m1_round(const float* t, long long n, signed char* codes) {
  for (long long i = 0; i < n; ++i) codes[i] = (signed char)e2m1_round_sw(t[i]);
}

// e2m1_value of every code against the level table; returns the number of mismatches (bitwise, so -0 counts)
int hc_e2m1_value_mismatches(float* values) {
  int bad = 0;
  for (unsigned int c = 0; c < 16; ++c) {
    values[c] = e2m1_value(c);
    const float want = (c & 8u) ? -kE2M1Magnitude[c & 7u] : kE2M1Magnitude[c & 7u];
    if (f32_bits(values[c]) != f32_bits(want)) ++bad;
  }
  return bad;
}

// closed-form thresholds of one scale: theta[j] (j = 0 .. 13) and the number of violations of the definition (theta
// reaches level j + 1, its predecessor does not, theta equals the neighbour-float search)
int hc_e2m1_thresholds(float scale, float* theta) {
  int bad = 0;
  for (int j = 0; j < kE2M1Thresholds; ++j) {
    theta[j] = e2m1_threshold(scale, j);
    const float target = e2m1_grid_level(j + 1);
    const float below = ordered_float(ordered_key(theta[j]) - 1u);
    if (!e2m1_reaches(theta[j], scale, target)) ++bad;
    if (e2m1_reaches(below, scale, target)) ++bad;
    if (theta[j] != e2m1_threshold_search(scale, j)) ++bad;
  }
  return bad;
}

void hc_e2m1_scales(float absmax, int nc, float* scale) {
  const Levels L = make_levels(4);
  const ClipGrid g = make_clip_grid(absmax, nc);
  for (int c = 0; c < nc; ++c) scale[c] = SearchGrid<true>::scale(clip_candidate(g, c), L);
}

// per-candidate sums on the E2M1 grid as float64, in the two forms the kernels use:
//   direct      every element with the exact division, the group recipe of numerics.cuh (groups of 8, float32 over a
//               64-element block, float64 across blocks), fixed point
//   thresholds  exact thresholds, counts and fixed-point prefix sums below each (from a sorted copy), summation by parts
// and the argmin of the threshold form.
void hc_e2m1_sums(const float* x, long long n, float absmax, int nc, double* direct, double* thresholds, int* best) {
  const Levels L = make_levels(4);
  using G = SearchGrid<true>;
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
    for (int j = 0; j < kE2M1Thresholds; ++j) {
      const float theta = G::threshold(s, j, L);
      const long long cnt = std::lower_bound(xs.begin(), xs.end(), theta) - xs.begin();  // #{x < theta}
      double term = G::term(s, j, L, cnt, pre[cnt], fx.unit);
      if (j == kE2M1Thresholds - 1) term += closing_term(s, G::top(L), n, pre[n], fx.unit);
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
