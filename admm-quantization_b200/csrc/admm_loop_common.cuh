// admm_loop_common.cuh - the pieces of the ADMM inner loop (source/admm.py:55-65) that the loop kernels share.  The
// shared-memory kernels (admm_loop_resident.cuh, admm_loop_cluster.cuh, admm_loop_tap.cuh) take all of them: report
// bookkeeping, projection parameters, clip search, P3 element step and residual sums.  The general kernel
// (admm_loop.cu) takes the CTA sum and the candidate scale; its report and projection code stay inline, where moving
// them changed its register allocation.  The parity rules of the small kernels live here once: the NaN semantics of a
// degenerate range, the order of the fixed-point sums, the float32 residual sums flushed every 16 elements.
#pragma once
#include "search.cuh"

namespace admmq {

constexpr int kResBins = 2048;   // linear bins of the shared-memory clip search over [-absmax, absmax]

__device__ __forceinline__ int res_bin_of(float x, float bmul) {
  const float t = fma_rn(x, bmul, 12582912.0f + (float)(kResBins / 2));
  const int b = (int)__float_as_uint(t) - 0x4B400000;
  return min(max(b, 0), kResBins - 1);
}

// ---- report: admmq_loop_report of one call, filled identically by every thread; `writer` names the one that stores it
struct LoopReport {
  admmq_loop_report rep;
  unsigned long long t_begin, t_mark;
  // false (and the report written) when the ridge inverse failed: the loop then touches nothing
  __device__ __forceinline__ bool begin(const float* rho, const int* inv_status, admmq_loop_report* out, bool writer) {
    rep.iterations = 0;
    rep.status = 0;
    rep.rho = *rho;
    rep.scale = 0.0f;
    rep.r = 0.0f;
    rep.s = 0.0f;
    rep.best_index = -1;
    rep.absmax = 0.0f;
    rep.phase_ns[0] = rep.phase_ns[1] = rep.phase_ns[2] = rep.phase_ns[3] = 0ull;
    if (inv_status != nullptr && *inv_status != 0) {
      rep.status = *inv_status;
      if (writer) *out = rep;
      return false;
    }
    return true;
  }
  __device__ __forceinline__ void start() { t_begin = t_mark = global_ns(); }
  __device__ __forceinline__ void lap(int phase) {
    const unsigned long long now = global_ns();
    rep.phase_ns[phase] += now - t_mark;
    t_mark = now;
  }
  // a degenerate range: the reference would carry NaN through every remaining iteration
  __device__ __forceinline__ void nonfinite() {
    rep.status |= ADMMQ_ST_NONFINITE;
    rep.r = __int_as_float(0x7fc00000);
    rep.s = __int_as_float(0x7fc00000);
  }
  __device__ __forceinline__ void finish(admmq_loop_report* out, bool writer) {
    rep.phase_ns[3] = global_ns() - t_begin;
    if (writer) *out = rep;
  }
};

// ---- projection parameters of an iteration from the min / max keys of V (G: the grid of the instantiation)
struct Projection {
  float tmin, tmax, absmax;
  QParams qp;       // scale still 0 for the clip search: it comes from the argmin (clip_scale)
  bool degenerate;  // no finite, non-zero range: H becomes NaN (every scheme follows the reference's NaN propagation)
};
template <Grid G>
__device__ __forceinline__ Projection projection_from_keys(unsigned int kmax, unsigned int kinv, int scheme, int bits,
                                                           const Levels& L) {
  Projection pj;
  pj.tmax = key_float(kmax);
  pj.tmin = key_float(~kinv);
  pj.absmax = fmaxf(fabsf(pj.tmin), fabsf(pj.tmax));
  if (pj.tmin != pj.tmin || pj.tmax != pj.tmax) pj.absmax = __int_as_float(0x7fc00000);
  if (clip_search_scheme<G>(scheme)) {
    pj.qp.scheme = scheme;
    pj.qp.bits = bits;
    pj.qp.aux = 0.0f;
    pj.qp.n = 0.0f;
    pj.qp.scale = 0.0f;
    pj.degenerate = !(pj.absmax > 0.0f) || isinf(pj.absmax);
  } else {
    pj.degenerate = (pj.absmax != pj.absmax) || isinf(pj.absmax);
    pj.qp = params_from_minmax(scheme, bits, pj.tmin, pj.tmax, L);
  }
  return pj;
}

// ---- sum over the CTA of four per-thread doubles (fixed order), result valid in every thread; sm.red is [4][kWarps]
template <class Smem>
__device__ __forceinline__ void cta_sum4(double v[4], Smem& sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < 4; ++q) v[q] = warp_sum(v[q]);
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int q = 0; q < 4; ++q) sm.red[q][warp] = v[q];
  }
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) s += sm.red[q][w];
    v[q] = s;
  }
}

// r and s of the cluster kernels from every CTA's residual slot (rank order), and the exit test r < eps && s < eps
// (:62-65); every CTA evaluates it identically
__device__ __forceinline__ bool cluster_converged(const double (*slots)[4], int C, float eps, admmq_loop_report& rep) {
  double tot[4] = {0.0, 0.0, 0.0, 0.0};
  for (int rk = 0; rk < C; ++rk)
#pragma unroll
    for (int q = 0; q < 4; ++q) tot[q] += slots[rk][q];
  rep.r = div_rn((float)tot[0], (float)tot[1]);
  rep.s = div_rn((float)tot[2], (float)tot[3]);
  return rep.r < eps && rep.s < eps;
}

// ---- P3 of the shared-memory kernels, one element: H = Q(V), U += H - H_ls, next RHS, residual sums
__device__ __forceinline__ float rhs_of(float f, float rho, float h, float u) {   // F + rho (H + U)   (:56)
  return add_rn(f, mul_rn(rho, add_rn(h, u)));
}

// the four residual sums: float32 over 16 elements at a time, float64 beyond
struct ResidualSums {
  float f0 = 0.0f, f1 = 0.0f, f2 = 0.0f, f3 = 0.0f;
  double sums[4] = {0.0, 0.0, 0.0, 0.0};
  int cnt = 0;
  __device__ __forceinline__ void flush() {
    sums[0] += (double)f0;
    sums[1] += (double)f1;
    sums[2] += (double)f2;
    sums[3] += (double)f3;
  }
  // sums[q] for a run-time q without a dynamic index (which would move the whole accumulator to local memory)
  __device__ __forceinline__ double total(int q) const {
    return q == 0 ? sums[0] : q == 1 ? sums[1] : q == 2 ? sums[2] : sums[3];
  }
  __device__ __forceinline__ void add(float d1, float hq, float d2, float un) {
    f0 = fmaf(d1, d1, f0);  // sum (H - H_ls)^2     (:62)
    f1 = fmaf(hq, hq, f1);  // sum H^2
    f2 = fmaf(d2, d2, f2);  // sum (H - H_prev)^2   (:63)
    f3 = fmaf(un, un, f3);  // sum U^2
    if (++cnt == 16) {
      flush();
      f0 = f1 = f2 = f3 = 0.0f;
      cnt = 0;
    }
  }
};

struct ElementStep {
  float hq, un, code, rhs_next;
};
template <Grid G>
__device__ __forceinline__ ElementStep p3_element(float hls, float u, float hp, float fv, float rho, const QParams& qp,
                                                  const Levels& L, bool degenerate, ResidualSums& res) {
  ElementStep o;
  const float v = sub_rn(hls, u);
  o.code = 0.0f;
  if constexpr (G == kGridE2M1)
    o.hq = degenerate ? __int_as_float(0x7fc00000) : e2m1_quantize(v, qp.scale, o.code);
  else if constexpr (G == kGridFP)
    o.hq = degenerate ? __int_as_float(0x7fc00000) : fp_quantize(v, qp.scale, L.fmt, o.code);
  else
    o.hq = degenerate ? __int_as_float(0x7fc00000) : quantize_value(v, qp, L, o.code);   // H = Q(H_ls - U)   (:59)
  const float d1 = sub_rn(o.hq, hls);
  o.un = add_rn(u, d1);                                                                // U += H - H_ls     (:60)
  res.add(d1, o.hq, sub_rn(o.hq, hp), o.un);
  o.rhs_next = rhs_of(fv, rho, o.hq, o.un);
  return o;
}

// ---- clip search of the shared-memory kernels: fixed-point sums of squared errors of the n elements value(0 .. n-1)
// for the candidates [c0, c1) into sm.acc, in the threshold form (numerics.cuh; histogram + counting sort into sm.X,
// one thread per (candidate, threshold) pair) or, for abs-max outside [2^-40, 2^40], the plain evaluation of every
// (element, candidate) pair.  The per-candidate sums are integers over a fixed element order: the same bits whatever
// the thread that adds a term.
template <Grid G, class Smem, class Value>
__device__ inline void smem_candidate_sums(Smem& sm, int n, Value value, float absmax, int Nc, int c0, int c1,
                                           const Levels L, int bits) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const ClipGrid g = make_clip_grid(absmax, Nc);
  const double unit_inv = fixed_point_unit_inv((double)n, absmax);
  if (!binned_range_ok(absmax)) {
    for (int c = c0 + tid; c < c1; c += kThreads) {
      const float s = SearchGrid<G>::scale(clip_candidate(g, c), L);
      double tot = 0.0;
      for (int e = 0; e < n; ++e) {
        const float d = SearchGrid<G>::dev(value(e), s, L);
        tot += (double)mul_rn(d, d);
      }
      sm.acc[c] = (unsigned long long)__double2ll_rn(tot * unit_inv);
    }
    __syncthreads();
    return;
  }
  const FixX fx = make_fix_x(absmax);
  const float bmul = div_rn((float)(kResBins / 2), absmax);
  const int nthr = SearchGrid<G>::thresholds(bits, L);
  const int ncand = c1 - c0;
  const int npairs = ncand * nthr;
  for (int c = c0 + tid; c < c1; c += kThreads) {
    sm.scale[c] = SearchGrid<G>::scale(clip_candidate(g, c), L);
    sm.acc[c] = 0ull;
  }
  float* sorted = sm.X;
  for (int b = tid; b < kResBins; b += kThreads) {
    sm.cnt[b] = 0u;
    sm.slo[b] = 0u;
    sm.shi[b] = 0u;
  }
  __syncthreads();
  // pass 1: histogram (count + 64-bit fixed-point sum per bin) and the sum of squares
  double x2 = 0.0;
  for (int e = tid; e < n; e += kThreads) {
    const float x = value(e);
    const int b = res_bin_of(x, bmul);
    atomicAdd(&sm.cnt[b], 1u);
    const long long f = fix_x(x, fx);
    const unsigned int lo = (unsigned int)f, hi = (unsigned int)((unsigned long long)f >> 32);
    const unsigned int old = atomicAdd(&sm.slo[b], lo);
    atomicAdd(&sm.shi[b], hi + ((old + lo < old) ? 1u : 0u));
    const double xd = (double)x;
    x2 = fma(xd, xd, x2);
  }
  __syncthreads();
  // exclusive scan over the bins: thread t owns kResBins / kThreads consecutive bins
  {
    constexpr int kPer = kResBins / kThreads;
    const int b0 = tid * kPer;
    unsigned int c[kPer], lo[kPer], hi[kPer];
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      c[i] = sm.cnt[b0 + i];
      lo[i] = sm.slo[b0 + i];
      hi[i] = sm.shi[b0 + i];
    }
    unsigned int ct = 0u;
    unsigned long long st = 0ull;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      ct += c[i];
      st += ((unsigned long long)hi[i] << 32) | lo[i];
    }
    unsigned int ci = ct;
    unsigned long long si = st;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int nc = __shfl_up_sync(0xffffffffu, ci, o);
      const unsigned long long ns = __shfl_up_sync(0xffffffffu, si, o);
      if (lane >= o) {
        ci += nc;
        si += ns;
      }
    }
    if (lane == 31) {
      sm.wcnt[warp] = ci;
      sm.wsum[warp] = si;
    }
    __syncthreads();
    unsigned int rc = ci - ct;
    unsigned long long rs = si - st;
    for (int w = 0; w < warp; ++w) {
      rc += sm.wcnt[w];
      rs += sm.wsum[w];
    }
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      const unsigned int cc = c[i];
      const unsigned long long ss = ((unsigned long long)hi[i] << 32) | lo[i];
      sm.cnt[b0 + i] = rc;
      sm.slo[b0 + i] = (unsigned int)rs;
      sm.shi[b0 + i] = (unsigned int)(rs >> 32);
      rc += cc;
      rs += ss;
    }
  }
  __syncthreads();
  // pass 2: counting-sort scatter into X (cnt[b] runs from the start to the end of bin b)
  for (int e = tid; e < n; e += kThreads) {
    const float x = value(e);
    const unsigned int pos = atomicAdd(&sm.cnt[res_bin_of(x, bmul)], 1u);
    sorted[pos] = x;
  }
  __syncthreads();
  // pass 3: one (candidate, threshold) pair per thread, candidates [c0, c1) only
  {
    long long ptot = 0ll;
    for (int w = 0; w < kWarps; ++w) ptot += (long long)sm.wsum[w];
    for (int p = tid; p < npairs; p += kThreads) {
      const int j = p / ncand, c = c0 + (p - j * ncand);
      const float s = sm.scale[c];
      const float theta = SearchGrid<G>::threshold(s, j, L);
      const int b = res_bin_of(theta, bmul);
      const unsigned int beg = b ? sm.cnt[b - 1] : 0u, end = sm.cnt[b];
      long long ps = (long long)(((unsigned long long)sm.shi[b] << 32) | sm.slo[b]);
      long long cn = (long long)beg;
      for (unsigned int i = beg; i < end; ++i) {
        const float x = sorted[i];
        if (x < theta) {
          ++cn;
          ps += fix_x(x, fx);
        }
      }
      double term = SearchGrid<G>::term(s, j, L, cn, ps, fx.unit);
      if (j == nthr - 1) term += closing_term(s, SearchGrid<G>::top(L), (long long)n, ptot, fx.unit);
      atomicAdd(&sm.acc[c], (unsigned long long)__double2ll_rn(term * unit_inv));
    }
  }
  // sum of squares, fixed order
  x2 = warp_sum(x2);
  __syncthreads();
  if (lane == 0) sm.red[0][warp] = x2;
  __syncthreads();
  double tot = 0.0;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) tot += sm.red[0][w];
  const long long x2f = __double2ll_rn(tot * unit_inv);
  for (int c = c0 + tid; c < c1; c += kThreads) {
    const long long f = (long long)sm.acc[c] + x2f;
    sm.acc[c] = (unsigned long long)max(f, 0ll);
  }
  __syncthreads();
}

}  // namespace admmq
