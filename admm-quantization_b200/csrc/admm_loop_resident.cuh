// admm_loop_resident.cuh - the ADMM inner loop (source/admm.py:55-65) for SMALL factors, run by ONE CTA with the
// loop state resident in shared memory (the 64 x 64 x 3 x 3 convolutions of ResNet-18: I x R = 64 x 134).
//
// The general kernel (admm_loop.cu) spreads a factor over many CTAs and pays three device-wide barriers and several
// L2 round trips per iteration for its scratch arrays; for a factor this small that latency is the whole cost (45 us
// per iteration on one CTA).  Here the scaled dual U, the ridge inverse Minv, H_ls, the next right-hand side and every
// scratch structure of the clip search live in shared memory (~210 KB), the phases are separated by __syncthreads
// only, and global memory is touched once per iteration and element: H (previous value in, new value out) and F.
//   P1  H_ls = RHS . Minv as float32 FMA register tiles (4 x 5 outputs per thread), operands from shared memory
//   P2  clip search in its threshold form (numerics.cuh / search.cuh) on V = H_ls - U, all counters in shared memory
//   P3  argmin, H = Q(V), U += H - H_ls, residual sums, next RHS; exit test r < eps && s < eps
// Results follow the same float32 recipe as the general kernel's parity mode (precision 0) up to the summation order
// of the ridge product.
#pragma once
#include "admm_loop_common.cuh"

namespace admmq {

constexpr int kResMaxElems = 8704;        // I * R  (64 x 136)
constexpr int kResMaxMinv = 136 * 136;    // R * Rp

struct ResidentParams {
  float* H;
  float* U;
  const float* F;
  const float* Minv;  // R x Rp, pad columns zero
  const float* rho;
  const int* inv_status;
  int I, R, Rp;
  int max_iter;
  float eps;
  int bits, scheme, Nc;
  int8_t* codes;
  admmq_loop_report* report;
};

struct __align__(16) ResidentSmem {
  float U[kResMaxElems];
  float Hls[kResMaxElems];
  float X[kResMaxElems];      // RHS during P1, elements grouped by bin during P2
  float Minv[kResMaxMinv];
  unsigned int cnt[kResBins];
  unsigned int slo[kResBins];
  unsigned int shi[kResBins];
  unsigned long long acc[kMaxCandidates];
  float scale[kMaxCandidates];
  unsigned long long wsum[kWarps];
  unsigned int wcnt[kWarps];
  unsigned int wkey[2][kWarps];
  double red[4][kWarps];
  unsigned long long best[kWarps];
};

template <Grid G>   // G: the grid of the clip search (numerics.cuh SearchGrid)
__global__ void __launch_bounds__(kThreads, 1) k_admm_loop_resident(const ResidentParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ResidentSmem& sm = *reinterpret_cast<ResidentSmem*>(smem_raw);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int I = p.I, R = p.R, Rp = p.Rp, n = I * R;
  LoopReport rb;
  admmq_loop_report& rep = rb.rep;
  if (!rb.begin(p.rho, p.inv_status, p.report, t == 0)) return;
  rb.start();
  const float rho = rep.rho;
  const Levels L = make_levels(p.bits, G == kGridFP ? p.scheme : 0);
  // ---- state into shared memory; RHS = F + rho (H + U) for the first iteration (:56)
  for (int e = t; e < R * Rp; e += kThreads) sm.Minv[e] = p.Minv[e];
  for (int e = t; e < n; e += kThreads) {
    const float u = p.U[e];
    sm.U[e] = u;
    sm.X[e] = rhs_of(p.F[e], rho, p.H[e], u);
  }
  __syncthreads();
  // P1 mapping: 4 rows x 5 columns per thread
  const int tiles_n = (R + 4) / 5, tiles_m = (I + 3) / 4;
  for (int j = 1; j < p.max_iter; ++j) {  // range(1, max_iter), :55
    // ---------------- P1: H_ls = RHS . Minv, abs-max of V = H_ls - U
    unsigned int kmax = 0u, kinv = 0u;
    for (int tile = t; tile < tiles_m * tiles_n; tile += kThreads) {
      const int i0 = (tile / tiles_n) * 4, n0 = (tile % tiles_n) * 5;
      float acc[4][5];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 5; ++b) acc[a][b] = 0.0f;
      const float* r0 = sm.X + (size_t)min(i0, I - 1) * R;
      const float* r1 = sm.X + (size_t)min(i0 + 1, I - 1) * R;
      const float* r2 = sm.X + (size_t)min(i0 + 2, I - 1) * R;
      const float* r3 = sm.X + (size_t)min(i0 + 3, I - 1) * R;
      const float* mp = sm.Minv + n0;
#pragma unroll 2
      for (int k = 0; k < R; ++k) {
        const float a0 = r0[k], a1 = r1[k], a2 = r2[k], a3 = r3[k];
        float m[5];
#pragma unroll
        for (int b = 0; b < 5; ++b) m[b] = (n0 + b < Rp) ? mp[(size_t)k * Rp + b] : 0.0f;
#pragma unroll
        for (int b = 0; b < 5; ++b) {
          acc[0][b] = fmaf(a0, m[b], acc[0][b]);
          acc[1][b] = fmaf(a1, m[b], acc[1][b]);
          acc[2][b] = fmaf(a2, m[b], acc[2][b]);
          acc[3][b] = fmaf(a3, m[b], acc[3][b]);
        }
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 5; ++b) {
          const int i = i0 + a, c = n0 + b;
          if (i < I && c < R) {
            const int e = i * R + c;
            sm.Hls[e] = acc[a][b];
            const unsigned int k = float_key(sub_rn(acc[a][b], sm.U[e]));  // V = H_ls - U (:59)
            kmax = max(kmax, k);
            kinv = max(kinv, ~k);
          }
        }
    }
    kmax = warp_max_u32(kmax);
    kinv = warp_max_u32(kinv);
    if (lane == 0) {
      sm.wkey[0][warp] = kmax;
      sm.wkey[1][warp] = kinv;
    }
    __syncthreads();
    kmax = 0u;
    kinv = 0u;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      kmax = max(kmax, sm.wkey[0][w]);
      kinv = max(kinv, sm.wkey[1][w]);
    }
    rb.lap(0);
    // ---------------- P2
    const Projection pj = projection_from_keys<G>(kmax, kinv, p.scheme, p.bits, L);
    rep.absmax = pj.absmax;
    rep.iterations = j;
    QParams qp = pj.qp;
    if (clip_search_scheme<G>(p.scheme) && !pj.degenerate) {
      smem_candidate_sums<G>(sm, n, [&](int e) { return sub_rn(sm.Hls[e], sm.U[e]); }, pj.absmax, p.Nc, 0, p.Nc, L, p.bits);
      rep.best_index = cta_best_candidate<false>(sm.acc, p.Nc, pj.absmax, (double)n, sm.best);
      qp.scale = clip_scale<G>(pj.absmax, p.Nc, rep.best_index, L);
    }
    rep.scale = qp.scale;
    rb.lap(1);
    // ---------------- P3: H = Q(V), U += H - H_ls, residual sums, next RHS
    __syncthreads();  // everyone is done with X as the sorted array
    ResidualSums res;
    for (int e0 = t; e0 < n; e0 += kThreads * 4) {
      float hp[4], fv[4];
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int e = e0 + b * kThreads;
        if (e < n) {
          hp[b] = p.H[e];
          fv[b] = __ldg(p.F + e);
        }
      }
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int e = e0 + b * kThreads;
        if (e < n) {
          const ElementStep o = p3_element<G>(sm.Hls[e], sm.U[e], hp[b], fv[b], rho, qp, L, pj.degenerate, res);
          p.H[e] = o.hq;
          sm.U[e] = o.un;
          sm.X[e] = o.rhs_next;
          if (p.codes != nullptr) p.codes[e] = (int8_t)o.code;
        }
      }
    }
    res.flush();
    if (pj.degenerate) {  // uniform
      rb.nonfinite();
      break;
    }
    cta_sum4(res.sums, sm);  // (contains the barriers that publish U and X for the next iteration)
    rep.r = div_rn((float)res.sums[0], (float)res.sums[1]);
    rep.s = div_rn((float)res.sums[2], (float)res.sums[3]);
    rb.lap(2);
    if (rep.r < p.eps && rep.s < p.eps) {
      rep.status |= ADMMQ_ST_CONVERGED;
      break;
    }
  }
  __syncthreads();
  for (int e = t; e < n; e += kThreads) p.U[e] = sm.U[e];
  rb.finish(p.report, t == 0);
}

inline bool resident_fits(int I, int R, int Rp, int num_attempts) {
  return (long long)I * R <= kResMaxElems && (long long)R * Rp <= kResMaxMinv && num_attempts <= kMaxCandidates;
}

}  // namespace admmq
