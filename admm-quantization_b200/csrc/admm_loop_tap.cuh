// admm_loop_tap.cuh - the ADMM inner loop (source/admm.py:55-65) for the TAP FACTOR of a wide convolution: few rows
// (the 3 x 3 = 9 kernel taps, I <= 9) and a large rank (R = 278 ... 1365), on ONE THREAD-BLOCK CLUSTER of 8 CTAs.
//
// In the general kernel (admm_loop.cu) such a factor is pure latency: ~10 k elements spread over the layer's 30+ CTAs
// cost 27 us per iteration - three device-wide barriers, a few hundred elements per CTA, every CTA repeating the 3000
// thresholds of the clip search.  Here the COLUMNS of the factor and the CANDIDATES of the clip search are split over
// the CTAs of a cluster (admm_loop_cluster.cuh splits rows; with 9 rows that would leave CTAs idle and make every CTA
// stream the whole inverse):
//   P1  every CTA holds the whole right-hand side (I x Rp floats) in shared memory and forms H_ls = RHS . Minv for ITS
//       column strip: thread (column group, k-slice) accumulates 4 columns x I rows over its k-slice with float32 FMAs,
//       rows of Minv read as float4 from L2 (the strip of the inverse, 0.65 MB at R = 1141, is the only global traffic
//       of the iteration); k-slices summed in fixed order; V = H_ls - U and the min / max keys go to EVERY CTA's shared
//       memory                                                              -- cluster barrier 1
//   P2  every CTA histograms and sorts ALL elements (replicated) and evaluates the thresholds of ITS candidates only;
//       a candidate's sum is broadcast                                      -- cluster barrier 2
//   P3  argmin, H = Q(V), U += H - H_ls, residual sums for the own columns; the new right-hand side of the own columns
//       and the residual partial sums go to every CTA                       -- cluster barrier 3, exit test
// Same float32 recipe as the general kernel's column-strip product up to the order of the k-slices.
#pragma once
#include <cstddef>
#include "admm_loop_common.cuh"
#include "admm_loop_cluster.cuh"

namespace admmq {

constexpr int kTapMaxElems = 12288;   // I * Rp (right-hand side, V, sorted elements: 48 KB each)
constexpr int kTapMaxRows = 9;      // the 3 x 3 taps (the k-slice scratch of P1 is sized for 9 rows x 512 threads)
constexpr int kTapMaxOwn = 3072;      // I * (columns of one CTA)
constexpr int kTapCtas = 8;

struct __align__(16) TapSmem {
  float rhs[kTapMaxElems];      // the whole right-hand side, row pitch Rp (pad columns zero)
  float Vall[kTapMaxElems];     // all elements of V, dense (row pitch R), written by every CTA of the cluster
  float X[kTapMaxElems];        // elements grouped by bin during P2; k-slice partial sums during P1 (with cnt .. shi)
  unsigned int cnt[kResBins];
  unsigned int slo[kResBins];
  unsigned int shi[kResBins];
  float U[kTapMaxOwn];          // own columns: [row][own column]
  float Hls[kTapMaxOwn];
  unsigned long long acc[kMaxCandidates];
  unsigned long long cand[kMaxCandidates];
  float scale[kMaxCandidates];
  double slots[kTapCtas][4];
  unsigned int keys[kTapCtas][2];
  unsigned long long wsum[kWarps];
  unsigned int wcnt[kWarps];
  unsigned int wkey[2][kWarps];
  double red[4][kWarps];
  unsigned long long best[kWarps];
};
static_assert(sizeof(TapSmem) <= 227 * 1024, "tap-factor loop state must fit the shared memory of one SM");
// the k-slice partial sums of P1 (kThreads x MI x 4 floats) live in X + cnt + slo + shi, which are dead during P1
static_assert((size_t)kThreads * kTapMaxRows * 4 * sizeof(float) <= sizeof(float) * kTapMaxElems + 3 * sizeof(unsigned int) * kResBins,
              "P1 scratch must fit the arrays it aliases");
static_assert(offsetof(TapSmem, cnt) == offsetof(TapSmem, X) + sizeof(float) * kTapMaxElems &&
              offsetof(TapSmem, shi) == offsetof(TapSmem, cnt) + 2 * sizeof(unsigned int) * kResBins, "X, cnt, slo, shi are contiguous");

template <int MI, Grid G>   // G: the grid of the clip search (numerics.cuh SearchGrid)
__global__ void __launch_bounds__(kThreads, 1) k_admm_loop_tap(const ResidentParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TapSmem& sm = *reinterpret_cast<TapSmem*>(smem_raw);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int I = p.I, R = p.R, Rp = p.Rp, n = I * R;
  const int rank = (int)cl_rank(), C = (int)cl_size();
  LoopReport rb;
  admmq_loop_report& rep = rb.rep;
  // inv_status is uniform over the cluster: nobody reaches a barrier
  if (!rb.begin(p.rho, p.inv_status, p.report, rank == 0 && t == 0)) return;
  rb.start();
  const float rho = rep.rho;
  const Levels L = make_levels(p.bits, G == kGridFP ? p.scheme : 0);
  // own columns [n0, n1) (a multiple of four per CTA) and own candidates [c0, c1)
  const int cps = ((R + C - 1) / C + 3) / 4 * 4;
  const int n0 = min(R, rank * cps), n1 = min(R, n0 + cps), w = n1 - n0;
  const int own = I * w;
  const int cand_per = (p.Nc + C - 1) / C;
  const int c0 = min(p.Nc, rank * cand_per), c1 = min(p.Nc, c0 + cand_per);
  // ---- the whole right-hand side F + rho (H + U) for the first iteration (:56), own U
  for (int e = t; e < I * Rp; e += kThreads) {
    const int i = e / Rp, c = e - i * Rp;
    sm.rhs[e] = (c < R) ? rhs_of(p.F[i * R + c], rho, p.H[i * R + c], p.U[i * R + c]) : 0.0f;
  }
  for (int e = t; e < own; e += kThreads) {
    const int i = e / w, c = e - i * w;
    sm.U[e] = p.U[i * R + n0 + c];
  }
  cl_sync();   // every CTA of the cluster is running (remote shared memory may be written from here on)
  float* part = sm.X;   // k-slice partial sums: [thread][MI][4]
  const int cg = (w + 3) >> 2;                 // float4 column groups of the own strip (n0 + 4 cg <= Rp)
  const int ks = cg > 0 ? kThreads / cg : 0;   // k-slices
  const int s_id = cg > 0 ? t / cg : 0, c_id = cg > 0 ? t - s_id * cg : 0;
  int done = 0;
  for (int j = 1; j < p.max_iter; ++j) {  // range(1, max_iter), :55
    // ---------------- P1: H_ls = RHS . Minv for the own column strip
    unsigned int kmax = 0u, kinv = 0u;
    if (cg > 0) {
      float acc[MI][4];
#pragma unroll
      for (int i = 0; i < MI; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0f;
      if (s_id < ks) {
        const float* mp = p.Minv + n0 + 4 * c_id;
        // groups of four consecutive rows of Minv (k = 4 g .. 4 g + 3, g = s, s + ks, ...): the four RHS values of a factor
        // row are one 16-byte shared-memory load for 16 FMAs; two groups in flight
        constexpr int kG = 2;
        const int ngroups = (R + 3) >> 2;
        for (int gq = s_id; gq < ngroups; gq += ks * kG) {
          float4 m[kG][4];
#pragma unroll
          for (int u = 0; u < kG; ++u) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int k = 4 * (gq + u * ks) + q;
              m[u][q] = (k < R) ? __ldg(reinterpret_cast<const float4*>(mp + (size_t)k * Rp)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
#pragma unroll
          for (int u = 0; u < kG; ++u) {
            const int g = gq + u * ks;
            if (g < ngroups) {
#pragma unroll
              for (int i = 0; i < MI; ++i) {
                if (i < I) {
                  const float4 r4 = *reinterpret_cast<const float4*>(&sm.rhs[i * Rp + 4 * g]);
                  const float r[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    acc[i][0] = fmaf(r[q], m[u][q].x, acc[i][0]);
                    acc[i][1] = fmaf(r[q], m[u][q].y, acc[i][1]);
                    acc[i][2] = fmaf(r[q], m[u][q].z, acc[i][2]);
                    acc[i][3] = fmaf(r[q], m[u][q].w, acc[i][3]);
                  }
                }
              }
            }
          }
        }
#pragma unroll
        for (int i = 0; i < MI; ++i)
          *reinterpret_cast<float4*>(&part[(size_t)t * (MI * 4) + i * 4]) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
      }
    }
    __syncthreads();
    for (int o = t; o < own; o += kThreads) {
      const int i = o / w, nn = o - i * w;
      const int cc = nn >> 2, q = nn & 3;
      // fixed order: four interleaved partial sums over the k-slices, then ((h0 + h1) + (h2 + h3))
      float h4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      const float* rp = &part[(size_t)cc * (MI * 4) + i * 4 + q];
      int sl = 0;
      for (; sl + 3 < ks; sl += 4) {
#pragma unroll
        for (int a = 0; a < 4; ++a) h4[a] = add_rn(h4[a], rp[(size_t)((sl + a) * cg) * (MI * 4)]);
      }
      for (; sl < ks; ++sl) h4[sl & 3] = add_rn(h4[sl & 3], rp[(size_t)(sl * cg) * (MI * 4)]);
      const float h = add_rn(add_rn(h4[0], h4[1]), add_rn(h4[2], h4[3]));
      sm.Hls[o] = h;
      const float v = sub_rn(h, sm.U[o]);   // V = H_ls - U (:59)
      const unsigned int key = float_key(v);
      kmax = max(kmax, key);
      kinv = max(kinv, ~key);
      const int e = i * R + n0 + nn;
      for (int rk = 0; rk < C; ++rk) cl_store(cl_map(&sm.Vall[e], (unsigned int)rk), v);
    }
    kmax = warp_max_u32(kmax);
    kinv = warp_max_u32(kinv);
    if (lane == 0) {
      sm.wkey[0][warp] = kmax;
      sm.wkey[1][warp] = kinv;
    }
    __syncthreads();
    if (t < 2 * C) {   // this CTA's keys into slot `rank` of every CTA
      unsigned int k = 0u;
      for (int wq = 0; wq < kWarps; ++wq) k = max(k, sm.wkey[t & 1][wq]);
      cl_store(cl_map(&sm.keys[rank][t & 1], (unsigned int)(t >> 1)), k);
    }
    cl_sync();   // ---- barrier 1: V and the keys are everywhere
    kmax = 0u;
    kinv = 0u;
    for (int rk = 0; rk < C; ++rk) {
      kmax = max(kmax, sm.keys[rk][0]);
      kinv = max(kinv, sm.keys[rk][1]);
    }
    rb.lap(0);
    // ---------------- P2
    const Projection pj = projection_from_keys<G>(kmax, kinv, p.scheme, p.bits, L);
    rep.absmax = pj.absmax;
    rep.iterations = j;
    done = j;
    QParams qp = pj.qp;
    const bool search = clip_search_scheme<G>(p.scheme) && !pj.degenerate;
    if (search) {
      smem_candidate_sums<G>(sm, n, [&](int e) { return sm.Vall[e]; }, pj.absmax, p.Nc, c0, c1, L, p.bits);
      for (int c = c0 + t; c < c1; c += kThreads) {
        const unsigned long long v = sm.acc[c];
        for (int rk = 0; rk < C; ++rk) cl_store(cl_map(&sm.cand[c], (unsigned int)rk), v);
      }
    }
    cl_sync();   // ---- barrier 2: every candidate's sum is everywhere (nobody reads V / the sorted array any more)
    if (search) {
      rep.best_index = cta_best_candidate<false>(sm.cand, p.Nc, pj.absmax, (double)n, sm.best);
      qp.scale = clip_scale<G>(pj.absmax, p.Nc, rep.best_index, L);
    }
    rep.scale = qp.scale;
    rb.lap(1);
    // ---------------- P3: H = Q(V), U += H - H_ls, residual sums, next RHS (to every CTA) - own columns
    ResidualSums res;
    for (int o = t; o < own; o += kThreads) {
      const int i = o / w, nn = o - i * w;
      const int e = i * R + n0 + nn;
      const float hp = p.H[e];
      const float fv = __ldg(p.F + e);
      const ElementStep s = p3_element<G>(sm.Hls[o], sm.U[o], hp, fv, rho, qp, L, pj.degenerate, res);
      p.H[e] = s.hq;
      sm.U[o] = s.un;
      for (int rk = 0; rk < C; ++rk) cl_store(cl_map(&sm.rhs[i * Rp + n0 + nn], (unsigned int)rk), s.rhs_next);
      if (p.codes != nullptr) p.codes[e] = (int8_t)s.code;
    }
    res.flush();
    if (pj.degenerate) {  // uniform
      rb.nonfinite();
      break;
    }
    cta_sum4(res.sums, sm);
    if (t < 4 * C) cl_store(cl_map(&sm.slots[rank][t & 3], (unsigned int)(t >> 2)), res.total(t & 3));
    cl_sync();   // ---- barrier 3: the next right-hand side and the residual sums are everywhere
    const bool converged = cluster_converged(sm.slots, C, p.eps, rep);
    rb.lap(2);
    if (converged) {
      rep.status |= ADMMQ_ST_CONVERGED;
      break;
    }
  }
  cl_sync();   // no CTA leaves while its shared memory may still be written
  rep.iterations = done;
  for (int o = t; o < own; o += kThreads) {
    const int i = o / w, nn = o - i * w;
    p.U[i * R + n0 + nn] = sm.U[o];
  }
  rb.finish(p.report, rank == 0 && t == 0);
}

// Eligible: few rows, everything fits the shared-memory arrays, a budget of at least one cluster - and a rank up to
// kTapMaxRank: the product streams the CTA's strip of the inverse with float32 FMAs, 1.5 MFMA per CTA at R = 1141, which
// eight SMs do slower than the general kernel's thirty-odd.  Measured per iteration (9 x R; cluster of 8 against the
// general kernel on 7 / 33 CTAs): R = 278: 13.0 us against 23.1, R = 566: 19.7 against 28.1 / 26.9, R = 1141: 38.0
// against 49.3 / 28.0.
constexpr int kTapMaxRank = 640;
inline bool tap_cluster_fits(int I, int R, int Rp, int num_attempts, int budget) {
  if (I > kTapMaxRows || R > kTapMaxRank || budget < kTapCtas || num_attempts > kMaxCandidates) return false;
  const int cps = ((R + kTapCtas - 1) / kTapCtas + 3) / 4 * 4;
  return (long long)I * Rp <= kTapMaxElems && (long long)I * cps <= kTapMaxOwn && cps >= 4;
}

}  // namespace admmq
