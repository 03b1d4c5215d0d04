// admm_loop_cluster.cuh - the ADMM inner loop (source/admm.py:55-65) for SMALL factors on ONE THREAD-BLOCK CLUSTER:
// 2, 4 or 8 CTAs (one per SM) that share the factor through distributed shared memory.
//
// The single-CTA resident kernel (admm_loop_resident.cuh) keeps the whole loop state of a 64 x 134 factor in one SM's
// shared memory but runs every phase on that one SM: 35 us per iteration, of which 15 us are the ridge product out of
// shared memory and 15 us the clip search (8.6 k elements to histogram and sort, 3000 (candidate, threshold) pairs).
// Here the ROWS of the factor are split over the CTAs of a cluster and the CANDIDATES of the clip search as well:
//   P1  every CTA forms H_ls = RHS . Minv for ITS rows (Minv replicated in every CTA's shared memory, 4 rows x 1 column
//       per thread, operands from shared memory, products and sums in float64: with so few rows per CTA the FP64 pipe
//       is not the limit, and H_ls is then the correctly rounded product with the float32 inverse) and V = H_ls - U; it
//       stores its rows of V and its min / max keys into EVERY CTA's shared memory (st.shared::cluster)
//                                                                            -- cluster barrier 1
//   P2  every CTA histograms and counting-sorts ALL elements of V (replicated: 8.6 k elements, ~4 us) and evaluates
//       the thresholds of ITS share of the candidates only (25 of 200 on 8 CTAs); a candidate's sum is complete inside
//       one CTA, which broadcasts it to every CTA                            -- cluster barrier 2
//   P3  argmin, H = Q(V), U += H - H_ls, next RHS and the residual sums for the CTA's own rows; the partial sums go to
//       every CTA.  The exit test r < eps && s < eps of iteration j is evaluated after barrier 1 of iteration j + 1: P1
//       touches neither H, U nor RHS, so the speculative P1 is simply dropped when the test fires - two barriers per
//       iteration instead of three.
// Arithmetic: every output of the ridge product is accumulated over k in ascending order whatever the cluster size, and
// the candidate sums are integers / fixed point over the same element order, so H and U are bit-identical for clusters
// of 2, 4 and 8 CTAs; against the single-CTA kernel (float32 FMAs) they differ by the rounding of the product only
// (tests/test_gpu_parity_r2.py).
#pragma once
#include "admm_loop_common.cuh"
#include "admm_loop_resident.cuh"

namespace admmq {

constexpr int kClMaxOwn = kResMaxElems / 2;   // elements of a CTA's own rows (at least two CTAs share the factor)
constexpr int kClMaxCtas = 8;                 // portable cluster size

struct __align__(16) ClusterSmem {
  float Minv[kResMaxMinv];      // R x Rp, rows R .. Rp-1 zero
  float Vall[kResMaxElems];     // all rows of V = H_ls - U, written by every CTA of the cluster (dense, row pitch R)
  float X[kResMaxElems];        // own rows of RHS as float64 (row pitch Rp) during P1 / P3; all elements grouped by bin during P2
  float U[kClMaxOwn];           // own rows, dense
  float Hls[kClMaxOwn];
  unsigned int cnt[kResBins];
  unsigned int slo[kResBins];
  unsigned int shi[kResBins];
  unsigned long long acc[kMaxCandidates];    // own candidates' fixed-point sums
  unsigned long long cand[kMaxCandidates];   // every candidate's sum (each written by the CTA that owns the candidate)
  float scale[kMaxCandidates];
  double slots[kClMaxCtas][4];               // residual partial sums of every CTA
  unsigned int keys[kClMaxCtas][2];          // min / max keys of every CTA's rows
  unsigned long long wsum[kWarps];
  unsigned int wcnt[kWarps];
  unsigned int wkey[2][kWarps];
  double red[4][kWarps];
  unsigned long long best[kWarps];
};
static_assert(sizeof(ClusterSmem) <= 227 * 1024, "cluster loop state must fit the shared memory of one SM");

__device__ __forceinline__ unsigned int cl_rank() {
  unsigned int r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ unsigned int cl_size() {
  unsigned int r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
// release / acquire at cluster scope: shared-memory stores into other CTAs issued before the barrier are visible after it
__device__ __forceinline__ void cl_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory variable in CTA `rank` of the cluster
__device__ __forceinline__ unsigned int cl_map(const void* p, unsigned int rank) {
  unsigned int local = (unsigned int)__cvta_generic_to_shared(p), remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local), "r"(rank));
  return remote;
}
__device__ __forceinline__ void cl_store(unsigned int addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ void cl_store(unsigned int addr, unsigned int v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void cl_store(unsigned int addr, unsigned long long v) {
  asm volatile("st.shared::cluster.u64 [%0], %1;" ::"r"(addr), "l"(v) : "memory");
}
__device__ __forceinline__ void cl_store(unsigned int addr, double v) {
  asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

template <Grid G>   // G: the grid of the clip search (numerics.cuh SearchGrid)
__global__ void __launch_bounds__(kThreads, 1) k_admm_loop_cluster(const ResidentParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ClusterSmem& sm = *reinterpret_cast<ClusterSmem*>(smem_raw);
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
  // own rows [i0, i1) and own candidates [c0, c1)
  const int rows_per = (I + C - 1) / C;
  const int i0 = min(I, rank * rows_per), i1 = min(I, i0 + rows_per);
  const int own_rows = i1 - i0, own = own_rows * R;
  const int e_base = i0 * R;                 // first own element in the dense factor
  const int cand_per = (p.Nc + C - 1) / C;
  const int c0 = min(p.Nc, rank * cand_per), c1 = min(p.Nc, c0 + cand_per);
  // ---- state into shared memory; RHS = F + rho (H + U) for the first iteration (:56), row pitch Rp, pad columns zero
  for (int e = t; e < Rp * Rp; e += kThreads) sm.Minv[e] = (e < R * Rp) ? p.Minv[e] : 0.0f;
  double* rhs = reinterpret_cast<double*>(sm.X);   // own rows of RHS (float32 values, widened once), row pitch Rp
  for (int e = t; e < own; e += kThreads) {
    const int il = e / R, c = e - il * R;
    const float u = p.U[e_base + e];
    sm.U[e] = u;
    rhs[il * Rp + c] = (double)rhs_of(p.F[e_base + e], rho, p.H[e_base + e], u);
  }
  cl_sync();   // every CTA of the cluster is running (remote shared memory may be written from here on)
  const int row_groups = (own_rows + 3) / 4;
  bool pending = false;   // residual sums of the previous iteration wait for their (deferred) exit test
  int done = 0;
  for (int j = 1; j < p.max_iter; ++j) {  // range(1, max_iter), :55
    // ---------------- P1: H_ls = RHS . Minv for the own rows (4 rows x 1 column per thread), V to every CTA
    unsigned int kmax = 0u, kinv = 0u;
    for (int item = t; item < row_groups * R; item += kThreads) {
      const int rg = item / R, col = item - rg * R;
      const int r0 = rg * 4;
      const double* x0 = rhs + (size_t)min(r0, own_rows - 1) * Rp;
      const double* x1 = rhs + (size_t)min(r0 + 1, own_rows - 1) * Rp;
      const double* x2 = rhs + (size_t)min(r0 + 2, own_rows - 1) * Rp;
      const double* x3 = rhs + (size_t)min(r0 + 3, own_rows - 1) * Rp;
      const float* mp = sm.Minv + col;
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll 2
      for (int k = 0; k < R; ++k) {   // (the pad columns of RHS are overwritten by the sort of P2: never read)
        const double m = (double)mp[(size_t)k * Rp];
        a0 = fma(x0[k], m, a0);
        a1 = fma(x1[k], m, a1);
        a2 = fma(x2[k], m, a2);
        a3 = fma(x3[k], m, a3);
      }
      const float acc[4] = {(float)a0, (float)a1, (float)a2, (float)a3};
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int il = r0 + a;
        if (il < own_rows) {
          const int e = il * R + col;
          sm.Hls[e] = acc[a];
          const float v = sub_rn(acc[a], sm.U[e]);   // V = H_ls - U (:59)
          const unsigned int key = float_key(v);
          kmax = max(kmax, key);
          kinv = max(kinv, ~key);
          for (int rk = 0; rk < C; ++rk) cl_store(cl_map(&sm.Vall[e_base + e], (unsigned int)rk), v);
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
    if (t < 2 * C) {   // this CTA's keys into slot `rank` of every CTA
      unsigned int k = 0u;
      for (int w = 0; w < kWarps; ++w) k = max(k, sm.wkey[t & 1][w]);
      cl_store(cl_map(&sm.keys[rank][t & 1], (unsigned int)(t >> 1)), k);
    }
    cl_sync();   // ---- barrier 1: V, keys (and the previous iteration's residual sums) are everywhere
    // exit test of iteration j - 1 (:62-65); the speculative P1 above touched neither H, U nor RHS
    if (pending && cluster_converged(sm.slots, C, p.eps, rep)) {
      rep.status |= ADMMQ_ST_CONVERGED;
      pending = false;
      break;
    }
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
    cl_sync();   // ---- barrier 2: every candidate's sum is everywhere (and nobody reads V / the sorted array any more)
    if (search) {
      rep.best_index = cta_best_candidate<false>(sm.cand, p.Nc, pj.absmax, (double)n, sm.best);
      qp.scale = clip_scale<G>(pj.absmax, p.Nc, rep.best_index, L);
    }
    rep.scale = qp.scale;
    rb.lap(1);
    // ---------------- P3: H = Q(V), U += H - H_ls, residual sums, next RHS - own rows
    ResidualSums res;
    for (int e = t; e < own; e += kThreads) {
      const int il = e / R, c = e - il * R;
      const float hp = p.H[e_base + e];
      const float fv = __ldg(p.F + e_base + e);
      const ElementStep o = p3_element<G>(sm.Hls[e], sm.U[e], hp, fv, rho, qp, L, pj.degenerate, res);
      p.H[e_base + e] = o.hq;
      sm.U[e] = o.un;
      rhs[il * Rp + c] = (double)o.rhs_next;
      if (p.codes != nullptr) p.codes[e_base + e] = (int8_t)o.code;
    }
    res.flush();
    if (pj.degenerate) {  // uniform
      rb.nonfinite();
      pending = false;
      break;
    }
    cta_sum4(res.sums, sm);  // (contains the barriers that publish U and X for the next iteration)
    if (t < 4 * C) cl_store(cl_map(&sm.slots[rank][t & 3], (unsigned int)(t >> 2)), res.total(t & 3));
    pending = true;
    rb.lap(2);
  }
  cl_sync();   // the last residual sums are everywhere; no CTA leaves while its shared memory may still be written
  if (pending && cluster_converged(sm.slots, C, p.eps, rep)) rep.status |= ADMMQ_ST_CONVERGED;
  rep.iterations = done;
  for (int e = t; e < own; e += kThreads) p.U[e_base + e] = sm.U[e];
  rb.finish(p.report, rank == 0 && t == 0);
}

// Size of the cluster for a factor: the largest power of two in {8, 4} within the budget for which a CTA's own rows fit
// its shared-memory arrays; 0 = not eligible (a CTA without rows still takes its share of the candidates).  Two CTAs are
// not worth it: measured 36.4 us per iteration on 64 x 134 against 35.8 us for the single-CTA kernel (26.1 us on four
// CTAs, 17.9 us on eight).
inline int cluster_ctas_for(int I, int R, int Rp, int num_attempts, int budget) {
  if ((long long)I * R > kResMaxElems || (long long)Rp * Rp > kResMaxMinv || num_attempts > kMaxCandidates) return 0;
  for (int c = kClMaxCtas; c >= 4; c >>= 1) {
    if (c > budget) continue;
    const long long rows = (I + c - 1) / c;
    if (rows * R <= kClMaxOwn && 2 * rows * Rp <= kResMaxElems) return c;   // own RHS rows as float64 in the X array
  }
  return 0;
}

}  // namespace admmq
