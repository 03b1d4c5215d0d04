// admm_loop.cu - the persistent ADMM inner loop (admmq_admm_iteration) and the ridge-system
// inverse (admmq_spd_inverse).  Replaces admm_iteration() of source/admm.py:51-67.
//
// One cooperative launch (one CTA per SM) runs ALL max_iter-1 inner iterations; per iteration
//   P1  H_ls = RHS . Minv            RHS = F + rho (H + U)                                (:56-57)
//       precision 0: float64-accumulating tiles against the float64 inverse (parity mode: the correctly rounded
//       solve); precision 1: 3xTF32 on tcgen05/TMEM, operands fetched by TMA (tc_gemm.cuh; throughput mode);
//       precision 2 and shapes that do not fill a tensor-core tile: float32 FFMA tiles, column strips for <= 16 rows;
//       admmq_split_loop: elementwise (two-block splitting)
//       epilogue: abs-max key of V = H_ls - U                                          (:59, q.py:129)
//   --- device-wide barrier
//   P2  per-candidate squared-error sums of the clip search over V (search.cuh)         (q.py:136-139)
//   --- device-wide barrier
//   P3  argmin -> scale; H = Q(V); U += H - H_ls; residual sums; next RHS              (:59-63, q.py:141-144)
//   --- device-wide barrier; the exit test r < eps && s < eps (:64-65) of iteration j is evaluated after the first
//       barrier of iteration j + 1 (P1 touches no result, so the speculative product is dropped when the test fires)
// State (H, U, F, H_ls, RHS, Minv) stays L2 resident for the whole call: per iteration the
// algorithmic traffic is 16 B per element of H plus one pass over Minv, all served from L2.
// A small factor on a budget of one CTA takes the shared-memory-resident kernel of admm_loop_resident.cuh instead.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include "search.cuh"
#include "admm_loop_common.cuh"
#include "spd_inverse.cuh"
#include "tc_gemm.cuh"
#include "admm_loop_resident.cuh"
#include "admm_loop_cluster.cuh"
#include "admm_loop_tap.cuh"

namespace admmq {

constexpr int kKeySlots = 3;

// B operand of the tensor-core ridge product: pre-split hi / lo parts of Minv fetched by TMA straight into the operand
// stages (1: no conversion work, twice the L2 traffic for B) or the float32 Minv itself, split tile by tile by the
// converter warps (0).  See DESIGN.md 5 for the measurements behind the default.
#ifndef ADMMQ_LOOP_PS
#define ADMMQ_LOOP_PS 1
#endif
constexpr bool kLoopPS = ADMMQ_LOOP_PS != 0;

struct LoopHeader {  // start of the workspace; zeroed by cudaMemsetAsync before every call
  unsigned int barrier_loop;
  unsigned int pad[3];
  unsigned int keys[kKeySlots][4];  // rotating {max key, ~min key, -, -} of V
  unsigned int smid_mask[8];        // diagnostics: bit s is set when a CTA of the last launch ran on SM s (%smid)
};
static_assert(sizeof(LoopHeader) <= 256, "the header page is 256 bytes");

struct IterationHeader {  // admmq_admm_iteration only: scalars handed from the inverse to the loop
  unsigned int barrier_inv;
  int status;  // ADMMQ_E_NOT_PD from the inverse
  float rho;
  unsigned int pad;
};

struct LoopParams {
  CUtensorMap tm_rhs;      // TMA descriptors of RHS (I x R, ld Rp) and of the hi / lo tf32 parts of Minv (R x R, ld Rp);
  CUtensorMap tm_minv_hi;  // only used by the tensor-core variant of P1
  CUtensorMap tm_minv_lo;
  float* MinvHi;           // R x Rp each, made from Minv by the kernel's prologue (tensor-core variant)
  float* MinvLo;
  int tc_bn;               // tile width of the tensor-core variant (multiple of 16, <= TCBN)
  float* H;         // the caller's dense I x R arrays: read by the prologue, written back after the last iteration
  float* U;
  const float* F;
  float* Hp;        // working copies with row pitch Rp (pad columns zero): every array of the loop then shares ONE element
  float* Up;        // index and is accessed in aligned 16-byte groups
  float* Fp;
  const float* H2;  // kDiagP1 only: the other block of the two-block splitting (scripts/factorize_lowrank.py:85)
  int I, R, Rp;
  int max_iter;
  float eps;
  int bits, scheme, Nc;
  float neg_zero;  // -0.0f as a run-time value (see search.cuh)
  int direct_below;  // chunks of at most this many elements per CTA take the direct form of the clip search
  int8_t* codes;
  admmq_loop_report* report;
  const float* rho;       // device scalar: trace(G)/R
  const int* inv_status;  // device scalar or nullptr
  LoopHeader* hdr;
  unsigned long long* cand;  // [kKeySlots][kMaxCandidates]
  double* slots;             // [gridDim.x][4]
  float* Hls;                // I x Rp
  float* V;                  // I x R flat: H_ls - U, the projection input of this iteration (source/admm.py:59)
  float* RHS;                // I x Rp (pad columns stay zero)
  const float* Minv;         // R x Rp
  const double* Minv64;      // R x Rp float64 inverse (parity mode, kF64P1) or nullptr
};

// P1 shared memory: two K-groups (256 threads each) work on alternating 16-deep slabs of the same
// output tile and are summed at the end, so that 16 warps hide the L2 latency of the operand loads.
template <int BM, int BN>
struct __align__(16) GemmSmem {
  float a[2][16][BM + 4];
  float b[2][16][BN + 4];
  float red[BM * BN];
};

struct ResidualSmem {
  double red[4][kWarps];
};

__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

// P1: every CTA takes tiles round-robin; each K-group of 256 threads as (BM/TM) x (BN/TN).
template <int BM, int BN, int TM, int TN>
__device__ void gemm_phase(const LoopParams& p, GemmSmem<BM, BN>& gs, unsigned int* keys) {
  constexpr int TX = BN / TN, TY = BM / TM;
  static_assert(TX * TY == 256, "thread tiling must cover the tile with one K-group");
  const int kg = threadIdx.x >> 8, t = threadIdx.x & 255, tx = t % TX, ty = t / TX;
  const int I = p.I, R = p.R, Rp = p.Rp;
  const int tilesN = (R + BN - 1) / BN, tilesM = (I + BM - 1) / BM;
  const int nslab = (R + 15) / 16, nstep = (nslab + 1) / 2;   // slab = 2 * step + kg
  const int arow = t >> 2, akq = (t & 3) * 4;                 // A loader: BM rows x 4 float4
  const int brow = t / (BN / 4), bc4 = (t % (BN / 4)) * 4;    // B loader: 16 rows x BN/4 float4
  unsigned int kmax = 0u, kinv = 0u;
  for (int tile = blockIdx.x; tile < tilesM * tilesN; tile += gridDim.x) {
    const int i0 = (tile / tilesN) * BM, n0 = (tile % tilesN) * BN;
    float acc[TM][TN];
#pragma unroll
    for (int m = 0; m < TM; ++m)
#pragma unroll
      for (int n = 0; n < TN; ++n) acc[m][n] = 0.0f;
    float4 ra = make_float4(0.f, 0.f, 0.f, 0.f), rb = ra;
    auto fetch = [&](int step) {
      const int k0 = (2 * step + kg) * 16;
      ra = make_float4(0.f, 0.f, 0.f, 0.f);
      rb = ra;
      if (t < BM * 4 && i0 + arow < I && k0 + akq < Rp) ra = ldcg4(p.RHS + (size_t)(i0 + arow) * Rp + k0 + akq);
      if (t < 4 * BN && k0 + brow < R && n0 + bc4 < Rp) rb = __ldg(reinterpret_cast<const float4*>(p.Minv + (size_t)(k0 + brow) * Rp + n0 + bc4));
    };
    fetch(0);
    for (int step = 0; step < nstep; ++step) {
      __syncthreads();
      if (t < BM * 4) {
        gs.a[kg][akq + 0][arow] = ra.x;
        gs.a[kg][akq + 1][arow] = ra.y;
        gs.a[kg][akq + 2][arow] = ra.z;
        gs.a[kg][akq + 3][arow] = ra.w;
      }
      if (t < 4 * BN) *reinterpret_cast<float4*>(&gs.b[kg][brow][bc4]) = rb;
      __syncthreads();
      if (step + 1 < nstep) fetch(step + 1);
#pragma unroll
      for (int kk = 0; kk < 16; ++kk) {
        float av[TM], bv[TN];
#pragma unroll
        for (int m = 0; m < TM; ++m) av[m] = gs.a[kg][kk][ty * TM + m];
#pragma unroll
        for (int n = 0; n < TN; ++n) bv[n] = gs.b[kg][kk][tx * TN + n];
#pragma unroll
        for (int m = 0; m < TM; ++m)
#pragma unroll
          for (int n = 0; n < TN; ++n) acc[m][n] = fmaf(av[m], bv[n], acc[m][n]);
      }
    }
    // K-group 1 hands its partial tile to K-group 0 (fixed order: acc0 + acc1)
    __syncthreads();
    if (kg == 1) {
#pragma unroll
      for (int m = 0; m < TM; ++m)
#pragma unroll
        for (int n = 0; n < TN; ++n) gs.red[(ty * TM + m) * BN + tx * TN + n] = acc[m][n];
    }
    __syncthreads();
    if (kg == 0) {
#pragma unroll
      for (int m = 0; m < TM; ++m)
#pragma unroll
        for (int n = 0; n < TN; ++n) {
          const int i = i0 + ty * TM + m, c = n0 + tx * TN + n;
          if (i < I && c < R) {
            const float h = add_rn(acc[m][n], gs.red[(ty * TM + m) * BN + tx * TN + n]);
            p.Hls[(size_t)i * Rp + c] = h;
            const float v = sub_rn(h, __ldcg(p.Up + (size_t)i * Rp + c));  // V = H_ls - U (:59)
            p.V[(size_t)i * R + c] = v;
            const unsigned int k = float_key(v);
            kmax = max(kmax, k);
            kinv = max(kinv, ~k);
          }
        }
    }
  }
  kmax = warp_max_u32(kmax);
  kinv = warp_max_u32(kinv);
  if ((threadIdx.x & 31) == 0 && (kmax | kinv) != 0u) {
    atomicMax(&keys[0], kmax);
    atomicMax(&keys[1], kinv);
  }
}

// P1 of the PARITY mode (precision 0): H_ls = fl32( RHS . Minv64 ) with the inverse kept in float64 and every product
// and sum formed in float64, i.e. the correctly rounded solution of the ridge system (up to one double rounding) -
// what LAPACK's float32 potrs (source/admm.py:56) approximates to 3e-7.  Same tiling as gemm_phase: two K-groups on
// alternating 16-deep slabs, summed in fixed order.  FP64 FMAs run at half the FP32 rate on B200; this mode exists for
// the bit-level comparisons, not for throughput.
template <int BM, int BN>
struct __align__(16) GemmSmem64 {
  float a[2][16][BM + 4];
  double b[2][16][BN + 2];
  double red[BM * BN];
};

template <int BM, int BN, int TM, int TN>
__device__ void gemm_phase_f64(const LoopParams& p, GemmSmem64<BM, BN>& gs, unsigned int* keys) {
  constexpr int TX = BN / TN, TY = BM / TM;
  static_assert(TX * TY == 256, "thread tiling must cover the tile with one K-group");
  const int kg = threadIdx.x >> 8, t = threadIdx.x & 255, tx = t % TX, ty = t / TX;
  const int I = p.I, R = p.R, Rp = p.Rp;
  const int tilesN = (R + BN - 1) / BN, tilesM = (I + BM - 1) / BM;
  const int nslab = (R + 15) / 16, nstep = (nslab + 1) / 2;   // slab = 2 * step + kg
  unsigned int kmax = 0u, kinv = 0u;
  for (int tile = blockIdx.x; tile < tilesM * tilesN; tile += gridDim.x) {
    const int i0 = (tile / tilesN) * BM, n0 = (tile % tilesN) * BN;
    double acc[TM][TN];
#pragma unroll
    for (int m = 0; m < TM; ++m)
#pragma unroll
      for (int n = 0; n < TN; ++n) acc[m][n] = 0.0;
    for (int step = 0; step < nstep; ++step) {
      const int k0 = (2 * step + kg) * 16;
      __syncthreads();
      for (int idx = t; idx < BM * 16; idx += 256) {  // A slab, transposed into [k][row]
        const int row = idx >> 4, kk = idx & 15;
        gs.a[kg][kk][row] = (i0 + row < I && k0 + kk < R) ? __ldcg(p.RHS + (size_t)(i0 + row) * Rp + k0 + kk) : 0.0f;
      }
      for (int idx = t; idx < 16 * BN; idx += 256) {  // B slab
        const int kk = idx / BN, c = idx - kk * BN;
        gs.b[kg][kk][c] = (k0 + kk < R && n0 + c < R) ? __ldg(p.Minv64 + (size_t)(k0 + kk) * Rp + n0 + c) : 0.0;
      }
      __syncthreads();
#pragma unroll 4
      for (int kk = 0; kk < 16; ++kk) {
        double av[TM], bv[TN];
#pragma unroll
        for (int m = 0; m < TM; ++m) av[m] = (double)gs.a[kg][kk][ty * TM + m];
#pragma unroll
        for (int n = 0; n < TN; ++n) bv[n] = gs.b[kg][kk][tx * TN + n];
#pragma unroll
        for (int m = 0; m < TM; ++m)
#pragma unroll
          for (int n = 0; n < TN; ++n) acc[m][n] = fma(av[m], bv[n], acc[m][n]);
      }
    }
    __syncthreads();
    if (kg == 1) {
#pragma unroll
      for (int m = 0; m < TM; ++m)
#pragma unroll
        for (int n = 0; n < TN; ++n) gs.red[(ty * TM + m) * BN + tx * TN + n] = acc[m][n];
    }
    __syncthreads();
    if (kg == 0) {
#pragma unroll
      for (int m = 0; m < TM; ++m)
#pragma unroll
        for (int n = 0; n < TN; ++n) {
          const int i = i0 + ty * TM + m, c = n0 + tx * TN + n;
          if (i < I && c < R) {
            const float h = (float)(acc[m][n] + gs.red[(ty * TM + m) * BN + tx * TN + n]);
            p.Hls[(size_t)i * Rp + c] = h;
            const float v = sub_rn(h, __ldcg(p.Up + (size_t)i * Rp + c));  // V = H_ls - U (:59)
            p.V[(size_t)i * R + c] = v;
            const unsigned int k = float_key(v);
            kmax = max(kmax, k);
            kinv = max(kinv, ~k);
          }
        }
    }
  }
  kmax = warp_max_u32(kmax);
  kinv = warp_max_u32(kinv);
  if ((threadIdx.x & 31) == 0 && (kmax | kinv) != 0u) {
    atomicMax(&keys[0], kmax);
    atomicMax(&keys[1], kinv);
  }
}

// P1 for factors with very few rows (the 3 x 3 tap factor of a convolution: I = 9): a 128-row tensor-core tile or a
// 16 x 32 FFMA tile would idle on padding, and the product is really I matrix-vector products that stream Minv once.
// Every CTA owns a strip of output columns; inside the CTA thread (c, s) accumulates columns 4c .. 4c+3 of the strip
// over the k-slice {s, s + ks, ...} (Minv rows read as float4 from L2, the staged RHS from shared memory), and the
// k-slices are summed in fixed order through shared memory.
template <int MI>
struct __align__(16) SkinnySmem {
  static constexpr int kRhsFloats = 16384;  // I * Rp must fit (launch_loop checks)
  float rhs[kRhsFloats];
  float red[512 * MI * 4];
};

template <int MI>
__device__ void gemm_phase_skinny(const LoopParams& p, SkinnySmem<MI>& ss, unsigned int* keys) {
  const int I = p.I, R = p.R, Rp = p.Rp, t = threadIdx.x;
  const int cps = ((R + (int)gridDim.x - 1) / (int)gridDim.x + 3) / 4 * 4;
  const int n_begin = blockIdx.x * cps, n_end = min(R, n_begin + cps);
  unsigned int kmax = 0u, kinv = 0u;
  if (n_begin < R) {  // uniform per CTA
    __syncthreads();
    // stage RHS, four loads in flight per thread (the phase is a chain of L2 round trips otherwise)
    for (int e0 = t * 4; e0 < I * Rp; e0 += kThreads * 16) {
      float4 r[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * kThreads * 4;
        if (e < I * Rp) r[u] = ldcg4(p.RHS + e);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = e0 + u * kThreads * 4;
        if (e < I * Rp) *reinterpret_cast<float4*>(&ss.rhs[e]) = r[u];
      }
    }
    __syncthreads();
    for (int s0 = n_begin; s0 < n_end; s0 += 128) {
      const int w = min(128, n_end - s0);
      const int cg = (w + 3) >> 2;     // float4 column groups; s0 + 4 cg <= Rp, the pad columns of Minv are zero
      const int ks = kThreads / cg;    // k-slices
      const int s = t / cg, c = t - s * cg;
      float acc[MI][4];
#pragma unroll
      for (int i = 0; i < MI; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0f;
      if (s < ks) {
        const float* mp = p.Minv + s0 + 4 * c;
        // a thread takes groups of four consecutive rows of Minv (k = 4 g .. 4 g + 3, g = s, s + ks, ...): the four RHS
        // values of a factor row come as ONE 16-byte shared-memory load for 16 FMAs (one 4-byte load per 4 FMAs made
        // the loop issue and shared-memory-latency bound: ncu showed 140 instructions per row of Minv); kG groups in
        // flight.  Rows >= R of Minv do not exist (read as zero); the pad columns of RHS are zero.
        constexpr int kG = MI <= 9 ? 2 : 1;
        const int ngroups = (R + 3) >> 2;
        for (int g0 = s; g0 < ngroups; g0 += ks * kG) {
          float4 m[kG][4];
#pragma unroll
          for (int u = 0; u < kG; ++u) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int k = 4 * (g0 + u * ks) + q;
              m[u][q] = (k < R) ? __ldcg(reinterpret_cast<const float4*>(mp + (size_t)k * Rp)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
#pragma unroll
          for (int u = 0; u < kG; ++u) {
            const int g = g0 + u * ks;
            if (g < ngroups) {
#pragma unroll
              for (int i = 0; i < MI; ++i) {
                if (i < I) {
                  const float4 r4 = *reinterpret_cast<const float4*>(&ss.rhs[i * Rp + 4 * g]);
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
          *reinterpret_cast<float4*>(&ss.red[(size_t)t * (MI * 4) + i * 4]) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
      }
      __syncthreads();
      for (int o = t; o < I * w; o += kThreads) {
        const int i = o / w, nn = o - i * w;
        const int cc = nn >> 2, q = nn & 3;
        const int n = s0 + nn;
        const float u = __ldcg(p.Up + (size_t)i * Rp + n);  // requested before the (long) sum over the slices
        // fixed order: four interleaved partial sums over the k-slices, then ((h0 + h1) + (h2 + h3))
        float h4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        const float* rp = &ss.red[(size_t)cc * (MI * 4) + i * 4 + q];
        int sl = 0;
        for (; sl + 3 < ks; sl += 4) {
#pragma unroll
          for (int a = 0; a < 4; ++a) h4[a] = add_rn(h4[a], rp[(size_t)((sl + a) * cg) * (MI * 4)]);
        }
        for (; sl < ks; ++sl) h4[sl & 3] = add_rn(h4[sl & 3], rp[(size_t)(sl * cg) * (MI * 4)]);
        const float h = add_rn(add_rn(h4[0], h4[1]), add_rn(h4[2], h4[3]));
        p.Hls[(size_t)i * Rp + n] = h;
        const float v = sub_rn(h, u);  // V = H_ls - U (:59)
        p.V[(size_t)i * R + n] = v;
        const unsigned int k = float_key(v);
        kmax = max(kmax, k);
        kinv = max(kinv, ~k);
      }
      __syncthreads();
    }
  }
  kmax = warp_max_u32(kmax);
  kinv = warp_max_u32(kinv);
  if ((threadIdx.x & 31) == 0 && (kmax | kinv) != 0u) {
    atomicMax(&keys[0], kmax);
    atomicMax(&keys[1], kinv);
  }
}

// P1 of the two-block splitting W ~ W_q + W_r (scripts/factorize_lowrank.py:80-101): the least-squares step is
// elementwise, H_ = (rho (H + U) + W - H2) / (1 + rho) with p.F = W, evaluated in the reference's operation order.
// Every CTA works on the chunk of elements it also owns in P2 / P3 (I = 1, R = number of elements).
constexpr int kDiagP1 = -1000;
constexpr int kF64P1 = -2000;  // TCBN value of the parity mode: float64-accumulating tiles against Minv64
__device__ void elementwise_phase(const LoopParams& p, float rho, long long e0, long long e1, unsigned int* keys) {
  const float opr = add_rn(1.0f, rho);
  unsigned int kmax = 0u, kinv = 0u;
  for (long long e = e0 + threadIdx.x; e < e1; e += kThreads) {
    const float u = __ldcg(p.Up + e);   // I = 1: padded and dense indices coincide
    const float h = div_rn(sub_rn(add_rn(mul_rn(rho, add_rn(__ldcg(p.Hp + e), u)), p.F[e]), p.H2[e]), opr);   // :85
    p.Hls[e] = h;
    const float v = sub_rn(h, u);                                                                  // :88
    p.V[e] = v;
    const unsigned int k = float_key(v);
    kmax = max(kmax, k);
    kinv = max(kinv, ~k);
  }
  kmax = warp_max_u32(kmax);
  kinv = warp_max_u32(kinv);
  if ((threadIdx.x & 31) == 0 && (kmax | kinv) != 0u) {
    atomicMax(&keys[0], kmax);
    atomicMax(&keys[1], kinv);
  }
}

// P1 on the tensor cores: 128 x bn tiles (bn = p.tc_bn <= TCBN) of H_ls = RHS . Minv^T (Minv is symmetric) in 3xTF32;
// Minv comes pre-split into its tf32 hi / lo parts (constant over the call, made by the kernel's prologue).
template <int TCBN>
__device__ void gemm_phase_tc(const LoopParams& p, unsigned char* smem_tiles, tc::Pipe& pipe, tc::PipeState& st,
                              unsigned int* keys) {
  const int I = p.I, R = p.R, Rp = p.Rp, bn = p.tc_bn;
  const int tilesN = (R + bn - 1) / bn, tilesM = (I + tc::kTileM - 1) / tc::kTileM;
  unsigned int kmax = 0u, kinv = 0u;
  // RHS was written with ordinary stores by other CTAs before the grid barrier; the TMA engine reads through the
  // async proxy
  asm volatile("fence.proxy.async;" ::: "memory");
  for (int tile = blockIdx.x; tile < tilesM * tilesN; tile += gridDim.x) {
    const int i0 = (tile / tilesN) * tc::kTileM, n0 = (tile % tilesN) * bn;
    const int next = tile + (int)gridDim.x;
    const bool has_next = next < tilesM * tilesN;
    tc::tile_3xtf32<TCBN, kLoopPS>(&p.tm_rhs, i0, &p.tm_minv_hi, &p.tm_minv_lo, n0, bn, R, smem_tiles, pipe, st,
                                has_next ? (next / tilesN) * tc::kTileM : -1, has_next ? (next % tilesN) * bn : -1);
    // epilogue over row-contiguous float4 groups of the tile parked in shared memory (coalesced global traffic)
    const float* tile_h = tc::acc_to_smem<TCBN, kLoopPS>(pipe, smem_tiles);
    using ET = tc::EpiTile<TCBN>;
    // U comes from L2 (working copy, row pitch Rp: one aligned 16-byte load per group): the loads of up to four groups
    // per thread are issued before the first use, so the epilogue pays two L2 round trips per tile instead of eight
    constexpr int kIt = (ET::kGroups + kThreads - 1) / kThreads;
    constexpr int kChunk = kIt < 4 ? kIt : 4;
#pragma unroll
    for (int c0 = 0; c0 < kIt; c0 += kChunk) {
      float4 u[kChunk];
#pragma unroll
      for (int j = 0; j < kChunk; ++j) {
        const int g = (c0 + j) * kThreads + (int)threadIdx.x;
        const int row = g / ET::kGroupsPerRow, c4 = (g - row * ET::kGroupsPerRow) * 4;
        const int i = i0 + row, n = n0 + c4;
        u[j] = (c0 + j < kIt && g < ET::kGroups && c4 < bn && i < I && n < R)
                   ? ldcg4(p.Up + (unsigned int)i * (unsigned int)Rp + (unsigned int)n) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int j = 0; j < kChunk; ++j) {
        const int g = (c0 + j) * kThreads + (int)threadIdx.x;
        const int row = g / ET::kGroupsPerRow, c4 = (g - row * ET::kGroupsPerRow) * 4;
        const int i = i0 + row, n = n0 + c4;
        if (c0 + j < kIt && g < ET::kGroups && c4 < bn && i < I && n < R) {
          const float4 h4 = *reinterpret_cast<const float4*>(tile_h + ET::offset(row, c4 >> 2));
          const float h[4] = {h4.x, h4.y, h4.z, h4.w};
          const float uu[4] = {u[j].x, u[j].y, u[j].z, u[j].w};
          *reinterpret_cast<float4*>(p.Hls + (unsigned int)i * (unsigned int)Rp + (unsigned int)n) = h4;  // n + 3 < Rp: pad columns hold the zero-filled product
          const unsigned int e = (unsigned int)i * (unsigned int)R + (unsigned int)n;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (n + q < R) {
              const float d = sub_rn(h[q], uu[q]);  // V = H_ls - U (:59)
              p.V[e + q] = d;
              const unsigned int k = float_key(d);
              kmax = max(kmax, k);
              kinv = max(kinv, ~k);
            }
          }
        }
      }
    }
    __syncthreads();  // the staging tile lives in the operand stages the next tile's producers write
  }
  kmax = warp_max_u32(kmax);
  kinv = warp_max_u32(kinv);
  if ((threadIdx.x & 31) == 0 && (kmax | kinv) != 0u) {
    atomicMax(&keys[0], kmax);
    atomicMax(&keys[1], kinv);
  }
}

__global__ void __launch_bounds__(kInvThreads, 1) k_spd_inverse(InvParams p) {
  __shared__ InvSmem sm;
  GridBarrier bar;
  bar.init(p.barrier);
  spd_inverse_body(p, sm, bar);
}

template <int BM, int BN, int TCBN>
union LoopSmem {
  SearchSmem search;
  GemmSmem<BM, BN> gemm;
  GemmSmem64<BM, BN> gemm64;
  ResidualSmem res;
  unsigned char tc_tiles[TCBN > 0 ? tc::TileSmem<(TCBN > 0 ? TCBN : 16), kLoopPS>::kBytes : 16];
  SkinnySmem<(TCBN < 0 && TCBN != kDiagP1 && TCBN != kF64P1 ? -TCBN : 1)> skinny;
};

// Totals of the per-CTA residual slots, formed redundantly by every warp: lane c takes the CTAs c, c + 32, ... in
// order, then a xor butterfly (the same association in every lane, warp and CTA, so every thread of the grid holds
// bit-identical totals) - no shared memory and no CTA barrier on the path of the exit test.
__device__ __forceinline__ void slot_totals(const double* slots, int ctas, double tot[4]) {
  tot[0] = tot[1] = tot[2] = tot[3] = 0.0;
  for (int c = threadIdx.x & 31; c < ctas; c += 32) {
    const double2 a = __ldcg(reinterpret_cast<const double2*>(slots + (size_t)c * 4));
    const double2 b = __ldcg(reinterpret_cast<const double2*>(slots + (size_t)c * 4 + 2));
    tot[0] += a.x;
    tot[1] += a.y;
    tot[2] += b.x;
    tot[3] += b.y;
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) tot[q] = warp_sum(tot[q]);
}

// TCBN = 0: P1 as float32 FFMA tiles (BM x BN, TM x TN per thread); TCBN = 16 / 32 / 64: P1 on the tensor cores;
// TCBN = -MI: P1 for factors with at most MI rows (gemm_phase_skinny); TCBN = kDiagP1: elementwise P1 of the
// two-block splitting (elementwise_phase); TCBN = kF64P1: float64-accumulating tiles against the float64 inverse
// (parity mode, gemm_phase_f64).  G: the grid of the clip search (numerics.cuh SearchGrid); the E2M1 and FP8 / FP6
// instantiations run no other scheme.
template <int BM, int BN, int TM, int TN, int TCBN, Grid G>
__global__ void __launch_bounds__(kThreads, 1) k_admm_loop(const __grid_constant__ LoopParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  LoopSmem<BM, BN, TCBN>& sm = *reinterpret_cast<LoopSmem<BM, BN, TCBN>*>(smem_raw);
  __shared__ tc::Pipe pipe;
  __shared__ unsigned int cta_keys[2];   // this CTA's {max key, ~min key} of V, merged here before they go to the header
  tc::PipeState pst;
  const int t = threadIdx.x;
  if (t < 2) cta_keys[t] = 0u;           // (visible to all warps after the barrier that ends the prologue)
  LoopHeader* hdr = p.hdr;
  admmq_loop_report rep;
  rep.iterations = 0;
  rep.status = 0;
  rep.rho = *p.rho;
  rep.scale = 0.0f;
  rep.r = 0.0f;
  rep.s = 0.0f;
  rep.best_index = -1;
  rep.absmax = 0.0f;
  rep.phase_ns[0] = rep.phase_ns[1] = rep.phase_ns[2] = rep.phase_ns[3] = 0ull;
  if (p.inv_status != nullptr && *p.inv_status != 0) {  // G + rho I was not positive definite: nothing is touched
    rep.status = *p.inv_status;
    if (blockIdx.x == 0 && t == 0) *p.report = rep;
    return;
  }
  if constexpr (TCBN > 0) tc::pipe_setup(pipe, pst, p.neg_zero);
  const unsigned long long t_begin = global_ns();
  unsigned long long t_mark = t_begin;
  auto lap = [&](int phase) {
    const unsigned long long now = global_ns();
    rep.phase_ns[phase] += now - t_mark;
    t_mark = now;
  };
  GridBarrier bar;
  bar.init(&hdr->barrier_loop);
  if (t == 0) {   // where the grid runs (tools / bench.py --placement read the mask from the workspace header)
    unsigned int smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    atomicOr(&hdr->smid_mask[(smid >> 5) & 7], 1u << (smid & 31));
  }
  const float rho = rep.rho;
  const int R = p.R, Rp = p.Rp;
  const long long N = (long long)p.I * R;
  const long long cs = chunk_size(N, gridDim.x);
  const long long e0 = min(N, (long long)blockIdx.x * cs), e1 = min(N, e0 + cs);
  const Levels L = make_levels(p.bits, G == kGridFP ? p.scheme : 0);
  const float qnan = __int_as_float(0x7fc00000);
  // P3 and the copies around the loop walk the working arrays (row pitch Rp) in aligned groups of four floats: groups
  // [g0, g1) belong to this CTA, thread t takes g0 + t, g0 + t + kThreads, ...  Only the last group of a row can hold
  // pad columns (Rp - R <= 3 of them).
  const unsigned int gpr = (unsigned int)Rp >> 2;                       // groups per row
  unsigned int g0, g1;
  {
    const unsigned int gtot = (unsigned int)p.I * gpr;
    const unsigned int gcs = (gtot + gridDim.x - 1) / gridDim.x;
    g0 = min(gtot, blockIdx.x * gcs);
    g1 = min(gtot, g0 + gcs);
  }
  // (row, column group) of the thread's first group and the step of kThreads groups are recomputed where they are used
  // (one integer division per phase) instead of being carried in registers through the tensor-core phase
#define ADMMQ_GROUP_WALK()                                                                                       \
  const unsigned int grow0 = (g0 + (unsigned int)t) / gpr, gcol0 = (g0 + (unsigned int)t) - grow0 * gpr;         \
  const unsigned int gdrow = (unsigned int)kThreads / gpr, gdcol = (unsigned int)kThreads - gdrow * gpr;         \
  const int last_valid = R - 4 * (int)(gpr - 1) /* valid columns of a row's last group (1 .. 4) */

  if constexpr (TCBN > 0 && kLoopPS) {  // tf32 hi / lo parts of Minv for the tensor-core product (same split as the A operand)
    const long long n4 = (long long)R * Rp / 4;
    for (long long e = (long long)blockIdx.x * kThreads + t; e < n4; e += (long long)gridDim.x * kThreads) {
      float4 hi, lo;
      tc::split4(__ldg(reinterpret_cast<const float4*>(p.Minv) + e), pst.nz2, hi, lo);
      reinterpret_cast<float4*>(p.MinvHi)[e] = hi;
      reinterpret_cast<float4*>(p.MinvLo)[e] = lo;
    }
  }
  // working copies of H, U, F and RHS = F + rho * (H + U) for the first iteration (:56); pad columns are zero
  {
    ADMMQ_GROUP_WALK();
    unsigned int row = grow0, cg = gcol0;
    for (unsigned int g = g0 + (unsigned int)t; g < g1; g += kThreads) {
      const int nv = (cg == gpr - 1) ? last_valid : 4;
      const size_t e = (size_t)row * R + 4 * cg;
      float h[4], u[4], f[4], rhs[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const bool ok = q < nv;
        h[q] = ok ? p.H[e + q] : 0.0f;
        u[q] = ok ? p.U[e + q] : 0.0f;
        f[q] = (ok && TCBN != kDiagP1) ? p.F[e + q] : 0.0f;
        rhs[q] = ok ? add_rn(f[q], mul_rn(rho, add_rn(h[q], u[q]))) : 0.0f;
      }
      reinterpret_cast<float4*>(p.Hp)[g] = make_float4(h[0], h[1], h[2], h[3]);
      reinterpret_cast<float4*>(p.Up)[g] = make_float4(u[0], u[1], u[2], u[3]);
      reinterpret_cast<float4*>(p.Hls)[g] = make_float4(0.f, 0.f, 0.f, 0.f);   // its pad columns are read (and ignored) by P3
      if constexpr (TCBN != kDiagP1) {
        reinterpret_cast<float4*>(p.Fp)[g] = make_float4(f[0], f[1], f[2], f[3]);
        reinterpret_cast<float4*>(p.RHS)[g] = make_float4(rhs[0], rhs[1], rhs[2], rhs[3]);
      }
      row += gdrow;
      cg += gdcol;
      if (cg >= gpr) {
        cg -= gpr;
        ++row;
      }
    }
  }
  bar.sync();

  bool pending = false;   // the residual slots of the last finished iteration have not been tested yet
  auto residuals_below_eps = [&]() {
    double tot[4];
    slot_totals(p.slots, (int)gridDim.x, tot);
    rep.r = div_rn((float)tot[0], (float)tot[1]);
    rep.s = div_rn((float)tot[2], (float)tot[3]);
    return rep.r < p.eps && rep.s < p.eps;
  };
  for (int j = 1; j < p.max_iter; ++j) {  // range(1, max_iter), :55
    const int slot = j % kKeySlots, next_slot = (j + 1) % kKeySlots;
    // ---------------- P1
    // the warps' min / max keys are merged in shared memory first: two global atomics per CTA instead of two per warp
    // (a grid of 148 CTAs otherwise sends 4.7 k atomics to the same two L2 words every iteration)
    if constexpr (TCBN > 0) gemm_phase_tc<TCBN>(p, sm.tc_tiles, pipe, pst, cta_keys);
    else if constexpr (TCBN == kDiagP1) elementwise_phase(p, rho, e0, e1, cta_keys);
    else if constexpr (TCBN == kF64P1) gemm_phase_f64<BM, BN, TM, TN>(p, sm.gemm64, cta_keys);
    else if constexpr (TCBN < 0) gemm_phase_skinny<-TCBN>(p, sm.skinny, cta_keys);
    else gemm_phase<BM, BN, TM, TN>(p, sm.gemm, cta_keys);
    __syncthreads();
    if (t == 0) {
      if ((cta_keys[0] | cta_keys[1]) != 0u) {
        atomicMax(&hdr->keys[slot][0], cta_keys[0]);
        atomicMax(&hdr->keys[slot][1], cta_keys[1]);
      }
      cta_keys[0] = cta_keys[1] = 0u;
    }
    if (blockIdx.x == 0) {  // recycle the accumulators of iteration j+1 (last read in iteration j-2)
      if (t < 4) hdr->keys[next_slot][t] = 0u;
      for (int c = t; c < p.Nc; c += kThreads) p.cand[(size_t)next_slot * kMaxCandidates + c] = 0ull;
    }
    bar.sync();
    lap(0);
    // ---------------- exit test of iteration j - 1 (:62-65), evaluated identically by every thread of the grid.  It is
    // deferred past this iteration's P1: the residual slots are complete after the barrier that ended iteration j - 1,
    // P1 touches neither H, U, the codes nor the report, so a speculative P1 is simply dropped when the test fires, and
    // the slots' L2 round trip overlaps the one of the min / max keys below instead of standing alone after a barrier.
    if (pending && residuals_below_eps()) {
      rep.status |= ADMMQ_ST_CONVERGED;
      pending = false;
      break;
    }
    pending = false;
    // ---------------- P2
    const float tmax = key_float(__ldcg(&hdr->keys[slot][0]));
    const float tmin = key_float(~__ldcg(&hdr->keys[slot][1]));
    float absmax = fmaxf(fabsf(tmin), fabsf(tmax));
    if (tmin != tmin || tmax != tmax) absmax = qnan;
    rep.absmax = absmax;
    rep.iterations = j;
    QParams qp;
    qp.scheme = p.scheme;
    qp.bits = p.bits;
    qp.aux = 0.0f;
    qp.n = 0.0f;
    qp.scale = 0.0f;
    bool degenerate = false;
    if (clip_search_scheme<G>(p.scheme)) {
      degenerate = !(absmax > 0.0f) || isinf(absmax);
      if (!degenerate) {
        unsigned long long* cand = p.cand + (size_t)slot * kMaxCandidates;
        cta_candidate_sums<G>(p.V, e0, e1, absmax, p.Nc, L, p.bits, (double)N, cand, sm.search, p.neg_zero, kFormAuto, p.direct_below);
        bar.sync();
        lap(1);
        // ---------------- P3
        rep.best_index = cta_best_candidate<true>(cand, p.Nc, absmax, (double)N, sm.search.direct.key);
        qp.scale = clip_scale<G>(absmax, p.Nc, rep.best_index, L);
      }
    } else {
      degenerate = (absmax != absmax) || isinf(absmax);
      qp = params_from_minmax(p.scheme, p.bits, tmin, tmax, L);
    }
    rep.scale = qp.scale;
    // clip-search scheme: the code comes from x * (1 / scale) + magic-number rounding (numerics.cuh dev_fast, the
    // shortcut the direct search uses); the rare quotient too close to a rounding boundary is redone with the exact
    // division, so the codes stay those of rint(fl(x / scale)).  The E2M1 and FP8 / FP6 grids take the exact division
    // throughout.
    const bool fast_code = G == kGridInt && p.scheme == ADMMQ_Q_MSEMINMAX_SYMMETRIC && !degenerate;
    const float rcp_scale = fast_code ? div_rn(1.0f, qp.scale) : 0.0f;
    double sums[4] = {0.0, 0.0, 0.0, 0.0};
    {
      // batches of kBatch groups (4 elements each) per thread: all 16-byte loads of a batch are issued before the first
      // dependent use, so the phase runs at L2 bandwidth instead of one L2 round trip per element; every array shares
      // the group index (working copies with row pitch Rp), one IMAD.WIDE per address
      constexpr int kBatch = 2;
      ADMMQ_GROUP_WALK();
      unsigned int row = grow0, cg = gcol0;
      unsigned int g = g0 + (unsigned int)t;
      while (g < g1) {
        unsigned int gg[kBatch], eb[kBatch];
        int nvb[kBatch];
        float4 hls4[kBatch], u4[kBatch], hp4[kBatch], fv4[kBatch];
#pragma unroll
        for (int b = 0; b < kBatch; ++b) {
          gg[b] = g;
          nvb[b] = (cg == gpr - 1) ? last_valid : 4;
          eb[b] = row * (unsigned int)R + 4u * cg;   // dense index of the group's first element (codes)
          if (g < g1) {
            hls4[b] = ldcg4(p.Hls + 4u * g);
            u4[b] = ldcg4(p.Up + 4u * g);
            hp4[b] = ldcg4(p.Hp + 4u * g);
            if constexpr (TCBN != kDiagP1) fv4[b] = ldcg4(p.Fp + 4u * g);
          }
          g += kThreads;
          row += gdrow;
          cg += gdcol;
          if (cg >= gpr) {
            cg -= gpr;
            ++row;
          }
        }
        float f0 = 0.0f, f1 = 0.0f, f2 = 0.0f, f3 = 0.0f;   // float32 partial sums over at most 4 * kBatch elements, float64 beyond
        f32x2 a0 = 0ull, a1 = 0ull, a2 = 0ull, a3 = 0ull;     // the same sums of the packed path (even / odd lanes)
#pragma unroll
        for (int b = 0; b < kBatch; ++b) {
          if (gg[b] < g1 && fast_code && nvb[b] == 4) {
            // Full group, clip-search scheme: two elements per instruction (packed f32x2 IEEE operations: the same
            // roundings as the scalar code below, half the issue slots - the phase is issue bound).  Products that the
            // reference rounds on their own (code * scale, rho * (H + U)) are formed as fma(a, b, -0.0) with the -0.0
            // from a kernel parameter, which ptxas cannot contract into the following add (see search.cuh).
            const f32x2 nz2 = pack2(p.neg_zero, p.neg_zero), sc2 = pack2(qp.scale, qp.scale), rc2 = pack2(rcp_scale, rcp_scale);
            const f32x2 magic = pack2(12582912.0f, 12582912.0f), nmagic = pack2(-12582912.0f, -12582912.0f);
            const ulonglong2 hl = *reinterpret_cast<const ulonglong2*>(&hls4[b]), uu = *reinterpret_cast<const ulonglong2*>(&u4[b]);
            const ulonglong2 hpp = *reinterpret_cast<const ulonglong2*>(&hp4[b]);
            const f32x2 hls2[2] = {hl.x, hl.y}, u2[2] = {uu.x, uu.y}, hp2[2] = {hpp.x, hpp.y};
            f32x2 hq2[2], un2[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const f32x2 v2 = sub2(hls2[h], u2[h]);
              float t0, t1, v0, v1;
              unpack2(mul2(v2, rc2), t0, t1);
              t0 = fminf(fmaxf(t0, L.fast_lo), L.fast_hi);
              t1 = fminf(fmaxf(t1, L.fast_lo), L.fast_hi);
              const f32x2 tc2 = pack2(t0, t1);
              const f32x2 k2 = add2(add2(tc2, magic), nmagic);
              float c0, c1, r0, r1;
              unpack2(k2, c0, c1);
              unpack2(sub2(tc2, k2), r0, r1);
              c0 = copysignf(c0, t0);   // rint keeps the sign of a quotient in (-0.5, 0); the magic sum returns +0
              c1 = copysignf(c1, t1);
              if (!(fmaxf(fabsf(r0), fabsf(r1)) <= L.fast_thr)) {   // rare: too close to a rounding boundary
                unpack2(v2, v0, v1);
                if (!(fabsf(r0) <= L.fast_thr)) c0 = code_exact(v0, qp.scale, L);
                if (!(fabsf(r1) <= L.fast_thr)) c1 = code_exact(v1, qp.scale, L);
              }
              if (p.codes != nullptr) {
                p.codes[eb[b] + 2 * h] = (int8_t)c0;
                p.codes[eb[b] + 2 * h + 1] = (int8_t)c1;
              }
              const f32x2 hq = fma2(pack2(c0, c1), sc2, nz2);            // H = Q(H_ls - U)   (:59)
              const f32x2 d1 = sub2(hq, hls2[h]);
              const f32x2 un = add2(u2[h], d1);                         // U += H - H_ls     (:60)
              const f32x2 d2 = sub2(hq, hp2[h]);
              a0 = fma2(d1, d1, a0);   // sum (H - H_ls)^2     (:62)
              a1 = fma2(hq, hq, a1);   // sum H^2
              a2 = fma2(d2, d2, a2);   // sum (H - H_prev)^2   (:63)
              a3 = fma2(un, un, a3);   // sum U^2
              hq2[h] = hq;
              un2[h] = un;
            }
            ulonglong2 ho, uo;
            ho.x = hq2[0]; ho.y = hq2[1];
            uo.x = un2[0]; uo.y = un2[1];
            reinterpret_cast<ulonglong2*>(p.Hp)[gg[b]] = ho;
            reinterpret_cast<ulonglong2*>(p.Up)[gg[b]] = uo;
            if constexpr (TCBN != kDiagP1) {
              const f32x2 rho2 = pack2(rho, rho);
              const ulonglong2 ff = *reinterpret_cast<const ulonglong2*>(&fv4[b]);
              ulonglong2 ro;
              ro.x = add2(ff.x, fma2(rho2, add2(hq2[0], un2[0]), nz2));   // F + rho * (H + U), the product rounded on its own
              ro.y = add2(ff.y, fma2(rho2, add2(hq2[1], un2[1]), nz2));
              reinterpret_cast<ulonglong2*>(p.RHS)[gg[b]] = ro;
            }
          } else if (gg[b] < g1) {
            const float hls[4] = {hls4[b].x, hls4[b].y, hls4[b].z, hls4[b].w};
            const float u[4] = {u4[b].x, u4[b].y, u4[b].z, u4[b].w};
            const float hp[4] = {hp4[b].x, hp4[b].y, hp4[b].z, hp4[b].w};
            float hq4[4], un4[4], rhs4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float v = sub_rn(hls[q], u[q]);
              float code = 0.0f, hq;                                               // H = Q(H_ls - U)   (:59)
              if (fast_code) {
                const float tq = fminf(fmaxf(mul_rn(v, rcp_scale), L.fast_lo), L.fast_hi);
                code = sub_rn(add_rn(tq, 12582912.0f), 12582912.0f);
                const bool near_tie = !(fabsf(sub_rn(tq, code)) <= L.fast_thr);
                code = copysignf(code, tq);  // rint keeps the sign of a quotient in (-0.5, 0); the magic sum returns +0
                if (near_tie) code = code_exact(v, qp.scale, L);
                hq = mul_rn(code, qp.scale);
              } else if constexpr (G == kGridE2M1) {
                hq = degenerate ? qnan : e2m1_quantize(v, qp.scale, code);
              } else if constexpr (G == kGridFP) {
                hq = degenerate ? qnan : fp_quantize(v, qp.scale, L.fmt, code);
              } else {
                hq = degenerate ? qnan : quantize_value(v, qp, L, code);
              }
              const float d1 = sub_rn(hq, hls[q]);
              float un = add_rn(u[q], d1);                                         // U += H - H_ls     (:60)
              const float d2 = sub_rn(hq, hp[q]);
              if (q < nvb[b]) {
                f0 = fmaf(d1, d1, f0);  // sum (H - H_ls)^2     (:62)
                f1 = fmaf(hq, hq, f1);  // sum H^2
                f2 = fmaf(d2, d2, f2);  // sum (H - H_prev)^2   (:63)
                f3 = fmaf(un, un, f3);  // sum U^2
                if (p.codes != nullptr) p.codes[eb[b] + q] = (int8_t)code;
              } else {                  // pad column: stays zero
                hq = 0.0f;
                un = 0.0f;
              }
              hq4[q] = hq;
              un4[q] = un;
            }
            reinterpret_cast<float4*>(p.Hp)[gg[b]] = make_float4(hq4[0], hq4[1], hq4[2], hq4[3]);
            reinterpret_cast<float4*>(p.Up)[gg[b]] = make_float4(un4[0], un4[1], un4[2], un4[3]);
            if constexpr (TCBN != kDiagP1) {
              const float fv[4] = {fv4[b].x, fv4[b].y, fv4[b].z, fv4[b].w};
#pragma unroll
              for (int q = 0; q < 4; ++q) rhs4[q] = (q < nvb[b]) ? add_rn(fv[q], mul_rn(rho, add_rn(hq4[q], un4[q]))) : 0.0f;
              reinterpret_cast<float4*>(p.RHS)[gg[b]] = make_float4(rhs4[0], rhs4[1], rhs4[2], rhs4[3]);
            }
          }
        }
        {
          float e, o;
          unpack2(a0, e, o); f0 = add_rn(f0, add_rn(e, o));
          unpack2(a1, e, o); f1 = add_rn(f1, add_rn(e, o));
          unpack2(a2, e, o); f2 = add_rn(f2, add_rn(e, o));
          unpack2(a3, e, o); f3 = add_rn(f3, add_rn(e, o));
        }
        sums[0] += (double)f0;
        sums[1] += (double)f1;
        sums[2] += (double)f2;
        sums[3] += (double)f3;
      }
    }
    if (degenerate) {  // uniform: the reference would carry NaN through every remaining iteration
      rep.status |= ADMMQ_ST_NONFINITE;
      rep.r = qnan;
      rep.s = qnan;
      break;
    }
    cta_sum4(sums, sm.res);
    if (t < 4) p.slots[(size_t)blockIdx.x * 4 + t] = sums[t];
    bar.sync();
    lap(2);
    pending = true;   // r, s of this iteration: tested after the next P1, or below when this was the last iteration
  }
  if (pending && residuals_below_eps()) rep.status |= ADMMQ_ST_CONVERGED;
  // the caller's dense H and U (every CTA copies the groups it updated itself in P3: no barrier needed)
  if (p.max_iter > 1) {
    ADMMQ_GROUP_WALK();
    unsigned int row = grow0, cg = gcol0;
    for (unsigned int g = g0 + (unsigned int)t; g < g1; g += kThreads) {
      const int nv = (cg == gpr - 1) ? last_valid : 4;
      const size_t e = (size_t)row * R + 4 * cg;
      const float4 h4 = reinterpret_cast<const float4*>(p.Hp)[g], u4 = reinterpret_cast<const float4*>(p.Up)[g];
      const float h[4] = {h4.x, h4.y, h4.z, h4.w}, u[4] = {u4.x, u4.y, u4.z, u4.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (q < nv) {
          p.H[e + q] = h[q];
          p.U[e + q] = u[q];
        }
      }
      row += gdrow;
      cg += gdcol;
      if (cg >= gpr) {
        cg -= gpr;
        ++row;
      }
    }
  }
#undef ADMMQ_GROUP_WALK
  rep.phase_ns[3] = global_ns() - t_begin;
  if (blockIdx.x == 0 && t == 0) *p.report = rep;
  if constexpr (TCBN > 0) tc::pipe_teardown(pipe);
}

// ------------------------------------------------------------------------------------ host side
struct LoopLayout {  // workspace of admmq_admm_loop
  size_t header, cand, slots, hls, rhs, v, hp, up, fp, minv_hi, minv_lo, total;
  int Rp;
};

static LoopLayout loop_layout(int I, int R, int grid, bool with_minv_parts = true) {
  LoopLayout l;
  l.Rp = (R + 3) / 4 * 4;
  size_t off = 0;
  auto take = [&off](size_t bytes) {
    const size_t o = off;
    off += align_up(bytes, 256);
    return o;
  };
  l.header = take(sizeof(LoopHeader));
  l.cand = take((size_t)kKeySlots * kMaxCandidates * sizeof(unsigned long long));
  l.slots = take((size_t)grid * 4 * sizeof(double));
  l.rhs = take((size_t)I * l.Rp * sizeof(float));
  l.hls = take((size_t)I * l.Rp * sizeof(float));
  l.v = take((size_t)I * R * sizeof(float));
  l.hp = take((size_t)I * l.Rp * sizeof(float));
  l.up = take((size_t)I * l.Rp * sizeof(float));
  l.fp = take(with_minv_parts ? (size_t)I * l.Rp * sizeof(float) : 0);   // not used by the two-block splitting
  l.minv_hi = take(with_minv_parts ? (size_t)R * l.Rp * sizeof(float) : 0);
  l.minv_lo = take(with_minv_parts ? (size_t)R * l.Rp * sizeof(float) : 0);
  l.total = off;
  return l;
}

struct IterationLayout {  // workspace of admmq_admm_iteration = scalars + Minv + inverse scratch + loop workspace
  size_t header, minv, minv64, inv_ws, loop_ws, total;
};

static size_t spd_scratch_bytes(int R) {
  const size_t Rb = (size_t)((R + kNB - 1) / kNB) * kNB;
  return 2 * align_up(Rb * Rb * sizeof(double), 256);
}

static IterationLayout iteration_layout(int I, int R, int grid) {
  IterationLayout l;
  const int Rp = (R + 3) / 4 * 4;
  size_t off = 0;
  auto take = [&off](size_t bytes) {
    const size_t o = off;
    off += align_up(bytes, 256);
    return o;
  };
  l.header = take(sizeof(IterationHeader));
  l.minv = take((size_t)R * Rp * sizeof(float));
  l.minv64 = take((size_t)R * Rp * sizeof(double));
  l.inv_ws = take(spd_scratch_bytes(R));
  l.loop_ws = take(loop_layout(I, R, grid).total);
  l.total = off;
  return l;
}

// experiment knob / default of LoopParams::direct_below
static int direct_below_default() {
  static const int v = getenv("ADMMQ_DIRECT_BELOW") ? atoi(getenv("ADMMQ_DIRECT_BELOW")) : 0;
  return v;
}

constexpr int kTileFixed = 16;   // cost of a tensor-core tile that does not depend on its width, in columns of width
                                 // (measured per tile at K = 1141: 10.5 / 15.3 / 23 / 32 us at 32 / 48 / 80 / 128 columns)
constexpr int kMaxGrid = 1024;  // workspaces are sized for any cooperative grid up to this many CTAs

static int coop_grid(const DeviceProps& dp, int max_ctas) {
  return (max_ctas > 0 && max_ctas < dp.sm_count) ? max_ctas : dp.sm_count;
}

static int launch_spd_inverse(const float* G, int R, float* Minv, double* Minv64, int ldm, float* rho_out, int* status,
                              unsigned int* barrier, double* Lw, double* Xw, int grid, cudaStream_t stream) {
  InvParams ip;
  ip.G = G;
  ip.R = R;
  ip.nb = (R + kNB - 1) / kNB;
  ip.Rb = ip.nb * kNB;
  ip.ldm = ldm;
  ip.Lw = Lw;
  ip.Xw = Xw;
  ip.Minv = Minv;
  ip.Minv64 = Minv64;
  ip.rho_out = rho_out;
  ip.status = status;
  ip.barrier = barrier;
  void* args[] = {&ip};
  ADMMQ_CUDA_OK(cudaLaunchCooperativeKernel((const void*)k_spd_inverse, dim3(grid), dim3(kInvThreads), args, 0, stream));
  count_launches(1);
  return ADMMQ_OK;
}

// tile shape for P1: minimise waves * tile cost (relative FFMA efficiencies measured on B200)
static int pick_tile(int I, int R, int grid) {
  const int bm[3] = {64, 32, 16}, bn[3] = {64, 32, 32};
  const double eff[3] = {1.0, 0.55, 0.40};
  int best = 0;
  double best_cost = 1e300;
  for (int c = 0; c < 3; ++c) {
    const long long tiles = (long long)((I + bm[c] - 1) / bm[c]) * ((R + bn[c] - 1) / bn[c]);
    const long long waves = (tiles + grid - 1) / grid;
    const double cost = (double)waves * bm[c] * bn[c] / eff[c];
    if (cost < best_cost) {
      best_cost = cost;
      best = c;
    }
  }
  return best;
}

static int check_loop_args(const char* who, const void* H, const void* U, const void* F, const void* M, const void* report,
                           int I, int R, int bits, int qscheme, int num_attempts) {
  if (H == nullptr || U == nullptr || F == nullptr || M == nullptr || report == nullptr || I <= 0 || R <= 0)
    return fail(ADMMQ_E_BADARG, "%s: null pointer or empty shape", who);
  if (bits < 1 || bits > 8) return fail(ADMMQ_E_BADARG, "%s: bits must be in 1..8, got %d", who, bits);
  if (!known_scheme(qscheme)) return fail(ADMMQ_E_BADARG, "%s: unknown qscheme %d", who, qscheme);
  if (int e = check_scheme_bits(who, qscheme, bits)) return e;
  if (has_clip_search(qscheme) && (num_attempts < 1 || num_attempts > kMaxCandidates))
    return fail(ADMMQ_E_BADARG, "%s: num_attempts must be in 1..%d", who, kMaxCandidates);
  if ((long long)I * ((R + 3) / 4 * 4) >= (1ll << 31)) return fail(ADMMQ_E_UNSUPPORTED, "%s: I * (R rounded up to 4) must be < 2^31", who);
  return ADMMQ_OK;
}

// The loop kernel of a call: one decision for launch_loop and admmq_admm_loop_kernel (include/admmq.h lists the ids).
static int select_loop_kernel(int I, int R, int num_attempts, int precision, int grid) {
  const int Rp = (R + 3) / 4 * 4;
  static const bool no_resident = getenv("ADMMQ_NO_RESIDENT") != nullptr;  // diagnostics: force the general kernel
  static const bool no_cluster = getenv("ADMMQ_NO_CLUSTER") != nullptr;    // diagnostics: never take the cluster kernel
  static const bool no_tap = getenv("ADMMQ_NO_TAP") != nullptr;            // diagnostics: never take the tap-factor cluster kernel
  const int ccl = (precision != 0 && !no_resident && !no_cluster && grid >= 4) ? cluster_ctas_for(I, R, Rp, num_attempts, grid) : 0;
  if ((grid == 1 || ccl >= 4) && precision != 0 && !no_resident && resident_fits(I, R, Rp, num_attempts)) {
    // a small factor: the shared-memory-resident loop on one CTA (admm_loop_resident.cuh) or, with a budget of at
    // least four CTAs, on a thread-block cluster that splits rows and clip candidates (admm_loop_cluster.cuh)
    if (ccl == 8) return ADMMQ_LOOP_CLUSTER8;
    if (ccl == 4) return ADMMQ_LOOP_CLUSTER4;
    return ADMMQ_LOOP_RESIDENT;
  }
  // the tap factor of a wide convolution (9 x R): one cluster of 8 CTAs, columns and clip candidates split (admm_loop_tap.cuh)
  if (precision != 0 && !no_tap && !no_cluster && tap_cluster_fits(I, R, Rp, num_attempts, grid)) return ADMMQ_LOOP_TAP;
  if (precision == 0)  // parity mode: float64-accumulating tiles against the float64 inverse
    return pick_tile(I, R, grid) == 0 ? ADMMQ_LOOP_F64_64 : ADMMQ_LOOP_F64_32;
  if (I <= 16 && (long long)I * Rp <= SkinnySmem<16>::kRhsFloats) return I <= 9 ? ADMMQ_LOOP_SKINNY9 : ADMMQ_LOOP_SKINNY16;
  // tensor-core P1 only pays off when the factor has enough rows to fill a good part of a 128-row tile
  if (precision == 1 && I >= 64 && R >= 32) {
    const int tilesM = (I + tc::kTileM - 1) / tc::kTileM;
    // tile width (multiple of 16): a tile costs a fixed part (fill, drain, epilogue set-up) plus bn columns of
    // tensor-core work; minimise waves * (kTileFixed + bn), ties go to the wider tile.  Widths above 128 (one
    // accumulator, shallower raw ring: ~5 % dearer per column) exist for the wave structure: 4 x 8 tiles of width 144
    // cover 512 x 1141 in ONE wave on 32 .. 35 CTAs where 4 x 9 of width 128 need two
    int tcbn = kLoopPS ? 128 : 64;
    long long best = -1;
    for (int bn = (kLoopPS ? 160 : 64); bn >= 16; bn -= 16) {
      const long long tiles = (long long)tilesM * ((R + bn - 1) / bn);
      const long long cost = ((tiles + grid - 1) / grid) * (kTileFixed + bn) * (bn > 128 ? 105 : 100);
      if (best < 0 || cost < best) {
        best = cost;
        tcbn = bn;
      }
    }
    static const int force_bn = getenv("ADMMQ_LOOP_BN") ? atoi(getenv("ADMMQ_LOOP_BN")) : 0;   // experiment knob
    if (force_bn >= 16 && force_bn <= (kLoopPS ? 160 : 64) && (force_bn & 15) == 0) tcbn = force_bn;
    return ADMMQ_LOOP_TC + tcbn;
  }
  switch (pick_tile(I, R, grid)) {
    case 0: return ADMMQ_LOOP_FFMA64;
    case 1: return ADMMQ_LOOP_FFMA32;
    default: return ADMMQ_LOOP_FFMA16;
  }
}

// the instantiation of a kernel for a scheme's grid (grid_of)
template <class F>
static F by_grid(Grid g, F int_grid, F e2m1, F fp) {
  return g == kGridE2M1 ? e2m1 : g == kGridFP ? fp : int_grid;
}

// kernel function and dynamic shared memory of a general loop kernel id (not the shared-memory kernels)
template <Grid G>
static void general_kernel(int kid, const void** fn, size_t* smem) {
  switch (kid) {
    case ADMMQ_LOOP_F64_64: *fn = (const void*)k_admm_loop<64, 64, 4, 4, kF64P1, G>; *smem = sizeof(LoopSmem<64, 64, kF64P1>); break;
    case ADMMQ_LOOP_F64_32: *fn = (const void*)k_admm_loop<32, 32, 2, 2, kF64P1, G>; *smem = sizeof(LoopSmem<32, 32, kF64P1>); break;
    case ADMMQ_LOOP_SKINNY9: *fn = (const void*)k_admm_loop<16, 32, 1, 2, -9, G>; *smem = sizeof(LoopSmem<16, 32, -9>); break;
    case ADMMQ_LOOP_SKINNY16: *fn = (const void*)k_admm_loop<16, 32, 1, 2, -16, G>; *smem = sizeof(LoopSmem<16, 32, -16>); break;
    case ADMMQ_LOOP_FFMA64: *fn = (const void*)k_admm_loop<64, 64, 4, 4, 0, G>; *smem = sizeof(LoopSmem<64, 64, 0>); break;
    case ADMMQ_LOOP_FFMA32: *fn = (const void*)k_admm_loop<32, 32, 2, 2, 0, G>; *smem = sizeof(LoopSmem<32, 32, 0>); break;
    case ADMMQ_LOOP_FFMA16: *fn = (const void*)k_admm_loop<16, 32, 1, 2, 0, G>; *smem = sizeof(LoopSmem<16, 32, 0>); break;
    default: {  // ADMMQ_LOOP_TC + tile width
      const int tcbn = kid - ADMMQ_LOOP_TC;
      if (tcbn > 128) {
        *fn = (const void*)k_admm_loop<16, 32, 1, 2, (kLoopPS ? 160 : 64), G>;
        *smem = sizeof(LoopSmem<16, 32, (kLoopPS ? 160 : 64)>);
      } else if (tcbn > 64) {
        *fn = (const void*)k_admm_loop<16, 32, 1, 2, (kLoopPS ? 128 : 64), G>;
        *smem = sizeof(LoopSmem<16, 32, (kLoopPS ? 128 : 64)>);
      } else if (tcbn > 32) {
        *fn = (const void*)k_admm_loop<16, 32, 1, 2, 64, G>;
        *smem = sizeof(LoopSmem<16, 32, 64>);
      } else if (tcbn > 16) {
        *fn = (const void*)k_admm_loop<16, 32, 1, 2, 32, G>;
        *smem = sizeof(LoopSmem<16, 32, 32>);
      } else {
        *fn = (const void*)k_admm_loop<16, 32, 1, 2, 16, G>;
        *smem = sizeof(LoopSmem<16, 32, 16>);
      }
    }
  }
}

// one launch of a shared-memory loop kernel on a thread-block cluster of `ctas` CTAs (the whole grid)
static int launch_cluster(void (*kernel)(ResidentParams), int ctas, size_t smem, const ResidentParams& rp, cudaStream_t stream) {
  ADMMQ_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(ctas);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = ctas;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  ADMMQ_CUDA_OK(cudaLaunchKernelEx(&cfg, kernel, rp));
  count_launches(1);
  return ADMMQ_OK;
}

static int launch_loop(float* H, float* U, const float* F, const float* Minv, const double* Minv64, const float* rho,
                       const int* inv_status, int I, int R, int max_iter, float eps, int bits, int qscheme, int num_attempts, int precision,
                       int8_t* codes, admmq_loop_report* report, char* ws, int grid, cudaStream_t stream) {
  const LoopLayout l = loop_layout(I, R, grid);
  const int kid = select_loop_kernel(I, R, num_attempts, precision, grid);
  const Grid qgrid = grid_of(qscheme);
  if (kid == ADMMQ_LOOP_RESIDENT || kid == ADMMQ_LOOP_CLUSTER4 || kid == ADMMQ_LOOP_CLUSTER8 || kid == ADMMQ_LOOP_TAP) {
    ResidentParams rp;
    rp.H = H;
    rp.U = U;
    rp.F = F;
    rp.Minv = Minv;
    rp.rho = rho;
    rp.inv_status = inv_status;
    rp.I = I;
    rp.R = R;
    rp.Rp = l.Rp;
    rp.max_iter = max_iter;
    rp.eps = eps;
    rp.bits = bits;
    rp.scheme = qscheme;
    rp.Nc = has_clip_search(qscheme) ? num_attempts : 0;
    rp.codes = codes;
    rp.report = report;
    if (kid == ADMMQ_LOOP_TAP)
      return launch_cluster(by_grid(qgrid, k_admm_loop_tap<kTapMaxRows, kGridInt>, k_admm_loop_tap<kTapMaxRows, kGridE2M1>,
                                    k_admm_loop_tap<kTapMaxRows, kGridFP>),
                            kTapCtas, sizeof(TapSmem), rp, stream);
    if (kid != ADMMQ_LOOP_RESIDENT)
      return launch_cluster(by_grid(qgrid, k_admm_loop_cluster<kGridInt>, k_admm_loop_cluster<kGridE2M1>, k_admm_loop_cluster<kGridFP>),
                            kid == ADMMQ_LOOP_CLUSTER8 ? 8 : 4, sizeof(ClusterSmem), rp, stream);
    void (*resident)(ResidentParams) =
        by_grid(qgrid, k_admm_loop_resident<kGridInt>, k_admm_loop_resident<kGridE2M1>, k_admm_loop_resident<kGridFP>);
    ADMMQ_CUDA_OK(cudaFuncSetAttribute(resident, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ResidentSmem)));
    resident<<<1, kThreads, sizeof(ResidentSmem), stream>>>(rp);
    ADMMQ_CUDA_OK(cudaGetLastError());
    count_launches(1);
    return ADMMQ_OK;
  }
  // header + candidate accumulators (RHS and the working copies, pad columns included, are written by the kernel's prologue)
  ADMMQ_CUDA_OK(cudaMemsetAsync(ws, 0, l.slots, stream));
  LoopParams p;
  p.H = H;
  p.U = U;
  p.F = F;
  p.I = I;
  p.R = R;
  p.Rp = l.Rp;
  p.max_iter = max_iter;
  p.eps = eps;
  p.bits = bits;
  p.scheme = qscheme;
  p.Nc = has_clip_search(qscheme) ? num_attempts : 0;
  p.neg_zero = -0.0f;
  p.direct_below = direct_below_default();
  p.codes = codes;
  p.report = report;
  p.rho = rho;
  p.inv_status = inv_status;
  p.hdr = (LoopHeader*)(ws + l.header);
  p.cand = (unsigned long long*)(ws + l.cand);
  p.slots = (double*)(ws + l.slots);
  p.Hls = (float*)(ws + l.hls);
  p.V = (float*)(ws + l.v);
  p.RHS = (float*)(ws + l.rhs);
  p.Hp = (float*)(ws + l.hp);
  p.Up = (float*)(ws + l.up);
  p.Fp = (float*)(ws + l.fp);
  p.Minv = Minv;
  p.Minv64 = Minv64;
  p.MinvHi = (float*)(ws + l.minv_hi);
  p.MinvLo = (float*)(ws + l.minv_lo);
  p.tc_bn = 0;
  void* args[] = {&p};
  const void* fn = nullptr;
  size_t smem = 0;
  if (kid < ADMMQ_LOOP_TC) {
    memset(&p.tm_rhs, 0, sizeof(CUtensorMap));
    memset(&p.tm_minv_hi, 0, sizeof(CUtensorMap));
    memset(&p.tm_minv_lo, 0, sizeof(CUtensorMap));
  }
  if (kid > ADMMQ_LOOP_TC) {
    const int tcbn = kid - ADMMQ_LOOP_TC;
    p.tc_bn = tcbn;
    if (int e = tc::make_operand_tmap(&p.tm_rhs, p.RHS, I, R, l.Rp, tc::kTileM)) return e;
    if (int e = tc::make_operand_tmap(&p.tm_minv_hi, kLoopPS ? p.MinvHi : Minv, R, R, l.Rp, tcbn)) return e;
    if (int e = tc::make_operand_tmap(&p.tm_minv_lo, kLoopPS ? p.MinvLo : Minv, R, R, l.Rp, tcbn)) return e;
  }
  if (qgrid == kGridE2M1) general_kernel<kGridE2M1>(kid, &fn, &smem);
  else if (qgrid == kGridFP) general_kernel<kGridFP>(kid, &fn, &smem);
  else general_kernel<kGridInt>(kid, &fn, &smem);
  ADMMQ_CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ADMMQ_CUDA_OK(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kThreads), args, smem, stream));
  count_launches(1);
  return ADMMQ_OK;
}

}  // namespace admmq

using namespace admmq;

extern "C" int admmq_padded_ld(int R) { return (R + 3) / 4 * 4; }

extern "C" size_t admmq_spd_inverse_workspace_bytes(int R) {
  if (R <= 0) return 0;
  return 256 + spd_scratch_bytes(R);
}

extern "C" int admmq_spd_inverse(const float* G, int R, float* Minv, double* Minv64, float* rho_out, int* status,
                                 int max_ctas, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (G == nullptr || Minv == nullptr || rho_out == nullptr || status == nullptr || R <= 0)
    return fail(ADMMQ_E_BADARG, "admmq_spd_inverse: bad argument");
  if (workspace == nullptr || workspace_bytes < admmq_spd_inverse_workspace_bytes(R) || ((uintptr_t)workspace & 255) != 0)
    return fail(ADMMQ_E_WORKSPACE, "admmq_spd_inverse: workspace too small or not 256-byte aligned");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  if (!dp.coop) return fail(ADMMQ_E_UNSUPPORTED, "device does not support cooperative launch");
  char* ws = (char*)workspace;
  ADMMQ_CUDA_OK(cudaMemsetAsync(ws, 0, 256, stream));
  ADMMQ_CUDA_OK(cudaMemsetAsync(status, 0, sizeof(int), stream));
  double* Lw = (double*)(ws + 256);
  double* Xw = (double*)(ws + 256 + spd_scratch_bytes(R) / 2);
  return launch_spd_inverse(G, R, Minv, Minv64, admmq_padded_ld(R), rho_out, status, (unsigned int*)ws, Lw, Xw, coop_grid(dp, max_ctas), stream);
}

extern "C" int admmq_admm_loop_kernel(int I, int R, int num_attempts, int precision, int grid) {
  if (I <= 0 || R <= 0 || grid <= 0 || precision < 0 || precision > 2)
    return fail(ADMMQ_E_BADARG, "admmq_admm_loop_kernel: bad argument");
  return select_loop_kernel(I, R, num_attempts, precision, grid);
}

extern "C" size_t admmq_admm_loop_workspace_bytes(int I, int R, int num_attempts) {
  (void)num_attempts;
  if (I <= 0 || R <= 0) return 0;
  return loop_layout(I, R, kMaxGrid).total;
}

extern "C" int admmq_admm_loop(float* H, float* U, const float* F, const float* Minv, const double* Minv64,
                               const float* rho, const int* inv_status, int I, int R, int max_iter, float eps, int bits, int qscheme,
                               int num_attempts, int precision, int max_ctas, int8_t* codes, admmq_loop_report* report,
                               void* workspace, size_t workspace_bytes, void* stream_) {
  if (int e = check_loop_args("admmq_admm_loop", H, U, F, Minv, report, I, R, bits, qscheme, num_attempts)) return e;
  if (rho == nullptr) return fail(ADMMQ_E_BADARG, "admmq_admm_loop: rho is null");
  if (precision < 0 || precision > 2) return fail(ADMMQ_E_BADARG, "admmq_admm_loop: precision must be 0, 1 or 2");
  if (precision == 0 && Minv64 == nullptr)
    return fail(ADMMQ_E_BADARG, "admmq_admm_loop: precision 0 (parity mode) needs the float64 inverse Minv64 of admmq_spd_inverse");
  if (((uintptr_t)Minv & 15) != 0) return fail(ADMMQ_E_BADARG, "admmq_admm_loop: Minv must be 16-byte aligned");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  if (!dp.coop) return fail(ADMMQ_E_UNSUPPORTED, "device does not support cooperative launch");
  if (workspace == nullptr || workspace_bytes < admmq_admm_loop_workspace_bytes(I, R, num_attempts) ||
      ((uintptr_t)workspace & 255) != 0)
    return fail(ADMMQ_E_WORKSPACE, "admmq_admm_loop: workspace needs %zu bytes, 256-byte aligned",
                admmq_admm_loop_workspace_bytes(I, R, num_attempts));
  return launch_loop(H, U, F, Minv, Minv64, rho, inv_status, I, R, max_iter, eps, bits, qscheme, num_attempts, precision,
                     codes, report, (char*)workspace, coop_grid(dp, max_ctas), (cudaStream_t)stream_);
}

// ---- two-block splitting W ~ W_q + W_r (scripts/factorize_lowrank.py): the quantized block's inner loop
extern "C" size_t admmq_split_loop_workspace_bytes(int64_t n, int num_attempts) {
  (void)num_attempts;
  if (n <= 0 || n >= (1ll << 31)) return 0;
  return loop_layout(1, (int)n, kMaxGrid, false).total;
}

extern "C" int admmq_split_loop(float* H, float* U, const float* W, const float* H2, int64_t n, float rho, int max_iter,
                                float eps, int bits, int qscheme, int num_attempts, int max_ctas, int8_t* codes,
                                admmq_loop_report* report, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (n <= 0 || n >= (1ll << 31)) return fail(ADMMQ_E_UNSUPPORTED, "admmq_split_loop: n must be in 1 .. 2^31-1");
  if (int e = check_loop_args("admmq_split_loop", H, U, W, H2, report, 1, (int)n, bits, qscheme, num_attempts)) return e;
  if (!(rho > 0.0f)) return fail(ADMMQ_E_BADARG, "admmq_split_loop: rho must be positive");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  if (!dp.coop) return fail(ADMMQ_E_UNSUPPORTED, "device does not support cooperative launch");
  if (workspace == nullptr || workspace_bytes < admmq_split_loop_workspace_bytes(n, num_attempts) ||
      ((uintptr_t)workspace & 255) != 0)
    return fail(ADMMQ_E_WORKSPACE, "admmq_split_loop: workspace needs %zu bytes, 256-byte aligned",
                admmq_split_loop_workspace_bytes(n, num_attempts));
  const int grid = coop_grid(dp, max_ctas);
  char* ws = (char*)workspace;
  const LoopLayout l = loop_layout(1, (int)n, grid, false);
  ADMMQ_CUDA_OK(cudaMemsetAsync(ws, 0, l.slots, stream));
  // rho lives in the (zeroed) header page: pad[] of LoopHeader is unused by the kernel
  LoopHeader* hdr = (LoopHeader*)(ws + l.header);
  ADMMQ_CUDA_OK(cudaMemcpyAsync(&hdr->pad[0], &rho, sizeof(float), cudaMemcpyHostToDevice, stream));
  LoopParams p;
  memset(&p, 0, sizeof(p));
  p.H = H;
  p.U = U;
  p.F = W;
  p.H2 = H2;
  p.I = 1;
  p.R = (int)n;
  p.Rp = l.Rp;
  p.max_iter = max_iter;
  p.eps = eps;
  p.bits = bits;
  p.scheme = qscheme;
  p.Nc = has_clip_search(qscheme) ? num_attempts : 0;
  p.neg_zero = -0.0f;
  p.codes = codes;
  p.report = report;
  p.rho = reinterpret_cast<const float*>(&hdr->pad[0]);
  p.inv_status = nullptr;
  p.hdr = hdr;
  p.cand = (unsigned long long*)(ws + l.cand);
  p.slots = (double*)(ws + l.slots);
  p.Hls = (float*)(ws + l.hls);
  p.V = (float*)(ws + l.v);
  p.Hp = (float*)(ws + l.hp);
  p.Up = (float*)(ws + l.up);
  p.Fp = nullptr;
  p.RHS = nullptr;
  p.Minv = nullptr;
  void* args[] = {&p};
  const void* fn = by_grid(grid_of(qscheme), (const void*)k_admm_loop<16, 32, 1, 2, kDiagP1, kGridInt>,
                           (const void*)k_admm_loop<16, 32, 1, 2, kDiagP1, kGridE2M1>,
                           (const void*)k_admm_loop<16, 32, 1, 2, kDiagP1, kGridFP>);
  const size_t smem = sizeof(LoopSmem<16, 32, kDiagP1>);
  ADMMQ_CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ADMMQ_CUDA_OK(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kThreads), args, smem, stream));
  count_launches(1);
  return ADMMQ_OK;
}

extern "C" size_t admmq_admm_iteration_workspace_bytes(int I, int R, int num_attempts) {
  (void)num_attempts;
  if (I <= 0 || R <= 0) return 0;
  return iteration_layout(I, R, kMaxGrid).total;
}

extern "C" int admmq_admm_iteration(float* H, float* U, const float* F, const float* G, int I, int R, int max_iter,
                                    float eps, int bits, int qscheme, int num_attempts, int precision, int max_ctas,
                                    int8_t* codes, admmq_loop_report* report, void* workspace, size_t workspace_bytes,
                                    void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (int e = check_loop_args("admmq_admm_iteration", H, U, F, G, report, I, R, bits, qscheme, num_attempts)) return e;
  if (precision < 0 || precision > 2) return fail(ADMMQ_E_BADARG, "admmq_admm_iteration: precision must be 0, 1 or 2");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  if (!dp.coop) return fail(ADMMQ_E_UNSUPPORTED, "device does not support cooperative launch");
  const int grid = coop_grid(dp, max_ctas);
  const IterationLayout l = iteration_layout(I, R, kMaxGrid);
  if (workspace == nullptr || workspace_bytes < l.total || ((uintptr_t)workspace & 255) != 0)
    return fail(ADMMQ_E_WORKSPACE, "admmq_admm_iteration: workspace needs %zu bytes, 256-byte aligned", l.total);
  char* ws = (char*)workspace;
  ADMMQ_CUDA_OK(cudaMemsetAsync(ws + l.header, 0, 256, stream));
  IterationHeader* ih = (IterationHeader*)(ws + l.header);
  float* Minv = (float*)(ws + l.minv);
  double* Minv64 = precision == 0 ? (double*)(ws + l.minv64) : nullptr;
  if (int e = launch_spd_inverse(G, R, Minv, Minv64, admmq_padded_ld(R), &ih->rho, &ih->status, &ih->barrier_inv,
                                 (double*)(ws + l.inv_ws), (double*)(ws + l.inv_ws + spd_scratch_bytes(R) / 2), grid, stream))
    return e;
  return launch_loop(H, U, F, Minv, Minv64, &ih->rho, &ih->status, I, R, max_iter, eps, bits, qscheme, num_attempts,
                     precision, codes, report, ws + l.loop_ws, grid, stream);
}
