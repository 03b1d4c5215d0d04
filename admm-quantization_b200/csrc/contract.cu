// contract.cu - the per-sweep dense contractions in PARITY mode (float64 accumulation on
// CUDA cores): Gram-Hadamard, mode-n unfolding, MTTKRP and the reconstruction error.
// Reference call sites: scripts/factorize.py:215-217, 226-227, 236-237, 246-253 (3-D) and
// :276-277, 286-287, 296-297 (2-D); source/admm.py:14-15; source/utils.py:60-74.
//
// These run 3 (+2) times per outer sweep against 3 x 999 inner iterations, i.e. < 1 % of the
// time; accumulating in float64 makes F and G the correctly rounded float32 values of the exact
// contraction, which is what keeps the solver on the reference's trajectory (SURVEY App. E.2).
// The 3xTF32 tcgen05 MTTKRP (throughput mode) lives in mttkrp_tc.cu.
#include <algorithm>
#include "common.cuh"
#include "numerics.cuh"

namespace admmq {

constexpr int kCT = 256;  // threads per CTA
constexpr int kBK = 16;   // depth of one shared-memory slab

// ---------------------------------------------------------------------------- Gram-Hadamard
// G[a,b] = fl32(sum_k U1[k,a] U1[k,b]) * fl32(sum_k U2[k,a] U2[k,b]); 32x32 outputs per CTA.
// T = float: the solver's Gram (each Gram rounded to float32 before the float32 Hadamard product, like the reference's
// float32 matmuls); T = double: the ALS / EPC initialisation (source/parafac_epc.py runs in float64), everything double.
template <typename T>
__global__ void __launch_bounds__(kCT) k_gram_hadamard(const T* __restrict__ U1, int n1,
                                                      const T* __restrict__ U2, int n2, int R,
                                                      T* __restrict__ G) {
  __shared__ double sa[kBK][33], sb[kBK][33];
  const int a0 = blockIdx.y * 32, b0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8; each thread: rows ty, ty+8, ty+16, ty+24
  T prod[4] = {(T)1, (T)1, (T)1, (T)1};
  for (int m = 0; m < 2; ++m) {
    const T* U = (m == 0) ? U1 : U2;
    const int n = (m == 0) ? n1 : n2;
    if (U == nullptr) continue;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int k0 = 0; k0 < n; k0 += kBK) {
      __syncthreads();
      for (int i = threadIdx.x; i < kBK * 32; i += kCT) {
        const int kk = i >> 5, c = i & 31;
        const int k = k0 + kk;
        sa[kk][c] = (k < n && a0 + c < R) ? (double)U[(size_t)k * R + a0 + c] : 0.0;
        sb[kk][c] = (k < n && b0 + c < R) ? (double)U[(size_t)k * R + b0 + c] : 0.0;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < kBK; ++kk) {
        const double bv = sb[kk][tx];
#pragma unroll
        for (int r = 0; r < 4; ++r) acc[r] = fma(sa[kk][ty + 8 * r], bv, acc[r]);
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if constexpr (sizeof(T) == 4) prod[r] = (m == 0) ? (float)acc[r] : mul_rn((float)prod[r], (float)acc[r]);
      else prod[r] = (m == 0) ? acc[r] : prod[r] * acc[r];
    }
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int a = a0 + ty + 8 * r, b = b0 + tx;
    if (a < R && b < R) G[(size_t)a * R + b] = prod[r];
  }
}

// ---------------------------------------------------------------------------- unfolding
__global__ void __launch_bounds__(kCT) k_unfold3(const float* __restrict__ W, int I, int J, int K, int mode,
                                                float* __restrict__ out) {
  const long long n = (long long)I * J * K;
  for (long long o = (long long)blockIdx.x * kCT + threadIdx.x; o < n; o += (long long)gridDim.x * kCT) {
    long long i, j, k;
    if (mode == 0) {
      i = o / ((long long)J * K); j = (o / K) % J; k = o % K;
    } else if (mode == 1) {  // (J, I, K)
      j = o / ((long long)I * K); i = (o / K) % I; k = o % K;
    } else {                 // (K, I, J)
      k = o / ((long long)I * J); i = (o / J) % I; j = o % J;
    }
    out[o] = W[(i * J + j) * K + k];
  }
}

// ---------------------------------------------------------------------------- MTTKRP (float64 accumulate)
// F[m, r] = sum_p Wn[m, p] * X[p / ny, r] * Y[p % ny, r]; tile BM x 64, split over p into gridDim.z slices.
// TI / TO = float: the solver's parity-mode MTTKRP (float32 operands, result = correctly rounded float32 of the exact
// contraction); TI = TO = double: the ALS / EPC initialisation - the Khatri-Rao operand is formed on the fly from the two
// factors, never materialised (source/parafac_epc.py via tensorly's unfolding_dot_khatri_rao builds (I J) x R in memory).
template <int BM, typename TI, typename TO>
__global__ void __launch_bounds__(kCT) k_mttkrp_f64(const TI* __restrict__ Wn, int M, long long P,
                                                   const TI* __restrict__ X, const TI* __restrict__ Y,
                                                   int ny, int R, long long p_per_split,
                                                   double* __restrict__ partial, TO* __restrict__ F) {
  constexpr int BN = 64;
  constexpr int TM = BM / 16;  // rows per thread (16 x 16 thread grid); thread tx owns the columns tx, tx + 16, tx + 32, tx + 48:
                               // a half warp reads 16 consecutive doubles of the Khatri-Rao slab (tx * 4 + b was a 4-way bank
                               // conflict: 0.556 -> 0.435 ms on the 512 x 4608 x 1141 float64 MTTKRP; same sums, same order)
  __shared__ double sw[kBK][BM + 1], skr[kBK][BN + 2];
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const long long pb = (long long)blockIdx.z * p_per_split, pe = min(P, pb + p_per_split);
  double acc[TM][4];
#pragma unroll
  for (int a = 0; a < TM; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
  for (long long p0 = pb; p0 < pe; p0 += kBK) {
    __syncthreads();
    for (int i = threadIdx.x; i < BM * kBK; i += kCT) {
      const int row = i / kBK, kk = i % kBK;
      const long long p = p0 + kk;
      sw[kk][row] = (m0 + row < M && p < pe) ? (double)Wn[(size_t)(m0 + row) * P + p] : 0.0;
    }
    for (int i = threadIdx.x; i < BN * kBK; i += kCT) {
      const int kk = i / BN, c = i % BN;
      const long long p = p0 + kk;
      double v = 0.0;
      if (p < pe && n0 + c < R) {
        const long long xi = p / ny;
        v = (double)X[(size_t)xi * R + n0 + c];
        if (Y != nullptr) v *= (double)Y[(size_t)(p - xi * ny) * R + n0 + c];
      }
      skr[kk][c] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kBK; ++kk) {
      double bv[4];
#pragma unroll
      for (int b = 0; b < 4; ++b) bv[b] = skr[kk][tx + 16 * b];
#pragma unroll
      for (int a = 0; a < TM; ++a) {
        const double av = sw[kk][ty * TM + a];
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = fma(av, bv[b], acc[a][b]);
      }
    }
  }
#pragma unroll
  for (int a = 0; a < TM; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int m = m0 + ty * TM + a, r = n0 + tx + 16 * b;
      if (m < M && r < R) {
        if (gridDim.z == 1) F[(size_t)m * R + r] = (TO)acc[a][b];
        else partial[((size_t)blockIdx.z * M + m) * R + r] = acc[a][b];
      }
    }
}

template <typename TO>
__global__ void __launch_bounds__(kCT) k_sum_partials(const double* __restrict__ partial, int splits, long long n,
                                                     TO* __restrict__ F) {
  for (long long i = (long long)blockIdx.x * kCT + threadIdx.x; i < n; i += (long long)gridDim.x * kCT) {
    double s = 0.0;
    for (int z = 0; z < splits; ++z) s += partial[(size_t)z * n + i];  // fixed order
    F[i] = (TO)s;
  }
}

// ---------------------------------------------------------------------------- reconstruction error
// tile (64 rows of A) x (64 columns p of the mode-0 unfolding); the reconstruction element is the
// float32 rounding of the float64 inner product (torch.einsum's output dtype), the difference and
// its square are float32 (source/admm.py:15), the two sums are float64 per CTA, reduced in fixed order.
__global__ void __launch_bounds__(kCT) k_recon_error(const float* __restrict__ W0, int M, long long P,
                                                    const float* __restrict__ A, const float* __restrict__ X,
                                                    const float* __restrict__ Y, int ny, int R,
                                                    double* __restrict__ cta_sums) {
  constexpr int BM = 64, BN = 64;
  __shared__ double sa[kBK][BM + 1], skr[kBK][BN + 1];
  __shared__ double red[2][kCT / 32];
  const int m0 = blockIdx.y * BM;
  const long long q0 = (long long)blockIdx.x * BN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
  for (int r0 = 0; r0 < R; r0 += kBK) {
    __syncthreads();
    for (int i = threadIdx.x; i < BM * kBK; i += kCT) {
      const int row = i / kBK, kk = i % kBK;
      sa[kk][row] = (m0 + row < M && r0 + kk < R) ? (double)A[(size_t)(m0 + row) * R + r0 + kk] : 0.0;
    }
    for (int i = threadIdx.x; i < BN * kBK; i += kCT) {
      const int c = i / kBK, kk = i % kBK;
      const long long p = q0 + c;
      double v = 0.0;
      if (p < P && r0 + kk < R) {
        const long long xi = p / ny;
        v = (double)X[(size_t)xi * R + r0 + kk];
        if (Y != nullptr) v *= (double)Y[(size_t)(p - xi * ny) * R + r0 + kk];
      }
      skr[kk][c] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kBK; ++kk) {
      double bv[4];
#pragma unroll
      for (int b = 0; b < 4; ++b) bv[b] = skr[kk][tx * 4 + b];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const double av = sa[kk][ty * 4 + a];
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = fma(av, bv[b], acc[a][b]);
      }
    }
  }
  double num = 0.0, den = 0.0;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int m = m0 + ty * 4 + a;
      const long long p = q0 + tx * 4 + b;
      if (m < M && p < P) {
        const float w = W0[(size_t)m * P + p];
        const float d = sub_rn(w, (float)acc[a][b]);
        num += (double)mul_rn(d, d);
        den += (double)mul_rn(w, w);
      }
    }
  num = warp_sum(num);
  den = warp_sum(den);
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = num;
    red[1][threadIdx.x >> 5] = den;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double n2 = 0.0, d2 = 0.0;
    for (int w = 0; w < kCT / 32; ++w) {
      n2 += red[0][w];
      d2 += red[1][w];
    }
    const size_t cta = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
    cta_sums[2 * cta] = n2;
    cta_sums[2 * cta + 1] = d2;
  }
}

__global__ void __launch_bounds__(kCT) k_sum_pairs(const double* __restrict__ cta_sums, long long ctas,
                                                  double* __restrict__ out2) {
  __shared__ double red[2][kCT];
  double n = 0.0, d = 0.0;
  for (long long i = threadIdx.x; i < ctas; i += kCT) {  // fixed assignment, fixed order
    n += cta_sums[2 * i];
    d += cta_sums[2 * i + 1];
  }
  red[0][threadIdx.x] = n;
  red[1][threadIdx.x] = d;
  __syncthreads();
  for (int s = kCT / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      red[0][threadIdx.x] += red[0][threadIdx.x + s];
      red[1][threadIdx.x] += red[1][threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out2[0] = red[0][0];
    out2[1] = red[1][0];
  }
}

int select_mttkrp_kernel(int M, int nx, int ny, int R, int precision, int sms, int* grid, int* splits);  // tc_gemm.cu

template <typename TI, typename TO>
static int launch_mttkrp_f64(const TI* Wn, int M, const TI* X, int nx, const TI* Y, int ny, int R, TO* F, void* workspace,
                             size_t workspace_bytes, cudaStream_t stream) {
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  const long long P = (long long)nx * ny;
  int splits;
  const int bm = select_mttkrp_kernel(M, nx, ny, R, 0, dp.sm_count, nullptr, &splits) == ADMMQ_MTTKRP_F64_16 ? 16 : 64;
  // without room for the partials (admmq_mttkrp_workspace_bytes) the sum over p runs in one slice
  if (splits > 1 && (workspace == nullptr || workspace_bytes < (size_t)splits * M * R * sizeof(double))) splits = 1;
  const long long per = ((P + splits - 1) / splits + kBK - 1) / kBK * kBK;
  dim3 grid((R + 63) / 64, (M + bm - 1) / bm, splits);
  if (bm == 16) k_mttkrp_f64<16, TI, TO><<<grid, kCT, 0, stream>>>(Wn, M, P, X, Y, ny, R, per, (double*)workspace, F);
  else k_mttkrp_f64<64, TI, TO><<<grid, kCT, 0, stream>>>(Wn, M, P, X, Y, ny, R, per, (double*)workspace, F);
  if (splits > 1) {
    const long long n = (long long)M * R;
    k_sum_partials<TO><<<(int)std::min<long long>((n + kCT - 1) / kCT, 148 * 8), kCT, 0, stream>>>((const double*)workspace,
                                                                                                splits, n, F);
  }
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(splits > 1 ? 2 : 1);
  return ADMMQ_OK;
}

// Column 2-norms of an n x R float64 factor (one warp-wide column strip of 32 columns per CTA, 8 row groups summed in
// fixed order); a zero norm is reported as 1 (the column is left alone, like the restated cp_anc does).
__global__ void __launch_bounds__(kCT) k_column_norms(const double* __restrict__ U, int n, int R, double* __restrict__ norms) {
  __shared__ double red[kCT / 32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  double s = 0.0;
  if (c < R)
    for (int k = ty; k < n; k += kCT / 32) {
      const double v = U[(size_t)k * R + c];
      s = fma(v, v, s);
    }
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && c < R) {
    double t = 0.0;
    for (int w = 0; w < kCT / 32; ++w) t += red[w][tx];
    const double nrm = sqrt(t);
    norms[c] = nrm == 0.0 ? 1.0 : nrm;
  }
}
// U[:, c] /= norms[c]; carry[c] *= norms[c] (the scale the caller moves into another factor), carry may be null
__global__ void __launch_bounds__(kCT) k_scale_columns(double* __restrict__ U, int n, int R, const double* __restrict__ norms,
                                                      double* __restrict__ carry) {
  const long long tot = (long long)n * R;
  for (long long i = (long long)blockIdx.x * kCT + threadIdx.x; i < tot; i += (long long)gridDim.x * kCT) {
    const int c = (int)(i % R);
    U[i] = U[i] / norms[c];
    if (carry != nullptr && i < R) carry[i] *= norms[i];
  }
}

}  // namespace admmq

using namespace admmq;

extern "C" int admmq_gram_hadamard(const float* U1, int n1, const float* U2, int n2, int R, float* G, void* stream_) {
  if (U1 == nullptr || G == nullptr || n1 <= 0 || R <= 0 || (U2 != nullptr && n2 <= 0))
    return fail(ADMMQ_E_BADARG, "admmq_gram_hadamard: bad argument");
  dim3 grid((R + 31) / 32, (R + 31) / 32);
  k_gram_hadamard<float><<<grid, kCT, 0, (cudaStream_t)stream_>>>(U1, n1, U2, n2, R, G);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

extern "C" int admmq_unfold3(const float* W, int I, int J, int K, int mode, float* out, void* stream_) {
  if (W == nullptr || out == nullptr || I <= 0 || J <= 0 || K <= 0 || mode < 0 || mode > 2)
    return fail(ADMMQ_E_BADARG, "admmq_unfold3: bad argument");
  const long long n = (long long)I * J * K;
  const int g = (int)std::min<long long>((n + kCT - 1) / kCT, 148 * 16);
  k_unfold3<<<g, kCT, 0, (cudaStream_t)stream_>>>(W, I, J, K, mode, out);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

namespace admmq {
size_t mttkrp_tc_workspace_bytes(int M, int nx, int ny, int R);
int mttkrp_tc(const float* V, int M, const float* X, int nx, const float* Y, int ny, int R, float* F,
              void* workspace, size_t workspace_bytes, cudaStream_t stream);
}  // namespace admmq

extern "C" size_t admmq_mttkrp_workspace_bytes(int M, int nx, int ny, int R, int precision) {
  if (precision == 1) return mttkrp_tc_workspace_bytes(M, nx, ny, R);
  DeviceProps dp;
  const int sms = (device_props(&dp) == ADMMQ_OK) ? dp.sm_count : 148;
  int splits;
  select_mttkrp_kernel(M, nx, std::max(ny, 1), R, 0, sms, nullptr, &splits);
  return align_up((size_t)splits * M * R * sizeof(double), 256);  // split-K partials
}

extern "C" int admmq_mttkrp(const float* Wn, int M, const float* X, int nx, const float* Y, int ny, int R, float* F,
                            int precision, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (Wn == nullptr || X == nullptr || F == nullptr || M <= 0 || nx <= 0 || R <= 0 || (Y != nullptr && ny <= 0))
    return fail(ADMMQ_E_BADARG, "admmq_mttkrp: bad argument");
  if (Y == nullptr) ny = 1;
  if (precision == 1) {
    // the tensor-core form contracts the large index first and needs the (m, y, x) permutation of the tensor; for a
    // matrix (ny == 1, nx % 4 == 0) the unfolding itself is that operand
    if (ny == 1 && (nx & 3) == 0) return mttkrp_tc(Wn, M, X, nx, nullptr, 1, R, F, workspace, workspace_bytes, stream);
    return fail(ADMMQ_E_UNSUPPORTED, "admmq_mttkrp: precision 1 on a 3-way tensor takes the permuted operand: use "
                                     "admmq_permute_myx once per layer and admmq_mttkrp_tc");
  }
  if (precision != 0) return fail(ADMMQ_E_BADARG, "admmq_mttkrp: precision must be 0 (f64 accumulate) or 1 (3xTF32)");
  return launch_mttkrp_f64<float, float>(Wn, M, X, nx, Y, ny, R, F, workspace, workspace_bytes, stream);
}

// ---- float64 pieces of the ALS / EPC initialisation (source/parafac_epc.py:12-82; tensorly parafac, musco cp_anc)
extern "C" size_t admmq_mttkrp_f64_workspace_bytes(int M, int nx, int ny, int R) {
  return admmq_mttkrp_workspace_bytes(M, nx, ny, R, 0);
}

extern "C" int admmq_mttkrp_f64(const double* Wn, int M, const double* X, int nx, const double* Y, int ny, int R,
                                double* F, void* workspace, size_t workspace_bytes, void* stream_) {
  if (Wn == nullptr || X == nullptr || F == nullptr || M <= 0 || nx <= 0 || R <= 0 || (Y != nullptr && ny <= 0))
    return fail(ADMMQ_E_BADARG, "admmq_mttkrp_f64: bad argument");
  if (Y == nullptr) ny = 1;
  return launch_mttkrp_f64<double, double>(Wn, M, X, nx, Y, ny, R, F, workspace, workspace_bytes, (cudaStream_t)stream_);
}

extern "C" int admmq_gram_hadamard_f64(const double* U1, int n1, const double* U2, int n2, int R, double* G, void* stream_) {
  if (U1 == nullptr || G == nullptr || n1 <= 0 || R <= 0 || (U2 != nullptr && n2 <= 0))
    return fail(ADMMQ_E_BADARG, "admmq_gram_hadamard_f64: bad argument");
  dim3 grid((R + 31) / 32, (R + 31) / 32);
  k_gram_hadamard<double><<<grid, kCT, 0, (cudaStream_t)stream_>>>(U1, n1, U2, n2, R, G);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

extern "C" int admmq_normalize_columns_f64(double* U, int n, int R, double* norms, double* carry, void* stream_) {
  if (U == nullptr || norms == nullptr || n <= 0 || R <= 0) return fail(ADMMQ_E_BADARG, "admmq_normalize_columns_f64: bad argument");
  cudaStream_t stream = (cudaStream_t)stream_;
  k_column_norms<<<(R + 31) / 32, kCT, 0, stream>>>(U, n, R, norms);
  const long long tot = (long long)n * R;
  k_scale_columns<<<(int)std::min<long long>((tot + kCT - 1) / kCT, 148 * 8), kCT, 0, stream>>>(U, n, R, norms, carry);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(2);
  return ADMMQ_OK;
}

extern "C" size_t admmq_recon_error_workspace_bytes(int M, int nx, int ny) {
  const long long P = (long long)nx * std::max(ny, 1);
  const size_t ctas = (size_t)((M + 63) / 64) * (size_t)((P + 63) / 64);
  return align_up(ctas * 2 * sizeof(double), 256);
}

extern "C" int admmq_recon_error(const float* W0, int M, const float* A, const float* X, int nx, const float* Y,
                                 int ny, int R, double* out2, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (W0 == nullptr || A == nullptr || X == nullptr || out2 == nullptr || M <= 0 || nx <= 0 || R <= 0)
    return fail(ADMMQ_E_BADARG, "admmq_recon_error: bad argument");
  if (Y == nullptr) ny = 1;
  if (workspace == nullptr || workspace_bytes < admmq_recon_error_workspace_bytes(M, nx, ny))
    return fail(ADMMQ_E_WORKSPACE, "admmq_recon_error: workspace too small");
  const long long P = (long long)nx * ny;
  dim3 grid((unsigned)((P + 63) / 64), (M + 63) / 64);
  k_recon_error<<<grid, kCT, 0, stream>>>(W0, M, P, A, X, Y, ny, R, (double*)workspace);
  k_sum_pairs<<<1, kCT, 0, stream>>>((const double*)workspace, (long long)grid.x * grid.y, out2);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(2);
  return ADMMQ_OK;
}
