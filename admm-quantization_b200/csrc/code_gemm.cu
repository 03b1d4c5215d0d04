// code_gemm.cu - CP layers on the FP8 tensor cores from their factor codes (DESIGN.md 2d):
//   k_codes_to_fp8        factor codes -> FP8 operand bytes (exact: the byte's value is the grid level), optionally
//                         transposed, pad columns zeroed
//   k_fp8_quantize_rows   per-row dynamic E4M3 activations: s_m = fl(amax_m / 448), q = cvt.rn.satfinite.e4m3(fl(x / s_m))
//   k_code_gemm           D = fl(acc * fl(s_a[m] * s_w)) (+ bias[n]), acc = A8 . B8^T summed by tcgen05.mma kind::f8f6f4
//                         in float32 over K in a fixed order (no split-K: the result does not depend on the grid)
#include <algorithm>
#include <cstdlib>
#include "numerics.cuh"
#include "tc_gemm.cuh"

namespace admmq {

namespace {

constexpr int kCgThreads = 192;     // warp 0: TMA, warp 1: MMA (and the TMEM allocation), warps 2 .. 5: epilogue
constexpr int kCgBlockK = 128;      // codes per K-block: one 128-byte swizzle row
constexpr int kCgUmmaK = 32;        // k per tcgen05.mma.kind::f8f6f4
constexpr int kCgTileM = 128;
constexpr int kCgStageBudget = 192 * 1024;

// Operand stages and tensor memory of a tile of up to BN columns: two accumulators of BN float32 columns, so that the
// epilogue of one tile overlaps the MMAs of the next.
template <int BN>
struct CgSmem {
  static_assert(BN == 128 || BN == 256, "BN must be 128 or 256");
  static constexpr int kABytes = kCgTileM * kCgBlockK;    // 16 KB
  static constexpr int kBBytes = BN * kCgBlockK;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = kCgStageBudget / kStageBytes;   // 6 (BN = 128) or 4 (BN = 256)
  static constexpr int kBytes = kStages * kStageBytes + 1024;    // + slack for the 1024-byte alignment of SWIZZLE_128B
  static constexpr unsigned int kTmemCols = 2 * BN;
  static_assert(kBytes <= 227 * 1024, "tile does not fit in shared memory");
};

struct CgPipe {
  unsigned long long full[6], empty[6];      // operand stage landed / consumed by the MMAs
  unsigned long long acc_full[2], acc_empty[2];
  unsigned int tmem_base;
};

struct CgMaps {
  CUtensorMap a, b;
};

__device__ __forceinline__ void umma_f8f6f4(unsigned int d_tmem, unsigned long long a_desc, unsigned long long b_desc,
                                            unsigned int idesc, unsigned int accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// instruction descriptor: D = F32, A / B formats (kind::f8f6f4: E4M3 = 0, E5M2 = 1), both K-major, M = 128, N = bn
__host__ __device__ constexpr unsigned int cg_idesc(int bn, unsigned int a_fmt, unsigned int b_fmt) {
  return (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | ((unsigned int)(bn >> 3) << 17) | ((unsigned int)(kCgTileM >> 4) << 24);
}

// Persistent: CTA b computes tiles b, b + grid, ... (row-major over 128 x bn tiles).  Barrier phases: fill number n of a
// stage / accumulator completes phase n - 1, so its parity is (n - 1) & 1; a producer waits for the previous use to
// have been released, which for the first use is the parity-1 phase a fresh barrier counts as complete.
template <int BN>
__global__ void __launch_bounds__(kCgThreads, 1)
k_code_gemm(const __grid_constant__ CgMaps maps, int M, int N, int K, int bn, unsigned int idesc,
            const float* __restrict__ a_scale, const float* __restrict__ b_scale, const float* __restrict__ bias,
            float* __restrict__ D, int ldd) {
  using S = CgSmem<BN>;
  constexpr int kNS = S::kStages;
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  __shared__ CgPipe pipe;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned int base = (tc::smem_u32(smem_dyn) + 1023u) & ~1023u;
  const int tilesM = (M + kCgTileM - 1) / kCgTileM, tilesN = (N + bn - 1) / bn;
  const int tiles = tilesM * tilesN;
  const int nkb = (K + kCgBlockK - 1) / kCgBlockK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kNS; ++s) {
      tc::mbar_init(&pipe.full[s], 1);
      tc::mbar_init(&pipe.empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&pipe.acc_full[b], 1);
      tc::mbar_init(&pipe.acc_empty[b], 4);
    }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc(&pipe.tmem_base, S::kTmemCols);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const unsigned int tmem = pipe.tmem_base;

  if (warp == 0) {
    // ---------------- TMA: A (128 rows) and B (bn rows) of one K-block per stage
    if (lane == 0) {
      tc::tma_prefetch_desc(&maps.a);
      tc::tma_prefetch_desc(&maps.b);
    }
    if (tc::elect_one()) {
      const unsigned int tx = (unsigned int)((kCgTileM + bn) * kCgBlockK);
      unsigned int it = 0;
      for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const int m0 = (tile / tilesN) * kCgTileM, n0 = (tile % tilesN) * bn;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = (int)(it % kNS);
          tc::mbar_wait(&pipe.empty[s], ((it / kNS) & 1u) ^ 1u);
          const unsigned int sa = base + (unsigned int)(s * S::kStageBytes);
          tc::mbar_expect_tx(&pipe.full[s], tx);
          tc::tma_load_2d(sa, &maps.a, kb * kCgBlockK, m0, &pipe.full[s]);
          tc::tma_load_2d(sa + (unsigned int)S::kABytes, &maps.b, kb * kCgBlockK, n0, &pipe.full[s]);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---------------- MMA: the whole warp runs the loop, one elected lane issues
    unsigned int it = 0, tl = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++tl) {
      const unsigned int ab = tl & 1u;
      tc::mbar_wait(&pipe.acc_empty[ab], ((tl >> 1) & 1u) ^ 1u);
      tc::tc_fence_after();
      const unsigned int acc = tmem + ab * (unsigned int)BN;
      for (int kb = 0; kb < nkb; ++kb, ++it) {
        const int s = (int)(it % kNS);
        tc::mbar_wait(&pipe.full[s], (it / kNS) & 1u);
        tc::tc_fence_after();
        if (tc::elect_one()) {
          const unsigned int sa = base + (unsigned int)(s * S::kStageBytes);
          const unsigned long long da = tc::make_desc(sa), db = tc::make_desc(sa + (unsigned int)S::kABytes);
#pragma unroll
          for (int k = 0; k < kCgBlockK / kCgUmmaK; ++k) {
            const unsigned long long adv = (unsigned long long)((k * kCgUmmaK) >> 4);   // +32 bytes per k-step
            umma_f8f6f4(acc, da + adv, db + adv, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          tc::umma_commit(&pipe.empty[s]);
          if (kb + 1 == nkb) tc::umma_commit(&pipe.acc_full[ab]);
        }
        __syncwarp();
      }
    }
  } else {
    // ---------------- epilogue: warp w reads TMEM lanes 32 (w % 4) .. +31 = tile rows, 16 columns per tcgen05.ld
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const float sw = __ldg(b_scale);
    const bool vec = ((ldd & 3) == 0) && ((reinterpret_cast<uintptr_t>(D) & 15) == 0);
    unsigned int tl = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++tl) {
      const unsigned int ab = tl & 1u;
      const int m0 = (tile / tilesN) * kCgTileM, n0 = (tile % tilesN) * bn;
      const int i = m0 + row;
      const float sc = i < M ? __fmul_rn(__ldg(a_scale + i), sw) : 0.0f;
      float* drow = D + (size_t)(i < M ? i : 0) * (size_t)ldd;
      tc::mbar_wait(&pipe.acc_full[ab], (tl >> 1) & 1u);
      tc::tc_fence_after();
      const unsigned int taddr = tmem + ((unsigned int)(q * 32) << 16) + ab * (unsigned int)BN;
      for (int c0 = 0; c0 < bn; c0 += 16) {
        unsigned int r[16];
        tc::tmem_load<16>(taddr + (unsigned int)c0, r);
        tc::tmem_load_wait();
        if (i < M) {
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int n = n0 + c0 + j;
            v[j] = __fmul_rn(__uint_as_float(r[j]), sc);
            if (bias != nullptr && n < N) v[j] = __fadd_rn(v[j], __ldg(bias + n));
          }
          const int n = n0 + c0;
          if (vec && n + 16 <= N) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              *reinterpret_cast<float4*>(drow + n + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (n + j < N) drow[n + j] = v[j];
          }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&pipe.acc_empty[ab]);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_free(tmem, S::kTmemCols);
}

// One warp per row: the row's abs-max (NaN propagates), s = fl(amax / 448), codes of fl(x / s) by the hardware
// conversion, four columns per lane and store, pad columns [K, ldq) zero.
__global__ void __launch_bounds__(256) k_fp8_quantize_rows(const float* __restrict__ x, int ldx, int M, int K,
                                                             unsigned char* __restrict__ q, int ldq, float* __restrict__ scale) {
  const int lane = threadIdx.x & 31;
  const int row = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (row >= M) return;
  const float* xr = x + (size_t)row * ldx;
  float amax = 0.0f;
  for (int k = lane; k < K; k += 32) {
    const float a = fabsf(__ldg(xr + k));
    amax = (a > amax || a != a) ? a : amax;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float a = __shfl_xor_sync(0xffffffffu, amax, o);
    amax = (a > amax || a != a) ? a : amax;
  }
  float s;
  if (!(amax <= 3.402823466e38f)) s = __int_as_float(0x7fffffff);   // NaN or infinite abs-max: the row's outputs are NaN
  else s = __fdiv_rn(amax, 448.0f);                                  // 0 for amax == 0 or on underflow
  unsigned int* qr = reinterpret_cast<unsigned int*>(q + (size_t)row * ldq);
  for (int c = lane * 4; c < ldq; c += 128) {
    unsigned int word = 0u;
    if (s != 0.0f) {
      float t[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) t[j] = c + j < K ? __fdiv_rn(__ldg(xr + c + j), s) : 0.0f;
      unsigned short lo, hi;
      asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(lo) : "f"(t[1]), "f"(t[0]));   // first source -> upper byte
      asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(hi) : "f"(t[3]), "f"(t[2]));
      word = (unsigned int)lo | ((unsigned int)hi << 16);
    }
    qr[c >> 2] = word;
  }
  if (lane == 0) scale[row] = s;
}

// out (rows_out x ldo): out[r, c] = byte of codes[r, c] (transpose = 0) or of codes[c, r] (transpose = 1); codes is
// rows x cols, contiguous.  Columns [cols_out, ldo) are zero.
__global__ void __launch_bounds__(256) k_codes_to_fp8(const signed char* __restrict__ codes, int rows, int cols, int scheme,
                                                        int transpose, unsigned char* __restrict__ out, int ldo) {
  const int rows_out = transpose ? cols : rows, cols_out = transpose ? rows : cols;
  const long long tot = (long long)rows_out * ldo;
  for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < tot; o += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(o / ldo), c = (int)(o - (long long)r * ldo);
    unsigned int b = 0u;
    if (c < cols_out) b = code_to_fp8(scheme, (int)codes[transpose ? (size_t)c * cols + r : (size_t)r * cols + c]);
    out[o] = (unsigned char)b;
  }
}

constexpr long long kIndexLimit = 1LL << 31;

}  // namespace

// The tile width of a code GEMM: the multiple of 16 up to 256 that fills whole waves of 128 x bn tiles (the MTTKRP's
// rule, tc::wave_cost with a fixed part of 16 columns).  ADMMQ_CODE_GEMM_BN forces a width (a test knob, read per call).
int code_gemm_tile_width(int M, int N, int sms, int* grid) {
  const long long tilesM = (M + kCgTileM - 1) / kCgTileM;
  int bn = 256;
  long long best = -1;
  for (int w = 256; w >= 16; w -= 16) {
    const long long cost = tc::wave_cost(tilesM, N, w, sms, 16);
    if (best < 0 || cost < best) {
      best = cost;
      bn = w;
    }
  }
  if (const char* force = getenv("ADMMQ_CODE_GEMM_BN")) {
    const int w = atoi(force);
    if (w >= 16 && w <= 256 && (w & 15) == 0) bn = w;
  }
  if (grid != nullptr) *grid = (int)std::min<long long>(tilesM * ((N + bn - 1) / bn), sms);
  return bn;
}

template <int BN>
static int launch_code_gemm(const CgMaps& maps, int M, int N, int K, int bn, unsigned int idesc, const float* sa,
                            const float* sw, const float* bias, float* D, int ldd, int grid, cudaStream_t stream) {
  const int smem = CgSmem<BN>::kBytes;
  ADMMQ_CUDA_OK(cudaFuncSetAttribute(k_code_gemm<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  k_code_gemm<BN><<<grid, kCgThreads, smem, stream>>>(maps, M, N, K, bn, idesc, sa, sw, bias, D, ldd);
  return ADMMQ_OK;
}

}  // namespace admmq

using namespace admmq;

extern "C" int admmq_fp8_operand_format(int bits, int qscheme) {
  const int f = fp8_operand_format(qscheme, bits);
  if (f >= 0) return f;
  if (qscheme == ADMMQ_Q_MINMAX || qscheme == ADMMQ_Q_AFFINE)
    return fail(ADMMQ_E_BADARG, "fp8 operand: the %s grid is offset by its minimum / zero point, so its levels are not "
                "codes times one scale", qscheme == ADMMQ_Q_MINMAX ? "tensor_minmax" : "tensor_affine");
  if (qscheme == ADMMQ_Q_MSEMINMAX_SYMMETRIC || qscheme == ADMMQ_Q_SYMMETRIC)
    return fail(ADMMQ_E_BADARG, "fp8 operand: integer codes need bits 1 .. 5 (|code| <= 16 is exact in E4M3; 17 is not), "
                "got bits = %d", bits);
  const char* name;
  const int want = scheme_bits(qscheme, &name);
  if (want != 0) return fail(ADMMQ_E_BADARG, "fp8 operand: %s needs bits = %d, got %d", name, want, bits);
  return fail(ADMMQ_E_BADARG, "fp8 operand: unknown qscheme id %d", qscheme);
}

extern "C" int admmq_codes_to_fp8(const int8_t* codes, int rows, int cols, int bits, int qscheme, int transpose,
                                  uint8_t* out, int ldo, void* stream) {
  if (int e = admmq_fp8_operand_format(bits, qscheme); e < 0) return e;
  const int cols_out = transpose ? rows : cols, rows_out = transpose ? cols : rows;
  if (codes == nullptr || out == nullptr || rows <= 0 || cols <= 0)
    return fail(ADMMQ_E_BADARG, "admmq_codes_to_fp8: null pointer or empty shape");
  if ((ldo & 15) != 0 || ldo < cols_out)
    return fail(ADMMQ_E_BADARG, "admmq_codes_to_fp8: ldo = %d must be a multiple of 16 and >= %d", ldo, cols_out);
  if ((long long)rows_out * ldo >= kIndexLimit || (long long)rows * cols >= kIndexLimit)
    return fail(ADMMQ_E_UNSUPPORTED, "admmq_codes_to_fp8: shape past the 32-bit indexing limit");
  const long long tot = (long long)rows_out * ldo;
  const int blocks = (int)std::min<long long>((tot + 255) / 256, 148 * 8);
  k_codes_to_fp8<<<blocks, 256, 0, (cudaStream_t)stream>>>((const signed char*)codes, rows, cols, qscheme, transpose,
                                                          out, ldo);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

extern "C" int admmq_fp8_quantize_rows(const float* x, int ldx, int M, int K, uint8_t* q, int ldq, float* scale,
                                       void* stream) {
  if (K <= 0 || M <= 0 || x == nullptr || q == nullptr || scale == nullptr)
    return fail(ADMMQ_E_BADARG, "admmq_fp8_quantize_rows: null pointer or empty shape (M = %d, K = %d)", M, K);
  if (ldx < K || (ldq & 15) != 0 || ldq < K || ((uintptr_t)q & 15) != 0)
    return fail(ADMMQ_E_BADARG, "admmq_fp8_quantize_rows: ldx = %d must be >= K = %d, ldq = %d a multiple of 16 and >= K, "
                "q 16-byte aligned", ldx, K, ldq);
  if ((long long)M * ldx >= kIndexLimit || (long long)M * ldq >= kIndexLimit)
    return fail(ADMMQ_E_UNSUPPORTED, "admmq_fp8_quantize_rows: shape past the 32-bit indexing limit");
  const int blocks = (int)(((long long)M * 32 + 255) / 256);
  k_fp8_quantize_rows<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, ldx, M, K, q, ldq, scale);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

extern "C" int admmq_code_gemm_kernel(int M, int N, int K, int sm_count, int* grid) {
  if (M <= 0 || N <= 0 || K <= 0 || sm_count <= 0) return fail(ADMMQ_E_BADARG, "admmq_code_gemm_kernel: bad argument");
  return code_gemm_tile_width(M, N, sm_count, grid);
}

extern "C" int admmq_code_gemm(const uint8_t* A8, int lda, const float* a_scale, int M, const uint8_t* B8, int ldb,
                               const float* b_scale, int b_format, int N, int K, const float* bias, float* D, int ldd,
                               void* stream) {
  if (A8 == nullptr || B8 == nullptr || a_scale == nullptr || b_scale == nullptr || D == nullptr || M <= 0 || N <= 0 ||
      K <= 0)
    return fail(ADMMQ_E_BADARG, "admmq_code_gemm: null pointer or empty shape (M = %d, N = %d, K = %d)", M, N, K);
  if ((lda & 15) != 0 || (ldb & 15) != 0 || lda < K || ldb < K || ldd < N || ((uintptr_t)A8 & 15) != 0 ||
      ((uintptr_t)B8 & 15) != 0)
    return fail(ADMMQ_E_BADARG, "admmq_code_gemm: lda = %d, ldb = %d must be multiples of 16 and >= K = %d, ldd >= N, "
                "A8 / B8 16-byte aligned", lda, ldb, K);
  if (b_format != ADMMQ_Q_MSEMINMAX_E4M3 && b_format != ADMMQ_Q_MSEMINMAX_E5M2)
    return fail(ADMMQ_E_BADARG, "admmq_code_gemm: b_format must be ADMMQ_Q_MSEMINMAX_E4M3 or _E5M2, got %d", b_format);
  if ((long long)M * lda >= kIndexLimit || (long long)N * ldb >= kIndexLimit || (long long)M * ldd >= kIndexLimit)
    return fail(ADMMQ_E_UNSUPPORTED, "admmq_code_gemm: shape past the 32-bit indexing limit");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  if (dp.cc_major != 10) return fail(ADMMQ_E_UNSUPPORTED, "admmq_code_gemm needs an sm_100 device (tcgen05)");
  int grid;
  const int bn = code_gemm_tile_width(M, N, dp.sm_count, &grid);
  CgMaps maps;
  if (int e = tc::make_tmap_2d(&maps.a, CU_TENSOR_MAP_DATA_TYPE_UINT8, A8, M, K, (size_t)lda, kCgBlockK, kCgTileM)) return e;
  if (int e = tc::make_tmap_2d(&maps.b, CU_TENSOR_MAP_DATA_TYPE_UINT8, B8, N, K, (size_t)ldb, kCgBlockK, bn)) return e;
  const unsigned int idesc = cg_idesc(bn, 0u, b_format == ADMMQ_Q_MSEMINMAX_E5M2 ? 1u : 0u);
  cudaStream_t st = (cudaStream_t)stream;
  const int e = bn > 128 ? launch_code_gemm<256>(maps, M, N, K, bn, idesc, a_scale, b_scale, bias, D, ldd, grid, st)
                         : launch_code_gemm<128>(maps, M, N, K, bn, idesc, a_scale, b_scale, bias, D, ldd, grid, st);
  if (e) return e;
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}
