// tc_gemm.cu - C = A . B^T in 3xTF32 on tcgen05 (admmq_gemm_nt), the stand-alone form of the tile product that
// the persistent ADMM loop uses for its ridge product and that the tensor-core MTTKRP builds on.
#include <algorithm>
#include <cstdlib>
#include "tc_gemm.cuh"

namespace admmq {

namespace tc {
int make_operand_tmap(CUtensorMap* out, const float* base, int rows, int cols, int ld, int box_rows) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (encode == nullptr) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || fn == nullptr)
      return fail(ADMMQ_E_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    encode = (EncodeFn)fn;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)kAtomK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1u, 1u};
  const CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(ADMMQ_E_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return ADMMQ_OK;
}
}  // namespace tc

struct GemmMaps {
  CUtensorMap a, b, blo;  // blo: lo part of a pre-split B (PS), otherwise unused
};

template <int BN, bool PS>
__global__ void __launch_bounds__(tc::kThreadsTC, 1)
k_gemm_nt_tc(const __grid_constant__ GemmMaps maps, int M, int N, int K, float* __restrict__ C, int ldc, float neg_zero) {
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  __shared__ tc::Pipe pipe;
  tc::PipeState st;
  tc::pipe_setup(pipe, st, neg_zero);
  const int tilesM = (M + tc::kTileM - 1) / tc::kTileM, tilesN = (N + BN - 1) / BN;
  for (int tile = blockIdx.x; tile < tilesM * tilesN; tile += gridDim.x) {
    const int i0 = (tile / tilesN) * tc::kTileM, n0 = (tile % tilesN) * BN;
    const int next = tile + (int)gridDim.x;
    const bool has_next = next < tilesM * tilesN;
    tc::tile_3xtf32<BN, PS>(&maps.a, i0, &maps.b, &maps.blo, n0, BN, K, smem_dyn, pipe, st,
                               has_next ? (next / tilesN) * tc::kTileM : -1, has_next ? (next % tilesN) * BN : -1);
    const float* tile_c = tc::acc_to_smem<BN, PS>(pipe, smem_dyn);
    using ET = tc::EpiTile<BN>;
    const bool vec = ((ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
#pragma unroll
    for (int g0 = 0; g0 < ET::kGroups; g0 += tc::kThreadsTC) {
      const int g = g0 + (int)threadIdx.x;
      const int row = g / ET::kGroupsPerRow, c4 = (g - row * ET::kGroupsPerRow) * 4;
      const int i = i0 + row, n = n0 + c4;
      if (g < ET::kGroups && i < M && n < N) {
        const float4 h4 = *reinterpret_cast<const float4*>(tile_c + ET::offset(row, c4 >> 2));
        float* dst = C + (size_t)i * ldc + n;
        if (vec && n + 3 < N) {
          *reinterpret_cast<float4*>(dst) = h4;
        } else {
          const float h[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (n + q < N) dst[q] = h[q];
        }
      }
    }
    __syncthreads();
  }
  tc::pipe_teardown(pipe);
}

// MTTKRP with the fold of the small tensor index inside the epilogue (mttkrp_tc.cu):
//   F[m, r] = sum_y Y[y, r] * T[(m, y), r],   T = A . B^T with A rows (m, y) = the (m, y, x)-permuted tensor, B = X^T.
// A tile takes mg = 128 / ny whole m (rows m0 * ny .. +mg * ny - 1 of A; the TMA box still loads 128 rows, the extra
// ones belong to the next tile and are ignored), so the fold over y happens on the accumulator parked in shared memory
// and T never goes to global memory.  float64 accumulation over y like the stand-alone fold kernel.
template <int BN>
__global__ void __launch_bounds__(tc::kThreadsTC, 1)
k_mttkrp_fold_tc(const __grid_constant__ GemmMaps maps, int Mout, int ny, int N, int K, int bn, const float* __restrict__ Y,
                 float* __restrict__ F, float neg_zero) {
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  __shared__ tc::Pipe pipe;
  tc::PipeState st;
  tc::pipe_setup(pipe, st, neg_zero);
  const int mg = tc::kTileM / ny;  // m per tile
  // bn <= BN (a multiple of 16) is the tile width actually computed: chosen on the host so that the tiles fill whole
  // waves of the grid (37 x 12 tiles of width 96 are exactly 3 waves of 148 for 512 x 512 x 9 at R = 1141)
  const int tilesM = (Mout + mg - 1) / mg, tilesN = (N + bn - 1) / bn;
  for (int tile = blockIdx.x; tile < tilesM * tilesN; tile += gridDim.x) {
    const int m0 = (tile / tilesN) * mg, n0 = (tile % tilesN) * bn;
    const int next = tile + (int)gridDim.x;
    const bool has_next = next < tilesM * tilesN;
    tc::tile_3xtf32<BN, true>(&maps.a, m0 * ny, &maps.b, &maps.blo, n0, bn, K, smem_dyn, pipe, st,
                              has_next ? (next / tilesN) * mg * ny : -1, has_next ? (next % tilesN) * bn : -1);
    const float* tile_c = tc::acc_to_smem<BN, true>(pipe, smem_dyn);
    using ET = tc::EpiTile<BN>;
    for (int idx = threadIdx.x; idx < mg * bn; idx += tc::kThreadsTC) {
      const int ml = idx / bn, c = idx - ml * bn;
      const int m = m0 + ml, n = n0 + c;
      if (m < Mout && n < N) {
        double acc = 0.0;
        for (int y = 0; y < ny; ++y)
          acc = fma((double)__ldg(Y + (size_t)y * N + n), (double)tile_c[ET::offset(ml * ny + y, c >> 2) + (c & 3)], acc);
        F[(size_t)m * N + n] = (float)acc;
      }
    }
    __syncthreads();
  }
  tc::pipe_teardown(pipe);
}

// The same contraction when the folded index is LONG (ny > 128: the tap factor of a convolution, F (9 x R) folded over the
// 512 input channels): a 128-row tile of A covers rows (m, y) of at most two consecutive m.  The tile folds its rows
// with their weights Y[y, n] into two float64 partial sums per column (slot 0: the tile's first m, slot 1: the next
// one), written to partial[(tile_row * 2 + slot) * N + n]; k_fold_partials adds the partials of every m in tile order.
// The intermediate T = A . B^T (M * ny x N floats: 21 MB for 9 x 512 x 1141) never exists.
template <int BN>
__global__ void __launch_bounds__(tc::kThreadsTC, 1)
k_mttkrp_foldlong_tc(const __grid_constant__ GemmMaps maps, int rows, int ny, int N, int K, int bn, const float* __restrict__ Y,
                     double* __restrict__ partial, float neg_zero) {
  extern __shared__ __align__(16) unsigned char smem_dyn[];
  __shared__ tc::Pipe pipe;
  tc::PipeState st;
  tc::pipe_setup(pipe, st, neg_zero);
  const int tilesM = (rows + tc::kTileM - 1) / tc::kTileM, tilesN = (N + bn - 1) / bn;
  for (int tile = blockIdx.x; tile < tilesM * tilesN; tile += gridDim.x) {
    const int tr = tile / tilesN, r0 = tr * tc::kTileM, n0 = (tile % tilesN) * bn;
    const int next = tile + (int)gridDim.x;
    const bool has_next = next < tilesM * tilesN;
    tc::tile_3xtf32<BN, true>(&maps.a, r0, &maps.b, &maps.blo, n0, bn, K, smem_dyn, pipe, st,
                              has_next ? (next / tilesN) * tc::kTileM : -1, has_next ? (next % tilesN) * bn : -1);
    const float* tile_c = tc::acc_to_smem<BN, true>(pipe, smem_dyn);
    using ET = tc::EpiTile<BN>;
    const int m_first = r0 / ny;
    // thread -> (column c, quarter q): the four quarters of a column are neighbouring lanes and take rows q, q + 4, ...
    // (consecutive rows sit in different swizzle positions of the staging tile: no bank conflicts), summed in fixed
    // order ((q0 + q1) + (q2 + q3)) with two shuffles - the tile leaves no room for another shared-memory array
    const int c = threadIdx.x >> 2, q = threadIdx.x & 3;
    static_assert(BN * 4 == tc::kThreadsTC, "one thread per (column, quarter)");
    double a0 = 0.0, a1 = 0.0;
    const bool col_ok = c < bn && n0 + c < N;
    if (col_ok) {
      // rows q, q + 4, ... of the tile: (m, y) advance without a division; the weights Y[y, n] of eight rows are
      // requested before the first use (they come from L2: one round trip per batch instead of one per row)
      const int y_first = r0 - m_first * ny;          // y of the tile's first row
      const float* ycol = Y + n0 + c;
      constexpr int kB = 8;
      for (int i0 = 0; i0 < tc::kTileM / 4; i0 += kB) {
        float w[kB];
        int slot[kB];
#pragma unroll
        for (int b = 0; b < kB; ++b) {
          const int rr = (i0 + b) * 4 + q;
          int y = y_first + rr;
          slot[b] = y >= ny ? 1 : 0;
          if (y >= ny) y -= ny;
          w[b] = (r0 + rr < rows) ? __ldg(ycol + (size_t)y * N) : 0.0f;
        }
#pragma unroll
        for (int b = 0; b < kB; ++b) {
          const int rr = (i0 + b) * 4 + q;
          const double v = (double)w[b] * (double)tile_c[ET::offset(rr, c >> 2) + (c & 3)];
          if (slot[b] == 0) a0 += v;
          else a1 += v;
        }
      }
    }
    a0 += __shfl_xor_sync(0xffffffffu, a0, 1);
    a1 += __shfl_xor_sync(0xffffffffu, a1, 1);
    a0 += __shfl_xor_sync(0xffffffffu, a0, 2);
    a1 += __shfl_xor_sync(0xffffffffu, a1, 2);
    if (col_ok && q == 0) {
      partial[((size_t)tr * 2 + 0) * N + n0 + c] = a0;
      partial[((size_t)tr * 2 + 1) * N + n0 + c] = a1;
    }
    __syncthreads();
  }
  tc::pipe_teardown(pipe);
}

// F[m, n] = sum over the row tiles that hold rows of m, in tile order (fixed: deterministic)
__global__ void __launch_bounds__(256) k_fold_partials(const double* __restrict__ partial, int M, int ny, int N, float* __restrict__ F) {
  const long long tot = (long long)M * N;
  for (long long o = (long long)blockIdx.x * 256 + threadIdx.x; o < tot; o += (long long)gridDim.x * 256) {
    const int m = (int)(o / N), n = (int)(o - (long long)m * N);
    const int t_first = (int)(((long long)m * ny) / tc::kTileM), t_last = (int)(((long long)(m + 1) * ny - 1) / tc::kTileM);
    double acc = 0.0;
    for (int t = t_first; t <= t_last; ++t) {
      const int slot = m - (int)(((long long)t * tc::kTileM) / ny);   // 0 or 1 (ny > 128: a tile spans at most two m)
      acc += partial[((size_t)t * 2 + slot) * N + n];
    }
    F[o] = (float)acc;
  }
}

// ---------------------------------------------------------------------------- launch choices
// Tile widths come from a wave model: a tile costs a fixed part plus bn columns of tensor-core work, and the width
// minimises waves * (fixed + bn); ties go to the wider tile (the candidates are tried widest first).
static long long wave_cost(long long tilesM, int N, int w, int sms, int fixed) {
  const long long tiles = tilesM * ((N + w - 1) / w);
  return ((tiles + sms - 1) / sms) * (fixed + w);
}

// gemm_nt: measured 3.3 + 0.225 bn us at K = 1141, i.e. a fixed part of 16 columns; 128-wide tiles need the pre-split
// B operand
static int gemm_tile_width(int M, int N, int sms, bool presplit) {
  const long long tilesM = (M + tc::kTileM - 1) / tc::kTileM;
  int bn = 16;
  long long best = -1;
  for (const int w : {128, 64, 32, 16}) {
    if (w == 128 && !presplit) continue;
    const long long cost = wave_cost(tilesM, N, w, sms, 16);
    if (best < 0 || cost < best) {
      best = cost;
      bn = w;
    }
  }
  return bn;
}

// The float64 MTTKRP splits its sum over p into slices of at least 256 (aim: ~2 waves of tiles, at most 64 slices);
// a slice is a whole number of 16-deep slabs, so rounding can leave fewer slices than asked for
static int mttkrp_f64_splits(int M, long long P, int R, int bm, int sms) {
  const long long tiles = (long long)((M + bm - 1) / bm) * ((R + 63) / 64);
  long long want = (2LL * sms + tiles - 1) / tiles;
  const long long max_by_depth = std::max<long long>(1, P / 256);
  want = std::min<long long>(std::max<long long>(1, std::min(want, max_by_depth)), 64);
  const long long per = ((P + want - 1) / want + 15) / 16 * 16;
  return (int)((P + per - 1) / per);
}

// The kernel an MTTKRP call runs: one decision for the launchers (launch_mttkrp_f64, mttkrp_fold_gemm,
// mttkrp_foldlong_gemm, and gemm_nt through gemm_tile_width) and admmq_mttkrp_kernel.  precision 1 is the
// permuted-operand call admmq_mttkrp_tc.  grid: CTAs of the contraction kernel; splits: slices of the float64 sum
// (1 on the tensor cores).  Honours ADMMQ_FOLD_BN.
int select_mttkrp_kernel(int M, int nx, int ny, int R, int precision, int sms, int* grid, int* splits) {
  int kid, g, s = 1;
  if (precision == 0) {
    const int bm = (M <= 16) ? 16 : 64;
    s = mttkrp_f64_splits(M, (long long)nx * ny, R, bm, sms);
    g = ((R + 63) / 64) * ((M + bm - 1) / bm) * s;
    kid = bm == 16 ? ADMMQ_MTTKRP_F64_16 : ADMMQ_MTTKRP_F64_64;
  } else if (ny == 1) {  // matrix: F = W . X
    const int bn = gemm_tile_width(M, R, sms, true);
    g = (int)std::min<long long>((long long)((M + tc::kTileM - 1) / tc::kTileM) * ((R + bn - 1) / bn), sms);
    kid = ADMMQ_MTTKRP_GEMM + bn;
  } else {
    // fold: a tile takes mg = 128 / ny whole m, any multiple of 16 up to 128 wide; long fold (ny > 128): 128-row tiles,
    // 80 .. 128 wide (one thread per column of a 128-wide staging tile).  The fixed part of a tile (pipeline fill,
    // epilogue, fold) is worth ~40 columns at K = 512.
    const bool longf = ny > tc::kTileM;
    const long long tilesM = longf ? ((long long)M * ny + tc::kTileM - 1) / tc::kTileM
                                   : (M + tc::kTileM / ny - 1) / (tc::kTileM / ny);
    int bn = 128;
    long long best = -1;
    for (int w = 128; w >= (longf ? 80 : 16); w -= 16) {
      const long long cost = wave_cost(tilesM, R, w, sms, 40);
      if (best < 0 || cost < best) {
        best = cost;
        bn = w;
      }
    }
    if (const char* force = longf ? nullptr : getenv("ADMMQ_FOLD_BN")) {  // experiment knob, read per call
      const int w = atoi(force);
      if (w >= 16 && w <= 128 && (w & 15) == 0) bn = w;
    }
    g = (int)std::min<long long>(tilesM * ((R + bn - 1) / bn), sms);
    kid = (longf ? ADMMQ_MTTKRP_FOLDLONG : ADMMQ_MTTKRP_FOLD) + bn;
  }
  if (grid != nullptr) *grid = g;
  if (splits != nullptr) *splits = s;
  return kid;
}

template <int BN, bool PS>
static int launch_gemm(const GemmMaps& maps, int M, int N, int K, float* C, int ldc, int grid, cudaStream_t stream) {
  const int smem = tc::TileSmem<BN, PS>::kBytes;
  ADMMQ_CUDA_OK(cudaFuncSetAttribute(k_gemm_nt_tc<BN, PS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  k_gemm_nt_tc<BN, PS><<<grid, tc::kThreadsTC, smem, stream>>>(maps, M, N, K, C, ldc, -0.0f);
  return ADMMQ_OK;
}

// C = A . B^T.  B either as one float32 matrix (Blo == nullptr; split into tf32 hi / lo tile by tile on the fly) or
// pre-split by the caller into B (hi part) and Blo (lo part), both tf32-valued float32 with the same layout.
int gemm_nt(const float* A, int lda, int M, const float* B, const float* Blo, int ldb, int N, int K, float* C, int ldc,
            cudaStream_t stream) {
  if (A == nullptr || B == nullptr || C == nullptr || M <= 0 || N <= 0 || K <= 0)
    return fail(ADMMQ_E_BADARG, "admmq_gemm_nt: null pointer or empty shape");
  if ((lda & 3) || (ldb & 3) || lda < K || ldb < K || ldc < N || ((uintptr_t)A & 15) || ((uintptr_t)B & 15) || ((uintptr_t)Blo & 15))
    return fail(ADMMQ_E_BADARG, "admmq_gemm_nt: lda/ldb must be multiples of 4 and >= K, A/B 16-byte aligned, ldc >= N");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  if (dp.cc_major != 10) return fail(ADMMQ_E_UNSUPPORTED, "admmq_gemm_nt needs an sm_100 device (tcgen05)");
  const int tilesM = (M + tc::kTileM - 1) / tc::kTileM;
  const int bn = gemm_tile_width(M, N, dp.sm_count, Blo != nullptr);
  const int tiles = tilesM * ((N + bn - 1) / bn);
  const int grid = std::min(tiles, dp.sm_count);
  GemmMaps maps;
  if (int e = tc::make_operand_tmap(&maps.a, A, M, K, lda, tc::kTileM)) return e;
  if (int e = tc::make_operand_tmap(&maps.b, B, N, K, ldb, bn)) return e;
  if (int e = tc::make_operand_tmap(&maps.blo, Blo != nullptr ? Blo : B, N, K, ldb, bn)) return e;
  int e = ADMMQ_OK;
  if (Blo != nullptr) {
    e = bn == 128 ? launch_gemm<128, true>(maps, M, N, K, C, ldc, grid, stream)
                  : (bn == 64 ? launch_gemm<64, true>(maps, M, N, K, C, ldc, grid, stream)
                              : (bn == 32 ? launch_gemm<32, true>(maps, M, N, K, C, ldc, grid, stream)
                                          : launch_gemm<16, true>(maps, M, N, K, C, ldc, grid, stream)));
  } else {
    e = bn == 64 ? launch_gemm<64, false>(maps, M, N, K, C, ldc, grid, stream)
                 : (bn == 32 ? launch_gemm<32, false>(maps, M, N, K, C, ldc, grid, stream)
                             : launch_gemm<16, false>(maps, M, N, K, C, ldc, grid, stream));
  }
  if (e) return e;
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

// F (Mout x N) = fold_y( V ((Mout * ny) x K, ld ldv) . Bhi/Blo (N x K, ld ldb)^T , Y (ny x N) ), see k_mttkrp_fold_tc
int mttkrp_fold_gemm(const float* V, int ldv, int Mout, int ny, const float* B, const float* Blo, int ldb, int N, int K,
                     const float* Y, float* F, cudaStream_t stream) {
  if (ny < 1 || ny > tc::kTileM) return fail(ADMMQ_E_UNSUPPORTED, "mttkrp_fold_gemm: ny must be in 1..128");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  if (dp.cc_major != 10) return fail(ADMMQ_E_UNSUPPORTED, "the tensor-core MTTKRP needs an sm_100 device (tcgen05)");
  int grid;
  const int bn = select_mttkrp_kernel(Mout, K, ny, N, 1, dp.sm_count, &grid, nullptr) - ADMMQ_MTTKRP_FOLD;
  GemmMaps maps;
  if (int e = tc::make_operand_tmap(&maps.a, V, Mout * ny, K, ldv, tc::kTileM)) return e;
  if (int e = tc::make_operand_tmap(&maps.b, B, N, K, ldb, bn)) return e;
  if (int e = tc::make_operand_tmap(&maps.blo, Blo, N, K, ldb, bn)) return e;
  if (bn > 64) {
    const int smem = tc::TileSmem<128, true>::kBytes;
    ADMMQ_CUDA_OK(cudaFuncSetAttribute(k_mttkrp_fold_tc<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k_mttkrp_fold_tc<128><<<grid, tc::kThreadsTC, smem, stream>>>(maps, Mout, ny, N, K, bn, Y, F, -0.0f);
  } else {
    const int smem = tc::TileSmem<64, true>::kBytes;
    ADMMQ_CUDA_OK(cudaFuncSetAttribute(k_mttkrp_fold_tc<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k_mttkrp_fold_tc<64><<<grid, tc::kThreadsTC, smem, stream>>>(maps, Mout, ny, N, K, bn, Y, F, -0.0f);
  }
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

size_t mttkrp_foldlong_partial_bytes(int Mout, int ny, int N) {
  const long long rows = (long long)Mout * ny;
  return (size_t)((rows + tc::kTileM - 1) / tc::kTileM) * 2 * (size_t)N * sizeof(double);
}

// F (Mout x N) = fold_y( V ((Mout * ny) x K) . B^T , Y ) for ny > 128, see k_mttkrp_foldlong_tc; partial: workspace of
// mttkrp_foldlong_partial_bytes
int mttkrp_foldlong_gemm(const float* V, int ldv, int Mout, int ny, const float* B, const float* Blo, int ldb, int N, int K,
                         const float* Y, float* F, double* partial, cudaStream_t stream) {
  if (ny <= tc::kTileM) return fail(ADMMQ_E_UNSUPPORTED, "mttkrp_foldlong_gemm: ny must exceed 128");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  if (dp.cc_major != 10) return fail(ADMMQ_E_UNSUPPORTED, "the tensor-core MTTKRP needs an sm_100 device (tcgen05)");
  const int rows = Mout * ny;
  int grid;
  const int bn = select_mttkrp_kernel(Mout, K, ny, N, 1, dp.sm_count, &grid, nullptr) - ADMMQ_MTTKRP_FOLDLONG;
  GemmMaps maps;
  if (int e = tc::make_operand_tmap(&maps.a, V, rows, K, ldv, tc::kTileM)) return e;
  if (int e = tc::make_operand_tmap(&maps.b, B, N, K, ldb, bn)) return e;
  if (int e = tc::make_operand_tmap(&maps.blo, Blo, N, K, ldb, bn)) return e;
  const int smem = tc::TileSmem<128, true>::kBytes;
  ADMMQ_CUDA_OK(cudaFuncSetAttribute(k_mttkrp_foldlong_tc<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  k_mttkrp_foldlong_tc<128><<<grid, tc::kThreadsTC, smem, stream>>>(maps, rows, ny, N, K, bn, Y, partial, -0.0f);
  const long long tot = (long long)Mout * N;
  k_fold_partials<<<(int)std::min<long long>((tot + 255) / 256, 148 * 4), 256, 0, stream>>>(partial, Mout, ny, N, F);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(2);
  return ADMMQ_OK;
}

}  // namespace admmq

using namespace admmq;

extern "C" int admmq_gemm_nt(const float* A, int lda, int M, const float* B, int ldb, int N, int K, float* C, int ldc,
                             void* stream_) {
  return gemm_nt(A, lda, M, B, nullptr, ldb, N, K, C, ldc, (cudaStream_t)stream_);
}

extern "C" int admmq_mttkrp_kernel(int M, int nx, int ny, int R, int precision, int sm_count, int* grid, int* splits) {
  if (M <= 0 || nx <= 0 || ny <= 0 || R <= 0 || sm_count <= 0 || precision < 0 || precision > 1)
    return fail(ADMMQ_E_BADARG, "admmq_mttkrp_kernel: bad argument");
  return select_mttkrp_kernel(M, nx, ny, R, precision, sm_count, grid, splits);
}
