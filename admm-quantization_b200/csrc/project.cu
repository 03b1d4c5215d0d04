// project.cu - standalone projection onto the b-bit grid (admmq_project).
// Replaces quantize_tensor / quantize_tensor_mse / min_max_quantize of
// source/quantization.py:48-144 for the tensor_* schemes.
//
// Three launches on the caller's stream:
//   k_minmax_keys   min and max of x as order-preserving integer keys (atomicMax)
//   k_mse_sums      per-candidate squared-error sums (only for the clip-search schemes: tensor_mseminmax_symmetric,
//                   tensor_mseminmax_e2m1 and the FP8 / FP6 grids, k_mse_sums_fp)
//   k_apply         argmin (redundantly per CTA) + quantize + codes
// HBM traffic: x is read 2x (4x for the clip search), xq written once: 12-20 B/element.  The clip search runs in its
// threshold form (search.cuh / numerics.cuh): O(1) work per element plus (2^bits - 1) * num_attempts thresholds per
// CTA, instead of num_attempts evaluations per element (kept as the direct form for extreme magnitudes and as a
// cross-check, admmq_clip_search_sums).
#include "search.cuh"

namespace admmq {

struct ProjectHeader {        // lives at the start of the workspace, zeroed by cudaMemsetAsync
  unsigned int max_key;       // max over float_key(x)
  unsigned int inv_min_key;   // max over ~float_key(x)  ==  ~min key
  unsigned int pad[2];
};

__global__ void __launch_bounds__(kThreads) k_minmax_keys(const float* x, long long n, ProjectHeader* hdr) {
  unsigned int kmax = 0u, kinv = 0u;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) {
    const unsigned int k = float_key(x[i]);
    kmax = max(kmax, k);
    kinv = max(kinv, ~k);
  }
  kmax = warp_max_u32(kmax);
  kinv = warp_max_u32(kinv);
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&hdr->max_key, kmax);
    atomicMax(&hdr->inv_min_key, kinv);
  }
}

__device__ __forceinline__ void read_minmax(const ProjectHeader* hdr, float& tmin, float& tmax, float& absmax) {
  tmax = key_float(__ldcg(&hdr->max_key));
  tmin = key_float(~__ldcg(&hdr->inv_min_key));
  absmax = fmaxf(fabsf(tmin), fabsf(tmax));  // source/quantization.py:129
  if (tmin != tmin || tmax != tmax) absmax = __int_as_float(0x7fc00000);
}

template <Grid G>
__device__ __forceinline__ void mse_sums(const float* x, long long n, int bits, int fmt, int Nc, const ProjectHeader* hdr,
                                         unsigned long long* cand_sums, float neg_zero, int form) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SearchSmem& sm = *reinterpret_cast<SearchSmem*>(smem_raw);
  float tmin, tmax, absmax;
  read_minmax(hdr, tmin, tmax, absmax);
  if (!(absmax > 0.0f) || isinf(absmax)) return;  // all-zero / non-finite input: output is NaN (k_apply)
  const Levels L = make_levels(bits, fmt);
  const long long cs = chunk_size(n, gridDim.x);
  const long long e0 = min(n, (long long)blockIdx.x * cs), e1 = min(n, e0 + cs);
  cta_candidate_sums<G>(x, e0, e1, absmax, Nc, L, bits, (double)n, cand_sums, sm, neg_zero, form);
}
// the integer and the E2M1 grid
template <Grid G>
__global__ void __launch_bounds__(kThreads) k_mse_sums(const float* x, long long n, int bits, int Nc,
                                                      const ProjectHeader* hdr, unsigned long long* cand_sums,
                                                      float neg_zero, int form) {
  mse_sums<G>(x, n, bits, 0, Nc, hdr, cand_sums, neg_zero, form);
}
// the FP8 / FP6 grids: the format (the scheme id) is one more parameter
__global__ void __launch_bounds__(kThreads) k_mse_sums_fp(const float* x, long long n, int bits, int Nc,
                                                         const ProjectHeader* hdr, unsigned long long* cand_sums,
                                                         float neg_zero, int form, int fmt) {
  mse_sums<kGridFP>(x, n, bits, fmt, Nc, hdr, cand_sums, neg_zero, form);
}

// G: the integer grid runs the reference's four schemes, the E2M1 and FP8 / FP6 instantiations their own schemes
template <Grid G>
__global__ void __launch_bounds__(kThreads) k_apply(const float* x, long long n, int bits, int scheme, int Nc,
                                                   const ProjectHeader* hdr, const unsigned long long* cand_sums,
                                                   const float* tmin_in, const float* tmax_in, float* xq,
                                                   int8_t* codes, float* info) {
  __shared__ unsigned long long wkey[kWarps];
  float tmin, tmax, absmax;
  read_minmax(hdr, tmin, tmax, absmax);
  const Levels L = make_levels(bits, G == kGridFP ? scheme : 0);
  QParams p;
  int best = -1;
  bool nan_fill = false;
  if (clip_search_scheme<G>(scheme)) {
    p.scheme = scheme;
    p.bits = bits;
    p.aux = 0.0f;
    p.n = 0.0f;
    if (!(absmax > 0.0f) || isinf(absmax)) {
      nan_fill = true;  // reference: scale 0 or inf/NaN -> every output NaN (SURVEY App. A.3 item 6)
      p.scale = __int_as_float(0x7fc00000);
    } else {
      best = cta_best_candidate<true>(cand_sums, Nc, absmax, (double)n, wkey);
      p.scale = clip_scale<G>(absmax, Nc, best, L);
    }
  } else {
    if (scheme == ADMMQ_Q_AFFINE && tmin_in != nullptr && tmax_in != nullptr) {
      tmin = *tmin_in;
      tmax = *tmax_in;
    }
    p = params_from_minmax(scheme, bits, tmin, tmax, L);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && info != nullptr) {
    info[0] = p.scale;
    info[1] = p.aux;
    info[2] = (float)best;
    info[3] = absmax;
  }
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < n; i += (long long)gridDim.x * kThreads) {
    float code = 0.0f;
    float v;
    if (nan_fill) {
      v = __int_as_float(0x7fc00000);
    } else if constexpr (G == kGridE2M1) {
      v = e2m1_quantize(x[i], p.scale, code);
    } else if constexpr (G == kGridFP) {
      v = fp_quantize(x[i], p.scale, L.fmt, code);
    } else {
      v = quantize_value(x[i], p, L, code);
    }
    xq[i] = v;
    if (codes != nullptr) codes[i] = (int8_t)code;
  }
}

// per-candidate sums of squared errors as float64 (admmq_clip_search_sums)
__global__ void k_sums_to_double(const unsigned long long* cand_sums, const ProjectHeader* hdr, long long n, int Nc,
                                 double* out) {
  float tmin, tmax, absmax;
  read_minmax(hdr, tmin, tmax, absmax);
  const double unit = fixed_point_unit((double)n, absmax);
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < Nc; c += gridDim.x * blockDim.x)
    out[c] = (double)(long long)cand_sums[c] * unit;
}

// E2M1 codes of t by the hardware conversion (admmq_e2m1_encode)
__global__ void k_e2m1_encode(const float* t, long long n, int8_t* codes) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    codes[i] = (int8_t)e2m1_code(t[i]);
}

// FP8 / FP6 codes of t by the hardware conversion (admmq_fp_encode)
__global__ void k_fp_encode(const float* t, long long n, int fmt, int8_t* codes) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    codes[i] = (int8_t)fp_code(fmt, t[i]);
}

}  // namespace admmq

using namespace admmq;

extern "C" size_t admmq_project_workspace_bytes(int64_t n, int num_attempts) {
  (void)n;
  const int nc = num_attempts > 0 ? num_attempts : 1;
  return align_up(sizeof(ProjectHeader), 256) + align_up((size_t)nc * sizeof(unsigned long long), 256);
}

static int launch_mse_sums(const float* x, int64_t n, int bits, int qscheme, int num_attempts, ProjectHeader* hdr,
                           unsigned long long* cand, int form, int max_ctas, const DeviceProps& dp, cudaStream_t stream) {
  // one chunk of >= 512 elements per CTA, at most one CTA per SM
  const long long want = (n + 511) / 512;
  int g = (int)std::max<long long>(1, std::min<long long>((long long)dp.sm_count, want));
  if (max_ctas > 0) g = std::min(g, max_ctas);
  if (grid_of(qscheme) == kGridFP) {
    ADMMQ_CUDA_OK(cudaFuncSetAttribute(k_mse_sums_fp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SearchSmem)));
    k_mse_sums_fp<<<g, kThreads, sizeof(SearchSmem), stream>>>(x, n, bits, num_attempts, hdr, cand, -0.0f, form, qscheme);
    return ADMMQ_OK;
  }
  auto kernel = grid_of(qscheme) == kGridE2M1 ? k_mse_sums<kGridE2M1> : k_mse_sums<kGridInt>;
  ADMMQ_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SearchSmem)));
  kernel<<<g, kThreads, sizeof(SearchSmem), stream>>>(x, n, bits, num_attempts, hdr, cand, -0.0f, form);
  return ADMMQ_OK;
}

extern "C" int admmq_clip_search_sums_scheme(const float* x, int64_t n, int bits, int qscheme, int num_attempts, int method,
                                             int max_ctas, double* sums, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (x == nullptr || sums == nullptr || n <= 0) return fail(ADMMQ_E_BADARG, "admmq_clip_search_sums: null pointer or n <= 0");
  if (bits < 1 || bits > 8) return fail(ADMMQ_E_BADARG, "admmq_clip_search_sums: bits must be in 1..8, got %d", bits);
  if (!has_clip_search(qscheme)) return fail(ADMMQ_E_BADARG, "admmq_clip_search_sums: qscheme %d has no clip search", qscheme);
  if (int e = check_scheme_bits("admmq_clip_search_sums", qscheme, bits)) return e;
  if (num_attempts < 1 || num_attempts > kMaxCandidates)
    return fail(ADMMQ_E_BADARG, "admmq_clip_search_sums: num_attempts must be in 1..%d", kMaxCandidates);
  if (method != 0 && method != 1) return fail(ADMMQ_E_BADARG, "admmq_clip_search_sums: method must be 0 (direct) or 1 (thresholds)");
  if (workspace == nullptr || workspace_bytes < admmq_project_workspace_bytes(n, num_attempts) ||
      ((uintptr_t)workspace & 15) != 0)
    return fail(ADMMQ_E_WORKSPACE, "admmq_clip_search_sums: workspace too small or misaligned");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  ProjectHeader* hdr = (ProjectHeader*)workspace;
  unsigned long long* cand = (unsigned long long*)((char*)workspace + align_up(sizeof(ProjectHeader), 256));
  ADMMQ_CUDA_OK(cudaMemsetAsync(workspace, 0, admmq_project_workspace_bytes(n, num_attempts), stream));
  const int g_stream = (int)std::min<long long>((long long)dp.sm_count * 4, (n + kThreads * 4 - 1) / (kThreads * 4));
  k_minmax_keys<<<std::max(g_stream, 1), kThreads, 0, stream>>>(x, n, hdr);
  if (int e = launch_mse_sums(x, n, bits, qscheme, num_attempts, hdr, cand, method == 0 ? kFormDirect : kFormThresholds,
                              max_ctas, dp, stream))
    return e;
  k_sums_to_double<<<(num_attempts + 255) / 256, 256, 0, stream>>>(cand, hdr, n, num_attempts, sums);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(3);
  return ADMMQ_OK;
}

extern "C" int admmq_clip_search_sums(const float* x, int64_t n, int bits, int num_attempts, int method, int max_ctas,
                                      double* sums, void* workspace, size_t workspace_bytes, void* stream) {
  return admmq_clip_search_sums_scheme(x, n, bits, ADMMQ_Q_MSEMINMAX_SYMMETRIC, num_attempts, method, max_ctas, sums,
                                       workspace, workspace_bytes, stream);
}

extern "C" int admmq_e2m1_encode(const float* t, int64_t n, int8_t* codes, void* stream_) {
  if (t == nullptr || codes == nullptr || n <= 0) return fail(ADMMQ_E_BADARG, "admmq_e2m1_encode: null pointer or n <= 0");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  const int g = (int)std::max<long long>(1, std::min<long long>((long long)dp.sm_count * 4, (n + 255) / 256));
  k_e2m1_encode<<<g, 256, 0, (cudaStream_t)stream_>>>(t, n, codes);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

extern "C" int admmq_fp_encode(const float* t, int64_t n, int qscheme, int8_t* codes, void* stream_) {
  if (t == nullptr || codes == nullptr || n <= 0) return fail(ADMMQ_E_BADARG, "admmq_fp_encode: null pointer or n <= 0");
  if (!fp_format_id(qscheme)) return fail(ADMMQ_E_BADARG, "admmq_fp_encode: qscheme %d is no FP8 / FP6 grid", qscheme);
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  const int g = (int)std::max<long long>(1, std::min<long long>((long long)dp.sm_count * 4, (n + 255) / 256));
  k_fp_encode<<<g, 256, 0, (cudaStream_t)stream_>>>(t, n, qscheme, codes);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(1);
  return ADMMQ_OK;
}

extern "C" int admmq_project(const float* x, int64_t n, int bits, int qscheme, int num_attempts,
                             const float* tmin, const float* tmax, float* xq, int8_t* codes, float* info,
                             void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (x == nullptr || xq == nullptr || n <= 0) return fail(ADMMQ_E_BADARG, "admmq_project: null pointer or n <= 0");
  if (bits < 1 || bits > 8) return fail(ADMMQ_E_BADARG, "admmq_project: bits must be in 1..8, got %d", bits);
  if (!known_scheme(qscheme)) return fail(ADMMQ_E_BADARG, "admmq_project: unknown qscheme %d", qscheme);
  if (int e = check_scheme_bits("admmq_project", qscheme, bits)) return e;
  if (has_clip_search(qscheme) && (num_attempts < 1 || num_attempts > kMaxCandidates))
    return fail(ADMMQ_E_BADARG, "admmq_project: num_attempts must be in 1..%d, got %d", kMaxCandidates, num_attempts);
  if (workspace == nullptr || workspace_bytes < admmq_project_workspace_bytes(n, num_attempts) ||
      ((uintptr_t)workspace & 15) != 0)
    return fail(ADMMQ_E_WORKSPACE, "admmq_project: workspace too small or misaligned");
  DeviceProps dp;
  if (int e = device_props(&dp)) return e;
  ProjectHeader* hdr = (ProjectHeader*)workspace;
  unsigned long long* cand = (unsigned long long*)((char*)workspace + align_up(sizeof(ProjectHeader), 256));
  ADMMQ_CUDA_OK(cudaMemsetAsync(workspace, 0, admmq_project_workspace_bytes(n, num_attempts), stream));
  const long long max_ctas = (long long)dp.sm_count * 4;
  const int g_stream = (int)std::min<long long>(max_ctas, (n + kThreads * 4 - 1) / (kThreads * 4));
  k_minmax_keys<<<std::max(g_stream, 1), kThreads, 0, stream>>>(x, n, hdr);
  if (has_clip_search(qscheme)) {
    if (int e = launch_mse_sums(x, n, bits, qscheme, num_attempts, hdr, cand, kFormAuto, 0, dp, stream)) return e;
  }
  const Grid qgrid = grid_of(qscheme);
  auto apply = qgrid == kGridE2M1 ? k_apply<kGridE2M1> : qgrid == kGridFP ? k_apply<kGridFP> : k_apply<kGridInt>;
  apply<<<std::max(g_stream, 1), kThreads, 0, stream>>>(x, n, bits, qscheme, num_attempts, hdr, cand, tmin, tmax, xq,
                                                        codes, info);
  ADMMQ_CUDA_OK(cudaGetLastError());
  count_launches(has_clip_search(qscheme) ? 3 : 2);
  return ADMMQ_OK;
}
