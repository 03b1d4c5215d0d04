// common.cuh - error plumbing, device-wide barrier and small reduction helpers.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include "../../include/admmq.h"

namespace admmq {

// ---- thread-local error string behind admmq_last_error() -------------------------------
char* error_buffer();
int fail(int code, const char* fmt, ...);

#define ADMMQ_CUDA_OK(expr)                                                                   \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess)                                                                    \
      return ::admmq::fail(ADMMQ_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                           __FILE__, __LINE__);                                               \
  } while (0)

// process-wide count of kernel launches (admmq_launch_count)
void count_launches(int n);

struct DeviceProps {
  int sm_count = 0, cc_major = 0, cc_minor = 0, coop = 0;
  size_t smem_optin = 0;
  int device = -1;
};
int device_props(DeviceProps* out);

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- the quantization schemes as the entry points check them (include/admmq.h)
// the width a scheme requires and its name: the E2M1 and FP8 / FP6 grids have one; 0 for the reference's schemes
inline int scheme_bits(int scheme, const char** name) {
  switch (scheme) {
    case ADMMQ_Q_MSEMINMAX_E2M1: *name = "tensor_mseminmax_e2m1"; return 4;
    case ADMMQ_Q_MSEMINMAX_E4M3: *name = "tensor_mseminmax_e4m3"; return 8;
    case ADMMQ_Q_MSEMINMAX_E5M2: *name = "tensor_mseminmax_e5m2"; return 8;
    case ADMMQ_Q_MSEMINMAX_E3M2: *name = "tensor_mseminmax_e3m2"; return 6;
    case ADMMQ_Q_MSEMINMAX_E2M3: *name = "tensor_mseminmax_e2m3"; return 6;
    default: *name = nullptr; return 0;
  }
}
inline bool known_scheme(int scheme) {
  const char* name;
  return (scheme >= ADMMQ_Q_MSEMINMAX_SYMMETRIC && scheme <= ADMMQ_Q_AFFINE) || scheme_bits(scheme, &name) != 0;
}
// the scale comes from the clip search: tensor_mseminmax_symmetric and every fixed-width grid
inline bool has_clip_search(int scheme) {
  const char* name;
  return scheme == ADMMQ_Q_MSEMINMAX_SYMMETRIC || scheme_bits(scheme, &name) != 0;
}
// ADMMQ_OK, or the failure for a width the scheme does not take
inline int check_scheme_bits(const char* who, int scheme, int bits) {
  const char* name;
  const int want = scheme_bits(scheme, &name);
  if (want != 0 && bits != want) return fail(ADMMQ_E_BADARG, "%s: %s needs bits = %d, got %d", who, name, want, bits);
  return ADMMQ_OK;
}

#if defined(__CUDACC__)
// ---- device-wide barrier for cooperative (co-resident) grids ----------------------------
// Monotonic ticket counter in global memory: barrier k completes when the counter reaches
// k * gridDim.x.  The CTA's writes are ordered before thread 0's arrival by bar.sync (CTA scope) followed by the
// gpu-scope RELEASE of the arrival itself (release is cumulative over the writes thread 0 has observed through the
// barrier), and other CTAs' writes are ordered before the departure by the gpu-scope ACQUIRE load that sees the final
// count, again extended to the whole CTA by bar.sync - no separate membar.gl on either side (each cost ~0.4 us with
// stores in flight).  Data produced by other CTAs is read with ld.global.cg (L2) afterwards, so no L1 staleness is
// possible.
struct GridBarrier {
  unsigned int* counter;
  unsigned int target;
  __device__ __forceinline__ void init(unsigned int* c) {
    counter = c;
    target = 0;
  }
  __device__ __forceinline__ void sync() {
    __syncthreads();
    target += gridDim.x;
    if (threadIdx.x == 0) {
      asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(counter), "r"(1u) : "memory");
      unsigned int seen;
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
      } while ((int)(seen - target) < 0);
    }
    __syncthreads();
  }
};

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ float ldcg(const float* p) { return __ldcg(p); }
__device__ __forceinline__ double ldcg(const double* p) { return __ldcg(p); }
__device__ __forceinline__ long long ldcg(const long long* p) { return __ldcg(p); }
__device__ __forceinline__ unsigned int ldcg(const unsigned int* p) { return __ldcg(p); }
__device__ __forceinline__ int ldcg(const int* p) { return __ldcg(p); }

// order-preserving map float -> uint32 (larger float <=> larger key); NaN maps above +inf
__device__ __forceinline__ unsigned int float_key(float f) {
  const unsigned int b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_float(unsigned int k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ unsigned int warp_max_u32(unsigned int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
#endif  // __CUDACC__

}  // namespace admmq
