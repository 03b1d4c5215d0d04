// search.cuh - CTA-level building blocks of the clip-search projection
// (quantize_tensor_mse, source/quantization.py:118-144), shared by the standalone
// projection kernels (project.cu) and the persistent ADMM loop (admm_loop.cu).
//
// Two forms of the per-candidate squared-error sums (cta_candidate_sums dispatches):
//   * the THRESHOLD form (cta_candidate_sums_binned, what the product runs): histogram + counting sort of the CTA's
//     elements, then one exact float32 threshold per (candidate, level) - O(1) work per element, see numerics.cuh;
//   * the DIRECT form (cta_candidate_sums_direct): every (element, candidate) pair evaluated with the reference's
//     float32 operations - kept for abs-max outside [2^-40, 2^40] and as the cross-check of the parity tests.
// Direct form, work split: the CTA's elements are staged through shared memory (cp.async, double buffered); every warp walks its
// slice of the stage in aligned groups of 8 elements read as warp-wide broadcasts (2 x LDS.128),
// and each LANE owns kCPL candidates (scale and 1/scale in registers, duplicated into both
// halves of a packed f32x2 register) -> no per-candidate warp reduction.  One candidate
// evaluation is ~6 issue slots: the multiplies/adds run as packed FFMA2/FADD2/FMUL2 on two
// elements at a time, only the clamp (FMNMX) and the boundary check (FMNMX3) are scalar.
// Group sums follow the group_sum8 / 64-element block recipe of numerics.cuh, go into float64 per lane, and the
// CTA total is converted to fixed point and added to the global per-candidate accumulators
// with integer atomics (order independent => deterministic for any grid size).
#pragma once
#include "common.cuh"
#include "numerics.cuh"

namespace admmq {

constexpr int kThreads = 512;               // CTA size of every kernel that uses these helpers
constexpr int kWarps = kThreads / 32;
constexpr int kCPL = 7;                     // candidates per lane per pass (200 = 6.25 * 32)
constexpr int kCandPerPass = 32 * kCPL;     // 224
constexpr int kStage = 4096;                // elements staged in shared memory at a time
constexpr int kGroup = kSumGroup;           // accumulation group (aligned, see numerics.cuh)
constexpr int kMaxCandidates = 1024;        // num_attempts limit (custom_benchmark.py uses 1000)
constexpr int kChunkAlign = 64;             // CTA chunks are multiples of this many elements

struct DirectSmem {
  __align__(16) float stage[2][kStage];  // double buffered: cp.async fills one while the warps evaluate the other
  double red[kWarps * kCandPerPass];
  unsigned long long key[kWarps];
};

// threshold ("binned") form of the search, see numerics.cuh
constexpr int kBins = 8192;        // linear bins over [-absmax, absmax]
constexpr int kBinSlots = kBins + kBins / 8;  // see bin_slot()
// elements sorted by bin in shared memory at a time: as many as fit next to the bin arrays in the 227 KB of a CTA (every
// further stage repeats the fixed costs of the scan and the threshold pass: a 20.7 k chunk took 27 us as two stages)
constexpr int kStageCap = 23296;
constexpr int kLoadBatch = 5;      // float4 loads in flight per thread
struct BinnedSmem {
  __align__(16) float sorted[kStageCap];   // the stage's elements grouped by bin
  // the three per-bin arrays are indexed by bin_slot(bin): four padding words after every 32 bins
  __align__(16) unsigned int cnt[kBinSlots];   // per-bin counts -> start offsets -> end offsets
  __align__(16) unsigned int slo[kBinSlots];   // per-bin fixed-point sums (low / high word) -> exclusive prefix sums
  __align__(16) unsigned int shi[kBinSlots];
  unsigned long long acc[kMaxCandidates];  // per-candidate fixed-point totals of this CTA (folded once per stage)
  unsigned int part[3][kMaxCandidates];    // the current stage's terms in three 21-bit slices (plain 32-bit adds, no return)
  float scale[kMaxCandidates];
  double mid[256];                         // per level: the midpoint of code_threshold() (depends on the level only)
  unsigned int odd[256];                   // ... and the parity of y*'s mantissa
  unsigned long long wsum[kWarps];
  unsigned int wcnt[kWarps];
  double red[kWarps];
};

union SearchSmem {
  DirectSmem direct;
  BinnedSmem binned;
};
static_assert(sizeof(SearchSmem) + 512 <= 227 * 1024, "the search scratch must fit the dynamic shared memory of one CTA");

// ---- packed pairs of float32 (two independent IEEE round-to-nearest operations per instruction).
// NOTE: ptxas fuses a single-use mul.rn.f32x2 feeding an add/sub.rn.f32x2 into one FFMA2 (unlike the
// scalar .rn forms), and it also folds fma(a, b, -0.0) back into a multiply when the -0.0 is a visible
// constant.  The product k*scale must be rounded on its own (the reference rounds `codes * scale`, then
// `x - xq`), so it is written as fma(k, scale, nz) with nz = -0.0 taken from a KERNEL PARAMETER, which
// ptxas cannot constant-fold: adding -0.0 is the identity for every value including both zeros.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// Elements [e0, e1) of the flattened tensor belong to this CTA.
__host__ __device__ inline long long chunk_size(long long n, int ctas) {
  long long c = (n + ctas - 1) / ctas;
  return (c + kChunkAlign - 1) / kChunkAlign * kChunkAlign;
}

// One candidate (scale s, 1/s duplicated in both halves) on two elements x = (x0, x1):
// acc += d*d per half with d = x - k*s, k = clamp(rint(x/s)) via the reciprocal + magic-number
// shortcut (numerics.cuh dev_fast); `worst` collects the distance of the quotient from its rounded value.
// 7 FMA-pipe (FMUL2, 4 x FADD2, 2 x FFMA2) + 2.5 ALU-pipe instructions per two evaluations.  (A 6-instruction variant
// that rounds the product with an FMA and takes the residual with a second FMA measured 13 % SLOWER on B200: four
// three-operand FFMA2 per pair lose more to register-bank conflicts than the saved FADD2 gains.)
__device__ __forceinline__ void eval_pair(f32x2 x, f32x2 s, f32x2 rc, const Levels& L, f32x2 magic, f32x2 nmagic,
                                          f32x2 nzero, f32x2& acc, float& worst) {
  const f32x2 t = mul2(x, rc);
  float t0, t1;
  unpack2(t, t0, t1);
  t0 = fminf(fmaxf(t0, L.fast_lo), L.fast_hi);
  t1 = fminf(fmaxf(t1, L.fast_lo), L.fast_hi);
  const f32x2 tc = pack2(t0, t1);
  const f32x2 k = add2(add2(tc, magic), nmagic);
  float f0, f1;
  unpack2(sub2(tc, k), f0, f1);
  worst = max3(worst, fabsf(f0), fabsf(f1));
  const f32x2 d = sub2(x, fma2(k, s, nzero));
  acc = fma2(d, d, acc);
}

// Adds this CTA's share of sum_e (x_e - Q_c(x_e))^2 for every candidate c < Nc into
// cand_sums[c] (fixed point, see numerics.cuh).  The CTA's elements are v[e0 .. e1) (contiguous).  On the E2M1 and the
// FP8 / FP6 grids every element takes the exact division; the summation recipe is the same.
template <Grid G = kGridInt>
__device__ inline void cta_candidate_sums_direct(const float* __restrict__ v, long long e0, long long e1, float absmax,
                                                 int Nc, const Levels L, double n_total, unsigned long long* cand_sums,
                                                 DirectSmem& sm, float opaque_neg_zero) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (e0 >= e1) return;  // uniform per CTA
  const ClipGrid g = make_clip_grid(absmax, Nc);
  const double unit_inv = fixed_point_unit_inv(n_total, absmax);
  const f32x2 magic = pack2(12582912.0f, 12582912.0f), nmagic = pack2(-12582912.0f, -12582912.0f);
  const f32x2 nzero = pack2(opaque_neg_zero, opaque_neg_zero);
  const bool vec_ok = ((reinterpret_cast<uintptr_t>(v + e0) & 15) == 0);  // e0 and kStage are multiples of 64
  const int nstage = (int)((e1 - e0 + kStage - 1) / kStage);
  // asynchronous fill of one stage buffer (16-byte copies when the source is aligned, 4-byte otherwise)
  auto fill = [&](int st) {
    const long long base = e0 + (long long)st * kStage;
    const int cnt = (int)min((long long)kStage, e1 - base);
    float* dst = sm.stage[st & 1];
    if (vec_ok) {
      for (int i = threadIdx.x * 4; i + 3 < cnt; i += kThreads * 4)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned int)__cvta_generic_to_shared(dst + i)),
                     "l"(v + base + i) : "memory");
      for (int i = (cnt & ~3) + threadIdx.x; i < cnt; i += kThreads)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned int)__cvta_generic_to_shared(dst + i)),
                     "l"(v + base + i) : "memory");
    } else {
      for (int i = threadIdx.x; i < cnt; i += kThreads)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned int)__cvta_generic_to_shared(dst + i)),
                     "l"(v + base + i) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  for (int c0 = 0; c0 < Nc; c0 += kCandPerPass) {
    f32x2 sc[kCPL], rc[kCPL];
    // per-lane float64 accumulators live in shared memory (sm.red[warp][candidate slot]): they are touched once per
    // 64-element block, and keeping them out of the register file keeps the 512-thread CTA under 128 registers
    double* dacc = &sm.red[warp * kCandPerPass + lane];
    __syncthreads();  // the previous pass / phase is done with both stage buffers and with sm.red
#pragma unroll
    for (int j = 0; j < kCPL; ++j) {
      const int c = c0 + j * 32 + lane;
      const float s = (c < Nc) ? SearchGrid<G>::scale(clip_candidate(g, c), L) : 1.0f;
      const float r = (c < Nc) ? div_rn(1.0f, s) : 0.0f;
      sc[j] = pack2(s, s);
      rc[j] = pack2(r, r);
      dacc[j * 32] = 0.0;
    }
    fill(0);
    for (int st = 0; st < nstage; ++st) {
      const long long base = e0 + (long long)st * kStage;
      const int cnt = (int)min((long long)kStage, e1 - base);
      const int cnt8 = (cnt + kGroup - 1) / kGroup * kGroup;  // zero padding contributes exactly 0
      float* stage = sm.stage[st & 1];
      if (st + 1 < nstage) {
        fill(st + 1);  // buffer (st+1)&1 was released by the barrier at the end of iteration st-1
        asm volatile("cp.async.wait_group 1;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
      if (threadIdx.x < cnt8 - cnt) stage[cnt + threadIdx.x] = 0.0f;
      __syncthreads();
      // warp slice, multiple of kSumBlock (base and e0 are multiples of kChunkAlign = kSumBlock)
      int per = (cnt8 + kWarps - 1) / kWarps;
      per = (per + kSumBlock - 1) / kSumBlock * kSumBlock;
      const int wb = min(warp * per, cnt8), we = min(wb + per, cnt8);
      float bacc[kCPL];
#pragma unroll
      for (int j = 0; j < kCPL; ++j) bacc[j] = 0.0f;
      for (int gb = wb; gb < we; gb += kGroup) {
        const ulonglong2 va = *reinterpret_cast<const ulonglong2*>(&stage[gb]);
        const ulonglong2 vb = *reinterpret_cast<const ulonglong2*>(&stage[gb + 4]);
        const f32x2 xs[4] = {va.x, va.y, vb.x, vb.y};
        f32x2 acc[kCPL];
        float worst = 0.0f;
        if constexpr (G == kGridInt) {
#pragma unroll
          for (int j = 0; j < kCPL; ++j) {
            acc[j] = 0ull;  // (+0.0f, +0.0f)
#pragma unroll
            for (int q = 0; q < 4; ++q) eval_pair(xs[q], sc[j], rc[j], L, magic, nmagic, nzero, acc[j], worst);
          }
        }
        // integer grid, rare: a quotient too close to a rounding boundary (or non-finite); the other grids: always
        if (G != kGridInt || !(worst <= L.fast_thr)) {
#pragma unroll
          for (int j = 0; j < kCPL; ++j) {
            float s0, s1, even = 0.0f, odd = 0.0f;
            unpack2(sc[j], s0, s1);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              float x0, x1;
              unpack2(xs[q], x0, x1);
              const float d0 = SearchGrid<G>::dev(x0, s0, L), d1 = SearchGrid<G>::dev(x1, s0, L);
              even = fma_rn(d0, d0, even);
              odd = fma_rn(d1, d1, odd);
            }
            acc[j] = pack2(even, odd);
          }
        }
#pragma unroll
        for (int j = 0; j < kCPL; ++j) {
          float even, odd;
          unpack2(acc[j], even, odd);
          bacc[j] = add_rn(bacc[j], add_rn(even, odd));
        }
        if (((gb + kGroup) & (kSumBlock - 1)) == 0 || gb + kGroup >= we) {  // end of an aligned 64-element block
#pragma unroll
          for (int j = 0; j < kCPL; ++j) {
            dacc[j * 32] += (double)bacc[j];
            bacc[j] = 0.0f;
          }
        }
      }
      __syncthreads();  // everyone is done with this buffer: it may be refilled two stages from now
    }
    // fixed-order reduction over the CTA's warps (the last stage ended with a barrier), one integer atomic per candidate
    if (threadIdx.x < kCandPerPass && c0 + (int)threadIdx.x < Nc) {
      double tot = 0.0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) tot += sm.red[w * kCandPerPass + threadIdx.x];
      const long long fx = __double2ll_rn(tot * unit_inv);
      atomicAdd(cand_sums + c0 + threadIdx.x, (unsigned long long)fx);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Threshold form (numerics.cuh): per stage of <= kStageCap elements
//   pass 1  histogram over kBins linear bins: count + 64-bit fixed-point sum per bin (shared-memory atomics; the 64-bit
//           sum as two 32-bit atomics with carry), sum of squares in float64
//   scan    exclusive prefix over the bins
//   pass 2  counting-sort scatter of the elements into `sorted` (grouped by bin)
//   pass 3  one (candidate, threshold) pair per thread: exact threshold, its bin, prefix + the bin's elements compared
//           one by one -> C, P -> float64 term -> fixed point -> per-candidate shared accumulator (three 21-bit slices)
// bin(x) is monotone in x, so every element in a lower bin is below the threshold and every element in a higher bin
// is not; only the threshold's own bin (kStageCap / kBins = 3 elements on average, ~7 in the central bins of bell-shaped data) is inspected.
__device__ __forceinline__ int bin_of(float x, float bmul) {
  const float t = fma_rn(x, bmul, 12582912.0f + (float)(kBins / 2));  // rne(x * bmul) + kBins / 2 in the low mantissa bits
  const int b = (int)__float_as_uint(t) - 0x4B400000;
  return min(max(b, 0), kBins - 1);
}

// A 64-bit fixed-point term f is accumulated as three 21-bit slices f = a0 + a1 2^21 + a2 2^42 (a2 signed): at most
// 2^8 terms per candidate and stage keep every slice inside 32 bits, and 32-bit shared-memory adds need no return
// value (the 64-bit shared atomic is a compare-and-swap loop).
__device__ __forceinline__ long long fold_slices(unsigned int a0, unsigned int a1, unsigned int a2) {
  return (long long)a0 + ((long long)a1 << 21) + (long long)((unsigned long long)(long long)(int)a2 << 42);
}

// Position of a bin in the per-bin arrays.  The scan reads 16 consecutive bins per thread as four 16-byte words; with
// the bins stored densely the threads of a quarter warp start 64 bytes apart and every such access is a 4-way bank
// conflict (ncu: 16 wavefronts instead of 4).  Four padding words after every 32 bins put the eight threads of a
// quarter warp on eight different groups of four banks.
__device__ __forceinline__ int bin_slot(int b) { return b + ((b >> 5) << 2); }

__device__ __forceinline__ float4 load_group4(const float* __restrict__ p, int gi, int ngroups, int cnt, bool vec_ok) {
  float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
  if (gi < ngroups) {
    const int i = gi * 4;
    if (vec_ok && i + 3 < cnt) {
      x = __ldcg(reinterpret_cast<const float4*>(p + i));
    } else {
      x.x = __ldcg(p + i);
      if (i + 1 < cnt) x.y = __ldcg(p + i + 1);
      if (i + 2 < cnt) x.z = __ldcg(p + i + 2);
      if (i + 3 < cnt) x.w = __ldcg(p + i + 3);
    }
  }
  return x;
}

template <Grid G = kGridInt>
__device__ inline void cta_candidate_sums_binned(const float* __restrict__ v, long long e0, long long e1, float absmax,
                                                 int Nc, const Levels L, int bits, double n_total,
                                                 unsigned long long* cand_sums, BinnedSmem& sm) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (e0 >= e1) return;  // uniform per CTA
  const ClipGrid g = make_clip_grid(absmax, Nc);
  const double unit_inv = fixed_point_unit_inv(n_total, absmax);
  const FixX fx = make_fix_x(absmax);
  const float bmul = div_rn((float)(kBins / 2), absmax);
  const int nthr = SearchGrid<G>::thresholds(bits, L);  // thresholds per candidate
  const int npairs = Nc * nthr;
  const bool vec_ok = ((reinterpret_cast<uintptr_t>(v + e0) & 15) == 0);
  __syncthreads();  // the previous phase is done with the shared memory
  for (int c = tid; c < Nc; c += kThreads) {
    sm.scale[c] = SearchGrid<G>::scale(clip_candidate(g, c), L);
    sm.acc[c] = 0ull;
    sm.part[0][c] = sm.part[1][c] = sm.part[2][c] = 0u;
  }
  for (int j = tid; j < nthr; j += kThreads) {
    const ThresholdMid tm = SearchGrid<G>::mid(j, L);
    sm.mid[j] = tm.mid;
    sm.odd[j] = tm.odd ? 1u : 0u;
  }
  double x2 = 0.0;
  for (long long base = e0; base < e1; base += kStageCap) {
    const int cnt = (int)min((long long)kStageCap, e1 - base);
    const int ngroups = (cnt + 3) >> 2;
    const float* __restrict__ src = v + base;
    for (int b = tid * 4; b < kBinSlots; b += kThreads * 4) {
      *reinterpret_cast<uint4*>(&sm.cnt[b]) = make_uint4(0u, 0u, 0u, 0u);
      *reinterpret_cast<uint4*>(&sm.slo[b]) = make_uint4(0u, 0u, 0u, 0u);
      *reinterpret_cast<uint4*>(&sm.shi[b]) = make_uint4(0u, 0u, 0u, 0u);
    }
    if (base != e0) {  // fold the previous stage's slices (its pass 3 ended with a barrier)
      for (int c = tid; c < Nc; c += kThreads) {
        sm.acc[c] += (unsigned long long)fold_slices(sm.part[0][c], sm.part[1][c], sm.part[2][c]);
        sm.part[0][c] = sm.part[1][c] = sm.part[2][c] = 0u;
      }
    }
    __syncthreads();
    // ---- pass 1: histogram
    for (int g0 = tid; g0 < ngroups; g0 += kThreads * kLoadBatch) {
      float4 xs[kLoadBatch];
#pragma unroll
      for (int u = 0; u < kLoadBatch; ++u) xs[u] = load_group4(src, g0 + u * kThreads, ngroups, cnt, vec_ok);
#pragma unroll
      for (int u = 0; u < kLoadBatch; ++u) {
        const int gi = g0 + u * kThreads;
        if (gi < ngroups) {
          const float xe[4] = {xs[u].x, xs[u].y, xs[u].z, xs[u].w};
          const int nv = min(4, cnt - gi * 4);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (q < nv) {
              const int b = bin_slot(bin_of(xe[q], bmul));
              atomicAdd(&sm.cnt[b], 1u);
              const long long f = fix_x(xe[q], fx);
              const unsigned int lo = (unsigned int)f, hi = (unsigned int)((unsigned long long)f >> 32);
              const unsigned int old = atomicAdd(&sm.slo[b], lo);
              atomicAdd(&sm.shi[b], hi + ((old + lo < old) ? 1u : 0u));
              const double xd = (double)xe[q];
              x2 = fma(xd, xd, x2);
            }
          }
        }
      }
    }
    __syncthreads();
    // ---- exclusive scan over the bins: thread t owns kBins / kThreads consecutive bins
    {
      constexpr int kPer = kBins / kThreads;
      static_assert(kPer % 4 == 0 && kPer * kThreads == kBins, "bins per thread");
      static_assert(kPer <= 32 && 32 % kPer == 0, "a thread's bins share one padded block");
      const int b0 = bin_slot(tid * kPer);
      unsigned int c[kPer], lo[kPer], hi[kPer];
#pragma unroll
      for (int i = 0; i < kPer; i += 4) {
        *reinterpret_cast<uint4*>(&c[i]) = *reinterpret_cast<const uint4*>(&sm.cnt[b0 + i]);
        *reinterpret_cast<uint4*>(&lo[i]) = *reinterpret_cast<const uint4*>(&sm.slo[b0 + i]);
        *reinterpret_cast<uint4*>(&hi[i]) = *reinterpret_cast<const uint4*>(&sm.shi[b0 + i]);
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
        c[i] = rc;
        lo[i] = (unsigned int)rs;
        hi[i] = (unsigned int)(rs >> 32);
        rc += cc;
        rs += ss;
      }
#pragma unroll
      for (int i = 0; i < kPer; i += 4) {
        *reinterpret_cast<uint4*>(&sm.cnt[b0 + i]) = *reinterpret_cast<const uint4*>(&c[i]);
        *reinterpret_cast<uint4*>(&sm.slo[b0 + i]) = *reinterpret_cast<const uint4*>(&lo[i]);
        *reinterpret_cast<uint4*>(&sm.shi[b0 + i]) = *reinterpret_cast<const uint4*>(&hi[i]);
      }
    }
    __syncthreads();
    // ---- pass 2: scatter (cnt[b] runs from the start to the end of bin b)
    for (int g0 = tid; g0 < ngroups; g0 += kThreads * kLoadBatch) {
      float4 xs[kLoadBatch];
#pragma unroll
      for (int u = 0; u < kLoadBatch; ++u) xs[u] = load_group4(src, g0 + u * kThreads, ngroups, cnt, vec_ok);
#pragma unroll
      for (int u = 0; u < kLoadBatch; ++u) {
        const int gi = g0 + u * kThreads;
        if (gi < ngroups) {
          const float xe[4] = {xs[u].x, xs[u].y, xs[u].z, xs[u].w};
          const int nv = min(4, cnt - gi * 4);
          unsigned int pos[4];
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (q < nv) pos[q] = atomicAdd(&sm.cnt[bin_slot(bin_of(xe[q], bmul))], 1u);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (q < nv) sm.sorted[pos[q]] = xe[q];
        }
      }
    }
    __syncthreads();
    // ---- pass 3: thresholds.  pair p = j * Nc + c: neighbouring threads take neighbouring candidates of the same
    // level, whose thresholds fall into neighbouring bins and whose accumulators are distinct.  (Working on two pairs
    // at a time to hide the dependent chain was measured: no gain, the phase is issue bound.)
    {
      long long ptot = 0ll;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) ptot += (long long)sm.wsum[w];
      // fix_x() split into its two integer parts, accumulated separately (int32 is enough for 512 elements at a time)
      auto take = [&](float x, float theta, int& sth, int& stl, int& below) {
        const float hb = fma_rn(x, fx.p2a, 12582912.0f);
        const float r = fma_rn(x, fx.p2a, -sub_rn(hb, 12582912.0f));
        const float lb = fma_rn(r, 1048576.0f, 12582912.0f);
        const bool in = x < theta;
        sth += in ? (int)__float_as_uint(hb) - 0x4B400000 : 0;
        stl += in ? (int)__float_as_uint(lb) - 0x4B400000 : 0;
        below += in ? 1 : 0;
      };
      // (level, candidate) of the thread's pairs without a division per pair
      int j = tid / Nc, c = tid - j * Nc;
      const int dj = kThreads / Nc, dc = kThreads - dj * Nc;
      for (int p = tid; p < npairs; p += kThreads, j += dj, c += dc) {
        if (c >= Nc) {
          c -= Nc;
          ++j;
        }
        const float s = sm.scale[c];
        const float theta = code_threshold_from_mid(s, sm.mid[j], sm.odd[j] != 0u);
        const int bin = bin_of(theta, bmul), b = bin_slot(bin);
        const unsigned int beg = bin ? sm.cnt[bin_slot(bin - 1)] : 0u, end = sm.cnt[b];
        long long ps = (long long)(((unsigned long long)sm.shi[b] << 32) | sm.slo[b]);
        long long cn = (long long)beg;
        // the threshold's own bin, two elements per step
        for (unsigned int i0 = beg; i0 < end; i0 += 512u) {
          const unsigned int i1 = min(end, i0 + 512u);
          int sth = 0, stl = 0, below = 0;
          unsigned int i = i0;
          for (; i + 1u < i1; i += 2u) {
            const float x0 = sm.sorted[i], x1 = sm.sorted[i + 1u];
            take(x0, theta, sth, stl, below);
            take(x1, theta, sth, stl, below);
          }
          if (i < i1) take(sm.sorted[i], theta, sth, stl, below);
          cn += below;
          ps += (long long)sth * 1048576ll + (long long)stl;
        }
        double term = SearchGrid<G>::term(s, j, L, cn, ps, fx.unit);
        if (j == nthr - 1) term += closing_term(s, SearchGrid<G>::top(L), (long long)cnt, ptot, fx.unit);
        const long long f = __double2ll_rn(term * unit_inv);
        atomicAdd(&sm.part[0][c], (unsigned int)(f & 0x1fffffll));
        atomicAdd(&sm.part[1][c], (unsigned int)((f >> 21) & 0x1fffffll));
        atomicAdd(&sm.part[2][c], (unsigned int)(int)(f >> 42));
      }
    }
    __syncthreads();
  }
  // ---- sum of squares: fixed-order reduction over the CTA, then one integer atomic per candidate
  x2 = warp_sum(x2);
  if (lane == 0) sm.red[warp] = x2;
  __syncthreads();
  double tot = 0.0;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) tot += sm.red[w];
  const long long x2f = __double2ll_rn(tot * unit_inv);
  for (int c = tid; c < Nc; c += kThreads) {
    const long long f = (long long)sm.acc[c] + fold_slices(sm.part[0][c], sm.part[1][c], sm.part[2][c]) + x2f;  // >= 0 up to rounding
    atomicAdd(cand_sums + c, (unsigned long long)max(f, 0ll));
  }
}

// Dispatch: threshold form when absmax is in its supported range and the form is the cheaper one, direct evaluation
// otherwise (and on request)
constexpr int kFormAuto = 0, kFormDirect = 1, kFormThresholds = 2;
// cost of one (candidate, threshold) pair in (element, candidate) evaluations of the direct form: measured ~1.1 ns against
// ~69 ps on B200 (tools/time_search.py crossover: break-even near 5 k elements per CTA with 8 bits, 1.3 k with 6, and
// no difference below 1 k with 4)
constexpr int kPairsPerElement = 18;
template <Grid G = kGridInt>
__device__ inline void cta_candidate_sums(const float* __restrict__ v, long long e0, long long e1, float absmax, int Nc,
                                          const Levels L, int bits, double n_total, unsigned long long* cand_sums,
                                          SearchSmem& sm, float opaque_neg_zero, int form = kFormAuto, int direct_below = 0) {
  // Both forms give the same sums up to the last fixed-point unit, so each CTA may take the cheaper one for its chunk: the threshold form
  // pays per (candidate, threshold) pair and stage on top of O(1) per element, the direct form per (element, candidate);
  // with 8 bits (255 thresholds) the direct form wins below ~4.6 k elements per stage, with 4 bits never in practice.
  const long long elems = e1 - e0;
  const long long stages = (elems + kStageCap - 1) / kStageCap;
  // ... and below `direct_below` elements per CTA the fixed costs of the threshold form (zeroing and scanning 8192 bins,
  // (2^bits - 1) x candidates thresholds however few elements there are) dominate: small factors spread over many CTAs
  // (up to 4 bits = 15 thresholds the threshold form is never the slower one: measured inside the loop 10.8 against 13.4 us
  // per iteration at 214 elements per CTA, and equal in the stand-alone search at 285, profiles/r1g_search_crossover.txt)
  const bool direct_is_cheaper = (bits > 4 && (long long)((1 << bits) - 1) * stages * kPairsPerElement > elems) || elems <= direct_below;
  const bool want_direct = form == kFormDirect || (form == kFormAuto && direct_is_cheaper);
  if (!want_direct && binned_range_ok(absmax))
    cta_candidate_sums_binned<G>(v, e0, e1, absmax, Nc, L, bits, n_total, cand_sums, sm.binned);
  else
    cta_candidate_sums_direct<G>(v, e0, e1, absmax, Nc, L, n_total, cand_sums, sm.direct, opaque_neg_zero);
}

// First index of the smallest MSE (torch.argmin, source/quantization.py:141), evaluated redundantly by every CTA from
// the fixed-point sums: global sums written by other CTAs are read with __ldcg (Ldcg), sums in shared memory with plain
// loads.  wkey is kWarps words of shared scratch that no thread may still be reading.  Returns the index to all threads.
template <bool Ldcg>
__device__ inline int cta_best_candidate(const unsigned long long* cand_sums, int Nc, float absmax, double n_total,
                                         unsigned long long* wkey) {
  const double unit = fixed_point_unit(n_total, absmax);
  const float nf = (float)n_total;
  unsigned long long best = ~0ull;
  for (int c = threadIdx.x; c < Nc; c += kThreads) {
    const long long fx = (long long)(Ldcg ? __ldcg(cand_sums + c) : cand_sums[c]);
    const float mse = mse_from_fixed(fx, unit, nf);
    const unsigned long long key = ((unsigned long long)float_key(mse) << 32) | (unsigned int)c;
    best = min(best, key);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0) wkey[threadIdx.x >> 5] = best;
  __syncthreads();
  unsigned long long b = wkey[0];
#pragma unroll
  for (int w = 1; w < kWarps; ++w) b = min(b, wkey[w]);
  return (int)(b & 0xffffffffu);
}

static_assert(kFmtE4M3 == ADMMQ_Q_MSEMINMAX_E4M3 && kFmtE5M2 == ADMMQ_Q_MSEMINMAX_E5M2 &&
              kFmtE3M2 == ADMMQ_Q_MSEMINMAX_E3M2 && kFmtE2M3 == ADMMQ_Q_MSEMINMAX_E2M3, "the FP format is the scheme id");

// The scheme takes its scale from the clip search, in a kernel instantiated for grid G: quantize_tensor_mse on the
// integer grid or on the E2M1 grid.  A kernel instantiated for the E2M1 or the FP8 / FP6 grids runs no other scheme;
// the integer grid's instantiations never see an FP8 / FP6 scheme (grid_of).
template <Grid G = kGridInt>
__host__ __device__ __forceinline__ bool clip_search_scheme(int scheme) {
  return G != kGridInt || scheme == ADMMQ_Q_MSEMINMAX_SYMMETRIC || scheme == ADMMQ_Q_MSEMINMAX_E2M1;
}

// which instantiation runs a scheme (host side)
inline Grid grid_of(int scheme) {
  return scheme == ADMMQ_Q_MSEMINMAX_E2M1 ? kGridE2M1 : fp_format_id(scheme) ? kGridFP : kGridInt;
}

// scale of clip candidate `best` (source/quantization.py:141-144)
template <Grid G = kGridInt>
__device__ __forceinline__ float clip_scale(float absmax, int Nc, int best, const Levels& L) {
  return SearchGrid<G>::scale(clip_candidate(make_clip_grid(absmax, Nc), best), L);
}

// Parameters of the non-search schemes from the tensor's min / max (source/quantization.py:48-66, 91-106)
__device__ inline QParams params_from_minmax(int scheme, int bits, float tmin, float tmax, const Levels& L) {
  QParams p;
  p.scheme = scheme;
  p.bits = bits;
  p.n = (float)((1u << bits) - 1u);
  p.aux = 0.0f;
  p.scale = 0.0f;
  if (scheme == ADMMQ_Q_MINMAX) {
    p.scale = sub_rn(tmax, tmin);
    p.aux = tmin;
  } else if (scheme == ADMMQ_Q_SYMMETRIC) {
    const float a = fabsf(tmin);
    p.scale = div_rn(mul_rn(2.0f, (a > tmax) ? a : tmax), L.denom);
  } else if (scheme == ADMMQ_Q_AFFINE) {
    p.scale = div_rn(sub_rn(tmax, tmin), L.denom);
    p.aux = affine_zero_point(tmin, p.scale, L);
  }
  return p;
}

// value on the grid and its integer code for any scheme
__device__ __forceinline__ float quantize_value(float x, const QParams& p, const Levels& L, float& code) {
  if (p.scheme == ADMMQ_Q_MINMAX) {
    float level;
    const float v = minmax_value(x, p, level);
    code = (p.bits == 1) ? level : level - (float)(1 << (p.bits - 1));
    return v;
  }
  if (p.scheme == ADMMQ_Q_AFFINE) return affine_value(x, p, L, code);
  code = code_exact(x, p.scale, L);
  // tensor_symmetric multiplies the INTEGER code by the scale (source/quantization.py:95 `.to(int)`),
  // which has no negative zero; the clip search (:127, :144) stays in float and keeps -0.
  if (p.scheme == ADMMQ_Q_SYMMETRIC) code = add_rn(code, 0.0f);
  return mul_rn(code, p.scale);
}

}  // namespace admmq
