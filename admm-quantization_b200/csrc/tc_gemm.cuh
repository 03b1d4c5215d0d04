// tc_gemm.cuh - 3xTF32 tile product on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
//   D[128 x bn] (TMEM, float32) = A[128 x K] . B[bn x K]^T          A, B: float32, K-major, bn <= BN, bn % 16 == 0
//
// Every float32 operand x is split as x = hi + lo + O(2^-22 |x|) with hi = tf32_rn(x), lo = tf32_rn(x - hi), and
// the tile is accumulated as (lo.hi + hi.lo) + hi.hi by three tcgen05.mma.kind::tf32 per 8-deep k-step: the two
// cross terms into one TMEM accumulator, hi.hi into another, added small-terms-first by the epilogue.  This keeps
// float32-level accuracy (the dropped lo.lo term and the split residuals are 2^-22 relative) at 1/3 of the TF32 rate.
//
// Operand paths.  Measured on B200: with BOTH operands in shared memory one tcgen05.mma of 128 x N x 8 tf32 costs
// ~90 cycles for every N <= 64 - the tensor core re-reads the 128-row A slab (32 bytes from each of 128 rows) for
// every instruction - so narrow tiles, which this path needs to keep 148 SMs busy on 512 x 1141 outputs, were
// MMA-issue bound.  The A operand therefore lives in TENSOR MEMORY (TS form of tcgen05.mma): lane = tile row,
// column = k, written there by the converter warps with tcgen05.st, and only the small B slab (N rows x 32 bytes) is
// read from shared memory per instruction (measured 25 / 31 / 38 cycles per MMA at N = 32 / 48 / 64; floor N / 2).
//
// Staging (512 threads = MMA warp + TMA warp + 14 converter warps, see tile_3xtf32): A is fetched from global/L2 ONCE as
// float32 by TMA (cp.async.bulk.tensor, 128B swizzle, out-of-range rows/columns zero-filled by the hardware) into a
// raw ring in shared memory whose swizzle makes the row-per-lane read-back conflict free; each converter thread
// splits the chunks of ITS row (the hardware restricts a warp to TMEM lanes 32 * (w % 4) .. +31) into hi/lo in
// registers and stores them to TMEM.  B reaches the operand stage in the canonical K-major SWIZZLE_128B layout (row r
// of a K-block = 128 bytes; 16-byte chunk c of row r at chunk c ^ (r & 7); 8-row groups 1024 bytes apart) either
// through the same raw ring + conversion (PS = false) or, when the caller provides it pre-split (PS = true: the
// operand is constant over many products), by TMA directly.
#pragma once
#include <cuda.h>
#include <cstdint>
#include "common.cuh"

namespace admmq {
namespace tc {

constexpr int kThreadsTC = 512;
constexpr int kMmaWarp = 15;     // one elected lane issues the MMAs
constexpr int kTmaWarp = 14;     // one elected lane issues the TMA loads of the raw ring
constexpr int kTmaWarpB = 13;    // PS: one elected lane issues the TMA loads of B hi / lo into the operand stages
constexpr int kConverters = 13;  // warps 0 .. 12 convert operands
constexpr int kAtomK = 32;       // floats per 128-byte swizzle row
constexpr int kAtoms = 2;        // swizzle atoms along K per K-block
constexpr int kBlockK = kAtomK * kAtoms;  // 64: halves the per-block synchronisation cost of a 32-deep block
constexpr int kUmmaK = 8;        // k per tcgen05.mma.kind::tf32
constexpr int kMaxStages = 3;    // operand stages (B hi/lo swizzled in shared memory, A hi/lo in tensor memory)
constexpr int kTileM = 128;
constexpr int kPrefetchB = 2;     // operand stages whose B hi / lo may be requested across a tile boundary (PS)

constexpr int kMaxRawDepth = 4;  // K-blocks of raw float32 in flight (TMA): TileSmem::kRawDepth = 4 with PS, 3 without
constexpr int kStageCols = 2 * kBlockK;  // TMEM columns of one A stage: hi [0, 64), lo [64, 128)
constexpr int kTmemCols = 512;   // 2 accumulators + stages x 128: 64 + 3 x 128 (BN <= 32), 128 + 3 x 128 (BN = 64), 256 + 2 x 128 (BN = 128);
                                 // BN = 160: ONE accumulator of 160 (in 256) + 2 x 128

// PS ("pre-split B"): the B operand is given as two tf32-valued float32 matrices hi / lo made once by the caller (the
// ridge inverse is constant for all inner iterations of an ADMM call), fetched by TMA straight into the operand stage
// in the layout the MMA reads, so that the producer warps only convert A.
template <int BN, bool PS = false>
struct TileSmem {
  static_assert(BN == 16 || BN == 32 || BN == 64 || BN == 128 || BN == 160, "BN must be 16, 32, 64, 128 or 160");
  static_assert(PS || BN <= 64, "128-wide and wider tiles need the pre-split B operand (shared-memory budget)");
  // Tiles up to 128 columns keep TWO accumulators: hi.hi in one, the small cross terms lo.hi + hi.lo in the other,
  // added once by the epilogue.  That is not a nicety: the tensor core's accumulate rounds toward zero, so the error of
  // an accumulator grows with the number of MMAs added into it - measured on the 512 x 512 x 9 MTTKRP: 1.1e-6 of the
  // largest entry with the cross terms apart (K / 8 additions into the large accumulator), 3.2e-6 with all three
  // products in one (3 K / 8).  Tiles wider than 128 columns (BN = 160, used with bn = 144 / 160) leave tensor memory
  // room for ONE accumulator only next to the two operand stages; they take the 3x larger rounding error and exist
  // for the wave structure: 512 x 1141 is 4 x 9 tiles of width 128 but 4 x 8 of width 144 - ONE wave on 32 .. 35 CTAs
  // instead of two (ridge product 44 -> 32 us per iteration there).
  static constexpr bool kSingleAcc = BN > 128;
  // shared-memory / TMEM budgets: BN = 64 without PS: 2 x 32 + 3 x 48 KB; BN = 64 with PS: 3 x 32 + 4 x 32 KB;
  // BN = 128 (PS): 2 x 64 + 3 x 32 KB and 2 x 128 accumulator + 2 x 128 operand columns of tensor memory;
  // BN = 160 (PS): 2 x 80 + 2 x 32 KB and 256 (160 used) + 2 x 128 columns
  static constexpr int kStages = (BN >= 128 || (BN == 64 && !PS)) ? 2 : 3;
  static constexpr int kRawDepth = (BN == 160) ? 2 : ((BN == 128) ? 3 : (PS ? 4 : 3));
  static constexpr int kAccStride = (BN >= 128) ? 128 : ((BN == 64) ? 64 : 32);  // TMEM columns between the two accumulators
  static constexpr int kAccCols = 2 * kAccStride;   // hi.hi at +0, hi.lo + lo.hi at +stride; one accumulator of up to 256 columns for BN = 160
  static_assert(kAccCols + kStages * kStageCols <= kTmemCols, "tensor memory budget");
  static constexpr int kAAtomBytes = kTileM * 128;               // one 32-deep atom of A as raw float32
  static constexpr int kBAtomBytes = BN * 128;
  static constexpr int kABytes = kAtoms * kAAtomBytes;           // one K-block of A
  static constexpr int kBBytes = kAtoms * kBAtomBytes;
  static constexpr int kStageBytes = 2 * kBBytes;                // B_hi, B_lo (A goes to tensor memory)
  static constexpr int kRawBytes = kABytes + (PS ? 0 : kBBytes); // one K-block of raw float32
  static constexpr int kBytes = kStages * kStageBytes + kRawDepth * kRawBytes + 1024;  // + slack for 1024-byte alignment
  static_assert(kBytes <= 227 * 1024, "tile does not fit in shared memory");
};

struct Pipe {  // lives in shared memory (static), one per CTA
  unsigned long long raw_full[kMaxRawDepth];  // the TMA data of a K-block has landed
  unsigned long long raw_free[kMaxRawDepth];  // every converter warp has finished reading the slot
  unsigned long long stage_full[kMaxStages];
  unsigned long long stage_free[kMaxStages];
  unsigned long long b_full[kMaxStages];   // PS only: the TMA loads of B hi / lo into the stage have landed
  unsigned long long tile_done;
  unsigned int tmem_base;
  unsigned int pad;
};

struct PipeState {  // per-thread copy, uniform across the CTA
  unsigned int raw_uses[kMaxRawDepth];  // how often each raw slot has been filled so far
  unsigned int uses[kMaxStages];  // how often each stage has been filled / consumed so far
  unsigned int tiles;          // commits issued so far on tile_done
  unsigned int prefetched;     // the first K-blocks of the coming tile were already requested at the end of the previous one
  unsigned long long nz2;      // (-0.0f, -0.0f) as a run-time value (see split2)
#ifdef ADMMQ_TC_PROFILE
  long long cyc[6];            // producer: cp.async wait, stage_free wait, convert; mma: full wait, issue; all: tile_done wait
#endif
};
#ifdef ADMMQ_TC_PROFILE
#define TC_T0() const long long _t0 = clock64()
#define TC_ACC(i) st.cyc[i] += clock64() - _t0
#else
#define TC_T0()
#define TC_ACC(i)
#endif

__device__ __forceinline__ unsigned int smem_u32(const void* p) { return (unsigned int)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned int parity) {
  const unsigned int addr = smem_u32(bar);
  unsigned int ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (ok == 0u);
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cp_async16(unsigned int dst_smem, const void* src, bool valid) {
  const unsigned int sz = valid ? 16u : 0u;  // 0 source bytes => the 16 destination bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// arrive on `bar` once every cp.async issued so far by this thread has landed (the barrier's count includes it)
__device__ __forceinline__ void cp_async_arrive(unsigned long long* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// TMA: one arrival + `bytes` expected on `bar`, then a 2-D tile load (coordinates: c0 = innermost = column, c1 = row)
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned int bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(unsigned int dst_smem, const CUtensorMap* tmap, int c0, int c1,
                                            unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst_smem), "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}
// true in exactly one (always the same) lane of a fully active warp; the surrounding code stays warp-uniform,
// which lets ptxas keep MMA descriptors in uniform registers instead of broadcasting them lane by lane
__device__ __forceinline__ bool elect_one() {
  unsigned int pred = 0;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0u;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(unsigned int* slot, unsigned int cols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(unsigned int base, unsigned int cols) {  // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

__device__ __forceinline__ void umma_tf32(unsigned int d_tmem, unsigned long long a_desc, unsigned long long b_desc,
                                          unsigned int idesc, unsigned int accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TS form: A from tensor memory (lane = row, column = k), B from shared memory
__device__ __forceinline__ void umma_tf32_ts(unsigned int d_tmem, unsigned int a_tmem, unsigned long long b_desc,
                                             unsigned int idesc, unsigned int accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 8 consecutive columns of the calling thread's TMEM lane
__device__ __forceinline__ void tmem_store8(unsigned int taddr, const float v[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
               "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
               "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
__device__ __forceinline__ void tmem_store_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(unsigned long long* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// instruction descriptor: D = F32, A = B = TF32, both K-major, M = 128, N = BN
template <int BN>
__device__ __forceinline__ constexpr unsigned int make_idesc() {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned int)(BN >> 3) << 17) | ((unsigned int)(kTileM >> 4) << 24);
}
// shared-memory matrix descriptor, K-major SWIZZLE_128B: LBO = 1 (unused), SBO = 1024 B between 8-row groups,
// version 1 (sm_100), layout type 2
__device__ __forceinline__ unsigned long long make_desc(unsigned int smem_addr) {
  return (unsigned long long)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | ((unsigned long long)(1024 >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}

// hi/lo split of two packed float32 values in four FMA-pipe instructions (the conversion is issue bound: the integer
// form costs five half-rate ALU operations per element, cvt.rna.tf32 runs on the quarter-rate conversion pipe):
//   Veltkamp/Dekker: t = x * (2^13 + 1); hi = t - (t - x) is x rounded to nearest to 11 significant bits, i.e.
//   exactly a tf32 number; lo = x - hi is exact in float32 and |lo| <= 2^-11 |x|.
// lo keeps up to 13 significant bits; the tensor core reads the upper 19 bits of each 32-bit operand, so lo enters the
// product truncated to tf32 (error <= 2^-21 |x|, same order as the dropped lo.lo term).
// ptxas contracts a packed multiply into each packed add/sub that consumes it (it even duplicates the multiply), which
// turns hi = t - (t - x) into fma(x, c, -(fma(x, c, -x))) = x.  The product is therefore formed as fma(x, c, nz) with
// nz = (-0.0f, -0.0f) taken from a kernel parameter, which cannot be folded away.
__device__ __forceinline__ void split2(unsigned long long x, unsigned long long nz, unsigned long long& hi,
                                       unsigned long long& lo) {
  unsigned long long t, u;
  const unsigned long long c = 0x4600040046000400ull;  // (8193.0f, 8193.0f)
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(t) : "l"(x), "l"(c), "l"(nz));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(u) : "l"(t), "l"(x));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(hi) : "l"(t), "l"(u));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(lo) : "l"(x), "l"(hi));
}
__device__ __forceinline__ void split4(const float4 v, unsigned long long nz, float4& hi, float4& lo) {
  const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(&v);
  ulonglong2 h, l;
  split2(x.x, nz, h.x, l.x);
  split2(x.y, nz, h.y, l.y);
  hi = *reinterpret_cast<const float4*>(&h);
  lo = *reinterpret_cast<const float4*>(&l);
}

// byte offset of 16-byte chunk c (0..7) of row r inside a K-major SWIZZLE_128B tile
__device__ __forceinline__ unsigned int sw128(int r, int c) { return (unsigned int)(r * 128 + ((c ^ (r & 7)) << 4)); }

__device__ __forceinline__ void pipe_setup(Pipe& pipe, PipeState& st, float neg_zero) {
  const unsigned int tmem_cols = kTmemCols;
  asm("mov.b64 %0, {%1, %1};" : "=l"(st.nz2) : "f"(neg_zero));
  if (threadIdx.x == 0) {
    for (int d = 0; d < kMaxRawDepth; ++d) {
      mbar_init(&pipe.raw_full[d], 1);
      mbar_init(&pipe.raw_free[d], kConverters);
    }
    for (int s = 0; s < kMaxStages; ++s) {
      mbar_init(&pipe.stage_full[s], kConverters);
      mbar_init(&pipe.stage_free[s], 1);
      mbar_init(&pipe.b_full[s], 1);
    }
    mbar_init(&pipe.tile_done, 1);
    fence_barrier_init();
  }
  if (threadIdx.x < 32) tmem_alloc(&pipe.tmem_base, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  for (int s = 0; s < kMaxStages; ++s) st.uses[s] = 0u;
  for (int d = 0; d < kMaxRawDepth; ++d) st.raw_uses[d] = 0u;
  st.tiles = 0u;
  st.prefetched = 0u;
#ifdef ADMMQ_TC_PROFILE
  for (int i = 0; i < 6; ++i) st.cyc[i] = 0;
#endif
}
__device__ __forceinline__ void pipe_teardown(Pipe& pipe) {
  const unsigned int tmem_cols = kTmemCols;
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) tmem_free(pipe.tmem_base, tmem_cols);
}

// 4 consecutive columns of the calling thread's TMEM lane
__device__ __forceinline__ void tmem_store4(unsigned int taddr, const float4 v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(__float_as_uint(v.x)), "r"(__float_as_uint(v.y)), "r"(__float_as_uint(v.z)),
               "r"(__float_as_uint(v.w))
               : "memory");
}

// One 128 x bn tile (bn <= BN, a multiple of 16): the 128 rows of A starting at a_row0 against the bn rows of B starting
// at b_row0, over K columns.  tmA / tmB are TMA descriptors of the row-major float32 matrices with boxes {32, 128} and
// {32, bn} (make_operand_tmap); rows and columns outside the matrices read as zero.  With PS the B operand comes
// pre-split: tmB = hi part, tmBlo = lo part (both tf32-valued float32, same shape and box).
// On return the accumulators are complete in TMEM and visible to every thread (load_acc / acc_to_smem).
//
// Roles: warp 15 issues MMAs and the TMA loads of the raw ring.  Warps 0..14 convert: warp w writes TMEM lanes
// 32 * (w % 4) .. +31; the 16 chunks (4 k-columns each) of a K-block row are split 4/4/4/4 over the four warps of
// quarters 0-2 and 6/5/5 over warps 3, 7, 11 of quarter 3; without PS the B chunks go to the twelve warps of quarters
// 0-2, with PS warp 0 issues the TMA loads of B hi / lo into the stage as soon as the tensor pipe has released it.
// next_a_row0 / next_b_row0 >= 0 name the tile this CTA computes next: its first K-blocks are requested as soon as this
// tile no longer needs the buffers, so that the TMA latency overlaps the caller's epilogue.
//
// Roles (16 warps):
//   warp 15  MMA: waits for a stage (A hi/lo in tensor memory from the converters, B hi/lo in shared memory), issues
//            the 24 MMAs of the K-block, commits them to stage_free
//   warp 14  TMA: keeps the raw ring (float32 K-blocks of A, and of B without PS) filled; warp 13 (PS) the B hi/lo halves
//            of the operand stages; a slot / stage is refilled as soon as its previous content has been consumed
//            (measured: issuing the TMA loads from the MMA warp or from a converting warp stalls that warp for ~75
//            cycles per load and makes it the straggler of every K-block)
//   13 converters (warps 0 .. 12): warp w writes TMEM lanes 32 * (w % 4) .. +31; the 16 chunks (4 k-columns each) of a K-block row are
//            split 4/4/4/4 over the four warps of quarter 0 and 6/5/5 over the three warps of quarters 1-3; without
//            PS the B chunks are split over all converters
// Barrier phases: K-block j of this tile is fill number st.uses[j % kStages] + j / kStages + 1 of its stage (st.uses =
// fills before this tile, the same in every thread), raw slots likewise with st.raw_uses; nothing is mutated inside
// the loops, every thread adds the tile's counts at the end.
template <int BN, bool PS>
__device__ void tile_3xtf32(const CUtensorMap* tmA, int a_row0, const CUtensorMap* tmB, const CUtensorMap* tmBlo,
                            int b_row0, int bn, int K, unsigned char* smem_tiles, Pipe& pipe, PipeState& st,
                            int next_a_row0 = -1, int next_b_row0 = -1) {
  using TS = TileSmem<BN, PS>;
  constexpr int kChunksB = BN * 8 * kAtoms;  // 16-byte chunks of B per K-block
  constexpr int kRowChunks = 8 * kAtoms;     // 16-byte chunks per row per K-block
  constexpr int kNS = TS::kStages;
  constexpr int kRawDepth = TS::kRawDepth;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const unsigned int tiles_base = (smem_u32(smem_tiles) + 1023u) & ~1023u;
  unsigned char* tiles_ptr = smem_tiles + (tiles_base - smem_u32(smem_tiles));
  const unsigned int raw_base = tiles_base + (unsigned int)(kNS * TS::kStageBytes);
  unsigned char* raw_ptr = tiles_ptr + (size_t)kNS * TS::kStageBytes;
  const int nkb = (K + kBlockK - 1) / kBlockK;
  const unsigned int tmem = pipe.tmem_base;  // keep in a register: the asm memory clobbers would re-read it
  const unsigned int b_atom_tx = (unsigned int)(bn * 128);  // bytes one TMA box of B delivers
  // parity of the phase that completes with fill number n (n = 1, 2, ...) of a barrier: (n - 1) & 1
  auto fills_before = [&](int j) { return st.uses[j % kNS] + (unsigned int)(j / kNS); };        // stage fills before K-block j
  auto raw_before = [&](int j) { return st.raw_uses[j % kRawDepth] + (unsigned int)(j / kRawDepth); };

  if (warp == kMmaWarp) {
    // ---------------- MMA warp: the whole warp runs the loop, one elected lane issues
    const unsigned int idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned int)(bn >> 3) << 17) | ((unsigned int)(kTileM >> 4) << 24);
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % kNS;
      const unsigned int par = fills_before(kb) & 1u;
      { TC_T0(); mbar_wait(&pipe.stage_full[s], par); TC_ACC(3); }
      if constexpr (PS) { TC_T0(); mbar_wait(&pipe.b_full[s], par); TC_ACC(0); }
      tc_fence_after();
      TC_T0();
      const unsigned int a_col = tmem + (unsigned int)(TS::kAccCols + s * kStageCols);
      const unsigned int sb = tiles_base + (unsigned int)(s * TS::kStageBytes);
      const unsigned int first = kb != 0 ? 1u : 0u;
      unsigned long long* free_bar = &pipe.stage_free[s];
      unsigned long long* done_bar = &pipe.tile_done;
      const bool last = kb + 1 == nkb;
      if (elect_one()) {
#pragma unroll
        for (int a = 0; a < kAtoms; ++a) {
          const unsigned long long b_hi = make_desc(sb + (unsigned int)(a * TS::kBAtomBytes));
          const unsigned long long b_lo = make_desc(sb + (unsigned int)(TS::kBBytes + a * TS::kBAtomBytes));
#pragma unroll
          for (int ks = 0; ks < kAtomK / kUmmaK; ++ks) {
            const unsigned long long adv = (unsigned long long)((ks * kUmmaK * 4) >> 4);  // +32 bytes per k-step
            const unsigned int a_hi = a_col + (unsigned int)(a * kAtomK + ks * kUmmaK), a_lo = a_hi + (unsigned int)kBlockK;
            // the small cross terms get their own accumulator (added to hi.hi by the epilogue): this keeps them from
            // being absorbed into the large hi.hi sums and halves the dependent chain on each accumulator
            const unsigned int acc = (a | ks) != 0 ? 1u : first;
            if constexpr (TS::kSingleAcc) {   // one accumulator: small terms first within the k-step
              umma_tf32_ts(tmem, a_lo, b_hi + adv, idesc, acc);
              umma_tf32_ts(tmem, a_hi, b_lo + adv, idesc, 1u);
              umma_tf32_ts(tmem, a_hi, b_hi + adv, idesc, 1u);
            } else {
              umma_tf32_ts(tmem + (unsigned int)TS::kAccStride, a_lo, b_hi + adv, idesc, acc);
              umma_tf32_ts(tmem + (unsigned int)TS::kAccStride, a_hi, b_lo + adv, idesc, 1u);
              umma_tf32_ts(tmem, a_hi, b_hi + adv, idesc, acc);
            }
          }
        }
        umma_commit(free_bar);
        if (last) umma_commit(done_bar);
      }
      __syncwarp();
      TC_ACC(4);
    }
  } else if (warp == kTmaWarp) {
    // ---------------- TMA warp (one elected lane works)
    if (elect_one()) {
      auto fetch_raw = [&](int j, int arow, int brow) {  // K-block j of the tile with rows arow / brow into slot j % kRawDepth
        const int d = j % kRawDepth;
        const unsigned int slot = raw_base + (unsigned int)(d * TS::kRawBytes);
        mbar_expect_tx(&pipe.raw_full[d], (unsigned int)TS::kABytes + (PS ? 0u : (unsigned int)kAtoms * b_atom_tx));
#pragma unroll
        for (int a = 0; a < kAtoms; ++a) {
          tma_load_2d(slot + (unsigned int)(a * TS::kAAtomBytes), tmA, j * kBlockK + a * kAtomK, arow, &pipe.raw_full[d]);
          if constexpr (!PS)
            tma_load_2d(slot + (unsigned int)(TS::kABytes + a * TS::kBAtomBytes), tmB, j * kBlockK + a * kAtomK, brow,
                        &pipe.raw_full[d]);
        }
      };
      const int npre_raw = min(kRawDepth, nkb);
      unsigned int raw_fills[kRawDepth];  // fills of each raw slot so far (previous tiles + this one)
#pragma unroll
      for (int d = 0; d < kRawDepth; ++d) raw_fills[d] = st.raw_uses[d];
      // kb runs past nkb by kRawDepth: those steps request the next tile's first K-blocks (slot order restarts with
      // every tile, so the previous user of a slot is tracked per slot, not per K-block)
      for (int kb = 0; kb < nkb + kRawDepth; ++kb) {
        const bool cur = kb < nkb;
        const int j = cur ? kb : kb - nkb;
        const int d = j % kRawDepth;
        if (cur && st.prefetched != 0u && kb < npre_raw) {
          raw_fills[d] += 1u;  // requested at the end of the previous tile
        } else if (cur || (next_a_row0 >= 0 && j < npre_raw)) {
          // raw slot d is free once every converter warp has read its previous content
          if (raw_fills[d] > 0u) mbar_wait(&pipe.raw_free[d], (raw_fills[d] - 1u) & 1u);
          if (cur) {
            fetch_raw(j, a_row0, b_row0);
            raw_fills[d] += 1u;
          } else {
            fetch_raw(j, next_a_row0, next_b_row0);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == kTmaWarpB) {
    // ---------------- second TMA warp (PS only): B hi / lo straight into the operand stages.  A separate warp, so
    // that waiting for a stage to be released by the tensor pipe never delays the raw ring (and vice versa)
    if constexpr (PS) {
      if (elect_one()) {
        auto fetch_b = [&](int j, int brow) {
          const int s = j % kNS;
          const unsigned int sb = tiles_base + (unsigned int)(s * TS::kStageBytes);
          mbar_expect_tx(&pipe.b_full[s], 2u * (unsigned int)kAtoms * b_atom_tx);
#pragma unroll
          for (int a = 0; a < kAtoms; ++a) {
            tma_load_2d(sb + (unsigned int)(a * TS::kBAtomBytes), tmB, j * kBlockK + a * kAtomK, brow, &pipe.b_full[s]);
            tma_load_2d(sb + (unsigned int)(TS::kBBytes + a * TS::kBAtomBytes), tmBlo, j * kBlockK + a * kAtomK, brow, &pipe.b_full[s]);
          }
        };
        const int npre_b = min(min(kPrefetchB, kNS - 1), nkb);
        for (int kb = 0; kb < nkb; ++kb) {
          // stage kb % kNS: free once the MMAs of its previous fill have completed
          if (!(st.prefetched != 0u && kb < npre_b)) {
            const unsigned int fb = fills_before(kb);
            if (fb > 0u) mbar_wait(&pipe.stage_free[kb % kNS], (fb - 1u) & 1u);
            fetch_b(kb, b_row0);
          }
        }
        // every MMA of this tile has completed => all stages are free: B hi / lo of the next tile's first K-blocks go
        // into stages 0 .. kPrefetchB-1 (the caller's epilogue parks the accumulator in the LAST stage)
        if (next_a_row0 >= 0) {
          mbar_wait(&pipe.tile_done, st.tiles & 1u);
          for (int j = 0; j < npre_b; ++j) fetch_b(j, next_b_row0);
        }
      }
    }
    __syncwarp();
  } else {
    // ---------------- converters
    const int q = warp & 3, kgi = warp >> 2;
    const int ar = q * 32 + lane;  // tile row = TMEM lane of this thread
    // chunks (4 k-columns each) of the row this thread converts: 4/4/4/4 in quarter 0, 6/5/5 in quarters 1-3
    const int c_begin = (q >= 1) ? (kgi == 0 ? 0 : 1 + 5 * kgi) : kgi * (kRowChunks / 4);
    const int c_count = (q >= 1) ? (kgi == 0 ? 6 : 5) : kRowChunks / 4;
    const unsigned int lane_addr = tmem + ((unsigned int)(q * 32) << 16);
    // without PS: B chunk ids handled by this thread: bi0, bi0 + 13 * 32, ...
    const int cw = (q >= 1) ? 4 + (q - 1) * 3 + kgi : kgi;  // converter index 0 .. 12
    const int bi0 = cw * 32 + lane;
    for (int kb = 0; kb < nkb; ++kb) {
      const int d = kb % kRawDepth;
      const int s = kb % kNS;
      const unsigned int fb = fills_before(kb);
      { TC_T0(); if (fb > 0u) { mbar_wait(&pipe.stage_free[s], (fb - 1u) & 1u); tc_fence_after(); } TC_ACC(1); }
      { TC_T0(); mbar_wait(&pipe.raw_full[d], raw_before(kb) & 1u); TC_ACC(0); }  // K-block kb has landed
      TC_T0();
      const unsigned char* raw = raw_ptr + (size_t)d * TS::kRawBytes;
      const unsigned int col0 = lane_addr + (unsigned int)(TS::kAccCols + s * kStageCols);
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        if (i < c_count) {
          const int c = c_begin + i;  // chunk c of the row: atom c / 8, chunk c % 8 within the atom's 128-byte row
          const float4 v = *reinterpret_cast<const float4*>(raw + (c >> 3) * TS::kAAtomBytes + sw128(ar, c & 7));
          float4 hi, lo;
          split4(v, st.nz2, hi, lo);
          tmem_store4(col0 + (unsigned int)(c * 4), hi);
          tmem_store4(col0 + (unsigned int)(kBlockK + c * 4), lo);
        }
      }
      if constexpr (!PS) {
        unsigned char* stage = tiles_ptr + (size_t)s * TS::kStageBytes;
        for (int bi = bi0; bi < kChunksB; bi += kConverters * 32) {
          const int atom = bi / (BN * 8), lid = bi % (BN * 8);
          const unsigned int off = (unsigned int)(atom * TS::kBAtomBytes) + sw128(lid >> 3, lid & 7);
          const float4 v = *reinterpret_cast<const float4*>(raw + TS::kABytes + off);
          float4 hi, lo;
          split4(v, st.nz2, hi, lo);
          *reinterpret_cast<float4*>(stage + off) = hi;
          *reinterpret_cast<float4*>(stage + TS::kBBytes + off) = lo;
        }
      }
      tmem_store_wait();
      tc_fence_before();
      if constexpr (!PS) fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core's async proxy
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&pipe.raw_free[d]);
        mbar_arrive(&pipe.stage_full[s]);
      }
      TC_ACC(2);
    }
  }
  { TC_T0(); mbar_wait(&pipe.tile_done, st.tiles & 1u); TC_ACC(5); }
  // the tile's fills, identically in every thread
  for (int kb = 0; kb < nkb; ++kb) {
    st.uses[kb % kNS] += 1u;
    st.raw_uses[kb % kRawDepth] += 1u;
  }
  st.tiles += 1u;
  tc_fence_after();
  st.prefetched = next_a_row0 >= 0 ? 1u : 0u;
}

// Accumulator read-back for the calling warp: TMEM lanes 32 * (warp % 4) .. +31 (= tile rows), BN / 4 columns
// starting at (warp / 4) * BN / 4.  v[i] = D[row = 32 * (warp % 4) + lane][col0 + i] = (lo.hi + hi.lo) + hi.hi.
// (kAccStride does not depend on PS.)
// tcgen05.ld of N consecutive columns of the calling thread's TMEM lane; the registers are valid after tmem_load_wait()
template <int N>
__device__ __forceinline__ void tmem_load(unsigned int taddr, unsigned int r[N]) {
  if constexpr (N == 8) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
  } else if constexpr (N == 4) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
  } else {
    static_assert(N == 16, "unsupported width");
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
  }
}
__device__ __forceinline__ void tmem_load_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Accumulator read-back for the calling warp: TMEM lanes 32 * (warp % 4) .. +31 (= tile rows), BN / 4 columns
// starting at (warp / 4) * BN / 4.  v[i] = D[row = 32 * (warp % 4) + lane][col0 + i] = (lo.hi + hi.lo) + hi.hi.
// Both accumulators of a column block are requested before the single wait (one tensor-memory round trip per block
// instead of two; with BN / 4 <= 16 the whole read-back is one round trip).
template <int BN>
__device__ __forceinline__ void load_acc(const Pipe& pipe, float v[BN / 4], int& row, int& col0) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = warp & 3, cgp = warp >> 2;
  row = q * 32 + lane;
  col0 = cgp * (BN / 4);
  const unsigned int taddr = pipe.tmem_base + ((unsigned int)(q * 32) << 16) + (unsigned int)col0;
  constexpr int kCols = BN / 4;
  constexpr int kW = (kCols % 16 == 0) ? 16 : ((kCols % 8 == 0) ? 8 : 4);  // columns per tcgen05.ld (register pressure)
#pragma unroll
  for (int c0 = 0; c0 < kCols; c0 += kW) {
    unsigned int hh[kW];
    tmem_load<kW>(taddr + (unsigned int)c0, hh);
    if constexpr (TileSmem<BN, true>::kSingleAcc) {
      tmem_load_wait();
#pragma unroll
      for (int i = 0; i < kW; ++i) v[c0 + i] = __uint_as_float(hh[i]);
    } else {
      unsigned int cr[kW];
      tmem_load<kW>(taddr + (unsigned int)(TileSmem<BN, true>::kAccStride + c0), cr);
      tmem_load_wait();
#pragma unroll
      for (int i = 0; i < kW; ++i) v[c0 + i] = __uint_as_float(cr[i]) + __uint_as_float(hh[i]);
    }
  }
}

// all accumulator reads of this tile are done: the next tile may overwrite TMEM
__device__ __forceinline__ void release_acc() {
  tc_fence_before();
  __syncthreads();
}

// Epilogue staging.  A thread holds one ROW of the accumulator (TMEM lane = row), so writing results straight to
// row-major global memory touches 32 different rows per warp instruction (4 useful bytes per 32-byte sector, measured
// ~6-8 k cycles per 128 x 64 tile).  acc_to_smem() parks the tile in shared memory instead - in the LAST operand
// stage, which is idle once tile_done has completed and is not a target of the cross-tile prefetch - releases the
// accumulator and returns the tile, so that the caller can walk it in row-contiguous float4 groups (thread t -> group
// t, t + 512, ...; group g = row g / (BN / 4), columns 4 (g % (BN / 4)) .. +3, at EpiTile::offset(row, g % (BN / 4))).
// The caller must __syncthreads() after its last read and before the next tile_3xtf32().
template <int BN>
struct EpiTile {
  static constexpr int kGroupsPerRow = BN / 4;
  static constexpr int kGroups = kTileM * kGroupsPerRow;
  static_assert(kTileM * BN * 4 <= TileSmem<BN, true>::kStageBytes, "staging tile must fit in one operand stage");
  // float offset of float4 group g of `row`: rows of BN floats, groups XOR-swizzled so that both the per-row writes
  // (32 rows per warp) and the row-contiguous reads are bank-conflict free without padding
  __device__ static __forceinline__ int offset(int row, int g) {
    const int sw = (BN == 16) ? ((row >> 1) & 3) : (row & 7);
    return row * BN + ((g ^ sw) << 2);
  }
};
template <int BN, bool PS>
__device__ __forceinline__ const float* acc_to_smem(const Pipe& pipe, unsigned char* smem_tiles) {
  using TS = TileSmem<BN, PS>;
  const unsigned int tiles_base = (smem_u32(smem_tiles) + 1023u) & ~1023u;
  float* tile = reinterpret_cast<float*>(smem_tiles + (tiles_base - smem_u32(smem_tiles)) + (size_t)(TS::kStages - 1) * TS::kStageBytes);
  float v[BN / 4];
  int row, col0;
  load_acc<BN>(pipe, v, row, col0);
#pragma unroll
  for (int c = 0; c < BN / 4; c += 4)
    *reinterpret_cast<float4*>(tile + EpiTile<BN>::offset(row, (col0 + c) >> 2)) = make_float4(v[c], v[c + 1], v[c + 2], v[c + 3]);
  release_acc();
  return tile;
}

// Host: TMA descriptor of a row-major matrix of `dtype` elements (rows x cols, leading dimension ld_bytes, a multiple
// of 16, base 16-byte aligned) with box {box_cols columns, box_rows rows} and 128-byte swizzle; rows and columns outside
// the matrix read as zero.  Returns 0 or ADMMQ_E_CUDA.
int make_tmap_2d(CUtensorMap* out, CUtensorMapDataType dtype, const void* base, int rows, int cols, size_t ld_bytes,
                 int box_cols, int box_rows);
// ... of a float32 matrix (ld floats, ld % 4 == 0) with box {32 columns, box_rows rows}
int make_operand_tmap(CUtensorMap* out, const float* base, int rows, int cols, int ld, int box_rows);

// Host: tile widths come from a wave model.  A tile costs a fixed part plus w columns of tensor-core work, and the width
// minimises waves * (fixed + w); callers try the candidates widest first, so ties go to the wider tile.
inline long long wave_cost(long long tilesM, int N, int w, int sms, int fixed) {
  const long long tiles = tilesM * ((N + w - 1) / w);
  return ((tiles + sms - 1) / sms) * (fixed + w);
}

}  // namespace tc
}  // namespace admmq
