/*
 * admmq.h - C ABI of libadmmq.so: the B200 (sm_100a) kernels behind the
 * quantization-aware CP factorization hot path of KamikaziZen/admm-quantization.
 *
 * The reference has no FFI: its boundary is the Python API of source/admm.py,
 * source/quantization.py and the loop in scripts/factorize.py.  Every entry point
 * below names the reference call site it replaces (file:line relative to the
 * reference repository).  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *   - All data pointers are DEVICE pointers on the current CUDA device, float32
 *     row-major contiguous unless stated.  The caller owns every buffer, including
 *     workspaces (size them with the *_workspace_bytes functions); the library
 *     never allocates or frees device memory and keeps no pointer after return.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     the call returns without synchronising unless stated.
 *   - Return value: 0 on success, a negative ADMMQ_E_* code on failure; the message
 *     is available from admmq_last_error() (thread-local).  No C++ exception crosses.
 *   - There is no CPU fallback: without a CUDA device every compute call fails
 *     with ADMMQ_E_CUDA.
 */
#ifndef ADMMQ_H_
#define ADMMQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ADMMQ_VERSION 200 /* 0.2.0 */

#if defined(__GNUC__)
#define ADMMQ_API __attribute__((visibility("default")))
#else
#define ADMMQ_API
#endif

/* error codes */
#define ADMMQ_OK 0
#define ADMMQ_E_BADARG (-1)      /* ValueError / NotImplementedError on the Python side */
#define ADMMQ_E_WORKSPACE (-2)   /* workspace too small or misaligned */
#define ADMMQ_E_CUDA (-3)        /* CUDA runtime / launch failure (no device, OOM, ...) */
#define ADMMQ_E_NOT_PD (-4)      /* G + rho I not positive definite: torch.linalg.LinAlgError */
#define ADMMQ_E_UNSUPPORTED (-5) /* shape outside what the kernels handle */

/* quantization schemes, source/quantization.py:91-115 (tensor_* branches) */
#define ADMMQ_Q_MSEMINMAX_SYMMETRIC 0 /* 'tensor_mseminmax_symmetric' :107-108, :118-144 */
#define ADMMQ_Q_MINMAX 1              /* 'tensor_minmax'              :110-111, :48-66  */
#define ADMMQ_Q_SYMMETRIC 2           /* 'tensor_symmetric'           :91-95           */
#define ADMMQ_Q_AFFINE 3              /* 'tensor_affine'              :97-106          */
/* 'tensor_mseminmax_e2m1' (no counterpart in the reference; bits must be 4): the clip search of :118-144 onto the FP4
 * E2M1 grid s * {+-0, 0.5, 1, 1.5, 2, 3, 4, 6}, s = clip / 6; codes are the 4-bit E2M1 encodings 0 .. 15 (bit 3 sign,
 * bits 2-1 exponent, bit 0 mantissa), ready to pack into FP4 tensor-core operands.  Definition: DESIGN.md 2b. */
#define ADMMQ_Q_MSEMINMAX_E2M1 4
/* (id 5 is unassigned.)  The same clip search onto the FP8 and FP6 grids that tcgen05.mma kind::f8f6f4 reads, no
 * counterpart in the reference either: s * (every finite value of the format), s = clip / max, each with a fixed width.
 * Codes are the format's encodings: for FP8 the byte itself (a float8_e4m3fn / float8_e5m2 tensor viewed as int8), for
 * FP6 0 .. 63 (bit 5 sign, then the exponent bits, then the mantissa bits).  Definition: DESIGN.md 2c. */
#define ADMMQ_Q_MSEMINMAX_E4M3 6 /* 'tensor_mseminmax_e4m3'  bits 8, max 448   */
#define ADMMQ_Q_MSEMINMAX_E5M2 7 /* 'tensor_mseminmax_e5m2'  bits 8, max 57344 */
#define ADMMQ_Q_MSEMINMAX_E3M2 8 /* 'tensor_mseminmax_e3m2'  bits 6, max 28    */
#define ADMMQ_Q_MSEMINMAX_E2M3 9 /* 'tensor_mseminmax_e2m3'  bits 6, max 7.5   */

/* status bits written by the ADMM loop into admmq_loop_report.status */
#define ADMMQ_ST_CONVERGED 1 /* r < eps and s < eps fired (source/admm.py:64-65) */
#define ADMMQ_ST_NONFINITE 2 /* projection input had abs-max 0, inf or NaN: outputs are NaN like the reference */

ADMMQ_API int admmq_version(void);
ADMMQ_API const char* admmq_last_error(void);
/* sm count / compute capability of the current device; fails without one. */
ADMMQ_API int admmq_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Number of kernels this library has launched in the calling process so far (all threads).
 * bench.py differences it around the timed region for its "gpu_launches" claim. */
ADMMQ_API uint64_t admmq_launch_count(void);

/* ------------------------------------------------------------------ projection
 * Replaces quantize_tensor(tensor, bits, qscheme, **kw)  source/quantization.py:69-115
 * and quantize_tensor_mse(x, bits, num_attempts)          source/quantization.py:118-144.
 *   x, xq       n floats (xq may alias x)
 *   codes       n int8 integer codes or NULL (mse/symmetric: clamp(rint(x/scale),-q,q-1);
 *               affine: code incl. zero point; minmax: level index - 2^(bits-1); e2m1: the E2M1 encoding 0 .. 15;
 *               e4m3 / e5m2: the FP8 byte; e3m2 / e2m3: the FP6 encoding 0 .. 63)
 *   info        device float[4] or NULL: {scale, zero_point or min, chosen candidate index, abs-max}
 *   tmin,tmax   only for ADMMQ_Q_AFFINE: device float scalars or NULL (= tensor min/max) (:98-101)
 */
ADMMQ_API size_t admmq_project_workspace_bytes(int64_t n, int num_attempts);
ADMMQ_API int admmq_project(const float* x, int64_t n, int bits, int qscheme, int num_attempts,
                  const float* tmin, const float* tmax, float* xq, int8_t* codes, float* info,
                  void* workspace, size_t workspace_bytes, void* stream);
/* The per-candidate sums behind the argmin of source/quantization.py:136-141, sums[c] = sum((x - Q_c(x))**2) as
 * float64, for the parity tests: method 0 = direct evaluation of every (element, candidate) pair with the
 * reference's float32 operations, method 1 = the threshold form (csrc/numerics.cuh); the product lets every CTA take
 * whichever of the two is cheaper for its chunk (csrc/search.cuh, cta_candidate_sums).  max_ctas > 0
 * limits the grid (the result must not depend on it).  Workspace: admmq_project_workspace_bytes(n, num_attempts). */
ADMMQ_API int admmq_clip_search_sums(const float* x, int64_t n, int bits, int num_attempts, int method, int max_ctas,
                  double* sums, void* workspace, size_t workspace_bytes, void* stream);
/* The same sums for any clip-search scheme: qscheme ADMMQ_Q_MSEMINMAX_SYMMETRIC (= admmq_clip_search_sums),
 * ADMMQ_Q_MSEMINMAX_E2M1 (bits 4; 14 thresholds per candidate in the threshold form) or ADMMQ_Q_MSEMINMAX_E4M3 / E5M2
 * / E3M2 / E2M3 (bits 8 / 8 / 6 / 6; 252 / 246 / 62 / 62 thresholds). */
ADMMQ_API int admmq_clip_search_sums_scheme(const float* x, int64_t n, int bits, int qscheme, int num_attempts, int method,
                  int max_ctas, double* sums, void* workspace, size_t workspace_bytes, void* stream);
/* E2M1 codes (0 .. 15) of n floats t by the hardware conversion cvt.rn.satfinite.e2m1x2.f32: round to nearest, ties
 * to the even mantissa, saturating at +-6.  The projection's E2M1 codes are those of t = fl(x / scale). */
ADMMQ_API int admmq_e2m1_encode(const float* t, int64_t n, int8_t* codes, void* stream);
/* FP8 / FP6 codes of n floats t by the hardware conversion cvt.rn.satfinite.<fmt>x2.f32 for qscheme
 * ADMMQ_Q_MSEMINMAX_E4M3 / E5M2 / E3M2 / E2M3: round to nearest, ties to the even mantissa, saturating at +-max.  The
 * projection's codes are those of t = fl(x / scale). */
ADMMQ_API int admmq_fp_encode(const float* t, int64_t n, int qscheme, int8_t* codes, void* stream);

/* ------------------------------------------------------------------ per-sweep contractions
 * Gram-Hadamard  G = (U1^T U1) * (U2^T U2)   scripts/factorize.py:215,226,236 (3-D), :276,286 (2-D, U2 = NULL)
 *   U1 (n1 x R), U2 (n2 x R) or NULL, G (R x R).  Each Gram is accumulated in float64 and
 *   rounded to float32 before the float32 Hadamard product. */
ADMMQ_API int admmq_gram_hadamard(const float* U1, int n1, const float* U2, int n2, int R, float* G, void* stream);

/* Mode-n unfolding copy of a 3-way tensor (source/utils.py:60-74): out = reshape(moveaxis(W, mode, 0)). */
ADMMQ_API int admmq_unfold3(const float* W, int I, int J, int K, int mode, float* out, void* stream);

/* MTTKRP  F = Wn . KhatriRao(X, Y)   scripts/factorize.py:217,227,237 (einsum) and :277,287 (W@B, W.T@A)
 *   Wn  (M x P) row-major unfolding, P = nx*ny;  X (nx x R), Y (ny x R) or NULL (ny = 1, matrix case);
 *   KR row p = x*ny + y is X[x,:] * Y[y,:];  F (M x R).
 *   precision 0: float64 accumulation on CUDA cores (parity mode)
 *   precision 1: 3xTF32 tcgen05 tensor-core path; matrices only (ny = 1, nx % 4 == 0) - 3-way tensors use
 *                admmq_permute_myx + admmq_mttkrp_tc below, which need the permuted operand  */
ADMMQ_API size_t admmq_mttkrp_workspace_bytes(int M, int nx, int ny, int R, int precision);
ADMMQ_API int admmq_mttkrp(const float* Wn, int M, const float* X, int nx, const float* Y, int ny, int R,
                 float* F, int precision, void* workspace, size_t workspace_bytes, void* stream);

/* Tensor-core MTTKRP (3xTF32 on tcgen05): the contraction over the large index x runs as a GEMM against X alone,
 * T[(m,y), r] = sum_x V[(m,y), x] X[x, r], the small index y is folded afterwards, F[m, r] = sum_y Y[y, r] T[(m,y), r]
 * (float64 accumulation) - no Khatri-Rao operand is ever formed.
 *   admmq_permute_myx   V[(m, y), x] = Wn[m, x*ny + y]; V is (M*ny) x ldv with ldv = nx rounded up to 4 (pad columns
 *                       zeroed).  W is constant, so this runs once per layer and mode.
 *   admmq_mttkrp_tc     V as above, X (nx x R), Y (ny x R) or NULL (matrix case: V = Wn, T = F). */
ADMMQ_API int admmq_permute_myx(const float* Wn, int M, int nx, int ny, float* V, void* stream);
ADMMQ_API size_t admmq_mttkrp_tc_workspace_bytes(int M, int nx, int ny, int R);
ADMMQ_API int admmq_mttkrp_tc(const float* V, int M, const float* X, int nx, const float* Y, int ny, int R, float* F,
                    void* workspace, size_t workspace_bytes, void* stream);

/* The kernel an MTTKRP call runs on a device with sm_count SMs: precision 0 is admmq_mttkrp(..., 0, ...), precision 1
 * the permuted-operand call admmq_mttkrp_tc; ny = 1 for a matrix.  Pure host logic: needs no device, honours
 * ADMMQ_FOLD_BN (a forced width of the fold, read per call).  Returns one of the ids below, or ADMMQ_E_BADARG.
 *   grid    (or NULL) CTAs of the contraction kernel
 *   splits  (or NULL) slices of the float64 sum over p (precision 0, with the workspace that
 *           admmq_mttkrp_workspace_bytes asks for; a smaller one makes it 1); 1 on the tensor cores */
#define ADMMQ_MTTKRP_F64_16 1       /* float64-accumulating CUDA-core tiles of 16 x 64 (M <= 16) */
#define ADMMQ_MTTKRP_F64_64 2       /* ... of 64 x 64 */
#define ADMMQ_MTTKRP_GEMM 1000      /* + tile width (16, 32, 64, 128): matrix, 3xTF32 tcgen05 product F = W . X */
#define ADMMQ_MTTKRP_FOLD 2000      /* + tile width (16 .. 128, multiple of 16): 2 <= ny <= 128, y folded in the epilogue */
#define ADMMQ_MTTKRP_FOLDLONG 3000  /* + tile width (80 .. 128, multiple of 16): ny > 128, two float64 partials per tile */
ADMMQ_API int admmq_mttkrp_kernel(int M, int nx, int ny, int R, int precision, int sm_count, int* grid, int* splits);

/* Reconstruction error pieces for squared_relative_diff  source/admm.py:14-15 with the einsum of
 * scripts/factorize.py:246-253 (3-D) / :296-297 (2-D):  out2 (device double[2]) = { sum (W - [[A,X,Y]])^2, sum W^2 }.
 *   W0 (M x P) mode-0 unfolding, A (M x R), X (nx x R), Y (ny x R) or NULL.  The reconstruction is never stored. */
ADMMQ_API size_t admmq_recon_error_workspace_bytes(int M, int nx, int ny);
ADMMQ_API int admmq_recon_error(const float* W0, int M, const float* A, const float* X, int nx, const float* Y, int ny,
                      int R, double* out2, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ float64 pieces of the ALS + EPC initialisation
 * `parafac_epc` (source/parafac_epc.py:12-82) runs tensorly's ALS (`parafac`, :42-43) and musco's error-preserving
 * correction (`cp_anc`, :63) in float64; both spend their time in MTTKRP and Gram-Hadamard products (tensorly forms the
 * MTTKRP as unfolding x materialised Khatri-Rao: (I J) x R doubles, 2.4 GB for mode 2 of a 512 x 512 x 9 layer, every
 * pass).  Same contracts as admmq_mttkrp / admmq_gram_hadamard with float64 operands and results; the Khatri-Rao
 * operand is formed on the fly.  The R x R eigen-decomposition / linear solve of a mode update stays with the caller.
 *   admmq_normalize_columns_f64   norms[c] = ||U[:, c]||_2 (a zero norm is reported as 1), U[:, c] /= norms[c] in
 *                                 place, carry[c] *= norms[c] (carry may be NULL): the column normalisation that
 *                                 precedes every mode update of cp_anc, with the scale moved into another factor. */
ADMMQ_API size_t admmq_mttkrp_f64_workspace_bytes(int M, int nx, int ny, int R);
ADMMQ_API int admmq_mttkrp_f64(const double* Wn, int M, const double* X, int nx, const double* Y, int ny, int R,
                     double* F, void* workspace, size_t workspace_bytes, void* stream);
ADMMQ_API int admmq_gram_hadamard_f64(const double* U1, int n1, const double* U2, int n2, int R, double* G, void* stream);
ADMMQ_API int admmq_normalize_columns_f64(double* U, int n, int R, double* norms, double* carry, void* stream);

/* ------------------------------------------------------------------ tensor-core building block
 * C (M x N, ldc) = A (M x K, lda) . B (N x K, ldb)^T in 3xTF32 on tcgen05/TMEM: float32 operands are split into
 * tf32 hi + lo on the fly and accumulated as lo.hi + hi.lo + hi.hi in float32 (csrc/tc_gemm.cuh).  This is the tile
 * product behind the throughput mode of the ridge product (source/admm.py:56) and of the 2-D MTTKRP
 * (scripts/factorize.py:277,287).  lda, ldb multiples of 4 and >= K; columns [K, round_up(K, 4)) of A and B must be
 * readable and zero; A, B 16-byte aligned. */
ADMMQ_API int admmq_gemm_nt(const float* A, int lda, int M, const float* B, int ldb, int N, int K, float* C, int ldc,
                  void* stream);

/* ------------------------------------------------------------------ ridge system
 * rho = trace(G)/R and Minv = (G + rho I)^-1  (replaces torch.linalg.cholesky at source/admm.py:52-54;
 * the per-iteration cholesky_solve of :56 becomes a product with Minv).  Blocked float64 Cholesky +
 * triangular inverse run by one cooperative kernel; Minv is (R x ldm) float32, ldm = admmq_padded_ld(R).
 * Minv64 (R x ldm float64, or NULL): the same inverse before its rounding to float32 - the operand of the loop's
 * parity mode (precision 0).  status (device int): 0 or ADMMQ_E_NOT_PD.  rho_out: device float. */
ADMMQ_API int admmq_padded_ld(int R);
ADMMQ_API size_t admmq_spd_inverse_workspace_bytes(int R);
ADMMQ_API int admmq_spd_inverse(const float* G, int R, float* Minv, double* Minv64, float* rho_out, int* status,
                      int max_ctas, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ ADMM inner loop
 * Replaces admm_iteration(H, U, F, G, max_iter, eps, bits, qscheme)  source/admm.py:51-67.
 * One persistent cooperative kernel runs all max_iter-1 iterations: Minv product (:56), projection (:59),
 * dual update (:60), residuals and exit test (:62-65).  H (I x R) and U (I x R) are updated IN PLACE
 * (the Python wrapper returns a fresh H tensor and the caller's U, like the reference).
 *   codes   I*R int8 codes of the final H, or NULL
 *   report  device struct, see below
 * The call itself runs admmq_spd_inverse first (same stream). */
typedef struct admmq_loop_report {
  int32_t iterations; /* inner iterations executed (max_iter-1 unless the exit test fired) */
  int32_t status;     /* ADMMQ_ST_* bits, or a negative ADMMQ_E_* */
  float rho;          /* trace(G)/R */
  float scale;        /* grid scale of the last projection (mse/symmetric/affine); (max-min) for minmax */
  float r;            /* last primal residual  sum (H-H_ls)^2 / sum H^2      source/admm.py:62 */
  float s;            /* last dual residual    sum (H-H_prev)^2 / sum U^2    source/admm.py:63 */
  int32_t best_index; /* chosen clip candidate of the last projection, -1 for other schemes */
  float absmax;       /* abs-max of the last projection input */
  /* device-side profile of CTA 0 (%globaltimer, nanoseconds, barriers included in the phase they end):
   * [0] ridge product H_ls = RHS.Minv, [1] clip search, [2] quantize + dual + residuals + exit test,
   * [3] whole loop.  This is what a --profile run reports per layer without any host sync in the loop. */
  uint64_t phase_ns[4];
} admmq_loop_report;

/* max_ctas (admmq_spd_inverse and both loop entry points): size of the cooperative grid, 0 = one CTA per SM.
 *   Independent solves are latency bound on small factors (three device-wide barriers per iteration), so a caller
 *   with several solves gives each a share of the SMs and runs them concurrently on different streams: cooperative
 *   launches are gang scheduled, a grid that does not fit yet simply waits for SMs to free up.
 *
 * precision (both loop entry points): how the per-iteration ridge product H_ls = (F + rho (H + U)) . Minv is formed
 *   0  parity mode: float64 products and sums against the float64 inverse Minv64, rounded once to float32 - the
 *      correctly rounded solution of the ridge system, which LAPACK's float32 potrs in the reference approximates to
 *      ~3e-7; what the bit-level comparisons against the reference use (general kernel only, FP64 pipe)
 *   1  throughput mode: 3xTF32 on tcgen05 / tensor memory with TMA-fed operands; factors with < 64 rows take 2
 *   2  float32 FFMA on the CUDA cores (tiles; column strips for <= 16 rows; the shared-memory-resident kernel for a
 *      small factor on a budget of one CTA)
 *
 * Shapes: I * admmq_padded_ld(R) < 2^31 (ADMMQ_E_UNSUPPORTED otherwise; the kernels index elements with 32 bits).
 *
 * The loop alone, for callers that keep (Minv, rho) of a ridge system around (admmq_spd_inverse):
 *   Minv  R x admmq_padded_ld(R) float32, rho / inv_status device scalars written by admmq_spd_inverse
 *         (inv_status may be NULL; a non-zero value makes the loop return it in report->status untouched).
 *   Minv64  the float64 inverse (same shape) - required for precision 0, NULL otherwise. */
/* The kernel a loop call with this factor shape, precision and grid size runs (grid = the cooperative grid: max_ctas,
 * or the SM count when max_ctas is 0 or larger).  Pure host logic: needs no device, honours the ADMMQ_NO_RESIDENT /
 * ADMMQ_NO_CLUSTER / ADMMQ_NO_TAP switches and ADMMQ_LOOP_BN.  Returns one of the ids below, or ADMMQ_E_BADARG. */
#define ADMMQ_LOOP_RESIDENT 1  /* one CTA, the whole loop state in shared memory (admm_loop_resident.cuh) */
#define ADMMQ_LOOP_CLUSTER4 2  /* thread-block cluster of 4 CTAs, rows split (admm_loop_cluster.cuh) */
#define ADMMQ_LOOP_CLUSTER8 3  /* the same on 8 CTAs */
#define ADMMQ_LOOP_TAP 4       /* cluster of 8 CTAs for <= 9 rows, columns split (admm_loop_tap.cuh) */
#define ADMMQ_LOOP_SKINNY9 5   /* cooperative grid, column strips for <= 9 rows */
#define ADMMQ_LOOP_SKINNY16 6  /* cooperative grid, column strips for 10 .. 16 rows */
#define ADMMQ_LOOP_FFMA64 7    /* cooperative grid, float32 FFMA tiles of 64 x 64 */
#define ADMMQ_LOOP_FFMA32 8    /* ... of 32 x 32 */
#define ADMMQ_LOOP_FFMA16 9    /* ... of 16 x 32 */
#define ADMMQ_LOOP_F64_64 10   /* cooperative grid, float64 parity tiles (precision 0) of 64 x 64 */
#define ADMMQ_LOOP_F64_32 11   /* ... of 32 x 32 */
#define ADMMQ_LOOP_TC 1000     /* + tile width (16 .. 160, multiple of 16): cooperative grid, 3xTF32 tcgen05 product */
ADMMQ_API int admmq_admm_loop_kernel(int I, int R, int num_attempts, int precision, int grid);
ADMMQ_API size_t admmq_admm_loop_workspace_bytes(int I, int R, int num_attempts);
ADMMQ_API int admmq_admm_loop(float* H, float* U, const float* F, const float* Minv, const double* Minv64,
                    const float* rho, const int* inv_status, int I, int R, int max_iter, float eps, int bits, int qscheme,
                    int num_attempts, int precision, int max_ctas, int8_t* codes, admmq_loop_report* report,
                    void* workspace, size_t workspace_bytes, void* stream);

ADMMQ_API size_t admmq_admm_iteration_workspace_bytes(int I, int R, int num_attempts);
ADMMQ_API int admmq_admm_iteration(float* H, float* U, const float* F, const float* G, int I, int R,
                         int max_iter, float eps, int bits, int qscheme, int num_attempts, int precision,
                         int max_ctas, int8_t* codes, admmq_loop_report* report,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ two-block splitting  W ~ W_q + W_r
 * The quantized block's inner loop of scripts/factorize_lowrank.py:80-101 (`admm_iteration(H, U, W, H2, proj_func,
 * rho, max_iter, eps)` with proj_func = quantize_tensor): max_iter-1 iterations of
 *   H_ = (rho (H + U) + W - H2) / (1 + rho);  H = Q(H_ - U);  U += H - H_;  exit when r < eps and s < eps
 * in one persistent cooperative kernel (the least-squares step is elementwise, so there is no ridge product; clip
 * search, dual update, residuals and barriers are those of admmq_admm_loop).  H, U IN/OUT, W, H2 read-only, all n
 * floats.  The low-rank block's projection (an SVD truncation, :80-82) stays with the caller. */
ADMMQ_API size_t admmq_split_loop_workspace_bytes(int64_t n, int num_attempts);
ADMMQ_API int admmq_split_loop(float* H, float* U, const float* W, const float* H2, int64_t n, float rho, int max_iter,
                     float eps, int bits, int qscheme, int num_attempts, int max_ctas, int8_t* codes,
                     admmq_loop_report* report, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ whole outer loop
 * Replaces the AO-ADMM loop of scripts/factorize.py:207-266 (3-D: admmq_factorize_cp3) and :269-310 (2-D:
 * admmq_factorize_mat): up to max_iter_als sweeps of { Gram-Hadamard (:215), MTTKRP (:217), admm_iteration (:218),
 * re-projection (:222) } per mode, the two reconstruction errors (:246-253) and the stop rules (:259-263 / :303-307).
 *   W              device, (I, J, K) / (I, J) row-major float32
 *   A, B, C        device factors (I x R), (J x R), (K x R), IN/OUT; UA, UB, UC the scaled duals, IN/OUT (zero for a
 *                  fresh run, :209-212); Aq, Bq, Cq OUT: the re-projected factors of the last sweep
 *   loss_hist, loss_quant_hist   HOST float arrays with room for max_iter_als + 1 entries (rec_error, quant_rec_error
 *                  per sweep; one leading entry for the initial factors unless init_is_random, :192-201)
 *   sweeps_done    HOST int
 * Enqueues on `stream` and synchronises it once per sweep to read the errors (the reference synchronises there too).
 * Returns ADMMQ_E_NOT_PD when a ridge system is not positive definite (torch.linalg.LinAlgError in the reference). */
typedef struct admmq_factorize_params {
  int32_t max_iter_als;     /* --max_iter_als  (5000) */
  int32_t max_iter_admm;    /* --max_iter_admm (1000) */
  float eps;                /* 1e-8, exit test of admm_iteration  scripts/factorize.py:187 (compared in float32 like the
                               reference's 0-dim float32 tensors r, s against the Python float) */
  double tol;               /* 1e-5, stop rule on the error history  :186 - a Python float (double) in the reference */
  int32_t bits, qscheme, num_attempts;
  int32_t solve_precision;  /* see admmq_admm_loop */
  int32_t mttkrp_precision; /* 0 float64-accumulating CUDA-core MTTKRP, 1 3xTF32 tcgen05 */
  int32_t max_ctas;         /* cooperative-grid budget, 0 = every SM */
  int32_t init_is_random;   /* non-zero: no leading history entry (:192) */
} admmq_factorize_params;
ADMMQ_API size_t admmq_factorize_workspace_bytes(int ndim, const int* shape, int R, const admmq_factorize_params* params);
ADMMQ_API int admmq_factorize_cp3(const float* W, int I, int J, int K, int R, float* A, float* B, float* C,
                        float* UA, float* UB, float* UC, float* Aq, float* Bq, float* Cq,
                        const admmq_factorize_params* params, float* loss_hist, float* loss_quant_hist,
                        int* sweeps_done, void* workspace, size_t workspace_bytes, void* stream);
ADMMQ_API int admmq_factorize_mat(const float* W, int I, int J, int R, float* A, float* B, float* UA, float* UB,
                        float* Aq, float* Bq, const admmq_factorize_params* params, float* loss_hist,
                        float* loss_quant_hist, int* sweeps_done, void* workspace, size_t workspace_bytes, void* stream);

/* Independent solves side by side (layers x reduction rates x bit-widths): one descriptor per problem, each with its
 * own stream, workspace (admmq_factorize_workspace_bytes) and cooperative-grid budget params.max_ctas; the problems
 * are enqueued round by round (one outer sweep each) and overlap on the GPU.  Same results as one admmq_factorize_*
 * call per problem. */
typedef struct admmq_problem {
  const float* W;          /* device */
  int32_t ndim;            /* 2 or 3 */
  int32_t shape[3];
  int32_t rank;
  float* factors[3];       /* device, IN/OUT */
  float* duals[3];         /* device, IN/OUT */
  float* factors_q[3];     /* device, OUT */
  admmq_factorize_params params;
  float* loss_hist;        /* HOST, params.max_iter_als + 1 floats */
  float* loss_quant_hist;  /* HOST */
  int32_t* sweeps_done;    /* HOST */
  void* workspace;         /* device, 256-byte aligned */
  size_t workspace_bytes;
  void* stream;            /* cudaStream_t of this problem */
} admmq_problem;
ADMMQ_API int admmq_factorize_batch(int n_problems, const admmq_problem* problems);

#ifdef __cplusplus
}
#endif
#endif /* ADMMQ_H_ */
