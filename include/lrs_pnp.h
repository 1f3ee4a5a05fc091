/*
 * lrs_pnp.h — C ABI of liblrs_pnp.so, the B200 (sm_100a) implementation of the
 * LRS-PnP sparse-coding hot path (patch gather → masked ISTA against a
 * dictionary → overlap-sum scatter → closed-form ADMM update, plus the
 * singular-value-thresholding helpers).
 *
 * The reference (shuoli0708/LRS-PnP-DIP) has no FFI: its boundary is a set of
 * Python functions and the script body around them.  Each entry point below
 * names the reference lines it replaces (paths relative to the reference
 * checkout); lrs_pnp_dip_b200/ops.py binds them with ctypes and re-exports the
 * reference's own signatures.
 *
 * Conventions
 *  - extern "C", plain C types only.  Every function returns 0 on success or a
 *    negative LRS_E_* code; lrs_last_error() returns a thread-local message.
 *    No exception crosses this boundary.
 *  - Every pointer named *_dev is a DEVICE pointer owned by the caller; the
 *    library never allocates, frees or retains it.  Workspaces are sized by the
 *    matching *_workspace_bytes() query and passed in.
 *  - Matrices are row-major.  The unfolded cube is [R, C] (R = pixels, C =
 *    bands); patch matrices are [n, P] with n = bb*bb, element k of a patch =
 *    window(row k % bb, col k / bb), patches ordered with the ROW start
 *    varying fastest (main_LRS_PnP.py:94-105).
 *  - The last argument is the CUDA stream (cudaStream_t passed as void*).  All
 *    work is enqueued asynchronously on it; no hidden device synchronisation.
 *  - There is no CPU fallback: without a CUDA device every compute entry point
 *    fails with LRS_E_CUDA.
 *  - Batched forms (*_batch_*) serve B cubes of ONE geometry (same R, C, bb,
 *    s): every per-cube array is [B, ...] contiguous, cube b at offset b times
 *    the per-cube size, 1 <= B <= LRS_MAX_BATCH.  Slice b of a batched result
 *    is what the single-cube entry point gives for cube b (each single-cube
 *    entry point is the B = 1 call of the same launcher).
 */
#ifndef LRS_PNP_H_
#define LRS_PNP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRS_OK 0
#define LRS_E_ARG (-1)       /* invalid argument / unsupported shape */
#define LRS_E_CUDA (-2)      /* CUDA runtime error (message has the cudaError string) */
#define LRS_E_WORKSPACE (-3) /* workspace too small */

#define LRS_MAX_BATCH 65535 /* largest cube count of a batched entry point (the cube is a grid dimension) */

#define LRS_STEP_SPECTRAL 0 /* a = ||H||_2^2        main_LRS_PnP.py:134, ista.m:15 */
#define LRS_STEP_FROB4 1    /* a = 4*||H||_F^2      main_LRS_PnP_DIP_pro.py:190     */

#define LRS_DENOISE_SOFT 0
#define LRS_DENOISE_NLM 1
#define LRS_DENOISE_IDENTITY 2

/* engines of lrs_sparse_step_fused_f32 */
#define LRS_ENGINE_AUTO 0
#define LRS_ENGINE_SIMT 1   /* fp32 FFMA kernel (K in {64,128,192,256})                   */
#define LRS_ENGINE_TC 2     /* tcgen05/TMEM kernel, 3-pass fp16 split (n = 64, K in {64,128,192,256}) */
/* OR-ed into `engine`: the tcgen05 kernel's CTAs CLAIM their work items from a device counter instead of being dealt them,
 * for a launch that shares the GPU with another kernel (CTAs that start late take fewer items).  Costs ~4 % in cycles
 * (DESIGN 3), so it is meant for that launch only. */
#define LRS_ENGINE_DYNAMIC_TILES 0x100

typedef void* lrs_stream_t;

const char* lrs_last_error(void);
int lrs_version(void);
/* Number of CUDA kernels this library has launched in the calling process (monotonic). */
uint64_t lrs_launch_count(void);

/* ---- patch geometry: get_image_block's index logic, main_LRS_PnP.py:76-99 ------------------- */
/* Number of selected starts along an axis of `length` (stride s, last start appended iff
 * length % bb != 0) — host only. */
int64_t lrs_axis_count(int64_t length, int bb, int s);
/* starts_out[count] (host memory). */
int lrs_axis_starts(int64_t length, int bb, int s, int64_t* starts_out, int64_t count);
/* x_index / y_index (int64 [P], device) in reference order, and idx_Mat ([R-bb+1, C-bb+1] f32,
 * device; may be NULL). */
int lrs_patch_index_i64(int64_t R, int64_t C, int bb, int s, int64_t* x_index_dev, int64_t* y_index_dev,
                        float* idx_mat_dev, lrs_stream_t stream);

/* ---- im2col / col2im ----------------------------------------------------------------------- */
/* blocks[n,P] = patches of (X + L / mu) ; L_dev may be NULL (then plain X).
 * Replaces get_image_block, main_LRS_PnP.py:73-107 (calls at :244, :259, :328). */
int lrs_im2col_f32(const float* X_dev, const float* L_dev, float mu, int64_t R, int64_t C, int bb, int s,
                   float* blocks_dev, lrs_stream_t stream);
/* IMout[R,C] = overlap SUM of patches, float32 adds in ascending patch order (bit-exact with the
 * sequential loop main_LRS_PnP.py:332-339).  Deterministic gather, no atomics. */
int lrs_col2im_accum_f32(const float* blocks_dev, int64_t R, int64_t C, int bb, int s, float* imout_dev,
                         lrs_stream_t stream);
/* Batched im2col / col2im: X_dev, L_dev (may be NULL), imout_dev [B, R, C]; blocks_dev [n, B*P] with cube b in columns
 * [b*P, (b+1)*P).  The overlap sum of a cube keeps the sequential fp32 order of lrs_col2im_accum_f32. */
int lrs_im2col_batch_f32(const float* X_dev, const float* L_dev, float mu, int64_t B, int64_t R, int64_t C, int bb, int s,
                         float* blocks_dev, lrs_stream_t stream);
int lrs_col2im_accum_batch_f32(const float* blocks_dev, int64_t B, int64_t R, int64_t C, int bb, int s, float* imout_dev,
                               lrs_stream_t stream);
/* The same overlap sum fed one RANGE of column starts at a time (bb = 8, s = 1): blocks_dev holds only the patches
 * p in [ci_begin*nR, ci_end*nR) (nR = R-bb+1 row starts; [n, (ci_end-ci_begin)*nR] row-major — what
 * lrs_sparse_step_fused_f32 writes for that patch range) and imout_dev carries the running sum.  Patch order is
 * column-start-outer (main_LRS_PnP.py:94-99), so calling with ascending, contiguous ranges that start at 0 continues
 * every element's sequential fp32 sum exactly where the previous range left it: the result is bit-identical to
 * lrs_col2im_accum_f32 on the whole Phi_z (main_LRS_PnP.py:332-339) without ever materialising it.  imout_dev needs no
 * initialisation: an element's sum starts from 0 in the range that holds its first covering patch. */
int lrs_col2im_accum_range_f32(const float* blocks_dev, int64_t R, int64_t C, int bb, int s, int64_t ci_begin,
                               int64_t ci_end, float* imout_dev, lrs_stream_t stream);
/* Weight[R,C] of main_LRS_PnP.py:341 (analytic coverage count). */
int lrs_coverage_weight_f32(int64_t R, int64_t C, int bb, int s, float* weight_dev, lrs_stream_t stream);

/* ---- elementwise ---------------------------------------------------------------------------- */
/* out = sign(x)*max(|x|-tau,0): soft.m:4, soft_thresh main_LRS_PnP.py:128, Shrinkage_Operator :112,
 * l1_prox admm_utils.py:72. */
int lrs_soft_f32(const float* x_dev, float tau, float* out_dev, int64_t count, lrs_stream_t stream);
/* out = x + c*l  (Z = X + (1/mu_2)*lambda_2, main_LRS_PnP.py:315) */
int lrs_axpy_f32(const float* x_dev, const float* l_dev, float c, float* out_dev, int64_t count,
                 lrs_stream_t stream);

/* ---- step constants ------------------------------------------------------------------------- */
/* a[p] = 4*sum_i m[i,p]*||D[i,:]||^2 for explicit patch matrices; mask = (blocks_copy != 0).
 * main_LRS_PnP_DIP_pro.py:190. */
int lrs_step_frob4_f32(const float* blocks_copy_dev, const float* D_dev, int n, int K, int64_t P, float* a_dev,
                       lrs_stream_t stream);

/* Per-patch step constants for ANY mask (bb <= 8), in two stages; the caller merges equal words in between
 * (ops.patch_step_constants).  Together they replace np.linalg.norm(H, 2)**2 with H = D minus the patch's missing rows
 * (main_LRS_PnP.py:134, :276-289), paid per patch per outer iteration in the reference, by one value per distinct mask
 * pattern per dictionary; the result feeds a_patch_dev of lrs_sparse_step_fused_f32 or a_dev of lrs_ista_pnp_f32.
 *
 * words_dev[p - p_begin] for the patches p in [p_begin, p_end) (reference order): bit k set iff element k of the patch
 * (window row k % bb, column k / bb) is observed, Yobs != 0.0f as in the fused kernels (-0.0 missing, NaN observed).
 * Any stride. */
int lrs_patch_mask_words_u64(const float* Yobs_dev, int64_t R, int64_t C, int bb, int s, int64_t p_begin, int64_t p_end,
                             uint64_t* words_dev, lrs_stream_t stream);
/* a_dev[i] for each pattern word words_dev[i] (bit k = row k of D [n, K], n <= 64): LRS_STEP_SPECTRAL lambda_max of
 * G[S,S], G = D D^T in fp64 (fp64 Lanczos), LRS_STEP_FROB4 4 tr G[S,S]; the empty pattern gives exactly 0.  Equal words
 * give bit-identical values.  count_dev: NULL -> all max_count words; else a device int64 holding how many of the
 * max_count words to process (the launch is sized for max_count and reads the count on the device: no host
 * synchronisation).
 * Run on the 2^bb row-pattern words (bit k set iff bit k % bb of the row pattern is set: band-replicated masks,
 * main_LRS_PnP.py:188-192), it also fills a_table_dev of lrs_sparse_step_fused_f32: one table per dictionary. */
size_t lrs_spectral_patterns_workspace_bytes(int n);
int lrs_spectral_patterns_f32(const float* D_dev, int n, int K, const uint64_t* words_dev, int64_t max_count,
                              const int64_t* count_dev, int step, float* a_dev, void* workspace_dev, size_t workspace_bytes,
                              lrs_stream_t stream);

/* ---- batched soft-ISTA on explicit patch matrices ------------------------------------------- */
/* For every patch p: alpha=0; repeat Nit: alpha <- soft(alpha + D^T(m.*(y - D alpha))/a_p, lambda/(2 a_p))
 * with m = (blocks_copy[:,p] != 0)  [row deletion of main_LRS_PnP.py:276-289 in masked form],
 * then phi_z[:,p] = D alpha (full dictionary, :294/:302).  Patches with a_p <= 0 give alpha = 0.
 * Replaces the jj loop main_LRS_PnP.py:270-303 + ista :131-149 / ista.m:13-24.
 * coefs_dev [K,P] and phi_z_dev [n,P] may each be NULL.  Any n, K, P.
 * Engines (chosen per call, same results to <= 2e-5 relative, all denoisers): for P >= 8 and n, K >= 128 (the 36x36-patch
 * configurations) the two products of an iteration run as split-K tcgen05 GEMMs with a 3-pass fp16 operand split
 * (ista_tc.cu); every other shape, and the environment override LRS_ISTA_ENGINE=simt, uses the fp32 FFMA kernels.
 * lrs_ista_workspace_bytes covers whichever engine the shape may take. */
size_t lrs_ista_workspace_bytes(int n, int K, int64_t P);
int lrs_ista_soft_f32(const float* blocks_dev, const float* blocks_copy_dev, const float* D_dev, const float* a_dev,
                      float lambda_ista, int Nit, int n, int K, int64_t P, float* coefs_dev, float* phi_z_dev,
                      void* workspace_dev, size_t workspace_bytes, lrs_stream_t stream);

/* Plug-and-play variant: the same iteration with the proximal step replaced by a denoiser of the K x 1 gradient-step
 * vector — LRS_DENOISE_SOFT soft(g, T) (ista.m:23); LRS_DENOISE_NLM NLmeansfilter(g, 3, 3, h_scale*T)
 * (pnp_ista.m:30, NLmeansfilter.m:1-91; h_scale = 0.1 in the MATLAB file); LRS_DENOISE_IDENTITY none. */
int lrs_ista_pnp_f32(const float* blocks_dev, const float* blocks_copy_dev, const float* D_dev, const float* a_dev,
                     float lambda_ista, int Nit, int n, int K, int64_t P, int denoiser, float h_scale, float* coefs_dev,
                     float* phi_z_dev, void* workspace_dev, size_t workspace_bytes, lrs_stream_t stream);

/* ---- fused sparse step on the implicit patch set (bb = 8) ------------------------------------ */
/* phi_z[64,P] for all patches of V = X + L/mu_1, mask taken from Yobs != 0 (main_LRS_PnP.py:244,
 * 259-303) without materialising the patch matrices.  Step constants: a_patch_dev [P] if non-NULL,
 * else a_table_dev[256] indexed by the 8-bit validity pattern of the patch's 8 rows (bit i = row
 * r+i observed; requires band-replicated masks), else (both NULL) 4*||H||_F^2 computed in-kernel.
 * patch range [p_begin, p_end) in reference order lets callers shard / chunk; phi_z_dev holds
 * columns p_begin..p_end-1 (leading dimension p_end-p_begin). */
int lrs_sparse_step_fused_f32(const float* X_dev, const float* L_dev, float mu_1, const float* Yobs_dev,
                              const float* D_dev, int K, const float* a_patch_dev, const float* a_table_dev,
                              float lambda_ista, int Nit, int64_t R, int64_t C, int bb, int s, int64_t p_begin,
                              int64_t p_end, float* phi_z_dev, int engine, lrs_stream_t stream);

/* ---- closed-form X and multiplier update ------------------------------------------------------ */
/* X = (g*Y + mu1*IMout + mu2*U - lam1sum - lam2) / (g*MtM + mu1*Weight + mu2)   main_LRS_PnP.py:346
 * lam1 += mu1*(X - IMout) ; lam2 += mu2*(X - U)                                  :361-362
 * Weight and lam1sum (= lam1 added Weight times, sequential fp32 adds, :343) are derived from the
 * geometry in-kernel.  X_out, lam1 and lam2 are updated in place (lam1_dev/lam2_dev in/out).
 * The arrays hold `rows` rows that start at row `row_offset` of the full R_total x C matrix (a row
 * stripe of a sharded run; rows = R_total, row_offset = 0 for the whole matrix): the coverage
 * count is that of the FULL geometry. */
int lrs_admm_update_f32(const float* Y_dev, const float* MtM_dev, const float* imout_dev, const float* U_dev,
                        float* lam1_dev, float* lam2_dev, float* X_out_dev, float gamma, float mu_1, float mu_2,
                        int64_t rows, int64_t row_offset, int64_t R_total, int64_t C, int bb, int s,
                        lrs_stream_t stream);
/* The same update for B whole cubes [B, R, C] of one geometry (Weight and lam1sum shared). */
int lrs_admm_update_batch_f32(const float* Y_dev, const float* MtM_dev, const float* imout_dev, const float* U_dev,
                              float* lam1_dev, float* lam2_dev, float* X_out_dev, float gamma, float mu_1, float mu_2, int64_t B,
                              int64_t R, int64_t C, int bb, int s, lrs_stream_t stream);

/* ---- low-rank proximal step (SVT, main_LRS_PnP.py:118-124) via the band Gram matrix ------------ */
/* G[C,C] (fp64, device, accumulated INTO — caller zeroes) += Z^T Z with Z = X + c*L (L may be NULL). */
int lrs_gram_f64(const float* X_dev, const float* L_dev, float c, int64_t R, int64_t C, double* G_dev,
                 lrs_stream_t stream);
/* G[B,C,C] += Z_b^T Z_b for the B cubes Z_b = X_b + c*L_b of [B, R, C] arrays (caller zeroes G). */
int lrs_gram_batch_f64(const float* X_dev, const float* L_dev, float c, int64_t B, int64_t R, int64_t C, double* G_dev,
                       lrs_stream_t stream);
/* Symmetric eigen-decomposition of the band Gram matrix (fp64, symmetric positive semi-definite, 1 <= C <= 256) in ONE
 * launch: one-sided Jacobi over a thread-block cluster (csrc/jacobi_eig.cu) — replaces the eigh / SVD of
 * main_LRS_PnP.py:119 without a host synchronisation.  Outputs: lam_dev[C] eigenvalues (unsorted), Bt_dev[C*C] with row k
 * = lambda_k * v_k (the eigenvector scaled by its eigenvalue; "B form"), status_dev[3] = {sweeps run, 1 if not converged,
 * 1 if an eigenvalue is not finite}. */
int lrs_sym_eig_jacobi_f64(const double* G_dev, int C, double* lam_dev, double* Bt_dev, int* status_dev, lrs_stream_t stream);
/* B independent problems in one launch (one cluster each; clusters need not be co-resident): G_dev [B,C,C], lam_dev [B,C],
 * Bt_dev [B,C,C], status_dev [B,3]. */
int lrs_sym_eig_jacobi_batch_f64(const double* G_dev, int64_t B, int C, double* lam_dev, double* Bt_dev, int* status_dev,
                                 lrs_stream_t stream);
/* W[C,C] (f32) = V diag(max(1 - tau/sigma_k, 0)) V^T on the leading C x C block, sigma_k = sqrt(max(evals[k], 0)):
 * the shrinkage of main_LRS_PnP.py:121-123 on the n_eig >= C eigenpairs of the (possibly zero-bordered) Gram matrix.
 * V[i,k] is read at V_dev[i*v_row_stride + k*v_col_stride] (eigenvectors in columns, either storage order).
 * b_form != 0: column k holds lambda_k * v_k as lrs_sym_eig_jacobi_f64 returns it (v_row_stride = 1, v_col_stride = C). */
int lrs_svt_weights_f64(const double* evals_dev, const double* V_dev, int64_t v_row_stride, int64_t v_col_stride, int C,
                        int n_eig, double tau, int b_form, float* W_dev, lrs_stream_t stream);
/* B weight matrices W_dev [B,C,C]: eigenvalues of cube b at evals_dev + b*n_eig, its eigenvectors at
 * V_dev + b*v_batch_stride (the strides above within a cube). */
int lrs_svt_weights_batch_f64(const double* evals_dev, const double* V_dev, int64_t v_batch_stride, int64_t v_row_stride,
                              int64_t v_col_stride, int64_t B, int C, int n_eig, double tau, int b_form, float* W_dev,
                              lrs_stream_t stream);
/* U[R,C] = (X + c*L) * W, W [C,C] f32 = V diag(max(1 - tau/sigma, 0)) V^T from the caller's eigh. */
int lrs_svt_apply_f32(const float* X_dev, const float* L_dev, float c, const float* W_dev, int64_t R, int64_t C,
                      float* U_dev, lrs_stream_t stream);
/* U_b = (X_b + c*L_b) * W_b for B cubes: X, L, U [B, R, C], W [B, C, C]. */
int lrs_svt_apply_batch_f32(const float* X_dev, const float* L_dev, float c, const float* W_dev, int64_t B, int64_t R,
                            int64_t C, float* U_dev, lrs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LRS_PNP_H_ */
