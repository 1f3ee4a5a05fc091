/* Diagnostics of the tcgen05 engine — NOT part of the product ABI.
 *
 * These entry points exist only in lrs_pnp_dip_b200/csrc/liblrs_pnp_diag.so, the diagnostics build of the library (the
 * same sources compiled with -DLRS_DIAGNOSTICS plus tc_probe.cu).  The product library liblrs_pnp.so (include/lrs_pnp.h)
 * exports none of them and carries no timing instrumentation.  They have no counterpart in the reference; tests/ and
 * scripts/ use them to pin hardware behaviour (operand layouts, rounding), to replay the fused kernel's tile order on
 * the host, and to read the barrier-wait counters of an instrumented launch. */
#ifndef LRS_PNP_DIAG_H
#define LRS_PNP_DIAG_H

#include "lrs_pnp.h"

#ifdef __cplusplus
extern "C" {
#endif

/* C[128,N] = A[128,Kd] * B[N,Kd]^T through one CTA's tensor core with the operand layouts of the fused
 * kernel: A from shared memory (a_in_tmem = 0) or TMEM (1); B K-major (b_mn_major = 0) or MN-major (1),
 * SWIZZLE_NONE; f16 = 0: kind::tf32 on the fp32 data, 1: kind::f16 on the data rounded to fp16. */
int lrs_tc_probe_f32(const float* A_dev, const float* B_dev, float* C_dev, int N, int Kd, int a_in_tmem,
                     int b_mn_major, int f16, lrs_stream_t stream);
/* Barrier-wait cycle counters of the fused tcgen05 kernel (block 0), filled when the environment variable
 * LRS_TC_TIMING is set at the first launch; out32_host = uint64 [32] in HOST memory. */
int lrs_tc_timing_read(unsigned long long* out32_host);
/* HOST-side replay (no GPU needed) of the tile order the fused tcgen05 kernel uses for the patch range
 * [p_begin, p_end) on a device with `sms` SMs: visits_host[p - p_begin] is incremented once per lane that owns patch p
 * (the caller zeroes it; a correct walk leaves every entry at 1), tiles_host receives the number of tiles.  bb = 8. */
int lrs_debug_tile_walk(int64_t R, int64_t C, int bb, int s, int64_t p_begin, int64_t p_end, int sms, int* visits_host,
                        int64_t* tiles_host);
/* The same replay for the row-pattern tile order of the step-constant table mode: row_obs_host = R bytes, nonzero where
 * a row of the matrix is observed; order_host (nR ints, may be null) receives the row starts in tile order, which is
 * the stable sort of the row starts by the Gray rank of their 8-row validity word. */
int lrs_debug_tile_walk_ordered(int64_t R, int64_t C, int bb, int s, int64_t p_begin, int64_t p_end, int sms,
                                const unsigned char* row_obs_host, int* visits_host, int64_t* tiles_host, int* order_host);
/* HOST-side replay (no GPU needed) of the launch plan of lrs_ista_pnp_f32 for an [n, K] dictionary and P patches;
 * out_host = int64 [15] in HOST memory:
 *   [0]  engine by shape: 1 = tensor-core (ista_tc.cu; LRS_ISTA_ENGINE=simt still forces the FFMA engine), 0 = FFMA
 *   tensor-core plan (0 when [0] is 0): [1] Np = P rounded up to 16, [2] patch tiles of 256 columns, [3] width of the
 *   last tile, [4] pipeline stages, [5] S1 / [6] k blocks per split of D alpha, [7] S2 / [8] of D^T r, [9] / [10] k blocks
 *   of the last split of D alpha / D^T r
 *   FFMA engine (any shape): [11] / [12] k splits of the residual / gradient GEMM, [13] / [14] their rows per CTA
 *   (on a 148-SM device). */
int lrs_debug_ista_plan(int n, int K, int64_t P, int64_t* out_host);
/* HOST-side replay (no GPU needed) of ONE sweep of the parallel order of lrs_sym_eig_jacobi_f64 (csrc/jacobi_eig.cu) for C
 * columns: meets_host[p*C + q] (p < q; caller zeroes C*C ints) counts how often columns p and q are paired — a correct order
 * leaves every p < q at 1 —, conflicts_host the sub-rounds in which a column was used twice, subrounds_host their number. */
int lrs_debug_jacobi_schedule(int C, int* meets_host, int* conflicts_host, int* subrounds_host);
/* Cycle counts of MMA issue chains / TMEM load-store streams; out_dev = int64 [blocks*16]. */
int lrs_tc_microbench(int do_mma, int f16, int ts, int N, int nacc, int ldst, int depth, int reps, int blocks,
                      long long* out_dev, lrs_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LRS_PNP_DIAG_H */
