// Low-rank proximal step helpers (SVT, main_LRS_PnP.py:118-124) for tall-skinny Z [R, C], C = bands.
// SVT(Z, tau) = U soft(S, tau) V^T = Z * (V diag(max(1 - tau/sigma, 0)) V^T), with V, sigma^2 from the
// eigen-decomposition of the C x C Gram matrix Z^T Z.  The Gram matrix is accumulated in fp64 (products
// of two fp32 are exact in fp64), the small eigh is the caller's (host code), the recomposition is a
// fused  (X + c L) * W  GEMM.
#include "common.cuh"

namespace lrs {

int svt_apply_impl(const float* X, const float* L, float c, const float* W, int64_t R, int64_t C, float* U,
                   cudaStream_t st);

constexpr int GT = 64;       // output tile (bands x bands)
constexpr int GROWS = 16;    // rows staged per step

// grid.x = upper-triangular tile pairs, grid.y = row chunks.  256 threads, 4x4 fp64 accumulators each.
// The tiles are staged as fp64 (one conversion per loaded element instead of one per use: with fp32 tiles the F2F
// conversions, not the DFMA pipe, bound the kernel) and a thread's 4 + 4 operands are 16 columns apart, so the 16 lanes
// that differ in tx read 128 contiguous bytes (one wavefront) and the lanes that share ty read one broadcast word.
__global__ void __launch_bounds__(256) gram_kernel(const float* __restrict__ X, const float* __restrict__ L, float c,
                                                   int64_t R, int64_t C, int ntile, int64_t rows_per_block,
                                                   double* __restrict__ G) {
    __shared__ double Zi[GROWS][GT];
    __shared__ double Zj[GROWS][GT];
    // decode (ti <= tj) from the linear pair index
    int pair = blockIdx.x, ti = 0;
    while (pair >= ntile - ti) {
        pair -= ntile - ti;
        ++ti;
    }
    int tj = ti + pair;
    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const int64_t ci0 = (int64_t)ti * GT, cj0 = (int64_t)tj * GT;
    int64_t r_begin = blockIdx.y * rows_per_block;
    int64_t r_end = r_begin + rows_per_block < R ? r_begin + rows_per_block : R;
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    // software pipeline: the global loads of stage s+1 are in flight while stage s is multiplied (a block's stages would
    // otherwise each expose one DRAM latency: load -> barrier -> 16 x 16 DFMA -> barrier)
    constexpr int EPT = GROWS * GT / 256;                      // staged elements per thread and operand
    float vi[EPT], vj[EPT];
    auto fetch = [&](int64_t r0) {
#pragma unroll
        for (int q = 0; q < EPT; ++q) {
            const int e = tid + 256 * q, rr = e / GT, cc = e % GT;
            const int64_t r = r0 + rr;
            vi[q] = 0.f;
            vj[q] = 0.f;
            if (r < r_end) {
                if (ci0 + cc < C) {
                    int64_t o = r * C + ci0 + cc;
                    vi[q] = __ldg(X + o);
                    if (L) vi[q] = __fadd_rn(vi[q], __fmul_rn(c, __ldg(L + o)));
                }
                if (cj0 + cc < C) {
                    int64_t o = r * C + cj0 + cc;
                    vj[q] = __ldg(X + o);
                    if (L) vj[q] = __fadd_rn(vj[q], __fmul_rn(c, __ldg(L + o)));
                }
            }
        }
    };
    fetch(r_begin);
    for (int64_t r0 = r_begin; r0 < r_end; r0 += GROWS) {
#pragma unroll
        for (int q = 0; q < EPT; ++q) {
            const int e = tid + 256 * q, rr = e / GT, cc = e % GT;
            Zi[rr][cc] = (double)vi[q];
            Zj[rr][cc] = (double)vj[q];
        }
        __syncthreads();
        if (r0 + GROWS < r_end) fetch(r0 + GROWS);
#pragma unroll
        for (int rr = 0; rr < GROWS; ++rr) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = Zi[rr][ty + 16 * i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Zj[rr][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int64_t gi = ci0 + ty + 16 * i;
        if (gi >= C) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int64_t gj = cj0 + tx + 16 * j;
            if (gj >= C) continue;
            if (ti == tj) {
                atomicAdd(G + gi * C + gj, acc[i][j]);  // diagonal tile computes both triangles itself
            } else {
                atomicAdd(G + gi * C + gj, acc[i][j]);
                atomicAdd(G + gj * C + gi, acc[i][j]);
            }
        }
    }
}

// W[i,j] = sum_k V[i,k] w_k V[j,k],  w_k = max(1 - tau/sigma_k, 0),  sigma_k = sqrt(max(lambda_k, 0))  (fp64 sum, fp32 out):
// the singular-value shrinkage of main_LRS_PnP.py:121-123 expressed on the eigenpairs of the band Gram matrix.  One
// launch instead of a dozen elementwise / GEMM launches of host code between the eigensolver and the recomposition.
// V is addressed through its two strides (eigensolvers return column-major eigenvector matrices); only the leading
// C x C block of the n-eigenpair problem is produced (n > C for a zero-bordered problem, see ops.svt_weights).
// BFORM: column k of V holds b_k = lambda_k v_k (the one-sided Jacobi solver, jacobi_eig.cu), so w_k is divided by
// lambda_k^2; directions that are numerically zero (lambda_k <= 1e-12 lambda_max: b_k is rounding noise) get weight 0.
constexpr int WT = 16;
template <bool BFORM>
__global__ void __launch_bounds__(WT * WT) svt_weights_kernel(const double* __restrict__ evals, const double* __restrict__ V,
                                                              int64_t sr, int64_t sk, int C, int n, double tau,
                                                              float* __restrict__ W) {
    __shared__ double Vi[WT][WT + 1], Vj[WT][WT + 1], wk[WT], red[WT * WT / 32];
    const int tx = threadIdx.x % WT, ty = threadIdx.x / WT;
    const int i0 = blockIdx.y * WT, j0 = blockIdx.x * WT;
    double cut = 0.0;
    if (BFORM) {
        double mx = 0.0;
        for (int k = threadIdx.x; k < n; k += WT * WT) mx = fmax(mx, evals[k]);      // fmax drops NaN: handled per k below
        for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
        __syncthreads();
        for (int q = 0; q < WT * WT / 32; ++q) cut = fmax(cut, red[q]);
        cut *= 1e-12;
    }
    double acc = 0.0;
    for (int k0 = 0; k0 < n; k0 += WT) {
        const int k = k0 + tx;
        Vi[ty][tx] = (i0 + ty < C && k < n) ? V[(int64_t)(i0 + ty) * sr + (int64_t)k * sk] : 0.0;
        Vj[ty][tx] = (j0 + ty < C && k < n) ? V[(int64_t)(j0 + ty) * sr + (int64_t)k * sk] : 0.0;
        if (ty == 0) {
            double w = 0.0;
            if (k < n) {
                const double lam = evals[k];
                const double sigma = lam > 0.0 ? sqrt(lam) : 0.0;
                w = sigma > tau ? 1.0 - tau / sigma : 0.0;
                if (BFORM) w = lam > cut ? w / (lam * lam) : 0.0;
                if (!(lam - lam == 0.0)) w = lam - lam;             // NaN / Inf eigenvalues poison W (the caller checks them)
            }
            wk[tx] = w;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < WT; ++kk) acc = fma(Vi[ty][kk] * wk[kk], Vj[tx][kk], acc);
        __syncthreads();
    }
    if (i0 + ty < C && j0 + tx < C) W[(int64_t)(i0 + ty) * C + j0 + tx] = (float)acc;
}

}  // namespace lrs

using namespace lrs;

extern "C" {

int lrs_svt_weights_f64(const double* evals_dev, const double* V_dev, int64_t v_row_stride, int64_t v_col_stride, int C,
                        int n_eig, double tau, int b_form, float* W_dev, lrs_stream_t stream) {
    const char* fn = "lrs_svt_weights_f64";
    if (C <= 0 || n_eig < C || !evals_dev || !V_dev || !W_dev || v_row_stride == 0 || v_col_stride == 0 || !(tau >= 0.0))
        return fail_arg(fn, "bad arguments");
    dim3 grid((unsigned)((C + WT - 1) / WT), (unsigned)((C + WT - 1) / WT));
    if (b_form)
        svt_weights_kernel<true><<<grid, WT * WT, 0, (cudaStream_t)stream>>>(evals_dev, V_dev, v_row_stride, v_col_stride, C, n_eig, tau, W_dev);
    else
        svt_weights_kernel<false><<<grid, WT * WT, 0, (cudaStream_t)stream>>>(evals_dev, V_dev, v_row_stride, v_col_stride, C, n_eig, tau, W_dev);
    LRS_CHECK_LAUNCH(fn);
    return LRS_OK;
}

int lrs_gram_f64(const float* X_dev, const float* L_dev, float c, int64_t R, int64_t C, double* G_dev,
                 lrs_stream_t stream) {
    const char* fn = "lrs_gram_f64";
    if (R <= 0 || C <= 0 || !X_dev || !G_dev) return fail_arg(fn, "bad arguments");
    int sms = device_sm_count();
    if (sms <= 0) return check_cuda(fn, cudaErrorNoDevice);
    int ntile = (int)((C + GT - 1) / GT);
    int npairs = ntile * (ntile + 1) / 2;
    // row chunks: two whole waves of the 2 blocks an SM holds (126 registers x 256 threads) — 594 blocks on 296 slots ran
    // as three waves for two waves' worth of work — and at least 256 rows each
    int64_t want_chunks = ((int64_t)sms * 2 * 2) / npairs;
    if (want_chunks < 1) want_chunks = 1;
    int64_t rows_per_block = (R + want_chunks - 1) / want_chunks;
    if (rows_per_block < 256) rows_per_block = 256;
    rows_per_block = (rows_per_block + GROWS - 1) / GROWS * GROWS;
    int64_t chunks = (R + rows_per_block - 1) / rows_per_block;
    if (chunks > 65535) return fail_arg(fn, "R too large");
    dim3 grid(npairs, (unsigned)chunks);
    gram_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(X_dev, L_dev, c, R, C, ntile, rows_per_block, G_dev);
    LRS_CHECK_LAUNCH(fn);
    return LRS_OK;
}

int lrs_svt_apply_f32(const float* X_dev, const float* L_dev, float c, const float* W_dev, int64_t R, int64_t C,
                      float* U_dev, lrs_stream_t stream) {
    if (R <= 0 || C <= 0 || !X_dev || !W_dev || !U_dev) return fail_arg("lrs_svt_apply_f32", "bad arguments");
    return svt_apply_impl(X_dev, L_dev, c, W_dev, R, C, U_dev, (cudaStream_t)stream);
}

}  // extern "C"
