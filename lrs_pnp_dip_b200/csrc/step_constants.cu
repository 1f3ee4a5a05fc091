// Per-patch ISTA step constants for any observation mask (main_LRS_PnP.py:134, :276-289): a_p = ||M_p D||_2^2 with M_p
// the rows of the patch that are observed.  The reference pays one SVD per patch per outer iteration; here a patch's
// validity is packed into one 64-bit word (bb <= 8), equal words are merged by the caller (ops.patch_step_constants) and
// one fp64 Lanczos run per distinct word gives lambda_max(G[S,S]), G = D D^T.
#include "common.cuh"

namespace lrs {

// ------------------------------------------------------------------------------------------------
// Validity words.  Bit k of patch p = (Yobs[row start + k % bb, col start + k / bb] != 0.0f), the predicate of the fused
// kernels (sparse_fused_simt.cu, sparse_fused_tc.cu): -0.0 is missing, NaN is observed.
// A block owns WORD_TILE consecutive row starts of one column start.  It first packs the bb-column validity byte of
// every window row it needs (8 lanes read the bb floats of one row: 4 rows = 4 sectors per warp request, as
// im2col_s1_kernel reads its window) and then assembles the words from shared memory.  blockIdx.x runs over column
// starts, so the blocks resident together read neighbouring columns of the same rows and share their sectors in L2.
// ------------------------------------------------------------------------------------------------
constexpr int WORD_TILE = 256;

__global__ void __launch_bounds__(WORD_TILE) patch_mask_words_kernel(Geom g, const float* __restrict__ Y, int64_t p_begin,
                                                                     int64_t p_end, int64_t ci_first, int64_t n_tiles,
                                                                     unsigned long long* __restrict__ words) {
    // window rows: s <= bb -> the contiguous rows [start(first), start(last) + bb) <= (TILE-1)*bb + bb;
    //              s >  bb -> bb rows per patch, TILE*bb
    __shared__ unsigned char rowbits[WORD_TILE * 8];
    const int bb = g.bb;
    const bool dense = g.row.s <= bb;
    const int64_t ci = ci_first + blockIdx.x, nR = g.row.n;
    const int64_t cs = g.col.start(ci);
    for (int64_t tile = blockIdx.y; tile < n_tiles; tile += gridDim.y) {
        const int64_t ri0 = tile * WORD_TILE, pt = ci * nR + ri0;               // patch number of row start ri0
        const int64_t lo = p_begin > pt ? p_begin - pt : 0;
        int64_t hi = nR - ri0 < WORD_TILE ? nR - ri0 : WORD_TILE;
        if (p_end - pt < hi) hi = p_end - pt;
        if (lo >= hi) continue;                                                  // block-uniform
        const int mlo = (int)lo, mhi = (int)hi;
        const int64_t r0 = g.row.start(ri0 + mlo);
        const int wrows = dense ? (int)(g.row.start(ri0 + mhi - 1) - r0) + bb : (mhi - mlo) * bb;
        const int tot = (wrows * 8 + WORD_TILE - 1) / WORD_TILE * WORD_TILE;   // every lane runs every ballot
        for (int e = threadIdx.x; e < tot; e += WORD_TILE) {
            const int w = e >> 3, j = e & 7;
            bool ok = false;
            if (w < wrows && j < bb) {
                const int64_t r = dense ? r0 + w : g.row.start(ri0 + mlo + w / bb) + w % bb;
                ok = __ldg(Y + r * g.C + cs + j) != 0.0f;
            }
            const unsigned b = __ballot_sync(0xffffffffu, ok);
            if (j == 0 && w < wrows) rowbits[w] = (unsigned char)(b >> (threadIdx.x & 24));
        }
        __syncthreads();
        const int m = mlo + (int)threadIdx.x;
        if (m < mhi) {
            const int base = dense ? (int)(g.row.start(ri0 + m) - r0) : (m - mlo) * bb;
            unsigned long long word = 0;
            for (int i = 0; i < bb; ++i) {
                const unsigned b = rowbits[base + i];
                for (int j = 0; j < bb; ++j) word |= (unsigned long long)((b >> j) & 1u) << (i + bb * j);
            }
            words[pt + m - p_begin] = word;
        }
        __syncthreads();                                                         // rowbits is rewritten by the next tile
    }
}

// ------------------------------------------------------------------------------------------------
// One step constant per pattern word.  G = D D^T (fp64, 64 x 64, zero beyond n) stays in shared memory.
//
// LRS_STEP_SPECTRAL: lambda_max(G[S,S]) by fp64 Lanczos from the fixed start vector x_i = 1 + 0.01 i (i in S).  A warp
// carries PW patterns at once, so every G element read from shared memory feeds PW DFMAs; lane l holds elements l and
// l + 32 of each pattern's vectors.  The three-term recurrence is re-orthogonalised once against the current vector
// (no basis is stored: the largest Ritz value of finite-precision Lanczos converges to lambda_max whatever happens to
// the orthogonality of the others).  Every CHECK steps, on a breakdown (beta <= 1e-13 max alpha: the Krylov space is
// invariant) and at KMAX steps, the group of 8 lanes of a pattern brackets lambda_max(T_k) by 9-section with Sturm
// counts; the run stops when the value moved by <= 1e-14 relative since the previous check.
// LRS_STEP_FROB4: 4 tr G[S,S].
//
// Every sum has a fixed order (xor butterflies give all lanes the same bits), and a pattern's arithmetic does not depend
// on the patterns that share its warp: equal words give bit-identical values, in any position and on every call.
// ------------------------------------------------------------------------------------------------
constexpr int PW = 4;          // patterns per warp (= 32 lanes / 8-lane bisection groups)
constexpr int PWARPS = 4;      // warps per block
constexpr int KMAX = 128;      // Lanczos steps at most (2n)
constexpr int CHECK = 4;       // steps between convergence checks
constexpr int SECT_ROUNDS = 18;  // 9^-18 < 2^-57: the bracket [max alpha, Gershgorin bound <= 3 lambda_max] shrinks to rounding level
constexpr size_t PATTERN_SMEM = (64 * 64 + PWARPS * 64 * PW + 2 * PWARPS * KMAX * PW) * sizeof(double);

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

// Number of eigenvalues of the k x k tridiagonal (ta, tb) below x (LDL^T signs, LAPACK's pivmin guard).
__device__ __forceinline__ int sturm_below(const double* ta, const double* tb, int k, double x) {
    const double pivmin = 1e-290;
    double d = ta[0] - x;
    if (fabs(d) < pivmin) d = -pivmin;
    int c = d < 0.0;
    for (int i = 1; i < k; ++i) {
        const double b = tb[(i - 1) * PW];
        d = (ta[i * PW] - x) - b * b / d;
        if (fabs(d) < pivmin) d = -pivmin;
        c += d < 0.0;
    }
    return c;
}

__global__ void __launch_bounds__(PWARPS * 32) ddt64_kernel(const float* __restrict__ D, int n, int K, double* __restrict__ G) {
    for (int e = threadIdx.x + blockIdx.x * blockDim.x; e < 64 * 64; e += blockDim.x * gridDim.x) {
        const int i = e / 64, j = e % 64;
        double s = 0.0;
        if (i < n && j < n)
            for (int k = 0; k < K; ++k) s = fma((double)D[(int64_t)i * K + k], (double)D[(int64_t)j * K + k], s);
        G[e] = s;
    }
}

__global__ void __launch_bounds__(PWARPS * 32) spectral_patterns_kernel(const double* __restrict__ G0, int n,
                                                                        const unsigned long long* __restrict__ words,
                                                                        int64_t max_count, const int64_t* __restrict__ count_dev,
                                                                        int frob4, float* __restrict__ a) {
    extern __shared__ double smem[];
    int64_t count = max_count;
    if (count_dev) {
        const int64_t c = *count_dev;
        count = c < max_count ? c : max_count;
    }
    const int64_t block0 = (int64_t)blockIdx.x * PWARPS * PW;
    if (block0 >= count) return;                                   // beyond the distinct words: nothing to do
    double* G = smem;
    for (int e = threadIdx.x; e < 64 * 64; e += blockDim.x) G[e] = G0[e];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* vs = smem + 64 * 64 + warp * 64 * PW;                  // [64][PW]: the current vectors, broadcast to the warp
    double* ta = smem + 64 * 64 + PWARPS * 64 * PW + warp * KMAX * PW;   // [KMAX][PW] alpha_k
    double* tb = ta + PWARPS * KMAX * PW;                                  // [KMAX][PW] beta_k
    const unsigned long long nmask = n >= 64 ? ~0ull : (1ull << n) - 1;
    const int64_t p0 = block0 + warp * PW;

    bool m0[PW], m1[PW], act[PW];
    double v0[PW], v1[PW], u0[PW], u1[PW], beta[PW], amax[PW], theta[PW];
#pragma unroll
    for (int q = 0; q < PW; ++q) {
        const unsigned long long w = p0 + q < count ? words[p0 + q] & nmask : 0ull;
        m0[q] = (w >> lane) & 1ull;
        m1[q] = (w >> (lane + 32)) & 1ull;
        if (frob4) {
            const double s = warp_sum((m0[q] ? G[lane * 65] : 0.0) + (m1[q] ? G[(lane + 32) * 65] : 0.0));
            if (lane == 0 && p0 + q < count) a[p0 + q] = (float)(4.0 * s);
            act[q] = false;
            continue;
        }
        const double x0 = m0[q] ? 1.0 + 0.01 * lane : 0.0, x1 = m1[q] ? 1.0 + 0.01 * (lane + 32) : 0.0;
        const double nrm = sqrt(warp_sum(x0 * x0 + x1 * x1));
        act[q] = nrm > 0.0;
        if (!act[q] && lane == 0 && p0 + q < count) a[p0 + q] = 0.0f;  // empty pattern (or beyond count: not written)
        v0[q] = act[q] ? x0 / nrm : 0.0;
        v1[q] = act[q] ? x1 / nrm : 0.0;
        u0[q] = u1[q] = beta[q] = amax[q] = 0.0;
        theta[q] = -1.0;
    }
    const int grp = lane >> 3, sub = lane & 7;
    for (int k = 0; k < KMAX; ++k) {
        bool any = false;
#pragma unroll
        for (int q = 0; q < PW; ++q) any |= act[q];
        if (!any) break;                                           // warp-uniform: every lane holds the same flags
#pragma unroll
        for (int q = 0; q < PW; ++q) {
            vs[lane * PW + q] = v0[q];
            vs[(lane + 32) * PW + q] = v1[q];
        }
        __syncwarp();
        double w0[PW], w1[PW];
#pragma unroll
        for (int q = 0; q < PW; ++q) w0[q] = w1[q] = 0.0;
#pragma unroll 4
        for (int j = 0; j < n; ++j) {                              // w = G v (G symmetric: row j read along the lanes)
            const double g0 = G[j * 64 + lane], g1 = G[j * 64 + lane + 32];
            const double2 va = *reinterpret_cast<const double2*>(vs + j * PW);
            const double2 vb = *reinterpret_cast<const double2*>(vs + j * PW + 2);
            const double vj[PW] = {va.x, va.y, vb.x, vb.y};
#pragma unroll
            for (int q = 0; q < PW; ++q) {
                w0[q] = fma(g0, vj[q], w0[q]);
                w1[q] = fma(g1, vj[q], w1[q]);
            }
        }
        __syncwarp();                                              // vs is rewritten next step
        bool chk[PW], brk[PW];
#pragma unroll
        for (int q = 0; q < PW; ++q) {
            w0[q] = m0[q] ? w0[q] : 0.0;                           // G[S,S] v: rows outside S dropped
            w1[q] = m1[q] ? w1[q] : 0.0;
            double alpha = warp_sum(v0[q] * w0[q] + v1[q] * w1[q]);
            w0[q] = w0[q] - alpha * v0[q] - beta[q] * u0[q];
            w1[q] = w1[q] - alpha * v1[q] - beta[q] * u1[q];
            const double c = warp_sum(v0[q] * w0[q] + v1[q] * w1[q]);
            w0[q] -= c * v0[q];
            w1[q] -= c * v1[q];
            alpha += c;
            const double b = sqrt(warp_sum(w0[q] * w0[q] + w1[q] * w1[q]));
            if (act[q] && lane == 0) {
                ta[k * PW + q] = alpha;
                tb[k * PW + q] = b;
            }
            amax[q] = fmax(amax[q], alpha);
            brk[q] = b <= 1e-13 * amax[q];
            chk[q] = act[q] && ((k + 1) % CHECK == 0 || brk[q] || k + 1 == KMAX);
            if (act[q] && !brk[q]) {
                u0[q] = v0[q];
                u1[q] = v1[q];
                v0[q] = w0[q] / b;
                v1[q] = w1[q] / b;
            }
            beta[q] = b;
        }
        bool any_chk = false;
#pragma unroll
        for (int q = 0; q < PW; ++q) any_chk |= chk[q];
        if (!any_chk) continue;
        __syncwarp();                                              // alpha / beta of this step visible to the groups
        // lambda_max(T_{k+1}) of pattern grp by 9-section: 8 lanes, 8 points a round
        const int kk = k + 1;
        bool mine = false;
        double lo = 0.0;
#pragma unroll
        for (int q = 0; q < PW; ++q)
            if (q == grp) {
                mine = chk[q];
                lo = amax[q];                                      // lambda_max >= every diagonal entry
            }
        double hi = lo;
        if (mine)
            for (int i = 0; i < kk; ++i) {
                const double r = ta[i * PW + grp] + (i > 0 ? tb[(i - 1) * PW + grp] : 0.0) + (i + 1 < kk ? tb[i * PW + grp] : 0.0);
                hi = fmax(hi, r);
            }
        for (int round = 0; round < SECT_ROUNDS; ++round) {
            const double h = (hi - lo) / 9.0;
            const double x = lo + h * (sub + 1);
            const bool above = mine && sturm_below(ta + grp, tb + grp, kk, x) < kk;   // lambda_max >= x
            const unsigned t = __popc((__ballot_sync(0xffffffffu, above) >> (grp * 8)) & 0xffu);
            const double nlo = t > 0 ? lo + h * t : lo;
            hi = t < 8 ? lo + h * (t + 1) : hi;
            lo = nlo;
        }
        const double th = 0.5 * (lo + hi);
#pragma unroll
        for (int q = 0; q < PW; ++q) {
            const double tq = __shfl_sync(0xffffffffu, th, q * 8);
            if (!chk[q]) continue;
            const bool done = brk[q] || k + 1 == KMAX || (theta[q] >= 0.0 && fabs(tq - theta[q]) <= 1e-14 * tq);
            theta[q] = tq;
            if (done) {
                act[q] = false;
                if (lane == 0) a[p0 + q] = (float)(tq > 0.0 ? tq : 0.0);
            }
        }
    }
}

}  // namespace lrs

using namespace lrs;

extern "C" {

int lrs_patch_mask_words_u64(const float* Yobs_dev, int64_t R, int64_t C, int bb, int s, int64_t p_begin, int64_t p_end,
                             uint64_t* words_dev, lrs_stream_t stream) {
    const char* fn = "lrs_patch_mask_words_u64";
    Geom g;
    if (!make_geom(R, C, bb, s, g)) return fail_arg(fn, "need 0 < bb <= min(R,C) and s > 0");
    if (bb > 8) return fail_arg(fn, "a validity word holds bb*bb <= 64 bits (bb <= 8)");
    if (p_begin < 0 || p_end > g.P || p_begin > p_end) return fail_arg(fn, "patch range outside [0, P)");
    if (p_begin == p_end) return LRS_OK;
    if (!Yobs_dev || !words_dev) return fail_arg(fn, "null pointer");
    const int64_t nR = g.row.n, ci_first = p_begin / nR, ci_last = (p_end - 1) / nR;
    const int64_t n_tiles = (nR + WORD_TILE - 1) / WORD_TILE;
    dim3 grid((unsigned)(ci_last - ci_first + 1), (unsigned)(n_tiles < 65535 ? n_tiles : 65535));
    patch_mask_words_kernel<<<grid, WORD_TILE, 0, (cudaStream_t)stream>>>(g, Yobs_dev, p_begin, p_end, ci_first, n_tiles,
                                                                         (unsigned long long*)words_dev);
    LRS_CHECK_LAUNCH(fn);
    return LRS_OK;
}

size_t lrs_spectral_patterns_workspace_bytes(int n) { return n >= 1 && n <= 64 ? (size_t)64 * 64 * sizeof(double) : 0; }

int lrs_spectral_patterns_f32(const float* D_dev, int n, int K, const uint64_t* words_dev, int64_t max_count,
                              const int64_t* count_dev, int step, float* a_dev, void* workspace_dev, size_t workspace_bytes,
                              lrs_stream_t stream) {
    const char* fn = "lrs_spectral_patterns_f32";
    if (n < 1 || n > 64 || K <= 0 || max_count < 0) return fail_arg(fn, "need 1 <= n <= 64, K > 0, max_count >= 0");
    if (step != LRS_STEP_SPECTRAL && step != LRS_STEP_FROB4) return fail_arg(fn, "unknown step mode");
    if (!D_dev || (max_count > 0 && (!words_dev || !a_dev))) return fail_arg(fn, "null pointer");
    if (!workspace_dev || workspace_bytes < lrs_spectral_patterns_workspace_bytes(n)) {
        set_error(std::string(fn) + ": workspace smaller than lrs_spectral_patterns_workspace_bytes()");
        return LRS_E_WORKSPACE;
    }
    const int64_t blocks = (max_count + PWARPS * PW - 1) / (PWARPS * PW);
    if (blocks > 0x7fffffffLL) return fail_arg(fn, "max_count too large");
    cudaStream_t st = (cudaStream_t)stream;
    double* G = (double*)workspace_dev;
    ddt64_kernel<<<16, PWARPS * 32, 0, st>>>(D_dev, n, K, G);
    LRS_CHECK_LAUNCH(fn);
    if (blocks == 0) return LRS_OK;
    int rc = check_cuda(fn, cudaFuncSetAttribute(spectral_patterns_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)PATTERN_SMEM));
    if (rc != LRS_OK) return rc;
    spectral_patterns_kernel<<<(unsigned)blocks, PWARPS * 32, PATTERN_SMEM, st>>>(G, n, (const unsigned long long*)words_dev,
                                                                                 max_count, count_dev,
                                                                                 step == LRS_STEP_FROB4, a_dev);
    LRS_CHECK_LAUNCH(fn);
    return LRS_OK;
}

}  // extern "C"
