// Patch geometry, im2col / col2im and the elementwise ADMM kernels (all HBM-bound).
#include <atomic>

#include "common.cuh"

namespace lrs {

static thread_local std::string g_err;

void set_error(const std::string& msg) { g_err = msg; }

int fail_arg(const char* fn, const char* what) {
    g_err = std::string(fn) + ": " + what;
    return LRS_E_ARG;
}

int check_cuda(const char* fn, cudaError_t e) {
    if (e == cudaSuccess) return LRS_OK;
    g_err = std::string(fn) + ": CUDA error: " + cudaGetErrorString(e);
    return LRS_E_CUDA;
}

static std::atomic<unsigned long long> g_launches{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int device_sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    return n;
}

// ------------------------------------------------------------------------------------------------
// x_index / y_index / idx_Mat   (main_LRS_PnP.py:76-99)
// ------------------------------------------------------------------------------------------------
__global__ void patch_index_kernel(Geom g, int64_t* __restrict__ xi, int64_t* __restrict__ yi) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= g.P) return;
    int64_t ci = p / g.row.n, ri = p - ci * g.row.n;
    if (xi) xi[p] = g.row.start(ri);
    if (yi) yi[p] = g.col.start(ci);
}

__global__ void idx_mat_kernel(Geom g, float* __restrict__ m) {
    int64_t nr = g.R - g.bb + 1, nc = g.C - g.bb + 1;
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= nr * nc) return;
    int64_t r = i / nc, c = i - r * nc;
    bool rsel = (r % g.row.s == 0) || (g.row.n > g.row.n_reg && r == g.row.last);
    bool csel = (c % g.col.s == 0) || (g.col.n > g.col.n_reg && c == g.col.last);
    m[i] = (rsel && csel) ? 1.0f : 0.0f;
}

// ------------------------------------------------------------------------------------------------
// im2col: blocks[(i + bb*j)*ld + p] = V[(rs+i)*C + cs + j],  V = X (+ L/mu)
// thread = (patch p, window column j); loops the bb rows.  Writes are coalesced along p.
// Batch: cube b = blockIdx.z reads X, L at b*R*C and writes columns [b*P, (b+1)*P) of blocks [n, ld] (ld = B*P).
// ------------------------------------------------------------------------------------------------
__global__ void im2col_kernel(Geom g, const float* __restrict__ X, const float* __restrict__ L, float mu,
                              float* __restrict__ blocks, int64_t ld) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int j = blockIdx.y;
    if (p >= g.P) return;
    const int64_t cube = (int64_t)blockIdx.z * g.R * g.C;
    X += cube;
    if (L) L += cube;
    blocks += (int64_t)blockIdx.z * g.P;
    int64_t ci, ri;
    if (g.P <= 0x7fffffffLL) {  // 32-bit division on the common sizes
        const unsigned nr = (unsigned)g.row.n, pu = (unsigned)p;
        ci = pu / nr;
        ri = pu - (unsigned)ci * nr;
    } else {
        ci = p / g.row.n;
        ri = p - ci * g.row.n;
    }
    const int64_t rs = g.row.start(ri), cs = g.col.start(ci);
    const int bb = g.bb;
    const float* src = X + rs * g.C + cs + j;
    const float* lsrc = L ? L + rs * g.C + cs + j : nullptr;
    float* dst = blocks + (int64_t)(bb * j) * ld + p;
    for (int i = 0; i < bb; ++i) {
        float v = __ldg(src);
        if (lsrc) {
            v = __fadd_rn(v, __fdiv_rn(__ldg(lsrc), mu));
            lsrc += g.C;
        }
        *dst = v;
        src += g.C;
        dst += ld;
    }
}

// Stride-1 im2col: a block owns 128 consecutive row starts of one column start, stages their (128+bb-1) x bb window
// (plus the multiplier term) in shared memory with row-contiguous loads — 4 cache lines per warp request instead of the
// 32 of the thread-per-patch gather above, which is L1-wavefront bound — and then streams the bb*bb rows of `blocks`
// out, 512 contiguous bytes per row.
template <int IM2COL_TILE>
__global__ void __launch_bounds__(256) im2col_s1_kernel(Geom g, const float* __restrict__ X, const float* __restrict__ L,
                                                        float mu, float* __restrict__ blocks, int64_t ld) {
    extern __shared__ float win[];   // [(TILE + bb - 1)][bb + 1]
    const int64_t cube = (int64_t)blockIdx.z * g.R * g.C;    // batch: as im2col_kernel
    X += cube;
    if (L) L += cube;
    blocks += (int64_t)blockIdx.z * g.P;
    const int bb = g.bb, wld = bb + 1;
    const int64_t ri0 = blockIdx.x * (int64_t)IM2COL_TILE, ci = blockIdx.y;
    const int64_t nR = g.row.n;
    const int np = (int)(nR - ri0 < IM2COL_TILE ? nR - ri0 : IM2COL_TILE);   // patches of this tile
    const int wrows = np + bb - 1;
    for (int e = threadIdx.x; e < wrows * bb; e += blockDim.x) {
        const int wr = e / bb, wc = e - wr * bb;
        const int64_t src = (ri0 + wr) * g.C + ci + wc;
        float v = __ldg(X + src);
        if (L) v = __fadd_rn(v, __fdiv_rn(__ldg(L + src), mu));
        win[wr * wld + wc] = v;
    }
    __syncthreads();
    const int m = threadIdx.x % IM2COL_TILE, h = threadIdx.x / IM2COL_TILE, nh = blockDim.x / IM2COL_TILE;
    if (m >= np) return;
    float* dst = blocks + ci * nR + ri0 + m;
    for (int j = 0; j < bb; ++j) {                               // element k = i + bb*j = row i, column j of the patch
        float* d = dst + (int64_t)(bb * j + h) * ld;
        const float* w = win + (m + h) * wld + j;
        for (int i = h; i < bb; i += nh) {
            __stcs(d, *w);                                       // written once, read by a later kernel: stream it
            d += nh * ld;
            w += nh * wld;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// col2im: deterministic gather.  Each output element sums its covering patches in ascending patch
// order (column start outer, row start inner) with plain fp32 adds — the order of the sequential
// loop at main_LRS_PnP.py:332-339, so the result is bit-identical to it.
// 32x32 tile, threads run along r while gathering (coalesced along p), transposed through shared
// memory so the store runs along c.
// ------------------------------------------------------------------------------------------------
// Sum, in ascending row-start order, of the regular row starts [rlo, rhi] (+ the appended last start) of one column
// start.  `pc` points at blocks[(bb*j)*ld + ci*nR] (ld = leading dimension of blocks); consecutive row starts are one
// pointer step apart, so the walk costs an add per load (the kernel is instruction-issue bound otherwise: measured 56
// instructions per load).
__device__ __forceinline__ float col2im_column(const Geom& g, int64_t ld, const float* __restrict__ pc, int64_t r, int64_t rlo,
                                               int64_t nreg, bool rapp, float sum) {
    const int64_t step = 1 - (int64_t)g.row.s * ld;
    const float* pr = pc + (r - rlo * g.row.s) * ld + rlo;
    int64_t b = 0;
    for (; b + 8 <= nreg; b += 8) {  // 8 independent loads in flight, then the adds in patch order
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = __ldg(pr + u * step);
#pragma unroll
        for (int u = 0; u < 8; ++u) sum = __fadd_rn(sum, v[u]);
        pr += 8 * step;
    }
    for (; b < nreg; ++b) {
        sum = __fadd_rn(sum, __ldg(pr));
        pr += step;
    }
    if (rapp) sum = __fadd_rn(sum, __ldg(pc + (r - g.row.last) * ld + g.row.n_reg));
    return sum;
}

// Stride-1 specialisation (the dense-overlap geometry of cfg 4/5): no appended starts, no divisions, and for interior
// rows the BB row starts of a column start are BB loads at compile-time multiples of one pointer step — about four
// instructions per load instead of the generic path's 28 (ncu), which is what makes the kernel HBM-bound.
//
// Column-start RANGE mode: `blocks` holds only the patches of column starts [ci_begin, ci_end) (P = (ci_end - ci_begin) * nR
// columns), and every output element covered by them CONTINUES its running fp32 sum from `out` — or starts it from 0 when
// the range contains its first covering column start.  Patch order is column-start-outer, so feeding the ranges in
// ascending order reproduces the association of the sequential loop (main_LRS_PnP.py:332-339) bit for bit while only one
// range of Phi_z exists at a time.  Only output columns [ci_begin, ci_end + BB - 1) are touched.
// Batch (whole range only): cube b = blockIdx.z sums columns [b*P, (b+1)*P) of blocks [n, ld] into out + b*R*C.
template <int BB, int JU, int MINB>
__global__ void __launch_bounds__(256, MINB) col2im_s1_kernel(Geom g, const float* __restrict__ blocks, int64_t ld,
                                                              float* __restrict__ out, int64_t ci_begin, int64_t ci_end) {
    __shared__ float tile[32][33];
    const int64_t r0 = blockIdx.x * 32LL, c0 = ci_begin + blockIdx.y * 32LL;
    const int tx = threadIdx.x, ty = threadIdx.y;  // blockDim = (32, 8)
    const int64_t nR = g.row.n, nC = g.col.n;
    blocks += (int64_t)blockIdx.z * (ci_end - ci_begin) * nR;
    out += (int64_t)blockIdx.z * g.R * g.C;
    const int64_t step = 1 - ld, cstep = nR - (int64_t)BB * ld;
    const int64_t c_end = ci_end + BB - 1 < g.C ? ci_end + BB - 1 : g.C;   // one past the last output column touched
    for (int cc = ty; cc < 32; cc += 8) {
        const int64_t r = r0 + tx, c = c0 + cc;
        float sum = 0.0f;
        if (r < g.R && c < c_end) {
            const int64_t rlo = r - (BB - 1) > 0 ? r - (BB - 1) : 0, rhi = r < nR - 1 ? r : nR - 1;
            const int64_t clo_all = c - (BB - 1) > 0 ? c - (BB - 1) : 0, chi_all = c < nC - 1 ? c : nC - 1;
            const int64_t clo = clo_all > ci_begin ? clo_all : ci_begin, chi = chi_all < ci_end - 1 ? chi_all : ci_end - 1;
            const int nreg = (int)(rhi - rlo + 1), ncol = (int)(chi - clo + 1);
            if (clo > clo_all) sum = out[r * g.C + c];        // earlier ranges already added this element's first patches
            const float* pc = blocks + ((r - rlo) + (int64_t)BB * (c - clo)) * ld + (clo - ci_begin) * nR + rlo;
            if (nreg == BB) {
                int j = 0;
                for (; j + JU <= ncol; j += JU) {   // JU column starts = JU*BB independent loads in flight
                    float v[JU][BB];
#pragma unroll
                    for (int w = 0; w < JU; ++w)
#pragma unroll
                        for (int u = 0; u < BB; ++u) v[w][u] = __ldg(pc + w * cstep + u * step);
#pragma unroll
                    for (int w = 0; w < JU; ++w)
#pragma unroll
                        for (int u = 0; u < BB; ++u) sum = __fadd_rn(sum, v[w][u]);
                    pc += JU * cstep;
                }
                for (; j < ncol; ++j) {
                    float v[BB];
#pragma unroll
                    for (int u = 0; u < BB; ++u) v[u] = __ldg(pc + u * step);
#pragma unroll
                    for (int u = 0; u < BB; ++u) sum = __fadd_rn(sum, v[u]);
                    pc += cstep;
                }
            } else {
                for (int j = 0; j < ncol; ++j) {
                    const float* pr = pc;
                    for (int u = 0; u < nreg; ++u) {
                        sum = __fadd_rn(sum, __ldg(pr));
                        pr += step;
                    }
                    pc += cstep;
                }
            }
        }
        tile[cc][tx] = sum;
    }
    __syncthreads();
    for (int rr = ty; rr < 32; rr += 8) {
        const int64_t r = r0 + rr, c = c0 + tx;
        if (r < g.R && c < c_end) out[r * g.C + c] = tile[tx][rr];
    }
}

template <int TR, int TC, int TY>
__global__ void __launch_bounds__(TR * TY, 1536 / (TR * TY)) col2im_kernel(Geom g, const float* __restrict__ blocks, int64_t ld,
                                                                           float* __restrict__ out) {
    __shared__ float tile[TC][TR + 1];
    int64_t r0 = blockIdx.x * (int64_t)TR, c0 = blockIdx.y * (int64_t)TC;
    blocks += (int64_t)blockIdx.z * g.P;                   // batch: as col2im_s1_kernel
    out += (int64_t)blockIdx.z * g.R * g.C;
    int tx = threadIdx.x, ty = threadIdx.y;  // blockDim = (TR, TY)
    for (int cc = ty; cc < TC; cc += TY) {
        int64_t r = r0 + tx, c = c0 + cc;
        float sum = 0.0f;
        if (r < g.R && c < g.C) {
            int64_t rlo, rhi, clo, chi;
            bool rapp, capp;
            g.row.cover(r, rlo, rhi, rapp);
            g.col.cover(c, clo, chi, capp);
            const int64_t nreg = rhi - rlo + 1 > 0 ? rhi - rlo + 1 : 0;
            // regular column starts ci = clo..chi: j = c - ci*s; next ci: j -= s
            const float* pc = blocks + ((int64_t)g.bb * (c - clo * g.col.s)) * ld + clo * g.row.n;
            const int64_t cstep = g.row.n - (int64_t)g.bb * g.col.s * ld;
            for (int64_t ci = clo; ci <= chi; ++ci) {
                sum = col2im_column(g, ld, pc, r, rlo, nreg, rapp, sum);
                pc += cstep;
            }
            if (capp)
                sum = col2im_column(g, ld, blocks + ((int64_t)g.bb * (c - g.col.last)) * ld + g.col.n_reg * g.row.n, r, rlo,
                                    nreg, rapp, sum);
        }
        tile[cc][tx] = sum;
    }
    __syncthreads();
    for (int idx = ty * TR + tx; idx < TR * TC; idx += TR * TY) {
        const int rr = idx / TC, cc = idx % TC;
        int64_t r = r0 + rr, c = c0 + cc;
        if (r < g.R && c < g.C) out[r * g.C + c] = tile[cc][rr];
    }
}

constexpr int WEIGHT_ROWS = 32;     // unfolded rows per block (a block per row is launch-overhead bound: 21 % of the HBM peak)
__global__ void weight_kernel(Geom g, float* __restrict__ w) {
    const int64_t r0 = (int64_t)blockIdx.x * WEIGHT_ROWS;
    const int64_t c = blockIdx.y * (int64_t)blockDim.x + threadIdx.x;    // bands along the threads
    if (c >= g.C) return;
    const int wc = g.col.count(c);
    const int64_t r1 = r0 + WEIGHT_ROWS < g.R ? r0 + WEIGHT_ROWS : g.R;
    for (int64_t r = r0; r < r1; ++r) w[r * g.C + c] = (float)(g.row.count(r) * wc);
}

// ------------------------------------------------------------------------------------------------
// elementwise
// ------------------------------------------------------------------------------------------------
__global__ void soft_kernel(const float* __restrict__ x, float tau, float* __restrict__ out, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = soft_thr(x[i], tau);
}

__global__ void soft_kernel_v4(const float4* __restrict__ x, float tau, float4* __restrict__ out, int64_t n4) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n4; i += stride) {
        float4 v = x[i];
        v.x = soft_thr(v.x, tau);
        v.y = soft_thr(v.y, tau);
        v.z = soft_thr(v.z, tau);
        v.w = soft_thr(v.w, tau);
        out[i] = v;
    }
}

__global__ void axpy_kernel(const float* __restrict__ x, const float* __restrict__ l, float c,
                            float* __restrict__ out, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) out[i] = __fadd_rn(x[i], __fmul_rn(c, l[i]));
}

__global__ void step_frob4_kernel(const float* __restrict__ bc, const float* __restrict__ D, int n, int K, int64_t P,
                                  float* __restrict__ a) {
    extern __shared__ float rn[];  // ||D[i,:]||^2
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float s = 0.f;
        for (int k = 0; k < K; ++k) {
            float d = D[(int64_t)i * K + k];
            s = fmaf(d, d, s);
        }
        rn[i] = s;
    }
    __syncthreads();
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= P) return;
    float s = 0.f;
    for (int i = 0; i < n; ++i)
        if (bc[(int64_t)i * P + p] != 0.0f) s += rn[i];
    a[p] = 4.0f * s;
}

// X / multiplier update, main_LRS_PnP.py:346,361-362 — same fp32 operation order, no FMA contraction.
// A thread owns one band of ADMM_RPT consecutive unfolded rows: its 6 x ADMM_RPT loads are issued together and the
// ADMM_RPT chains of dependent adds of lambda1_summation (:343, one add per covering patch, up to bb^2 = 64 at stride 1)
// run interleaved, so the add latency of one element hides behind the others'.
constexpr int ADMM_RPT = 4;
__global__ void admm_update_kernel(Geom g, const float* __restrict__ Y, const float* __restrict__ M,
                                   const float* __restrict__ IM, const float* __restrict__ U, float* __restrict__ lam1,
                                   float* __restrict__ lam2, float* __restrict__ Xo, float gamma, float mu1, float mu2,
                                   int64_t rows, int64_t row_offset) {
    const int64_t r0 = (int64_t)blockIdx.x * ADMM_RPT;                   // ADMM_RPT unfolded rows per block row
    const int64_t c = blockIdx.y * (int64_t)blockDim.x + threadIdx.x;    // bands along the threads (coalesced)
    if (c >= g.C) return;
    const int64_t cube = (int64_t)blockIdx.z * rows * g.C;               // batch: cube b = blockIdx.z, geometry shared
    Y += cube;
    M += cube;
    IM += cube;
    U += cube;
    lam1 += cube;
    lam2 += cube;
    Xo += cube;
    const int wc = g.col.count(c);
    float l1[ADMM_RPT], l2[ADMM_RPT], im[ADMM_RPT], u[ADMM_RPT], y[ADMM_RPT], m[ADMM_RPT], l1s[ADMM_RPT];
    int W[ADMM_RPT], wmax = 0;
#pragma unroll
    for (int k = 0; k < ADMM_RPT; ++k) {
        const bool ok = r0 + k < rows;
        const int64_t idx = (ok ? r0 + k : r0) * g.C + c;
        W[k] = ok ? g.row.count(r0 + k + row_offset) * wc : 0;
        wmax = W[k] > wmax ? W[k] : wmax;
        l1[k] = lam1[idx];
        l2[k] = lam2[idx];
        im[k] = __ldg(IM + idx);
        u[k] = __ldg(U + idx);
        y[k] = __ldg(Y + idx);
        m[k] = __ldg(M + idx);
        l1s[k] = 0.0f;
    }
    bool uniform = true;
#pragma unroll
    for (int k = 0; k < ADMM_RPT; ++k) uniform = uniform && W[k] == wmax;
    if (uniform) {               // interior rows: every element is covered equally often — no per-add predicate
#pragma unroll 8
        for (int t = 0; t < wmax; ++t) {
#pragma unroll
            for (int k = 0; k < ADMM_RPT; ++k) l1s[k] = __fadd_rn(l1s[k], l1[k]);  // lambda1_summation (:343)
        }
    } else {
        for (int t = 0; t < wmax; ++t) {
#pragma unroll
            for (int k = 0; k < ADMM_RPT; ++k)
                if (t < W[k]) l1s[k] = __fadd_rn(l1s[k], l1[k]);  // one add per covering patch
        }
    }
#pragma unroll
    for (int k = 0; k < ADMM_RPT; ++k) {
        if (r0 + k >= rows) break;
        const int64_t idx = (r0 + k) * g.C + c;
        float num = __fadd_rn(__fmul_rn(gamma, y[k]), __fmul_rn(mu1, im[k]));
        num = __fadd_rn(num, __fmul_rn(mu2, u[k]));
        num = __fsub_rn(num, l1s[k]);
        num = __fsub_rn(num, l2[k]);
        const float den = __fadd_rn(__fadd_rn(__fmul_rn(gamma, m[k]), __fmul_rn(mu1, (float)W[k])), mu2);
        const float x = __fdiv_rn(num, den);
        Xo[idx] = x;
        lam1[idx] = __fadd_rn(l1[k], __fmul_rn(mu1, __fsub_rn(x, im[k])));
        lam2[idx] = __fadd_rn(l2[k], __fmul_rn(mu2, __fsub_rn(x, u[k])));
    }
}

static inline unsigned blocks_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

// Launchers shared by the single-cube entry points (B = 1) and their batched forms: B cubes of one geometry, [B, R, C]
// contiguous, cube b in grid z.
static int im2col_launch(const char* fn, const float* X_dev, const float* L_dev, float mu, int64_t B, int64_t R, int64_t C,
                         int bb, int s, float* blocks_dev, cudaStream_t st) {
    Geom g;
    if (!make_geom(R, C, bb, s, g)) return fail_arg(fn, "need 0 < bb <= min(R,C) and s > 0");
    if (B < 1 || B > LRS_MAX_BATCH) return fail_arg(fn, "need 1 <= B <= LRS_MAX_BATCH");
    if (!X_dev || !blocks_dev) return fail_arg(fn, "null pointer");
    if (L_dev && mu == 0.0f) return fail_arg(fn, "mu must be non-zero");
    // 256 row starts per block: measured 4.2-4.5 TB/s at cfg 4 (128: 3.9-4.3, 64: 3.3-3.5; thread-per-patch gather: 2.2)
    constexpr int tile = 256;
    const size_t win_bytes = (size_t)(tile + bb - 1) * (bb + 1) * sizeof(float);
    const int64_t ld = B * g.P;
    if (s == 1 && win_bytes <= 48 * 1024 && g.col.n <= 65535) {
        im2col_s1_kernel<tile><<<dim3(blocks_for(g.row.n, tile), (unsigned)g.col.n, (unsigned)B), 256, win_bytes, st>>>(
            g, X_dev, L_dev, mu, blocks_dev, ld);
    } else {
        dim3 grid(blocks_for(g.P, 128), bb, (unsigned)B);
        im2col_kernel<<<grid, 128, 0, st>>>(g, X_dev, L_dev, mu, blocks_dev, ld);
    }
    LRS_CHECK_LAUNCH(fn);
    return LRS_OK;
}

static int col2im_launch(const char* fn, const float* blocks_dev, int64_t B, int64_t R, int64_t C, int bb, int s,
                         float* imout_dev, cudaStream_t st) {
    Geom g;
    if (!make_geom(R, C, bb, s, g)) return fail_arg(fn, "need 0 < bb <= min(R,C) and s > 0");
    if (B < 1 || B > LRS_MAX_BATCH) return fail_arg(fn, "need 1 <= B <= LRS_MAX_BATCH");
    if (!blocks_dev || !imout_dev) return fail_arg(fn, "null pointer");
    dim3 grid(blocks_for(R, 32), blocks_for(C, 32), (unsigned)B);
    if (grid.y > 65535) return fail_arg(fn, "C too large");
    const int64_t ld = B * g.P;
    // measured at cfg 4 (B200): generic kernel 3.9 ms; stride-1 kernel 2.2-2.6 ms; two or four column starts in flight
    // per thread, 8 blocks/SM with 32 registers, or longer row tiles (128x8, 256x4) are all slower
    if (s == 1 && bb == 8)
        col2im_s1_kernel<8, 1, 6><<<grid, dim3(32, 8), 0, st>>>(g, blocks_dev, ld, imout_dev, 0, g.col.n);
    else col2im_kernel<32, 32, 8><<<grid, dim3(32, 8), 0, st>>>(g, blocks_dev, ld, imout_dev);
    LRS_CHECK_LAUNCH(fn);
    return LRS_OK;
}

static int admm_update_launch(const char* fn, const float* Y_dev, const float* MtM_dev, const float* imout_dev,
                              const float* U_dev, float* lam1_dev, float* lam2_dev, float* X_out_dev, float gamma, float mu_1,
                              float mu_2, int64_t B, int64_t rows, int64_t row_offset, int64_t R_total, int64_t C, int bb, int s,
                              cudaStream_t st) {
    Geom g;
    if (!make_geom(R_total, C, bb, s, g)) return fail_arg(fn, "need 0 < bb <= min(R,C) and s > 0");
    if (B < 1 || B > LRS_MAX_BATCH) return fail_arg(fn, "need 1 <= B <= LRS_MAX_BATCH");
    if (rows < 0 || row_offset < 0 || row_offset + rows > R_total) return fail_arg(fn, "row stripe outside the matrix");
    if (rows == 0) return LRS_OK;
    if (!Y_dev || !MtM_dev || !imout_dev || !U_dev || !lam1_dev || !lam2_dev || !X_out_dev) return fail_arg(fn, "null pointer");
    const int threads = C >= 256 ? 256 : (int)((C + 31) / 32 * 32);
    dim3 grid((unsigned)((rows + ADMM_RPT - 1) / ADMM_RPT), blocks_for(C, threads), (unsigned)B);
    if (rows > 2147483647LL || grid.y > 65535) return fail_arg(fn, "matrix too large");
    admm_update_kernel<<<grid, threads, 0, st>>>(g, Y_dev, MtM_dev, imout_dev, U_dev, lam1_dev, lam2_dev, X_out_dev, gamma, mu_1,
                                                 mu_2, rows, row_offset);
    LRS_CHECK_LAUNCH(fn);
    return LRS_OK;
}

}  // namespace lrs

using namespace lrs;

extern "C" {

const char* lrs_last_error(void) { return lrs::g_err.c_str(); }

int lrs_version(void) { return 103; }

uint64_t lrs_launch_count(void) { return (uint64_t)lrs::g_launches.load(); }

int64_t lrs_axis_count(int64_t length, int bb, int s) {
    Axis a;
    if (!make_axis(length, bb, s, a)) return -1;
    return a.n;
}

int lrs_axis_starts(int64_t length, int bb, int s, int64_t* starts_out, int64_t count) {
    Axis a;
    if (!make_axis(length, bb, s, a)) return fail_arg("lrs_axis_starts", "need 0 < bb <= length and s > 0");
    if (count != a.n || !starts_out) return fail_arg("lrs_axis_starts", "count does not match lrs_axis_count");
    for (int64_t i = 0; i < a.n; ++i) starts_out[i] = a.start(i);
    return LRS_OK;
}

int lrs_patch_index_i64(int64_t R, int64_t C, int bb, int s, int64_t* x_index_dev, int64_t* y_index_dev,
                        float* idx_mat_dev, lrs_stream_t stream) {
    Geom g;
    if (!make_geom(R, C, bb, s, g)) return fail_arg("lrs_patch_index_i64", "need 0 < bb <= min(R,C) and s > 0");
    cudaStream_t st = (cudaStream_t)stream;
    if (x_index_dev || y_index_dev) {
        patch_index_kernel<<<blocks_for(g.P, 256), 256, 0, st>>>(g, x_index_dev, y_index_dev);
        LRS_CHECK_LAUNCH("lrs_patch_index_i64");
    }
    if (idx_mat_dev) {
        int64_t tot = (R - bb + 1) * (C - bb + 1);
        idx_mat_kernel<<<blocks_for(tot, 256), 256, 0, st>>>(g, idx_mat_dev);
        LRS_CHECK_LAUNCH("lrs_patch_index_i64");
    }
    return LRS_OK;
}

int lrs_im2col_f32(const float* X_dev, const float* L_dev, float mu, int64_t R, int64_t C, int bb, int s,
                   float* blocks_dev, lrs_stream_t stream) {
    return im2col_launch("lrs_im2col_f32", X_dev, L_dev, mu, 1, R, C, bb, s, blocks_dev, (cudaStream_t)stream);
}

int lrs_im2col_batch_f32(const float* X_dev, const float* L_dev, float mu, int64_t B, int64_t R, int64_t C, int bb, int s,
                         float* blocks_dev, lrs_stream_t stream) {
    return im2col_launch("lrs_im2col_batch_f32", X_dev, L_dev, mu, B, R, C, bb, s, blocks_dev, (cudaStream_t)stream);
}

int lrs_col2im_accum_f32(const float* blocks_dev, int64_t R, int64_t C, int bb, int s, float* imout_dev,
                         lrs_stream_t stream) {
    return col2im_launch("lrs_col2im_accum_f32", blocks_dev, 1, R, C, bb, s, imout_dev, (cudaStream_t)stream);
}

int lrs_col2im_accum_batch_f32(const float* blocks_dev, int64_t B, int64_t R, int64_t C, int bb, int s, float* imout_dev,
                               lrs_stream_t stream) {
    return col2im_launch("lrs_col2im_accum_batch_f32", blocks_dev, B, R, C, bb, s, imout_dev, (cudaStream_t)stream);
}

int lrs_col2im_accum_range_f32(const float* blocks_dev, int64_t R, int64_t C, int bb, int s, int64_t ci_begin, int64_t ci_end,
                               float* imout_dev, lrs_stream_t stream) {
    const char* fn = "lrs_col2im_accum_range_f32";
    Geom g;
    if (!make_geom(R, C, bb, s, g)) return fail_arg(fn, "need 0 < bb <= min(R,C) and s > 0");
    if (s != 1 || bb != 8) return fail_arg(fn, "column-start ranges are implemented for bb = 8, stride 1 (the dense-overlap geometry)");
    if (!blocks_dev || !imout_dev) return fail_arg(fn, "null pointer");
    if (ci_begin < 0 || ci_end > g.col.n || ci_begin >= ci_end) return fail_arg(fn, "need 0 <= ci_begin < ci_end <= column starts");
    const int64_t c_end = ci_end + bb - 1 < C ? ci_end + bb - 1 : C;
    dim3 grid(blocks_for(R, 32), blocks_for(c_end - ci_begin, 32));
    if (grid.y > 65535) return fail_arg(fn, "C too large");
    col2im_s1_kernel<8, 1, 6><<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(g, blocks_dev, (ci_end - ci_begin) * g.row.n,
                                                                              imout_dev, ci_begin, ci_end);
    LRS_CHECK_LAUNCH(fn);
    return LRS_OK;
}

int lrs_coverage_weight_f32(int64_t R, int64_t C, int bb, int s, float* weight_dev, lrs_stream_t stream) {
    Geom g;
    if (!make_geom(R, C, bb, s, g)) return fail_arg("lrs_coverage_weight_f32", "need 0 < bb <= min(R,C) and s > 0");
    if (!weight_dev) return fail_arg("lrs_coverage_weight_f32", "null pointer");
    const int threads = C >= 256 ? 256 : (int)((C + 31) / 32 * 32);
    dim3 grid(blocks_for(R, WEIGHT_ROWS), blocks_for(C, threads));
    if (R > 2147483647LL || grid.y > 65535) return fail_arg("lrs_coverage_weight_f32", "matrix too large");
    weight_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(g, weight_dev);
    LRS_CHECK_LAUNCH("lrs_coverage_weight_f32");
    return LRS_OK;
}

int lrs_soft_f32(const float* x_dev, float tau, float* out_dev, int64_t count, lrs_stream_t stream) {
    if (count < 0 || (count > 0 && (!x_dev || !out_dev))) return fail_arg("lrs_soft_f32", "bad arguments");
    if (count == 0) return LRS_OK;
    int sms = device_sm_count();
    if (sms <= 0) return check_cuda("lrs_soft_f32", cudaErrorNoDevice);
    cudaStream_t st = (cudaStream_t)stream;
    bool v4 = ((uintptr_t)x_dev % 16 == 0) && ((uintptr_t)out_dev % 16 == 0) && (count % 4 == 0);
    if (v4) {
        int64_t n4 = count / 4;
        unsigned grid = (unsigned)std::min<int64_t>((n4 + 255) / 256, (int64_t)sms * 16);
        soft_kernel_v4<<<grid, 256, 0, st>>>((const float4*)x_dev, tau, (float4*)out_dev, n4);
    } else {
        unsigned grid = (unsigned)std::min<int64_t>((count + 255) / 256, (int64_t)sms * 16);
        soft_kernel<<<grid, 256, 0, st>>>(x_dev, tau, out_dev, count);
    }
    LRS_CHECK_LAUNCH("lrs_soft_f32");
    return LRS_OK;
}

int lrs_axpy_f32(const float* x_dev, const float* l_dev, float c, float* out_dev, int64_t count, lrs_stream_t stream) {
    if (count < 0 || (count > 0 && (!x_dev || !l_dev || !out_dev))) return fail_arg("lrs_axpy_f32", "bad arguments");
    if (count == 0) return LRS_OK;
    int sms = device_sm_count();
    if (sms <= 0) return check_cuda("lrs_axpy_f32", cudaErrorNoDevice);
    unsigned grid = (unsigned)std::min<int64_t>((count + 255) / 256, (int64_t)sms * 16);
    axpy_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x_dev, l_dev, c, out_dev, count);
    LRS_CHECK_LAUNCH("lrs_axpy_f32");
    return LRS_OK;
}

int lrs_step_frob4_f32(const float* blocks_copy_dev, const float* D_dev, int n, int K, int64_t P, float* a_dev,
                       lrs_stream_t stream) {
    if (n <= 0 || K <= 0 || P < 0 || !blocks_copy_dev || !D_dev || !a_dev)
        return fail_arg("lrs_step_frob4_f32", "bad arguments");
    if (P == 0) return LRS_OK;
    if ((size_t)n * sizeof(float) > 48 * 1024) return fail_arg("lrs_step_frob4_f32", "n too large");
    step_frob4_kernel<<<blocks_for(P, 128), 128, n * sizeof(float), (cudaStream_t)stream>>>(blocks_copy_dev, D_dev, n, K,
                                                                                         P, a_dev);
    LRS_CHECK_LAUNCH("lrs_step_frob4_f32");
    return LRS_OK;
}

int lrs_admm_update_f32(const float* Y_dev, const float* MtM_dev, const float* imout_dev, const float* U_dev,
                        float* lam1_dev, float* lam2_dev, float* X_out_dev, float gamma, float mu_1, float mu_2,
                        int64_t rows, int64_t row_offset, int64_t R_total, int64_t C, int bb, int s,
                        lrs_stream_t stream) {
    return admm_update_launch("lrs_admm_update_f32", Y_dev, MtM_dev, imout_dev, U_dev, lam1_dev, lam2_dev, X_out_dev, gamma,
                              mu_1, mu_2, 1, rows, row_offset, R_total, C, bb, s, (cudaStream_t)stream);
}

int lrs_admm_update_batch_f32(const float* Y_dev, const float* MtM_dev, const float* imout_dev, const float* U_dev,
                              float* lam1_dev, float* lam2_dev, float* X_out_dev, float gamma, float mu_1, float mu_2, int64_t B,
                              int64_t R, int64_t C, int bb, int s, lrs_stream_t stream) {
    return admm_update_launch("lrs_admm_update_batch_f32", Y_dev, MtM_dev, imout_dev, U_dev, lam1_dev, lam2_dev, X_out_dev,
                              gamma, mu_1, mu_2, B, R, 0, R, C, bb, s, (cudaStream_t)stream);
}

}  // extern "C"
