// Batched soft-ISTA on explicit patch matrices, any (n, K, P): two fp32 GEMM launches per
// iteration with the mask / residual / step / soft-threshold fused into the epilogues.
// This is the shape-generic engine (bundled configs: n = 1296, P = 144); the n = 64 stride-1 regime
// goes through sparse_fused_*.cu instead.
//
//   residual:  Rm[n,P] = m .* (Y - D A) * inv_a[p]          (A-operand D [n,K] row-major)
//   gradient:  A[K,P]  = soft(A + D^T Rm, T[p])             (A-operand D^T, read from D)
//   output:    Phi[n,P] = D A                               (full dictionary, main_LRS_PnP.py:294)
#include "common.cuh"

namespace lrs {

constexpr int BM = 64, BN = 64, BK = 16, TM = 4, TN = 4;

struct EpiResidual {
    __device__ __forceinline__ void slice(int64_t) {}  // c = D A  ->  Rm
    const float* Y;
    const float* BC;
    const float* inv_a;
    float* out;
    __device__ __forceinline__ void operator()(int64_t m, int64_t p, int64_t ld, float acc) const {
        int64_t o = m * ld + p;
        float v = (BC[o] != 0.0f) ? (Y[o] - acc) * inv_a[p] : 0.0f;
        out[o] = v;
    }
};
struct EpiGradient {
    __device__ __forceinline__ void slice(int64_t) {}  // c = D^T Rm  ->  A = soft(A + c, T)
    const float* T;
    float* A;
    __device__ __forceinline__ void operator()(int64_t m, int64_t p, int64_t ld, float acc) const {
        int64_t o = m * ld + p;
        A[o] = soft_thr(A[o] + acc, T[p]);
    }
};
struct EpiGradientPlain {
    __device__ __forceinline__ void slice(int64_t) {}  // c = D^T Rm  ->  G = A + c   (input of a plug-and-play denoiser; identity when G == A buffer)
    const float* A;
    float* G;
    __device__ __forceinline__ void operator()(int64_t m, int64_t p, int64_t ld, float acc) const {
        int64_t o = m * ld + p;
        G[o] = A[o] + acc;
    }
};
struct EpiStore {
    __device__ __forceinline__ void slice(int64_t) {}
    __device__ __forceinline__ void cube(int64_t off) { out += off; }     // batch of sgemm_kernel
    float* out;
    __device__ __forceinline__ void operator()(int64_t m, int64_t p, int64_t ld, float acc) const { out[m * ld + p] = acc; }
};
struct EpiPartial {  // split-K: raw partial sums into slice z of a [splits, M, N] buffer
    float* buf;
    __device__ __forceinline__ void slice(int64_t off) { buf += off; }
    __device__ __forceinline__ void operator()(int64_t m, int64_t p, int64_t ld, float acc) const { buf[m * ld + p] = acc; }
};
struct LoadPlain {
    const float* B;
    __device__ __forceinline__ float operator()(int64_t o) const { return __ldg(B + o); }
};
struct LoadAxpy {  // Z = X + c*L on the fly (SVT input, main_LRS_PnP.py:315)
    const float* X;
    const float* L;
    float c;
    __device__ __forceinline__ void cube(int64_t off) {
        X += off;
        if (L) L += off;
    }
    __device__ __forceinline__ float operator()(int64_t o) const {
        float v = __ldg(X + o);
        if (L) v = __fadd_rn(v, __fmul_rn(c, __ldg(L + o)));
        return v;
    }
};

// C[M,N] = op(A)[M,Kd] * B[Kd,N];  A stored row-major [M,Kd] (TRANS_A=false) or [Kd,M] (true).
// Batch: grid.z = problem z, A and C shifted by z * ac_stride, B by z * b_stride.
template <bool TRANS_A, class ALoad, class Epi>
__global__ void __launch_bounds__(256) sgemm_kernel(ALoad aload, const float* __restrict__ B, int64_t M, int64_t N,
                                                    int64_t Kd, Epi epi, int64_t ac_stride, int64_t b_stride) {
    aload.cube((int64_t)blockIdx.z * ac_stride);
    epi.cube((int64_t)blockIdx.z * ac_stride);
    B += (int64_t)blockIdx.z * b_stride;
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid % 16, ty = tid / 16;
    const int64_t m0 = blockIdx.y * (int64_t)BM, n0 = blockIdx.x * (int64_t)BN;
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    for (int64_t k0 = 0; k0 < Kd; k0 += BK) {
        // A tile -> As[k][m]
        if (TRANS_A) {
#pragma unroll
            for (int e = tid; e < BK * BM; e += 256) {
                int k = e / BM, m = e % BM;
                int64_t gk = k0 + k, gm = m0 + m;
                As[k][m] = (gk < Kd && gm < M) ? aload(gk * M + gm) : 0.f;
            }
        } else {
#pragma unroll
            for (int e = tid; e < BK * BM; e += 256) {
                int m = e / BK, k = e % BK;
                int64_t gk = k0 + k, gm = m0 + m;
                As[k][m] = (gk < Kd && gm < M) ? aload(gm * Kd + gk) : 0.f;
            }
        }
#pragma unroll
        for (int e = tid; e < BK * BN; e += 256) {
            int k = e / BN, n = e % BN;
            int64_t gk = k0 + k, gn = n0 + n;
            Bs[k][n] = (gk < Kd && gn < N) ? __ldg(B + gk * N + gn) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; ++i) a[i] = As[k][ty * TM + i];
#pragma unroll
            for (int j = 0; j < TN; ++j) b[j] = Bs[k][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        int64_t gm = m0 + ty * TM + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            int64_t gn = n0 + tx * TN + j;
            if (gn < N) epi(gm, gn, N, acc[i][j]);
        }
    }
}

// Software-pipelined variant for the ISTA GEMMs (plain pointer A operand): 48-column tiles (P = 144 = 3 x 48 on the
// bundled configs, no padded columns), BMv = 32 or 64 rows so that the tall-skinny problems fill the SMs, double-buffered
// shared memory with the next k-tile prefetched into registers while the current one is multiplied.
template <bool TRANS_A, class Epi, int BMv>
__global__ void __launch_bounds__(192) sgemm_pipe_kernel(const float* __restrict__ A, const float* __restrict__ B, int64_t M,
                                                         int64_t N, int64_t Kd, int64_t kchunk, Epi epi_in) {
    // split-K: block z multiplies k in [z*kchunk, (z+1)*kchunk) and hands its partial sums to slice z of the epilogue
    const int64_t kbeg = blockIdx.z * kchunk, kend = kbeg + kchunk < Kd ? kbeg + kchunk : Kd;
    Epi epi = epi_in;
    epi.slice((int64_t)blockIdx.z * M * N);
    constexpr int BNv = 48, TMv = BMv / 16, NT = 192;
    constexpr int NA = (BK * BMv + NT - 1) / NT, NB = BK * BNv / NT;
    __shared__ __align__(16) float As[2][BK][BMv + 4];
    __shared__ __align__(16) float Bs[2][BK][BNv + 4];
    const int tid = threadIdx.x, tx = tid % 12, ty = tid / 12;
    const int64_t m0 = blockIdx.y * (int64_t)BMv, n0 = blockIdx.x * (int64_t)BNv;
    float acc[TMv][4];
#pragma unroll
    for (int i = 0; i < TMv; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float ra[NA], rb[NB];

    auto gload = [&](int64_t k0) {
#pragma unroll
        for (int u = 0; u < NA; ++u) {
            const int e = tid + u * NT;
            float v = 0.f;
            if (e < BK * BMv) {
                const int k = TRANS_A ? e / BMv : e % BK, m = TRANS_A ? e % BMv : e / BK;
                const int64_t gk = k0 + k, gm = m0 + m;
                if (gk < kend && gm < M) v = __ldg(A + (TRANS_A ? gk * M + gm : gm * Kd + gk));
            }
            ra[u] = v;
        }
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            const int e = tid + u * NT, k = e / BNv, n = e % BNv;
            const int64_t gk = k0 + k, gn = n0 + n;
            rb[u] = (gk < kend && gn < N) ? __ldg(B + gk * N + gn) : 0.f;
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int u = 0; u < NA; ++u) {
            const int e = tid + u * NT;
            if (e < BK * BMv) {
                const int k = TRANS_A ? e / BMv : e % BK, m = TRANS_A ? e % BMv : e / BK;
                As[buf][k][m] = ra[u];
            }
        }
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            const int e = tid + u * NT;
            Bs[buf][e / BNv][e % BNv] = rb[u];
        }
    };

    const int64_t nk = (kend - kbeg + BK - 1) / BK;
    gload(kbeg);
    sstore(0);
    __syncthreads();
    for (int64_t kt = 0; kt < nk; ++kt) {
        const int buf = (int)(kt & 1);
        if (kt + 1 < nk) gload(kbeg + (kt + 1) * BK);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[TMv];
#pragma unroll
            for (int i = 0; i < TMv; ++i) a[i] = As[buf][k][ty * TMv + i];
            const float4 b = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
#pragma unroll
            for (int i = 0; i < TMv; ++i) {
                acc[i][0] = fmaf(a[i], b.x, acc[i][0]);
                acc[i][1] = fmaf(a[i], b.y, acc[i][1]);
                acc[i][2] = fmaf(a[i], b.z, acc[i][2]);
                acc[i][3] = fmaf(a[i], b.w, acc[i][3]);
            }
        }
        if (kt + 1 < nk) sstore(buf ^ 1);
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < TMv; ++i) {
        const int64_t gm = m0 + ty * TMv + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t gn = n0 + tx * 4 + j;
            if (gn < N) epi(gm, gn, N, acc[i][j]);
        }
    }
}

// Second pass of a split-K GEMM: add the slices in a fixed order (deterministic), then apply the fused epilogue.
template <class Epi>
__global__ void splitk_epilogue_kernel(const float* __restrict__ partial, int splits, int64_t M, int64_t N, Epi epi) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= M * N) return;
    float s = partial[e];
    for (int z = 1; z < splits; ++z) s += partial[(int64_t)z * M * N + e];
    const int64_t m = e / N;
    epi(m, e - m * N, N, s);
}

// Number of k-splits for an ISTA GEMM: enough CTAs for ~4 per SM on the small-P problems, none on the large ones.
int ista_splits(int64_t M, int64_t N, int64_t Kd) {
    const int64_t base = ((M + 31) / 32) * ((N + 47) / 48);
    int64_t sp = (592 + base - 1) / base;
    const int64_t by_k = Kd / (8 * BK);      // at least 8 k-tiles per split
    if (sp > by_k) sp = by_k;
    if (sp > 8) sp = 8;
    return sp < 1 ? 1 : (int)sp;
}

// Rows per CTA of an ISTA GEMM: 32 when split-K or when 64-row tiles would leave SMs idle, else 64.
int ista_row_tile(int64_t M, int64_t N, int splits, int sms) {
    const int64_t ncol = (N + 47) / 48;
    return (splits > 1 || ((M + 63) / 64) * ncol < 2 * (int64_t)(sms > 0 ? sms : 148)) ? 32 : 64;
}

__global__ void ista_prepare_kernel(const float* __restrict__ a, float lambda, int64_t P, float* __restrict__ inv_a,
                                    float* __restrict__ T) {
    int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= P) return;
    float av = a[p];
    bool ok = av > 0.0f && av < INFINITY;   // a <= 0, NaN or +inf: no step, the coefficients stay 0
    inv_a[p] = ok ? __fdiv_rn(1.0f, av) : 0.0f;
    T[p] = ok ? __fdiv_rn(lambda, __fmul_rn(2.0f, av)) : 0.0f;  // T = lambda/(2a), ista.m:17
}

// 1-D non-local means along the atom axis of G [K,P] (one column per patch): NLmeansfilter.m:18-91 on a K x 1 input
// with search radius 3 and patch radius 3 (pnp_ista.m:30), h = h_scale * T[p].  The symmetric padding (:24) makes
// the 7 window columns identical, so the 7x7 weighted distance reduces to 7 taps (row sums of make_kernel, :80-91).
__global__ void nlm_column_kernel(const float* __restrict__ G, const float* __restrict__ T, float h_scale, int K, int64_t P,
                                  float* __restrict__ out) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int k = blockIdx.y;
    if (p >= P) return;
    const float kw[7] = {1.0f / 21.0f, 4.0f / 35.0f, 71.0f / 315.0f, 71.0f / 315.0f, 71.0f / 315.0f, 4.0f / 35.0f, 1.0f / 21.0f};
    float x[13];  // G[k-6 .. k+6] with symmetric (edge-including mirror) extension, reflected as often as a short column
                  // needs (np.pad(..., mode="symmetric")): period 2K, the second half mirrored
#pragma unroll
    for (int u = 0; u < 13; ++u) {
        int idx = (k - 6 + u) % (2 * K);
        if (idx < 0) idx += 2 * K;
        if (idx >= K) idx = 2 * K - 1 - idx;
        x[u] = __ldg(G + (int64_t)idx * P + p);
    }
    const float h = h_scale * T[p];
    const float h2 = h * h, inv_h2 = h2 > 0.f ? 1.0f / h2 : INFINITY;
    // The reference's weights exp(-d / h^2) (double precision) are computed relative to the nearest window,
    // exp(-(d - dmin) / h^2): avg / sw is unchanged by the common factor exp(-dmin / h^2), which in fp32 underflows to 0
    // for every neighbour once dmin / h^2 > 87 and would return the input where the reference still averages.  A weight
    // is 0 where the reference's double-precision exp underflows (d / h^2 > 745); if all are, the input is returned (:80-84).
    float d[6];
    float dmin = INFINITY;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const int dr = j < 3 ? j - 3 : j - 2;
        d[j] = INFINITY;
        if (k + dr < 0 || k + dr >= K) continue;  // the search window is clipped to the real column (:46-49)
        float dd = 0.f;
#pragma unroll
        for (int u = -3; u <= 3; ++u) {
            float e = x[6 + u] - x[6 + dr + u];
            dd = fmaf(kw[u + 3] * e, e, dd);
        }
        d[j] = dd;
        dmin = fminf(dmin, dd);
    }
    float wmax = 0.f, avg = 0.f, sw = 0.f;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        const int dr = j < 3 ? j - 3 : j - 2;
        if (k + dr < 0 || k + dr >= K) continue;
        float w;
        if (!(h > 0.f)) w = d[j] == 0.f ? 1.f : 0.f;
        else if (d[j] == 0.f) w = 1.f;                                   // also when h^2 underflows
        else if (d[j] * inv_h2 > 745.0f) w = 0.f;
        else w = d[j] == dmin ? 1.f : __expf(-(d[j] - dmin) * inv_h2);
        wmax = fmaxf(wmax, w);
        sw += w;
        avg = fmaf(w, x[6 + dr], avg);
    }
    avg = fmaf(wmax, x[6], avg);
    sw += wmax;
    out[(int64_t)k * P + p] = sw > 0.f ? avg / sw : x[6];
}

template <bool TRANS_A, class ALoad, class Epi>
static int launch_gemm(const char* fn, ALoad al, const float* B, int64_t M, int64_t N, int64_t Kd, Epi epi,
                       cudaStream_t st, int64_t batch, int64_t ac_stride, int64_t b_stride) {
    dim3 grid((unsigned)((N + BN - 1) / BN), (unsigned)((M + BM - 1) / BM), (unsigned)batch);
    if (grid.y > 65535) return fail_arg(fn, "matrix too tall for this engine");
    sgemm_kernel<TRANS_A, ALoad, Epi><<<grid, 256, 0, st>>>(al, B, M, N, Kd, epi, ac_stride, b_stride);
    note_launch();
    return check_cuda(fn, cudaGetLastError());
}

// ISTA GEMMs: pipelined kernel; 32-row tiles when 64-row tiles would leave SMs idle, and split-K (partials in
// `scratch`, reduced in a fixed order by splitk_epilogue_kernel) when even those are too few CTAs.
template <bool TRANS_A, class Epi>
static int launch_gemm(const char* fn, LoadPlain al, const float* B, int64_t M, int64_t N, int64_t Kd, Epi epi,
                       cudaStream_t st, float* scratch = nullptr) {
    static int sms = device_sm_count();
    const int64_t ncol = (N + 47) / 48;
    const int splits = scratch ? ista_splits(M, N, Kd) : 1;
    const int bm = ista_row_tile(M, N, splits, sms);
    const bool small = bm == 32;
    dim3 grid((unsigned)ncol, (unsigned)((M + bm - 1) / bm), (unsigned)splits);
    if (grid.y > 65535) return fail_arg(fn, "matrix too tall for this engine");
    if (splits > 1) {
        const int64_t kchunk = ((Kd + splits - 1) / splits + BK - 1) / BK * BK;
        sgemm_pipe_kernel<TRANS_A, EpiPartial, 32><<<grid, 192, 0, st>>>(al.B, B, M, N, Kd, kchunk, EpiPartial{scratch});
        note_launch();
        int rc = check_cuda(fn, cudaGetLastError());
        if (rc != LRS_OK) return rc;
        splitk_epilogue_kernel<Epi><<<(unsigned)((M * N + 255) / 256), 256, 0, st>>>(scratch, splits, M, N, epi);
    } else if (small) {
        sgemm_pipe_kernel<TRANS_A, Epi, 32><<<grid, 192, 0, st>>>(al.B, B, M, N, Kd, Kd, epi);
    } else {
        sgemm_pipe_kernel<TRANS_A, Epi, 64><<<grid, 192, 0, st>>>(al.B, B, M, N, Kd, Kd, epi);
    }
    note_launch();
    return check_cuda(fn, cudaGetLastError());
}

// U[R,C] = (X + c L) W   — the recomposition GEMM of the Gram-based SVT (svt.cu declares it); for B cubes
// ([B, R, C] X, L, U and [B, C, C] W) cube b is grid z.
int svt_apply_impl(const float* X, const float* L, float c, const float* W, int64_t B, int64_t R, int64_t C, float* U,
                   cudaStream_t st) {
    // rows of Z play "M", W is the [Kd,N] operand
    dim3 grid((unsigned)((C + BN - 1) / BN), 1);
    int64_t rows_per_launch = 65535LL * BM;
    for (int64_t r0 = 0; r0 < R; r0 += rows_per_launch) {
        int64_t rows = R - r0 < rows_per_launch ? R - r0 : rows_per_launch;
        LoadAxpy al{X + r0 * C, L ? L + r0 * C : nullptr, c};
        int rc = launch_gemm<false>(B > 1 ? "lrs_svt_apply_batch_f32" : "lrs_svt_apply_f32", al, W, rows, C, C,
                                    EpiStore{U + r0 * C}, st, B, R * C, C * C);
        if (rc != LRS_OK) return rc;
    }
    return LRS_OK;
}

int nlm_columns(const char* fn, const float* G, const float* T, float h_scale, int K, int64_t P, float* A, cudaStream_t st) {
    if (K > 65535) return fail_arg(fn, "K too large for the NLM denoiser");
    dim3 grid((unsigned)((P + 127) / 128), (unsigned)K);
    nlm_column_kernel<<<grid, 128, 0, st>>>(G, T, h_scale, K, P, A);
    note_launch();
    return check_cuda(fn, cudaGetLastError());
}

}  // namespace lrs

using namespace lrs;

extern "C" {

size_t lrs_ista_workspace_bytes(int n, int K, int64_t P) {
    if (n <= 0 || K <= 0 || P < 0) return 0;
    // coefs [K,P] + denoiser input [K,P] + residual [n,P] + inv_a [P] + T [P] + split-K partials, each 256-byte aligned
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    const size_t s1 = (size_t)lrs::ista_splits(n, P, K) * n, s2 = (size_t)lrs::ista_splits(K, P, n) * K;
    const size_t part = (s1 > (size_t)n || s2 > (size_t)K) ? al((s1 > s2 ? s1 : s2) * (size_t)P * 4) : 0;
    const size_t simt = 2 * al((size_t)K * P * 4) + al((size_t)n * P * 4) + 2 * al((size_t)P * 4) + part;
    const size_t tcb = lrs::ista_tc_workspace_bytes(n, K, P);   // fp16 operand pieces of the tensor-core engine
    return simt > tcb ? simt : tcb;
}

int lrs_ista_soft_f32(const float* blocks_dev, const float* blocks_copy_dev, const float* D_dev, const float* a_dev,
                      float lambda_ista, int Nit, int n, int K, int64_t P, float* coefs_dev, float* phi_z_dev,
                      void* workspace_dev, size_t workspace_bytes, lrs_stream_t stream) {
    return lrs_ista_pnp_f32(blocks_dev, blocks_copy_dev, D_dev, a_dev, lambda_ista, Nit, n, K, P, LRS_DENOISE_SOFT, 1.0f,
                            coefs_dev, phi_z_dev, workspace_dev, workspace_bytes, stream);
}

int lrs_ista_pnp_f32(const float* blocks_dev, const float* blocks_copy_dev, const float* D_dev, const float* a_dev,
                     float lambda_ista, int Nit, int n, int K, int64_t P, int denoiser, float h_scale, float* coefs_dev,
                     float* phi_z_dev, void* workspace_dev, size_t workspace_bytes, lrs_stream_t stream) {
    const char* fn = "lrs_ista_pnp_f32";
    if (denoiser != LRS_DENOISE_SOFT && denoiser != LRS_DENOISE_NLM && denoiser != LRS_DENOISE_IDENTITY)
        return fail_arg(fn, "unknown denoiser");
    if (n <= 0 || K <= 0 || P < 0 || Nit < 0) return fail_arg(fn, "bad shape");
    if (!blocks_dev || !blocks_copy_dev || !D_dev || !a_dev) return fail_arg(fn, "null pointer");
    if (P == 0) return LRS_OK;
    if (workspace_bytes < lrs_ista_workspace_bytes(n, K, P) || !workspace_dev) {
        set_error(std::string(fn) + ": workspace smaller than lrs_ista_workspace_bytes()");
        return LRS_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    if (ista_tc_shape_ok(n, K, P) && ista_tc_enabled())
        return ista_tc_run(blocks_dev, blocks_copy_dev, D_dev, a_dev, lambda_ista, Nit, n, K, P, denoiser, h_scale, coefs_dev,
                           phi_z_dev, workspace_dev, workspace_bytes, st);
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    char* w = (char*)workspace_dev;
    float* A = (float*)w;
    w += al((size_t)K * P * 4);
    float* Gd = (float*)w;
    w += al((size_t)K * P * 4);
    float* Rm = (float*)w;
    w += al((size_t)n * P * 4);
    float* inv_a = (float*)w;
    w += al((size_t)P * 4);
    float* T = (float*)w;
    w += al((size_t)P * 4);
    float* scratch = (ista_splits(n, P, K) > 1 || ista_splits(K, P, n) > 1) ? (float*)w : nullptr;

    int rc = check_cuda(fn, cudaMemsetAsync(A, 0, (size_t)K * P * 4, st));  // x0 = 0  (ista.m:14)
    if (rc != LRS_OK) return rc;
    ista_prepare_kernel<<<(unsigned)((P + 255) / 256), 256, 0, st>>>(a_dev, lambda_ista, P, inv_a, T);
    LRS_CHECK_LAUNCH(fn);
    for (int it = 0; it < Nit; ++it) {
        rc = launch_gemm<false>(fn, LoadPlain{D_dev}, A, n, P, K, EpiResidual{blocks_dev, blocks_copy_dev, inv_a, Rm}, st, scratch);
        if (rc != LRS_OK) return rc;
        if (denoiser == LRS_DENOISE_SOFT) {
            rc = launch_gemm<true>(fn, LoadPlain{D_dev}, Rm, K, P, n, EpiGradient{T, A}, st, scratch);
        } else if (denoiser == LRS_DENOISE_IDENTITY) {
            rc = launch_gemm<true>(fn, LoadPlain{D_dev}, Rm, K, P, n, EpiGradientPlain{A, A}, st, scratch);
        } else {
            rc = launch_gemm<true>(fn, LoadPlain{D_dev}, Rm, K, P, n, EpiGradientPlain{A, Gd}, st, scratch);
            if (rc != LRS_OK) return rc;
            rc = nlm_columns(fn, Gd, T, h_scale, K, P, A, st);
        }
        if (rc != LRS_OK) return rc;
    }
    if (phi_z_dev) {
        rc = launch_gemm<false>(fn, LoadPlain{D_dev}, A, n, P, K, EpiStore{phi_z_dev}, st, scratch);
        if (rc != LRS_OK) return rc;
    }
    if (coefs_dev) {
        rc = check_cuda(fn, cudaMemcpyAsync(coefs_dev, A, (size_t)K * P * 4, cudaMemcpyDeviceToDevice, st));
        if (rc != LRS_OK) return rc;
    }
    return LRS_OK;
}

}  // extern "C"
