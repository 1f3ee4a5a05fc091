// Tensor-core engine of the explicit ISTA path (lrs_ista_pnp_f32: soft, NLM or identity update) for the LARGE-PATCH
// regime of the bundled configurations: n = bb^2 = 1296 pixels, K ~ 2592 atoms, P = 144 patches (main_LRS_PnP.py:131-149,
// 270-303; ista.m:13-24; 2304 patches for the 144 x 144 crop of main_LRS_PnP.m).  There the dictionary (13 MB) does not
// fit on chip and the two products of an iteration,
//     D alpha  [n x P] = D [n x K]  alpha [K x P]          and          D^T r  [K x P] = D^T [K x n]  r [n x P],
// are tall-skinny GEMMs against a few-hundred-column operand.  Each runs as ONE split-K launch of tcgen05 MMAs (M = 128
// rows per CTA, N = up to 256 patches per CTA, fp32 accumulators in TMEM) followed by a small reduce kernel that adds the
// split-K slices in a fixed order and applies the fused epilogue (mask + residual, or gradient step + soft threshold).
// The launches of a call are chained with programmatic dependent launch.
//
// fp32 accuracy comes from the same 3-pass fp16 operand split as the fused engine (sparse_fused_tc.cu, DESIGN 4.2):
//   x = x1 + x2, x1 = fp16(x), x2 = fp16(x - x1);   a b ~ a1 b1 + a2 b1 + a1 b2   (fp32 accumulate).
// The pieces of D (and of D^T, so that both products read a K-major A operand) are made once per call; the pieces of
// alpha and r are written by the reduce kernels.  Every operand is normalised by an exact power of two first — D by
// its largest entry, every patch column by its largest observed value — so the fp16 pieces are well scaled whatever
// the scale of the data, and the products are scaled back exactly in the reduce kernels.
#include <cuda_fp16.h>

#include <cstdlib>

#include "common.cuh"
#include "tc_common.cuh"

namespace lrs {
using namespace tc;

namespace {

constexpr int TG_BM = 128;         // rows of the A operand per CTA (TMEM lanes)
constexpr int TG_BK = 64;          // k per pipeline stage (4 MMA k-steps)
constexpr int TG_THREADS = 128;
constexpr float TS_D = 4.0f;       // D pieces  = fp16(4 sd D)
constexpr float TS_R = 0.25f;      // r pieces  = fp16(r' / 4)     (TS_D * TS_R = 1)
constexpr uint32_t A_PIECE = TG_BM * TG_BK * 2;     // 16 KB: [8 k-groups][128 rows][8 halves]

constexpr int TG_BN = 256;         // patches per tile of the B operand (MMA N)
__host__ __device__ inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
__host__ __device__ inline int64_t ptile_width(int64_t Np, int64_t t) { return Np - t * TG_BN < TG_BN ? Np - t * TG_BN : TG_BN; }
__host__ __device__ inline int64_t b_slot_halves(int64_t Np) { return 2 * (Np < TG_BN ? Np : TG_BN) * 64; }

__device__ __forceinline__ void split_h(float x, __half& h1, __half& h2) {
    h1 = __float2half_rn(x);
    h2 = __float2half_rn(x - __half2float(h1));
}

// 1-D bulk copy global -> shared (TMA engine, SASS UBLKCP), completion counted in bytes on an mbarrier (mbar_expect_tx)
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// Programmatic dependent launch: the 2*Nit+1 GEMM / reduce launches of a call form a chain in one stream.  Every kernel
// lets its successor start launching at once (its CTAs become resident as resources free up and run their set-up) and
// waits for its predecessor's results right before it first touches them.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// max |x| as float bits (non-negative floats order like their bit patterns)
__global__ void absmax_kernel(const float* __restrict__ x, int64_t n, unsigned* __restrict__ out) {
    float m = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        m = fmaxf(m, fabsf(x[i]));
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.f && m < INFINITY) atomicMax(out, __float_as_uint(m));
}

__device__ __forceinline__ float pow2_down_scale(const unsigned* dmax_bits) {   // sd: sd * max|D| in [0.5, 1)
    const float dmax = __uint_as_float(*dmax_bits);
    int ex = 0;
    if (dmax > 0.f) (void)frexpf(dmax, &ex);
    return ldexpf(1.0f, -ex);
}

// Operand pieces live in global memory as the exact images of the shared-memory stages, so that a stage is ONE
// contiguous bulk copy:
//   A tile (128 rows x 64 k), 32 KB:  halves  [piece][k/8][row][k%8]                 tile index = mtile * (Kp/64) + kblock
//   B tile (64 k x w patches):        halves  [piece][p/8][k][p%8]                   tile index = ptile * (Kp/64) + kblock
// The patch axis is cut into tiles of TG_BN = 256 columns (one MMA N, one TMEM accumulator); w is 256 except for the
// last tile.  Every B tile occupies a slot of 2 * min(Np, 256) * 64 halves.
__device__ __forceinline__ int64_t a_tile_offset(int64_t row, int64_t k, int64_t nkb) {
    return (((row >> 7) * nkb + (k >> 6)) << 14) + (((k & 63) >> 3) << 10) + ((row & 127) << 3) + (k & 7);
}

// D [n, K] -> fp16 pieces of 4 sd D, as A operand of D alpha (rows = pixels, k = atoms) and of D^T r (rows = atoms,
// k = pixels); the padding was zeroed by the caller.
__global__ void dict_pieces_kernel(const float* __restrict__ D, int n, int K, const unsigned* __restrict__ dmax_bits,
                                   __half* __restrict__ A1, int64_t nkb1, __half* __restrict__ A2, int64_t nkb2) {
    const float sc = pow2_down_scale(dmax_bits) * TS_D;
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= (int64_t)n * K) return;
    const int64_t i = e / K, k = e - i * K;
    __half h1, h2;
    split_h(D[e] * sc, h1, h2);
    const int64_t o1 = a_tile_offset(i, k, nkb1), o2 = a_tile_offset(k, i, nkb2);
    A1[o1] = h1;
    A1[o1 + 8192] = h2;
    A2[o2] = h1;
    A2[o2 + 8192] = h2;
}

// Per patch column: power-of-two normalisation of the operands, the scale-back factors of both products and the ISTA
// threshold T = lambda / (2a) (ista.m:15-17; a <= 0 marks a patch without any observed entry: coefficients stay 0).
//   residual pieces   = fp16 split of  m .* (y - D alpha) * sR ,  sR = 2^-ex(y) / 4       (NOT yet divided by a: with a
//                       large step constant r / a would fall into fp16's subnormal range)
//   coefficient pieces = fp16 split of  alpha * sA ,  sA = 2^-ex(y) * 2^ex(sqrt a)          (alpha ~ y / ||d||, a ~ ||d||^2)
__global__ void column_scales_kernel(const float* __restrict__ Y, int n, int64_t P, const unsigned* __restrict__ dmax_bits,
                                     const float* __restrict__ a, float lambda, float* __restrict__ sA,
                                     float* __restrict__ f1, float* __restrict__ f2, float* __restrict__ sR,
                                     float* __restrict__ T) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= P) return;
    float amax = 0.f;
    for (int i = 0; i < n; ++i) amax = fmaxf(amax, fabsf(Y[(int64_t)i * P + p]));
    int ex = 0;
    if (amax > 0.f && amax < INFINITY) (void)frexpf(amax, &ex);
    const float sd = pow2_down_scale(dmax_bits);
    const float av = a[p];
    const bool ok = av > 0.0f && av < INFINITY;
    int ea = 0;
    if (ok) (void)frexpf(sqrtf(av), &ea);
    sA[p] = ldexpf(1.0f, ea - ex);
    sR[p] = ldexpf(TS_R, -ex);
    f1[p] = ldexpf(1.0f, ex - ea) / (sd * TS_D);                               // D alpha   = (sum of MMAs) * f1
    f2[p] = ok ? __fdiv_rn(ldexpf(1.0f, ex) / sd, av) : 0.0f;                  // D^T r / a = (sum of MMAs) * f2   (TS_D TS_R = 1)
    T[p] = ok ? __fdiv_rn(lambda, __fmul_rn(2.0f, av)) : 0.0f;
}

struct GemmArgs {
    const __half* Ap;    // A tiles (see above), (Mp/128) x (Kp/64) of them
    const __half* Bp;    // B tiles, Kp/64 of them
    float* partial;      // [splits][M][N]
    int64_t M, N;        // logical output size
    int64_t Mp, Kp, Np;  // padded sizes (Mp % 128 == 0, Kp % 64 == 0, Np % 16 == 0)
    int kb_per_split;    // 64-wide k blocks per split
    int nkb_total;       // Kp / 64
};

// partial[z] = A[m0 : m0+128, k-range z] * B[k-range z, :]   with three MMAs per 16-wide k-step.
// A stage in shared memory (K-major canonical no-swizzle layout, LBO = 2048 between k-groups, SBO = 128 between row groups):
//     byte(m, k) = (k%8)*2 + (m%8)*16 + (m/8)*128 + (k/8)*2048          (+ piece * 16 KB)
// B stage (MN-major: 16-byte chunks = 8 consecutive patches, LBO = 128 between k-groups, SBO = 1024 between patch groups):
//     byte(nn, k) = (nn%8)*2 + (k%8)*16 + (k/8)*128 + (nn/8)*1024       (+ piece * Np*128)
// Warp 0 issues the MMAs, lane 0 of warp 1 drives the bulk copies, all four warps drain TMEM at the end.
template <int STAGES>
__global__ void __launch_bounds__(TG_THREADS, 1) tc_gemm_splitk_kernel(GemmArgs g) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ uint64_t bar_full[STAGES];
    __shared__ uint64_t bar_free[STAGES];
    __shared__ uint64_t bar_done;
    __shared__ uint32_t tmem_base_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    pdl_launch_dependents();
    const int pt = blockIdx.z;                                       // patch tile
    const uint32_t w = (uint32_t)ptile_width(g.Np, pt);              // its width (columns of the accumulator)
    const uint32_t b_piece = w * 128u, a_bytes = 2 * A_PIECE, b_bytes = 2 * b_piece;
    const uint32_t stage_bytes = a_bytes + (uint32_t)b_slot_halves(g.Np) * 2u;   // stage stride (widest tile)
    const int64_t m0 = blockIdx.x * (int64_t)TG_BM;
    const int z = blockIdx.y;
    const int kb0 = z * g.kb_per_split;
    const int nkb = g.nkb_total - kb0 < g.kb_per_split ? g.nkb_total - kb0 : g.kb_per_split;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&bar_full[s], 1);
            mbar_init(&bar_free[s], 1);
        }
        mbar_init(&bar_done, 1);
        mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&tmem_base_slot, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = tmem_base_slot;
    const uint32_t sbase = smem_u32(smem);
    pdl_wait();   // the B pieces come from the previous reduce kernel, which also still reads `partial`

    if (warp == 1 && lane == 0) {
        // ---- producer: one 32 KB bulk copy for the A stage, one for the B stage ----
        const __half* atile = g.Ap + (((int64_t)blockIdx.x * g.nkb_total + kb0) << 14);
        const int64_t slot = b_slot_halves(g.Np);
        const __half* btile = g.Bp + ((int64_t)pt * g.nkb_total + kb0) * slot;
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            if (kb >= STAGES) mbar_wait(&bar_free[s], (uint32_t)(((kb / STAGES) - 1) & 1));   // its MMAs have drained
            const uint32_t sa = sbase + (uint32_t)s * stage_bytes;
            mbar_expect_tx(&bar_full[s], a_bytes + b_bytes);
            bulk_g2s(sa, atile + ((int64_t)kb << 14), a_bytes, &bar_full[s]);
            bulk_g2s(sa + a_bytes, btile + (int64_t)kb * slot, b_bytes, &bar_full[s]);
        }
    } else if (warp == 0) {
        // ---- MMA issuer ----
        const uint32_t leader = elect_one();
        const uint32_t idesc = make_idesc_f16(128, (int)w, /*b_mn_major=*/true);
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % STAGES;
            mbar_wait(&bar_full[s], (uint32_t)((kb / STAGES) & 1));
            tc_fence_after();
            const uint32_t sa = sbase + (uint32_t)s * stage_bytes, sb = sa + a_bytes;
            const uint64_t a1 = make_smem_desc(sa, /*lbo=*/2048, /*sbo=*/128), a2 = make_smem_desc(sa + A_PIECE, 2048, 128);
            const uint64_t b1 = make_smem_desc(sb, /*lbo=*/128, /*sbo=*/1024), b2 = make_smem_desc(sb + b_piece, 128, 1024);
#pragma unroll
            for (int ks = 0; ks < TG_BK / 16; ++ks) {
                const uint64_t ao = (uint64_t)((2 * ks * 2048) >> 4), bo = (uint64_t)((2 * ks * 128) >> 4);
                if (leader) {
                    mma_f16_ss(tbase, a1 + ao, b1 + bo, idesc, !(kb == 0 && ks == 0));
                    mma_f16_ss(tbase, a2 + ao, b1 + bo, idesc, true);
                    mma_f16_ss(tbase, a1 + ao, b2 + bo, idesc, true);
                }
            }
            if (leader) mma_commit(&bar_free[s]);
            __syncwarp();
        }
        if (leader) mma_commit(&bar_done);
        __syncwarp();
    }
    __syncwarp();
    mbar_wait(&bar_done, 0);
    tc_fence_after();
    // epilogue: TMEM lane = output row; each thread writes its row's N partial sums
    {
        const int64_t m = m0 + 32 * warp + lane;
        float* dst = g.partial + ((int64_t)z * g.M + (m < g.M ? m : 0)) * g.N + (int64_t)pt * TG_BN;
        const int ncols = (int)(g.N - (int64_t)pt * TG_BN);          // logical columns left from this tile's first one
        const uint32_t lane_addr = tbase + ((uint32_t)(32 * warp) << 16);
        const bool vec = (g.N % 4 == 0);
        for (int c0 = 0; c0 < (int)w; c0 += 16) {
            uint32_t v[16];
            tmem_ld16(lane_addr + (uint32_t)c0, v);
            tmem_wait_ld();
            if (m < g.M) {
                if (vec) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4)
                        if (c0 + j < ncols)
                            *reinterpret_cast<float4*>(dst + c0 + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                                                  __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (c0 + j < ncols) dst[c0 + j] = __uint_as_float(v[j]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, 256);
}

// ---- reduce kernels: add the split-K slices in a fixed order, apply the epilogue, emit the next operand's pieces ----
// One thread owns 4 consecutive patches of one row = half a 16-byte chunk of each piece of the B tile image; up to eight
// slices are in flight per thread (the kernels are latency-bound: 1-2 MB of output against 10 MB of slices).
// (Measured alternative: reducing inside the GEMM kernel behind a per-row-tile arrival counter, cooperative launch —
//  23 us per product instead of 9.2 + 6.3 us: the 128 threads of a GEMM CTA cannot hide the L2 latency of its share.)
__device__ __forceinline__ float4 reduce4(const float* __restrict__ partial, int splits, int64_t MN, int64_t e0, int cnt) {
    float4 a;
    if (cnt == 4 && ((MN | e0) & 3) == 0) {
        const float4* q = reinterpret_cast<const float4*>(partial + e0);
        const int64_t st4 = MN / 4;
        a = q[0];
        int zz = 1;
        for (; zz + 8 <= splits; zz += 8) {
            float4 u[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) u[t] = q[(zz + t) * st4];
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                a.x += u[t].x; a.y += u[t].y; a.z += u[t].z; a.w += u[t].w;
            }
        }
        float4 u[8];
#pragma unroll
        for (int t = 0; t < 8; ++t)
            if (zz + t < splits) u[t] = q[(zz + t) * st4];
#pragma unroll
        for (int t = 0; t < 8; ++t)
            if (zz + t < splits) {
                a.x += u[t].x; a.y += u[t].y; a.z += u[t].z; a.w += u[t].w;
            }
        return a;
    }
    float s[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) s[j] = j < cnt ? partial[e0 + j] : 0.f;
    for (int zz = 1; zz < splits; ++zz) {
        const float* q = partial + (int64_t)zz * MN + e0;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < cnt) s[j] += q[j];
    }
    return make_float4(s[0], s[1], s[2], s[3]);
}
// patches 4*n4 .. 4*n4+3 of row `row` -> 8 bytes of each piece
__device__ __forceinline__ void store_pieces4(__half* __restrict__ Bp, int64_t row, int64_t n4, int64_t Np, int64_t nkb,
                                              const float (&v)[4]) {
    uint32_t w1[2], w2[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        __half a1, a2, b1, b2;
        split_h(v[2 * j], a1, a2);
        split_h(v[2 * j + 1], b1, b2);
        w1[j] = (uint32_t)__half_as_ushort(a1) | ((uint32_t)__half_as_ushort(b1) << 16);
        w2[j] = (uint32_t)__half_as_ushort(a2) | ((uint32_t)__half_as_ushort(b2) << 16);
    }
    // patch tile, k block, patch group of 8 within the tile, k within the block, half of the 16-byte chunk
    const int64_t p0 = 4 * n4, pt = p0 / TG_BN, pl = p0 - pt * TG_BN;
    __half* t = Bp + (pt * nkb + (row >> 6)) * b_slot_halves(Np) + (pl >> 3) * 512 + (row & 63) * 8 + ((pl >> 2) & 1) * 4;
    *reinterpret_cast<uint2*>(t) = make_uint2(w1[0], w1[1]);
    *reinterpret_cast<uint2*>(t + ptile_width(Np, pt) * 64) = make_uint2(w2[0], w2[1]);
}

// r = m .* (y - D alpha)  -> r pieces (the division by the step constant happens after D^T r, in f2)
__global__ void reduce_residual_kernel(const float* __restrict__ partial, int splits, int64_t n, int64_t P, int64_t Np,
                                       const float* __restrict__ Y, const float* __restrict__ BC,
                                       const float* __restrict__ f1, const float* __restrict__ sR,
                                       __half* __restrict__ B2p, int64_t nkb) {
    const int64_t nb4 = Np / 4, t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    pdl_launch_dependents();
    pdl_wait();
    if (t >= n * nb4) return;
    const int64_t i = t / nb4, n4 = t - i * nb4, p0 = 4 * n4, e0 = i * P + p0;
    const int cnt = P - p0 >= 4 ? 4 : (P - p0 > 0 ? (int)(P - p0) : 0);
    const float4 s4 = reduce4(partial, splits, n * P, e0, cnt);
    const float s[4] = {s4.x, s4.y, s4.z, s4.w};
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
        v[j] = (j < cnt && BC[e0 + j] != 0.0f) ? (Y[e0 + j] - s[j] * f1[p0 + j]) * sR[p0 + j] : 0.0f;
    store_pieces4(B2p, i, n4, Np, nkb, v);
}

// g = alpha + D^T r / a ;  GRAD_SOFT: alpha <- soft(g, T) (ista.m:21-23) ; GRAD_IDENTITY: alpha <- g ; both emit the
// pieces of the new alpha.  GRAD_PLAIN: G <- g for a plug-and-play denoiser that runs as its own kernel (pnp_ista.m:30).
enum { GRAD_SOFT = 0, GRAD_IDENTITY = 1, GRAD_PLAIN = 2 };
template <int MODE>
__global__ void reduce_gradient_kernel(const float* __restrict__ partial, int splits, int64_t K, int64_t P, int64_t Np,
                                       float* __restrict__ A, const float* __restrict__ T, const float* __restrict__ f2,
                                       const float* __restrict__ sA, __half* __restrict__ B1p, float* __restrict__ G,
                                       int64_t nkb) {
    const int64_t nb4 = Np / 4, t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    pdl_launch_dependents();
    pdl_wait();
    if (t >= K * nb4) return;
    const int64_t k = t / nb4, n4 = t - k * nb4, p0 = 4 * n4, e0 = k * P + p0;
    const int cnt = P - p0 >= 4 ? 4 : (P - p0 > 0 ? (int)(P - p0) : 0);
    const float4 s4 = reduce4(partial, splits, K * P, e0, cnt);
    const float s[4] = {s4.x, s4.y, s4.z, s4.w};
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        v[j] = 0.f;
        if (j < cnt) {
            const float g = A[e0 + j] + s[j] * f2[p0 + j];
            if (MODE == GRAD_PLAIN) {
                G[e0 + j] = g;
            } else {
                const float x = MODE == GRAD_SOFT ? soft_thr(g, T[p0 + j]) : g;
                A[e0 + j] = x;
                v[j] = x * sA[p0 + j];
            }
        }
    }
    if (MODE != GRAD_PLAIN) store_pieces4(B1p, k, n4, Np, nkb, v);
}

// pieces of a coefficient matrix that another kernel produced (the NLM denoiser)
__global__ void alpha_pieces_kernel(const float* __restrict__ A, int64_t K, int64_t P, int64_t Np, const float* __restrict__ sA,
                                    __half* __restrict__ B1p, int64_t nkb) {
    const int64_t nb4 = Np / 4, t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= K * nb4) return;
    const int64_t k = t / nb4, n4 = t - k * nb4, p0 = 4 * n4, e0 = k * P + p0;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = p0 + j < P ? A[e0 + j] * sA[p0 + j] : 0.f;
    store_pieces4(B1p, k, n4, Np, nkb, v);
}

// Phi_z = D alpha (full dictionary, main_LRS_PnP.py:294)
__global__ void reduce_store_kernel(const float* __restrict__ partial, int splits, int64_t n, int64_t P,
                                    const float* __restrict__ f1, float* __restrict__ phi) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= n * P) return;
    float s = partial[e];
    for (int zz = 1; zz < splits; ++zz) s += partial[(int64_t)zz * n * P + e];
    phi[e] = s * f1[e % P];
}

struct Plan {
    int64_t Mp1, Kp1, Mp2, Kp2, Np;
    int ntiles;             // patch tiles of TG_BN columns
    int S1, kb1, S2, kb2;   // splits and k blocks per split of both products
    size_t off_A, off_vec, off_dmax, off_A1, off_A2, off_B1, off_B2, off_part, off_G, total;
};

size_t al256(size_t b) { return (b + 255) / 256 * 256; }

void choose_splits(int64_t Mp, int64_t Kp, int ntiles, int sms, int& S, int& kb_per) {
    const int64_t mt = Mp / TG_BM * ntiles;   // output tiles; split k only as far as one wave of CTAs allows
    const int nkb = (int)(Kp / TG_BK);
    int s = (int)(sms / mt);
    if (s < 1) s = 1;
    if (s > nkb) s = nkb;
    kb_per = (nkb + s - 1) / s;
    S = (nkb + kb_per - 1) / kb_per;
}

Plan make_plan(int n, int K, int64_t P, int sms) {
    Plan pl;
    pl.Mp1 = round_up(n, TG_BM);
    pl.Kp1 = round_up(K, TG_BK);
    pl.Mp2 = round_up(K, TG_BM);
    pl.Kp2 = round_up(n, TG_BK);
    pl.Np = round_up(P, 16);
    pl.ntiles = (int)((pl.Np + TG_BN - 1) / TG_BN);
    choose_splits(pl.Mp1, pl.Kp1, pl.ntiles, sms, pl.S1, pl.kb1);
    choose_splits(pl.Mp2, pl.Kp2, pl.ntiles, sms, pl.S2, pl.kb2);
    size_t o = 0;
    pl.off_A = o;
    o += al256((size_t)K * P * 4);
    pl.off_vec = o;
    o += 5 * al256((size_t)P * 4);
    pl.off_dmax = o;
    o += 256;
    pl.off_A1 = o;
    o += al256((size_t)2 * pl.Mp1 * pl.Kp1 * 2);
    pl.off_A2 = o;
    o += al256((size_t)2 * pl.Mp2 * pl.Kp2 * 2);
    pl.off_B1 = o;
    o += al256((size_t)pl.ntiles * (pl.Kp1 / TG_BK) * b_slot_halves(pl.Np) * 2);
    pl.off_B2 = o;
    o += al256((size_t)pl.ntiles * (pl.Kp2 / TG_BK) * b_slot_halves(pl.Np) * 2);
    pl.off_part = o;
    const size_t p1 = (size_t)pl.S1 * n * P * 4, p2 = (size_t)pl.S2 * K * P * 4;
    o += al256(p1 > p2 ? p1 : p2);
    pl.off_G = o;                          // input of a plug-and-play denoiser
    o += al256((size_t)K * P * 4);
    pl.total = o;
    return pl;
}

constexpr int PLAN_SMS = 148;   // the workspace size must not depend on the device that later runs the call

}  // namespace

// Shapes the engine takes: a patch count that fits one MMA (N <= 256) and operands big enough to be worth the pieces.
bool ista_tc_shape_ok(int n, int K, int64_t P) { return P >= 8 && P <= (int64_t)65535 * TG_BN && n >= 128 && K >= 128; }

size_t ista_tc_workspace_bytes(int n, int K, int64_t P) { return ista_tc_shape_ok(n, K, P) ? make_plan(n, K, P, PLAN_SMS).total : 0; }

bool ista_tc_enabled() {
    const char* e = getenv("LRS_ISTA_ENGINE");   // "simt" forces the FFMA engine (tests compare the two)
    if (e && e[0] == 's') return false;
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return false;
    return major == 10;
}

// launch with the programmatic-stream-serialization attribute (see pdl_wait above)
template <class... KArgs, class... Args>
static cudaError_t launch_chained(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

template <int STAGES>
static int launch_tc_gemm(const char* fn, const GemmArgs& g, int splits, cudaStream_t st) {
    const size_t smem = (size_t)STAGES * (2 * A_PIECE + (size_t)b_slot_halves(g.Np) * 2);
    int rc = check_cuda(fn, cudaFuncSetAttribute(tc_gemm_splitk_kernel<STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (rc != LRS_OK) return rc;
    dim3 grid((unsigned)(g.Mp / TG_BM), (unsigned)splits, (unsigned)((g.Np + TG_BN - 1) / TG_BN));
    rc = check_cuda(fn, launch_chained(tc_gemm_splitk_kernel<STAGES>, grid, dim3(TG_THREADS), smem, st, g));
    note_launch();
    return rc;
}

static int tc_gemm(const char* fn, const GemmArgs& g, int splits, cudaStream_t st) {
    const size_t stage = 2 * A_PIECE + (size_t)b_slot_halves(g.Np) * 2;
    return 3 * stage <= 220 * 1024 ? launch_tc_gemm<3>(fn, g, splits, st) : launch_tc_gemm<2>(fn, g, splits, st);
}

int ista_tc_run(const float* blocks, const float* blocks_copy, const float* D, const float* a, float lambda, int Nit,
                int n, int K, int64_t P, int denoiser, float h_scale, float* coefs, float* phi, void* ws, size_t ws_bytes,
                cudaStream_t st) {
    const char* fn = "lrs_ista_pnp_f32";
    const Plan pl = make_plan(n, K, P, PLAN_SMS);
    if (ws_bytes < pl.total) {
        set_error(std::string(fn) + ": workspace smaller than lrs_ista_workspace_bytes()");
        return LRS_E_WORKSPACE;
    }
    char* w = (char*)ws;
    float* A = (float*)(w + pl.off_A);
    float* vec = (float*)(w + pl.off_vec);
    const size_t vs = al256((size_t)P * 4) / 4;
    float *sR = vec, *T = vec + vs, *sA = vec + 2 * vs, *f1 = vec + 3 * vs, *f2 = vec + 4 * vs;
    unsigned* dmax = (unsigned*)(w + pl.off_dmax);
    __half* A1 = (__half*)(w + pl.off_A1);
    __half* A2 = (__half*)(w + pl.off_A2);
    __half* B1 = (__half*)(w + pl.off_B1);
    __half* B2 = (__half*)(w + pl.off_B2);
    float* part = (float*)(w + pl.off_part);
    float* Gd = (float*)(w + pl.off_G);

    // x0 = 0 (ista.m:14), zero padding of every piece buffer, max |D|
    int rc = check_cuda(fn, cudaMemsetAsync(w + pl.off_A, 0, pl.off_part - pl.off_A, st));
    if (rc != LRS_OK) return rc;
    const int64_t nD = (int64_t)n * K;
    absmax_kernel<<<(unsigned)((nD + 1023) / 1024 < 592 ? (nD + 1023) / 1024 : 592), 256, 0, st>>>(D, nD, dmax);
    LRS_CHECK_LAUNCH(fn);
    dict_pieces_kernel<<<(unsigned)((nD + 255) / 256), 256, 0, st>>>(D, n, K, dmax, A1, pl.Kp1 / TG_BK, A2, pl.Kp2 / TG_BK);
    LRS_CHECK_LAUNCH(fn);
    column_scales_kernel<<<(unsigned)((P + 63) / 64), 64, 0, st>>>(blocks, n, P, dmax, a, lambda, sA, f1, f2, sR, T);
    LRS_CHECK_LAUNCH(fn);

    GemmArgs g1{A1, B1, part, n, P, pl.Mp1, pl.Kp1, pl.Np, pl.kb1, (int)(pl.Kp1 / TG_BK)};   // D alpha
    GemmArgs g2{A2, B2, part, K, P, pl.Mp2, pl.Kp2, pl.Np, pl.kb2, (int)(pl.Kp2 / TG_BK)};   // D^T r
    const int64_t nb4 = pl.Np / 4;
    const unsigned eb1 = (unsigned)((n * nb4 + 63) / 64), eb2 = (unsigned)((K * nb4 + 63) / 64);
    const unsigned es = (unsigned)(((int64_t)n * P + 255) / 256);
    for (int it = 0; it < Nit; ++it) {
        if ((rc = tc_gemm(fn, g1, pl.S1, st)) != LRS_OK) return rc;
        rc = check_cuda(fn, launch_chained(reduce_residual_kernel, dim3(eb1), dim3(64), 0, st, (const float*)part, pl.S1, (int64_t)n, P,
                                           pl.Np, blocks, blocks_copy, (const float*)f1, (const float*)sR, B2, pl.Kp2 / TG_BK));
        note_launch();
        if (rc != LRS_OK) return rc;
        if ((rc = tc_gemm(fn, g2, pl.S2, st)) != LRS_OK) return rc;
        if (denoiser == LRS_DENOISE_SOFT) {
            rc = check_cuda(fn, launch_chained(reduce_gradient_kernel<GRAD_SOFT>, dim3(eb2), dim3(64), 0, st, (const float*)part, pl.S2,
                                               (int64_t)K, P, pl.Np, A, (const float*)T, (const float*)f2, (const float*)sA, B1,
                                               (float*)nullptr, pl.Kp1 / TG_BK));
            note_launch();
            if (rc != LRS_OK) return rc;
        } else if (denoiser == LRS_DENOISE_IDENTITY) {
            rc = check_cuda(fn, launch_chained(reduce_gradient_kernel<GRAD_IDENTITY>, dim3(eb2), dim3(64), 0, st, (const float*)part,
                                               pl.S2, (int64_t)K, P, pl.Np, A, (const float*)T, (const float*)f2, (const float*)sA, B1,
                                               (float*)nullptr, pl.Kp1 / TG_BK));
            note_launch();
            if (rc != LRS_OK) return rc;
        } else {
            rc = check_cuda(fn, launch_chained(reduce_gradient_kernel<GRAD_PLAIN>, dim3(eb2), dim3(64), 0, st, (const float*)part, pl.S2,
                                               (int64_t)K, P, pl.Np, A, (const float*)T, (const float*)f2, (const float*)sA, B1, Gd, pl.Kp1 / TG_BK));
            note_launch();
            if (rc != LRS_OK) return rc;
            if ((rc = nlm_columns(fn, Gd, T, h_scale, K, P, A, st)) != LRS_OK) return rc;
            alpha_pieces_kernel<<<eb2, 64, 0, st>>>(A, K, P, pl.Np, sA, B1, pl.Kp1 / TG_BK);
            LRS_CHECK_LAUNCH(fn);
        }
    }
    if (phi) {
        if ((rc = tc_gemm(fn, g1, pl.S1, st)) != LRS_OK) return rc;
        reduce_store_kernel<<<es, 256, 0, st>>>(part, pl.S1, n, P, f1, phi);
        LRS_CHECK_LAUNCH(fn);
    }
    if (coefs) {
        rc = check_cuda(fn, cudaMemcpyAsync(coefs, A, (size_t)K * P * 4, cudaMemcpyDeviceToDevice, st));
        if (rc != LRS_OK) return rc;
    }
    return LRS_OK;
}

}  // namespace lrs
