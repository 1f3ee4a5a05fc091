// Symmetric eigen-decomposition of the band Gram matrix for the SVT (main_LRS_PnP.py:118-124; C = bands <= 256) as ONE
// kernel on a thread-block cluster: one-sided (Hestenes) Jacobi in fp64, the matrix columns distributed over the shared
// memories of the 8 CTAs of the cluster and exchanged through distributed shared memory.
//
// Why not the library: cuSOLVER's syevd takes 1.1-2.1 ms for these orders (a chain of ~150 small launches, profiles/
// r02_eigh_time.txt) and its status word forces a host synchronisation in the middle of every outer iteration; on 8 GPUs
// that replicated, serial 1.6 ms is 2 % of the 77 ms step.  Here the whole decomposition is one launch and nothing waits
// on the host.
//
// Method.  Start from B = G (symmetric positive semi-definite, fp64).  A rotation of columns (p, q) by the angle that
// makes them orthogonal is a right-multiplication by a Givens matrix; sweeping over all pairs until every pair is
// orthogonal gives B = G V with V orthogonal and B^T B diagonal, i.e. V holds eigenvectors of G and column k of B is
// lambda_k v_k with lambda_k = ||b_k||.  V is never formed: the SVT only needs
//        W = V f(Lambda) V^T = sum_k  b_k b_k^T  f(lambda_k) / lambda_k^2          (lrs_svt_weights_f64, B form)
// and directions with lambda_k <= tau^2 have weight 0, so the division never meets a small eigenvalue.
//
// Parallel order.  The columns form 16 blocks of w = ceil(C/16) columns; CTA i holds a "top" and a "bottom" block.  A
// sweep is the 15 rounds of a round-robin tournament of the blocks: in a round a CTA orthogonalises every (top, bottom)
// column pair — w sub-rounds of w disjoint pairs, one warp per pair, the rows of a column spread over the lanes — then
// the blocks move to their next CTA (top[0] stays, the others rotate) by plain stores into the neighbour's shared
// memory and one cluster barrier.  Pairs inside a block are rotated once per sweep (round 0).  Every pair of columns
// meets exactly once per sweep: C - 1 + (C mod 2) sub-rounds, the minimum for a parallel Jacobi order.
#include <cooperative_groups.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "tc_common.cuh"

namespace cg = cooperative_groups;

namespace lrs {
using namespace tc;

namespace {

constexpr int JC = 8;              // CTAs per cluster (portable maximum)
constexpr int JNB = 2 * JC;        // column blocks
constexpr int JMAXW = 16;          // columns per block  -> C <= 256
constexpr int JT = 32 * JMAXW;     // one warp per column pair of a sub-round

// ---- the parallel Jacobi order, as pure index arithmetic (also compiled for the host: lrs_debug_jacobi_schedule replays a
// sweep on the CPU and tests/test_host.py checks, without a GPU, that every pair of columns meets exactly once) ----
// block width for C columns: ceil(C / 16), bumped so that a slot (w x C doubles) is a whole number of 16-byte words
__host__ __device__ inline int jacobi_block_width(int C) {
    int w = (C + JNB - 1) / JNB;
    if ((w * C) & 1) ++w;
    return w;
}
// cross pairs: in sub-round s warp i pairs top column i with this bottom column
__host__ __device__ inline int jacobi_cross_partner(int i, int s, int w) {
    const int jb = i + s;
    return jb >= w ? jb - w : jb;
}
// pairs inside a block: circle method on `we` (even) players, sub-round s, pair i of we/2; columns >= w are byes
__host__ __device__ inline void jacobi_circle_pair(int i, int s, int we, int& ca, int& cb) {
    if (i == 0) {
        ca = we - 1;
        cb = s;
    } else {
        ca = (s + i) % (we - 1);
        cb = (s - i + (we - 1)) % (we - 1);
    }
}
// tournament move of the blocks after a round: top[0] stays, top[1] <- bot[0], top[i] <- top[i-1], bot[i] <- bot[i+1],
// bot[JC-1] <- top[JC-1]; destination (CTA, slot 0 = top / 1 = bottom) of CTA `rank`'s two blocks
__host__ __device__ inline void jacobi_move(int rank, int& top_to, int& top_slot, int& bot_to, int& bot_slot) {
    if (rank == 0) {
        top_to = 0;
        top_slot = 0;
        bot_to = 1 % JC;
        bot_slot = 0;
    } else {
        if (rank < JC - 1) {
            top_to = rank + 1;
            top_slot = 0;
        } else {
            top_to = rank;
            top_slot = 1;
        }
        bot_to = rank - 1;
        bot_slot = 1;
    }
}

// Orthogonalise columns p and q (n rows each, in shared memory) — one warp.  Returns the squared cosine of the angle it
// removed (0 if the pair was left alone).
//   tol2   = (tolerance on the cosine of the angle between the columns)^2
//   floor2 = squared norm below which a column counts as zero (1e-14 ||G||_F): the columns of a rank-deficient matrix
//            decay to rounding noise, which would otherwise be rotated against itself sweep after sweep
// The rotation angle costs one rsqrt, one reciprocal and one more rsqrt in fp64 (no division, no sqrt): the scalar chain
// of a pair is what bounds a sub-round, not the column arithmetic.
template <int JROWS>   // rows per lane: ceil(C / 32) rounded up to even
__device__ __forceinline__ float rotate_pair(double* __restrict__ p, double* __restrict__ q, int n, int lane, double tol2,
                                            double floor2) {
    double bp[JROWS], bq[JROWS];
#pragma unroll
    for (int k = 0; k < JROWS; ++k) {
        const int r = lane + 32 * k;
        bp[k] = r < n ? p[r] : 0.0;
        bq[k] = r < n ? q[r] : 0.0;
    }
    // two accumulators per sum: the fp64 FMA has a 17-cycle dependent-issue latency (measured), the chain is what costs
    double a = bp[0] * bp[0], b = bq[0] * bq[0], g = bp[0] * bq[0];
    double a1 = bp[1] * bp[1], b1 = bq[1] * bq[1], g1 = bp[1] * bq[1];
#pragma unroll
    for (int k = 2; k < JROWS; k += 2) {
        a = fma(bp[k], bp[k], a);
        b = fma(bq[k], bq[k], b);
        g = fma(bp[k], bq[k], g);
        a1 = fma(bp[k + 1], bp[k + 1], a1);
        b1 = fma(bq[k + 1], bq[k + 1], b1);
        g1 = fma(bp[k + 1], bq[k + 1], g1);
    }
    a += a1;
    b += b1;
    g += g1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
        g += __shfl_xor_sync(0xffffffffu, g, o);
    }
    const double ab = a * b, g2 = g * g;
    if (!(g2 > tol2 * ab) || !(fmin(a, b) > floor2)) return 0.f;   // orthogonal already / a dead column / NaN
    // t = tan(theta) = smaller root of t^2 + 2 zeta t - 1, zeta = (b - a) / (2 g):  t = sign(d) h / (|d| + sqrt(d^2 + h^2))
    // (the hardware's approximate fp64 seeds, rsqrt / rcp.approx.ftz.f64, were tried for the angle: no faster, and their
    //  ~2^-8 accuracy leaves cosines of 1e-8 behind)
    const double d = b - a, h = 2.0 * g;
    const double x = fma(d, d, h * h);
    const double den = fma(x, rsqrt(x), fabs(d));
    const double t = (d >= 0.0 ? h : -h) * __drcp_rn(den);
    const double c = rsqrt(fma(t, t, 1.0)), s = c * t;            // c^2 + s^2 = 1 to fp64 whatever the accuracy of t
#pragma unroll
    for (int k = 0; k < JROWS; ++k) {
        const int r = lane + 32 * k;
        if (r < n) {
            p[r] = fma(c, bp[k], -s * bq[k]);
            q[r] = fma(s, bp[k], c * bq[k]);
        }
    }
    // only pairs of columns that can matter (norm above 1e-12 ||G||_F: lrs_svt_weights_f64 drops the others) keep the
    // iteration going; noise columns of a rank-deficient matrix are still rotated but never ask for another sweep
    return fmin(a, b) > 1e4 * floor2 ? fmaxf((float)(g2 / ab), 1e-37f) : 0.f;
}

// ---- distributed-shared-memory plumbing: bulk copies between the shared memories of two CTAs of the cluster (TMA engine),
// completion counted in bytes on an mbarrier of the DESTINATION CTA (mbar_expect_tx) ----
__device__ __forceinline__ uint32_t map_to_rank(uint32_t local_smem_addr, int rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void bulk_s2s(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes, uint32_t bar_cluster) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_cluster),
                 "r"(src_cta), "r"(bytes), "r"(bar_cluster)
                 : "memory");
}

// status[0] = sweeps run, status[1] = 1 if the last sweep still rotated by more than the stopping angle (not converged),
// status[2] = 1 if an eigenvalue is not finite (a diverged ADMM state reaches the SVT as a NaN / Inf Gram matrix).
//
// Shared memory: buf[phase 2][slot 2 (top, bottom)][w columns x n rows + 2 trailer doubles]; the trailer carries the block
// number, so a slot travels as ONE bulk copy.  Protocol of a round (no CTA ever waits for a barrier it has just arrived at):
//   1. rotate the pairs of the current phase;
//   2. wait for the cluster barrier armed in the PREVIOUS round — every CTA has then received that round's blocks, i.e.
//      nobody's copy engine still reads the buffers this round's copies are about to overwrite;
//   3. one thread arms its own mbarrier for the two incoming slots and sends its two slots to their next owners;
//   4. wait for the incoming slots (own mbarrier), arm the cluster barrier, switch phase.
// The stopping rule needs no verification sweep: Jacobi converges quadratically, so a sweep whose largest rotated cosine
// was below 3e-5 leaves cosines of order 1e-9.
//
// Batch: cluster q = blockIdx.x / JC solves problem q (G at q*n*n, lam at q*n, Bt at q*n*n, status at q*3).  Clusters
// never communicate, so they need not be resident at the same time: a batch larger than the GPU runs in waves.
template <int JROWS>
__global__ void __cluster_dims__(JC, 1, 1) __launch_bounds__(JT, 1)
    jacobi_eig_kernel(const double* __restrict__ G, int n, int w, double tol2, double stop2, int max_sweeps,
                      double* __restrict__ lam, double* __restrict__ Bt, int* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char jsm[];
    double* buf = reinterpret_cast<double*>(jsm);
    __shared__ __align__(8) uint64_t bar[2];               // incoming slots of phase 0 / 1 have landed
    __shared__ unsigned max_cos2[2][JC];                   // float bits of every CTA's largest rotated cos^2 of the sweep
    __shared__ unsigned my_max;
    __shared__ double fro[JT / 32];
    cg::cluster_group cl = cg::this_cluster();
    const int rank = (int)cl.block_rank();
    const int64_t prob = blockIdx.x / JC;
    G += prob * n * n;
    lam += prob * n;
    Bt += prob * n * n;
    status += prob * 3;
    const int tid = threadIdx.x, nthr = blockDim.x, warp = tid >> 5, lane = tid & 31;
    const size_t slot_sz = (size_t)w * n, slot_stride = slot_sz + 2;
    const uint32_t slot_bytes = (uint32_t)(slot_stride * sizeof(double));
    auto slot = [&](int ph, int s) { return buf + ((size_t)ph * 2 + s) * slot_stride; };

    // initial deal: CTA i holds blocks i (top) and i + JC (bottom); block b = columns [b w, b w + w) (zero beyond C)
    for (int s = 0; s < 2; ++s) {
        const int b = rank + s * JC;
        double* dst = slot(0, s);
        for (int e = tid; e < (int)slot_sz; e += nthr) {
            const int j = e / n, r = e - j * n, col = b * w + j;
            dst[e] = col < n ? G[(size_t)col * n + r] : 0.0;      // G is symmetric: column col = row col (coalesced)
        }
        if (tid == 0) dst[slot_sz] = (double)b;
    }
    if (tid == 0) {
        my_max = 0;
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_fence_init();
    }
    // ||G||_F^2 (every CTA computes the same sum in the same order): scale of the dead-column floor
    double floor2;
    {
        double f = 0.0;
        for (int e = tid; e < n * n; e += nthr) f = fma(G[e], G[e], f);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) f += __shfl_xor_sync(0xffffffffu, f, o);
        if (lane == 0) fro[warp] = f;
        __syncthreads();
        f = 0.0;
        for (int q = 0; q < nthr / 32; ++q) f += fro[q];
        floor2 = 1e-28 * f;
    }
    __syncthreads();
    cl.sync();                                             // barriers initialised, every CTA resident before remote traffic

    float wmax = 0.f;                                      // this warp's largest rotated cos^2 of the sweep (uniform in the warp)
    auto rotate = [&](double* p, double* q) { wmax = fmaxf(wmax, rotate_pair<JROWS>(p, q, n, lane, tol2, floor2)); };

    int ph = 0, sweep = 0;
    unsigned uses[2] = {0, 0};
    bool armed = false, more = true;
    for (; sweep < max_sweeps && more; ++sweep) {
        for (int round = 0; round < JNB - 1; ++round) {
            double* top = slot(ph, 0);
            double* bot = slot(ph, 1);
            // every (top, bottom) pair: sub-round s pairs top column i with bottom column (i + s) mod w
            for (int s = 0; s < w; ++s) {
                if (warp < w) rotate(top + (size_t)warp * n, bot + (size_t)jacobi_cross_partner(warp, s, w) * n);
                __syncthreads();
            }
            if (round == 0 && w > 1) {
                // pairs inside a block, once per sweep: circle method on we = w rounded up to even players; the first
                // we/2 warps serve the top block, the next we/2 the bottom block
                const int we = w + (w & 1), half = we / 2;
                for (int s = 0; s < we - 1; ++s) {
                    if (warp < we) {
                        const int sl = warp / half, i = warp - sl * half;
                        int ca, cb;
                        jacobi_circle_pair(i, s, we, ca, cb);
                        if (ca < w && cb < w) {
                            double* base = sl ? bot : top;
                            rotate(base + (size_t)ca * n, base + (size_t)cb * n);
                        }
                    }
                    __syncthreads();
                }
            }
            // tournament move: top[0] stays, top[1] <- bot[0], top[i] <- top[i-1], bot[i] <- bot[i+1], bot[JC-1] <- top[JC-1]
            const int nph = ph ^ 1;
            if (round == JNB - 2) {                                // end of the sweep: gather the warps' maxima (off the sub-round path)
                if (lane == 0 && wmax > 0.f) atomicMax(&my_max, __float_as_uint(wmax));   // positive floats order like their bits
                wmax = 0.f;
                __syncthreads();
            }
            if (armed) cl.barrier_wait();                          // step 2: last round's blocks have landed everywhere
            if (tid == 0) {
                int top_to, top_slot, bot_to, bot_slot;
                jacobi_move(rank, top_to, top_slot, bot_to, bot_slot);
                if (round == JNB - 2) {                            // end of the sweep: my largest rotation to every CTA
                    for (int pr = 0; pr < JC; ++pr) cl.map_shared_rank(&max_cos2[0][0], pr)[(sweep & 1) * JC + rank] = my_max;
                    my_max = 0;
                }
                fence_async_smem();                                // the rotations' stores -> copy engine
                mbar_expect_tx(&bar[nph], 2 * slot_bytes);
                bulk_s2s(map_to_rank(smem_u32(slot(nph, top_slot)), top_to), smem_u32(top), slot_bytes,
                         map_to_rank(smem_u32(&bar[nph]), top_to));
                bulk_s2s(map_to_rank(smem_u32(slot(nph, bot_slot)), bot_to), smem_u32(bot), slot_bytes,
                         map_to_rank(smem_u32(&bar[nph]), bot_to));
            }
            mbar_wait(&bar[nph], uses[nph] & 1);                   // step 4
            ++uses[nph];
            cl.barrier_arrive();
            armed = true;
            ph = nph;
        }
        cl.barrier_wait();                                         // sweep boundary: everybody's max_cos2 is visible
        armed = false;
        float m = 0.f;
        for (int pr = 0; pr < JC; ++pr) m = fmaxf(m, __uint_as_float(max_cos2[sweep & 1][pr]));
        more = (double)m > stop2;
    }

    // results: eigenvalue = column norm; columns written as rows of Bt (Bt[k, :] = b_k, coalesced)
    bool bad = false;
    for (int s = 0; s < 2; ++s) {
        const double* src = slot(ph, s);
        const int b = (int)src[slot_sz];
        for (int j = warp; j < w; j += nthr / 32) {
            const int col = b * w + j;
            if (col >= n) continue;
            double a = 0.0;
            for (int r = lane; r < n; r += 32) {
                const double v = src[(size_t)j * n + r];
                Bt[(size_t)col * n + r] = v;
                a = fma(v, v, a);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            const double l = sqrt(a);
            if (lane == 0) lam[col] = l;
            bad = bad || !(l - l == 0.0);
        }
    }
    if (bad && lane == 0) atomicExch(status + 2, 1);
    if (rank == 0 && tid == 0) {
        status[0] = sweep;
        status[1] = more ? 1 : 0;
    }
    cl.sync();                                                     // no CTA leaves while a peer may still address it
}

}  // namespace
}  // namespace lrs

using namespace lrs;

static int jacobi_launch(const char* fn, const double* G_dev, int64_t B, int C, double* lam_dev, double* Bt_dev, int* status_dev,
                         cudaStream_t st) {
    if (C < 1 || C > JNB * JMAXW) return fail_arg(fn, "need 1 <= C <= 256");
    if (B < 1 || B > LRS_MAX_BATCH) return fail_arg(fn, "need 1 <= B <= LRS_MAX_BATCH");
    if (!G_dev || !lam_dev || !Bt_dev || !status_dev) return fail_arg(fn, "null pointer");
    const int w = jacobi_block_width(C);                           // even slot size: the exchange moves 16-byte words
    if (w > JMAXW) return fail_arg(fn, "need 1 <= C <= 256");
    const size_t smem = (size_t)4 * ((size_t)w * C + 2) * sizeof(double);
    // rotate pairs whose cosine exceeds 1e-11; stop after a sweep whose largest rotated cosine was below 3e-5 (quadratic
    // convergence: what is left is of order 1e-9, two decades below what the fp32 weights W can resolve); 30 sweeps is far beyond the 7-9 a Gram matrix takes (14 for a spectrum
    // graded over 10 decades; exactly rank-deficient or degenerate matrices converge linearly in this parallel order: 17-22)
    const int we = w + (w & 1);
    auto launch = [&](auto kern) -> int {
        int rc = check_cuda(fn, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (rc != LRS_OK) return rc;
        rc = check_cuda(fn, cudaMemsetAsync(status_dev, 0, (size_t)B * 3 * sizeof(int), st));
        if (rc != LRS_OK) return rc;
        kern<<<(unsigned)(B * JC), 32 * we, smem, st>>>(G_dev, C, w, 1e-22, 1e-9, 30, lam_dev, Bt_dev, status_dev);
        return LRS_OK;
    };
    const int rows = (C + 31) / 32;                    // rows of a column per lane
    int rc = rows <= 2 ? launch(jacobi_eig_kernel<2>) : rows <= 4 ? launch(jacobi_eig_kernel<4>)
           : rows <= 6 ? launch(jacobi_eig_kernel<6>) : launch(jacobi_eig_kernel<8>);
    if (rc != LRS_OK) return rc;
    note_launch();
    return check_cuda(fn, cudaGetLastError());
}

extern "C" int lrs_sym_eig_jacobi_f64(const double* G_dev, int C, double* lam_dev, double* Bt_dev, int* status_dev,
                                      lrs_stream_t stream) {
    return jacobi_launch("lrs_sym_eig_jacobi_f64", G_dev, 1, C, lam_dev, Bt_dev, status_dev, (cudaStream_t)stream);
}

extern "C" int lrs_sym_eig_jacobi_batch_f64(const double* G_dev, int64_t B, int C, double* lam_dev, double* Bt_dev,
                                            int* status_dev, lrs_stream_t stream) {
    return jacobi_launch("lrs_sym_eig_jacobi_batch_f64", G_dev, B, C, lam_dev, Bt_dev, status_dev, (cudaStream_t)stream);
}

#ifdef LRS_DIAGNOSTICS
#include "../../include/lrs_pnp_diag.h"

// HOST replay of one sweep of the kernel's parallel order for C columns: meets_host[p * C + q] (p < q, caller zeroes) counts
// how often columns p and q are paired; conflicts_host receives the number of sub-rounds in which a column appeared twice.
extern "C" int lrs_debug_jacobi_schedule(int C, int* meets_host, int* conflicts_host, int* subrounds_host) {
    const char* fn = "lrs_debug_jacobi_schedule";
    if (C < 1 || C > JNB * JMAXW || !meets_host || !conflicts_host || !subrounds_host) return lrs::fail_arg(fn, "bad arguments");
    const int w = jacobi_block_width(C), N = JNB * w;
    if (w > JMAXW) return lrs::fail_arg(fn, "need 1 <= C <= 256");
    int top[JC], bot[JC];
    for (int i = 0; i < JC; ++i) {
        top[i] = i;
        bot[i] = i + JC;
    }
    int conflicts = 0, subrounds = 0;
    std::vector<int> used(N);
    auto meet = [&](int p, int q) {
        if (used[p]++ || used[q]++) ++conflicts;
        if (p < C && q < C) ++meets_host[(p < q ? p : q) * C + (p < q ? q : p)];
    };
    for (int round = 0; round < JNB - 1; ++round) {
        for (int s = 0; s < w; ++s) {                                  // cross pairs, all CTAs in parallel
            std::fill(used.begin(), used.end(), 0);
            for (int c = 0; c < JC; ++c)
                for (int i = 0; i < w; ++i) meet(top[c] * w + i, bot[c] * w + jacobi_cross_partner(i, s, w));
            ++subrounds;
        }
        if (round == 0 && w > 1) {
            const int we = w + (w & 1), half = we / 2;
            for (int s = 0; s < we - 1; ++s) {
                std::fill(used.begin(), used.end(), 0);
                for (int c = 0; c < JC; ++c)
                    for (int warp = 0; warp < we; ++warp) {
                        const int sl = warp / half, i = warp - sl * half;
                        int ca, cb;
                        jacobi_circle_pair(i, s, we, ca, cb);
                        if (ca < w && cb < w) meet((sl ? bot[c] : top[c]) * w + ca, (sl ? bot[c] : top[c]) * w + cb);
                    }
                ++subrounds;
            }
        }
        int ntop[JC], nbot[JC], filled = 0;
        for (int i = 0; i < JC; ++i) ntop[i] = nbot[i] = -1;
        for (int r = 0; r < JC; ++r) {
            int tt, ts, bt, bs;
            jacobi_move(r, tt, ts, bt, bs);
            (ts ? nbot : ntop)[tt] = top[r];
            (bs ? nbot : ntop)[bt] = bot[r];
        }
        for (int i = 0; i < JC; ++i) filled += (ntop[i] >= 0) + (nbot[i] >= 0);
        if (filled != 2 * JC) return lrs::fail_arg(fn, "the tournament move left a slot empty");
        for (int i = 0; i < JC; ++i) {
            top[i] = ntop[i];
            bot[i] = nbot[i];
        }
    }
    *conflicts_host = conflicts;
    *subrounds_host = subrounds;
    return LRS_OK;
}
#endif  // LRS_DIAGNOSTICS
