// Fused sparse-coding step on the implicit patch set — tcgen05 / TMEM engine (bb = 8, n = 64, K in {64,128,192,256}).
//
// Same contract as the FFMA engine (sparse_fused_simt.cu): for every selected 8x8 window of the unfolded
// matrix run Nit soft-ISTA iterations against D and write Phi_z = D alpha (main_LRS_PnP.py:259-303,
// ista.m:13-24).  Here the two contractions of every iteration run on the 5th-generation tensor cores:
//
//   tile        128 row starts of one column start = the 128 TMEM lanes = MMA M (in the step-constant table mode the
//               row starts are ordered by their row-validity pattern, so most tiles hold one pattern)
//   GEMM-B      G[128 x K]    = alpha + r D        A operand = residual pieces in shared memory (SS form), two atom
//                                                  halves, accumulated IN PLACE onto the fp32 state in TMEM; only the
//                                                  window rows observed in the tile, two rows per 16-pixel k-step
//   epilogue    alpha = soft(G, T)                 tcgen05.ld -> registers -> tcgen05.st, 64-atom chunks
//   GEMM-A      Da[128 x 64]  = alpha D^T          A operand = alpha pieces staged in TMEM (TS form)
//   epilogue    r = m .* (y - Da / a)              fp16 pieces to shared memory, one 16-pixel k-step at a time
//
// Inside the kernel pixel i of a window is 8 * row + col (the reference's order is row + 8 * col), so that an 8-pixel
// core-matrix group (a K group of GEMM-B, an N group of GEMM-A) is one window row: the residual is exactly zero on a
// row no patch of the tile observes, and GEMM-B and the residual epilogue skip such rows.  Phi_z is stored in the
// reference's order.
//
// so alpha (128 KB per tile) never leaves TMEM during the Nit iterations; HBM sees 3 gathers and one
// Phi_z store per patch.
//
// fp32 accuracy on the tensor cores: every fp32 operand x is split into two fp16 pieces x = x1 + x2
// (x1 = fp16(x), x2 = fp16(x - x1): 22 significant bits) and a product uses three MMAs
// a1 b1 + a2 b1 + a1 b2 accumulated in fp32 — the 3-pass split-precision scheme, here on kind::f16 rather
// than kind::tf32 because (measured on B200, tests/test_gpu_tc.py, DESIGN.md):
//   * D is the B operand of both GEMMs, K-major in one and MN-major in the other.  With 16-bit elements
//     the two SWIZZLE_NONE canonical layouts are transposes of each other, so ONE 64 KB copy of the two
//     D pieces serves both GEMMs.  MN-major tf32 operands only exist in the SWIZZLE_128B_BASE32B layout,
//     which would need a second copy: 2 x 128 KB > 227 KB of shared memory.
//   * an fp16 MMA covers K = 16 per instruction (tf32: 8) at the same cost: half the tensor-pipe time.
// Each patch is normalised by an exact power of two (max |y| -> [0.5, 1)) so the fp16 pieces never leave
// their range whatever the scale of the data; the result is scaled back exactly.
//
// Warp roles (384 threads, 1 CTA / SM, persistent over tiles; DESIGN.md 4.3-4.4 has the schedule and its history):
//   warp 0      MMA issuer (whole warp runs the loop, one elected lane issues)
//   warps 1-3   gather the NEXT tile's patch values into shared memory (warp 1 also owns the TMEM allocation)
//   warps 4-11  epilogue: warp w owns TMEM lanes 32*(w%4).. and column group (w-4)/4 of every 64-column chunk and
//               8 pixels of every 16-pixel GEMM-B k-step of its patch.  16 epilogue warps were measured slower.
//   setmaxnreg moves registers from warps 0-3 (88 per thread) to warps 4-11 (208 per thread).
#include <cuda_fp16.h>
#include <stdlib.h>

#include <atomic>
#include <mutex>
#include <type_traits>

#include "common.cuh"
#include "tc_common.cuh"

namespace lrs {
using namespace tc;

namespace {

constexpr int TILE = 128;
constexpr int NEPI = 8;                        // epilogue warps (8 measured faster than 16: the epilogue is issue-bound)
constexpr int NCG = NEPI / 4;                  // column groups per TMEM lane quarter
constexpr int CW = 64 / NCG;                   // columns (of a 64-column chunk) and pixels per epilogue thread
constexpr int NPX = 16 / NCG;                  // pixels of every 16-pixel GEMM-B k-step owned by one epilogue thread
static_assert(NPX == 8, "the residual epilogue moves its pixels with 8-column TMEM loads and 16-byte stores");
constexpr int FIRST_EPI = 4;                   // first epilogue warp (keeps warp % 4 == TMEM lane quarter)
constexpr int NTHREADS = 32 * (FIRST_EPI + NEPI);
// setmaxnreg works on warpgroups: warps 0-3 give registers to warps 4-11
constexpr int WG0_REGS = 88, EPI_REGS = 208;
static_assert(128 * WG0_REGS + 256 * EPI_REGS <= 384 * 168, "register budget of one CTA per SM");
constexpr int MAXCHUNK = 4;                    // soft-threshold / GEMM-A pipeline: K/64 chunks of 64 atoms, K <= 256
constexpr uint32_t COL_ALPHA = 0;    // [0,256)   fp32 state / GEMM-B accumulator
constexpr uint32_t COL_ACC = 256;    // [256,320) a1 D1 + a2 D1 ; [320,384) a1 D2
constexpr uint32_t COL_STG0 = 384;   // staging buffers: piece 1 in [+0,+32), piece 2 in [+32,+64)
constexpr uint32_t COL_STG1 = 448;   //   buffer 0 also carries the residual pieces between GEMM-A and GEMM-B
// The state kept in TMEM is at = a * alpha' (alpha' = alpha / 2^ex, the patch-normalised coefficients), so that the
// residual operand r = m .* (y' - D alpha') is O(1) whatever the step constant a is:
//     at <- soft(at + r D, lambda' / 2),      D alpha' = (D at) / a
// (soft is positively homogeneous: a * soft(g, T) = soft(a g, a T), and a T = lambda / 2).
constexpr float S_ALPHA = 1.0f;      // state pieces    = fp16(at)
constexpr float S_D = 4.0f;          // D pieces        = fp16(4 D)
constexpr float S_R = 0.25f;         // residual pieces = fp16(r / 4)  (S_R * S_D = 1: GEMM-B lands in the state's units)

// D pieces in shared memory, one copy for both GEMMs (bytes):
//   (k%8)*2 + (i%8)*16 + (8*piece + i/8)*128 + (k/8)*2048       i = kernel pixel (8 * row + col), k = atom
constexpr uint32_t D_SMEM_BYTES = 64 * 1024;
// GEMM-B takes the residual pieces as the A operand from SHARED memory (SS form) and the 256 atoms in two N = 128
// halves, so that the soft-threshold of the first half overlaps the MMAs of the second (an N = 128 MMA with A in
// shared memory runs at its 64-cycle MAC floor; with A in TMEM it would cost 88).
// residual pieces in shared memory, K-major A operand (bytes): (k%8)*2 + (m%8)*16 + (m/8)*128 + (k/8)*2048 + piece*16384
constexpr uint32_t R_SMEM_BYTES = 32 * 1024;
constexpr uint32_t R_SK = 2048, R_SM = 128, R_PIECE = 16 * 1024;
constexpr uint32_t D_SK = 2048, D_SI = 128;
// Next tile's patch values, gathered by the otherwise idle warps 1..3 while the current tile iterates:
// V = X + L/mu as [kernel pixel][patch] floats (32 KB) and the observed flags as [kernel pixel][patch] bytes (8 KB)
constexpr uint32_t G_SMEM_BYTES = 64 * TILE * 4 + 64 * TILE;
constexpr int NLOAD = 32 * (FIRST_EPI - 1);   // loader threads

struct __align__(8) Shared {
    uint64_t bar_R[4];        // epilogue -> MMA: residual pieces of pixel quarter ks are in shared memory (NEPI warps)
    uint64_t bar_B[2];        // MMA -> epilogue: GEMM-B complete for atom half h                              (commit)
    uint64_t bar_S[MAXCHUNK];   // epilogue -> MMA: soft-thresholded state pieces of chunk j are staged     (NEPI warps)
    uint64_t bar_A[MAXCHUNK];   // MMA -> epilogue: GEMM-A of chunk j complete (staging free / Da final)    (commit)
    uint64_t bar_T[2];        // epilogue -> MMA: first / second 16-atom halves of the LAST chunk are staged (NEPI warps)
    uint64_t bar_G_full;      // loader -> epilogue: the gathered values of the next tile are in shared memory (loader warps)
    uint64_t bar_G_free;      // epilogue -> loader: the gather buffer has been consumed                      (NEPI warps)
    uint32_t tmem_base;
    uint32_t ring_head;       // dynamic tile schedule: work items published so far (written by warp 1, lane 0)
    uint32_t ring[8];         //   the last 8 of them
    uint32_t ring_read[NTHREADS / 32];   // items every warp has read: a slot is reused only when all warps are past it
    uint32_t tiles_pub;       // tiles announced by the gather warps (the MMA warp does not walk: it only counts tiles)
    uint32_t walk_done;       // set after the last announcement
    float xmax[NCG][TILE];    // per-patch partial max |y| of the pixel groups
    float xsum[NCG][TILE];    // per-patch partial sum of valid row norms (in-kernel 4||H||_F^2)
    uint32_t xrow[NCG][TILE]; // validity bits of window column 0, the rows of each column group
    uint32_t rowor[2][FIRST_EPI - 1];   // per gather warp, by tile parity: window rows observed by a patch of the tile
    float rn[64];             // ||Dh[i,:]||^2 (normalised dictionary)
    uint32_t dmax_bits;       // max |D| as float bits
};

__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(32 * NEPI) : "memory"); }

__device__ __forceinline__ uint32_t pack_h2(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }

// Packed fp32 pairs (sm_100 add/sub/fma.f32x2 -> FADD2 / FFMA2): the epilogue is instruction-issue bound and every
// value it touches comes in pairs, so one instruction per two elements halves its FP32-pipe instruction count.  The
// results are the same IEEE round-to-nearest values as the scalar forms.
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t sub2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

// x (already scaled) -> two fp16 pieces, two values per 32-bit word
__device__ __forceinline__ void split_pair(float x0, float x1, uint32_t& p1, uint32_t& p2) {
    __half2 h = __floats2half2_rn(x0, x1);
    float l0, l1;
    // x - fp16(x) with the mixed-precision FMA of sm_100 (fma.rn.f32.f16 -> FHFMA): one instruction per element instead of
    // a conversion and half a packed subtract; the difference is exact either way
    const unsigned short hl = __half_as_ushort(__low2half(h)), hh = __half_as_ushort(__high2half(h));
    const unsigned short m1 = 0xBC00;   // -1.0 in fp16
    asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(l0) : "h"(hl), "h"(m1), "f"(x0));
    asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(l1) : "h"(hh), "h"(m1), "f"(x1));
    __half2 l = __floats2half2_rn(l0, l1);
    p1 = pack_h2(h);
    p2 = pack_h2(l);
}

// soft(g, T) = g - clamp(g, -T, T) for a pair.  clamp(g, -T, T) = sign(g) min(|g|, T) is ONE instruction per element
// (min.xorsign.abs -> FMNMX.XORSIGN: magnitude min(|g|, |T|), sign = sign(g) xor sign(T), T >= 0), then one packed
// subtract: three instructions per pair, exact (|g| <= T gives g - g = 0; beyond it g -/+ T is the single rounding of
// sign(g)(|g| - T), soft.m:4).  The two-min/max form takes five instructions per pair; the fma.sat forms on the FMA pipe
// were either inexact in the dead zone or slower (DESIGN.md 4.4).
__device__ __forceinline__ void soft_pair(float g0, float g1, float T, float& x0, float& x1) {
    float t0, t1;
    asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(t0) : "f"(g0), "f"(T));
    asm("min.xorsign.abs.f32 %0, %1, %2;" : "=f"(t1) : "f"(g1), "f"(T));
    upk2(sub2(pk2(g0, g1), pk2(t0, t1)), x0, x1);
}

template <int N> __device__ __forceinline__ void tmem_ldN(uint32_t a, uint32_t* r) {
    if constexpr (N == 8) tmem_ld8(a, r);
    else if constexpr (N == 16) tmem_ld16(a, r);
    else tmem_ld32(a, r);
}
template <int N> __device__ __forceinline__ void tmem_stN(uint32_t a, const uint32_t* r) {
    if constexpr (N == 8) tmem_st8(a, r);
    else if constexpr (N == 16) tmem_st16(a, r);
    else tmem_st32(a, r);
}

// Debug timing (LRS_TC_TIMING=1): cycles block 0 spends waiting at each barrier, summed over the run.
//   [0] total MMA-warp cycles  [1..4] wait bar_R[ks]  [5..8] wait bar_S[j]  [10] MMA iterations
//   [16] total epilogue (warp 2) cycles [17] wait bar_A[last] [18] wait bar_B [19],[20] wait bar_A[0],[1]
//   [21] residual phase [22] soft phase [23] tile prologue [24] final epilogue
__device__ unsigned long long g_tc_timing[32];

#define TSTAMP() (DBG ? clock64() : 0ll)

// Tile order.  A tile is TILE consecutive row starts of ONE column start, so its patches read a (TILE+7) x 8 window
// of the cube.  A CTA walks work items = (row block rb, chunk of column starts): consecutive tiles of an item shift
// the window by one column, so seven eighths of every gather hit lines the previous tile already pulled into L1/L2
// and DRAM sees each cube row block about once per item instead of once per tile.  Patch numbering (and the Phi_z
// column) stays the reference's p = ci * nR + ri (main_LRS_PnP.py:90-99).
struct TilePlan {
    int64_t ci0, ci_end;   // column starts touched by [p_begin, p_end)
    int64_t items;         // rblocks * cchunks
    int cchunks, cpc;      // chunks per row block, column starts per chunk
    unsigned* counter;     // device word, zero at launch: next unclaimed work item (nullptr: static round-robin deal)
    const int* order;      // row starts in tile order, nR of them (nullptr: ascending)
};

// Row starts are ordered by the rank of their 8-row validity word in the reflected Gray code, so that consecutive
// patterns differ in one row and a tile that straddles two patterns observes at most one row more than either.
__host__ __device__ __forceinline__ uint32_t pattern_rank(uint32_t w) {
    w ^= w >> 1;
    w ^= w >> 2;
    w ^= w >> 4;
    return w;
}

// Window rows of a tile, from the OR w of the observed flags of its patches: the observed rows ascending, padded with
// unobserved rows to an even count of at least 2, then the other rows; nibble j holds the j-th row.  GEMM-B k-step s
// (s < nks = half the padded count) takes the rows of nibbles 2s, 2s+1.  Padding rows are unobserved by every patch of
// the tile, so their residual is exactly zero.
__device__ __forceinline__ uint32_t tile_rows(uint32_t w, int& nks) {
    w &= 0xFFu;
    int c = __popc(w);
    while (c < 2 || (c & 1)) {
        w |= ~w & (w + 1);            // lowest unobserved row
        ++c;
    }
    nks = c >> 1;
    uint32_t list = 0;
    int j = 0;
#pragma unroll
    for (int r = 0; r < 8; ++r)
        if ((w >> r) & 1u) list |= (uint32_t)r << (4 * j++);
#pragma unroll
    for (int r = 0; r < 8; ++r)
        if (!((w >> r) & 1u)) list |= (uint32_t)r << (4 * j++);
    return list;
}

// The walker also compiles for the host (lrs_debug_tile_walk below replays a launch's tile order on the CPU, so the
// no-GPU test suite covers this integer logic); on the device the CTA index and the grid size stay special registers.
//
// Two deals (template parameter DYN of next()).  Static: item = CTA, CTA + grid, ... — also what the host replay walks.
// Dynamic: work items are CLAIMED — a CTA takes the next unclaimed item from a device-wide counter, so a CTA that starts late
// (its SM was busy with another kernel: the low-rank step's eigensolver runs beside the first launch of a sparse step) simply
// claims fewer items.  Warp 1 claims an item and publishes it in a small shared-memory ring; the other walking warps (gather,
// epilogue) read it from there and note how far they have read (a sub-range launch can skip many items in a row, so the
// claiming warp checks those notes before it reuses a slot).  The MMA warp does not walk in the dynamic instance: it counts
// the tiles the gather warps announce (see the kernel).
struct TileWalk {
    int64_t item;
    int rb = 0, ci = 0, c_hi = 0;
    int64_t stride_ = 0;                     // host replay only (never read on the device: optimised away)
    // The walker keeps NO extra state for the dynamic schedule (the epilogue warps have no register to spare): how many
    // items a warp has read is kept in shared memory (ring_read[warp]; ring_head for the claiming warp itself).
    __device__ TileWalk() : item((int64_t)blockIdx.x - (int64_t)gridDim.x) {}
    __host__ TileWalk(int64_t cta, int64_t grid) : item(cta - grid), stride_(grid) {}
    template <bool DYN>
    __host__ __device__ __forceinline__ int64_t next_item(const TilePlan& pl, Shared* sh_) {
#ifdef __CUDA_ARCH__
        if (!DYN) return item + gridDim.x;
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        const uint32_t k = *(volatile uint32_t*)(warp == 1 ? &sh_->ring_head : &sh_->ring_read[warp]);
        uint32_t it = 0;
        if (warp == 1) {                     // the claiming warp (whole warp, so that its lanes stay converged)
            __syncwarp();                    // every lane has read k before lane 0 moves ring_head
            if (lane == 0) {
                it = atomicAdd(pl.counter, 1u);
                if (k >= 8) {                // slot k & 7 still holds item k - 8: every other warp must have read it
                    for (int w = 2; w < NTHREADS / 32; ++w)      // warps 2.. walk (warp 0, the MMA warp, only counts tiles)
                        while (*(volatile uint32_t*)&sh_->ring_read[w] < k - 7) {
                        }
                }
                sh_->ring[k & 7] = it;
                __threadfence_block();
                *(volatile uint32_t*)&sh_->ring_head = k + 1;
            }
            it = __shfl_sync(0xffffffffu, it, 0);
        } else {
            while (*(volatile uint32_t*)&sh_->ring_head <= k) {
            }
            __threadfence_block();
            it = *(volatile uint32_t*)&sh_->ring[k & 7];
            __syncwarp();
            if (lane == 0) *(volatile uint32_t*)&sh_->ring_read[warp] = k + 1;
            __syncwarp();                    // the next call's lanes read the updated count
        }
        return (int64_t)it;
#else
        (void)pl;
        (void)sh_;
        return item + stride_;
#endif
    }
    // advance to this CTA's next tile holding at least one patch of [p_begin, p_end); pl and prm are the kernel
    // parameters (constant bank), so the walker itself only keeps a few values live across the iteration loop
    template <bool DYN = false>
    __host__ __device__ __forceinline__ bool next(const TilePlan& pl, const FusedParams& prm, Shared* sh = nullptr) {
        const int64_t nR = prm.g.row.n;
        for (;;) {
            if (ci + 1 < c_hi) {
                ++ci;
            } else {
                item = next_item<DYN>(pl, sh);
                if (item >= pl.items) return false;
                rb = (int)(item / pl.cchunks);
                ci = (int)(pl.ci0 + (item - (int64_t)rb * pl.cchunks) * pl.cpc);
                c_hi = ci + pl.cpc < (int)pl.ci_end ? ci + pl.cpc : (int)pl.ci_end;
                if (ci >= c_hi) {
                    c_hi = ci;
                    continue;
                }
            }
            // an ordered tile holds row starts from anywhere in its column: it is walked when the column meets the range
            int64_t r0 = 0, r1 = nR;
            if (!pl.order) {
                r0 = (int64_t)rb * TILE;
                r1 = r0 + TILE < nR ? r0 + TILE : nR;
            }
            if (ci * nR + r1 > prm.p_begin && ci * nR + r0 < prm.p_end) return true;
        }
    }
};

// Lane m of the current tile: its patch, the window origin and the Phi_z column.  A lane is idle (stores nothing) when its
// patch lies outside [p_begin, p_end): it still computes its own patch, whose observed rows join the tile's row set, so
// that the row set, and with it every result, does not depend on the launch's range.  A lane past the last row start
// computes some patch of the range (finite garbage) and adds nothing to the row set.
struct PatchRef {
    int64_t p, pi, rs, cs;
    bool valid;
};
__host__ __device__ __forceinline__ PatchRef tile_patch(const FusedParams& prm, const TilePlan& pl, const TileWalk& tw, int m) {
    const int64_t nR = prm.g.row.n;
    int64_t ci = tw.ci, ri = (int64_t)tw.rb * TILE + m;
    if (pl.order && ri < nR) {
#ifdef __CUDA_ARCH__
        ri = __ldg(pl.order + ri);
#else
        ri = pl.order[ri];
#endif
    }
    int64_t p = ci * nR + ri;
    PatchRef r;
    r.valid = ri < nR && p >= prm.p_begin && p < prm.p_end;
    r.pi = p - prm.p_begin;
    if (ri >= nR) {
        p = p < prm.p_begin ? prm.p_begin : prm.p_end - 1;
        if (tw.ci * nR + nR - 1 >= prm.p_begin && tw.ci * nR + nR - 1 < prm.p_end) p = tw.ci * nR + nR - 1;
        ci = p / nR;
        ri = p - ci * nR;
    }
    r.p = p;
    r.rs = prm.g.row.start(ri);
    r.cs = prm.g.col.start(ci);
    return r;
}

// KATOMS in {64, 128, 192, 256}: the state occupies TMEM columns [0, KATOMS); GEMM-B is issued in two halves of KATOMS/2 atoms.
// FOLD: the masks are band-replicated (the a_table step-constant mode, whose table is indexed by the validity of the 8 window
// rows): the mask is folded into the residual constants, see the residual phase.
// DYN: work items claimed dynamically (see TileWalk); the static instance keeps every loop of the MMA warp warp-uniform in the
// compiler's eyes — with the claimed item arriving through shared memory ptxas spills uniform registers around the MMA groups
// (+3.8 % cycles per launch, ncu tensor pipe 74.0 instead of 76.9 %) — so the dynamic instance is used only for the launch
// that has to share the GPU (the first of a sparse step, beside the eigensolver).
template <bool DBG, int KATOMS, bool FOLD, bool DYN>
__global__ void __launch_bounds__(NTHREADS, 1) sparse_fused_tc_kernel(FusedParams prm, TilePlan plan) {
    constexpr int NCHUNK = KATOMS / 64;
    constexpr int KH = KATOMS / 2;                    // atoms per GEMM-B half (MMA N)
    constexpr int FIRST_B1_CHUNK = (KH + 63) / 64 - ((KH % 64) ? 1 : 0);   // first chunk touching the second half
    static_assert(KATOMS % 64 == 0 && KATOMS >= 64 && KATOMS <= 256 && KH % 16 == 0, "unsupported K");
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* Dsm = smem;
    uint8_t* Rsm = smem + D_SMEM_BYTES;
    float* Gv = reinterpret_cast<float*>(smem + D_SMEM_BYTES + R_SMEM_BYTES);
    uint8_t* Gok = smem + D_SMEM_BYTES + R_SMEM_BYTES + 64 * TILE * 4;
    Shared& sh = *reinterpret_cast<Shared*>(smem + D_SMEM_BYTES + R_SMEM_BYTES + G_SMEM_BYTES);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t total = prm.p_end - prm.p_begin;
    const int Nit = prm.Nit;

    // ---- one-time setup: D -> fp16 pieces, barriers, TMEM -------------------------------------------
    // The dictionary is normalised by an exact power of two, Dh = sd * D with max |Dh| in [0.5, 1), so that its
    // fp16 pieces are well scaled whatever the scale of D.  In "hat" units alpha_h = alpha'/sd, a_h = a sd^2:
    //     at_h <- soft(at_h + r Dh, lambda' sd / 2),   D alpha' = (Dh at_h) / a_h      (at_h = a_h alpha_h)
    if (tid == 0) {
        sh.dmax_bits = 0u;
        sh.ring_head = 0u;
        sh.tiles_pub = 0u;
        sh.walk_done = 0u;
    }
    if (tid < NTHREADS / 32) sh.ring_read[tid] = 0u;
    __syncthreads();
    {
        float mx = 0.f;
        for (int e = tid; e < 64 * KATOMS; e += NTHREADS) mx = fmaxf(mx, fabsf(prm.D[e]));
        atomicMax(&sh.dmax_bits, __float_as_uint(mx));   // non-negative floats order like their bit patterns
    }
    __syncthreads();
    int dex = 0;
    {
        const float dmax = __uint_as_float(sh.dmax_bits);
        if (dmax > 0.f && dmax < INFINITY) (void)frexpf(dmax, &dex);
    }
    const float sd = ldexpf(1.0f, -dex);
    for (int e = tid; e < 64 * KATOMS; e += NTHREADS) {
        const int ir = e / KATOMS, k = e % KATOMS, i = 8 * (ir % 8) + ir / 8;   // reference pixel row + 8 col -> kernel pixel
        float v = prm.D[e] * (sd * S_D);
        __half h1 = __float2half_rn(v);
        __half h2 = __float2half_rn(v - __half2float(h1));
        uint32_t off = (uint32_t)((k % 8) * 2 + (i % 8) * 16) + (uint32_t)(i / 8) * D_SI + (uint32_t)(k / 8) * D_SK;
        *reinterpret_cast<__half*>(Dsm + off) = h1;
        *reinterpret_cast<__half*>(Dsm + off + 8 * D_SI) = h2;
    }
    if (tid < 64) {
        float s = 0.f;
        for (int k = 0; k < KATOMS; ++k) {
            float d = prm.D[tid * KATOMS + k] * sd;
            s = fmaf(d, d, s);
        }
        sh.rn[8 * (tid % 8) + tid / 8] = s;              // ||Dh[i,:]||^2, kernel pixel order
    }
    if (tid == 0) {
        mbar_init(&sh.bar_B[0], 1);
        mbar_init(&sh.bar_B[1], 1);
        for (int j = 0; j < 4; ++j) mbar_init(&sh.bar_R[j], NEPI);
        for (int j = 0; j < NCHUNK; ++j) {
            mbar_init(&sh.bar_S[j], NEPI);
            mbar_init(&sh.bar_A[j], 1);
        }
        mbar_init(&sh.bar_T[0], NEPI);
        mbar_init(&sh.bar_T[1], NEPI);
        mbar_init(&sh.bar_G_full, FIRST_EPI - 1);
        mbar_init(&sh.bar_G_free, NEPI);
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc(&sh.tmem_base, 512);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = sh.tmem_base;
    // warp-specialised register budget: the MMA / gather warpgroup (warps 0-3) gives registers to the two epilogue
    // warpgroups (168 each at launch: 128*88 + 256*208 = 384*168; 56/224 .. 104/200 measure the same within noise)
    if (warp < 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(WG0_REGS));
    else asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(EPI_REGS));

    if (warp == 0) {
        // ================================ MMA issuer ================================
        const uint32_t leader = elect_one();
        const uint32_t dbase = smem_u32(Dsm);
        const uint32_t idescB = make_idesc_f16(128, KATOMS, /*b_mn_major=*/true);
        const uint32_t idescA128 = make_idesc_f16(128, 128, false);
        const uint32_t idescA64 = make_idesc_f16(128, 64, false);
        // GEMM-B: B = D as (N = atoms, K = pixels), MN-major: 16-byte atom chunks SBO = D_SK apart, 8-pixel groups
        //         LBO = D_SI apart; k-step s covers the pixel groups (window rows) a < b of the tile's row list: its
        //         descriptor starts at group a with LBO = (b - a) D_SI.
        const uint64_t descB0 = make_smem_desc(dbase, /*lbo=*/0, /*sbo=*/D_SK);
        // GEMM-A: B = D as (N = pixels [D1;D2], K = atoms), K-major: 16-byte atom chunks LBO = D_SK apart, 8-pixel
        //         groups SBO = D_SI apart; k-step covers atom groups 2g, 2g+1.
        const uint64_t descA0 = make_smem_desc(dbase, /*lbo=*/D_SK, /*sbo=*/D_SI);
        uint32_t gi = 0;
        long long dbg[11] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        const long long t_begin = TSTAMP();
        // Dynamic instance: the MMA warp does not walk the tiles (it needs no coordinates); the gather warps announce every tile
        // they find and the vote makes the loop condition warp-uniform.  Static instance: the walker itself (all uniform).
        TileWalk twm;
        uint32_t nt = 0, tcount = 0;
        auto more_tiles = [&]() -> bool {
            if constexpr (DYN) {
                uint32_t have;
                for (;;) {
                    have = *(volatile uint32_t*)&sh.tiles_pub;
                    if (have > nt) break;
                    if (*(volatile uint32_t*)&sh.walk_done) {
                        __threadfence_block();
                        have = *(volatile uint32_t*)&sh.tiles_pub;   // the last announcement precedes walk_done
                        break;
                    }
                }
                const bool ok = __all_sync(0xffffffffu, have > nt);
                ++nt;
                return ok;
            } else {
                return twm.next<false>(plan, prm);
            }
        };
        for (; more_tiles(); ++tcount) {
            // The tile's row list: its row word was published with the gather, before the epilogue staged this tile's
            // first residual k-step (at least one k-step is always issued).
            mbar_wait(&sh.bar_R[0], gi & 1);
            int nks;
            const uint32_t rl = tile_rows(sh.rowor[tcount & 1][0] | sh.rowor[tcount & 1][1] | sh.rowor[tcount & 1][2], nks);
            for (int it = 0; it < Nit; ++it, ++gi) {
                const uint32_t par = gi & 1;
                // ---- GEMM-B: state += r D; k-step ks (two window rows) starts as soon as its residual is staged ----
                {
                    const uint32_t idescB128 = make_idesc_f16(128, KH, /*b_mn_major=*/true);
                    const uint64_t descR0 = make_smem_desc(smem_u32(Rsm), /*lbo=*/R_SK, /*sbo=*/R_SM);
                    // Half 0 takes every k-step as soon as its residual quarter is staged (its completion releases the first
                    // soft-threshold chunks), then half 1 runs the tile's nks k-steps.
#pragma unroll
                    for (int half = 0; half < 2; ++half) {
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            if (half == 0) {
                                long long w0 = TSTAMP();
                                mbar_wait(&sh.bar_R[ks], par);
                                if (DBG) dbg[1 + ks] += clock64() - w0;
                                tc_fence_after();
                            }
                            if (ks < nks) {
                                const uint32_t ra = (rl >> (8 * ks)) & 15u, rw = (rl >> (8 * ks + 4)) & 15u;
                                const uint64_t dk = (uint64_t)((ra * D_SI + half * (KH / 8) * D_SK) >> 4) |
                                                    ((uint64_t)(((rw - ra) * D_SI) >> 4) << 16);   // LBO: group b
                                const uint64_t d1 = descB0 + dk;
                                const uint64_t d2 = descB0 + dk + (uint64_t)((8 * D_SI) >> 4);
                                const uint64_t r1 = descR0 + (uint64_t)((2 * ks * R_SK) >> 4);
                                const uint64_t r2 = descR0 + (uint64_t)((R_PIECE + 2 * ks * R_SK) >> 4);
                                const uint32_t acc = tbase + COL_ALPHA + KH * half;
                                if (leader) {
                                    mma_f16_ss(acc, r1, d1, idescB128, !(it == 0 && ks == 0));
                                    mma_f16_ss(acc, r2, d1, idescB128, true);
                                    mma_f16_ss(acc, r1, d2, idescB128, true);
                                }
                            }
                            __syncwarp();
                        }
                        if (leader) mma_commit(&sh.bar_B[half]);
                        __syncwarp();
                    }
                }
                // ---- GEMM-A: Da = state D^T, chunk by chunk as the soft-threshold epilogue releases them ----
#pragma unroll
                for (int j = 0; j < NCHUNK; ++j) {
                    const uint32_t stg = tbase + ((j & 1) ? COL_STG1 : COL_STG0);
                    // the last chunk is released in two halves (k-steps {0,2}, then {1,3}: each column group stages its
                    // first 16 atoms, then its last 16), so only two k-steps of MMAs remain after the soft threshold ends
                    if (j == NCHUNK - 1) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            long long w1 = TSTAMP();
                            mbar_wait(&sh.bar_T[h], par);
                            if (DBG) dbg[5 + j] += clock64() - w1;
                            tc_fence_after();
#pragma unroll
                            for (int ks = h; ks < 4; ks += 2) {
                                const uint64_t d = descA0 + (uint64_t)(((8 * j + 2 * ks) * D_SK) >> 4);
                                if (leader) {
                                    mma_f16_ts(tbase + COL_ACC, stg + 8 * ks, d, idescA128, !(j == 0 && ks == 0));   // a1 [D1;D2]
                                    mma_f16_ts(tbase + COL_ACC, stg + 32 + 8 * ks, d, idescA64, true);                // a2 D1
                                }
                            }
                            __syncwarp();
                        }
                        if (leader) mma_commit(&sh.bar_A[j]);
                        __syncwarp();
                        continue;
                    }
                    long long w1 = TSTAMP();
                    mbar_wait(&sh.bar_S[j], par);
                    if (DBG) dbg[5 + j] += clock64() - w1;
                    tc_fence_after();
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        const uint64_t d = descA0 + (uint64_t)(((8 * j + 2 * ks) * D_SK) >> 4);
                        if (leader) {
                            mma_f16_ts(tbase + COL_ACC, stg + 8 * ks, d, idescA128, !(j == 0 && ks == 0));  // a1 [D1;D2]
                            mma_f16_ts(tbase + COL_ACC, stg + 32 + 8 * ks, d, idescA64, true);               // a2 D1
                        }
                    }
                    // staging-release commits are only needed when chunks share staging buffers (the last chunk, above,
                    // signals "Da complete")
                    if (j + 2 < NCHUNK && leader) mma_commit(&sh.bar_A[j]);
                    __syncwarp();
                }
                if (DBG) dbg[10] += 1;
            }
        }
        if (DBG && blockIdx.x == 0 && leader) {
            g_tc_timing[0] = clock64() - t_begin;
            for (int i = 1; i < 11; ++i) g_tc_timing[i] = dbg[i];
        }
    } else if (warp >= FIRST_EPI) {
        // ================================ epilogue warps ================================
        const int q = warp & 3;                     // TMEM lane quarter (hardware: warp % 4)
        const int cg = (warp - FIRST_EPI) >> 2;     // column group: CW of every 64 columns, pixels [CW*cg, CW*cg+CW)
        const int m = q * 32 + lane;                // patch within the tile = TMEM lane
        const uint32_t lane_addr = tbase + ((uint32_t)(q * 32) << 16);
        uint32_t gi = 0, tcount = 0;
        long long ed[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        const long long e_begin = TSTAMP();
        for (TileWalk tw; tw.next<DYN>(plan, prm, &sh);) {
            const long long tp0 = TSTAMP();
            // ---- tile prologue: gather my CW pixels, mask, step constant, scale.  Register slot c holds window row
            //      row(2*(c/8) + cg) of the tile's row list, column c%8: GEMM-B k-step s is shared by the two column
            //      groups (one row each), so that all warps finish it together and its MMAs start early ----
            const PatchRef pr = tile_patch(prm, plan, tw, m);
            const bool valid = pr.valid;
            const int64_t pi = pr.pi, p = pr.p;                 // Phi_z column; patch for the step constant
            float ysc[CW];
            uint32_t mbits = 0;
            float amax = 0.f, nsum = 0.f;
            mbar_wait(&sh.bar_G_full, tcount & 1);              // gathered by warps 1..3 during the previous tile
            // byte s of rlc: my row of k-step s in bits 0-3, bit 7 set when the tile issues k-step s
            uint32_t rlc;
            {
                int nks;
                const uint32_t rl = tile_rows(sh.rowor[tcount & 1][0] | sh.rowor[tcount & 1][1] | sh.rowor[tcount & 1][2], nks);
                rlc = (rl >> (4 * cg)) & 0x0F0F0F0Fu;
#pragma unroll
                for (int s4 = 0; s4 < 4; ++s4)
                    if (s4 < nks) rlc |= 0x80u << (8 * s4);
            }
#pragma unroll
            for (int c = 0; c < CW; ++c) {
                const int pix = 8 * (int)((rlc >> (8 * (c >> 3))) & 15u) + (c & 7);
                const float v = Gv[pix * TILE + m];
                const bool ok = Gok[pix * TILE + m] != 0;
                ysc[c] = v;
                if (ok) {
                    mbits |= 1u << c;
                    amax = fmaxf(amax, fabsf(v));
                    nsum += sh.rn[pix];
                }
            }
            uint32_t xr = 0;                                    // window column 0 of my rows
#pragma unroll
            for (int s4 = 0; s4 < 4; ++s4) xr |= ((mbits >> (8 * s4)) & 1u) << ((rlc >> (8 * s4)) & 15u);
            __syncwarp();
            if (lane == 0) mbar_arrive(&sh.bar_G_free);         // the loader may fetch the next tile
            ++tcount;
            sh.xmax[cg][m] = amax;
            sh.xsum[cg][m] = nsum;
            sh.xrow[cg][m] = xr;
            epi_barrier();
            float a = 0.f;
            amax = 0.f;
            uint32_t xrow = 0;
#pragma unroll
            for (int g2 = 0; g2 < NCG; ++g2) {
                amax = fmaxf(amax, sh.xmax[g2][m]);
                a += sh.xsum[g2][m];
                xrow |= sh.xrow[g2][m];
            }
            a *= 4.0f;                                              // 4 ||H||_F^2 (main_LRS_PnP_DIP_pro.py:190)
            if (prm.a_patch) a = __ldg(prm.a_patch + p) * (sd * sd);          // caller's a refers to D: a_h = a sd^2
            else if (prm.a_table) a = __ldg(prm.a_table + xrow) * (sd * sd);
            epi_barrier();  // exchange buffers are free for the next tile
            const bool ok_a = a > 0.0f;
            const float inv_a = ok_a ? __fdiv_rn(1.0f, a) : 0.0f;
            int ex = 0;
            // amax = f * 2^ex, f in [0.5, 1).  Subnormal maxima are treated as 0 (2^-ex would overflow; such a patch is
            // below fp32's normal range anyway and reconstructs to 0), and ex is capped so that 2^ex stays finite.
            if (amax >= 1.17549435e-38f && amax < INFINITY) (void)frexpf(amax, &ex);
            ex = ex > 127 ? 127 : ex;
            const float dn = ldexpf(1.0f, -ex), up = ldexpf(1.0f, ex);
            const float Tn = ok_a ? 0.5f * prm.lambda * dn * sd : 0.0f;  // a_h * T_h = lambda' sd / 2 (ista.m:17)
            const float c1 = S_R * dn;                            // y -> scaled residual units
            const float c2 = inv_a * S_R / (S_ALPHA * S_D);       // acc (= S_ALPHA S_D a D alpha') -> scaled residual units
#pragma unroll
            for (int c = 0; c < CW; ++c) ysc[c] = ((mbits >> c) & 1u) ? ysc[c] * c1 : 0.f;    // y' stored masked
            const uint64_t nc2 = pk2(-c2, -c2);
            // slots 8s .. 8s+7 hold one window row (see above): with a band-replicated mask bit 8s speaks for all of them
            uint64_t nc2m[4];
#pragma unroll
            for (int s4 = 0; s4 < 4; ++s4) {
                const float v = ((mbits >> (8 * s4)) & 1u) ? -c2 : 0.f;
                nc2m[s4] = pk2(v, v);
            }
            if (DBG) ed[7] += clock64() - tp0;

            for (int it = 0; it < Nit; ++it, ++gi) {
                const uint32_t par = gi & 1;
                const long long tr0 = TSTAMP();
                // ---- residual: r = m .* (y' - D at / a) -> fp16 pieces in staging buffer 0, one 16-pixel quarter at a
                //      time so that GEMM-B starts on the first quarters while the others are being computed ----
                if (it > 0) {
                    mbar_wait(&sh.bar_A[NCHUNK - 1], par ^ 1);
                    if (DBG) ed[1] += clock64() - tr0;
                    tc_fence_after();
                }
                // FOLD: band-replicated masks (validity depends on the window row only), so the mask is folded into four
                // packed constants nc2m[s] = -c2 .* m and into y' itself: r = y'm - (c2 m) Da needs no per-element
                // select (the selects run on the half-rate ALU pipe that bounds the epilogue).
                // K-steps past the tile's nks are not issued: their barriers are only arrived on, so that every quarter
                // barrier keeps one phase per iteration.
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {             // GEMM-B k-step = two window rows; my row of it
                    if ((rlc >> (8 * ks + 7)) & 1u) {
                        uint32_t p1[NPX / 2], p2[NPX / 2];
                        if (it > 0) {
                            uint32_t b0[NPX], b1[NPX];
                            const uint32_t col = COL_ACC + 8 * ((rlc >> (8 * ks)) & 15u);
                            tmem_ld8(lane_addr + col, b0);
                            tmem_ld8(lane_addr + col + 64, b1);
                            tmem_wait_ld();
#pragma unroll
                            for (int c = 0; c < NPX / 2; ++c) {
                                const int e = NPX * ks + 2 * c;
                                const uint64_t sm2 = add2(pk2(__uint_as_float(b0[2 * c]), __uint_as_float(b0[2 * c + 1])),
                                                          pk2(__uint_as_float(b1[2 * c]), __uint_as_float(b1[2 * c + 1])));
                                float r0, r1;
                                upk2(fma2(FOLD ? nc2m[ks] : nc2, sm2, pk2(ysc[e], ysc[e + 1])), r0, r1);
                                if (!FOLD) {
                                    r0 = ((mbits >> e) & 1u) ? r0 : 0.f;
                                    r1 = ((mbits >> (e + 1)) & 1u) ? r1 : 0.f;
                                }
                                split_pair(r0, r1, p1[c], p2[c]);
                            }
                        } else {
#pragma unroll
                            for (int c = 0; c < NPX / 2; ++c) {
                                const int e = NPX * ks + 2 * c;
                                split_pair(ysc[e], ysc[e + 1], p1[c], p2[c]);   // y' is stored masked
                            }
                        }
                        // my 8 pixels = k-group 2ks + cg of my row m: one 16-byte store per piece (a warp covers 512
                        // contiguous bytes per store: conflict-free), then publish to the async proxy
                        uint8_t* rrow = Rsm + (uint32_t)(m >> 3) * R_SM + (uint32_t)(m & 7) * 16 + (uint32_t)(NCG * ks + cg) * R_SK;
                        *reinterpret_cast<uint4*>(rrow) = make_uint4(p1[0], p1[1], p1[2], p1[3]);
                        *reinterpret_cast<uint4*>(rrow + R_PIECE) = make_uint4(p2[0], p2[1], p2[2], p2[3]);
                        fence_async_smem();
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&sh.bar_R[ks]);
                }
                // ---- soft threshold, 4 chunks of 64 atoms; my CW columns of each.  The load of chunk j+1 is in
                //      flight while chunk j is processed. ----
                const long long ts0 = TSTAMP();
                if (DBG) ed[5] += ts0 - tr0;
                mbar_wait(&sh.bar_B[0], par);
                if (DBG) ed[2] += clock64() - ts0;
                tc_fence_after();
                uint32_t ga[CW], gb[CW];
                tmem_ldN<CW>(lane_addr + COL_ALPHA + CW * cg, ga);
#pragma unroll
                for (int j = 0; j < NCHUNK; ++j) {
                    uint32_t* g = (j & 1) ? gb : ga;
                    uint32_t* gn = (j & 1) ? ga : gb;
                    uint32_t p1[CW / 2], p2[CW / 2];
                    const uint32_t col = COL_ALPHA + 64 * j + CW * cg;
                    if (j == FIRST_B1_CHUNK) {  // first chunk with atoms of the second GEMM-B half: no prefetch across it
                        mbar_wait(&sh.bar_B[1], par);
                        tc_fence_after();
                        tmem_ldN<CW>(lane_addr + col, g);
                    }
                    tmem_wait_ld();
                    if (j + 1 < NCHUNK && j + 1 != FIRST_B1_CHUNK) tmem_ldN<CW>(lane_addr + col + 64, gn);
                    const uint32_t stg = (j & 1) ? COL_STG1 : COL_STG0;
                    auto soft_pairs = [&](int c_lo, int c_hi) {
#pragma unroll
                        for (int c = c_lo; c < c_hi; ++c) {
                            float x0, x1;
                            soft_pair(__uint_as_float(g[2 * c]), __uint_as_float(g[2 * c + 1]), Tn, x0, x1);
                            g[2 * c] = __float_as_uint(x0);
                            g[2 * c + 1] = __float_as_uint(x1);
                            split_pair(x0 * S_ALPHA, x1 * S_ALPHA, p1[c], p2[c]);
                        }
                    };
                    auto wait_staging = [&]() {
                        if (j >= 2) {  // staging buffer (j&1) is free once GEMM-A of chunk j-2 has completed
                            const long long tw = TSTAMP();
                            mbar_wait(&sh.bar_A[j - 2], par);
                            if (DBG) ed[3 + (j - 2)] += clock64() - tw;
                            tc_fence_after();
                        }
                    };
                    // chunk j's "staged" signal is given in the middle of chunk j+1's arithmetic, when its TMEM stores have
                    // landed, instead of stalling on tcgen05.wait::st right after issuing them
                    auto flush_pending = [&]() {
                        if (j > 0) {
                            tmem_wait_st();
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&sh.bar_S[j - 1]);
                        }
                    };
                    if (j == NCHUNK - 1) {
                        // last chunk: my first 16 atoms (k-step 2 cg), then my last 16 (k-step 2 cg + 1), each released on its
                        // own barrier, so that only two k-steps of GEMM-A remain when the soft threshold ends
                        static_assert(CW == 32, "the tail split stages 16-atom halves with x16 / x8 TMEM stores");
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            soft_pairs(8 * h, 8 * h + 8);
                            if (h == 0) {
                                flush_pending();
                                wait_staging();
                            }
                            tmem_st16(lane_addr + col + 16 * h, g + 16 * h);
                            tmem_st8(lane_addr + stg + (CW / 2) * cg + 8 * h, p1 + 8 * h);
                            tmem_st8(lane_addr + stg + 32 + (CW / 2) * cg + 8 * h, p2 + 8 * h);
                            tmem_wait_st();
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&sh.bar_T[h]);
                        }
                    } else {
                        soft_pairs(0, CW / 4);
                        flush_pending();
                        soft_pairs(CW / 4, CW / 2);
                        wait_staging();
                        tmem_stN<CW>(lane_addr + col, g);
                        tmem_stN<CW / 2>(lane_addr + stg + (CW / 2) * cg, p1);
                        tmem_stN<CW / 2>(lane_addr + stg + 32 + (CW / 2) * cg, p2);
                    }
                }
                if (DBG) ed[6] += clock64() - ts0;
            }
            const long long tf0 = TSTAMP();
            // ---- Phi_z = D alpha_final (main_LRS_PnP.py:294): my CW pixels of my patch ----
            {
                uint32_t a0[CW], a1[CW];
                mbar_wait(&sh.bar_A[NCHUNK - 1], (gi - 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) {
                    tmem_ld8(lane_addr + COL_ACC + 16 * q4 + NPX * cg, a0 + NPX * q4);
                    tmem_ld8(lane_addr + COL_ACC + 64 + 16 * q4 + NPX * cg, a1 + NPX * q4);
                }
                tmem_wait_ld();
                tc_fence_before();   // order these loads before the next tile's MMAs (via bar_R)
                const float sc = up * inv_a / (S_ALPHA * S_D);
                if (valid) {
                    // slot c = kernel pixel 16*(c/8) + NPX*cg + c%8 = window row 2*(c/8) + cg, column c%8
#pragma unroll
                    for (int c = 0; c < CW; ++c)
                        __stcs(prm.phi + (int64_t)(2 * (c >> 3) + cg + 8 * (c & 7)) * total + pi,
                               (__uint_as_float(a0[c]) + __uint_as_float(a1[c])) * sc);   // streaming: keep the cube in L2
                }
            }
            if (DBG) ed[8] += clock64() - tf0;
        }
        if (DBG && blockIdx.x == 0 && warp == FIRST_EPI && lane == 0) {
            g_tc_timing[16] = clock64() - e_begin;
            for (int i = 1; i < 9; ++i) g_tc_timing[16 + i] = ed[i];
        }
    } else {
        // ================================ gather warps (1 .. FIRST_EPI-1) ================================
        // One tile ahead of the epilogue: V = X + L/mu and the observed flags of the next tile's 128 x 64 window values
        // go to shared memory while the current tile iterates, so the tile prologue no longer waits on global memory.
        const int lt = tid - 32;
        const int64_t C = prm.g.C;
        uint32_t t = 0;
        for (TileWalk tw; tw.next<DYN>(plan, prm, &sh); ++t) {
            if (DYN && tid == 32) *(volatile uint32_t*)&sh.tiles_pub = t + 1;      // announce the tile to the MMA warp
            if (t > 0) mbar_wait(&sh.bar_G_free, (t - 1) & 1);
            uint32_t rows = 0;                            // window rows with an observed entry in a patch of the tile
            for (int m = lt; m < TILE; m += NLOAD) {
                const PatchRef pr = tile_patch(prm, plan, tw, m);
                const bool own = (int64_t)tw.rb * TILE + m < prm.g.row.n;   // the lane holds a patch of the tile
                const float* xs = prm.X + pr.rs * C + pr.cs;
                const float* ys = prm.Yobs + pr.rs * C + pr.cs;
                const float* ls = prm.L ? prm.L + pr.rs * C + pr.cs : nullptr;
#pragma unroll 2
                for (int j = 0; j < 8; ++j) {            // window column j: kernel pixels j, 8 + j, .. 56 + j = rows 0..7
                    float v[8], o[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        v[i] = __ldg(xs + i * C + j);
                        o[i] = __ldg(ys + i * C + j);
                    }
                    if (ls) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v[i] = __fadd_rn(v[i], __fdiv_rn(__ldg(ls + i * C + j), prm.mu1));
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        Gv[(8 * i + j) * TILE + m] = v[i];
                        Gok[(8 * i + j) * TILE + m] = o[i] != 0.0f ? 1 : 0;
                        if (own && o[i] != 0.0f) rows |= 1u << i;
                    }
                }
            }
            rows = __reduce_or_sync(0xffffffffu, rows);
            if (lane == 0) sh.rowor[t & 1][warp - 1] = rows;   // tile t-2, the last reader of this slot, is done
            __syncwarp();
            if (lane == 0) mbar_arrive(&sh.bar_G_full);
        }
        if (DYN && tid == 32) {                            // no more tiles (after the last announcement)
            __threadfence_block();
            *(volatile uint32_t*)&sh.walk_done = 1u;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tbase, 512);
}

// ---- tile order of the step-constant table mode: row starts sorted by the Gray rank of their row-validity word ----
// The word uses the same bits as the table index (Yobs != 0 in the window's rows, column 0: table mode asserts
// band-replicated masks).  The order only decides which patches share a tile, never a result: the kernel derives a
// tile's row set from the gathered flags themselves.
__global__ void row_pattern_keys_kernel(const float* __restrict__ Yobs, Geom g, uint8_t* __restrict__ key) {
    const int64_t ri = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ri >= g.row.n) return;
    const float* y = Yobs + g.row.start(ri) * g.C;
    uint32_t w = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) w |= (__ldg(y + i * g.C) != 0.0f ? 1u : 0u) << i;
    key[ri] = (uint8_t)pattern_rank(w);
}

// Stable counting sort of n one-byte keys: CTA k writes the row starts with key k, ascending, after the count of smaller
// keys.  Thread t of every CTA reads the t-th contiguous share of the key array (the array is padded to a multiple of 16)
// twice, 16 keys per load: ~0.5 MB per CTA from L2 for the 262137 row starts of a 512 x 512 cube.  The result does not
// depend on timing, so every launch of a range sees the same tiles.
constexpr int SORT_THREADS = 1024;
__device__ __forceinline__ uint32_t key_matches(const uint8_t* key, int64_t n, int64_t i0, uint32_t k, bool below) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(key + i0));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t bits = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const uint32_t kj = (w[j >> 2] >> (8 * (j & 3))) & 0xFFu;
        if (i0 + j < n && (below ? kj < k : kj == k)) bits |= 1u << j;
    }
    return bits;
}
// exclusive prefix of v over the CTA; total receives the sum (every thread)
__device__ __forceinline__ uint32_t cta_exclusive_scan(uint32_t v, uint32_t* wsum, uint32_t& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t before = 0;
    total = 0;
    for (int w = 0; w < SORT_THREADS / 32; ++w) {
        const uint32_t t = wsum[w];
        before += w < warp ? t : 0u;
        total += t;
    }
    __syncthreads();   // wsum is reused by the next call
    return before + inc - v;
}
__global__ void __launch_bounds__(SORT_THREADS) row_order_kernel(const uint8_t* __restrict__ key, int64_t n, int* __restrict__ order) {
    __shared__ uint32_t wsum[SORT_THREADS / 32];
    const uint32_t k = blockIdx.x;
    const int64_t share = ((n + 16 * SORT_THREADS - 1) / (16 * SORT_THREADS)) * 16;
    const int64_t b = share * threadIdx.x, e = b + share < n ? b + share : n;
    uint32_t below = 0, mine = 0, total, base;
    for (int64_t i0 = b; i0 < e; i0 += 16) {
        below += __popc(key_matches(key, n, i0, k, true));
        mine += __popc(key_matches(key, n, i0, k, false));
    }
    uint32_t pos = cta_exclusive_scan(mine, wsum, total);
    if (total == 0) return;
    (void)cta_exclusive_scan(below, wsum, base);
    pos += base;
    for (int64_t i0 = b; i0 < e; i0 += 16)
        for (uint32_t bits = key_matches(key, n, i0, k, false); bits; bits &= bits - 1) order[pos++] = (int)(i0 + __ffs(bits) - 1);
}

}  // namespace

bool sparse_fused_tc_supported(const FusedParams& prm, int K) {
    if ((K != 64 && K != 128 && K != 192 && K != 256) || prm.g.bb != 8 || prm.Nit < 1) return false;
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return false;
    return major == 10;
}

// work items: every row block of TILE row starts, cut into enough column-start chunks that the persistent grid stays
// balanced (>= ~100 items per SM when the problem has them) while a chunk still reuses its window.
static TilePlan make_tile_plan(const FusedParams& prm, int sms) {
    const int64_t nR = prm.g.row.n;
    TilePlan plan;
    plan.ci0 = prm.p_begin / nR;
    plan.ci_end = (prm.p_end - 1) / nR + 1;
    const int64_t ncols = plan.ci_end - plan.ci0, rblocks = (nR + TILE - 1) / TILE;
    int64_t cchunks = (100 * (int64_t)sms + rblocks - 1) / rblocks;
    cchunks = cchunks < 1 ? 1 : (cchunks > ncols ? ncols : cchunks);
    plan.cpc = (int)((ncols + cchunks - 1) / cchunks);
    plan.cchunks = (int)((ncols + plan.cpc - 1) / plan.cpc);   // no empty chunks: every work item holds tiles
    plan.items = rblocks * plan.cchunks;
    plan.counter = nullptr;
    plan.order = nullptr;
    return plan;
}

// Claim counters of the dynamic tile schedule: a pool of words per device, one per launch in flight (a sparse step has two
// launches in flight on its two streams; 64 slots cannot wrap around a launch that is still running).
static unsigned* claim_counter(cudaStream_t st) {
    constexpr int SLOTS = 64, MAXDEV = 64;
    static unsigned* pool[MAXDEV] = {};
    static std::atomic<unsigned> seq{0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAXDEV) return nullptr;
    if (!pool[dev]) {
        static std::mutex mu;
        std::lock_guard<std::mutex> lock(mu);
        if (!pool[dev] && cudaMalloc(&pool[dev], SLOTS * sizeof(unsigned)) != cudaSuccess) {
            pool[dev] = nullptr;
            (void)cudaGetLastError();
            return nullptr;
        }
    }
    unsigned* c = pool[dev] + (seq.fetch_add(1) % SLOTS);
    if (cudaMemsetAsync(c, 0, sizeof(unsigned), st) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return c;
}

template <int K>
static int launch_tc(const FusedParams& prm, bool dynamic_tiles, cudaStream_t st) {
    const char* fn = "lrs_sparse_step_fused_f32";
    const size_t smem = D_SMEM_BYTES + R_SMEM_BYTES + G_SMEM_BYTES + sizeof(Shared);
    const bool fold = prm.a_table != nullptr && prm.a_patch == nullptr;
    using Kern = void (*)(FusedParams, TilePlan);
    auto pick = [&](auto dbg_c, bool dyn) -> Kern {
        constexpr bool DBGV = decltype(dbg_c)::value;
        if (dyn) return fold ? sparse_fused_tc_kernel<DBGV, K, true, true> : sparse_fused_tc_kernel<DBGV, K, false, true>;
        return fold ? sparse_fused_tc_kernel<DBGV, K, true, false> : sparse_fused_tc_kernel<DBGV, K, false, false>;
    };
#ifdef LRS_DIAGNOSTICS   // liblrs_pnp_diag.so only: barrier-wait counters (include/lrs_pnp_diag.h)
    static const bool dbg = getenv("LRS_TC_TIMING") != nullptr;
    Kern kern = dbg ? pick(std::true_type{}, dynamic_tiles) : pick(std::false_type{}, dynamic_tiles);
#else
    Kern kern = pick(std::false_type{}, dynamic_tiles);
#endif
    int rc = check_cuda(fn, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (rc != LRS_OK) return rc;
    int sms = device_sm_count();
    if (sms <= 0) return check_cuda(fn, cudaErrorNoDevice);
    TilePlan plan = make_tile_plan(prm, sms);
    unsigned grid = (unsigned)(plan.items < sms ? plan.items : sms);
    plan.counter = dynamic_tiles ? claim_counter(st) : nullptr;
    if (dynamic_tiles && !plan.counter) return fail_arg(fn, "no claim counter for the dynamic tile schedule");
    // table mode: tiles of row starts with one row-validity pattern, so that GEMM-B and the residual skip the rows none of
    // a tile's patches observes.  Scratch is stream-ordered on the launch stream.
    const int64_t nR = prm.g.row.n;
    void* scratch = nullptr;
    if (fold) {
        if (nR >= ((int64_t)1 << 30)) return fail_arg(fn, "too many row starts for the row-pattern tile order");
        const int64_t nkey = (nR + 15) / 16 * 16;
        rc = check_cuda(fn, cudaMallocAsync(&scratch, (size_t)nkey * 5, st));
        if (rc != LRS_OK) return rc;
        int* order = static_cast<int*>(scratch);
        uint8_t* key = reinterpret_cast<uint8_t*>(order + nkey);
        row_pattern_keys_kernel<<<(unsigned)((nR + 255) / 256), 256, 0, st>>>(prm.Yobs, prm.g, key);
        row_order_kernel<<<256, SORT_THREADS, 0, st>>>(key, nR, order);
        plan.order = order;
    }
    kern<<<grid, NTHREADS, smem, st>>>(prm, plan);
    note_launch();
    rc = check_cuda(fn, cudaGetLastError());
    if (scratch) {
        const int rc2 = check_cuda(fn, cudaFreeAsync(scratch, st));
        if (rc == LRS_OK) rc = rc2;
    }
    return rc;
}

int sparse_fused_tc_launch(const FusedParams& prm, int K, bool dynamic_tiles, cudaStream_t st) {
    if (!sparse_fused_tc_supported(prm, K))
        return fail_arg("lrs_sparse_step_fused_f32", "tcgen05 engine needs K in {64,128,192,256}, Nit >= 1 and an sm_100 device");
    switch (K) {
        case 64: return launch_tc<64>(prm, dynamic_tiles, st);
        case 128: return launch_tc<128>(prm, dynamic_tiles, st);
        case 192: return launch_tc<192>(prm, dynamic_tiles, st);
        default: return launch_tc<256>(prm, dynamic_tiles, st);
    }
}

#ifdef LRS_DIAGNOSTICS
int tc_timing_read(unsigned long long* out32) {
    return check_cuda("lrs_tc_timing_read", cudaMemcpyFromSymbol(out32, g_tc_timing, sizeof(unsigned long long) * 32));
}
#endif

}  // namespace lrs

#ifdef LRS_DIAGNOSTICS
#include <algorithm>
#include <numeric>
#include <vector>

#include "../../include/lrs_pnp_diag.h"

// Replays on the HOST the tile order a launch with `sms` SMs would use and counts how often every patch of
// [p_begin, p_end) is owned by a valid lane (must be exactly once); idle lanes must point at a patch of the matrix.
// row_obs_host (R bytes, or null: ascending row starts) gives the observed rows of the table mode's row-pattern order,
// which is returned in order_host (nR ints) when that is not null.
static int tile_walk_replay(const char* fn, int64_t R, int64_t C, int bb, int s, int64_t p_begin, int64_t p_end, int sms,
                            const uint8_t* row_obs_host, int* visits_host, int64_t* tiles_host, int* order_host) {
    lrs::FusedParams prm{};
    if (bb != 8 || !lrs::make_geom(R, C, bb, s, prm.g)) return lrs::fail_arg(fn, "need bb = 8 and a valid geometry");
    if (p_begin < 0 || p_end > prm.g.P || p_begin >= p_end || sms < 1 || !visits_host || !tiles_host)
        return lrs::fail_arg(fn, "bad range, sms or null pointer");
    prm.p_begin = p_begin;
    prm.p_end = p_end;
    lrs::TilePlan plan = lrs::make_tile_plan(prm, sms);
    std::vector<int> order;
    if (row_obs_host) {
        const int64_t nR = prm.g.row.n;
        std::vector<uint8_t> key(nR);
        for (int64_t ri = 0; ri < nR; ++ri) {
            uint32_t w = 0;
            for (int i = 0; i < 8; ++i) w |= (row_obs_host[prm.g.row.start(ri) + i] ? 1u : 0u) << i;
            key[ri] = (uint8_t)lrs::pattern_rank(w);
        }
        order.resize(nR);
        std::iota(order.begin(), order.end(), 0);
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key[a] < key[b]; });
        if (order_host) std::copy(order.begin(), order.end(), order_host);
        plan.order = order.data();
    }
    const int64_t grid = plan.items < sms ? plan.items : sms;
    int64_t tiles = 0;
    for (int64_t cta = 0; cta < grid; ++cta) {
        for (lrs::TileWalk tw(cta, grid); tw.next(plan, prm); ++tiles) {
            for (int m = 0; m < lrs::TILE; ++m) {
                const lrs::PatchRef pr = lrs::tile_patch(prm, plan, tw, m);
                if (pr.valid) ++visits_host[pr.pi];
                if (pr.p < 0 || pr.p >= prm.g.P || pr.rs < 0 || pr.rs + bb > R || pr.cs < 0 || pr.cs + bb > C)
                    return lrs::fail_arg(fn, "a lane points outside the matrix");
            }
        }
    }
    *tiles_host = tiles;
    return LRS_OK;
}

extern "C" int lrs_debug_tile_walk(int64_t R, int64_t C, int bb, int s, int64_t p_begin, int64_t p_end, int sms,
                                   int* visits_host, int64_t* tiles_host) {
    return tile_walk_replay("lrs_debug_tile_walk", R, C, bb, s, p_begin, p_end, sms, nullptr, visits_host, tiles_host,
                            nullptr);
}

extern "C" int lrs_debug_tile_walk_ordered(int64_t R, int64_t C, int bb, int s, int64_t p_begin, int64_t p_end, int sms,
                                           const uint8_t* row_obs_host, int* visits_host, int64_t* tiles_host,
                                           int* order_host) {
    const char* fn = "lrs_debug_tile_walk_ordered";
    if (!row_obs_host) return lrs::fail_arg(fn, "null row mask");
    return tile_walk_replay(fn, R, C, bb, s, p_begin, p_end, sms, row_obs_host, visits_host, tiles_host, order_host);
}

extern "C" int lrs_tc_timing_read(unsigned long long* out32_host) {
    if (!out32_host) return lrs::fail_arg("lrs_tc_timing_read", "null pointer");
    return lrs::tc_timing_read(out32_host);
}
#endif  // LRS_DIAGNOSTICS
