// Shared helpers for liblrs_pnp.so (sm_100a).  See include/lrs_pnp.h for the ABI contract.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "../../include/lrs_pnp.h"

namespace lrs {

void set_error(const std::string& msg);
int fail_arg(const char* fn, const char* what);
int check_cuda(const char* fn, cudaError_t e);
int device_sm_count();
void note_launch();  // counts kernel launches (lrs_launch_count)

#define LRS_CHECK_LAUNCH(fn)                                  \
    do {                                                      \
        ::lrs::note_launch();                                 \
        int _rc = ::lrs::check_cuda(fn, cudaGetLastError());  \
        if (_rc != LRS_OK) return _rc;                        \
    } while (0)

// One axis of get_image_block's selection (main_LRS_PnP.py:76-91): starts 0, s, 2s, ... <= len-bb,
// plus the last start len-bb iff len % bb != 0.  start(i) = min(i*s, len-bb) covers both.
struct Axis {
    int64_t len;
    int64_t last;   // len - bb
    int64_t n_reg;  // number of stride starts
    int64_t n;      // n_reg (+1 if the last start was appended)
    int bb;
    int s;

    __host__ __device__ __forceinline__ int64_t start(int64_t i) const {
        int64_t v = i * (int64_t)s;
        return v < last ? v : last;
    }
    // Range of regular start indices covering position x, [lo, hi]; appended start covers x iff
    // has_app() && x >= last.
    __host__ __device__ __forceinline__ void cover(int64_t x, int64_t& lo, int64_t& hi, bool& app) const {
        if (len <= 0x7fffffffLL) {  // 32-bit divisions (a 64-bit one is a ~100-instruction subroutine)
            const int xi = (int)x, t = xi - bb + 1, nr = (int)n_reg;
            const int l = t <= 0 ? 0 : (s == 1 ? t : (t + s - 1) / s), h = s == 1 ? xi : xi / s;
            lo = l;
            hi = h > nr - 1 ? nr - 1 : h;
        } else {
            int64_t t = x - bb + 1;
            lo = t <= 0 ? 0 : (t + s - 1) / s;
            hi = x / s;
            if (hi > n_reg - 1) hi = n_reg - 1;
        }
        app = (n > n_reg) && (x >= last);
    }
    __host__ __device__ __forceinline__ int count(int64_t x) const {
        if (len <= 0x7fffffffLL) {  // 32-bit arithmetic: the elementwise kernels call this per element
            const int xi = (int)x, t = xi - bb + 1, nr = (int)n_reg;
            int lo = t <= 0 ? 0 : (s == 1 ? t : (t + s - 1) / s), hi = s == 1 ? xi : xi / s;
            if (hi > nr - 1) hi = nr - 1;
            int c = hi - lo + 1;
            if (c < 0) c = 0;
            return c + (((n > n_reg) && (x >= last)) ? 1 : 0);
        }
        int64_t lo, hi;
        bool app;
        cover(x, lo, hi, app);
        int64_t c = hi - lo + 1;
        if (c < 0) c = 0;
        return (int)c + (app ? 1 : 0);
    }
};

inline bool make_axis(int64_t len, int bb, int s, Axis& a) {
    if (bb <= 0 || s <= 0 || len < bb) return false;
    a.len = len;
    a.bb = bb;
    a.s = s;
    a.last = len - bb;
    a.n_reg = a.last / s + 1;
    bool app = (len % bb) != 0 && ((a.n_reg - 1) * (int64_t)s != a.last);
    a.n = a.n_reg + (app ? 1 : 0);
    return true;
}

struct Geom {
    Axis row, col;
    int64_t R, C, P;
    int bb, n;
};

inline bool make_geom(int64_t R, int64_t C, int bb, int s, Geom& g) {
    if (!make_axis(R, bb, s, g.row) || !make_axis(C, bb, s, g.col)) return false;
    g.R = R;
    g.C = C;
    g.bb = bb;
    g.n = bb * bb;
    g.P = g.row.n * g.col.n;
    return true;
}

__device__ __forceinline__ float soft_thr(float x, float tau) {
    // sign(x)*max(|x|-tau,0)   (soft.m:4)
    return copysignf(fmaxf(__fsub_rn(fabsf(x), tau), 0.0f), x);
}

// Arguments of the fused sparse step (lrs_sparse_step_fused_f32), shared by both engines.
struct FusedParams {
    Geom g;
    const float* X;
    const float* L;
    const float* Yobs;
    const float* D;
    const float* a_patch;
    const float* a_table;
    float mu1, lambda;
    int Nit;
    int64_t p_begin, p_end;
    float* phi;
};

// ista_tc.cu: tensor-core engine of the explicit ISTA path (large patches, P <= 256)
bool ista_tc_shape_ok(int n, int K, int64_t P);
bool ista_tc_enabled();
size_t ista_tc_workspace_bytes(int n, int K, int64_t P);
int ista_tc_run(const float* blocks, const float* blocks_copy, const float* D, const float* a, float lambda, int Nit, int n,
                int K, int64_t P, int denoiser, float h_scale, float* coefs, float* phi, void* ws, size_t ws_bytes,
                cudaStream_t st);
// ista_generic.cu: split-K count and rows per CTA of the FFMA engine's GEMMs (M x N output, Kd deep)
int ista_splits(int64_t M, int64_t N, int64_t Kd);
int ista_row_tile(int64_t M, int64_t N, int splits, int sms);
// ista_generic.cu: A = NLmeansfilter(G, 3, 3, h_scale * T) column by column (NLmeansfilter.m:18-91)
int nlm_columns(const char* fn, const float* G, const float* T, float h_scale, int K, int64_t P, float* A, cudaStream_t st);

int sparse_fused_tc_launch(const FusedParams& prm, int K, bool dynamic_tiles, cudaStream_t st);  // sparse_fused_tc.cu
bool sparse_fused_tc_supported(const FusedParams& prm, int K);

}  // namespace lrs
