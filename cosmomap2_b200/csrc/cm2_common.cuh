// cosmomap2_b200 -- shared device/host helpers for the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/cosmomap2_b200.h"

namespace cm2 {

// ---- host side --------------------------------------------------------------------------
int set_error(int code, const char *fmt, ...);
void count_launch(int n = 1);
int sm_count();

#define CM2_REQUIRE(cond, msg)                                                     \
    do {                                                                           \
        if (!(cond)) return cm2::set_error(CM2_ERR_ARG, "%s: %s", __func__, msg);  \
    } while (0)

#define CM2_CUDA(call)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess)                                                               \
            return cm2::set_error(CM2_ERR_CUDA, "%s: %s", __func__, cudaGetErrorString(e__)); \
    } while (0)

#define CM2_LAUNCHED()                                                                        \
    do {                                                                                      \
        cm2::count_launch();                                                                  \
        cudaError_t e__ = cudaGetLastError();                                                 \
        if (e__ != cudaSuccess)                                                               \
            return cm2::set_error(CM2_ERR_CUDA, "%s: %s", __func__, cudaGetErrorString(e__)); \
    } while (0)

static inline bool aligned(const void *p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }
static inline cudaStream_t as_stream(cm2_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int64_t cdiv(int64_t n, int64_t d) { return (n + d - 1) / d; }

// grid of a grid-stride kernel with `ctas` CTAs of work: at least 1, at most per_sm per SM and at most max_ctas
static inline int capped_grid(int64_t ctas, int per_sm, int64_t max_ctas = INT64_MAX) {
    int64_t cap = (int64_t)sm_count() * per_sm;
    if (cap > max_ctas) cap = max_ctas;
    if (ctas > cap) ctas = cap;
    return (int)(ctas < 1 ? 1 : ctas);
}

// grid for a persistent grid-stride kernel: a multiple of the SM count
template <class Kernel>
static inline int persistent_grid(Kernel k, int block, size_t smem, int64_t work_blocks, int max_per_sm = 8) {
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, block, smem);
    return capped_grid(work_blocks, per_sm < 1 ? 1 : (per_sm > max_per_sm ? max_per_sm : per_sm));
}

// f(std::integral_constant<int, P>{}) for P = pol; any pol other than 1 or 2 runs P = 3, so callers check pol first
template <class F>
static inline auto with_pol(int pol, F f) {
    if (pol == 1) return f(std::integral_constant<int, 1>{});
    if (pol == 2) return f(std::integral_constant<int, 2>{});
    return f(std::integral_constant<int, 3>{});
}

// f(std::integral_constant<int, NK>{}) for NK = nk Legendre coefficients; any nk outside 2..4 runs NK = 5
template <class F>
static inline auto with_nk(int nk, F f) {
    switch (nk) {
        case 2: return f(std::integral_constant<int, 2>{});
        case 3: return f(std::integral_constant<int, 3>{});
        case 4: return f(std::integral_constant<int, 4>{});
        default: return f(std::integral_constant<int, 5>{});
    }
}

// one counted kernel launch; returns CM2_OK or the launch error
template <class... Params, class... Args>
static inline int launch(void (*kern)(Params...), int grid, int block, size_t smem, cudaStream_t st, Args... args) {
    kern<<<grid, block, smem, st>>>(args...);
    CM2_LAUNCHED();
    return CM2_OK;
}

// zero fill of n entries of nv 8-byte values (e.g. the map a scatter-add accumulates into)
static inline cudaError_t zero_fill(void *y, int64_t n, int nv, cudaStream_t st) {
    return n > 0 ? cudaMemsetAsync(y, 0, sizeof(double) * (size_t)n * nv, st) : cudaSuccess;
}

// ---- device side: streaming loads/stores (TOD is read once: keep it out of the way of the
// L2-resident map) --------------------------------------------------------------------------
#ifdef __CUDACC__
struct alignas(32) I8 { int v[8]; };
struct alignas(32) D4 { double v[4]; };

// 256-bit global loads (LDG.E.256, sm_100+), L1 no-allocate, L2 evict-first
__device__ __forceinline__ I8 ld_stream_i8(const int32_t *p) {
    I8 r;
    asm volatile("ld.global.L1::no_allocate.L2::evict_first.v8.s32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]),
                   "=r"(r.v[6]), "=r"(r.v[7])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ D4 ld_stream_d4(const double *p) {
    D4 r;
    asm volatile("ld.global.L1::no_allocate.L2::evict_first.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3])
                 : "l"(p));
    return r;
}
// same, but leave the line in L2 for a second pass of the same CTA (fused filter kernel)
__device__ __forceinline__ I8 ld_keep_i8(const int32_t *p) {
    I8 r;
    asm volatile("ld.global.L1::no_allocate.v8.s32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]),
                   "=r"(r.v[6]), "=r"(r.v[7])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ D4 ld_keep_d4(const double *p) {
    D4 r;
    asm volatile("ld.global.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                 : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream_d4(double *p, const D4 &v) {
    asm volatile("st.global.L1::no_allocate.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v.v[0]), "d"(v.v[1]),
                 "d"(v.v[2]), "d"(v.v[3])
                 : "memory");
}
// scalar tail loads: the .L2::evict_first priority form only exists for the 256-bit vectors
__device__ __forceinline__ int ld_stream_i1(const int32_t *p) { return __ldcs(p); }
__device__ __forceinline__ double ld_stream_d1(const double *p) { return __ldcs(p); }

// index of the last entry <= key in the ascending table[0..n), 0 when there is none
__device__ __forceinline__ int64_t last_le(const int64_t *table, int64_t n, int64_t key) {
    int64_t lo = 0, hi = n;
    while (hi - lo > 1) {
        int64_t mid = (lo + hi) >> 1;
        if (table[mid] <= key) lo = mid; else hi = mid;
    }
    return lo;
}

// (P x)_t of one sample from its pixel's POL map values xv and cos / sin 2 phi (not read for POL = 1): the one
// expression of the pointing apply (tod_pass.cu) and of the residual PSD loader (toeplitz_fft.cu)
template <int POL>
__device__ __forceinline__ double project(const double (&xv)[POL], double c, double s) {
    if constexpr (POL == 1) return xv[0];
    else if constexpr (POL == 2) return fma(xv[1], s, xv[0] * c);
    else return fma(xv[2], s, fma(xv[1], c, xv[0]));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic block sum: fixed shuffle tree + fixed order over warps.  `red` = 32 doubles smem.
__device__ __forceinline__ double block_sum(double v, double *red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    double t = 0.0;
    if (w == 0) {
        t = lane < nw ? red[lane] : 0.0;
        t = warp_sum(t);
    }
    return t;  // valid in warp 0
}
// z = M_BD r for pixel j: inv[npix][6] holds the upper triangle {a00,a01,a02,a11,a12,a22} of the per-pixel
// inverse block (zeros where the reference's |det| test fails, linearoperators.py:795, 821)
template <int POL>
__device__ __forceinline__ void bd_z(const double *__restrict__ inv, int64_t j, const double (&r)[POL], double (&z)[POL]) {
    if constexpr (POL == 1) {
        z[0] = __ldg(inv + 6 * j) * r[0];
    } else {
        const double2 *b2 = reinterpret_cast<const double2 *>(inv + 6 * j);
        if constexpr (POL == 2) {
            const double2 q1 = __ldg(b2 + 1), q2 = __ldg(b2 + 2);
            z[0] = q1.y * r[0] + q2.x * r[1];
            z[1] = q2.x * r[0] + q2.y * r[1];
        } else {
            const double2 q0 = __ldg(b2), q1 = __ldg(b2 + 1), q2 = __ldg(b2 + 2);
            z[0] = q0.x * r[0] + q0.y * r[1] + q1.x * r[2];
            z[1] = q0.y * r[0] + q1.y * r[1] + q2.x * r[2];
            z[2] = q1.x * r[0] + q2.x * r[1] + q2.y * r[2];
        }
    }
}

// ---- Legendre subscan filter helpers (filter_poly.cu, tod_pass.cu) ------------------------------
// Legendre P_0..P_{NK-1} at x by the three-term recurrence
template <int NK>
__device__ __forceinline__ void legendre(double x, double (&L)[NK]) {
    L[0] = 1.0;
    if constexpr (NK > 1) L[1] = x;
#pragma unroll
    for (int n = 1; n + 1 < NK; ++n) L[n + 1] = ((2 * n + 1) * x * L[n] - n * L[n - 1]) * (1.0 / (n + 1));
}

// c = G^-1 S for the symmetric positive definite NK x NK Gram matrix G (upper triangle packed row by
// row in g), by Cholesky on the diagonally scaled system.  One thread; every loop has compile-time
// bounds so the factor lives in registers.  Returns the smallest pivot of the scaled factorisation
// (1 = orthogonal basis; small = ill-conditioned: the caller then refines, see filter_refine_steps).
template <int NK>
__device__ __forceinline__ double gram_solve(const double *g, const double *S, double (&c)[NK]) {
    double A[NK][NK], dsc[NK], y[NK];
    double minpiv = 1.0;
    {
        int q = 0;
#pragma unroll
        for (int k = 0; k < NK; ++k) {
#pragma unroll
            for (int l = k; l < NK; ++l) { A[k][l] = g[q]; ++q; }
        }
    }
#pragma unroll
    for (int k = 0; k < NK; ++k) dsc[k] = A[k][k] > 0.0 ? rsqrt(A[k][k]) : 0.0;
#pragma unroll
    for (int k = 0; k < NK; ++k) {
#pragma unroll
        for (int l = k; l < NK; ++l) A[k][l] *= dsc[k] * dsc[l];
    }
    // A = R^T R, R upper triangular, stored in place of the upper triangle
#pragma unroll
    for (int k = 0; k < NK; ++k) {
        double piv = A[k][k];
#pragma unroll
        for (int m = 0; m < k; ++m) piv -= A[m][k] * A[m][k];
        minpiv = fmin(minpiv, piv);
        const double rkk = piv > 0.0 ? sqrt(piv) : 0.0;
        const double inv = rkk > 0.0 ? 1.0 / rkk : 0.0;
        A[k][k] = inv;                      // keep 1/r_kk on the diagonal
#pragma unroll
        for (int l = k + 1; l < NK; ++l) {
            double v = A[k][l];
#pragma unroll
            for (int m = 0; m < k; ++m) v -= A[m][k] * A[m][l];
            A[k][l] = v * inv;
        }
    }
#pragma unroll
    for (int k = 0; k < NK; ++k) {          // R^T y = D S
        double v = S[k] * dsc[k];
#pragma unroll
        for (int m = 0; m < k; ++m) v -= A[m][k] * y[m];
        y[k] = v * A[k][k];
    }
#pragma unroll
    for (int k = NK - 1; k >= 0; --k) {     // R z = y ; c = D z
        double v = y[k];
#pragma unroll
        for (int l = k + 1; l < NK; ++l) v -= A[k][l] * c[l];
        c[k] = v * A[k][k];
    }
#pragma unroll
    for (int k = 0; k < NK; ++k) c[k] *= dsc[k];
    return minpiv;
}

// The normal equations square the condition number of the basis.  With the Legendre basis of the
// interval spanned by the unflagged samples the Gram matrix is close to diagonal for any realistic
// flag pattern (pivots 0.3..1); a handful of unflagged samples at scattered positions can make it
// nearly singular.  Below this pivot the fit is corrected by refinement steps on the residual
// (c += G^-1 L^T (d - L c)): each step squares the relative error of the fitted values.
__device__ __forceinline__ int filter_refine_steps(double minpiv) { return minpiv < 1e-3 ? 2 : 0; }

// Deterministic CTA-wide sum of N values per thread: fixed shuffle tree, then warps in order.
// red: NW*N doubles, tot: N doubles of shared memory; tot is valid after the call (barrier inside).
template <int N, int NW>
__device__ __forceinline__ void block_sum_n(const double (&acc)[N], double *red, double *tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const double w = warp_sum(acc[i]);
        if (lane == 0) red[warp * N + i] = w;
    }
    __syncthreads();
    if (threadIdx.x < N) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) t += red[w * N + threadIdx.x];
        tot[threadIdx.x] = t;
    }
    __syncthreads();
}
#endif

}  // namespace cm2
