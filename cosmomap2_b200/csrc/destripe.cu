// cosmomap2_b200 -- the destriper operator over the run-compressed pointing (sm_100a), DESIGN.md section 4f.
//
// Baselines j (L samples, never straddling a noise block) carry an offset a_j spread over their unflagged samples by
// F.  With u_j = P^T 1_j kept run-compressed exactly as the subscan filter keeps it (filter_runs.cu: run_pix[r],
// run_mom[r] = {n, sum cos, sum sin}, baseline j = runs base_first[j] .. + base_nruns[j]) the destriper operator
//     (F^T W Z F + C_a^-1) a,   Z = I - P M_BD P^T W,   W = w_b per noise block
// is, with bw_j = w_b of baseline j's block and n_j its unflagged samples,
//     y   = sum_j bw_j a_j u_j                  k_base_scatter (RED per run)
//     m   = M_BD y                              cm2_bd_apply
//     q_j = bw_j (n_j a_j - u_j . m) + (C_a^-1 a)_j   k_base_dot (fixed-order sum per baseline)
// and never touches the TOD.  A baseline holds a handful of runs, so both kernels give each baseline a group of G
// lanes of a warp (G = 4 .. 32, chosen by the caller from the mean runs per baseline) rather than one CTA per
// segment as k_seg_mean does.
#include "cm2_common.cuh"

namespace cm2 {

constexpr int DB = 256;

// u_j . v for run r: n v_I + c v_Q + s v_U for the components POL has
template <int POL>
__device__ __forceinline__ double run_dot(const double *__restrict__ run_mom, int64_t r, const double *__restrict__ vp,
                                          double &n) {
    n = __ldcs(run_mom + 3 * r);
    if constexpr (POL == 1) return n * __ldg(vp);
    const double c = __ldcs(run_mom + 3 * r + 1), s = __ldcs(run_mom + 3 * r + 2);
    if constexpr (POL == 2) return fma(s, __ldg(vp + 1), c * __ldg(vp));
    else return fma(s, __ldg(vp + 2), fma(c, __ldg(vp + 1), n * __ldg(vp)));
}

// sum over the G lanes of a group (aligned lanes of one warp): a fixed xor tree, so the same bits every call
template <int G>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// y[POL p] += alpha bw_j c_j u_j for every run of every baseline j (bw NULL: 1)
template <int POL, int G>
__global__ void __launch_bounds__(DB) k_base_scatter(const int32_t *__restrict__ run_pix, const double *__restrict__ run_mom,
                                                     const int64_t *__restrict__ base_first,
                                                     const int32_t *__restrict__ base_nruns, int64_t nbase,
                                                     const double *__restrict__ c, const double *__restrict__ bw,
                                                     double alpha, double *__restrict__ y) {
    const int64_t ngroups = (int64_t)gridDim.x * (DB / G);
    const int lane = threadIdx.x % G;
    for (int64_t j = (int64_t)blockIdx.x * (DB / G) + threadIdx.x / G; j < nbase; j += ngroups) {
        const int nr = base_nruns[j];
        const double cj = alpha * c[j] * (bw ? bw[j] : 1.0);
        if (nr == 0 || cj == 0.0) continue;
        const int64_t f = base_first[j];
        for (int i = lane; i < nr; i += G) {
            const int64_t r = f + i;
            double *yp = y + (int64_t)POL * __ldcs(run_pix + r);
            if constexpr (POL == 1) {
                atomicAdd(yp, cj * __ldcs(run_mom + 3 * r));
            } else {
                const double cs = __ldcs(run_mom + 3 * r + 1), sn = __ldcs(run_mom + 3 * r + 2);
                if constexpr (POL == 3) atomicAdd(yp, cj * __ldcs(run_mom + 3 * r));
                atomicAdd(yp + POL - 2, cj * cs);
                atomicAdd(yp + POL - 1, cj * sn);
            }
        }
    }
}

// out_j = bw_j (n_j a_j - u_j . m) + add_j  (a NULL: 0; add NULL: 0); every lane of a warp runs the same trips
template <int POL, int G>
__global__ void __launch_bounds__(DB) k_base_dot(const int32_t *__restrict__ run_pix, const double *__restrict__ run_mom,
                                                 const int64_t *__restrict__ base_first,
                                                 const int32_t *__restrict__ base_nruns, int64_t nbase,
                                                 const double *__restrict__ bw, const double *__restrict__ a,
                                                 const double *__restrict__ m, const double *__restrict__ add,
                                                 double *__restrict__ out) {
    const int64_t ngroups = (int64_t)gridDim.x * (DB / G);
    const int lane = threadIdx.x % G;
    const int64_t warp_first = (int64_t)blockIdx.x * (DB / G) + (threadIdx.x & ~31) / G;
    for (int64_t jw = warp_first; jw < nbase; jw += ngroups) {
        const int64_t j = jw + (threadIdx.x & 31) / G;
        double um = 0.0, cnt = 0.0;
        if (j < nbase) {
            const int64_t f = base_first[j];
            const int nr = base_nruns[j];
            for (int i = lane; i < nr; i += G) {
                const int64_t r = f + i;
                double n;
                um += run_dot<POL>(run_mom, r, m + (int64_t)POL * __ldcs(run_pix + r), n);
                cnt += n;
            }
        }
        um = group_sum<G>(um);
        cnt = group_sum<G>(cnt);
        if (j < nbase && lane == 0) {
            const double aj = a ? a[j] : 0.0;
            out[j] = fma(bw[j], fma(cnt, aj, -um), add ? add[j] : 0.0);
        }
    }
}

// out_j = bw_j sum of d_t over the unflagged samples (pix_t >= 0) of [base_start[j], base_end[j]): a warp per
// baseline, a fixed-order sum.  A flagged sample is selected away, so NaN in flagged d does not reach the sums.
__global__ void __launch_bounds__(DB) k_base_tod_sums(const int32_t *__restrict__ pix, const double *__restrict__ d,
                                                      const int64_t *__restrict__ base_start,
                                                      const int64_t *__restrict__ base_end, int64_t nbase,
                                                      const double *__restrict__ bw, double *__restrict__ out) {
    const int64_t nwarps = (int64_t)gridDim.x * (DB / 32);
    const int lane = threadIdx.x & 31;
    for (int64_t j = (int64_t)blockIdx.x * (DB / 32) + threadIdx.x / 32; j < nbase; j += nwarps) {
        const int64_t a = base_start[j], b = base_end[j];
        double s = 0.0;
        for (int64_t t = a + lane; t < b; t += 32) {
            const double v = __ldcs(d + t);
            if (__ldcs(pix + t) >= 0) s += v;
        }
        s = warp_sum(s);
        if (lane == 0) out[j] = bw[j] * s;
    }
}

// f(std::integral_constant<int, G>{}) for a group of G = 4, 8, 16 or 32 lanes; callers check g first
template <class F>
static inline auto with_group(int g, F f) {
    switch (g) {
        case 4: return f(std::integral_constant<int, 4>{});
        case 8: return f(std::integral_constant<int, 8>{});
        case 16: return f(std::integral_constant<int, 16>{});
        default: return f(std::integral_constant<int, 32>{});
    }
}

static inline bool good_group(int g) { return g == 4 || g == 8 || g == 16 || g == 32; }

}  // namespace cm2

using namespace cm2;

extern "C" int cm2_destripe_scatter(const int32_t *run_pix, const double *run_mom, const int64_t *base_first,
                                    const int32_t *base_nruns, int64_t nbase, int pol, int group, const double *c,
                                    const double *bw, double alpha, double *y, int64_t npix, int accumulate,
                                    cm2_stream_t stream) {
    CM2_REQUIRE(nbase >= 0 && npix >= 0 && pol >= 1 && pol <= 3, "bad sizes");
    CM2_REQUIRE(good_group(group), "group must be 4, 8, 16 or 32 lanes");
    cudaStream_t st = as_stream(stream);
    if (!accumulate) CM2_CUDA(zero_fill(y, npix, pol, st));
    if (nbase == 0) return CM2_OK;
    CM2_REQUIRE(run_pix && run_mom && base_first && base_nruns && c && y, "NULL table or vector");
    return with_pol(pol, [&](auto P) {
        return with_group(group, [&](auto G) {
            return launch(k_base_scatter<P, G>, capped_grid(cdiv(nbase, DB / G), 8), DB, 0, st, run_pix, run_mom,
                          base_first, base_nruns, nbase, c, bw, alpha, y);
        });
    });
}

extern "C" int cm2_destripe_dot(const int32_t *run_pix, const double *run_mom, const int64_t *base_first,
                                const int32_t *base_nruns, int64_t nbase, int pol, int group, const double *bw,
                                const double *a, const double *m, const double *add, double *out, cm2_stream_t stream) {
    CM2_REQUIRE(nbase >= 0 && pol >= 1 && pol <= 3, "bad sizes");
    CM2_REQUIRE(good_group(group), "group must be 4, 8, 16 or 32 lanes");
    if (nbase == 0) return CM2_OK;
    CM2_REQUIRE(run_pix && run_mom && base_first && base_nruns && bw && m && out, "NULL table or vector");
    return with_pol(pol, [&](auto P) {
        return with_group(group, [&](auto G) {
            return launch(k_base_dot<P, G>, capped_grid(cdiv(nbase, DB / G), 8), DB, 0, as_stream(stream), run_pix,
                          run_mom, base_first, base_nruns, nbase, bw, a, m, add, out);
        });
    });
}

extern "C" int cm2_destripe_tod_sums(const int32_t *pix, const double *d, const int64_t *base_start,
                                     const int64_t *base_end, int64_t nbase, const double *bw, double *out,
                                     cm2_stream_t stream) {
    CM2_REQUIRE(nbase >= 0, "bad sizes");
    if (nbase == 0) return CM2_OK;
    CM2_REQUIRE(pix && d && base_start && base_end && bw && out, "NULL table or vector");
    return launch(k_base_tod_sums, capped_grid(cdiv(nbase, DB / 32), 8), DB, 0, as_stream(stream), pix, d, base_start,
                  base_end, nbase, bw, out);
}
