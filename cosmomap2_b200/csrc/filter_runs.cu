// cosmomap2_b200 -- single-TOD-pass y = P^T F P x for the subscan offset filter (sm_100a).
//
// F = I - Pi, Pi = per-subscan mean over the unflagged samples (FilterLO.mult,
// interfaces/linearoperators.py:129-168), so
//     P^T F P x = P^T P x  -  sum_k mu_k u_k ,   u_k = P^T 1_k ,  mu_k = (u_k . x) / n_k
// where 1_k is the indicator of the unflagged samples of subscan k.  u_k only depends on the
// pointing: it is stored once, run-compressed (a scan crosses a pixel in a run of consecutive
// samples): per run the pixel, the sample count n and sum(cos), sum(sin) -- 28 B per RUN instead of
// 20 B per SAMPLE.  An A-matvec is then
//     k_seg_mean         : CTA per subscan over the run table: mu_k = sum_runs (n I_p + C Q_p + S U_p) / sum n
//     k_amatvec_filter_mu: ONE pass over the TOD (tod_pass.cu): y += P^T (P x - mu_seg(t)) on the
//                          unflagged samples inside subscans -- the fused white kernel with a
//                          per-chunk segment lookup instead of a block-weight lookup.
// (A first version scattered the correction -mu_k u_k from the run table instead; its second RED
// stream cost 0.17 ms at configs[1] size, the mean pre-pass costs a fraction of that.)
// The two-pass kernel in tod_pass.cu (k_amatvec_filter) is kept as the no-extra-memory variant.
#include "cm2_common.cuh"

namespace cm2 {

constexpr int FB = 256;

// flags[t] = 1 where a run of equal pixel starts among the unflagged samples of a segment;
// pix_masked[t] = pix[t] inside segments, -1 elsewhere (pre-filled with -1 by the caller)
__global__ void __launch_bounds__(FB) k_runs_mark(const int32_t *__restrict__ pix, const int64_t *__restrict__ seg_start,
                                                  const int64_t *__restrict__ seg_end, int64_t nseg,
                                                  int32_t *__restrict__ flags, int32_t *__restrict__ pix_masked) {
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t a = seg_start[k], b = seg_end[k];
        for (int64_t t = a + threadIdx.x; t < b; t += FB) {
            const int32_t p = pix[t];
            const int32_t prev = t > a ? pix[t - 1] : -1;
            flags[t] = (p >= 0 && (t == a || prev != p)) ? 1 : 0;
            pix_masked[t] = p;
        }
    }
}

// one thread per run start: walk the run, accumulate (n, sum cos, sum sin); per segment the first
// run index and the number of runs
__global__ void __launch_bounds__(FB) k_runs_fill(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                  const double *__restrict__ sn, int pol,
                                                  const int64_t *__restrict__ seg_start, const int64_t *__restrict__ seg_end,
                                                  int64_t nseg, const int32_t *__restrict__ runidx,
                                                  int32_t *__restrict__ run_pix, double *__restrict__ run_mom,
                                                  int64_t *__restrict__ seg_first, int32_t *__restrict__ seg_nruns) {
    __shared__ int s_first, s_count;
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t a = seg_start[k], b = seg_end[k];
        if (threadIdx.x == 0) { s_first = 0x7fffffff; s_count = 0; }
        __syncthreads();
        for (int64_t t = a + threadIdx.x; t < b; t += FB) {
            const int32_t r = runidx[t];
            if (r < 0) continue;
            const int32_t p = pix[t];
            double n = 0.0, c = 0.0, s = 0.0;
            for (int64_t u = t; u < b && pix[u] == p; ++u) {
                n += 1.0;
                if (pol > 1) { c += cs[u]; s += sn[u]; }
            }
            run_pix[r] = p;
            run_mom[3 * (int64_t)r] = n;
            run_mom[3 * (int64_t)r + 1] = c;
            run_mom[3 * (int64_t)r + 2] = s;
            atomicMin(&s_first, r);
            atomicAdd(&s_count, 1);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            seg_first[k] = s_count > 0 ? s_first : 0;
            seg_nruns[k] = s_count;
        }
        __syncthreads();
    }
}

template <int POL>
__global__ void __launch_bounds__(FB) k_seg_mean(const int32_t *__restrict__ run_pix, const double *__restrict__ run_mom,
                                                 const int64_t *__restrict__ seg_first, const int32_t *__restrict__ seg_nruns,
                                                 int64_t nseg, const double *__restrict__ x, double *__restrict__ mu) {
    __shared__ double red[32];
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t f = seg_first[k];
        const int nr = seg_nruns[k];
        double dsum = 0.0, cnt = 0.0;
        for (int i = threadIdx.x; i < nr; i += FB) {
            const int64_t r = f + i;
            const int32_t p = __ldcs(run_pix + r);
            const double n = __ldcs(run_mom + 3 * r), c = __ldcs(run_mom + 3 * r + 1), s = __ldcs(run_mom + 3 * r + 2);
            const double *xp = x + (int64_t)POL * p;
            if constexpr (POL == 1) dsum = fma(n, __ldg(xp), dsum);
            else if constexpr (POL == 2) dsum = fma(s, __ldg(xp + 1), fma(c, __ldg(xp), dsum));
            else dsum = fma(s, __ldg(xp + 2), fma(c, __ldg(xp + 1), fma(n, __ldg(xp), dsum)));
            cnt += n;
        }
        const double ts = block_sum(dsum, red);
        const double tc = block_sum(cnt, red);
        if (threadIdx.x == 0) mu[k] = tc > 0.0 ? ts / tc : 0.0;
    }
}

// ---- Legendre filter (poly_order >= 1): the same single-TOD-pass scheme ----------------------------
// F_K d = d - sum_k c_k L_k(x_t) on the unflagged samples of a subscan, x_t = -1 + 2 (t - a)/(len - 1)
// (FilterLO.polyfilter, interfaces/linearoperators.py:170-204).  The coefficients are linear in the
// Legendre moments S_l = sum_{unflagged t} L_l(x_t) d_t:  c = W S  with W fixed by the pointing --
// diag(1/||L_k||^2) for a subscan without flags (the reference's non-orthogonal sum, :196-200), the
// inverse Gram matrix of the unflagged rows otherwise (the least-squares fit its QR step amounts to,
// :190-194).  With d = P x the moments come from a run table like the offset filter's, each run carrying
// sum L_l, sum L_l cos, sum L_l sin.  Set-up: k_poly_gram (W and the smallest Cholesky pivot per subscan;
// the host keeps the well-conditioned subscans for this path and sends the others to the per-subscan
// kernel), k_poly_runs_fill.  Per A-matvec: k_poly_seg_coef, then k_amatvec_filter_poly_mu (tod_pass.cu).
__device__ __forceinline__ double seg_step(int64_t len) { return len > 1 ? 2.0 / (double)(len - 1) : 0.0; }

template <int NK>
__global__ void __launch_bounds__(FB) k_poly_gram(const int32_t *__restrict__ pix, const int64_t *__restrict__ seg_start,
                                                  const int64_t *__restrict__ seg_end, int64_t nseg,
                                                  double *__restrict__ W, double *__restrict__ info) {
    constexpr int NG = NK * (NK + 1) / 2;
    __shared__ double red[(FB / 32) * (NG + 1)];
    __shared__ double tot[NG + 1];
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t a = seg_start[k], b = seg_end[k];
        const double step = seg_step(b - a);
        double acc[NG + 1];
#pragma unroll
        for (int i = 0; i <= NG; ++i) acc[i] = 0.0;
        for (int64_t t = a + threadIdx.x; t < b; t += FB) {
            if (pix[t] >= 0) {
                double L[NK];
                legendre<NK>(fma((double)(t - a), step, -1.0), L);
                int q = 0;
#pragma unroll
                for (int r = 0; r < NK; ++r) {
#pragma unroll
                    for (int c = r; c < NK; ++c) { acc[q] = fma(L[r], L[c], acc[q]); ++q; }
                }
                acc[NG] += 1.0;
            }
        }
        block_sum_n<NG + 1, FB / 32>(acc, red, tot);
        if (threadIdx.x == 0) {
            double *Wk = W + k * (NK * NK);
            const double cnt = tot[NG];
            double minpiv = 1.0;
#pragma unroll
            for (int i = 0; i < NK * NK; ++i) Wk[i] = 0.0;
            if (!(cnt > (double)(NK - 1))) {
                minpiv = 0.0;                             // too few samples: the reference skips the subscan (:185-187)
            } else if (cnt == (double)(b - a)) {          // no flag: coefficient of L_k is (L_k . d) / ||L_k||^2
                int q = 0;
#pragma unroll
                for (int r = 0; r < NK; ++r) { Wk[r * NK + r] = 1.0 / tot[q]; q += NK - r; }
            } else {
#pragma unroll
                for (int l = 0; l < NK; ++l) {
                    double e[NK], c[NK];
#pragma unroll
                    for (int r = 0; r < NK; ++r) e[r] = r == l ? 1.0 : 0.0;
                    minpiv = gram_solve<NK>(tot, e, c);
#pragma unroll
                    for (int r = 0; r < NK; ++r) Wk[r * NK + l] = c[r];
                }
            }
            info[2 * k] = cnt;
            info[2 * k + 1] = minpiv;
        }
        __syncthreads();
    }
}

// one thread per run start (runidx >= 0): Legendre-weighted sums of the run
template <int NK>
__global__ void __launch_bounds__(FB) k_poly_runs_fill(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                       const double *__restrict__ sn, int pol,
                                                       const int64_t *__restrict__ seg_start,
                                                       const int64_t *__restrict__ seg_end, int64_t nseg,
                                                       const int32_t *__restrict__ runidx, int32_t *__restrict__ run_pix,
                                                       double *__restrict__ run_mom, int64_t *__restrict__ seg_first,
                                                       int32_t *__restrict__ seg_nruns) {
    __shared__ int s_first, s_count;
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t a = seg_start[k], b = seg_end[k];
        const double step = seg_step(b - a);
        if (threadIdx.x == 0) { s_first = 0x7fffffff; s_count = 0; }
        __syncthreads();
        for (int64_t t = a + threadIdx.x; t < b; t += FB) {
            const int32_t r = runidx[t];
            if (r < 0) continue;
            const int32_t p = pix[t];
            double m1[NK], mc[NK], ms[NK];
#pragma unroll
            for (int i = 0; i < NK; ++i) m1[i] = mc[i] = ms[i] = 0.0;
            for (int64_t u = t; u < b && pix[u] == p; ++u) {
                double L[NK];
                legendre<NK>(fma((double)(u - a), step, -1.0), L);
                const double cu = pol > 1 ? cs[u] : 0.0, su = pol > 1 ? sn[u] : 0.0;
#pragma unroll
                for (int i = 0; i < NK; ++i) {
                    m1[i] += L[i];
                    mc[i] = fma(L[i], cu, mc[i]);
                    ms[i] = fma(L[i], su, ms[i]);
                }
            }
            run_pix[r] = p;
            double *dst = run_mom + (int64_t)r * (3 * NK);
#pragma unroll
            for (int i = 0; i < NK; ++i) { dst[i] = m1[i]; dst[NK + i] = mc[i]; dst[2 * NK + i] = ms[i]; }
            atomicMin(&s_first, r);
            atomicAdd(&s_count, 1);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            seg_first[k] = s_count > 0 ? s_first : 0;
            seg_nruns[k] = s_count;
        }
        __syncthreads();
    }
}

// coef[k][:] = W_k S_k,  S_k[l] = sum over the subscan's runs of (m1_l I_p + mc_l Q_p + ms_l U_p)
template <int POL, int NK>
__global__ void __launch_bounds__(FB) k_poly_seg_coef(const int32_t *__restrict__ run_pix, const double *__restrict__ run_mom,
                                                      const int64_t *__restrict__ seg_first,
                                                      const int32_t *__restrict__ seg_nruns, int64_t nseg,
                                                      const double *__restrict__ W, const double *__restrict__ x,
                                                      double *__restrict__ coef) {
    __shared__ double red[(FB / 32) * NK];
    __shared__ double tot[NK];
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t f = seg_first[k];
        const int nr = seg_nruns[k];
        double S[NK];
#pragma unroll
        for (int l = 0; l < NK; ++l) S[l] = 0.0;
        for (int i = threadIdx.x; i < nr; i += FB) {
            const int64_t r = f + i;
            const int32_t p = __ldcs(run_pix + r);
            const double *m = run_mom + r * (3 * NK);
            const double *xp = x + (int64_t)POL * p;
            if constexpr (POL == 1) {
                const double xi = __ldg(xp);
#pragma unroll
                for (int l = 0; l < NK; ++l) S[l] = fma(__ldcs(m + l), xi, S[l]);
            } else if constexpr (POL == 2) {
                const double xq = __ldg(xp), xu = __ldg(xp + 1);
#pragma unroll
                for (int l = 0; l < NK; ++l) S[l] = fma(__ldcs(m + 2 * NK + l), xu, fma(__ldcs(m + NK + l), xq, S[l]));
            } else {
                const double xi = __ldg(xp), xq = __ldg(xp + 1), xu = __ldg(xp + 2);
#pragma unroll
                for (int l = 0; l < NK; ++l)
                    S[l] = fma(__ldcs(m + 2 * NK + l), xu, fma(__ldcs(m + NK + l), xq, fma(__ldcs(m + l), xi, S[l])));
            }
        }
        block_sum_n<NK, FB / 32>(S, red, tot);
        if (threadIdx.x < NK) {
            const double *Wk = W + k * (NK * NK) + threadIdx.x * NK;
            double c = 0.0;
#pragma unroll
            for (int l = 0; l < NK; ++l) c = fma(Wk[l], tot[l], c);
            coef[k * NK + threadIdx.x] = c;
        }
        __syncthreads();
    }
}

}  // namespace cm2

using namespace cm2;

extern "C" int cm2_filter_runs_mark(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                                    int64_t nt, int32_t *flags, int32_t *pix_masked, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0 && nseg >= 0, "bad sizes");
    cudaStream_t st = as_stream(stream);
    if (nt > 0) {
        CM2_CUDA(cudaMemsetAsync(flags, 0, sizeof(int32_t) * (size_t)nt, st));
        CM2_CUDA(cudaMemsetAsync(pix_masked, 0xff, sizeof(int32_t) * (size_t)nt, st));   // -1 everywhere
    }
    if (nt == 0 || nseg == 0) return CM2_OK;
    return launch(k_runs_mark, capped_grid(nseg, 8), FB, 0, st, pix, seg_start, seg_end, nseg, flags, pix_masked);
}

extern "C" int cm2_filter_runs_fill(const int32_t *pix, const double *c, const double *s, int pol,
                                    const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                                    const int32_t *runidx, int32_t *run_pix, double *run_mom, int64_t *seg_first,
                                    int32_t *seg_nruns, cm2_stream_t stream) {
    CM2_REQUIRE(nseg >= 0 && pol >= 1 && pol <= 3, "bad sizes");
    if (nseg == 0) return CM2_OK;
    return launch(k_runs_fill, capped_grid(nseg, 8), FB, 0, as_stream(stream), pix, c, s, pol, seg_start, seg_end, nseg,
                  runidx, run_pix, run_mom, seg_first, seg_nruns);
}

extern "C" int cm2_filter_seg_mean(const int32_t *run_pix, const double *run_mom, const int64_t *seg_first,
                                   const int32_t *seg_nruns, int64_t nseg, int pol, const double *x, double *mu,
                                   cm2_stream_t stream) {
    CM2_REQUIRE(nseg >= 0 && pol >= 1 && pol <= 3, "bad sizes");
    if (nseg == 0) return CM2_OK;
    const int g = capped_grid(nseg, 8);
    return with_pol(pol, [&](auto P) {
        return launch(k_seg_mean<P>, g, FB, 0, as_stream(stream), run_pix, run_mom, seg_first, seg_nruns, nseg, x, mu);
    });
}

/* ---- Legendre variant of the run table (poly_order 1..4) --------------------------------------- */
extern "C" int cm2_filter_poly_gram(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                                    int poly_order, double *W, double *info, cm2_stream_t stream) {
    CM2_REQUIRE(nseg >= 0, "bad sizes");
    if (poly_order < 1 || poly_order > 4)
        return set_error(CM2_ERR_UNSUPPORTED, "run-table Legendre filter: poly_order=%d, orders 1..4 are supported", poly_order);
    if (nseg == 0) return CM2_OK;
    const int g = capped_grid(nseg, 8);
    return with_nk(poly_order + 1, [&](auto NK) {
        return launch(k_poly_gram<NK>, g, FB, 0, as_stream(stream), pix, seg_start, seg_end, nseg, W, info);
    });
}

extern "C" int cm2_filter_poly_runs_fill(const int32_t *pix, const double *c, const double *s, int pol,
                                         const int64_t *seg_start, const int64_t *seg_end, int64_t nseg, int poly_order,
                                         const int32_t *runidx, int32_t *run_pix, double *run_mom, int64_t *seg_first,
                                         int32_t *seg_nruns, cm2_stream_t stream) {
    CM2_REQUIRE(nseg >= 0 && pol >= 1 && pol <= 3, "bad sizes");
    if (poly_order < 1 || poly_order > 4)
        return set_error(CM2_ERR_UNSUPPORTED, "run-table Legendre filter: poly_order=%d, orders 1..4 are supported", poly_order);
    if (nseg == 0) return CM2_OK;
    const int g = capped_grid(nseg, 8);
    return with_nk(poly_order + 1, [&](auto NK) {
        return launch(k_poly_runs_fill<NK>, g, FB, 0, as_stream(stream), pix, c, s, pol, seg_start, seg_end, nseg, runidx,
                      run_pix, run_mom, seg_first, seg_nruns);
    });
}

extern "C" int cm2_filter_poly_seg_coef(const int32_t *run_pix, const double *run_mom, const int64_t *seg_first,
                                        const int32_t *seg_nruns, int64_t nseg, int pol, int poly_order, const double *W,
                                        const double *x, double *coef, cm2_stream_t stream) {
    CM2_REQUIRE(nseg >= 0 && pol >= 1 && pol <= 3, "bad sizes");
    if (poly_order < 1 || poly_order > 4)
        return set_error(CM2_ERR_UNSUPPORTED, "run-table Legendre filter: poly_order=%d, orders 1..4 are supported", poly_order);
    if (nseg == 0) return CM2_OK;
    const int g = capped_grid(nseg, 8);
    return with_pol(pol, [&](auto P) {
        return with_nk(poly_order + 1, [&](auto NK) {
            return launch(k_poly_seg_coef<P, NK>, g, FB, 0, as_stream(stream), run_pix, run_mom, seg_first, seg_nruns, nseg,
                          W, x, coef);
        });
    });
}
