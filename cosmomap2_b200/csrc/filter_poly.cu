// cosmomap2_b200 -- SURVEY 8(f) rows either side of the solve (sm_100a):
//
//   cm2_filter_poly_apply     subscan filter, one CTA per subscan, the subscan staged in shared memory
//                             poly_order = 0 : offset removal        (FilterLO.mult       linearoperators.py:129-168)
//                             poly_order > 0 : Legendre polynomials  (FilterLO.polyfilter linearoperators.py:170-204)
//   cm2_ground_filter_apply   v - G (G^T G)^-1 G^T v over ground bins (GroundFilterLO     linearoperators.py:24-61)
//   cm2_reorganize_map        interleaved cut-sky solution -> full-sky HEALPix arrays
//                                                                    (reorganize_map      healpy_functions.py:50-105)
//
// The subscan filter reads d and pix ONCE (12 B/sample) and writes out once (8 B/sample): the samples
// of a subscan wait in shared memory between the reduction pass and the subtraction pass, and the
// CTA of subscan k also zero-fills the gap in front of it, so no memset of the output is needed.
#include <climits>

#include "cm2_common.cuh"

namespace cm2 {

constexpr int FB = 256;          // threads per CTA
constexpr int FP_MAXNK = 8;      // poly_order <= 7

// ---- mbarrier + 1-D bulk copy (TMA engine, UBLKCP) ------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completes on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    uint32_t spins = 0;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
        if (!done && ++spins > (1u << 24)) __trap();      // a lost copy becomes an error, never a hang
    } while (!done);
}

// Shared-memory scratch of one CTA for filter_segment
template <int NK, bool OFFSET, int NT>
struct FilterScratch {
    static constexpr int NG = OFFSET ? 0 : NK * (NK + 1) / 2;
    static constexpr int NR = NK + NG;
    double red[(NT / 32) * NR > 32 ? (NT / 32) * NR : 32];
    double tot[NR];
    double coef[NK];
    int cnt, jmin, jmax, skip, refine;
};

// One subscan [a, a+len) by the NT threads of a CTA.  getd(j) / getf(j) return sample j of the subscan
// and whether it is unflagged (from shared memory, or global memory beyond the staged window).
// NK = poly_order + 1.  OFFSET (NK == 1): the reference's poly_order = 0 path, where the mean over
// the unflagged (pix != -1) samples is subtracted from EVERY sample of the subscan (:165).
// Otherwise the Legendre path: unflagged = pix >= 0 (:174); a subscan with <= poly_order unflagged
// samples is skipped (:185-187); without flags p = sum_k (b_k . d) b_k with b_k = L_k/||L_k|| on the
// full grid (:196-200, NOT an exact projector: the sampled L_k are not orthogonal); with flags the
// basis is re-orthonormalised by QR on the unflagged rows (:190-194), i.e. p is the least-squares
// polynomial of degree <= poly_order -- computed here from the Gram matrix in the Legendre basis of
// the interval spanned by the unflagged samples (same span, well conditioned); flagged samples -> 0.
// fill != 0: every sample of the subscan is written (zeros where the reference leaves the
// zero-initialised output untouched); fill == 0: only what the reference assigns is written.
// Ends with a CTA barrier (the staged window may be reused afterwards).
template <int NK, bool OFFSET, int NT, class GetD, class GetF>
__device__ __forceinline__ void filter_segment(GetD getd, GetF getf, int64_t a, int64_t len64, double *__restrict__ out,
                                               int fill, FilterScratch<NK, OFFSET, NT> &sh) {
    constexpr int NR = FilterScratch<NK, OFFSET, NT>::NR;
    constexpr int NW = NT / 32;
    const int tid = threadIdx.x, lane = tid & 31;
    const int len = len64 > 0 ? (int)len64 : 0;          // subscans are shorter than 2^31 samples (checked on the host)
    double *__restrict__ oa = out + a;
    if (tid == 0) { sh.cnt = 0; sh.jmin = INT_MAX; sh.jmax = -1; }
    __syncthreads();
    // ---- pass 1: count, first / last unflagged sample, (offset path) sum ------------------------
    int cnt = 0, jmin = INT_MAX, jmax = -1;
    double sum = 0.0;
#pragma unroll 4
    for (int j = tid; j < len; j += NT) {
        if (getf(j)) {
            ++cnt;
            jmin = min(jmin, j);
            jmax = j;
            if (OFFSET) sum += getd(j);
        }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    jmin = __reduce_min_sync(0xffffffffu, jmin);
    jmax = __reduce_max_sync(0xffffffffu, jmax);
    if (lane == 0 && cnt > 0) { atomicAdd(&sh.cnt, cnt); atomicMin(&sh.jmin, jmin); atomicMax(&sh.jmax, jmax); }
    if constexpr (OFFSET) {
        const double tsum = block_sum(sum, sh.red);      // two barriers inside: sh.cnt is complete after it
        if (tid == 0) {
            const double mean = tsum / (double)sh.cnt;    // 0/0 = NaN like the reference (:154, 163)
            sh.skip = (sh.cnt == 0) || isinf(mean) || isnan(mean);
            sh.coef[0] = mean;
        }
        __syncthreads();
        const double mu = sh.coef[0];
        if (!sh.skip) {
#pragma unroll 4
            for (int j = tid; j < len; j += NT) __stcs(oa + j, getd(j) - mu);
        } else if (fill) {
            for (int j = tid; j < len; j += NT) __stcs(oa + j, 0.0);
        }
    } else {
        __syncthreads();
        const int n = sh.cnt;
        if (n <= NK - 1) {                                // block-uniform: too few samples (:185-187)
            if (fill)
                for (int j = tid; j < len; j += NT) __stcs(oa + j, 0.0);
        } else {
            const bool full = n == len;
            const int j0 = full ? 0 : sh.jmin;
            const int j1 = full ? len - 1 : sh.jmax;
            const double step = 2.0 / (double)(j1 - j0);
            // x_j of this thread's m-th sample (j = tid + m NT): x0 + m dx, one fma instead of an int -> fp64
            // conversion per sample
            const double x0 = fma((double)(tid - j0), step, -1.0), dx = (double)NT * step;
            // ---- pass 2: S_k = sum L_k d and the Gram matrix over the unflagged samples -------------
            double acc[NR];
#pragma unroll
            for (int i = 0; i < NR; ++i) acc[i] = 0.0;
            if (full) {                                  // no flag: only the diagonal ||L_k||^2 is needed
                double m = 0.0;
#pragma unroll 2
                for (int j = tid; j < len; j += NT, m += 1.0) {
                    const double v = getd(j);
                    double L[NK];
                    legendre<NK>(fma(m, dx, x0), L);
                    int q = NK;
#pragma unroll
                    for (int r = 0; r < NK; ++r) {
                        acc[r] = fma(L[r], v, acc[r]);
                        acc[q] = fma(L[r], L[r], acc[q]);
                        q += NK - r;
                    }
                }
            } else {
                double m = 0.0;
#pragma unroll 2
                for (int j = tid; j < len; j += NT, m += 1.0) {
                    const bool f = getf(j);
                    const double v = getd(j);
                    double L[NK], Lw[NK];
                    legendre<NK>(fma(m, dx, x0), L);
#pragma unroll
                    for (int r = 0; r < NK; ++r) Lw[r] = f ? L[r] : 0.0;    // branch-free: flagged samples add 0
                    int q = NK;
#pragma unroll
                    for (int r = 0; r < NK; ++r) {
                        acc[r] = fma(Lw[r], v, acc[r]);
#pragma unroll
                        for (int c = r; c < NK; ++c) { acc[q] = fma(Lw[r], L[c], acc[q]); ++q; }
                    }
                }
            }
            block_sum_n<NR, NW>(acc, sh.red, sh.tot);
            if (tid == 0) {
                sh.refine = 0;
                if (full) {
                    int q = NK;
                    for (int r = 0; r < NK; ++r) {
                        sh.coef[r] = sh.tot[q] > 0.0 ? sh.tot[r] / sh.tot[q] : 0.0;   // (b_k . d) / ||L_k||^2
                        q += NK - r;
                    }
                } else {
                    double c[NK];
                    sh.refine = filter_refine_steps(gram_solve<NK>(sh.tot + NK, sh.tot, c));
                    for (int r = 0; r < NK; ++r) sh.coef[r] = c[r];
                }
            }
            __syncthreads();
            const int nref = sh.refine;                   // block-uniform, 0 unless ill-conditioned
            for (int it = 0; it < nref; ++it) {
                double c[NK], racc[NK];
#pragma unroll
                for (int r = 0; r < NK; ++r) { c[r] = sh.coef[r]; racc[r] = 0.0; }
                double m = 0.0;
                for (int j = tid; j < len; j += NT, m += 1.0) {
                    if (!getf(j)) continue;
                    double L[NK];
                    legendre<NK>(fma(m, dx, x0), L);
                    double res = getd(j);
#pragma unroll
                    for (int r = 0; r < NK; ++r) res = fma(-c[r], L[r], res);
#pragma unroll
                    for (int r = 0; r < NK; ++r) racc[r] = fma(L[r], res, racc[r]);
                }
                block_sum_n<NK, NW>(racc, sh.red, sh.tot);    // tot[0..NK) = L^T (d - L c); the Gram matrix stays
                if (tid == 0) {
                    double dc[NK];
                    gram_solve<NK>(sh.tot + NK, sh.tot, dc);
                    for (int r = 0; r < NK; ++r) sh.coef[r] += dc[r];
                }
                __syncthreads();
            }
            // ---- pass 3: subtract and write ----------------------------------------------------------
            double c[NK];
#pragma unroll
            for (int r = 0; r < NK; ++r) c[r] = sh.coef[r];
            double m = 0.0;
#pragma unroll 2
            for (int j = tid; j < len; j += NT, m += 1.0) {
                const bool f = full || getf(j);
                double L[NK];
                legendre<NK>(fma(m, dx, x0), L);
                double p = 0.0;
#pragma unroll
                for (int r = 0; r < NK; ++r) p = fma(c[r], L[r], p);
                if (f) __stcs(oa + j, getd(j) - p);
                else if (fill) __stcs(oa + j, 0.0);
            }
        }
    }
    __syncthreads();
}

// zero-fill of the gap in front of subscan k (and behind the last one): sorted tables only
template <int NT>
__device__ __forceinline__ void fill_gap(const int64_t *__restrict__ seg_end, int64_t k, int64_t nseg, int64_t a, int64_t b,
                                         int64_t nt, double *__restrict__ out) {
    const int64_t g0 = k == 0 ? 0 : seg_end[k - 1];
    for (int64_t t = g0 + threadIdx.x; t < a; t += NT) __stcs(out + t, 0.0);
    if (k == nseg - 1)
        for (int64_t t = b + threadIdx.x; t < nt; t += NT) __stcs(out + t, 0.0);
}

// ---- variant A: one CTA per subscan, staged by ordinary loads (any subscan length) --------------------
template <int NK, bool OFFSET>
__global__ void __launch_bounds__(FB) k_filter_poly(const int32_t *__restrict__ pix, const int64_t *__restrict__ seg_start,
                                                    const int64_t *__restrict__ seg_end, int64_t nseg,
                                                    const double *__restrict__ d, double *__restrict__ out, int64_t nt,
                                                    int cap, int fill) {
    extern __shared__ double sm[];
    double *sd = sm;                                     // cap staged samples
    uint8_t *sf = reinterpret_cast<uint8_t *>(sm + cap);   // cap flags (1 = unflagged)
    __shared__ FilterScratch<NK, OFFSET, FB> sh;
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t a = seg_start[k], b = seg_end[k];
        const int64_t len = b - a;
        if (fill) fill_gap<FB>(seg_end, k, nseg, a, b, nt, out);
        const int64_t nst = len < cap ? len : cap;
        for (int64_t j = threadIdx.x; j < nst; j += FB) {
            const int p = __ldcs(pix + a + j);
            sd[j] = __ldcs(d + a + j);
            sf[j] = OFFSET ? (p != -1) : (p >= 0);
        }
        __syncthreads();
        if (len <= cap) {                                // block-uniform: the whole subscan is on chip
            filter_segment<NK, OFFSET, FB>([&](int j) { return sd[j]; }, [&](int j) { return sf[j] != 0; }, a, len, out,
                                           fill, sh);
        } else {
            auto getd = [&](int j) { return j < cap ? sd[j] : d[a + j]; };
            auto getf = [&](int j) {
                if (j < cap) return sf[j] != 0;
                const int p = pix[a + j];
                return OFFSET ? (p != -1) : (p >= 0);
            };
            filter_segment<NK, OFFSET, FB>(getd, getf, a, len, out, fill, sh);
        }
    }
}

// ---- variant B: persistent CTAs, subscans streamed through a ring of shared-memory stages by the TMA
// engine (cp.async.bulk + mbarrier): while the CTA reduces and writes subscan i, the copies of
// subscans i+1 .. i+nstage-1 are in flight, so DRAM latency is never exposed.  The copied window is
// the 4-sample-aligned hull [a & ~3, min(roundup4(b), nt & ~3)) of d (8 B) and pix (4 B); the <= 3
// samples of the last subscan beyond nt & ~3 are read directly.
constexpr int TB = 512;
constexpr int TMA_MAX_STAGES = 4;

template <int NK, bool OFFSET>
__global__ void __launch_bounds__(TB, 1) k_filter_poly_tma(const int32_t *__restrict__ pix, const int64_t *__restrict__ seg_start,
                                                           const int64_t *__restrict__ seg_end, int64_t nseg,
                                                           const double *__restrict__ d, double *__restrict__ out, int64_t nt,
                                                           int capw, int nstage, int fill) {
    extern __shared__ __align__(128) unsigned char smraw[];
    __shared__ FilterScratch<NK, OFFSET, TB> sh;
    __shared__ __align__(8) uint64_t full[TMA_MAX_STAGES];
    const size_t stage_bytes = (size_t)capw * 12;
    const int64_t nt4 = nt & ~(int64_t)3;
    if (threadIdx.x == 0) {
        for (int s = 0; s < nstage; ++s) mbar_init(&full[s], 1);
        mbar_init_fence();
    }
    __syncthreads();
    if ((int64_t)blockIdx.x >= nseg) return;
    const int64_t nmine = (nseg - blockIdx.x + gridDim.x - 1) / gridDim.x;
    auto issue = [&](int64_t i) {                          // thread 0: start the copies of my i-th subscan
        const int64_t k = blockIdx.x + i * gridDim.x;
        const int s = (int)(i % nstage);
        const int64_t a = seg_start[k], b = seg_end[k];
        const int64_t a4 = a & ~(int64_t)3;
        int64_t e4 = (b + 3) & ~(int64_t)3;
        if (e4 > nt4) e4 = nt4;
        const int64_t n = e4 > a4 ? e4 - a4 : 0;           // multiple of 4
        unsigned char *base = smraw + s * stage_bytes;
        mbar_arrive_expect_tx(&full[s], (uint32_t)(n * 12));
        if (n > 0) {
            bulk_g2s(base, d + a4, (uint32_t)(n * 8), &full[s]);
            bulk_g2s(base + (size_t)capw * 8, pix + a4, (uint32_t)(n * 4), &full[s]);
        }
    };
    if (threadIdx.x == 0)
        for (int64_t i = 0; i < nstage - 1 && i < nmine; ++i) issue(i);
    for (int64_t i = 0; i < nmine; ++i) {
        const int64_t k = blockIdx.x + i * gridDim.x;
        const int s = (int)(i % nstage);
        // the stage refilled here was read during iteration i-1, which ended with a CTA barrier
        if (threadIdx.x == 0 && i + nstage - 1 < nmine) issue(i + nstage - 1);
        const int64_t a = seg_start[k], b = seg_end[k];
        const int64_t len = b - a;
        if (fill) fill_gap<TB>(seg_end, k, nseg, a, b, nt, out);
        const int64_t a4 = a & ~(int64_t)3;
        int64_t e4 = (b + 3) & ~(int64_t)3;
        if (e4 > nt4) e4 = nt4;
        const double *sd = reinterpret_cast<const double *>(smraw + s * stage_bytes) + (a - a4);
        const int *sp = reinterpret_cast<const int *>(smraw + s * stage_bytes + (size_t)capw * 8) + (a - a4);
        const int64_t nsm = e4 - a;                        // samples of the subscan present in the stage
        mbar_wait(&full[s], (uint32_t)((i / nstage) & 1));
        if (nsm >= len) {                                // block-uniform: every sample came with the bulk copy
            filter_segment<NK, OFFSET, TB>([&](int j) { return sd[j]; },
                                           [&](int j) { return OFFSET ? (sp[j] != -1) : (sp[j] >= 0); }, a, len, out, fill,
                                           sh);
        } else {                                         // the <= 3 last samples of the TOD
            auto getd = [&](int j) { return j < nsm ? sd[j] : d[a + j]; };
            auto getf = [&](int j) {
                const int p = j < nsm ? sp[j] : pix[a + j];
                return OFFSET ? (p != -1) : (p >= 0);
            };
            filter_segment<NK, OFFSET, TB>(getd, getf, a, len, out, fill, sh);
        }
    }
}

template <int NK, bool OFFSET>
static int launch_filter_poly(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                              int64_t max_seg_len, const double *d, double *out, int64_t nt, int fill, int use_tma,
                              cudaStream_t st) {
    // variant B when at least two stages of the longest subscan fit into 200 kB of shared memory
    const int64_t capw = (max_seg_len + 8 + 3) / 4 * 4;
    const int64_t budget = 200 * 1024;
    int nstage = (int)(budget / (capw * 12));
    if (nstage > TMA_MAX_STAGES) nstage = TMA_MAX_STAGES;
    // measured (1e8 samples, 8000-sample subscans): B wins up to order 2 (order 0: 0.31 vs 0.50 ms; order 1:
    // 0.39 vs 0.46 ms); from order 3 on the kernel is bound by fp64 issue and A's larger number of
    // resident warps wins (0.53 vs 0.57 ms)
    if (use_tma && NK <= 3 && nstage >= 2 && aligned(d, 16) && aligned(pix, 16)) {
        // no more stages than subscans per CTA make use of
        const int64_t per_cta = (nseg + sm_count() - 1) / sm_count();
        if (nstage > per_cta + 1) nstage = (int)(per_cta + 1);
        if (nstage < 2) nstage = 2;
        const size_t smem = (size_t)capw * 12 * nstage;
        auto kern = k_filter_poly_tma<NK, OFFSET>;
        CM2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        return launch(kern, capped_grid(nseg, 1), TB, smem, st, pix, seg_start, seg_end, nseg, d, out, nt, (int)capw, nstage,
                      fill);
    }
    // variant A: shared-memory window of the longest subscan, up to 24 000 samples (216 kB); longer
    // subscans re-read their tail from global memory (L2)
    int64_t cap64 = (max_seg_len + 15) / 16 * 16;
    if (cap64 > 24000) cap64 = 24000;
    if (cap64 < 16) cap64 = 16;
    const int cap = (int)cap64;
    const size_t smem = (size_t)cap * 9;
    auto kern = k_filter_poly<NK, OFFSET>;
    CM2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return launch(kern, persistent_grid(kern, FB, smem, nseg), FB, smem, st, pix, seg_start, seg_end, nseg, d, out, nt, cap,
                  fill);
}

// ---- ground-template filter: out = v - bins[g] / hits[g] ---------------------------------------
__global__ void __launch_bounds__(FB) k_ground_sub(const int32_t *__restrict__ g, const double *__restrict__ bins,
                                                   const int64_t *__restrict__ hits, const double *__restrict__ v,
                                                   double *__restrict__ out, int64_t nt) {
    const int64_t nchunk = (nt + 3) / 4;
    for (int64_t ch = (int64_t)blockIdx.x * FB + threadIdx.x; ch < nchunk; ch += (int64_t)gridDim.x * FB) {
        const int64_t t0 = ch * 4;
        if (t0 + 4 <= nt) {
            const int4 gi = __ldcs(reinterpret_cast<const int4 *>(g + t0));
            D4 x = ld_stream_d4(v + t0);
            const int gg[4] = {gi.x, gi.y, gi.z, gi.w};
            int prev = -1;
            double m = 0.0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (gg[j] >= 0) {
                    if (gg[j] != prev) {          // ground bins change slowly along a scan: one lookup per run
                        const int64_t h = __ldg(hits + gg[j]);
                        m = h > 0 ? __ldg(bins + gg[j]) / (double)h : 0.0;   // 1x1 M_BD: x / counts where counts > 0
                        prev = gg[j];
                    }
                    x.v[j] -= m;
                }
            }
            st_stream_d4(out + t0, x);
        } else {
            for (int64_t t = t0; t < nt; ++t) {
                const int b = g[t];
                double m = 0.0;
                if (b >= 0) { const int64_t h = hits[b]; m = h > 0 ? bins[b] / (double)h : 0.0; }
                out[t] = v[t] - m;
            }
        }
    }
}

// ---- map output: out[k][obspix[p]] = map[pol p + k], zero elsewhere ----------------------------------
__global__ void __launch_bounds__(FB) k_reorganize(const double *__restrict__ map, const int64_t *__restrict__ obspix,
                                                   int64_t npix, int pol, int64_t hnpix, double *__restrict__ out) {
    for (int64_t p = (int64_t)blockIdx.x * FB + threadIdx.x; p < npix; p += (int64_t)gridDim.x * FB) {
        const int64_t o = obspix[p];
        for (int k = 0; k < pol; ++k) out[(int64_t)k * hnpix + o] = map[(int64_t)pol * p + k];
    }
}

}  // namespace cm2

using namespace cm2;

static int g_filter_tma = 1;

extern "C" int cm2_filter_poly_max_order(void) { return FP_MAXNK - 1; }

extern "C" int cm2_filter_poly_apply(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                                     int64_t max_seg_len, int poly_order, int sorted, const double *d, double *out,
                                     int64_t nt, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0 && nseg >= 0 && max_seg_len >= 0, "bad sizes");
    CM2_REQUIRE(d != out, "in-place filtering is not supported");
    CM2_REQUIRE(max_seg_len < INT_MAX, "subscans longer than 2^31 samples are not supported");
    if (poly_order < 0 || poly_order >= FP_MAXNK)
        return set_error(CM2_ERR_UNSUPPORTED, "poly_order=%d: orders 0..%d are supported", poly_order, FP_MAXNK - 1);
    cudaStream_t st = as_stream(stream);
    const int fill = sorted && nseg > 0;
    if (!fill) CM2_CUDA(zero_fill(out, nt, 1, st));
    if (nt == 0 || nseg == 0) return CM2_OK;
    const int tma = g_filter_tma;
#define CM2_FP(NKv, OFFv) launch_filter_poly<NKv, OFFv>(pix, seg_start, seg_end, nseg, max_seg_len, d, out, nt, fill, tma, st)
    switch (poly_order) {
        case 0: return CM2_FP(1, true);
        case 1: return CM2_FP(2, false);
        case 2: return CM2_FP(3, false);
        case 3: return CM2_FP(4, false);
        case 4: return CM2_FP(5, false);
        case 5: return CM2_FP(6, false);
        case 6: return CM2_FP(7, false);
        default: return CM2_FP(8, false);
    }
#undef CM2_FP
}

/* development switch: 0 = always the ordinary-load variant (A), 1 = TMA-pipelined variant (B) when it fits */
extern "C" int cm2_filter_poly_set_tma(int on) {
    const int old = g_filter_tma;
    g_filter_tma = on != 0;
    return old;
}

extern "C" int cm2_ground_filter_sub(const int32_t *ground, int64_t nt, int64_t nbins, const int64_t *hits,
                                     const double *bins, const double *v, double *out, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0 && nbins >= 0, "bad sizes");
    CM2_REQUIRE(aligned(ground, 32) && aligned(v, 32) && aligned(out, 32), "TOD vectors must be 32-byte aligned");
    if (nt == 0) return CM2_OK;
    return launch(k_ground_sub, capped_grid(cdiv(cdiv(nt, 4), FB), 8), FB, 0, as_stream(stream), ground, bins, hits, v, out,
                  nt);
}

extern "C" int cm2_ground_filter_apply(const int32_t *ground, int64_t nt, int64_t nbins, const int64_t *hits,
                                       const double *v, double *bins, double *out, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0 && nbins >= 0, "bad sizes");
    // bins = G^T v: the pol = 1 scatter-add with run aggregation (ground bins change slowly along a scan)
    int rc = cm2_pointing_apply_t(ground, nullptr, nullptr, nt, 1, v, bins, nbins, stream);
    if (rc) return rc;
    return cm2_ground_filter_sub(ground, nt, nbins, hits, bins, v, out, stream);
}

extern "C" int cm2_reorganize_map(const double *map, const int64_t *obspix, int64_t npix, int pol, int64_t healpix_npix,
                                  double *out, cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && healpix_npix >= 0, "bad sizes");
    CM2_REQUIRE(pol >= 1 && pol <= 3, "pol must be 1, 2 or 3");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(out, healpix_npix, pol, st));
    if (npix == 0 || healpix_npix == 0) return CM2_OK;
    return launch(k_reorganize, capped_grid(cdiv(npix, FB), 8), FB, 0, st, map, obspix, npix, pol, healpix_npix, out);
}
