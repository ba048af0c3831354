// cosmomap2_b200 -- library-level C ABI (errors, device info) and the deterministic sorted P^T.
#include <atomic>
#include <cstdarg>
#include <cstdio>

#include "cm2_common.cuh"

namespace cm2 {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};
static int g_sm_count = 0;

int set_error(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int sm_count() {
    if (g_sm_count == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            g_sm_count = n;
        else
            return 148;
    }
    return g_sm_count;
}

// one warp per pixel, fixed summation order: lane l adds entries l, l+32, ... then a fixed tree
template <int POL>
__global__ void __launch_bounds__(256) k_apply_t_sorted(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ perm,
                                                        const double *__restrict__ cs, const double *__restrict__ sn,
                                                        const double *__restrict__ d, double *__restrict__ y, int64_t npix) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * 8;
    for (int64_t j = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); j < npix; j += nwarps) {
        const int64_t a = rowptr[j], b = rowptr[j + 1];
        double acc[POL];
#pragma unroll
        for (int k = 0; k < POL; ++k) acc[k] = 0.0;
        for (int64_t e = a + lane; e < b; e += 32) {
            const int64_t t = perm[e];
            const double v = d[t];
            if constexpr (POL == 1) {
                acc[0] += v;
            } else if constexpr (POL == 2) {
                acc[0] = fma(v, cs[t], acc[0]);
                acc[1] = fma(v, sn[t], acc[1]);
            } else {
                acc[0] += v;
                acc[1] = fma(v, cs[t], acc[1]);
                acc[2] = fma(v, sn[t], acc[2]);
            }
        }
#pragma unroll
        for (int k = 0; k < POL; ++k) acc[k] = warp_sum(acc[k]);
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < POL; ++k) y[POL * j + k] = acc[k];
        }
    }
}

}  // namespace cm2

using namespace cm2;

extern "C" int cm2_version(void) { return 100; }

extern "C" const char *cm2_last_error(void) { return g_err; }

extern "C" int64_t cm2_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" int cm2_device_info(int *sm, int64_t *l2_bytes, int *cc) {
    int dev = 0;
    CM2_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    CM2_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm) *sm = p.multiProcessorCount;
    if (l2_bytes) *l2_bytes = p.l2CacheSize;
    if (cc) *cc = p.major * 10 + p.minor;
    return CM2_OK;
}

extern "C" int cm2_pointing_apply_t_sorted(const int64_t *rowptr, const int32_t *perm, const double *c, const double *s,
                                           int pol, const double *d, double *y, int64_t npix, cm2_stream_t stream) {
    CM2_REQUIRE(pol >= 1 && pol <= 3, "No valid polarization key set! (1=I, 2=QU, 3=IQU)");
    CM2_REQUIRE(npix >= 0, "npix < 0");
    if (npix == 0) return CM2_OK;
    const int g = capped_grid(cdiv(npix, 8), 8);   // one pixel per warp
    return with_pol(pol, [&](auto P) {
        return launch(k_apply_t_sorted<P>, g, 256, 0, as_stream(stream), rowptr, perm, c, s, d, y, npix);
    });
}
