// cosmomap2_b200 -- deflation space, coarse operator and two-level preconditioner (sm_100a).
//
//   cm2_defl_zt_apply   out = Z^T X      (DeflationLO.rmult linearoperators.py:1056; E build :1019)
//   cm2_defl_z_apply    y = beta y0 + alpha Z c          (DeflationLO.mult :1047-1050)
//   cm2_coarse_apply    c = Einv v                        (CoarseLO.mult_eig :984)
//   cm2_m2_apply        y = M_BD (v - AZ c) + Z c, c = Einv Z^T v
//                       (src/test_M2_precond_onto_real_data.py:109-112; reads Z twice, AZ once)
//
// Z is tall-skinny (n x r, column-major, r <= 64): these are HBM-bound streaming kernels
// (8 r bytes per row), so they run on the fp64 pipes with coalesced 128-bit column reads; the
// r x r work is negligible.
#include "cm2_common.cuh"

namespace cm2 {

constexpr int DB = 256;
constexpr int DG_MAX = 1024;   // max CTAs of the Z^T x reduction

// partial[blockIdx.x * r + c] = sum over this CTA's rows of Z[row, c] * x[row].
// RC columns are accumulated per pass (RC = 32 covers r <= 32 in ONE pass over x and Z); every
// thread keeps RC independent column streams in flight per row.
template <int RC>
__global__ void __launch_bounds__(DB) k_zt_partial(const double *__restrict__ Z, int64_t n, int r, int64_t ldz,
                                                   const double *__restrict__ x, double *__restrict__ partial) {
    __shared__ double red[32];
    for (int c0 = 0; c0 < r; c0 += RC) {
        double acc[RC];
#pragma unroll
        for (int c = 0; c < RC; ++c) acc[c] = 0.0;
        const int nc = r - c0 < RC ? r - c0 : RC;
        if (nc == RC) {
            for (int64_t i = (int64_t)blockIdx.x * DB + threadIdx.x; i < n; i += (int64_t)gridDim.x * DB) {
                const double xi = x[i];
                double z[RC];
#pragma unroll
                for (int c = 0; c < RC; ++c) z[c] = __ldcs(Z + i + (int64_t)(c0 + c) * ldz);
#pragma unroll
                for (int c = 0; c < RC; ++c) acc[c] = fma(z[c], xi, acc[c]);
            }
        } else {
            for (int64_t i = (int64_t)blockIdx.x * DB + threadIdx.x; i < n; i += (int64_t)gridDim.x * DB) {
                const double xi = x[i];
#pragma unroll
                for (int c = 0; c < RC; ++c)
                    if (c < nc) acc[c] = fma(__ldcs(Z + i + (int64_t)(c0 + c) * ldz), xi, acc[c]);
            }
        }
#pragma unroll
        for (int c = 0; c < RC; ++c) {
            const double t = block_sum(acc[c], red);
            if (threadIdx.x == 0 && c < nc) partial[(int64_t)blockIdx.x * r + c0 + c] = t;
        }
    }
}

static void launch_zt_partial(int g, cudaStream_t st, const double *Z, int64_t n, int r, int64_t ldz, const double *x,
                              double *partial) {
    if (r <= 8) k_zt_partial<8><<<g, DB, 0, st>>>(Z, n, r, ldz, x, partial);
    else if (r <= 16) k_zt_partial<16><<<g, DB, 0, st>>>(Z, n, r, ldz, x, partial);
    else k_zt_partial<32><<<g, DB, 0, st>>>(Z, n, r, ldz, x, partial);
}

// out[c] = sum_b partial[b*r + c] in CTA order (deterministic); optional out = Einv * (that)
__global__ void __launch_bounds__(DB) k_zt_final(const double *__restrict__ partial, int nb, int r,
                                                 const double *__restrict__ Einv, double *__restrict__ t_out,
                                                 double *__restrict__ c_out) {
    extern __shared__ double st[];   // r doubles
    for (int c = threadIdx.x; c < r; c += DB) {
        double s = 0.0;
        for (int b = 0; b < nb; ++b) s += partial[(int64_t)b * r + c];
        st[c] = s;
        if (t_out) t_out[c] = s;
    }
    __syncthreads();
    if (Einv != nullptr) {
        for (int i = threadIdx.x; i < r; i += DB) {
            double s = 0.0;
            for (int j = 0; j < r; ++j) s = fma(Einv[i + (int64_t)j * r], st[j], s);
            c_out[i] = s;
        }
    }
}

__global__ void __launch_bounds__(DB) k_z_apply(const double *__restrict__ Z, int64_t n, int r, int64_t ldz,
                                                const double *__restrict__ coef, double alpha, double beta,
                                                const double *__restrict__ y0, double *__restrict__ y) {
    extern __shared__ double sc[];
    for (int c = threadIdx.x; c < r; c += DB) sc[c] = coef[c];
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * DB + threadIdx.x; i < n; i += (int64_t)gridDim.x * DB) {
        double s = 0.0;
#pragma unroll 8
        for (int c = 0; c < r; ++c) s = fma(__ldcs(Z + i + (int64_t)c * ldz), sc[c], s);
        const double b = (y0 != nullptr && beta != 0.0) ? beta * y0[i] : 0.0;
        y[i] = fma(alpha, s, b);
    }
}

__global__ void __launch_bounds__(DB) k_coarse_apply(const double *__restrict__ Einv, int r, const double *__restrict__ v,
                                                     double *__restrict__ c) {
    extern __shared__ double sv[];
    for (int j = threadIdx.x; j < r; j += DB) sv[j] = v[j];
    __syncthreads();
    for (int i = threadIdx.x; i < r; i += DB) {
        double s = 0.0;
        for (int j = 0; j < r; ++j) s = fma(Einv[i + (int64_t)j * r], sv[j], s);
        c[i] = s;
    }
}

// per pixel: u = v - AZ c ; y = Minv u + Z c
template <int POL>
__global__ void __launch_bounds__(DB) k_m2_finish(const double *__restrict__ Z, const double *__restrict__ AZ, int r, int64_t ld,
                                                  const double *__restrict__ coef, const double *__restrict__ inv, int64_t npix,
                                                  const double *__restrict__ v, double *__restrict__ y) {
    extern __shared__ double sc[];
    for (int c = threadIdx.x; c < r; c += DB) sc[c] = coef[c];
    __syncthreads();
    for (int64_t j = (int64_t)blockIdx.x * DB + threadIdx.x; j < npix; j += (int64_t)gridDim.x * DB) {
        double u[POL], zc[POL];
#pragma unroll
        for (int k = 0; k < POL; ++k) { u[k] = v[POL * j + k]; zc[k] = 0.0; }
#pragma unroll 8
        for (int c = 0; c < r; ++c) {
            const double cc = sc[c];
#pragma unroll
            for (int k = 0; k < POL; ++k) {
                u[k] = fma(-__ldcs(AZ + POL * j + k + (int64_t)c * ld), cc, u[k]);
                zc[k] = fma(__ldcs(Z + POL * j + k + (int64_t)c * ld), cc, zc[k]);
            }
        }
        const double *b = inv + 6 * j;
        if constexpr (POL == 1) {
            y[j] = fma(b[0], u[0], zc[0]);
        } else if constexpr (POL == 2) {
            y[2 * j] = b[3] * u[0] + b[4] * u[1] + zc[0];
            y[2 * j + 1] = b[4] * u[0] + b[5] * u[1] + zc[1];
        } else {
            y[3 * j] = b[0] * u[0] + b[1] * u[1] + b[2] * u[2] + zc[0];
            y[3 * j + 1] = b[1] * u[0] + b[3] * u[1] + b[4] * u[2] + zc[1];
            y[3 * j + 2] = b[2] * u[0] + b[4] * u[1] + b[5] * u[2] + zc[2];
        }
    }
}

}  // namespace cm2

using namespace cm2;

extern "C" int64_t cm2_defl_work_doubles(int r) { return (int64_t)DG_MAX * r + 2 * (int64_t)r; }

extern "C" int cm2_defl_zt_apply(const double *Z, int64_t n, int r, int64_t ldz, const double *X, int ncols_x,
                                 int64_t ldx, double *out, double *work, cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0 && r >= 1 && ncols_x >= 1 && ldz >= n, "bad sizes");
    CM2_REQUIRE(work != nullptr, "work (cm2_defl_work_doubles) required");
    cudaStream_t st = as_stream(stream);
    const int g = capped_grid(cdiv(n, DB), 2, DG_MAX);   // 128 regs/thread -> 2 resident CTAs/SM: one wave
    for (int k = 0; k < ncols_x; ++k) {
        launch_zt_partial(g, st, Z, n, r, ldz, X + (int64_t)k * ldx, work);
        CM2_LAUNCHED();
        k_zt_final<<<1, DB, sizeof(double) * r, st>>>(work, g, r, nullptr, out + (int64_t)k * r, nullptr);
        CM2_LAUNCHED();
    }
    return CM2_OK;
}

extern "C" int cm2_defl_z_apply(const double *Z, int64_t n, int r, int64_t ldz, const double *c, double alpha,
                                double beta, const double *y0, double *y, cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0 && r >= 1 && ldz >= n, "bad sizes");
    if (n == 0) return CM2_OK;
    return launch(k_z_apply, capped_grid(cdiv(n, DB), 8, DG_MAX), DB, sizeof(double) * r, as_stream(stream), Z, n, r, ldz, c,
                  alpha, beta, y0, y);
}

extern "C" int cm2_coarse_apply(const double *Einv, int r, const double *v, double *c, cm2_stream_t stream) {
    CM2_REQUIRE(r >= 1, "r < 1");
    k_coarse_apply<<<1, DB, sizeof(double) * r, as_stream(stream)>>>(Einv, r, v, c);
    CM2_LAUNCHED();
    return CM2_OK;
}

// ---- banded two-level apply ---------------------------------------------------------------------------
// For a subdomain coarse space (deflationlib.scan_coarse_space) column k of Z is the intensity indicator of the
// pixels of band k, so Z has ONE non-zero per pixel and A Z is banded: (A z_k) lives on band k and its two
// neighbours.  The same y = M_BD (v - AZ c) + Z c, c = Einv Z^T v then reads band[npix] (int32) and
// azb[npix][pol][3] (the entries of AZ in columns band-1, band, band+1, cyclic) instead of 3 r doubles per map
// element: 172 B per IQU pixel instead of 2304 at r = 32.
// Z^T v = per-band sums of the intensity component.  Deterministic: every warp adds into its own r accumulators in
// program order (a warp whose 32 pixels span several bands handles them band by band), warps are added in warp
// order, CTAs in CTA order by k_zt_final.
constexpr int BAND_RMAX = 64;

template <int POL>
__global__ void __launch_bounds__(DB) k_band_sums(const int32_t *__restrict__ band, int64_t npix, int r,
                                                  const double *__restrict__ v, double *__restrict__ partial) {
    __shared__ double acc[DB / 32][BAND_RMAX];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = lane; k < r; k += 32) acc[warp][k] = 0.0;
    __syncwarp();
    const int64_t nchunks = (npix + 31) / 32;
    const int64_t nwarps = (int64_t)gridDim.x * (DB / 32);
    // a warp walks CONSECUTIVE chunks of 32 pixels (bands are contiguous ranges of the pixel order, so a whole
    // stretch of chunks belongs to one band and is summed in registers before it touches shared memory)
    const int64_t per = (nchunks + nwarps - 1) / nwarps;
    const int64_t w = (int64_t)blockIdx.x * (DB / 32) + warp;
    const int64_t c0 = w * per, c1 = c0 + per < nchunks ? c0 + per : nchunks;
    int cur = -1;
    double run = 0.0;
    for (int64_t c = c0; c < c1; ++c) {
        const int64_t p = c * 32 + lane;
        const int b = p < npix ? __ldg(band + p) : -1;
        const double x = (p < npix && b >= 0) ? v[(int64_t)POL * p] : 0.0;
        const int b0 = __shfl_sync(0xffffffffu, b, 0);
        if (__all_sync(0xffffffffu, b == b0 || b < 0) && b0 >= 0) {       // one band (the common case)
            if (b0 != cur) {
                if (cur >= 0) {
                    const double t = warp_sum(run);
                    if (lane == 0) acc[warp][cur] += t;
                }
                cur = b0;
                run = 0.0;
            }
            run += x;
        } else {                                                            // several bands inside these 32 pixels
            if (cur >= 0) {
                const double t = warp_sum(run);
                if (lane == 0) acc[warp][cur] += t;
                cur = -1;
                run = 0.0;
            }
            unsigned todo = __ballot_sync(0xffffffffu, b >= 0);
            while (todo) {
                const int leader = __ffs(todo) - 1;
                const int bl = __shfl_sync(0xffffffffu, b, leader);
                const double t = warp_sum(b == bl ? x : 0.0);
                if (lane == 0) acc[warp][bl] += t;
                todo &= ~__ballot_sync(0xffffffffu, b == bl);
            }
        }
    }
    if (cur >= 0) {
        const double t = warp_sum(run);
        if (lane == 0) acc[warp][cur] += t;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < r; k += DB) {
        double t = 0.0;
#pragma unroll
        for (int ww = 0; ww < DB / 32; ++ww) t += acc[ww][k];
        partial[(int64_t)blockIdx.x * r + k] = t;
    }
}

template <int POL>
__global__ void __launch_bounds__(DB) k_m2_banded_finish(const int32_t *__restrict__ band, const double *__restrict__ azb, int r,
                                                         const double *__restrict__ coef, const double *__restrict__ inv,
                                                         int64_t npix, const double *__restrict__ v, double *__restrict__ y) {
    extern __shared__ double sc[];
    for (int k = threadIdx.x; k < r; k += DB) sc[k] = coef[k];
    __syncthreads();
    for (int64_t j = (int64_t)blockIdx.x * DB + threadIdx.x; j < npix; j += (int64_t)gridDim.x * DB) {
        const int b = __ldg(band + j);
        double u[POL], z[POL];
        double c0 = 0.0;
        if (b >= 0) {
            const double cm = sc[b == 0 ? r - 1 : b - 1], cp = sc[b == r - 1 ? 0 : b + 1];
            c0 = sc[b];
            const double *a = azb + (int64_t)3 * POL * j;
#pragma unroll
            for (int k = 0; k < POL; ++k)
                u[k] = v[(int64_t)POL * j + k] - (__ldcs(a + 3 * k) * cm + __ldcs(a + 3 * k + 1) * c0 + __ldcs(a + 3 * k + 2) * cp);
        } else {
#pragma unroll
            for (int k = 0; k < POL; ++k) u[k] = v[(int64_t)POL * j + k];
        }
        bd_z<POL>(inv, j, u, z);
        z[0] += c0;                                  // Z c: the intensity component of band b
#pragma unroll
        for (int k = 0; k < POL; ++k) y[(int64_t)POL * j + k] = z[k];
    }
}

extern "C" int cm2_m2_apply(const double *Z, const double *AZ, int64_t n, int r, int64_t ld, const double *Einv,
                            const double *bd_inv, int64_t npix, int pol, const double *v, double *y, double *work,
                            cm2_stream_t stream) {
    CM2_REQUIRE(pol >= 1 && pol <= 3 && n == npix * pol && r >= 1 && ld >= n, "bad sizes");
    CM2_REQUIRE(work != nullptr, "work (cm2_defl_work_doubles) required");
    cudaStream_t st = as_stream(stream);
    const int g = capped_grid(cdiv(n, DB), 2, DG_MAX);
    double *coef = work + (int64_t)DG_MAX * r;   // r doubles: c = Einv Z^T v
    launch_zt_partial(g, st, Z, n, r, ld, v, work);
    CM2_LAUNCHED();
    k_zt_final<<<1, DB, sizeof(double) * r, st>>>(work, g, r, Einv, nullptr, coef);
    CM2_LAUNCHED();
    const int g2 = capped_grid(cdiv(npix, DB), 8, DG_MAX);
    return with_pol(pol, [&](auto P) {
        return launch(k_m2_finish<P>, g2, DB, sizeof(double) * r, st, Z, AZ, r, ld, coef, bd_inv, npix, v, y);
    });
}


// y = M_BD (v - AZ c) + Z c, c = Einv Z^T v for a subdomain coarse space given in banded form (see k_band_sums):
// band[npix] = column of Z whose indicator contains the pixel (-1: none), azb[npix][pol][3] = AZ[pol*p + k, band-1 |
// band | band+1 (cyclic)].  Requires pol = 1 or 3 (the indicator sits on the intensity component), 3 <= r <= 64.
extern "C" int cm2_m2_banded_apply(const int32_t *band, const double *azb, int r, const double *Einv, const double *bd_inv,
                                   int64_t npix, int pol, const double *v, double *y, double *work, cm2_stream_t stream) {
    CM2_REQUIRE((pol == 1 || pol == 3) && r >= 3 && r <= BAND_RMAX && npix >= 0, "bad sizes (pol 1 or 3, 3 <= r <= 64)");
    CM2_REQUIRE(work != nullptr && band != nullptr && azb != nullptr, "NULL argument");
    if (npix == 0) return CM2_OK;
    cudaStream_t st = as_stream(stream);
    const int g = capped_grid(cdiv(npix, DB), 2, DG_MAX);
    double *coef = work + (int64_t)DG_MAX * r;
    if (pol == 1) k_band_sums<1><<<g, DB, 0, st>>>(band, npix, r, v, work);
    else k_band_sums<3><<<g, DB, 0, st>>>(band, npix, r, v, work);
    CM2_LAUNCHED();
    k_zt_final<<<1, DB, sizeof(double) * r, st>>>(work, g, r, Einv, nullptr, coef);
    CM2_LAUNCHED();
    const int g2 = capped_grid(cdiv(npix, DB), 8, DG_MAX);
    const size_t sm = sizeof(double) * r;
    if (pol == 1) k_m2_banded_finish<1><<<g2, DB, sm, st>>>(band, azb, r, coef, bd_inv, npix, v, y);
    else k_m2_banded_finish<3><<<g2, DB, sm, st>>>(band, azb, r, coef, bd_inv, npix, v, y);
    CM2_LAUNCHED();
    return CM2_OK;
}
