// cosmomap2_b200 -- pixel-domain kernels and set-up passes (sm_100a).
//
//   cm2_angles, cm2_pix_narrow/widen          input conversion (process_ces.py:493-494)
//   cm2_weights_mask / old2new / compact / relabel   (process_ces.py:192-349, 403-425, 544-555)
//   cm2_bd_build / cm2_bd_apply / cm2_bdfwd_apply    (linearoperators.py:700-859)
//
// Per-pixel coefficient arrays are interleaved [npix][6] fp64 (48 B/pixel, 16-B aligned rows):
//   mom = {h, c, s, c2, cs, s2}            inv = {i00, i01, i02, i11, i12, i22}
// (both are the upper triangle of the symmetric 3x3 block [[h,c,s],[c,c2,cs],[s,cs,s2]] or its inverse)
// so a pixel's coefficients arrive in three 128-bit loads and a warp reads 1.5 kB contiguous.
#include "cm2_common.cuh"

namespace cm2 {

constexpr int PB = 256;

__global__ void __launch_bounds__(PB) k_angles(const double *__restrict__ phi, int64_t nt, double *__restrict__ c,
                                               double *__restrict__ s) {
    for (int64_t i = (int64_t)blockIdx.x * PB + threadIdx.x; i < nt; i += (int64_t)gridDim.x * PB) {
        double sv, cv;
        sincos(2.0 * phi[i], &sv, &cv);
        c[i] = cv;
        s[i] = sv;
    }
}

__global__ void __launch_bounds__(PB) k_narrow(const int64_t *__restrict__ a, int64_t n, int32_t *__restrict__ b) {
    for (int64_t i = (int64_t)blockIdx.x * PB + threadIdx.x; i < n; i += (int64_t)gridDim.x * PB) b[i] = (int32_t)a[i];
}
__global__ void __launch_bounds__(PB) k_widen(const int32_t *__restrict__ a, int64_t n, int64_t *__restrict__ b) {
    for (int64_t i = (int64_t)blockIdx.x * PB + threadIdx.x; i < n; i += (int64_t)gridDim.x * PB) b[i] = (int64_t)a[i];
}

// process_ces.py:491, 544-555.  NaN conditions (unobserved pixels: 0/0) compare false -> dropped.
__global__ void __launch_bounds__(PB) k_mask(const double *__restrict__ mom, int64_t npix, int pol, double thr,
                                             int32_t *__restrict__ good) {
    for (int64_t j = (int64_t)blockIdx.x * PB + threadIdx.x; j < npix; j += (int64_t)gridDim.x * PB) {
        const double *m = mom + 6 * j;
        int g;
        if (pol == 1) {
            g = m[0] > 0.0;
        } else {
            // exactly the reference's operation order, every operation rounded on its own (no FMA
            // contraction): with bit-identical moments the mask is bit-identical to NumPy's
            const double c2 = m[3], cs = m[4], s2 = m[5];
            const double det = __dsub_rn(__dmul_rn(c2, s2), __dmul_rn(cs, cs));
            const double tr = __dadd_rn(c2, s2);
            const double sq = __dsqrt_rn(__dsub_rn(__ddiv_rn(__dmul_rn(tr, tr), 4.), det));
            const double lmax = __dadd_rn(__ddiv_rn(tr, 2.), sq), lmin = __dsub_rn(__ddiv_rn(tr, 2.), sq);
            const double cond = fabs(__ddiv_rn(lmax, lmin));
            g = cond <= thr;
            if (pol == 3) g = g && (m[0] > 2.0);
        }
        good[j] = g;
    }
}

// Deterministic moments in the reference's own summation order: one thread per pixel walks the
// pixel's samples in time order (perm = stable argsort of pix) and accumulates with the serial
// loop's association and rounding -- (w*c)*c etc., no FMA -- so every moment is bit-identical to
// process_ces.py:480-542 run on the same inputs.  One-off set-up pass; gathers are uncoalesced.
__global__ void __launch_bounds__(PB) k_moments_sorted(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ perm,
                                                       const double *__restrict__ cs, const double *__restrict__ sn,
                                                       const double *__restrict__ wsamp, const double *__restrict__ wblk,
                                                       int64_t nblocks, int64_t blocksize, const int64_t *__restrict__ bstart,
                                                       int pol, double *__restrict__ mom, int64_t npix) {
    for (int64_t j = (int64_t)blockIdx.x * PB + threadIdx.x; j < npix; j += (int64_t)gridDim.x * PB) {
        double h = 0., c1 = 0., s1 = 0., c2 = 0., cs2 = 0., s2 = 0.;
        for (int64_t e = rowptr[j]; e < rowptr[j + 1]; ++e) {
            const int64_t t = perm[e];
            double w = 1.0;
            if (wsamp) w = wsamp[t];
            else if (wblk) {
                const int64_t b = bstart == nullptr ? t / blocksize : last_le(bstart, nblocks, t);
                w = wblk[b < nblocks ? b : nblocks - 1];
            }
            if (pol == 1) { h = __dadd_rn(h, w); continue; }
            const double c = cs[t], s = sn[t];
            const double wc = __dmul_rn(w, c), ws = __dmul_rn(w, s);
            if (pol == 3) {
                h = __dadd_rn(h, w);
                c1 = __dadd_rn(c1, wc);
                s1 = __dadd_rn(s1, ws);
            }
            c2 = __dadd_rn(c2, __dmul_rn(wc, c));
            s2 = __dadd_rn(s2, __dmul_rn(ws, s));
            cs2 = __dadd_rn(cs2, __dmul_rn(ws, c));
        }
        double *m = mom + 6 * j;
        m[0] = h; m[1] = c1; m[2] = s1; m[3] = c2; m[4] = cs2; m[5] = s2;
    }
}

// ---- exclusive scan of int32 flags (three-phase, deterministic) ------------------------------
constexpr int SCAN_ITEMS = 8;                  // flags per thread
constexpr int SCAN_TILE = PB * SCAN_ITEMS;     // flags per block

__device__ __forceinline__ int block_excl_scan(int v, int *smem, int *total) {
    // exclusive scan of one int per thread over the block; smem: 32 ints
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) smem[w] = inc;
    __syncthreads();
    if (w == 0) {
        int s = lane < (PB / 32) ? smem[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += t;
        }
        smem[lane] = s;  // inclusive over warps
    }
    __syncthreads();
    const int woff = w == 0 ? 0 : smem[w - 1];
    *total = smem[PB / 32 - 1];
    return woff + inc - v;
}

__global__ void __launch_bounds__(PB) k_scan_partials(const int32_t *__restrict__ good, int64_t n, int64_t *__restrict__ part) {
    __shared__ int sm[32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) cnt += (base + i < n) ? (good[base + i] != 0) : 0;
    int total;
    block_excl_scan(cnt, sm, &total);
    if (threadIdx.x == 0) part[blockIdx.x] = total;
}

// single block: exclusive scan of the per-tile totals in place; grand total -> *total_out
__global__ void __launch_bounds__(PB) k_scan_tops(int64_t *__restrict__ part, int64_t nparts, int64_t *__restrict__ total_out) {
    __shared__ int64_t carry;
    __shared__ int sm[32];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t b0 = 0; b0 < nparts; b0 += PB) {
        const int64_t i = b0 + threadIdx.x;
        const int v = i < nparts ? (int)part[i] : 0;  // each tile total <= SCAN_TILE
        int total;
        const int ex = block_excl_scan(v, sm, &total);
        const int64_t c = carry;
        if (i < nparts) part[i] = c + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry = c + total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(PB) k_scan_apply(const int32_t *__restrict__ good, int64_t n, const int64_t *__restrict__ part,
                                                   int32_t *__restrict__ old2new) {
    __shared__ int sm[32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int g[SCAN_ITEMS];
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        g[i] = (base + i < n) ? (good[base + i] != 0) : 0;
        cnt += g[i];
    }
    int total;
    int64_t off = part[blockIdx.x] + block_excl_scan(cnt, sm, &total);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        if (base + i < n) old2new[base + i] = g[i] ? (int32_t)off : -1;
        off += g[i];
    }
}

template <class T>
__global__ void __launch_bounds__(PB) k_compact_rows(const T *__restrict__ src, const int32_t *__restrict__ old2new, int64_t npix,
                                                     int width, T *__restrict__ dst) {
    const int64_t total = npix * width;
    for (int64_t i = (int64_t)blockIdx.x * PB + threadIdx.x; i < total; i += (int64_t)gridDim.x * PB) {
        const int64_t j = i / width;
        const int k = (int)(i - j * width);
        const int32_t nw = old2new[j];
        if (nw >= 0) dst[(int64_t)nw * width + k] = src[i];
    }
}

__global__ void __launch_bounds__(PB) k_relabel(int32_t *__restrict__ pix, int64_t nt, const int32_t *__restrict__ old2new) {
    for (int64_t i = (int64_t)blockIdx.x * PB + threadIdx.x; i < nt; i += (int64_t)gridDim.x * PB) {
        const int32_t p = pix[i];
        if (p != -1) pix[i] = __ldg(old2new + p);
    }
}

// ---- M_BD -------------------------------------------------------------------------------------
// linearoperators.py:789-801, 820-826: closed-form inverse, zero block where the test fails
__global__ void __launch_bounds__(PB) k_bd_build(const double *__restrict__ mom, int64_t npix, int pol, double *__restrict__ inv) {
    for (int64_t j = (int64_t)blockIdx.x * PB + threadIdx.x; j < npix; j += (int64_t)gridDim.x * PB) {
        const double *m = mom + 6 * j;
        const double h = m[0], c = m[1], s = m[2], c2 = m[3], cs = m[4], s2 = m[5];
        double o[6] = {0, 0, 0, 0, 0, 0};
        if (pol == 1) {
            if (h > 0.0) o[0] = 1.0 / h;
        } else if (pol == 2) {
            const double det = (c2 * s2) - (cs * cs);
            if (fabs(det) > 1e-5) {
                o[3] = s2 / det;
                o[4] = -cs / det;
                o[5] = c2 / det;
            }
        } else {
            const double det = h * (c2 * s2 - cs * cs) - c * c * s2 - s * s * c2 + 2. * c * s * cs;
            if (fabs(det) > 1e-5) {
                o[0] = (c2 * s2 - cs * cs) / det;
                o[1] = (s * cs - c * s2) / det;
                o[2] = (c * cs - s * c2) / det;
                o[3] = (h * s2 - s * s) / det;
                o[4] = (s * c - h * cs) / det;
                o[5] = (h * c2 - c * c) / det;
            }
        }
        double *d = inv + 6 * j;
#pragma unroll
        for (int k = 0; k < 6; ++k) d[k] = o[k];
    }
}

// y = S x with S the symmetric per-pixel block packed as {00,01,02,11,12,22}; pol=2 uses
// {11,12,22} on (Q,U); pol=1 uses {00}.  Serves M_BD (inv) and BlockDiagonalLO (mom).
template <int POL>
__global__ void __launch_bounds__(PB) k_block_apply(const double *__restrict__ blk, int64_t npix, const double *__restrict__ x,
                                                    double *__restrict__ y) {
    for (int64_t j = (int64_t)blockIdx.x * PB + threadIdx.x; j < npix; j += (int64_t)gridDim.x * PB) {
        const double2 *b2 = reinterpret_cast<const double2 *>(blk + 6 * j);
        if constexpr (POL == 1) {
            y[j] = __ldg(blk + 6 * j) * x[j];
        } else if constexpr (POL == 2) {
            const double2 q1 = __ldg(b2 + 1), q2 = __ldg(b2 + 2);  // {02,11} {12,22}
            const double x0 = x[2 * j], x1 = x[2 * j + 1];
            y[2 * j] = q1.y * x0 + q2.x * x1;
            y[2 * j + 1] = q2.x * x0 + q2.y * x1;
        } else {
            const double2 q0 = __ldg(b2), q1 = __ldg(b2 + 1), q2 = __ldg(b2 + 2);
            const double x0 = x[3 * j], x1 = x[3 * j + 1], x2 = x[3 * j + 2];
            y[3 * j] = q0.x * x0 + q0.y * x1 + q1.x * x2;
            y[3 * j + 1] = q0.y * x0 + q1.y * x1 + q2.x * x2;
            y[3 * j + 2] = q1.x * x0 + q2.x * x1 + q2.y * x2;
        }
    }
}

}  // namespace cm2

using namespace cm2;

extern "C" int cm2_angles(const double *phi, int64_t nt, double *c, double *s, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0, "nt < 0");
    if (nt == 0) return CM2_OK;
    return launch(k_angles, capped_grid(cdiv(nt, PB), 8), PB, 0, as_stream(stream), phi, nt, c, s);
}

extern "C" int cm2_pix_narrow(const int64_t *pix64, int64_t nt, int32_t *pix32, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0, "nt < 0");
    if (nt == 0) return CM2_OK;
    return launch(k_narrow, capped_grid(cdiv(nt, PB), 8), PB, 0, as_stream(stream), pix64, nt, pix32);
}

extern "C" int cm2_pix_widen(const int32_t *pix32, int64_t nt, int64_t *pix64, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0, "nt < 0");
    if (nt == 0) return CM2_OK;
    return launch(k_widen, capped_grid(cdiv(nt, PB), 8), PB, 0, as_stream(stream), pix32, nt, pix64);
}

extern "C" int cm2_weights_mask(const double *mom, int64_t npix, int pol, double threshold_cond, int32_t *good,
                                cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && pol >= 1 && pol <= 3, "bad npix/pol");
    if (npix == 0) return CM2_OK;
    return launch(k_mask, capped_grid(cdiv(npix, PB), 8), PB, 0, as_stream(stream), mom, npix, pol, threshold_cond, good);
}

extern "C" int cm2_weights_moments_sorted(const int64_t *rowptr, const int32_t *perm, const double *c, const double *s,
                                          const double *w, const double *wblk, int64_t nblocks, int64_t blocksize,
                                          const int64_t *blk_start, int pol, double *mom, int64_t npix,
                                          cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && pol >= 1 && pol <= 3, "bad npix/pol");
    CM2_REQUIRE(wblk == nullptr || nblocks > 0, "nblocks must be > 0 when block weights are given");
    if (npix == 0) return CM2_OK;
    return launch(k_moments_sorted, capped_grid(cdiv(npix, PB), 8), PB, 0, as_stream(stream), rowptr, perm, c, s, w, wblk,
                  nblocks, blocksize, blk_start, pol, mom, npix);
}

extern "C" int64_t cm2_scan_scratch_bytes(int64_t n) {
    int64_t parts = (n + SCAN_TILE - 1) / SCAN_TILE;
    return (parts + 1) * (int64_t)sizeof(int64_t);
}

extern "C" int cm2_weights_old2new(const int32_t *good, int64_t npix, int32_t *old2new, int64_t *npix_new_dev,
                                   void *scratch, cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0, "npix < 0");
    cudaStream_t st = as_stream(stream);
    if (npix == 0) {
        CM2_CUDA(cudaMemsetAsync(npix_new_dev, 0, sizeof(int64_t), st));
        return CM2_OK;
    }
    int64_t parts = (npix + SCAN_TILE - 1) / SCAN_TILE;
    CM2_REQUIRE(parts < (int64_t)1 << 31, "npix too large");
    int64_t *part = reinterpret_cast<int64_t *>(scratch);
    k_scan_partials<<<(int)parts, PB, 0, st>>>(good, npix, part);
    CM2_LAUNCHED();
    k_scan_tops<<<1, PB, 0, st>>>(part, parts, npix_new_dev);
    CM2_LAUNCHED();
    k_scan_apply<<<(int)parts, PB, 0, st>>>(good, npix, part, old2new);
    CM2_LAUNCHED();
    return CM2_OK;
}

extern "C" int cm2_compact_rows_f64(const double *src, const int32_t *old2new, int64_t npix, int width, double *dst,
                                    cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && width > 0, "bad npix/width");
    if (npix == 0) return CM2_OK;
    return launch(k_compact_rows<double>, capped_grid(cdiv(npix * width, PB), 8), PB, 0, as_stream(stream), src, old2new,
                  npix, width, dst);
}

extern "C" int cm2_compact_rows_i64(const int64_t *src, const int32_t *old2new, int64_t npix, int width, int64_t *dst,
                                    cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && width > 0, "bad npix/width");
    if (npix == 0) return CM2_OK;
    return launch(k_compact_rows<int64_t>, capped_grid(cdiv(npix * width, PB), 8), PB, 0, as_stream(stream), src, old2new,
                  npix, width, dst);
}

extern "C" int cm2_relabel(int32_t *pix, int64_t nt, const int32_t *old2new, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0, "nt < 0");
    if (nt == 0) return CM2_OK;
    return launch(k_relabel, capped_grid(cdiv(nt, PB), 8), PB, 0, as_stream(stream), pix, nt, old2new);
}

extern "C" int cm2_bd_build(const double *mom, int64_t npix, int pol, double *inv, cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && pol >= 1 && pol <= 3, "bad npix/pol");
    if (npix == 0) return CM2_OK;
    return launch(k_bd_build, capped_grid(cdiv(npix, PB), 8), PB, 0, as_stream(stream), mom, npix, pol, inv);
}

static int block_apply(const double *blk, int64_t npix, int pol, const double *x, double *y, cm2_stream_t stream) {
    if (npix < 0 || pol < 1 || pol > 3) return set_error(CM2_ERR_ARG, "bad npix/pol");
    if (!aligned(blk, 16)) return set_error(CM2_ERR_ARG, "block coefficients must be 16-byte aligned");
    if (npix == 0) return CM2_OK;
    const int g = capped_grid(cdiv(npix, PB), 8);
    return with_pol(pol, [&](auto P) { return launch(k_block_apply<P>, g, PB, 0, as_stream(stream), blk, npix, x, y); });
}

extern "C" int cm2_bd_apply(const double *inv, int64_t npix, int pol, const double *x, double *y, cm2_stream_t stream) {
    return block_apply(inv, npix, pol, x, y, stream);
}

extern "C" int cm2_bdfwd_apply(const double *mom, int64_t npix, int pol, const double *x, double *y, cm2_stream_t stream) {
    return block_apply(mom, npix, pol, x, y, stream);
}
