// cosmomap2_b200 -- PCG vector work on the device (sm_100a).
//
// Restates the recurrence of scipy.sparse.linalg.cg (scipy/_isolve/iterative.py:405-431), which the
// reference calls at src/test_BD_precond_onto_real_data.py:47 and
// src/test_M2_precond_onto_real_data.py:117.  All scalars live in a 16-double device workspace:
//   scal[0]=rho  [1]=rho_prev  [2]=p.q  [3]=|r|^2  [4]=alpha  [5]=beta  [6]=atol
//   scal[7]=done flag (||r|| < atol, SciPy's exit test)  [8]=iterations completed  [9..15] spare
// so an iteration needs no host round trip, and every update kernel is a no-op once `done` is set:
// the host may launch iterations ahead of reading the flag and x still freezes at exactly the
// iteration SciPy would have returned.
//
// Reductions are deterministic: fixed per-thread order, fixed shuffle tree, per-CTA partials summed
// in CTA order by the last CTA to finish (ticket).  The partial/ticket scratch is one device-global
// area: call these entry points from one stream at a time.
#include <cooperative_groups.h>

#include "cm2_common.cuh"

namespace cg = cooperative_groups;

namespace cm2 {

constexpr int VB = 256;
constexpr int MAXP = 2048;  // max CTAs of a reduction kernel

__device__ double g_part[3][MAXP];   // rows 0,1: reduction partials; row 2: p.q partials of k_bd_iter
__device__ unsigned int g_ticket;

// CTA-level: write up to two partials, last CTA reduces all partials in order; returns true in
// thread 0 of the last CTA with the totals in tot[0..NR)
template <int NR>
__device__ __forceinline__ bool finish_reduce(const double (&v)[NR], double *red, double (&tot)[NR]) {
    __shared__ bool last;
    double t[NR];
#pragma unroll
    for (int k = 0; k < NR; ++k) t[k] = block_sum(v[k], red);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < NR; ++k) g_part[k][blockIdx.x] = t[k];
        __threadfence();
        const unsigned int tk = atomicAdd(&g_ticket, 1u);
        last = (tk == gridDim.x - 1);
    }
    __syncthreads();
    if (!last) return false;
    __threadfence();
#pragma unroll
    for (int k = 0; k < NR; ++k) {
        double s = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += VB) s += ((volatile double *)g_part[k])[i];
        tot[k] = block_sum(s, red);
    }
    if (threadIdx.x == 0) {
        g_ticket = 0;
        return true;
    }
    return false;
}

__global__ void __launch_bounds__(VB) k_dot(const double *__restrict__ a, const double *__restrict__ b, int64_t n,
                                            double *__restrict__ out) {
    __shared__ double red[32];
    double s[1] = {0.0}, tot[1];
    for (int64_t i = (int64_t)blockIdx.x * VB + threadIdx.x; i < n; i += (int64_t)gridDim.x * VB) s[0] = fma(a[i], b[i], s[0]);
    if (finish_reduce<1>(s, red, tot)) *out = tot[0];
}

__global__ void __launch_bounds__(VB) k_axpby(double alpha, const double *__restrict__ x, double beta, double *__restrict__ y,
                                              int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * VB + threadIdx.x; i < n; i += (int64_t)gridDim.x * VB) {
        const double yi = beta == 0.0 ? 0.0 : beta * y[i];
        y[i] = fma(alpha, x[i], yi);
    }
}

// ---- generic-M path ------------------------------------------------------------------------
// reset: |r|^2, atol, done flag, iteration counter
__global__ void __launch_bounds__(VB) k_reset(const double *__restrict__ r, int64_t n, double *__restrict__ scal, double atol) {
    __shared__ double red[32];
    double s[1] = {0.0}, tot[1];
    for (int64_t i = (int64_t)blockIdx.x * VB + threadIdx.x; i < n; i += (int64_t)gridDim.x * VB) s[0] = fma(r[i], r[i], s[0]);
    if (finish_reduce<1>(s, red, tot)) {
        scal[0] = 0.0; scal[1] = 0.0; scal[2] = 0.0; scal[4] = 0.0; scal[5] = 0.0;
        scal[3] = tot[0];
        scal[6] = atol;
        scal[7] = (sqrt(tot[0]) < atol) ? 1.0 : 0.0;
        scal[8] = 0.0;
    }
}

// rho = r.z ; beta = rho/rho_prev (0 on the first iteration)
__global__ void __launch_bounds__(VB) k_rho(const double *__restrict__ r, const double *__restrict__ z, int64_t n,
                                            double *__restrict__ scal) {
    __shared__ double red[32];
    if (scal[7] != 0.0) return;
    double s[1] = {0.0}, tot[1];
    for (int64_t i = (int64_t)blockIdx.x * VB + threadIdx.x; i < n; i += (int64_t)gridDim.x * VB) s[0] = fma(r[i], z[i], s[0]);
    if (finish_reduce<1>(s, red, tot)) {
        scal[0] = tot[0];
        scal[5] = (scal[8] == 0.0) ? 0.0 : tot[0] / scal[1];
    }
}

// p = z + beta p  (p = z on the first iteration: p may be uninitialised)
__global__ void __launch_bounds__(VB) k_update_p(const double *__restrict__ z, double *__restrict__ p, int64_t n,
                                                 const double *__restrict__ scal) {
    if (scal[7] != 0.0) return;
    const bool first = scal[8] == 0.0;
    const double beta = scal[5];
    for (int64_t i = (int64_t)blockIdx.x * VB + threadIdx.x; i < n; i += (int64_t)gridDim.x * VB)
        p[i] = first ? z[i] : fma(beta, p[i], z[i]);
}

__global__ void __launch_bounds__(VB) k_pq(const double *__restrict__ p, const double *__restrict__ q, int64_t n,
                                           double *__restrict__ scal) {
    __shared__ double red[32];
    if (scal[7] != 0.0) return;
    double s[1] = {0.0}, tot[1];
    for (int64_t i = (int64_t)blockIdx.x * VB + threadIdx.x; i < n; i += (int64_t)gridDim.x * VB) s[0] = fma(p[i], q[i], s[0]);
    if (finish_reduce<1>(s, red, tot)) {
        scal[2] = tot[0];
        scal[4] = scal[0] / tot[0];
    }
}

__global__ void __launch_bounds__(VB) k_update_xr(const double *__restrict__ p, const double *__restrict__ q,
                                                  double *__restrict__ x, double *__restrict__ r, int64_t n,
                                                  double *__restrict__ scal) {
    __shared__ double red[32];
    if (scal[7] != 0.0) return;
    const double alpha = scal[4];
    double s[1] = {0.0}, tot[1];
    for (int64_t i = (int64_t)blockIdx.x * VB + threadIdx.x; i < n; i += (int64_t)gridDim.x * VB) {
        x[i] = fma(alpha, p[i], x[i]);
        const double ri = fma(-alpha, q[i], r[i]);
        r[i] = ri;
        s[0] = fma(ri, ri, s[0]);
    }
    if (finish_reduce<1>(s, red, tot)) {
        scal[3] = tot[0];
        scal[1] = scal[0];
        scal[8] += 1.0;
        scal[7] = (sqrt(tot[0]) < scal[6]) ? 1.0 : 0.0;
    }
}

// the scalars of a start, from tot = {r.z, |r|^2}
__device__ __forceinline__ void bd_reset_scalars(const double (&tot)[2], double *scal, double atol, double rtol, bool has_b) {
    const double atol_eff = (has_b && rtol > 0.0) ? fmax(atol, rtol * sqrt(tot[1])) : atol;
    scal[0] = tot[0]; scal[1] = 0.0; scal[2] = 0.0; scal[4] = 0.0; scal[5] = 0.0;
    scal[3] = tot[1];
    scal[6] = atol_eff;
    scal[7] = (sqrt(tot[1]) < atol_eff || (has_b && tot[1] == 0.0)) ? 1.0 : 0.0;
    scal[8] = 0.0;
    scal[9] = 0.0;                      // the sharded solver's failure word
    scal[10] = tot[1];                  // ||r||^2 at the start (||b||^2 for x0 = 0)
}

// ---- M = M_BD path: the preconditioner apply is pixel-local, so z = M r and rho = r.z ride in
// the same kernel that updates r (one pass over the pixel-domain vectors per iteration) ---------
// start: z = M r, rho = r.z, |r|^2, flags.  With b != nullptr it also performs the x0 = 0 start of
// the solve in the same pass: r = b, x = 0, and folds SciPy's atol = max(atol, rtol ||b||) in (rtol > 0).
template <int POL>
__global__ void __launch_bounds__(VB) k_bd_reset(const double *__restrict__ inv, int64_t npix, double *__restrict__ r,
                                                 double *__restrict__ z, double *__restrict__ scal, double atol, double rtol,
                                                 const double *__restrict__ b, double *__restrict__ x,
                                                 double *__restrict__ p0) {
    __shared__ double red[32];
    double s[2] = {0.0, 0.0}, tot[2];
    for (int64_t j = (int64_t)blockIdx.x * VB + threadIdx.x; j < npix; j += (int64_t)gridDim.x * VB) {
        double rv[POL], zv[POL];
        if (b != nullptr) {
#pragma unroll
            for (int k = 0; k < POL; ++k) {
                rv[k] = b[POL * j + k];
                r[POL * j + k] = rv[k];
                x[POL * j + k] = 0.0;
            }
        } else {
#pragma unroll
            for (int k = 0; k < POL; ++k) rv[k] = r[POL * j + k];
        }
        bd_z<POL>(inv, j, rv, zv);
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            z[POL * j + k] = zv[k];
            if (p0 != nullptr) p0[POL * j + k] = zv[k];     // first search direction p = z
            s[0] = fma(rv[k], zv[k], s[0]);
            s[1] = fma(rv[k], rv[k], s[1]);
        }
    }
    if (finish_reduce<2>(s, red, tot)) bd_reset_scalars(tot, scal, atol, rtol, b != nullptr);
}

// alpha = rho/pq ; x += alpha p ; r -= alpha q ; z = M r ; rho' = r.z ; |r|^2 ; beta' = rho'/rho
template <int POL>
__global__ void __launch_bounds__(VB) k_bd_update(const double *__restrict__ inv, int64_t npix, const double *__restrict__ p,
                                                  const double *__restrict__ q, double *__restrict__ x,
                                                  double *__restrict__ r, double *__restrict__ z, double *__restrict__ scal) {
    __shared__ double red[32];
    if (scal[7] != 0.0) return;
    const double alpha = scal[4];
    double s[2] = {0.0, 0.0}, tot[2];
    for (int64_t j = (int64_t)blockIdx.x * VB + threadIdx.x; j < npix; j += (int64_t)gridDim.x * VB) {
        double rv[POL], zv[POL];
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            const int64_t i = POL * j + k;
            x[i] = fma(alpha, p[i], x[i]);
            rv[k] = fma(-alpha, q[i], r[i]);
            r[i] = rv[k];
        }
        bd_z<POL>(inv, j, rv, zv);
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            z[POL * j + k] = zv[k];
            s[0] = fma(rv[k], zv[k], s[0]);
            s[1] = fma(rv[k], rv[k], s[1]);
        }
    }
    if (finish_reduce<2>(s, red, tot)) {
        const double rho_old = scal[0];
        scal[1] = rho_old;
        scal[0] = tot[0];
        scal[5] = tot[0] / rho_old;
        scal[3] = tot[1];
        scal[8] += 1.0;
        scal[7] = (sqrt(tot[1]) < scal[6]) ? 1.0 : 0.0;
    }
}

// ---- the whole pixel-domain tail of an M_BD iteration in ONE cooperative launch -----------------
//   pq = p.q ; alpha = rho/pq ; x += alpha p ; r -= alpha q ; z = M r ; rho' = r.z ; |r|^2 ;
//   beta' = rho'/rho ; p = z + beta' p   (the NEXT iteration's search direction) ; flags
// Two grid-wide barriers replace two kernel boundaries; reductions stay deterministic (per-CTA
// partials summed in CTA order, by every CTA identically).
__device__ __forceinline__ double sum_partials(const double *part, int nb, double *red) {
    double s = 0.0;
    for (int i = threadIdx.x; i < nb; i += VB) s += ((volatile const double *)part)[i];
    __shared__ double bc;
    const double t = block_sum(s, red);
    if (threadIdx.x == 0) bc = t;
    __syncthreads();
    const double out = bc;
    __syncthreads();
    return out;
}

template <int POL>
__global__ void __launch_bounds__(VB) k_bd_iter(const double *__restrict__ inv, int64_t npix, double *__restrict__ p,
                                                const double *__restrict__ q, double *__restrict__ x, double *__restrict__ r,
                                                double *__restrict__ z, double *__restrict__ scal) {
    __shared__ double red[32];
    if (scal[7] != 0.0) return;     // uniform over the grid: nobody reaches a grid barrier
    cg::grid_group grid = cg::this_grid();
    const double rho = scal[0];
    const int64_t n = npix * POL;
    const int64_t stride = (int64_t)gridDim.x * VB;
    // phase 1: p.q
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * VB + threadIdx.x; i < n; i += stride) s = fma(p[i], q[i], s);
    s = block_sum(s, red);
    if (threadIdx.x == 0) g_part[2][blockIdx.x] = s;
    grid.sync();
    const double pq = sum_partials(g_part[2], gridDim.x, red);
    const double alpha = rho / pq;
    // phase 2: x, r, z and the two reductions
    double s0 = 0.0, s1 = 0.0;
    for (int64_t j = (int64_t)blockIdx.x * VB + threadIdx.x; j < npix; j += stride) {
        double rv[POL], zv[POL];
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            const int64_t i = POL * j + k;
            x[i] = fma(alpha, p[i], x[i]);
            rv[k] = fma(-alpha, q[i], r[i]);
            r[i] = rv[k];
        }
        bd_z<POL>(inv, j, rv, zv);
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            z[POL * j + k] = zv[k];
            s0 = fma(rv[k], zv[k], s0);
            s1 = fma(rv[k], rv[k], s1);
        }
    }
    s0 = block_sum(s0, red);
    s1 = block_sum(s1, red);
    if (threadIdx.x == 0) { g_part[0][blockIdx.x] = s0; g_part[1][blockIdx.x] = s1; }
    grid.sync();
    const double rho_new = sum_partials(g_part[0], gridDim.x, red);
    const double rr = sum_partials(g_part[1], gridDim.x, red);
    const double beta = rho_new / rho;
    // phase 3: next search direction (same pixel -> thread mapping as phase 2: z is this thread's own)
    for (int64_t j = (int64_t)blockIdx.x * VB + threadIdx.x; j < npix; j += stride) {
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            const int64_t i = POL * j + k;
            p[i] = fma(beta, p[i], z[i]);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        scal[1] = rho;
        scal[0] = rho_new;
        scal[2] = pq;
        scal[3] = rr;
        scal[4] = alpha;
        scal[5] = beta;
        scal[8] += 1.0;
        scal[7] = (sqrt(rr) < scal[6]) ? 1.0 : 0.0;
    }
}

// ---- coalesced M_BD tail: the kernels above give each thread one pixel and touch v[POL j + k] with
// 8-byte accesses at a POL*8-byte stride, so a warp store writes 8 of every 24 bytes of the sectors
// it touches (POL = 3).  The kernels below give each warp tiles of TP consecutive pixels, i.e. the
// contiguous span [POL TP t, POL TP (t+1)) of every pixel-domain vector; lane l moves the 16-byte
// pieces 2(l + 32k), k < POL, of that span.  z = M_BD r needs whole pixels: the warp transposes
// through its own shared-memory slot (flat layout in, lane = pixel out) and inv, POL = 3, is staged
// the same way.  k_bd_iter_tiled keeps p in registers and q, then r and z, in shared memory from
// phase 1 to phase 3: p, q, x, r and inv are read once, x, r and p written once, z never leaves the
// chip (216 B/pixel at POL = 3 instead of k_bd_iter's 336).
constexpr int TP = 64;            // pixels per warp tile
constexpr int TB = 256;           // threads per CTA of the tiled kernels (== VB: sum_partials strides by VB)
constexpr int TW = TB / 32;
// Tiles per warp k_bd_iter_tiled holds on chip (its npix bound: TPW TP pixels per warp of the co-resident grid) and
// the CTAs per SM its register budget targets; CTAs per SM the start kernel's register budget targets.  Chosen by
// the sweep in DESIGN section 5; the macros exist so that the sweep can be repeated.
#ifndef CM2_BD_TPW
#define CM2_BD_TPW 4
#endif
#ifndef CM2_BD_ITER_CTAS
#define CM2_BD_ITER_CTAS 2
#endif
#ifndef CM2_BD_RESET_CTAS
#define CM2_BD_RESET_CTAS 4
#endif
constexpr int TPW = CM2_BD_TPW;
static_assert(TB == VB, "sum_partials and finish_reduce stride by VB");

template <int POL>
constexpr int tile_smem_doubles(int tiles) { return TW * (tiles * POL * TP + (POL == 3 ? 6 * TP : 0)); }

__device__ __forceinline__ double2 ld2(const double *__restrict__ v, int64_t e, int64_t n) {
    if (e + 1 < n) return *reinterpret_cast<const double2 *>(v + e);
    return make_double2(e < n ? v[e] : 0.0, 0.0);
}
__device__ __forceinline__ void st2(double *__restrict__ v, int64_t e, int64_t n, double2 a) {
    if (e + 1 < n) *reinterpret_cast<double2 *>(v + e) = a;
    else if (e < n) v[e] = a.x;
}

// z = M_BD r for the pixels j0 .. j0+TP-1 of one tile.  sv holds the tile's r in flat layout and
// receives z in its place; lane handles pixels lane and lane + 32 and adds r.z to s0 and |r|^2 to s1.
// POL = 3 stages the tile's inv blocks (6 TP doubles, coalesced) in sinv; POL 1 and 2 use a third or
// half of each 48-byte block and read it in place.  Ends with a __syncwarp: sv and sinv may be reused.
// the tile's inv blocks in lane pieces (POL = 3 only: 6 TP doubles, 16-byte pieces 2(lane + 32k), k < 6)
template <int POL>
__device__ __forceinline__ void tile_inv_load(const double *__restrict__ inv, int64_t j0, int64_t npix, int lane,
                                              double2 (&iv)[6]) {
    if constexpr (POL == 3) {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const int64_t e = 6 * j0 + 2 * (lane + 32 * k);
            iv[k] = e < 6 * npix ? __ldg(reinterpret_cast<const double2 *>(inv + e)) : make_double2(0.0, 0.0);
        }
    }
}

// iv: the tile's inv pieces from tile_inv_load (POL = 3; unused otherwise)
template <int POL>
__device__ __forceinline__ void tile_z(const double2 (&iv)[6], const double *__restrict__ inv, double *sinv, double *sv,
                                       int64_t j0, int64_t npix, int lane, double &s0, double &s1) {
    if constexpr (POL == 3) {
#pragma unroll
        for (int k = 0; k < 6; ++k) reinterpret_cast<double2 *>(sinv)[lane + 32 * k] = iv[k];
    }
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int pp = lane + 32 * h;
        if (j0 + pp < npix) {
            double rv[POL], zv[POL];
#pragma unroll
            for (int k = 0; k < POL; ++k) rv[k] = sv[POL * pp + k];
            if constexpr (POL == 3) {
                const double2 *b2 = reinterpret_cast<const double2 *>(sinv) + 3 * pp;
                const double2 q0 = b2[0], q1 = b2[1], q2 = b2[2];
                zv[0] = q0.x * rv[0] + q0.y * rv[1] + q1.x * rv[2];
                zv[1] = q0.y * rv[0] + q1.y * rv[1] + q2.x * rv[2];
                zv[2] = q1.x * rv[0] + q2.x * rv[1] + q2.y * rv[2];
            } else {
                bd_z<POL>(inv, j0 + pp, rv, zv);
            }
#pragma unroll
            for (int k = 0; k < POL; ++k) {
                sv[POL * pp + k] = zv[k];
                s0 = fma(rv[k], zv[k], s0);
                s1 = fma(rv[k], rv[k], s1);
            }
        }
    }
    __syncwarp();
}

// x0 = 0 start with the first search direction: r = b, x = 0, p0 = z = M r, rho, |r|^2, flags.
// Reads b and inv, writes r, x and p0 (144 B/pixel at POL = 3); z is not stored.
template <int POL>
__global__ void __launch_bounds__(TB, CM2_BD_RESET_CTAS) k_bd_reset_tiled(const double *__restrict__ inv, int64_t npix, double *__restrict__ r,
                                                       double *__restrict__ scal, double atol, double rtol,
                                                       const double *__restrict__ b, double *__restrict__ x,
                                                       double *__restrict__ p0) {
    extern __shared__ double2 tsm[];
    __shared__ double red[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *sv = reinterpret_cast<double *>(tsm) + warp * (POL * TP);
    double *sinv = reinterpret_cast<double *>(tsm) + TW * POL * TP + warp * (6 * TP);
    const int64_t n = npix * POL, ntile = (npix + TP - 1) / TP;
    double s[2] = {0.0, 0.0}, tot[2];
    for (int64_t t = (int64_t)blockIdx.x * TW + warp; t < ntile; t += (int64_t)gridDim.x * TW) {
        const int64_t e0 = t * (POL * TP);
        double2 iv[6];
        tile_inv_load<POL>(inv, t * TP, npix, lane, iv);       // in flight together with b
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            const int o = 2 * (lane + 32 * k);
            const double2 bv = ld2(b, e0 + o, n);
            st2(r, e0 + o, n, bv);
            st2(x, e0 + o, n, make_double2(0.0, 0.0));
            reinterpret_cast<double2 *>(sv)[o / 2] = bv;
        }
        tile_z<POL>(iv, inv, sinv, sv, t * TP, npix, lane, s[0], s[1]);
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            const int o = 2 * (lane + 32 * k);
            st2(p0, e0 + o, n, reinterpret_cast<const double2 *>(sv)[o / 2]);
        }
        __syncwarp();
    }
    if (finish_reduce<2>(s, red, tot)) bd_reset_scalars(tot, scal, atol, rtol, true);
}

// k_bd_iter's recurrence with the tiled IO.  Warp w of the W in the grid owns tiles w, w + W, ...,
// w + (TPW-1) W: the launch requires npix <= W TPW TP.
template <int POL>
__global__ void __launch_bounds__(TB, CM2_BD_ITER_CTAS) k_bd_iter_tiled(const double *__restrict__ inv, int64_t npix, double *__restrict__ p,
                                                         const double *__restrict__ q, double *__restrict__ x,
                                                         double *__restrict__ r, double *__restrict__ scal) {
    extern __shared__ double2 tsm[];
    __shared__ double red[32];
    if (scal[7] != 0.0) return;     // uniform over the grid: nobody reaches a grid barrier
    cg::grid_group grid = cg::this_grid();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *stash = reinterpret_cast<double *>(tsm) + warp * (TPW * POL * TP);    // q, then r, then z
    double *sinv = reinterpret_cast<double *>(tsm) + TW * TPW * POL * TP + warp * (6 * TP);
    const int64_t n = npix * POL, ntile = (npix + TP - 1) / TP;
    const int64_t w = (int64_t)blockIdx.x * TW + warp, nw = (int64_t)gridDim.x * TW;
    const double rho = scal[0];
    double2 pv[TPW][POL];
    // phase 1: p.q ; p stays in registers, q goes to the warp's slot
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < TPW; ++i) {
        const int64_t t = w + nw * i, e0 = t * (POL * TP);
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            const int o = 2 * (lane + 32 * k);
            pv[i][k] = make_double2(0.0, 0.0);
            if (t < ntile) {
                pv[i][k] = ld2(p, e0 + o, n);
                const double2 qv = ld2(q, e0 + o, n);
                reinterpret_cast<double2 *>(stash + i * (POL * TP))[o / 2] = qv;
                s = fma(pv[i][k].x, qv.x, s);
                s = fma(pv[i][k].y, qv.y, s);
            }
        }
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) g_part[2][blockIdx.x] = s;
    grid.sync();
    const double pq = sum_partials(g_part[2], gridDim.x, red);
    const double alpha = rho / pq;
    // phase 2: x += alpha p ; r -= alpha q ; z = M r (replaces q in the slot) ; r.z ; |r|^2
    double s0 = 0.0, s1 = 0.0;
#pragma unroll
    for (int i = 0; i < TPW; ++i) {
        const int64_t t = w + nw * i, e0 = t * (POL * TP);
        if (t < ntile) {
            double *sv = stash + i * (POL * TP);
#pragma unroll
            for (int k = 0; k < POL; ++k) {
                const int o = 2 * (lane + 32 * k);
                double2 xv = ld2(x, e0 + o, n), rv = ld2(r, e0 + o, n);
                const double2 qv = reinterpret_cast<const double2 *>(sv)[o / 2];
                xv.x = fma(alpha, pv[i][k].x, xv.x);
                xv.y = fma(alpha, pv[i][k].y, xv.y);
                rv.x = fma(-alpha, qv.x, rv.x);
                rv.y = fma(-alpha, qv.y, rv.y);
                st2(x, e0 + o, n, xv);
                st2(r, e0 + o, n, rv);
                reinterpret_cast<double2 *>(sv)[o / 2] = rv;
            }
            double2 iv[6];       // loaded after x and r: loading it with them needs 24 more registers
            tile_inv_load<POL>(inv, t * TP, npix, lane, iv);
            tile_z<POL>(iv, inv, sinv, sv, t * TP, npix, lane, s0, s1);
        }
    }
    s0 = block_sum(s0, red);
    s1 = block_sum(s1, red);
    if (threadIdx.x == 0) { g_part[0][blockIdx.x] = s0; g_part[1][blockIdx.x] = s1; }
    grid.sync();
    const double rho_new = sum_partials(g_part[0], gridDim.x, red);
    const double rr = sum_partials(g_part[1], gridDim.x, red);
    const double beta = rho_new / rho;
    // phase 3: p = z + beta p
#pragma unroll
    for (int i = 0; i < TPW; ++i) {
        const int64_t t = w + nw * i, e0 = t * (POL * TP);
        if (t < ntile) {
            const double *sv = stash + i * (POL * TP);
#pragma unroll
            for (int k = 0; k < POL; ++k) {
                const int o = 2 * (lane + 32 * k);
                const double2 zv = reinterpret_cast<const double2 *>(sv)[o / 2];
                st2(p, e0 + o, n, make_double2(fma(beta, pv[i][k].x, zv.x), fma(beta, pv[i][k].y, zv.y)));
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        scal[1] = rho;
        scal[0] = rho_new;
        scal[2] = pq;
        scal[3] = rr;
        scal[4] = alpha;
        scal[5] = beta;
        scal[8] += 1.0;
        scal[7] = (sqrt(rr) < scal[6]) ? 1.0 : 0.0;
    }
}

// ---- launch geometry, computed once per (device, POL) instead of once per launch ---------------------
constexpr int MAXDEV = 64;
struct TailGeom {
    int ready;
    int iter_grid;          // co-resident CTAs of k_bd_iter_tiled (0: unusable)
    int reset_grid;         // CTAs of a k_bd_reset_tiled launch over a large npix
    int strided_iter_grid;  // co-resident CTAs of k_bd_iter (capped at 4 per SM as before)
};
static TailGeom g_geom[MAXDEV][3];

template <int POL>
static const TailGeom &tail_geom() {
    int dev = 0;
    cudaGetDevice(&dev);
    TailGeom &g = g_geom[dev < 0 || dev >= MAXDEV ? 0 : dev][POL - 1];
    if (g.ready) return g;
    const int sms = sm_count();
    int per_sm = 0;
    const size_t smi = sizeof(double) * tile_smem_doubles<POL>(TPW);
    if (cudaFuncSetAttribute(k_bd_iter_tiled<POL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smi) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bd_iter_tiled<POL>, TB, smi) != cudaSuccess)
        per_sm = 0;
    g.iter_grid = (int)std::min<int64_t>((int64_t)sms * per_sm, MAXP);
    per_sm = 0;
    const size_t smr = sizeof(double) * tile_smem_doubles<POL>(1);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bd_reset_tiled<POL>, TB, smr) != cudaSuccess) per_sm = 1;
    g.reset_grid = (int)std::min<int64_t>((int64_t)sms * std::max(1, std::min(per_sm, CM2_BD_RESET_CTAS)), MAXP);
    per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bd_iter<POL>, VB, 0);
    g.strided_iter_grid = (int)std::min<int64_t>((int64_t)sms * std::max(1, std::min(per_sm, 4)), MAXP);
    cudaGetLastError();
    // a benign race: two host threads on one device compute the same values; `ready` is set after them
    g.ready = 1;
    return g;
}

// the largest npix k_bd_iter_tiled covers on the current device (above it cm2_pcg_bd_iter runs k_bd_iter)
template <int POL>
static int64_t tiled_iter_max_npix() { return (int64_t)tail_geom<POL>().iter_grid * TW * TPW * TP; }

}  // namespace cm2

using namespace cm2;

extern "C" int cm2_dot(const double *a, const double *b, int64_t n, double *out, cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0, "n < 0");
    return launch(k_dot, capped_grid(cdiv(n, VB), 4, MAXP), VB, 0, as_stream(stream), a, b, n, out);
}

extern "C" int cm2_axpby(double alpha, const double *x, double beta, double *y, int64_t n, cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0, "n < 0");
    if (n == 0) return CM2_OK;
    return launch(k_axpby, capped_grid(cdiv(n, VB), 4, MAXP), VB, 0, as_stream(stream), alpha, x, beta, y, n);
}

extern "C" int cm2_pcg_reset(const double *r, int64_t n, double *scal, double atol, cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0, "n < 0");
    return launch(k_reset, capped_grid(cdiv(n, VB), 4, MAXP), VB, 0, as_stream(stream), r, n, scal, atol);
}

extern "C" int cm2_pcg_update_p(const double *r, const double *z, double *p, int64_t n, double *scal,
                                cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0, "n < 0");
    cudaStream_t st = as_stream(stream);
    const int g = capped_grid(cdiv(n, VB), 4, MAXP);
    k_rho<<<g, VB, 0, st>>>(r, z, n, scal);
    CM2_LAUNCHED();
    return launch(k_update_p, g, VB, 0, st, z, p, n, scal);
}

extern "C" int cm2_pcg_update_xr(const double *p, const double *q, double *x, double *r, int64_t n, double *scal,
                                 cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0, "n < 0");
    cudaStream_t st = as_stream(stream);
    const int g = capped_grid(cdiv(n, VB), 4, MAXP);
    k_pq<<<g, VB, 0, st>>>(p, q, n, scal);
    CM2_LAUNCHED();
    return launch(k_update_xr, g, VB, 0, st, p, q, x, r, n, scal);
}

// development/test hook (cm2_pcg_bd_tail_strided): run the one-thread-per-pixel kernels at every npix
static int g_force_strided = 0;

template <int POL>
static int launch_bd_reset_tiled(const double *inv, int64_t npix, double *r, double *scal, double atol, double rtol,
                                 const double *b, double *x, double *p0, cudaStream_t st) {
    const int64_t need = (npix + TP * TW - 1) / (TP * TW);
    const int g = (int)std::max<int64_t>(1, std::min<int64_t>(need, tail_geom<POL>().reset_grid));
    return launch(k_bd_reset_tiled<POL>, g, TB, sizeof(double) * tile_smem_doubles<POL>(1), st, inv, npix, r, scal, atol, rtol,
                  b, x, p0);
}

extern "C" int cm2_pcg_bd_reset(const double *inv, int64_t npix, int pol, double *r, double *z, double *scal,
                                double atol, double rtol, const double *b, double *x, double *p0, cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && pol >= 1 && pol <= 3, "bad npix/pol");
    CM2_REQUIRE(aligned(inv, 16), "inverse blocks must be 16-byte aligned");
    CM2_REQUIRE((b == nullptr) == (x == nullptr), "b and x go together");
    cudaStream_t st = as_stream(stream);
    // the x0 = 0 start that hands out p0 = z needs no z: coalesced tiles when the vectors allow 16-byte access
    if (b != nullptr && p0 != nullptr && !g_force_strided && aligned(b, 16) && aligned(r, 16) && aligned(x, 16) &&
        aligned(p0, 16))
        return with_pol(pol, [&](auto P) { return launch_bd_reset_tiled<P>(inv, npix, r, scal, atol, rtol, b, x, p0, st); });
    const int g = capped_grid(cdiv(npix, VB), 4, MAXP);
    return with_pol(pol, [&](auto P) {
        return launch(k_bd_reset<P>, g, VB, 0, st, inv, npix, r, z, scal, atol, rtol, b, x, p0);
    });
}

extern "C" int cm2_pcg_bd_update_p(const double *z, double *p, int64_t n, double *scal, cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0, "n < 0");
    return launch(k_update_p, capped_grid(cdiv(n, VB), 4, MAXP), VB, 0, as_stream(stream), z, p, n, scal);
}

extern "C" int cm2_pcg_bd_update(const double *inv, int64_t npix, int pol, const double *p, const double *q, double *x,
                                 double *r, double *z, double *scal, cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && pol >= 1 && pol <= 3, "bad npix/pol");
    CM2_REQUIRE(aligned(inv, 16), "inverse blocks must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    const int64_t n = npix * pol;
    k_pq<<<capped_grid(cdiv(n, VB), 4, MAXP), VB, 0, st>>>(p, q, n, scal);
    CM2_LAUNCHED();
    const int g = capped_grid(cdiv(npix, VB), 4, MAXP);
    return with_pol(pol, [&](auto P) { return launch(k_bd_update<P>, g, VB, 0, st, inv, npix, p, q, x, r, z, scal); });
}

// test hook (cm2_pcg_bd_iter_refuse): make the cooperative launch fail the way a GPU that refuses
// cooperative launches does (too many CTAs for co-residency), to exercise the fallback
static int g_refuse_coop = 0;

template <int POL>
static int launch_bd_iter(const double *inv, int64_t npix, double *p, const double *q, double *x, double *r, double *z,
                          double *scal, cudaStream_t st) {
    const TailGeom &geo = tail_geom<POL>();
    // all CTAs co-resident: grid barriers are safe
    const bool tiled = !g_force_strided && geo.iter_grid > 0 && npix <= tiled_iter_max_npix<POL>() && aligned(p, 16) && aligned(q, 16) &&
                       aligned(x, 16) && aligned(r, 16);
    int64_t g = tiled ? geo.iter_grid : geo.strided_iter_grid;
    const int64_t need = tiled ? (npix + TP * TW - 1) / (TP * TW) : (npix + VB - 1) / VB;
    if (need < g) g = need < 1 ? 1 : need;
    if (g_refuse_coop) g = (int64_t)sm_count() * 64;     // more CTAs than can be co-resident: the launch is refused
    cudaError_t e;
    if (tiled) {
        void *args[] = {(void *)&inv, (void *)&npix, (void *)&p, (void *)&q, (void *)&x, (void *)&r, (void *)&scal};
        e = cudaLaunchCooperativeKernel((const void *)k_bd_iter_tiled<POL>, dim3((unsigned)g), dim3(TB), args,
                                        sizeof(double) * tile_smem_doubles<POL>(TPW), st);
    } else {
        void *args[] = {(void *)&inv, (void *)&npix, (void *)&p, (void *)&q, (void *)&x, (void *)&r, (void *)&z, (void *)&scal};
        e = cudaLaunchCooperativeKernel((const void *)k_bd_iter<POL>, dim3((unsigned)g), dim3(VB), args, 0, st);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();      // clear the runtime's sticky last-error: the caller falls back to the 3-kernel tail
        return set_error(CM2_ERR_CUDA, "cm2_pcg_bd_iter: %s", cudaGetErrorString(e));
    }
    count_launch();
    return CM2_OK;
}

extern "C" int cm2_pcg_bd_iter_refuse(int on) {
    const int old = g_refuse_coop;
    g_refuse_coop = on ? 1 : 0;
    return old;
}

extern "C" int cm2_pcg_bd_tail_strided(int on) {
    const int old = g_force_strided;
    g_force_strided = on ? 1 : 0;
    return old;
}

extern "C" int64_t cm2_pcg_bd_iter_max_npix(int pol) {
    if (pol < 1 || pol > 3) return 0;
    return with_pol(pol, [](auto P) { return tiled_iter_max_npix<P>(); });
}

extern "C" int cm2_pcg_bd_iter(const double *inv, int64_t npix, int pol, double *p, const double *q, double *x,
                               double *r, double *z, double *scal, cm2_stream_t stream) {
    CM2_REQUIRE(npix >= 0 && pol >= 1 && pol <= 3, "bad npix/pol");
    CM2_REQUIRE(aligned(inv, 16), "inverse blocks must be 16-byte aligned");
    cudaStream_t st = as_stream(stream);
    return with_pol(pol, [&](auto P) { return launch_bd_iter<P>(inv, npix, p, q, x, r, z, scal, st); });
}
