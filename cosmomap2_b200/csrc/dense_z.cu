// cosmomap2_b200 -- the dense tall-skinny contractions of the deflation path on the fp64 tensor cores
// (sm_100a, DMMA: mma.sync.m8n8k4.f64).
//
//   cm2_dense_gram      C = X^T Y        (r1 x r2 from two n x r matrices, ONE pass over X and Y)
//                       E = Z^T (A Z):  CoarseLO.__init__ -> dgemm(Z, Az.T), interfaces/linearoperators.py:1019,
//                       utilities/linear_algebra_funcs.py:16-29
//   cm2_dense_combine   Z = V U          (n x r from the n x m Krylov basis and the m x r Ritz matrix)
//                       Ritz vectors:   find_ritz_eigenvalues / kp.utils.ritz, interfaces/deflationlib.py:204-219;
//                       build_Z :140-184; the thick restart of the device eigsh
//
// Tall-skinny matrices are column-major with a leading dimension (each column contiguous in HBM).
// Both kernels stream the tall matrices exactly once with 256-bit loads and are bound by HBM (gram:
// 8 (r1 + r2) bytes per row against 2 r1 r2 flop) or by the fp64 tensor pipe (combine at r = 32:
// 8 flop per byte of V).  The m8n8k4 fragments are filled straight from global memory:
//   * gram: A[i][k] = X[k][i], B[k][j] = Y[k][j]; the k index (rows of X, Y) is summed over, so the four
//     MMAs of a 16-row chunk may use ANY assignment of rows to k slots as long as A and B agree: lane
//     (g, t) loads rows k0 + 4t .. k0 + 4t + 3 of column 8 mb + g with one LDG.256 and feeds element s
//     to MMA s.  Per chunk and lane: MB + NB loads, 4 MB NB DMMAs.
//   * combine: A[row][k] = V[row][k]; the 8 rows of an m-block are independent, so lane (g, t) takes rows
//     R0 + 4g .. R0 + 4g + 3 of column k0 + t (one LDG.256) and row R0 + 4g + mb belongs to m-block mb; the
//     C fragments then hold 4 consecutive rows per lane and column: 256-bit stores.  U sits in shared
//     memory (padded so that the B-fragment reads are bank-conflict free).
// Reductions are deterministic: warps are added in warp order inside a CTA, CTA partials in CTA order
// by a second tiny kernel.
#include "cm2_common.cuh"

namespace cm2 {

constexpr int GR_THREADS = 128;          // 4 warps per CTA
constexpr int GR_MAXCTA = 1184;          // 148 SMs x 8

__device__ __forceinline__ void dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// 4 consecutive rows [k, k+4) of column `col` (nullptr = a padding column: zeros), rows >= n read as 0
__device__ __forceinline__ void load4(const double *__restrict__ col, int64_t k, int64_t n, bool vec, double (&v)[4]) {
    if (col == nullptr) {
        v[0] = v[1] = v[2] = v[3] = 0.0;
    } else if (vec && k + 4 <= n) {
        const D4 t = ld_stream_d4(col + k);
        v[0] = t.v[0]; v[1] = t.v[1]; v[2] = t.v[2]; v[3] = t.v[3];
    } else {
#pragma unroll
        for (int s = 0; s < 4; ++s) v[s] = (k + s < n) ? __ldcs(col + k + s) : 0.0;
    }
}

// partial[cta][(8 MB) x (8 NB)] (column-major, ld = 8 MB) = sum over the CTA's 16-row chunks of X^T Y
template <int MB, int NB>
__global__ void __launch_bounds__(GR_THREADS) k_gram_partial(const double *__restrict__ X, int64_t ldx, int r1,
                                                             const double *__restrict__ Y, int64_t ldy, int r2, int64_t n,
                                                             bool vec, double *__restrict__ partial) {
    constexpr int NW = GR_THREADS / 32;
    __shared__ double sacc[NW][MB * NB * 64];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const double *xc[MB], *yc[NB];
#pragma unroll
    for (int mb = 0; mb < MB; ++mb) xc[mb] = (8 * mb + g < r1) ? X + (int64_t)(8 * mb + g) * ldx : nullptr;
#pragma unroll
    for (int nb = 0; nb < NB; ++nb) yc[nb] = (8 * nb + g < r2) ? Y + (int64_t)(8 * nb + g) * ldy : nullptr;
    double acc[MB][NB][2];
#pragma unroll
    for (int mb = 0; mb < MB; ++mb)
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
    const int64_t nchunks = (n + 15) / 16;
    const int64_t nwarps = (int64_t)gridDim.x * NW;
    for (int64_t c = (int64_t)blockIdx.x * NW + warp; c < nchunks; c += nwarps) {
        const int64_t k = c * 16 + 4 * t;
        double a[MB][4], b[NB][4];
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) load4(xc[mb], k, n, vec, a[mb]);
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) load4(yc[nb], k, n, vec, b[nb]);
#pragma unroll
        for (int s = 0; s < 4; ++s)
#pragma unroll
            for (int mb = 0; mb < MB; ++mb)
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) dmma(acc[mb][nb][0], acc[mb][nb][1], a[mb][s], b[nb][s]);
    }
    // C fragment: row i = 8 mb + g, columns j = 8 nb + 2 t + {0, 1}
#pragma unroll
    for (int mb = 0; mb < MB; ++mb)
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) {
            sacc[warp][(8 * mb + g) + (8 * MB) * (8 * nb + 2 * t)] = acc[mb][nb][0];
            sacc[warp][(8 * mb + g) + (8 * MB) * (8 * nb + 2 * t + 1)] = acc[mb][nb][1];
        }
    __syncthreads();
    for (int e = threadIdx.x; e < MB * NB * 64; e += GR_THREADS) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) s += sacc[w][e];
        partial[(int64_t)blockIdx.x * (MB * NB * 64) + e] = s;
    }
}

// out[i + ldo j] = sum over CTAs (in order) of partial[cta][i + ldp j]
__global__ void k_gram_final(const double *__restrict__ partial, int ncta, int ldp, int stride, int r1, int r2,
                             double *__restrict__ out, int64_t ldo) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < r1 * r2; e += gridDim.x * blockDim.x) {
        const int i = e % r1, j = e / r1;
        double s = 0.0;
        for (int b = 0; b < ncta; ++b) s += partial[(int64_t)b * stride + i + ldp * j];
        out[i + ldo * j] = s;
    }
}

template <int MB, int NB>
static void launch_gram(int grid, cudaStream_t st, const double *X, int64_t ldx, int r1, const double *Y, int64_t ldy, int r2,
                        int64_t n, bool vec, double *partial) {
    k_gram_partial<MB, NB><<<grid, GR_THREADS, 0, st>>>(X, ldx, r1, Y, ldy, r2, n, vec, partial);
}

static int blocks_for(int r) { return r <= 8 ? 1 : (r <= 16 ? 2 : 4); }

// ---- combine ---------------------------------------------------------------------------------------
constexpr int CB_THREADS = 256;

// Z[:, j0 + j] = sum_i V[:, i] U[i, j0 + j] for j < r (<= 8 NB); U staged in shared memory as
// su[k + mpad j], mpad = 4 (mod 16) >= m rounded up to a multiple of 4, zero padded.
template <int NB>
__global__ void __launch_bounds__(CB_THREADS) k_combine(const double *__restrict__ V, int64_t ldv, int64_t n, int m,
                                                        const double *__restrict__ U, int64_t ldu, int r,
                                                        double *__restrict__ Z, int64_t ldz, int mpad, bool vec) {
    extern __shared__ double su[];
    for (int e = threadIdx.x; e < mpad * 8 * NB; e += CB_THREADS) {
        const int k = e % mpad, j = e / mpad;
        su[e] = (k < m && j < r) ? U[k + ldu * j] : 0.0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int64_t ntiles = (n + 31) / 32;
    const int64_t nwarps = (int64_t)gridDim.x * (CB_THREADS / 32);
    const int m4 = (m + 3) & ~3;
    for (int64_t tile = (int64_t)blockIdx.x * (CB_THREADS / 32) + (threadIdx.x >> 5); tile < ntiles; tile += nwarps) {
        const int64_t row = tile * 32 + 4 * g;               // this lane's rows: row .. row + 3 (m-block mb <-> row + mb)
        double acc[4][NB][2];
#pragma unroll
        for (int mb = 0; mb < 4; ++mb)
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) acc[mb][nb][0] = acc[mb][nb][1] = 0.0;
#pragma unroll 2
        for (int k0 = 0; k0 < m4; k0 += 4) {
            double a[4];
            load4(k0 + t < m ? V + (int64_t)(k0 + t) * ldv : nullptr, row, n, vec, a);
            double b[NB];
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) b[nb] = su[k0 + t + mpad * (8 * nb + g)];
#pragma unroll
            for (int mb = 0; mb < 4; ++mb)
#pragma unroll
                for (int nb = 0; nb < NB; ++nb) dmma(acc[mb][nb][0], acc[mb][nb][1], a[mb], b[nb]);
        }
        // C fragment of (mb, nb): row + mb, columns 8 nb + 2 t + {0, 1}
#pragma unroll
        for (int nb = 0; nb < NB; ++nb)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int j = 8 * nb + 2 * t + e;
                if (j >= r) continue;
                double *zc = Z + (int64_t)j * ldz + row;
                if (vec && row + 4 <= n) {
                    D4 o;
#pragma unroll
                    for (int mb = 0; mb < 4; ++mb) o.v[mb] = acc[mb][nb][e];
                    st_stream_d4(zc, o);
                } else {
#pragma unroll
                    for (int mb = 0; mb < 4; ++mb)
                        if (row + mb < n) zc[mb] = acc[mb][nb][e];
                }
            }
    }
}

template <int NB>
static int launch_combine(const double *V, int64_t ldv, int64_t n, int m, const double *U, int64_t ldu, int r, double *Z,
                          int64_t ldz, bool vec, cudaStream_t st) {
    int mpad = (m + 3) & ~3;
    while ((mpad & 15) != 4) mpad += 4;
    const size_t smem = sizeof(double) * (size_t)mpad * 8 * NB;
    auto kern = k_combine<NB>;
    if (smem > 200 * 1024) return set_error(CM2_ERR_UNSUPPORTED, "cm2_dense_combine: m = %d is too large for one panel", m);
    CM2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t tiles = (n + 31) / 32;
    return launch(kern, persistent_grid(kern, CB_THREADS, smem, (tiles + 7) / 8, 4), CB_THREADS, smem, st, V, ldv, n, m, U,
                  ldu, r, Z, ldz, mpad, vec);
}

}  // namespace cm2

using namespace cm2;

extern "C" int64_t cm2_dense_gram_work_doubles(void) { return (int64_t)GR_MAXCTA * 32 * 32; }

/* out (r1 x r2, column-major, leading dimension ldo) = X^T Y; X: n x r1 (ldx), Y: n x r2 (ldy), column-major.
 * One pass over X and Y per 32 x 32 panel of out (r1, r2 <= 32: exactly one). */
extern "C" int cm2_dense_gram(const double *X, int64_t ldx, int r1, const double *Y, int64_t ldy, int r2, int64_t n,
                              double *out, int64_t ldo, double *work, cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0 && r1 >= 1 && r2 >= 1 && ldx >= n && ldy >= n && ldo >= r1, "bad sizes");
    CM2_REQUIRE(work != nullptr, "work (cm2_dense_gram_work_doubles) required");
    cudaStream_t st = as_stream(stream);
    const bool vec = aligned(X, 32) && aligned(Y, 32) && (ldx % 4 == 0) && (ldy % 4 == 0);
    const int grid = capped_grid(cdiv(cdiv(n, 16), 4), 4, GR_MAXCTA);
    for (int i0 = 0; i0 < r1; i0 += 32) {
        for (int j0 = 0; j0 < r2; j0 += 32) {
            const int p1 = r1 - i0 < 32 ? r1 - i0 : 32, p2 = r2 - j0 < 32 ? r2 - j0 : 32;
            const int mb = blocks_for(p1), nb = blocks_for(p2);
            const double *Xp = X + (int64_t)i0 * ldx, *Yp = Y + (int64_t)j0 * ldy;
#define CM2_GRAM(MB, NB) launch_gram<MB, NB>(grid, st, Xp, ldx, p1, Yp, ldy, p2, n, vec, work)
            if (mb == 1 && nb == 1) CM2_GRAM(1, 1);
            else if (mb == 1 && nb == 2) CM2_GRAM(1, 2);
            else if (mb == 1 && nb == 4) CM2_GRAM(1, 4);
            else if (mb == 2 && nb == 1) CM2_GRAM(2, 1);
            else if (mb == 2 && nb == 2) CM2_GRAM(2, 2);
            else if (mb == 2 && nb == 4) CM2_GRAM(2, 4);
            else if (mb == 4 && nb == 1) CM2_GRAM(4, 1);
            else if (mb == 4 && nb == 2) CM2_GRAM(4, 2);
            else CM2_GRAM(4, 4);
#undef CM2_GRAM
            CM2_LAUNCHED();
            k_gram_final<<<4, 256, 0, st>>>(work, grid, 8 * mb, mb * nb * 64, p1, p2, out + i0 + ldo * (int64_t)j0, ldo);
            CM2_LAUNCHED();
        }
    }
    return CM2_OK;
}

/* Z (n x r, ldz) = V (n x m, ldv) U (m x r, ldu), all column-major; Z must not overlap V. */
extern "C" int cm2_dense_combine(const double *V, int64_t ldv, int64_t n, int m, const double *U, int64_t ldu, int r,
                                 double *Z, int64_t ldz, cm2_stream_t stream) {
    CM2_REQUIRE(n >= 0 && m >= 1 && r >= 1 && ldv >= n && ldz >= n && ldu >= m, "bad sizes");
    if (n == 0) return CM2_OK;
    cudaStream_t st = as_stream(stream);
    const bool vec = aligned(V, 32) && aligned(Z, 32) && (ldv % 4 == 0) && (ldz % 4 == 0);
    for (int j0 = 0; j0 < r; j0 += 32) {
        const int p = r - j0 < 32 ? r - j0 : 32;
        const double *Up = U + (int64_t)j0 * ldu;
        double *Zp = Z + (int64_t)j0 * ldz;
        int rc;
        if (p <= 8) rc = launch_combine<1>(V, ldv, n, m, Up, ldu, p, Zp, ldz, vec, st);
        else if (p <= 16) rc = launch_combine<2>(V, ldv, n, m, Up, ldu, p, Zp, ldz, vec, st);
        else rc = launch_combine<4>(V, ldv, n, m, Up, ldu, p, Zp, ldz, vec, st);
        if (rc) return rc;
    }
    return CM2_OK;
}
