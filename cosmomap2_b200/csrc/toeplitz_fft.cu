// cosmomap2_b200 -- banded symmetric Toeplitz apply by overlap-save FFT in shared memory (sm_100a).
//
// ToeplitzLO.mult (interfaces/linearoperators.py:582-595) is y_j = sum_{|k|<L} a_|k| v_{j-k} with
// zero boundaries: 2(2L-1) flop/sample done directly, i.e. 16 382 flop/sample at the L = 4096 of
// configs[2] -- 100x more time than the 16 B/sample of HBM traffic.  Here each CTA takes one window
// of NF = 2M real samples (M complex points, 128 kB of shared memory), runs an in-place DIF FFT
// (radix-2 stages fused into one radix-16 and three radix-8 passes; output bit-reversed), applies the real, even transfer function of the band in the
// bit-reversed domain, runs the inverse in-place DIT FFT (input bit-reversed, output natural) and
// writes the NF - 2(L-1) alias-free outputs.  No reordering pass, no global scratch.
//
// Real-input packing: z[n] = x[2n] + i x[2n+1] (the window as it lies in memory).  With
// E = FFT(even samples), O = FFT(odd samples), w = exp(-2 pi i/NF), H the (real, even) DFT of the
// circularly arranged band:  Hs = (H[k]+H[k+M])/2, Hd = (H[k]-H[k+M])/2,
//     W[k] = (Hs + i Hd w^-k) E[k] + (Hd w^k + i Hs) O[k]
// is the packed spectrum of the filtered window (derivation in DESIGN.md); C1 = Hs + i Hd w^-k and
// C2 = Hd w^k + i Hs are precomputed per noise block on the host, 1/M folded in.
//
// Bound: the L1/shared-memory data pipe (each fused pass moves 32 B per point, 4 passes per transform, the
// first and the last of the window fused with the global load / store), ~60x fewer flops than the direct
// form at L = 4096.
#include <cooperative_groups.h>

#include "cm2_common.cuh"

namespace cm2 {

constexpr int FFT_LOG2M = 13;
constexpr int FFT_M = 1 << FFT_LOG2M;   // complex points per window
constexpr int FFT_NF = 2 * FFT_M;       // real samples per window (16384)

__device__ __forceinline__ double2 cmul(double2 a, double2 b) {
    return make_double2(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}

// Twiddle tables: one compact table per pass so that consecutive butterflies read consecutive
// 16-byte entries (indexing one table tw[t] = exp(-2 pi i t / M) with the stride of the pass cost up
// to 32 L1 wavefronts per warp load and kept the LSU data pipe at 90 %; ncu, profiles/).  A radix-8
// pass with eighth-size q = 2^lq needs ONE entry per butterfly, w8 = exp(-2 pi i pos / (8 q)) for
// pos in [0, q), stored at tw[q + pos]; every other twiddle of the pass follows from it:
//   half-size 4q: w8 * exp(-2 pi i m/8), m = 0..3   half-size 2q: w8^2, -i w8^2   half-size q: w8^4
__global__ void k_fft_twiddles(double2 *__restrict__ tw) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;      // i = q + pos
    if (i >= 1 && i < FFT_M / 4) {
        const int lq = 31 - __clz(i);
        const int q = 1 << lq, pos = i - q;
        double sn, cs;
        sincospi(-2.0 * (double)pos / (double)(8 * q), &sn, &cs);
        tw[i] = make_double2(cs, sn);
    }
    if (i < FFT_M / 16) {     // radix-16 first / last pass: w16 = exp(-2 pi i pos / M) at tw[M/4 + pos]
        double sn, cs;
        sincospi(-2.0 * (double)i / (double)FFT_M, &sn, &cs);
        tw[FFT_M / 4 + i] = make_double2(cs, sn);
    }
}

// pair mode: W^n = exp(-2 pi i n / (2 M)), n < M -- the twiddles of the radix-2 stage that joins two CTAs
__global__ void k_fft_twiddles_pair(double2 *__restrict__ tw2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < FFT_M) {
        double sn, cs;
        sincospi(-(double)i / (double)FFT_M, &sn, &cs);
        tw2[i] = make_double2(cs, sn);
    }
}

// x * (1 - i)/sqrt2, x * (-i), x * (-1 - i)/sqrt2 and their conjugate counterparts
__device__ __forceinline__ double2 rot1(double2 x) { return make_double2(0.70710678118654752440 * (x.x + x.y), 0.70710678118654752440 * (x.y - x.x)); }
__device__ __forceinline__ double2 rot2(double2 x) { return make_double2(x.y, -x.x); }
__device__ __forceinline__ double2 rot3(double2 x) { return make_double2(0.70710678118654752440 * (x.y - x.x), -0.70710678118654752440 * (x.x + x.y)); }
__device__ __forceinline__ double2 rot1c(double2 x) { return make_double2(0.70710678118654752440 * (x.x - x.y), 0.70710678118654752440 * (x.x + x.y)); }
__device__ __forceinline__ double2 rot2c(double2 x) { return make_double2(-x.y, x.x); }
__device__ __forceinline__ double2 rot3c(double2 x) { return make_double2(-0.70710678118654752440 * (x.x + x.y), 0.70710678118654752440 * (x.x - x.y)); }
// decimation-in-frequency butterfly: (a, b) -> (a + b, (a - b) w); decimation in time: (a, b) -> (a + b w, a - b w)
__device__ __forceinline__ void dif(double2 &a, double2 &b, double2 w) {
    const double2 t = make_double2(a.x - b.x, a.y - b.y);
    a = make_double2(a.x + b.x, a.y + b.y);
    b = cmul(t, w);
}
__device__ __forceinline__ void dit(double2 &a, double2 &b, double2 w) {
    const double2 t = cmul(b, w);
    b = make_double2(a.x - t.x, a.y - t.y);
    a = make_double2(a.x + t.x, a.y + t.y);
}

// x * (cr + i ci)
__device__ __forceinline__ double2 rotc(double2 x, double cr, double ci) {
    return make_double2(fma(x.x, cr, -x.y * ci), fma(x.x, ci, x.y * cr));
}
constexpr double C16 = 0.92387953251128675613, S16 = 0.38268343236508977173, R2H = 0.70710678118654752440;

// The 16-point butterfly of the first forward pass (decimation in frequency, half-sizes 8q .. q) and of
// the last inverse pass (decimation in time, q .. 8q; INV selects conjugate twiddles): one table entry
// w16 = exp(-+2 pi i pos / 16q), every other twiddle derived from it.
template <bool INV>
__device__ __forceinline__ void butterfly16(double2 (&v)[16], double2 w16) {
    constexpr double sg = INV ? 1.0 : -1.0;               // sign of the imaginary part of exp(-+ i ...)
    const double2 w8 = cmul(w16, w16), w4 = cmul(w8, w8), w2 = cmul(w4, w4);
    const double2 wa[8] = {w16, rotc(w16, C16, sg * S16), rotc(w16, R2H, sg * R2H), rotc(w16, S16, sg * C16),
                           rotc(w16, 0.0, sg), rotc(w16, -S16, sg * C16), rotc(w16, -R2H, sg * R2H),
                           rotc(w16, -C16, sg * S16)};
    const double2 wb[4] = {w8, rotc(w8, R2H, sg * R2H), rotc(w8, 0.0, sg), rotc(w8, -R2H, sg * R2H)};
    const double2 wc[2] = {w4, rotc(w4, 0.0, sg)};
    if (!INV) {
#pragma unroll
        for (int m = 0; m < 8; ++m) dif(v[m], v[m + 8], wa[m]);
#pragma unroll
        for (int h = 0; h < 16; h += 8) {
#pragma unroll
            for (int m = 0; m < 4; ++m) dif(v[h + m], v[h + m + 4], wb[m]);
        }
#pragma unroll
        for (int h = 0; h < 16; h += 4) { dif(v[h], v[h + 2], wc[0]); dif(v[h + 1], v[h + 3], wc[1]); }
#pragma unroll
        for (int p = 0; p < 16; p += 2) dif(v[p], v[p + 1], w2);
    } else {
#pragma unroll
        for (int p = 0; p < 16; p += 2) dit(v[p], v[p + 1], w2);
#pragma unroll
        for (int h = 0; h < 16; h += 4) { dit(v[h], v[h + 2], wc[0]); dit(v[h + 1], v[h + 3], wc[1]); }
#pragma unroll
        for (int h = 0; h < 16; h += 8) {
#pragma unroll
            for (int m = 0; m < 4; ++m) dit(v[h + m], v[h + m + 4], wb[m]);
        }
#pragma unroll
        for (int m = 0; m < 8; ++m) dit(v[m], v[m + 8], wa[m]);
    }
}

// The 8-point butterfly of the forward radix-8 passes (decimation in frequency, half-sizes 4q, 2q, q) and of the
// inverse ones (decimation in time, q, 2q, 4q; INV: w8 is already conjugated and the rotations are the conjugate ones).
template <bool INV>
__device__ __forceinline__ void butterfly8(double2 (&v)[8], double2 w8) {
    const double2 w4 = cmul(w8, w8), w2 = cmul(w4, w4);
    if (!INV) {
        dif(v[0], v[4], w8);                       // half-size 4q
        dif(v[1], v[5], rot1(w8));
        dif(v[2], v[6], rot2(w8));
        dif(v[3], v[7], rot3(w8));
        const double2 w4r = rot2(w4);
        dif(v[0], v[2], w4);                       // half-size 2q
        dif(v[1], v[3], w4r);
        dif(v[4], v[6], w4);
        dif(v[5], v[7], w4r);
        dif(v[0], v[1], w2);                       // half-size q
        dif(v[2], v[3], w2);
        dif(v[4], v[5], w2);
        dif(v[6], v[7], w2);
    } else {
        dit(v[0], v[1], w2);                       // half-size q
        dit(v[2], v[3], w2);
        dit(v[4], v[5], w2);
        dit(v[6], v[7], w2);
        const double2 w4r = rot2c(w4);
        dit(v[0], v[2], w4);                       // half-size 2q
        dit(v[1], v[3], w4r);
        dit(v[4], v[6], w4);
        dit(v[5], v[7], w4r);
        dit(v[0], v[4], w8);                       // half-size 4q
        dit(v[1], v[5], rot1c(w8));
        dit(v[2], v[6], rot2c(w8));
        dit(v[3], v[7], rot3c(w8));
    }
}

// One radix-8 pass of eighth-size q = 2^lq through the transform in zs, in place, ending with a barrier: butterfly8<INV>
// with the pass's twiddle tw[q + pos] (conjugated for INV).  tid = threadIdx.x, read by the kernel (see fft_forward).
template <int FFT_THREADS, bool INV>
__device__ __forceinline__ void pass8(int tid, const double2 *__restrict__ tw, int lq) {
    extern __shared__ double2 zs[];
#define z(i) zs[(i) + ((i) >> 3)]
    const int q = 1 << lq;
    // NB butterflies per thread and loop trip, every input loaded before the first output is stored: the loads of the
    // second butterfly overlap the arithmetic of the first (the compiler cannot move them above the stores itself: same
    // shared-memory array)
    constexpr int NB = (FFT_M / 8) % (2 * FFT_THREADS) == 0 ? 2 : 1;
    for (int j = tid; j < FFT_M / 8; j += NB * FFT_THREADS) {
        double2 v[NB][8];
        int i0[NB];
        double2 w8[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            const int jb = j + b * FFT_THREADS;
            const int pos = jb & (q - 1);
            i0[b] = ((jb >> lq) << (lq + 3)) + pos;
#pragma unroll
            for (int m = 0; m < 8; ++m) v[b][m] = z(i0[b] + m * q);
            w8[b] = __ldg(tw + q + pos);
            if (INV) w8[b].y = -w8[b].y;
        }
#pragma unroll
        for (int b = 0; b < NB; ++b) {
            butterfly8<INV>(v[b], w8[b]);
#pragma unroll
            for (int m = 0; m < 8; ++m) z(i0[b] + m * q) = v[b][m];
        }
    }
    __syncthreads();
#undef z
}

// The even- and odd-sample spectra of the packed real transform at frequency k from Z_k and Z_{M-k}:
// E_k = (Z_k + conj Z_{M-k}) / 2,  O_k = (Z_k - conj Z_{M-k}) / 2i
__device__ __forceinline__ void split_packed(double2 zk, double2 zm, double2 &Ek, double2 &Ok) {
    Ek = make_double2(0.5 * (zk.x + zm.x), 0.5 * (zk.y - zm.y));
    Ok = make_double2(0.5 * (zk.y + zm.y), -0.5 * (zk.x - zm.x));
}

// The forward FFT of one window, decimation in frequency, natural in -> bit-reversed out, in place in zs (one pad
// element per 8 points).  Radix-2 stages are fused into passes whose points stay in registers: one radix-16 pass
// (4 stages) + radix-8 passes (3 stages each), so a transform makes 4 passes through shared memory instead of 13.
// The FIRST pass takes its inputs from the window loader, load16(i0, q, v) fills v[m] = point i0 + m q of the window
// (from global memory: the window never makes a separate trip through shared memory); before_store() runs between
// that pass's butterflies and its shared-memory stores.  Ends with a barrier: the spectrum is complete in zs.
// tid = threadIdx.x, read by the kernel: a read in here carries no __launch_bounds__ range, and once merged with the
// kernel's own read it widens that range and changes the kernel's code.
template <int FFT_THREADS, class Load16, class BeforeStore>
__device__ __forceinline__ void fft_forward(int tid, const double2 *__restrict__ tw, Load16 &&load16,
                                            BeforeStore &&before_store) {
    extern __shared__ double2 zs[];
#define z(i) zs[(i) + ((i) >> 3)]
    static_assert(FFT_LOG2M % 3 == 1 && FFT_LOG2M >= 4, "one radix-16 pass + radix-8 passes");
    {   // first pass: radix-16 (half-sizes M/2 .. M/16)
        constexpr int lq = FFT_LOG2M - 4, q = 1 << lq;
        for (int j = tid; j < FFT_M / 16; j += FFT_THREADS) {
            const int pos = j & (q - 1);
            const int i0 = ((j >> lq) << (lq + 4)) + pos;
            double2 v[16];
            load16(i0, q, v);
            butterfly16<false>(v, __ldg(tw + FFT_M / 4 + pos));
            before_store();
#pragma unroll
            for (int m = 0; m < 16; ++m) z(i0 + m * q) = v[m];
        }
        __syncthreads();
    }
    for (int lq = FFT_LOG2M - 7; lq >= 0; lq -= 3) pass8<FFT_THREADS, false>(tid, tw, lq);
#undef z
}

// ---- window sources of k_toeplitz_fft ---------------------------------------------------------------------------
// Without a generator the window is read from d, zero outside the noise block (the apply's non-circulant boundary).
// NoiseWindow: the window is generated, w_b(r) for the offsets r from the block start, for every integer r (no
// boundary): one Philox4x32-10 call per pair p = r / 2 (counter (lo p, hi p, id_b, realization), key (lo seed,
// hi seed)) and Box-Muller, w(2p) = rho cospi(2 u2), w(2p+1) = rho sinpi(2 u2), rho = sqrt(-2 ln u1),
// u1 = (a + 1) 2^-53 from x0:x1, u2 = c 2^-53 from x2:x3 (DESIGN.md section 4d).  Overlapping windows regenerate
// the same samples, so the result depends on (seed, realization, id_b, offset) only.
// ADD_: out += n instead of out = n.
template <bool ADD_>
struct NoiseWindow {
    static constexpr bool ADD = ADD_;
    uint64_t seed;
    const int64_t *ids;      // id_b = (uint32) ids[b]; nullptr: b
    uint32_t realization;
};

__device__ __forceinline__ double2 philox_normal_pair(uint64_t seed, uint32_t id, uint32_t realization, int64_t p) {
    uint32_t c0 = (uint32_t)p, c1 = (uint32_t)((uint64_t)p >> 32), c2 = id, c3 = realization;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
    }
    const uint64_t a = ((((uint64_t)c0) << 32) | c1) >> 11, c = ((((uint64_t)c2) << 32) | c3) >> 11;
    const double u1 = __ull2double_rn(a + 1) * 0x1p-53, u2 = __ull2double_rn(c) * 0x1p-53;     // both exact
    const double rho = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    return make_double2(rho * cs, rho * sn);
}

// one CTA per window.  win_first[b] = first window index of noise block b (prefix, nblocks+1).
// PAIR: a window of 2 NF = 32768 samples on a CLUSTER of two CTAs (one 16384-point complex transform split by one
// radix-2 stage).  With z the packed window, W = exp(-2 pi i / 2M): CTA 0 transforms u[n] = z[n] + z[n+M] (the even
// frequencies), CTA 1 v[n] = (z[n] - z[n+M]) W^n (the odd ones) -- both read both halves of the window from global
// memory / L2, so the forward stage needs no exchange.  The packed-real partner of frequency k is 2M - k, which has
// the parity of k: the transfer step stays inside a CTA (partner position M - k' for the even half, M - 1 - k', i.e.
// the complemented physical position, for the odd half).  The inverse transforms give U (CTA 0) and V (CTA 1);
// the window is U[n] + conj(W^n) V[n] (first half, written by CTA 0) and U[n] - conj(W^n) V[n] (second half,
// CTA 1): each CTA reads the other's result over distributed shared memory.  At 4096 coefficients 75 % of a window
// is alias-free instead of 50 %.
// Gen: empty (the apply: the window is read from d) or one NoiseWindow<ADD> (the simulation: the window is generated,
// d is unused; ADD: out += result).  An empty pack keeps the apply's instantiations, names and parameters as they were.
template <int FFT_THREADS, bool PAIR = false, class... Gen>
__global__ void __launch_bounds__(FFT_THREADS, 1)
    k_toeplitz_fft(const double2 *__restrict__ coef,   // [nblocks][2][M]: C1 then C2, indexed by PHYSICAL (bit-reversed) position
                   const double2 *__restrict__ tw, int L, int64_t nblocks, int64_t blocksize,
                   const int64_t *__restrict__ start, const int64_t *__restrict__ win_first,
                   const double *__restrict__ d, double *__restrict__ out, int64_t nt,
                   const double2 *__restrict__ tw2, Gen... gen) {
    static_assert(sizeof...(Gen) <= 1, "at most one window generator");
    constexpr bool GEN = sizeof...(Gen) == 1;
    constexpr bool ADD = GEN && (Gen::ADD && ...);
    uint64_t seed = 0;
    const int64_t *ids = nullptr;
    uint32_t realization = 0;
    ((seed = gen.seed, ids = gen.ids, realization = gen.realization), ...);
    extern __shared__ double2 zs[];   // M complex points, one pad element per 8 (bank-conflict relief)
#define z(i) zs[(i) + ((i) >> 3)]
    // the stores of the alias-free outputs: plain writes, or out += result (ADD)
    auto put2 = [&](int64_t t, double2 r) {
        double2 *o = reinterpret_cast<double2 *>(out + t);
        if constexpr (ADD) {
            const double2 x = *o;
            r = make_double2(x.x + r.x, x.y + r.y);
        }
        *o = r;
    };
    auto put1 = [&](int64_t t, double r) {
        if constexpr (ADD) out[t] += r;
        else out[t] = r;
    };
    // window positions [HD, HD + S) are alias-free; HD = L - 1 rounded up to even and S even, so that a window
    // starts on an even sample whenever its noise block does and the window moves as 16-byte pairs
    const int HD = (L - 1) + ((L - 1) & 1);
    const int S = ((PAIR ? 2 * FFT_NF : FFT_NF) - HD - (L - 1)) & ~1;
    const int64_t nwin = win_first[nblocks];
    unsigned crank = 0;
    if constexpr (PAIR) asm("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
    const int64_t win0 = PAIR ? (blockIdx.x >> 1) : blockIdx.x, winstep = PAIR ? (gridDim.x >> 1) : gridDim.x;
    bool join_pending = false;      // PAIR: arrived at the barrier that ends a window's join, not yet waited for
    for (int64_t win = win0; win < nwin; win += winstep) {
        // last_le(win_first, nblocks, win), written out: the shared helper (or lo declared first) swaps the operands of
        // one subtraction in this kernel's SASS
        int64_t hi = nblocks, lo = 0;
        while (hi - lo > 1) {
            int64_t mid = (lo + hi) >> 1;
            if (win_first[mid] <= win) lo = mid; else hi = mid;
        }
        const int64_t b = lo;
        const int64_t bs = start ? start[b] : b * blocksize;
        const int64_t be = start ? start[b + 1] : (b + 1 == nblocks ? nt : (b + 1) * blocksize);
        const int64_t j0 = bs + (win - win_first[b]) * S;     // first output of this window
        const int64_t w0 = j0 - HD;                           // first input sample of the window
        const bool al = ((w0 & 1) == 0) && (((uintptr_t)d | (uintptr_t)out) & 15) == 0;
        __syncthreads();
        // ---- forward FFT (fft_forward): the window's inputs straight from global memory, zero outside the noise
        // block (the non-circulant boundary)
        uint32_t idb = 0;
        if constexpr (GEN) idb = ids ? (uint32_t)ids[b] : (uint32_t)b;
        auto winload1 = [&](int i) {
            const int64_t t = w0 + 2 * (int64_t)i;
            if constexpr (GEN) return philox_normal_pair(seed, idb, realization, (t - bs) >> 1);   // t - bs even
            double2 v;
            if (al && t >= bs && t + 1 < be) return *reinterpret_cast<const double2 *>(d + t);
            v.x = (t >= bs && t < be) ? d[t] : 0.0;
            v.y = (t + 1 >= bs && t + 1 < be) ? d[t + 1] : 0.0;
            return v;
        };
        auto load16 = [&](int i0, int q, double2 (&v)[16]) {
            if constexpr (!PAIR) {
#pragma unroll
                for (int m = 0; m < 16; ++m) v[m] = winload1(i0 + m * q);
            } else {
                // both halves of the 2M-point window: explicit groups of 4 points with every load of a group
                // issued before its first use (a, b and the joining twiddle: 12 loads in flight per thread)
#pragma unroll
                for (int g = 0; g < 16; g += 4) {
                    double2 a[4], b[4], w[4];
#pragma unroll
                    for (int m = 0; m < 4; ++m) {
                        a[m] = winload1(i0 + (g + m) * q);
                        b[m] = winload1(i0 + (g + m) * q + FFT_M);
                        w[m] = __ldg(tw2 + i0 + (g + m) * q);
                    }
#pragma unroll
                    for (int m = 0; m < 4; ++m) {
                        if (crank == 0) v[g + m] = make_double2(a[m].x + b[m].x, a[m].y + b[m].y);
                        else v[g + m] = cmul(make_double2(a[m].x - b[m].x, a[m].y - b[m].y), w[m]);
                    }
                }
            }
        };
        auto before_store = [&] {
            if constexpr (PAIR) {
                // split-phase cluster barrier: the partner may still be reading this CTA's half of the PREVIOUS
                // window; it had this window's loads and 16-point butterflies to finish doing so
                if (join_pending) {
                    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
                    join_pending = false;
                }
            }
        };
        fft_forward<FFT_THREADS>(threadIdx.x, tw, load16, before_store);
        // ---- transfer function on the packed spectrum, in bit-reversed storage.  Every thread walks
        // PHYSICAL positions pk (consecutive lanes -> consecutive elements and coefficients: the
        // coefficient tables are stored by physical position) and computes W[k] alone, reading its
        // partner Z[M-k] but not the partner's coefficients (the first version handled the pair
        // (k, M-k) in one thread and paid two scattered 16-byte global loads per pair for them).
        // All reads, a barrier, then all writes: the update is in place.
        const double2 *c1 = coef + (PAIR ? (int64_t)(2 * b + crank) : (int64_t)b) * 2 * FFT_M;
        const double2 *c2 = c1 + FFT_M;
        constexpr int NPOS = FFT_M / FFT_THREADS;
        double2 res[NPOS];
#pragma unroll
        for (int i = 0; i < NPOS; ++i) {
            const int pk = threadIdx.x + i * FFT_THREADS;
            const int k = __brev((unsigned)pk) >> (32 - FFT_LOG2M);
            const int km = (FFT_M - k) & (FFT_M - 1);
            const int pm = (PAIR && crank == 1) ? (FFT_M - 1 - pk) : (int)(__brev((unsigned)km) >> (32 - FFT_LOG2M));
            double2 Ek, Ok;
            split_packed(z(pk), z(pm), Ek, Ok);
            const double2 a1 = cmul(__ldg(c1 + pk), Ek), a2 = cmul(__ldg(c2 + pk), Ok);
            res[i] = make_double2(a1.x + a2.x, a1.y + a2.y);
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < NPOS; ++i) z(threadIdx.x + i * FFT_THREADS) = res[i];
        __syncthreads();
        // ---- inverse FFT, decimation in time, bit-reversed in -> natural out (conjugate twiddles):
        // radix-8 passes (half-sizes q, 2q, 4q), then the radix-16 pass whose outputs -- the window in
        // natural order -- go straight to global memory
        for (int lq = 0; lq + 4 < FFT_LOG2M; lq += 3) pass8<FFT_THREADS, true>(threadIdx.x, tw, lq);
        {
            constexpr int lq = FFT_LOG2M - 4, q = 1 << lq;
            for (int j = threadIdx.x; j < FFT_M / 16; j += FFT_THREADS) {
                const int pos = j & (q - 1);
                const int i0 = ((j >> lq) << (lq + 4)) + pos;
                double2 v[16];
#pragma unroll
                for (int m = 0; m < 16; ++m) v[m] = z(i0 + m * q);
                double2 w16 = __ldg(tw + FFT_M / 4 + pos);
                w16.y = -w16.y;
                butterfly16<true>(v, w16);
                if constexpr (PAIR) {
#pragma unroll
                    for (int m = 0; m < 16; ++m) z(i0 + m * q) = v[m];      // U (CTA 0) / V (CTA 1), natural order
                } else {
                    // the alias-free samples, window positions [L-1, L-1+S)
#pragma unroll
                    for (int m = 0; m < 16; ++m) {
                        const int r0 = 2 * (i0 + m * q) - HD;             // output index of v.x within the window's S outputs (even)
                        if (r0 < 0 || r0 >= S) continue;
                        if (al && j0 + r0 + 1 < be) { put2(j0 + r0, v[m]); continue; }
                        if (j0 + r0 < be) put1(j0 + r0, v[m].x);
                        if (j0 + r0 + 1 < be) put1(j0 + r0 + 1, v[m].y);
                    }
                }
            }
        }
        if constexpr (PAIR) {
            // the radix-2 stage that joins the two CTAs: this CTA's half of the window from U and V
            namespace cg = cooperative_groups;
            cg::cluster_group cl = cg::this_cluster();
            cl.sync();                                                  // both inverse transforms are complete
            const double2 *rz = cl.map_shared_rank(zs, crank ^ 1u);
            constexpr int NU = 8;                                        // points per thread and trip, loads first
            for (int n0 = threadIdx.x; n0 < FFT_M; n0 += NU * FFT_THREADS) {
                double2 own[NU], oth[NU], w[NU];
#pragma unroll
                for (int u = 0; u < NU; ++u) {
                    const int n = n0 + u * FFT_THREADS;
                    own[u] = z(n);
                    oth[u] = rz[n + (n >> 3)];
                    w[u] = __ldg(tw2 + n);
                }
#pragma unroll
                for (int u = 0; u < NU; ++u) {
                    const int n = n0 + u * FFT_THREADS;
                    const int r0 = 2 * (n + (crank ? FFT_M : 0)) - HD;   // even
                    if (r0 < 0 || r0 >= S) continue;                    // aliased head / tail of the window
                    w[u].y = -w[u].y;
                    const double2 U = crank ? oth[u] : own[u], V = crank ? own[u] : oth[u];
                    const double2 t = cmul(w[u], V);
                    const double2 r = crank ? make_double2(U.x - t.x, U.y - t.y) : make_double2(U.x + t.x, U.y + t.y);
                    if (al && j0 + r0 + 1 < be) { put2(j0 + r0, r); continue; }
                    if (j0 + r0 < be) put1(j0 + r0, r.x);
                    if (j0 + r0 + 1 < be) put1(j0 + r0 + 1, r.y);
                }
            }
            // the partner has read my half once it, too, arrives here; waited for before the next window's first
            // shared-memory store (or before the CTA exits)
            asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
            join_pending = true;
        }
    }
    if constexpr (PAIR) {
        if (join_pending) asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    }
}

#undef z

// win_first[b] = first window index of noise block b (prefix, nblocks+1), a block of n samples holding
// n >= span ? (n - span) / hop + 1 : 0 windows (overlap-save apply: span 1, hop S, i.e. ceil(n / S); Welch: span NF, hop M)
__global__ void k_win_first(int64_t nblocks, int64_t blocksize, const int64_t *__restrict__ start, int64_t nt, int span,
                            int hop, int64_t *__restrict__ win_first) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int64_t acc = 0;
        for (int64_t b = 0; b < nblocks; ++b) {
            win_first[b] = acc;
            const int64_t bs = start ? start[b] : b * blocksize;
            const int64_t be = start ? start[b + 1] : (b + 1 == nblocks ? nt : (b + 1) * blocksize);
            acc += be - bs >= span ? (be - bs - span) / hop + 1 : 0;
        }
        win_first[nblocks] = acc;
    }
}

// ---- Welch periodogram sums per noise block (cm2_noise_psd) ------------------------------------------------------
// Windows of NF samples at hop M from each block's first sample; x_t = h_t m_t d_t with the periodic Hann window
// h_t = sin^2(pi t / NF) (hann[t], built once) and m_t = 0 where pix < 0 (a select: flagged d never enters).  The
// forward transform is fft_forward's; the packed spectrum Z gives E_k = (Z_k + conj Z_{M-k}) / 2,
// O_k = (Z_k - conj Z_{M-k}) / 2i and X_k = E_k + w^k O_k (w = exp(-2 pi i / NF), tw2[k]), X_M = E_0 - O_0.
//
// Deterministic: CTA c takes the contiguous windows [c per, (c+1) per), per = ceil(nwin / grid).  Thread t owns the
// physical positions t + i FFT_THREADS (and thread 0 also bin M) and adds |X_k|^2 into acc[] in shared memory, in
// window order; at the end of each run of windows of one block the CTA writes acc (natural frequency order) and its
// sum of (h m)^2 to slot c + b of the scratch.  Slot ids are distinct (the block of CTA c+1's first window is >= that of
// CTA c's last one), at most grid + nblocks - 1 of them.  k_psd_sum then adds each block's slots in CTA (= window) order.
constexpr int PSD_THREADS = 256;    // 128 registers per thread (512 threads) spill in the radix-16 pass
constexpr int PSD_SLOT = FFT_M + 2;    // S(0..M), W

// ---- sample sources of k_noise_psd ------------------------------------------------------------------------------
// Without a source the samples are d_t.  Residual<POL>: the samples are the map residual r_t = d_t - (P x)_t, with
// (P x)_t = project<POL> of x[POL pix_t ..] and cos / sin 2 phi_t (not read for POL = 1): the expression of
// k_pointing_apply, so r_t is bit for bit d_t - P.mult(x)_t.  Where pix_t < 0 nothing is gathered and the existing
// select masks the sample (DESIGN.md section 4e).  pix is required with a Residual.
template <int POL_>
struct Residual {
    static constexpr int POL = POL_;
    const double *cs, *sn;      // cos 2 phi, sin 2 phi: nt values each (POL > 1)
    const double *x;            // the map: POL values per pixel, every pixel id < its pixel count
};

__global__ void k_hann(double *__restrict__ hann) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < FFT_NF) {
        const double s = sinpi((double)t / (double)FFT_NF);
        hann[t] = s * s;
    }
}

// Src: empty (the samples are d) or one Residual<POL> (the samples are d - P x).  An empty pack keeps the kernel's
// parameters and code as they were.
template <class... Src>
__global__ void __launch_bounds__(PSD_THREADS, 1)
    k_noise_psd(const double2 *__restrict__ tw, const double2 *__restrict__ tw2, const double *__restrict__ hann,
                int64_t nblocks, int64_t blocksize, const int64_t *__restrict__ start,
                const int64_t *__restrict__ win_first, const double *__restrict__ d, const int32_t *__restrict__ pix,
                int64_t nt, double *__restrict__ slots, Src... src) {
    static_assert(sizeof...(Src) <= 1, "at most one sample source");
    constexpr bool RES = sizeof...(Src) == 1;
    constexpr int POL = (Src::POL * ... * 1);
    const double *cs = nullptr, *sn = nullptr, *xmap = nullptr;
    ((cs = src.cs, sn = src.sn, xmap = src.x), ...);
    extern __shared__ double2 zs[];
#define z(i) zs[(i) + ((i) >> 3)]
    double *acc = reinterpret_cast<double *>(zs + FFT_M + FFT_M / 8);     // [M + 1], by physical position; M last
    double *wrun = acc + FFT_M + 1;         // [2][PSD_THREADS]: each thread's sum of (h m)^2 over the run, compensated
    __shared__ double red[32];
    constexpr int NPOS = FFT_M / PSD_THREADS;
    const int tid = threadIdx.x;
    const int64_t nwin = win_first[nblocks];
    const int64_t per = (nwin + gridDim.x - 1) / gridDim.x;
    const int64_t wlo = (int64_t)blockIdx.x * per;
    const int64_t whi = wlo + per < nwin ? wlo + per : nwin;
    if (wlo >= whi) return;
#pragma unroll
    for (int i = 0; i < NPOS; ++i) acc[tid + i * PSD_THREADS] = 0.0;
    if (tid == 0) acc[FFT_M] = 0.0;
    wrun[tid] = wrun[PSD_THREADS + tid] = 0.0;
    int64_t b = last_le(win_first, nblocks, wlo);
    for (int64_t win = wlo; win < whi; ++win) {
        const int64_t bs = start ? start[b] : b * blocksize;
        const int64_t t0 = bs + (win - win_first[b]) * FFT_M;      // the window lies inside the block
        const double *dw = d + t0;
        const int32_t *pw = pix ? pix + t0 : nullptr;
        const bool ald = ((uintptr_t)dw & 15) == 0, alp = ((uintptr_t)pw & 7) == 0;
        const double *cw = POL > 1 ? cs + t0 : nullptr, *sw = POL > 1 ? sn + t0 : nullptr;
        const bool alc = ((((uintptr_t)cw) | (uintptr_t)sw) & 15) == 0;
        __syncthreads();                    // the previous window's power step has read zs
        // this thread's sum of (h m)^2 over the run, compensated (Neumaier), in shared memory: as registers across the
        // transform it spills
        auto wadd = [&](double a) {
            const double ws = wrun[tid], s = ws + a;
            wrun[PSD_THREADS + tid] += fabs(ws) >= fabs(a) ? (ws - s) + a : (a - s) + ws;
            wrun[tid] = s;
        };
        // r_t = d_t - (P x)_t for an unflagged sample (Residual); a flagged one is returned as is and selected away
        auto resid = [&](double dv, int p, double c, double s) {
            if (p < 0) return dv;
            double xv[POL];
#pragma unroll
            for (int k = 0; k < POL; ++k) xv[k] = __ldg(xmap + (int64_t)POL * p + k);
            return dv - project<POL>(xv, c, s);
        };
        auto load16 = [&](int i0, int q, double2 (&v)[16]) {
            // groups of 4 points, every load of a group issued before its first use (48 loads in flight spill; the
            // residual's cos / sin and x gathers fit: 217 / 240 / 250 registers at POL 1 / 2 / 3, no spill)
#pragma unroll
            for (int g = 0; g < 16; g += 4) {
                double2 x[4], h[4], c[4], s[4];
                int2 p[4];
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    const int i = i0 + (g + m) * q;
                    x[m] = ald ? __ldcs(reinterpret_cast<const double2 *>(dw) + i) : make_double2(__ldcs(dw + 2 * i), __ldcs(dw + 2 * i + 1));
                    h[m] = __ldg(reinterpret_cast<const double2 *>(hann) + i);
                    p[m] = !pw ? make_int2(0, 0)
                               : alp ? __ldcs(reinterpret_cast<const int2 *>(pw) + i) : make_int2(__ldcs(pw + 2 * i), __ldcs(pw + 2 * i + 1));
                    if constexpr (RES && POL > 1) {
                        c[m] = alc ? __ldcs(reinterpret_cast<const double2 *>(cw) + i) : make_double2(__ldcs(cw + 2 * i), __ldcs(cw + 2 * i + 1));
                        s[m] = alc ? __ldcs(reinterpret_cast<const double2 *>(sw) + i) : make_double2(__ldcs(sw + 2 * i), __ldcs(sw + 2 * i + 1));
                    } else {
                        c[m] = s[m] = make_double2(0.0, 0.0);
                    }
                }
                if constexpr (RES) {
#pragma unroll
                    for (int m = 0; m < 4; ++m)
                        x[m] = make_double2(resid(x[m].x, p[m].x, c[m].x, s[m].x), resid(x[m].y, p[m].y, c[m].y, s[m].y));
                }
                double a[4];
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    const bool g0 = p[m].x >= 0, g1 = p[m].y >= 0;
                    v[g + m] = make_double2(g0 ? h[m].x * x[m].x : 0.0, g1 ? h[m].y * x[m].y : 0.0);
                    a[m] = (g0 ? h[m].x * h[m].x : 0.0) + (g1 ? h[m].y * h[m].y : 0.0);
                }
                wadd((a[0] + a[1]) + (a[2] + a[3]));      // the group's 8 terms pairwise: 3 roundings deep
            }
        };
        fft_forward<PSD_THREADS>(tid, tw, load16, [] {});
        // ---- power step: |X_k|^2 for this thread's positions
#pragma unroll
        for (int i = 0; i < NPOS; ++i) {
            const int pk = tid + i * PSD_THREADS;
            const int k = __brev((unsigned)pk) >> (32 - FFT_LOG2M);
            const int pm = __brev((unsigned)((FFT_M - k) & (FFT_M - 1))) >> (32 - FFT_LOG2M);
            double2 Ek, Ok;
            split_packed(z(pk), z(pm), Ek, Ok);
            const double2 wO = cmul(__ldg(tw2 + k), Ok);
            const double2 X = make_double2(Ek.x + wO.x, Ek.y + wO.y);
            acc[pk] += fma(X.x, X.x, X.y * X.y);
            if (pk == 0) {
                const double xm = Ek.x - Ok.x;                     // E_0, O_0 are real
                acc[FFT_M] += xm * xm;
            }
        }
        if (win + 1 == whi || win + 1 == win_first[b + 1]) {
            // end of this CTA's run in block b: slot blockIdx.x + b
            double *slot = slots + ((int64_t)blockIdx.x + b) * PSD_SLOT;
#pragma unroll
            for (int i = 0; i < NPOS; ++i) {
                const int pk = tid + i * PSD_THREADS;
                slot[__brev((unsigned)pk) >> (32 - FFT_LOG2M)] = acc[pk];
                acc[pk] = 0.0;
            }
            if (tid == 0) {
                slot[FFT_M] = acc[FFT_M];
                acc[FFT_M] = 0.0;
            }
            const double wt = block_sum(wrun[tid] + wrun[PSD_THREADS + tid], red);
            if (tid == 0) slot[FFT_M + 1] = wt;
            wrun[tid] = wrun[PSD_THREADS + tid] = 0.0;
            while (b + 1 < nblocks && win + 1 >= win_first[b + 1]) ++b;
        }
    }
#undef z
}

// psd[b][k] = sum over the CTAs c that hold windows of block b (ascending) of slot (c + b), k = 0..M; wsum[b] likewise
// from entry M + 1.  A block without windows gets zeros.
__global__ void k_psd_sum(const int64_t *__restrict__ win_first, int64_t nblocks, int psd_grid,
                          const double *__restrict__ slots, double *__restrict__ psd, double *__restrict__ wsum) {
    const int64_t nwin = win_first[nblocks];
    const int64_t per = (nwin + psd_grid - 1) / psd_grid;      // as in k_noise_psd
    const int64_t n = nblocks * PSD_SLOT;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = e / PSD_SLOT;
        const int k = (int)(e - b * PSD_SLOT);
        const int64_t w0 = win_first[b], w1 = win_first[b + 1];
        double s = 0.0;
        if (w1 > w0) {
            for (int64_t c = w0 / per; c <= (w1 - 1) / per; ++c) s += slots[(c + b) * PSD_SLOT + k];
        }
        if (k <= FFT_M) psd[b * (FFT_M + 1) + k] = s;
        else wsum[b] = s;
    }
}

}  // namespace cm2

using namespace cm2;

// The scratch of both launchers begins with the twiddle tables: tw (M entries, the radix-16 and radix-8 passes), then
// tw2 (M entries, W^n = exp(-2 pi i n / 2M)).  Each launcher's own tables follow from byte TWIDDLE_BYTES.
constexpr int64_t TWIDDLE_BYTES = 2 * (int64_t)FFT_M * (int64_t)sizeof(double2);
constexpr size_t FFT_SMEM = sizeof(double2) * (FFT_M + FFT_M / 8);      // zs: M points, one pad element per 8

extern "C" int cm2_toeplitz_fft_points(void) { return FFT_M; }

// scratch: the twiddles, then win_first (nblocks + 1)
extern "C" int64_t cm2_toeplitz_fft_scratch_bytes(int64_t nblocks) {
    return TWIDDLE_BYTES + (nblocks + 1) * (int64_t)sizeof(int64_t) + 64;
}

// The block partition, checked first by both launchers
static int check_partition(int64_t nblocks, int64_t blocksize, const int64_t *blk_start, int64_t nt) {
    CM2_REQUIRE(nt >= 0 && nblocks > 0, "bad sizes");
    CM2_REQUIRE(blk_start != nullptr || blocksize > 0, "blocksize must be > 0");
    CM2_REQUIRE(blk_start != nullptr || nblocks - 1 <= nt / blocksize, "equal blocks past nt: (nblocks-1)*blocksize > nt");
    return CM2_OK;
}

// The set-up of both launchers after their argument checks: the twiddle tables at the head of scratch (built when
// init != 0) and the window plan win_first for windows of `span` samples at `hop`
static int plan_windows(void *scratch, int init, int64_t nblocks, int64_t blocksize, const int64_t *blk_start,
                        int64_t nt, int span, int hop, int64_t *win_first, cudaStream_t st) {
    double2 *tw = static_cast<double2 *>(scratch);
    if (init) {
        k_fft_twiddles<<<(FFT_M / 4 + 255) / 256, 256, 0, st>>>(tw);
        k_fft_twiddles_pair<<<(FFT_M + 255) / 256, 256, 0, st>>>(tw + FFT_M);
        CM2_LAUNCHED();
    }
    k_win_first<<<1, 1, 0, st>>>(nblocks, blocksize, blk_start, nt, span, hop, win_first);
    CM2_LAUNCHED();
    return CM2_OK;
}

// one launch of an overlap-save kernel: persistent CTAs (grid), or 2-CTA clusters (PAIR, grid = 2 x clusters)
template <bool PAIR, class... Params, class... Args>
static int fft_run(void (*kern)(Params...), int threads, int grid, size_t smem, cudaStream_t st, Args... args) {
    CM2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if constexpr (!PAIR) {
        kern<<<grid, threads, smem, st>>>(args...);
        CM2_LAUNCHED();
        return CM2_OK;
    }
    // one window per 2-CTA cluster (distributed shared memory for the joining stage)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CM2_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
    count_launch();
    return CM2_OK;
}

// 512 threads per CTA, one CTA per SM: the 16-point butterflies of the first / last pass need the 128 registers per
// thread that 512 threads leave.  The simulation runs at 512 threads too (at 256 it spills nothing but takes 1.15-1.5x
// as long, DESIGN.md section 4d).
template <bool PAIR, class... Gen>
static int fft_kernel(int grid, cudaStream_t st, const double2 *cf, const double2 *tw, int nband, int64_t nblocks,
                      int64_t blocksize, const int64_t *blk_start, const int64_t *win_first, const double *d,
                      double *out, int64_t nt, const double2 *tw2, Gen... gen) {
    return fft_run<PAIR>(k_toeplitz_fft<512, PAIR, Gen...>, 512, grid, FFT_SMEM, st, cf, tw, nband, nblocks, blocksize,
                         blk_start, win_first, d, out, nt, tw2, gen...);
}

// The overlap-save launcher of the apply (no generator, d the input) and of the noise simulation (one NoiseWindow,
// d = nullptr): argument checks, window plan and grid in one place.
template <class... Gen>
static int fft_launch(const double *coef, int nband, int64_t nblocks, int64_t blocksize, const int64_t *blk_start,
                      const double *d, double *out, int64_t nt, void *scratch, int init, int pair, cudaStream_t st,
                      Gen... gen) {
    if (int rc = check_partition(nblocks, blocksize, blk_start, nt)) return rc;
    CM2_REQUIRE(nband >= 1, "nband must be >= 1");
    CM2_REQUIRE(pair == 0 || pair == 1, "pair must be 0 or 1");
    CM2_REQUIRE(2 * (nband - 1) < (pair ? FFT_NF : FFT_NF / 2), "band too wide for the overlap-save window (4096 coefficients; 8192 in pair mode)");
    CM2_REQUIRE(scratch != nullptr && aligned(scratch, 16) && aligned(coef, 16), "scratch/coef must be 16-byte aligned");
    constexpr bool GEN = sizeof...(Gen) == 1;
    CM2_REQUIRE(GEN || d != out, "in-place Toeplitz apply is not supported");
    CM2_REQUIRE(!GEN || nt == 0 || out != nullptr, "out is required");
    if (nt == 0) return CM2_OK;
    const int HD = (nband - 1) + ((nband - 1) & 1);
    const int S = ((pair ? 2 * FFT_NF : FFT_NF) - HD - (nband - 1)) & ~1;       // as in the kernel
    int64_t *win_first = reinterpret_cast<int64_t *>(static_cast<char *>(scratch) + TWIDDLE_BYTES);
    if (int rc = plan_windows(scratch, init, nblocks, blocksize, blk_start, nt, 1, S, win_first, st)) return rc;
    const double2 *tw = static_cast<const double2 *>(scratch), *tw2 = tw + FFT_M;
    const double2 *cf = reinterpret_cast<const double2 *>(coef);
    const int64_t nwin_ub = nt / S + nblocks + 1;
    if (pair) {
        int64_t ncl = sm_count() / 2;
        if (nwin_ub < ncl) ncl = nwin_ub;
        return fft_kernel<true>((int)(2 * ncl), st, cf, tw, nband, nblocks, blocksize, blk_start, win_first, d, out, nt,
                                tw2, gen...);
    }
    return fft_kernel<false>(capped_grid(nwin_ub, 1), st, cf, tw, nband, nblocks, blocksize, blk_start, win_first, d,
                             out, nt, tw2, gen...);
}

// coef: device, [nblocks][2][M] complex (C1, C2 stored at the bit-reversed position of their frequency, 1/M folded in);
// pair = 1: 32768-sample windows on 2-CTA clusters, coef [nblocks][2 (CTA: even / odd frequencies)][2][M] of the
// 2M-point packed transform, entry p of CTA c = C[2 brev(p) + c], 1/(2M) folded in;
// scratch: cm2_toeplitz_fft_scratch_bytes(nblocks) bytes, `init` != 0 builds the twiddle tables in it
extern "C" int cm2_noise_toeplitz_fft_apply(const double *coef, int nband, int64_t nblocks, int64_t blocksize,
                                            const int64_t *blk_start, const double *d, double *out, int64_t nt,
                                            void *scratch, int init, int pair, cm2_stream_t stream) {
    return fft_launch(coef, nband, nblocks, blocksize, blk_start, d, out, nt, scratch, init, pair, as_stream(stream));
}

// n_t = sum_{|k|<L} h_b[|k|] w_b(t - k - s_b) per noise block, w_b the Philox / Box-Muller stream of NoiseWindow keyed on
// (seed, realization, block_ids[b] or b); out = n (add = 0) or out += n (add != 0).  coef, scratch, init, pair as
// for cm2_noise_toeplitz_fft_apply.
extern "C" int cm2_noise_simulate(const double *coef, int nband, int64_t nblocks, int64_t blocksize,
                                  const int64_t *blk_start, const int64_t *block_ids, uint64_t seed, uint32_t realization,
                                  double *out, int64_t nt, int add, void *scratch, int init, int pair,
                                  cm2_stream_t stream) {
    if (add)
        return fft_launch(coef, nband, nblocks, blocksize, blk_start, nullptr, out, nt, scratch, init, pair,
                          as_stream(stream), NoiseWindow<true>{seed, block_ids, realization});
    return fft_launch(coef, nband, nblocks, blocksize, blk_start, nullptr, out, nt, scratch, init, pair,
                      as_stream(stream), NoiseWindow<false>{seed, block_ids, realization});
}

// scratch: the twiddles, Hann window (NF doubles), win_first (nblocks + 1), one slot of M + 2 doubles per (CTA, block)
// run: at most (CTAs of the current device) + nblocks
extern "C" int64_t cm2_noise_psd_scratch_bytes(int64_t nblocks) {
    if (nblocks < 1) return 0;
    return TWIDDLE_BYTES + (int64_t)sizeof(double) * (FFT_NF + 2 * cdiv(nblocks + 1, 2) +
                                                      ((int64_t)sm_count() + nblocks) * PSD_SLOT);
}

// The Welch launcher of cm2_noise_psd (no source: the samples are d) and cm2_noise_psd_residual (one Residual<POL>):
// argument checks, tables, window plan, grid and the slot sums in one place.
template <class... Src>
static int psd_launch(const double *d, const int32_t *pix, int64_t nblocks, int64_t blocksize, const int64_t *blk_start,
                      int64_t nt, double *psd, double *wsum, void *scratch, int init, cudaStream_t st, Src... src) {
    if (int rc = check_partition(nblocks, blocksize, blk_start, nt)) return rc;
    CM2_REQUIRE(d != nullptr && psd != nullptr && wsum != nullptr, "d, psd and wsum are required");
    CM2_REQUIRE(scratch != nullptr && aligned(scratch, 16), "scratch (cm2_noise_psd_scratch_bytes) must be 16-byte aligned");
    // cm2_noise_psd writes zero sums for an empty TOD; the residual entry point writes nothing
    if (sizeof...(Src) == 1 && nt == 0) return CM2_OK;
    double *hann = reinterpret_cast<double *>(static_cast<char *>(scratch) + TWIDDLE_BYTES);
    int64_t *win_first = reinterpret_cast<int64_t *>(hann + FFT_NF);
    double *slots = reinterpret_cast<double *>(win_first) + 2 * cdiv(nblocks + 1, 2);
    if (int rc = plan_windows(scratch, init, nblocks, blocksize, blk_start, nt, FFT_NF, FFT_M, win_first, st)) return rc;
    if (init) {
        if (int rc = launch(k_hann, FFT_NF / 256, 256, 0, st, hann)) return rc;
    }
    const double2 *tw = static_cast<const double2 *>(scratch), *tw2 = tw + FFT_M;
    // one CTA per SM (the transform's shared memory), never more CTAs than windows could exist
    const size_t smem = FFT_SMEM + sizeof(double) * (FFT_M + 1 + 2 * PSD_THREADS);
    const int grid = capped_grid(nt / FFT_M + 1, 1);
    CM2_CUDA(cudaFuncSetAttribute(k_noise_psd<Src...>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (int rc = launch(k_noise_psd<Src...>, grid, PSD_THREADS, smem, st, tw, tw2, (const double *)hann, nblocks,
                        blocksize, blk_start, (const int64_t *)win_first, d, pix, nt, slots, src...))
        return rc;
    const int64_t n = nblocks * PSD_SLOT;
    return launch(k_psd_sum, capped_grid(cdiv(n, 256), 8), 256, 0, st, (const int64_t *)win_first, nblocks, grid,
                  (const double *)slots, psd, wsum);
}

extern "C" int cm2_noise_psd(const double *d, const int32_t *pix, int64_t nblocks, int64_t blocksize,
                             const int64_t *blk_start, int64_t nt, double *psd, double *wsum, void *scratch, int init,
                             cm2_stream_t stream) {
    return psd_launch(d, pix, nblocks, blocksize, blk_start, nt, psd, wsum, scratch, init, as_stream(stream));
}

// cm2_noise_psd of r = d - P x (Residual): pix is the pointing's own pixel table and masks as in cm2_noise_psd
extern "C" int cm2_noise_psd_residual(const double *d, const int32_t *pix, const double *cos2phi, const double *sin2phi,
                                      int pol, const double *x, int64_t nblocks, int64_t blocksize,
                                      const int64_t *blk_start, int64_t nt, double *psd, double *wsum, void *scratch,
                                      int init, cm2_stream_t stream) {
    CM2_REQUIRE(d != nullptr && pix != nullptr && x != nullptr, "d, pix and x are required");
    CM2_REQUIRE(pol >= 1 && pol <= 3, "pol must be 1, 2 or 3");
    CM2_REQUIRE(pol == 1 || (cos2phi != nullptr && sin2phi != nullptr), "cos2phi and sin2phi are required for pol > 1");
    return with_pol(pol, [&](auto P) {
        return psd_launch(d, pix, nblocks, blocksize, blk_start, nt, psd, wsum, scratch, init, as_stream(stream),
                          Residual<P>{cos2phi, sin2phi, x});
    });
}
