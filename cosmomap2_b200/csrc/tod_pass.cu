// cosmomap2_b200 -- time-domain passes over the TOD (sm_100a).
//
//   cm2_pointing_apply      d = P x            gather     (linearoperators.py:356-384,411-438,463-497)
//   cm2_pointing_apply_t    y = P^T d          scatter    (linearoperators.py:385-410,439-462,498-526)
//   cm2_amatvec_white       y = P^T diag(w) P x, fused, no TOD temporary
//   cm2_weights_moments     per-pixel moments of P^T diag(w) P (process_ces.py:480-542,125-189)
//   cm2_hits_i64            integer hit counts
//
// Data layout in HBM: pix int32[nt], cos2phi fp64[nt], sin2phi fp64[nt] (20 B/sample), maps
// interleaved fp64.  Every warp walks tiles of 32*K consecutive samples; lane l owns the K=8
// consecutive samples [tile*256 + 8l, +8) and reads them with 256-bit streaming loads
// (L2 evict-first, so the multi-GB TOD stream does not evict the L2-resident map).
//
// Scatter-add: a scan crosses a pixel in a run of consecutive samples, so (1) each lane compresses
// its 8 samples into runs in registers, (2) the open runs at lane boundaries are merged across the
// warp with a segmented shuffle scan, (3) one fp64 RED per (run, Stokes component) goes to L2.
// Random pointing degenerates gracefully to one RED per sample and component.
#include <cstdint>
#include <type_traits>

#include "cm2_common.cuh"

namespace cm2 {

constexpr int K = 8;          // consecutive samples per lane
constexpr int TILE = 32 * K;  // samples per warp tile
constexpr int BLOCK = 256;
constexpr unsigned FULL = 0xffffffffu;

struct BlockW {
    const double *w;       // per-block weights, nullptr = unit weights
    int64_t nblocks;
    int64_t blocksize;     // equal-size blocks when start == nullptr
    const int64_t *start;  // nblocks+1 block boundaries, or nullptr
    uint64_t magic;        // ceil(2^64 / blocksize): t / blocksize == umul64hi(t, magic) for t < 2^32 (0: unused)
};

static BlockW make_blockw(const double *w, int64_t nblocks, int64_t blocksize, const int64_t *start) {
    BlockW bw{w, nblocks, blocksize, start, 0};
    if (start == nullptr && blocksize > 1) bw.magic = ~(uint64_t)0 / (uint64_t)blocksize + 1;
    return bw;
}

__device__ __forceinline__ int64_t block_of(const BlockW &bw, int64_t t) {
    if (bw.start == nullptr) {
        // division by the invariant block size as one 64x64 -> high-64 multiply (exact for t < 2^32)
        if (bw.magic != 0 && ((uint64_t)t >> 32) == 0) return (int64_t)__umul64hi((uint64_t)t, bw.magic);
        return t / bw.blocksize;
    }
    return last_le(bw.start, bw.nblocks, t);
}

// weights of the K samples starting at t0 (one lookup when the chunk sits inside one block)
__device__ __forceinline__ void chunk_weights(const BlockW &bw, int64_t t0, int64_t nt, double (&w)[K]) {
    if (bw.w == nullptr) {
#pragma unroll
        for (int j = 0; j < K; ++j) w[j] = 1.0;
        return;
    }
    int64_t b0 = block_of(bw, t0);
    if (b0 >= bw.nblocks) b0 = bw.nblocks - 1;
    int64_t bend = bw.start ? bw.start[b0 + 1] : (b0 + 1) * bw.blocksize;
    if (t0 + K <= bend) {
        double w0 = __ldg(bw.w + b0);
#pragma unroll
        for (int j = 0; j < K; ++j) w[j] = w0;
    } else {
#pragma unroll
        for (int j = 0; j < K; ++j) {
            int64_t t = t0 + j;
            int64_t b = t < nt ? block_of(bw, t) : b0;
            if (b >= bw.nblocks) b = bw.nblocks - 1;
            w[j] = __ldg(bw.w + b);
        }
    }
}

// Order in which the persistent warps walk the tiles.  S = 1: time order.  S > 1: the tile sequence is cut into
// S streams of T tiles (S = number of detector timelines) and walked round-robin over the streams, so that all
// detectors are processed at the same scan time: they sweep the same sky rows then, and the part of x / y the
// kernel touches stays in L2 when the map itself (24 B/pixel each) is larger than L2.  In time order every
// detector timeline is one pass over the WHOLE map.
struct TileOrder {
    unsigned S, T;
    __device__ __forceinline__ int64_t count() const { return (int64_t)S * T; }
    __device__ __forceinline__ int64_t tile(int64_t v) const {
        if (S == 1) return v;
        const unsigned q = (unsigned)v / S, r = (unsigned)v - q * S;
        return (int64_t)r * T + q;
    }
    // first v' in {v, v + step, ...} below count() whose tile exists; sets tile = -1 at the end
    __device__ __forceinline__ int64_t next(int64_t v, int64_t step, int64_t ntiles, int64_t &t) const {
        const int64_t nv = count();
        for (; v < nv; v += step) {
            t = tile(v);
            if (t < ntiles) return v;
        }
        t = -1;
        return v;
    }
};

static TileOrder make_order(int64_t nt, int64_t nstreams) {
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    TileOrder o{1u, (unsigned)ntiles};
    if (nstreams > 1 && nstreams <= 65536 && ntiles >= 4 * nstreams && ntiles < ((int64_t)1 << 31)) {
        o.S = (unsigned)nstreams;
        o.T = (unsigned)((ntiles + nstreams - 1) / nstreams);
    }
    return o;
}

// Cache policy of the TOD loads.  STREAM: L2 evict-first, for data read once.  KEEP: default L2 priority, for the
// per-subscan kernels whose CTA reads the same samples again in a second pass.
enum Cache { STREAM, KEEP };

template <Cache CP = STREAM>
__device__ __forceinline__ void load_pix(const int32_t *__restrict__ pix, int64_t t0, int64_t nt, int (&p)[K]) {
    if (t0 + K <= nt) {
        I8 v = CP == KEEP ? ld_keep_i8(pix + t0) : ld_stream_i8(pix + t0);
#pragma unroll
        for (int j = 0; j < K; ++j) p[j] = v.v[j];
    } else {
#pragma unroll
        for (int j = 0; j < K; ++j) p[j] = (t0 + j < nt) ? (CP == KEEP ? pix[t0 + j] : ld_stream_i1(pix + t0 + j)) : -1;
    }
}

template <Cache CP = STREAM>
__device__ __forceinline__ void load_f64(const double *__restrict__ a, int64_t t0, int64_t nt, double (&c)[K]) {
    if (t0 + K <= nt) {
        D4 v0 = CP == KEEP ? ld_keep_d4(a + t0) : ld_stream_d4(a + t0);
        D4 v1 = CP == KEEP ? ld_keep_d4(a + t0 + 4) : ld_stream_d4(a + t0 + 4);
#pragma unroll
        for (int j = 0; j < 4; ++j) { c[j] = v0.v[j]; c[4 + j] = v1.v[j]; }
    } else {
#pragma unroll
        for (int j = 0; j < K; ++j) c[j] = (t0 + j < nt) ? (CP == KEEP ? a[t0 + j] : ld_stream_d1(a + t0 + j)) : 0.0;
    }
}

// Packed pixel stream (cm2_pack_pointing): one 64-bit word per lane of K samples, word t0 / K for the samples
// t0 .. t0 + K - 1, so a warp tile reads 256 contiguous bytes instead of 1 kB of int32 ids.  lo = bits 0..31, signed:
//   lo >= 0  b0 = lo, b1 = b0 + (int16) bits 32..47, codes = bits 48..63: sample j is (code & 2 ? b1 : b0) + (code & 1),
//            code = (codes >> 2j) & 3.  A raster sweep crosses each pixel in a run of samples and steps to the next
//            pixel or, at a row change, jumps by about a row length: two bases cover both.
//   lo == -1 every sample of the lane is flagged (-1).  The packer leaves bits 32..63 zero, so the decode of the
//            lo >= 0 case yields -1 for all K samples too.
//   lo == -2 escape: the lane reads its pixels from the int32 array.  Lanes that mix flagged and unflagged
//            samples, lanes the two bases do not cover, and a last lane of fewer than K samples escape.
constexpr int PK_FLAGGED = -1, PK_ESCAPE = -2;

__device__ __forceinline__ uint64_t ld_stream_u64(const uint64_t *p) {
    // the .L2::evict_first form of ld needs a 256-bit vector; an evict-first access policy does the same for 64 bits
    uint64_t pol, r;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.b64 %0, [%1], %2;" : "=l"(r) : "l"(p), "l"(pol));
    return r;
}

// The packed word of the lane at t0, PK_ESCAPE for a lane of fewer than K samples.  The load and the decode are apart
// (unpack_pix) so that the escape branch, which needs the word, does not hold back the work between them.
__device__ __forceinline__ uint64_t load_packed(const uint64_t *__restrict__ pk, int64_t t0, int64_t nt) {
    return t0 + K <= nt ? ld_stream_u64(pk + t0 / K) : (uint64_t)(uint32_t)PK_ESCAPE;
}

__device__ __forceinline__ void unpack_pix(uint64_t wd, const int32_t *__restrict__ pix, int64_t t0, int64_t nt,
                                           int (&p)[K]) {
    const int b0 = (int)(uint32_t)wd;
    if (b0 == PK_ESCAPE) {
        load_pix(pix, t0, nt, p);
        return;
    }
    const int b1 = b0 + (int)(int16_t)(uint16_t)(wd >> 32);
    const unsigned codes = (unsigned)(wd >> 48);
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const unsigned code = (codes >> (2 * j)) & 3u;
        p[j] = ((code & 2u) ? b1 : b0) + (int)(code & 1u);
    }
}

// pixels and, for POL > 1, cos / sin of the K samples starting at t0
template <int POL, Cache CP = STREAM>
__device__ __forceinline__ void load_tod(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                         const double *__restrict__ sn, int64_t t0, int64_t nt, int (&p)[K],
                                         double (&c)[K], double (&s)[K]) {
    load_pix<CP>(pix, t0, nt, p);
    if (POL > 1) { load_f64<CP>(cs, t0, nt, c); load_f64<CP>(sn, t0, nt, s); }
}

// the packed word of the K samples q (format above)
__device__ __forceinline__ uint64_t pack_lane(const int (&q)[K]) {
    bool all_flagged = true, any_flagged = false;
    int b0 = q[0];
#pragma unroll
    for (int j = 0; j < K; ++j) {
        all_flagged &= q[j] == -1;
        any_flagged |= q[j] < 0;
        b0 = min(b0, q[j]);
    }
    if (all_flagged) return (uint32_t)PK_FLAGGED;
    if (any_flagged) return (uint32_t)PK_ESCAPE;
    // b0 = the smallest pixel covers {b0, b0 + 1}; b1 = the smallest pixel above those covers {b1, b1 + 1}
    int b1 = b0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        if (q[j] - b0 > 1 && (b1 == b0 || q[j] < b1)) b1 = q[j];
    }
    if (b1 - b0 > INT16_MAX) return (uint32_t)PK_ESCAPE;
    uint64_t codes = 0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const int d0 = q[j] - b0, d1 = q[j] - b1;
        unsigned code;
        if (d0 <= 1) code = (unsigned)d0;
        else if (d1 <= 1) code = 2u + (unsigned)d1;
        else return (uint32_t)PK_ESCAPE;
        codes |= (uint64_t)code << (2 * j);
    }
    return (uint64_t)(uint32_t)b0 | ((uint64_t)(uint16_t)(b1 - b0) << 32) | (codes << 48);
}

// x values of the K samples; one gather per run start, copied along the run
template <int POL>
__device__ __forceinline__ void gather_x(const double *__restrict__ x, const int (&p)[K], double (&xv)[K][POL]) {
#pragma unroll
    for (int j = 0; j < K; ++j) {
        const bool nw = (j == 0) || (p[j] != p[j - 1]);
#pragma unroll
        for (int k = 0; k < POL; ++k) xv[j][k] = 0.0;
        if (nw && p[j] >= 0) {
            const double *xp = x + (int64_t)POL * p[j];
#pragma unroll
            for (int k = 0; k < POL; ++k) xv[j][k] = __ldg(xp + k);
        }
    }
#pragma unroll
    for (int j = 1; j < K; ++j) {
        if (p[j] == p[j - 1]) {
#pragma unroll
            for (int k = 0; k < POL; ++k) xv[j][k] = xv[j - 1][k];
        }
    }
}

template <int POL>
__device__ __forceinline__ double project(const double (&xv)[POL], double c, double s) {
    if constexpr (POL == 1) return xv[0];
    else if constexpr (POL == 2) return fma(xv[1], s, xv[0] * c);
    else return fma(xv[2], s, fma(xv[1], c, xv[0]));
}

// (P x) of sample j of the chunk (c, s are not read for POL = 1)
template <int POL>
__device__ __forceinline__ double project(const double (&xv)[K][POL], const double (&c)[K], const double (&s)[K], int j) {
    return project<POL>(xv[j], POL > 1 ? c[j] : 0.0, POL > 1 ? s[j] : 0.0);
}

// P^T contribution of sample j of the chunk with TOD value v[j]: the contrib functor of run_compress / run_scatter
template <int POL>
__device__ __forceinline__ auto pt_contrib(const double (&v)[K], const double (&c)[K], const double (&s)[K]) {
    return [&v, &c, &s](int j, double (&o)[POL]) {
        if constexpr (POL == 1) { o[0] = v[j]; }
        else if constexpr (POL == 2) { o[0] = v[j] * c[j]; o[1] = v[j] * s[j]; }
        else { o[0] = v[j]; o[1] = v[j] * c[j]; o[2] = v[j] * s[j]; }
    };
}

template <int NV, int STRIDE>
__device__ __forceinline__ void emit(double *__restrict__ y, int pix, const double (&v)[NV]) {
    if (pix >= 0) {
        double *dst = y + (int64_t)STRIDE * pix;
#pragma unroll
        for (int k = 0; k < NV; ++k) atomicAdd(dst + k, v[k]);  // result unused -> RED.E.ADD.F64
    }
}

// Run-compressed, warp-merged scatter-add of K samples per lane, in two phases so that a kernel
// can issue the next tile's loads between them:
//   run_compress: each lane folds its K samples into runs; complete interior runs are emitted,
//                 the first and the last (open) run stay in registers (RunState);
//   run_merge   : open runs are merged across lanes with a segmented shuffle scan and emitted.
// contrib(j, out[NV]) yields the NV values sample j adds to pixel p[j].  All 32 lanes must call.
template <int NV>
struct RunState {
    double acc[NV];    // partial of the run open at the end of the lane (== the only run if single)
    double head[NV];   // partial of the lane's first run (when the lane holds more than one run)
    int ph, pt;        // pixel of the first / last run
    bool single;

    // the state before the first tile: run_merge emits nothing for it
    __device__ __forceinline__ static RunState empty() {
        RunState rs;
        rs.ph = rs.pt = -1;
        rs.single = true;
#pragma unroll
        for (int k = 0; k < NV; ++k) rs.acc[k] = rs.head[k] = 0.0;
        return rs;
    }
};

template <int NV, int STRIDE, class F>
__device__ __forceinline__ void run_compress(double *__restrict__ y, const int (&p)[K], F contrib, RunState<NV> &rs) {
    int cur = p[0];
    rs.single = true;
    contrib(0, rs.acc);
#pragma unroll
    for (int k = 0; k < NV; ++k) rs.head[k] = 0.0;
#pragma unroll
    for (int j = 1; j < K; ++j) {
        double v[NV];
        contrib(j, v);
        if (p[j] != cur) {
            if (rs.single) {
#pragma unroll
                for (int k = 0; k < NV; ++k) rs.head[k] = rs.acc[k];
                rs.single = false;
            } else {
                emit<NV, STRIDE>(y, cur, rs.acc);
            }
            cur = p[j];
#pragma unroll
            for (int k = 0; k < NV; ++k) rs.acc[k] = v[k];
        } else {
#pragma unroll
            for (int k = 0; k < NV; ++k) rs.acc[k] += v[k];
        }
    }
    rs.ph = p[0];
    rs.pt = cur;
}

template <int NV, int STRIDE>
__device__ __forceinline__ void run_merge(double *__restrict__ y, RunState<NV> &rs) {
    const int lane = threadIdx.x & 31;
    const int pt_prev = __shfl_up_sync(FULL, rs.pt, 1);
    const int ph_next = __shfl_down_sync(FULL, rs.ph, 1);
    const bool cont_prev = (lane > 0) && (pt_prev == rs.ph);   // my first run continues the previous lane's last
    const bool cont_next = (lane < 31) && (ph_next == rs.pt);  // my last run continues into the next lane
    // segmented inclusive scan of the open partial over lanes; a lane starts a segment unless it
    // is one single run that continues the previous lane
    bool f = !(rs.single && cont_prev);
    if (__any_sync(FULL, !f)) {
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            double up[NV];
#pragma unroll
            for (int k = 0; k < NV; ++k) up[k] = __shfl_up_sync(FULL, rs.acc[k], d);
            const int fu = __shfl_up_sync(FULL, (int)f, d);
            if (lane >= d) {
                if (!f) {
#pragma unroll
                    for (int k = 0; k < NV; ++k) rs.acc[k] += up[k];
                }
                f = f || (fu != 0);
            }
        }
    }
    // rs.acc = partial of the run that is open at the end of this lane (carry-out)
    double cin[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) cin[k] = __shfl_up_sync(FULL, rs.acc[k], 1);
    if (!rs.single) {
        if (cont_prev) {
#pragma unroll
            for (int k = 0; k < NV; ++k) rs.head[k] += cin[k];
        }
        emit<NV, STRIDE>(y, rs.ph, rs.head);
    }
    if (!cont_next) emit<NV, STRIDE>(y, rs.pt, rs.acc);
}

template <int NV, int STRIDE, class F>
__device__ __forceinline__ void run_scatter(double *__restrict__ y, const int (&p)[K], F contrib) {
    RunState<NV> rs;
    run_compress<NV, STRIDE>(y, p, contrib, rs);
    run_merge<NV, STRIDE>(y, rs);
}

// ------------------------------------------------------------------------------------------
template <int POL>
__global__ void __launch_bounds__(BLOCK) k_pointing_apply(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                          const double *__restrict__ sn, int64_t nt,
                                                          const double *__restrict__ x, double *__restrict__ d) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    for (int64_t tile = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5); tile < ntiles; tile += nwarps) {
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        if (t0 >= nt) continue;
        int p[K];
        double c[K], s[K], xv[K][POL], out[K];
        load_tod<POL>(pix, cs, sn, t0, nt, p, c, s);
        gather_x<POL>(x, p, xv);
#pragma unroll
        for (int j = 0; j < K; ++j) out[j] = p[j] >= 0 ? project<POL>(xv, c, s, j) : 0.0;
        if (t0 + K <= nt) {
            D4 a, b;
#pragma unroll
            for (int j = 0; j < 4; ++j) { a.v[j] = out[j]; b.v[j] = out[4 + j]; }
            st_stream_d4(d + t0, a);
            st_stream_d4(d + t0 + 4, b);
        } else {
#pragma unroll
            for (int j = 0; j < K; ++j) if (t0 + j < nt) d[t0 + j] = out[j];
        }
    }
}

template <int POL>
__global__ void __launch_bounds__(BLOCK) k_pointing_apply_t(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                            const double *__restrict__ sn, int64_t nt,
                                                            const double *__restrict__ d, double *__restrict__ y) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    for (int64_t tile = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5); tile < ntiles; tile += nwarps) {
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        int p[K];
        double c[K], s[K], v[K];
        load_pix(pix, t0, nt, p);
        load_f64(d, t0, nt, v);
        if (POL > 1) { load_f64(cs, t0, nt, c); load_f64(sn, t0, nt, s); }
        run_scatter<POL, POL>(y, p, pt_contrib<POL>(v, c, s));
    }
}

// Fused y = P^T diag(w) P x.  The next tile's pix/cos/sin loads are issued between the compress
// and the merge phase of the current tile, so their DRAM latency overlaps the shuffles and REDs.
// WS = true: per-sample weights bw.w[t] (blocks of one sample: the pixel-sorted pointing copy), read as a stream.
// PK = true: the pixels come from the packed stream pk (8 B per lane instead of 32), int32 pix for escape lanes.
template <int POL, bool ILV, bool WS = false, bool PK = false>
__global__ void __launch_bounds__(BLOCK) k_amatvec_white(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                         const double *__restrict__ sn, int64_t nt, BlockW bw, TileOrder ord,
                                                         const double *__restrict__ x, double *__restrict__ y,
                                                         const uint64_t *__restrict__ pk) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    // The open runs of the previous tile (rs) are merged AFTER the loads of the current tile have been
    // issued, so DRAM latency overlaps the shuffles and REDs of the merge.  One load site per loop trip
    // (the loop-carried state is rs, 15 registers, not the 40 registers of p/c/s: the first version
    // carried p/c/s across the back edge and spent 79 register moves per tile on it).
    // ILV = false: time order (the instantiation measured on configs[1]); true: detector-interleaved (TileOrder).
    RunState<POL> rs = RunState<POL>::empty();
    const int64_t nv = ILV ? ord.count() : ntiles;
    const int64_t vt0 = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5);
    // PK: the packed word is loaded one trip ahead (2 registers), so the decode and the x gather do not wait for it
    uint64_t wd_next = 0;
    if constexpr (PK) wd_next = load_packed(pk, (ILV ? ord.tile(vt0) : vt0) * TILE + (int64_t)lane * K, nt);
    for (int64_t vt = vt0; vt < nv; vt += nwarps) {
        uint64_t wd = 0;
        if constexpr (PK) {
            wd = wd_next;
            const int64_t vn = vt + nwarps;
            wd_next = load_packed(pk, vn < nv ? (ILV ? ord.tile(vn) : vn) * TILE + (int64_t)lane * K : nt, nt);
        }
        int64_t tile = vt;
        if constexpr (ILV) {
            tile = ord.tile(vt);
            if (tile >= ntiles) continue;       // the last stream may be short
        }
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        int p[K];
        double c[K], s[K];
        if constexpr (PK) {
            if (POL > 1) { load_f64(cs, t0, nt, c); load_f64(sn, t0, nt, s); }
        } else {
            load_tod<POL>(pix, cs, sn, t0, nt, p, c, s);
        }
        run_merge<POL, POL>(y, rs);             // previous tile (the empty state on the first trip emits nothing)
        if constexpr (PK) unpack_pix(wd, pix, t0, nt, p);
        double w[K], xv[K][POL], v[K];
        if constexpr (WS) load_f64(bw.w, t0, nt, w);
        gather_x<POL>(x, p, xv);
        if constexpr (!WS) chunk_weights(bw, t0 < nt ? t0 : nt - 1, nt, w);
#pragma unroll
        for (int j = 0; j < K; ++j) v[j] = w[j] * project<POL>(xv, c, s, j);
        run_compress<POL, POL>(y, p, pt_contrib<POL>(v, c, s), rs);
    }
    run_merge<POL, POL>(y, rs);
}

// packed[l] = the packed word of lane l (samples 8 l .. 8 l + 7), one thread per lane; *nescape += escape lanes
__global__ void __launch_bounds__(BLOCK) k_pack_pointing(const int32_t *__restrict__ pix, int64_t nt,
                                                         uint64_t *__restrict__ packed, unsigned long long *__restrict__ nescape) {
    const int64_t nlanes = (nt + K - 1) / K;
    unsigned nesc = 0;
    for (int64_t l = (int64_t)blockIdx.x * BLOCK + threadIdx.x; l < nlanes; l += (int64_t)gridDim.x * BLOCK) {
        uint64_t wd = (uint32_t)PK_ESCAPE;
        if (l * K + K <= nt) {
            const I8 v = ld_stream_i8(pix + l * K);
            wd = pack_lane(v.v);
        }
        nesc += (int)(uint32_t)wd == PK_ESCAPE;
        packed[l] = wd;
    }
    nesc = __reduce_add_sync(FULL, nesc);
    if ((threadIdx.x & 31) == 0 && nesc) atomicAdd(nescape, (unsigned long long)nesc);
}

// Variant of k_amatvec_white with the scatter STAGED through shared memory: when the pixels of a warp tile span
// fewer than `wpix` pixels (a raster sweep along a pixel row: 256 / samples-per-pixel consecutive pixels), the
// lanes add their runs into a per-warp shared-memory window (fp64 CAS adds; collisions only where a run crosses a
// lane boundary or the scan turns around inside the tile) and the warp then flushes the window with REDs to
// CONSECUTIVE doubles: a warp-wide RED covers 8 sectors of y instead of up to 32, and a pixel crossed in fewer
// than 8 samples costs POL doubles of one coalesced RED instead of POL REDs of its own.  Tiles that span more
// (row changes, tilted or random pointing) take the register path of k_amatvec_white.  The window is zero
// outside [sink, flush]: the flush clears what it reads.
template <int POL>
__device__ __forceinline__ void stage_flush(double *__restrict__ sm, double *__restrict__ y, int64_t base, int len) {
    const int lane = threadIdx.x & 31;
    __syncwarp();
    for (int i = lane; i < len; i += 32) {
        const double v = sm[i];
        if (v != 0.0) {
            sm[i] = 0.0;
            atomicAdd(y + base + i, v);
        }
    }
    __syncwarp();
}

template <int POL>
__global__ void __launch_bounds__(BLOCK) k_amatvec_white_staged(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                                const double *__restrict__ sn, int64_t nt, BlockW bw, TileOrder ord,
                                                                const double *__restrict__ x, double *__restrict__ y, int wpix) {
    extern __shared__ double stage_sm[];
    const int lane = threadIdx.x & 31;
    double *sm = stage_sm + (size_t)(threadIdx.x >> 5) * POL * wpix;
    for (int i = lane; i < POL * wpix; i += 32) sm[i] = 0.0;
    __syncwarp();
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    const int64_t nv = ord.count();
    int64_t base_prev = 0;
    int len_prev = 0;
    for (int64_t vt = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5); vt < nv; vt += nwarps) {
        const int64_t tile = ord.tile(vt);
        if (tile >= ntiles) continue;
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        int p[K];
        double c[K], s[K];
        load_tod<POL>(pix, cs, sn, t0, nt, p, c, s);
        if (len_prev) stage_flush<POL>(sm, y, base_prev, len_prev);   // previous tile, after this tile's loads were issued
        len_prev = 0;
        double w[K], xv[K][POL], v[K];
        gather_x<POL>(x, p, xv);
        chunk_weights(bw, t0 < nt ? t0 : nt - 1, nt, w);
#pragma unroll
        for (int j = 0; j < K; ++j) v[j] = w[j] * project<POL>(xv, c, s, j);
        int lo = INT32_MAX, hi = INT32_MIN;
#pragma unroll
        for (int j = 0; j < K; ++j) {
            if (p[j] >= 0) { lo = min(lo, p[j]); hi = max(hi, p[j]); }
        }
        lo = __reduce_min_sync(FULL, lo);
        hi = __reduce_max_sync(FULL, hi);
        if (hi < lo) continue;                                    // every sample of the tile is flagged
        auto contrib = pt_contrib<POL>(v, c, s);
        if ((int64_t)hi - lo < wpix) {                            // warp-uniform
            double acc[POL];
            int cur = p[0];
            contrib(0, acc);
#pragma unroll
            for (int j = 1; j <= K; ++j) {
                double o[POL];
                if (j < K) contrib(j, o);
                if (j == K || p[j] != cur) {
                    if (cur >= 0) {
                        double *dst = sm + (cur - lo) * POL;
#pragma unroll
                        for (int k = 0; k < POL; ++k) atomicAdd(dst + k, acc[k]);
                    }
                    if (j < K) {
                        cur = p[j];
#pragma unroll
                        for (int k = 0; k < POL; ++k) acc[k] = o[k];
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < POL; ++k) acc[k] += o[k];
                }
            }
            base_prev = (int64_t)POL * lo;
            len_prev = POL * (hi - lo + 1);
        } else {
            RunState<POL> rs;
            run_compress<POL, POL>(y, p, contrib, rs);
            run_merge<POL, POL>(y, rs);
        }
    }
    if (len_prev) stage_flush<POL>(sm, y, base_prev, len_prev);
}

// Fused y = P^T T P x for a short symmetric band (T = the banded Toeplitz blocks of
// BlockLO(offdiag=True), linearoperators.py:582-595, 672-674; the composition P.T*N*P of
// tests/test_2level_preconditioner.py:16-29), NLAG = nband-1 <= 8 lags: one pass over the TOD, no
// time-domain temporary (20 B/sample instead of the 28 + 16 + 28 of the chain P, T, P^T).
// Warp tiles OVERLAP: a warp loads 256 consecutive samples, the first and last HL lanes are halo
// (their P x is only input to the neighbours' band sums), the 256 - 16 HL samples in between are the
// tile's outputs.  P x of the tile goes through 2 kB of shared memory per warp, stored transposed
// (element (lane, j) at 32 j + lane: conflict-free for the store and for the neighbour reads, which
// have a fixed offset to 8 lane + j); every lane then reads its 2 NLAG neighbours once and slides
// the band over a register window.  Contributions never cross a noise block (the zero boundary of
// ToeplitzLO): masked by the block's [begin, end) on the rare lanes near a boundary; a lane whose
// own 8 samples straddle a boundary takes a per-sample path.
struct ToepW {
    const double *band;    // [nblocks][nband]: a_0 .. a_{nband-1} per block
    int nband;
    BlockW blk;            // block geometry (w unused)
};

template <int POL, int NLAG>
__global__ void __launch_bounds__(BLOCK) k_amatvec_toeplitz(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                            const double *__restrict__ sn, int64_t nt, ToepW tw,
                                                            const double *__restrict__ x, double *__restrict__ y) {
    constexpr int HL = (NLAG + K - 1) / K;     // halo lanes on either side
    constexpr int VAL = TILE - 2 * HL * K;     // output samples per tile
    __shared__ double sv_all[BLOCK / 32][TILE];
    double *sv = sv_all[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + VAL - 1) / VAL;
    RunState<POL> rs = RunState<POL>::empty();
    for (int64_t tile = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5); tile < ntiles; tile += nwarps) {
        const int64_t t0 = tile * VAL - HL * K + (int64_t)lane * K;   // multiple of 8: the 256-bit loads stay aligned
        int p[K];
        double c[K], s[K];
        if (t0 >= 0) {
            load_tod<POL>(pix, cs, sn, t0, nt, p, c, s);
        } else {
#pragma unroll
            for (int j = 0; j < K; ++j) { p[j] = -1; c[j] = 0.0; s[j] = 0.0; }
        }
        run_merge<POL, POL>(y, rs);            // previous tile, after this tile's loads have been issued
        double v[K];
        {
            double xv[K][POL];
            gather_x<POL>(x, p, xv);
#pragma unroll
            for (int j = 0; j < K; ++j) v[j] = p[j] >= 0 ? project<POL>(xv, c, s, j) : 0.0;
        }
#pragma unroll
        for (int j = 0; j < K; ++j) sv[32 * j + lane] = v[j];
        __syncwarp();
        double out[K];
        const bool active = lane >= HL && lane < 32 - HL && t0 < nt;
        if (active) {
            int64_t b0 = block_of(tw.blk, t0);
            if (b0 >= tw.blk.nblocks) b0 = tw.blk.nblocks - 1;
            const int64_t bs = tw.blk.start ? __ldg(tw.blk.start + b0) : b0 * tw.blk.blocksize;
            int64_t be = tw.blk.start ? __ldg(tw.blk.start + b0 + 1) : (b0 + 1 == tw.blk.nblocks ? nt : (b0 + 1) * tw.blk.blocksize);
            if (be > nt) be = nt;
            if (t0 + K <= be) {                // the lane's 8 samples lie in one noise block (the common case)
                const double *a = tw.band + b0 * tw.nband;
                double ak[NLAG + 1];
#pragma unroll
                for (int k = 0; k <= NLAG; ++k) ak[k] = k < tw.nband ? __ldg(a + k) : 0.0;
                double w[K + 2 * NLAG];        // P x at t0 - NLAG .. t0 + K + NLAG - 1
#pragma unroll
                for (int m = 0; m < NLAG; ++m) {
                    const int il = K * lane - NLAG + m, ir = K * lane + K + m;
                    w[m] = (t0 - NLAG + m >= bs) ? sv[32 * (il & 7) + (il >> 3)] : 0.0;
                    w[NLAG + K + m] = (t0 + K + m < be) ? sv[32 * (ir & 7) + (ir >> 3)] : 0.0;
                }
#pragma unroll
                for (int j = 0; j < K; ++j) w[NLAG + j] = v[j];
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    double acc = ak[0] * w[NLAG + j];
#pragma unroll
                    for (int k = 1; k <= NLAG; ++k) acc = fma(ak[k], w[NLAG + j - k] + w[NLAG + j + k], acc);
                    out[j] = acc;
                }
            } else {                           // a block boundary inside the lane's samples: per sample
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const int64_t t = t0 + j;
                    out[j] = 0.0;
                    if (t >= nt) continue;
                    int64_t b = block_of(tw.blk, t);
                    if (b >= tw.blk.nblocks) b = tw.blk.nblocks - 1;
                    const int64_t s0 = tw.blk.start ? __ldg(tw.blk.start + b) : b * tw.blk.blocksize;
                    int64_t s1 = tw.blk.start ? __ldg(tw.blk.start + b + 1) : (b + 1 == tw.blk.nblocks ? nt : (b + 1) * tw.blk.blocksize);
                    if (s1 > nt) s1 = nt;
                    const double *a = tw.band + b * tw.nband;
                    double acc = __ldg(a) * v[j];
                    for (int k = 1; k <= NLAG && k < tw.nband; ++k) {
                        const int il = K * lane + j - k, ir = K * lane + j + k;
                        double nb = 0.0;
                        if (t - k >= s0) nb += sv[32 * (il & 7) + (il >> 3)];
                        if (t + k < s1) nb += sv[32 * (ir & 7) + (ir >> 3)];
                        acc = fma(__ldg(a + k), nb, acc);
                    }
                    out[j] = acc;
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < K; ++j) { out[j] = 0.0; p[j] = -1; }
        }
        __syncwarp();                          // all reads of sv done before the next tile overwrites it
        run_compress<POL, POL>(y, p, pt_contrib<POL>(out, c, s), rs);
    }
    run_merge<POL, POL>(y, rs);
}

// Fused y = P^T (P x - mu_seg) over the unflagged samples inside subscans: the offset-filtered
// A-matvec in ONE pass over the TOD, given the subscan means mu (k_seg_mean, filter_runs.cu).
// tile_seg[tile] = index of the first segment whose end lies beyond the tile's first sample.
struct SegInfo {
    const int64_t *start, *end;   // nseg, sorted, non-overlapping
    const double *mu;             // nseg
    const int32_t *tile_seg;      // ntiles: first segment ending beyond the tile's first sample
    const uint8_t *tile_flag;     // ntiles: 0 = tile outside every segment, 1 = inside one, 2 = mixed
    int64_t nseg;
};

template <int POL>
__global__ void __launch_bounds__(BLOCK) k_amatvec_filter_mu(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                             const double *__restrict__ sn, int64_t nt, SegInfo sg, TileOrder ord,
                                                             const double *__restrict__ x, double *__restrict__ y) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    // Three tiles are in flight per warp: the current one (registers), the next one (its TOD loads and its subscan
    // mean are issued before the merge of the current tile) and the one after (only its subscan lookup: flag and
    // segment index), so that mu[k0] of the next tile never waits for the load of k0 -- the lookups are a chain
    // tile -> segment -> mean of dependent L2 accesses otherwise.
    int64_t tile, tile2;
    int64_t v = ord.next((int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5), nwarps, ntiles, tile);
    if (tile < 0) return;
    int64_t v2 = ord.next(v + nwarps, nwarps, ntiles, tile2);
    int p[K];
    double c[K], s[K];
    int flag, k0, flag2 = 0, k02 = 0;
    double m0;
    {
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        load_tod<POL>(pix, cs, sn, t0, nt, p, c, s);
        flag = __ldg(sg.tile_flag + tile);
        k0 = __ldg(sg.tile_seg + tile);
        if (tile2 >= 0) { flag2 = __ldg(sg.tile_flag + tile2); k02 = __ldg(sg.tile_seg + tile2); }
        m0 = flag == 1 ? __ldg(sg.mu + k0) : 0.0;
    }
    while (tile >= 0) {
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        double mu[K];
        if (flag == 1) {                       // the whole tile lies inside subscan k0 (the common case)
#pragma unroll
            for (int j = 0; j < K; ++j) mu[j] = m0;
        } else if (flag == 0) {                // the whole tile lies in a gap
#pragma unroll
            for (int j = 0; j < K; ++j) { mu[j] = 0.0; p[j] = -1; }
        } else {                               // a subscan boundary falls inside the tile
            int64_t k = k0;
            while (k < sg.nseg && __ldg(sg.end + k) <= t0) ++k;
            int64_t a = k < sg.nseg ? __ldg(sg.start + k) : INT64_MAX, b = k < sg.nseg ? __ldg(sg.end + k) : INT64_MAX;
            double m = k < sg.nseg ? __ldg(sg.mu + k) : 0.0;
            if (t0 >= a && t0 + K <= b) {      // this lane's chunk is still inside one subscan
#pragma unroll
                for (int j = 0; j < K; ++j) mu[j] = m;
            } else if (t0 + K <= a) {          // ... or entirely in a gap
#pragma unroll
                for (int j = 0; j < K; ++j) { mu[j] = 0.0; p[j] = -1; }
            } else {                           // the boundary is inside this lane's 8 samples
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const int64_t t = t0 + j;
                    while (k < sg.nseg && t >= b) {
                        ++k;
                        a = k < sg.nseg ? __ldg(sg.start + k) : INT64_MAX;
                        b = k < sg.nseg ? __ldg(sg.end + k) : INT64_MAX;
                        m = k < sg.nseg ? __ldg(sg.mu + k) : 0.0;
                    }
                    if (t < a || k >= sg.nseg) p[j] = -1;
                    mu[j] = m;
                }
            }
        }
        RunState<POL> rs;
        {
            double xv[K][POL], vv[K];
            gather_x<POL>(x, p, xv);
#pragma unroll
            for (int j = 0; j < K; ++j) vv[j] = project<POL>(xv, c, s, j) - mu[j];
            run_compress<POL, POL>(y, p, pt_contrib<POL>(vv, c, s), rs);
        }
        int64_t tile3 = -1, v3 = v2;
        int flag3 = 0, k03 = 0;
        if (tile2 >= 0) {     // warp-uniform: the next tile's TOD loads and mean, the lookup of the tile after it
            const int64_t t1 = tile2 * TILE + (int64_t)lane * K;
            load_tod<POL>(pix, cs, sn, t1, nt, p, c, s);
            m0 = flag2 == 1 ? __ldg(sg.mu + k02) : 0.0;
            v3 = ord.next(v2 + nwarps, nwarps, ntiles, tile3);
            if (tile3 >= 0) { flag3 = __ldg(sg.tile_flag + tile3); k03 = __ldg(sg.tile_seg + tile3); }
        }
        run_merge<POL, POL>(y, rs);
        tile = tile2; flag = flag2; k0 = k02;
        tile2 = tile3; flag2 = flag3; k02 = k03; v2 = v3;
    }
}

// Fused y = P^T (P x - sum_k c_k L_k(x_t)) over the unflagged samples inside subscans: the Legendre-
// filtered A-matvec in ONE pass over the TOD, given the per-subscan coefficients (k_poly_seg_coef,
// filter_runs.cu).  Same tile / subscan lookup as k_amatvec_filter_mu; x_t = -1 + 2 (t - a)/(len - 1).
struct SegPoly {
    const int64_t *start, *end;   // nseg, sorted, non-overlapping (the subscans this path handles)
    const double *coef;           // nseg x NK
    const int32_t *tile_seg;
    const uint8_t *tile_flag;
    int64_t nseg;
};

template <int NK>
__device__ __forceinline__ double poly_eval(const double (&cf)[NK], double xt) {
    double L[NK];
    legendre<NK>(xt, L);
    double p = cf[0];
#pragma unroll
    for (int k = 1; k < NK; ++k) p = fma(cf[k], L[k], p);
    return p;
}

template <int POL, int NK>
__global__ void __launch_bounds__(BLOCK) k_amatvec_filter_poly_mu(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                                  const double *__restrict__ sn, int64_t nt, SegPoly sg, TileOrder ord,
                                                                  const double *__restrict__ x, double *__restrict__ y) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    RunState<POL> rs = RunState<POL>::empty();
    const int64_t nv = ord.count();
    for (int64_t vt = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5); vt < nv; vt += nwarps) {
        const int64_t tile = ord.tile(vt);
        if (tile >= ntiles) continue;          // the last stream may be short
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        int p[K];
        double c[K], s[K];
        load_tod<POL>(pix, cs, sn, t0, nt, p, c, s);
        const int flag = __ldg(sg.tile_flag + tile);
        const int k0 = __ldg(sg.tile_seg + tile);
        run_merge<POL, POL>(y, rs);            // previous tile, after this tile's loads have been issued
        double pv[K];                          // the polynomial at the lane's samples
        if (flag == 0) {                       // the whole tile lies in a gap
#pragma unroll
            for (int j = 0; j < K; ++j) { pv[j] = 0.0; p[j] = -1; }
        } else {
            int64_t k = k0;
            if (flag != 1) {
                while (k < sg.nseg && __ldg(sg.end + k) <= t0) ++k;
            }
            int64_t a = k < sg.nseg ? __ldg(sg.start + k) : INT64_MAX, b = k < sg.nseg ? __ldg(sg.end + k) : INT64_MAX;
            if (flag == 1 || (t0 >= a && t0 + K <= b)) {   // the lane's chunk lies inside one subscan
                double cf[NK];
#pragma unroll
                for (int i = 0; i < NK; ++i) cf[i] = __ldg(sg.coef + k * NK + i);
                const double step = b - a > 1 ? 2.0 / (double)(b - a - 1) : 0.0;
                const double x0 = fma((double)(t0 - a), step, -1.0);
#pragma unroll
                for (int j = 0; j < K; ++j) pv[j] = poly_eval<NK>(cf, fma((double)j, step, x0));
            } else if (t0 + K <= a) {                      // ... or entirely in a gap
#pragma unroll
                for (int j = 0; j < K; ++j) { pv[j] = 0.0; p[j] = -1; }
            } else {                                       // a subscan boundary inside the lane's 8 samples
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const int64_t t = t0 + j;
                    while (k < sg.nseg && t >= b) {
                        ++k;
                        a = k < sg.nseg ? __ldg(sg.start + k) : INT64_MAX;
                        b = k < sg.nseg ? __ldg(sg.end + k) : INT64_MAX;
                    }
                    pv[j] = 0.0;
                    if (k >= sg.nseg || t < a) { p[j] = -1; continue; }
                    double cf[NK];
#pragma unroll
                    for (int i = 0; i < NK; ++i) cf[i] = __ldg(sg.coef + k * NK + i);
                    const double step = b - a > 1 ? 2.0 / (double)(b - a - 1) : 0.0;
                    pv[j] = poly_eval<NK>(cf, fma((double)(t - a), step, -1.0));
                }
            }
        }
        double xv[K][POL], v[K];
        gather_x<POL>(x, p, xv);
#pragma unroll
        for (int j = 0; j < K; ++j) v[j] = project<POL>(xv, c, s, j) - pv[j];
        run_compress<POL, POL>(y, p, pt_contrib<POL>(v, c, s), rs);
    }
    run_merge<POL, POL>(y, rs);
}

// d = F P x for the offset filter in one pass (no P x temporary, no second pass for F): the subscan
// means of P x come from the run table (k_seg_mean), so d_t = (P x)_t - mu_seg(t) inside subscans --
// also on flagged samples, where (P x)_t = 0, exactly as FilterLO.mult subtracts the mean from them
// (linearoperators.py:165) -- and 0 in the gaps.  28 B/sample instead of 28 + 20.
template <int POL>
__global__ void __launch_bounds__(BLOCK) k_pointing_filter_mu(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                              const double *__restrict__ sn, int64_t nt, SegInfo sg,
                                                              const double *__restrict__ x, double *__restrict__ d) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    int64_t tile = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5);
    if (tile >= ntiles) return;
    // the subscan lookup of a tile (flag, segment index, and from it the mean) is a chain of dependent L2 accesses:
    // it is issued one trip ahead (flag / index two trips ahead), as in k_amatvec_filter_mu
    int flag = __ldg(sg.tile_flag + tile), k0 = __ldg(sg.tile_seg + tile);
    int flag2 = 0, k02 = 0;
    if (tile + nwarps < ntiles) { flag2 = __ldg(sg.tile_flag + tile + nwarps); k02 = __ldg(sg.tile_seg + tile + nwarps); }
    double m0 = flag == 1 ? __ldg(sg.mu + k0) : 0.0;
    for (; tile < ntiles; tile += nwarps) {
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        // next trip's mean and the lookup of the trip after it, before this tile's loads are waited for
        const double m0n = (tile + nwarps < ntiles && flag2 == 1) ? __ldg(sg.mu + k02) : 0.0;
        int flag3 = 0, k03 = 0;
        if (tile + 2 * nwarps < ntiles) { flag3 = __ldg(sg.tile_flag + tile + 2 * nwarps); k03 = __ldg(sg.tile_seg + tile + 2 * nwarps); }
        if (t0 < nt) {
            int p[K];
            double c[K], s[K], mu[K], xv[K][POL], out[K];
            bool in[K];
            load_tod<POL>(pix, cs, sn, t0, nt, p, c, s);
            if (flag == 1) {
#pragma unroll
                for (int j = 0; j < K; ++j) { mu[j] = m0; in[j] = true; }
            } else if (flag == 0) {
#pragma unroll
                for (int j = 0; j < K; ++j) { mu[j] = 0.0; in[j] = false; }
            } else {
                int64_t k = k0;
                while (k < sg.nseg && __ldg(sg.end + k) <= t0) ++k;
                int64_t a = k < sg.nseg ? __ldg(sg.start + k) : INT64_MAX, b = k < sg.nseg ? __ldg(sg.end + k) : INT64_MAX;
                double m = k < sg.nseg ? __ldg(sg.mu + k) : 0.0;
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const int64_t t = t0 + j;
                    while (k < sg.nseg && t >= b) {
                        ++k;
                        a = k < sg.nseg ? __ldg(sg.start + k) : INT64_MAX;
                        b = k < sg.nseg ? __ldg(sg.end + k) : INT64_MAX;
                        m = k < sg.nseg ? __ldg(sg.mu + k) : 0.0;
                    }
                    in[j] = k < sg.nseg && t >= a;
                    mu[j] = m;
                }
            }
#pragma unroll
            for (int j = 0; j < K; ++j) if (!in[j]) p[j] = -1;
            gather_x<POL>(x, p, xv);
#pragma unroll
            for (int j = 0; j < K; ++j) out[j] = in[j] ? (p[j] >= 0 ? project<POL>(xv, c, s, j) : 0.0) - mu[j] : 0.0;
            if (t0 + K <= nt) {
                D4 a, b;
#pragma unroll
                for (int j = 0; j < 4; ++j) { a.v[j] = out[j]; b.v[j] = out[4 + j]; }
                st_stream_d4(d + t0, a);
                st_stream_d4(d + t0 + 4, b);
            } else {
#pragma unroll
                for (int j = 0; j < K; ++j) if (t0 + j < nt) d[t0 + j] = out[j];
            }
        }
        flag = flag2; k0 = k02; m0 = m0n;
        flag2 = flag3; k02 = k03;
    }
}

// moments layout: mom[npix][6] = {h, c, s, c2, cs, s2}; pol=1 fills {h}, pol=2 {c2,cs,s2}, pol=3 all
template <int POL>
__global__ void __launch_bounds__(BLOCK) k_moments(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                   const double *__restrict__ sn, const double *__restrict__ wsamp,
                                                   BlockW bw, int64_t nt, double *__restrict__ mom) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    constexpr int NV = POL == 1 ? 1 : (POL == 2 ? 3 : 6);
    for (int64_t tile = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5); tile < ntiles; tile += nwarps) {
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        int p[K];
        double c[K], s[K], w[K];
        load_tod<POL>(pix, cs, sn, t0, nt, p, c, s);
        if (wsamp) load_f64(wsamp, t0, nt, w);
        else chunk_weights(bw, t0 < nt ? t0 : nt - 1, nt, w);
        double *base = mom + (POL == 2 ? 3 : 0);
        run_scatter<NV, 6>(base, p, [&](int j, double (&o)[NV]) {
            // same association as the reference loops: (w*c)*c, (w*s)*s, (w*s)*c
            if constexpr (POL == 1) { o[0] = w[j]; }
            else if constexpr (POL == 2) {
                o[0] = (w[j] * c[j]) * c[j]; o[1] = (w[j] * s[j]) * c[j]; o[2] = (w[j] * s[j]) * s[j];
            } else {
                o[0] = w[j]; o[1] = w[j] * c[j]; o[2] = w[j] * s[j];
                o[3] = (w[j] * c[j]) * c[j]; o[4] = (w[j] * s[j]) * c[j]; o[5] = (w[j] * s[j]) * s[j];
            }
        });
    }
}

__global__ void __launch_bounds__(BLOCK) k_hits(const int32_t *__restrict__ pix, int64_t nt, unsigned long long *__restrict__ hits) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (BLOCK / 32);
    const int64_t ntiles = (nt + TILE - 1) / TILE;
    for (int64_t tile = (int64_t)blockIdx.x * (BLOCK / 32) + (threadIdx.x >> 5); tile < ntiles; tile += nwarps) {
        const int64_t t0 = tile * TILE + (int64_t)lane * K;
        if (t0 >= nt) continue;
        int p[K];
        load_pix(pix, t0, nt, p);
        int cur = p[0];
        unsigned long long n = 1;
#pragma unroll
        for (int j = 1; j < K; ++j) {
            if (p[j] != cur) {
                if (cur >= 0) atomicAdd(hits + cur, n);
                cur = p[j];
                n = 1;
            } else {
                ++n;
            }
        }
        if (cur >= 0) atomicAdd(hits + cur, n);
    }
}


// ---- fused y = P^T F P x (offset filter) --------------------------------------------------------
// One CTA per subscan segment [a, b).  Pass 1 gathers d_t = (P x)_t, keeps it in shared memory and
// reduces the masked sum (fixed order -> deterministic mean); pass 2 scatters (d_t - mean) for the
// unflagged samples.  pix/cos/sin are read from HBM once (pass 1 leaves them in L2 for pass 2).
// Tiles are aligned to multiples of TILE in the global sample index so the 256-bit loads stay
// aligned; samples of a tile outside [a, b) are treated as flagged.
constexpr int SEG_SMEM = 12288;  // d_t values kept on chip per segment (96 kB dynamic smem, 2 CTAs/SM); longer -> recompute

template <int POL>
__global__ void __launch_bounds__(BLOCK) k_amatvec_filter(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                          const double *__restrict__ sn, int64_t nt,
                                                          const int64_t *__restrict__ seg_start,
                                                          const int64_t *__restrict__ seg_end, int64_t nseg,
                                                          const double *__restrict__ x, double *__restrict__ y) {
    extern __shared__ double sd[];   // SEG_SMEM doubles
    __shared__ double red[32];
    __shared__ double s_mean;
    __shared__ int s_skip;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t a = seg_start[k], b = seg_end[k];
        const int64_t tile0 = a / TILE, tile1 = (b + TILE - 1) / TILE;   // [tile0, tile1)
        const int64_t base = tile0 * TILE;
        const bool fits = (tile1 - tile0) * TILE <= SEG_SMEM;
        double sum = 0.0, cnt = 0.0;
        for (int64_t tile = tile0 + warp; tile < tile1; tile += BLOCK / 32) {
            const int64_t t0 = tile * TILE + (int64_t)lane * K;
            const int tb = (int)(tile * TILE - base);   // bank-conflict-free tile layout: (lane, j) at tb + 32 j + lane
            int p[K];
            double c[K], s[K], xv[K][POL];
            load_pix<KEEP>(pix, t0, nt, p);
#pragma unroll
            for (int j = 0; j < K; ++j) if (t0 + j < a || t0 + j >= b) p[j] = -1;
            if (POL > 1) { load_f64<KEEP>(cs, t0, nt, c); load_f64<KEEP>(sn, t0, nt, s); }
            gather_x<POL>(x, p, xv);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const double dv = p[j] >= 0 ? project<POL>(xv, c, s, j) : 0.0;
                if (p[j] >= 0) { sum += dv; cnt += 1.0; }
                if (fits) sd[tb + j * 32 + lane] = dv;
            }
        }
        const double tsum = block_sum(sum, red);
        const double tcnt = block_sum(cnt, red);
        if (threadIdx.x == 0) {
            s_skip = !(tcnt > 0.0);
            s_mean = tcnt > 0.0 ? tsum / tcnt : 0.0;
        }
        __syncthreads();
        if (!s_skip) {
            const double mu = s_mean;
            for (int64_t tile = tile0 + warp; tile < tile1; tile += BLOCK / 32) {
                const int64_t t0 = tile * TILE + (int64_t)lane * K;
                const int tb = (int)(tile * TILE - base);
                int p[K];
                double c[K], s[K], v[K];
                load_pix(pix, t0, nt, p);
#pragma unroll
                for (int j = 0; j < K; ++j) if (t0 + j < a || t0 + j >= b) p[j] = -1;
                if (POL > 1) { load_f64(cs, t0, nt, c); load_f64(sn, t0, nt, s); }
                if (fits) {
#pragma unroll
                    for (int j = 0; j < K; ++j) v[j] = sd[tb + j * 32 + lane] - mu;
                } else {
                    double xv[K][POL];
                    gather_x<POL>(x, p, xv);
#pragma unroll
                    for (int j = 0; j < K; ++j) v[j] = project<POL>(xv, c, s, j) - mu;
                }
                run_scatter<POL, POL>(y, p, pt_contrib<POL>(v, c, s));
            }
        }
        __syncthreads();
    }
}

// Fused y = P^T F_K P x with the Legendre subscan filter F_K (FilterLO.polyfilter,
// linearoperators.py:170-204; NK = poly_order + 1 >= 2): one CTA per subscan, no TOD temporary.
//   pass 1: the subscan's pixels and d = P x -> shared memory; number / first / last unflagged sample;
//           S_k = sum L_k d, G_kl = sum L_k L_l in the Legendre basis of the whole subscan
//   solve : c_k = S_k / G_kk without flags (the reference's literal sum over the sampled,
//           not exactly orthogonal, basis), else G c = S (QR re-orthonormalised basis, :190-194);
//           if G is ill-conditioned (flags leave only part of the subscan) the moments are redone
//           from shared memory in the basis of the interval the unflagged samples span
//   pass 2: scatter-add of d - sum_k c_k L_k over the unflagged samples
// cap = shared-memory window in samples (a multiple of TILE covering the longest subscan).
template <int POL, int NK>
__global__ void __launch_bounds__(BLOCK, 2) k_amatvec_filter_poly(const int32_t *__restrict__ pix, const double *__restrict__ cs,
                                                               const double *__restrict__ sn, int64_t nt,
                                                               const int64_t *__restrict__ seg_start,
                                                               const int64_t *__restrict__ seg_end, int64_t nseg,
                                                               const double *__restrict__ x, double *__restrict__ y, int cap) {
    constexpr int NR = NK + NK * (NK + 1) / 2;
    constexpr int NW = BLOCK / 32;
    extern __shared__ double sd[];                          // cap doubles, then cap ints
    int *sp = reinterpret_cast<int *>(sd + cap);
    __shared__ double red[NW * NR];
    __shared__ double tot[NR];
    __shared__ double coef[NK];
    __shared__ int s_cnt, s_jmin, s_jmax, s_refine, s_local;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t a = seg_start[k], b = seg_end[k];
        const int64_t tile0 = a / TILE, tile1 = (b + TILE - 1) / TILE;   // [tile0, tile1)
        const int64_t base = tile0 * TILE;
        const int len = (int)(b - a);
        if (threadIdx.x == 0) { s_cnt = 0; s_jmin = INT32_MAX; s_jmax = -1; }
        __syncthreads();
        // ---- pass 1 (the only read of pix): pixels and d = P x -> shared memory; number / first / last
        // unflagged sample; S and G in the Legendre basis of the WHOLE subscan (x = -1 + 2 j/(len-1)),
        // which is the reference's basis without flags and close to orthogonal with a few flags
        const double step_f = len > 1 ? 2.0 / (double)(len - 1) : 0.0;
        int cnt = 0, jmin = INT32_MAX, jmax = -1;
        double acc[NR];
#pragma unroll
        for (int i = 0; i < NR; ++i) acc[i] = 0.0;
        for (int64_t tile = tile0 + warp; tile < tile1; tile += NW) {
            const int64_t t0 = tile * TILE + (int64_t)lane * K;
            const int tb = (int)(tile * TILE - base);
            const double jb = (double)(int)(t0 - a);
            int p[K];
            double c[K], s[K], xv[K][POL];
            load_tod<POL, KEEP>(pix, cs, sn, t0, nt, p, c, s);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                if (t0 + j < a || t0 + j >= b || p[j] < 0) p[j] = -1;
                sp[tb + j * 32 + lane] = p[j];
            }
            gather_x<POL>(x, p, xv);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                double dv = 0.0;
                if (p[j] >= 0) {
                    const int jj = (int)(t0 - a) + j;
                    ++cnt;
                    jmin = min(jmin, jj);
                    jmax = max(jmax, jj);
                    dv = project<POL>(xv, c, s, j);
                    double L[NK];
                    legendre<NK>(fma(jb + (double)j, step_f, -1.0), L);
                    int q = NK;
#pragma unroll
                    for (int r = 0; r < NK; ++r) {
                        acc[r] = fma(L[r], dv, acc[r]);
#pragma unroll
                        for (int l = r; l < NK; ++l) { acc[q] = fma(L[r], L[l], acc[q]); ++q; }
                    }
                }
                sd[tb + j * 32 + lane] = dv;
            }
        }
        cnt = __reduce_add_sync(FULL, cnt);
        jmin = __reduce_min_sync(FULL, jmin);
        jmax = __reduce_max_sync(FULL, jmax);
        if (lane == 0 && cnt > 0) { atomicAdd(&s_cnt, cnt); atomicMin(&s_jmin, jmin); atomicMax(&s_jmax, jmax); }
        block_sum_n<NR, NW>(acc, red, tot);                  // barriers inside: the counters are complete after it
        const int n = s_cnt;
        if (n > NK - 1) {                                    // block-uniform (else: too few samples, :185-187)
            const bool full = n == len;
            if (threadIdx.x == 0) {
                s_refine = 0;
                s_local = 0;
                if (full) {                                  // the reference's literal sum_k (b_k . d) b_k
                    int q = NK;
#pragma unroll
                    for (int r = 0; r < NK; ++r) {
                        coef[r] = tot[q] > 0.0 ? tot[r] / tot[q] : 0.0;
                        q += NK - r;
                    }
                } else {
                    double cc[NK];
                    // ill-conditioned in the whole-subscan basis (the unflagged samples cluster in part of
                    // the subscan): redo the moments in the basis of the interval they span
                    s_local = gram_solve<NK>(tot + NK, tot, cc) < 1e-3;
#pragma unroll
                    for (int r = 0; r < NK; ++r) coef[r] = cc[r];
                }
            }
            __syncthreads();
            int j0 = 0;
            double step = step_f;
            if (s_local) {                                   // block-uniform, rare: shared memory only
                j0 = s_jmin;
                step = 2.0 / (double)(s_jmax - s_jmin);
#pragma unroll
                for (int i = 0; i < NR; ++i) acc[i] = 0.0;
                for (int64_t tile = tile0 + warp; tile < tile1; tile += NW) {
                    const int64_t t0 = tile * TILE + (int64_t)lane * K;
                    const int tb = (int)(tile * TILE - base);
                    const double jb = (double)((int)(t0 - a) - j0);
#pragma unroll
                    for (int j = 0; j < K; ++j) {
                        if (sp[tb + j * 32 + lane] < 0) continue;
                        const double dv = sd[tb + j * 32 + lane];
                        double L[NK];
                        legendre<NK>(fma(jb + (double)j, step, -1.0), L);
                        int q = NK;
#pragma unroll
                        for (int r = 0; r < NK; ++r) {
                            acc[r] = fma(L[r], dv, acc[r]);
#pragma unroll
                            for (int l = r; l < NK; ++l) { acc[q] = fma(L[r], L[l], acc[q]); ++q; }
                        }
                    }
                }
                block_sum_n<NR, NW>(acc, red, tot);
                if (threadIdx.x == 0) {
                    double cc[NK];
                    s_refine = filter_refine_steps(gram_solve<NK>(tot + NK, tot, cc));
#pragma unroll
                    for (int r = 0; r < NK; ++r) coef[r] = cc[r];
                }
                __syncthreads();
                const int nref = s_refine;
                for (int it = 0; it < nref; ++it) {
                    double cc[NK], racc[NK];
#pragma unroll
                    for (int r = 0; r < NK; ++r) { cc[r] = coef[r]; racc[r] = 0.0; }
                    for (int64_t tile = tile0 + warp; tile < tile1; tile += NW) {
                        const int64_t t0 = tile * TILE + (int64_t)lane * K;
                        const int tb = (int)(tile * TILE - base);
                        const double jb = (double)((int)(t0 - a) - j0);
#pragma unroll
                        for (int j = 0; j < K; ++j) {
                            if (sp[tb + j * 32 + lane] < 0) continue;
                            double L[NK];
                            legendre<NK>(fma(jb + (double)j, step, -1.0), L);
                            double res = sd[tb + j * 32 + lane];
#pragma unroll
                            for (int r = 0; r < NK; ++r) res = fma(-cc[r], L[r], res);
#pragma unroll
                            for (int r = 0; r < NK; ++r) racc[r] = fma(L[r], res, racc[r]);
                        }
                    }
                    block_sum_n<NK, NW>(racc, red, tot);
                    if (threadIdx.x == 0) {
                        double dc[NK];
                        gram_solve<NK>(tot + NK, tot, dc);
#pragma unroll
                        for (int r = 0; r < NK; ++r) coef[r] += dc[r];
                    }
                    __syncthreads();
                }
            }
            // ---- pass 2: scatter-add of d - sum_k c_k L_k over the unflagged samples
            double cf[NK];
#pragma unroll
            for (int r = 0; r < NK; ++r) cf[r] = coef[r];
            for (int64_t tile = tile0 + warp; tile < tile1; tile += NW) {
                const int64_t t0 = tile * TILE + (int64_t)lane * K;
                const int tb = (int)(tile * TILE - base);
                const double jb = (double)((int)(t0 - a) - j0);
                int p[K];
                double c[K], s[K], v[K];
#pragma unroll
                for (int j = 0; j < K; ++j) p[j] = sp[tb + j * 32 + lane];
                if (POL > 1) { load_f64(cs, t0, nt, c); load_f64(sn, t0, nt, s); }
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    double L[NK];
                    legendre<NK>(fma(jb + (double)j, step, -1.0), L);
                    double pj = 0.0;
#pragma unroll
                    for (int r = 0; r < NK; ++r) pj = fma(cf[r], L[r], pj);
                    v[j] = sd[tb + j * 32 + lane] - pj;
                }
                run_scatter<POL, POL>(y, p, pt_contrib<POL>(v, c, s));
            }
        }
        __syncthreads();
    }
}

// CTAs of BLOCK / 32 warp tiles that cover nt samples, `tile` of them per warp tile
static int64_t tod_blocks(int64_t nt, int64_t tile = TILE) {
    const int64_t ntiles = (nt + tile - 1) / tile;
    return (ntiles + (BLOCK / 32) - 1) / (BLOCK / 32);
}

// launch of a persistent kernel over `blocks` CTAs of work; a dynamic shared-memory size is also set as its limit
template <class... Params, class... Args>
static int launch_tod(void (*kern)(Params...), int64_t blocks, size_t smem, cudaStream_t st, Args... args) {
    if (smem > 0) CM2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return launch(kern, persistent_grid(kern, BLOCK, smem, blocks), BLOCK, smem, st, args...);
}

static int check_tod(const void *pix, const void *c, const void *s, int64_t nt, int pol) {
    if (nt < 0) return set_error(CM2_ERR_ARG, "nt < 0");
    if (pol < 1 || pol > 3) return set_error(CM2_ERR_ARG, "No valid polarization key set! pol=%d (1=I, 2=QU, 3=IQU)", pol);
    if (nt > 0 && pix == nullptr) return set_error(CM2_ERR_ARG, "pix is NULL");
    if (pol > 1 && nt > 0 && (c == nullptr || s == nullptr)) return set_error(CM2_ERR_ARG, "cos/sin required for pol>1");
    if (!aligned(pix, 32) || !aligned(c, 32) || !aligned(s, 32))
        return set_error(CM2_ERR_ARG, "TOD arrays must be 32-byte aligned");
    return CM2_OK;
}

}  // namespace cm2

using namespace cm2;

extern "C" int cm2_pointing_apply(const int32_t *pix, const double *c, const double *s, int64_t nt, int pol,
                                  const double *x, double *d, cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    CM2_REQUIRE(aligned(d, 32), "d must be 32-byte aligned");
    if (nt == 0) return CM2_OK;
    cudaStream_t st = as_stream(stream);
    return with_pol(pol, [&](auto P) { return launch_tod(k_pointing_apply<P>, tod_blocks(nt), 0, st, pix, c, s, nt, x, d); });
}

extern "C" int cm2_pointing_apply_t(const int32_t *pix, const double *c, const double *s, int64_t nt, int pol,
                                    const double *d, double *y, int64_t npix, cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    CM2_REQUIRE(aligned(d, 32), "d must be 32-byte aligned");
    CM2_REQUIRE(npix >= 0, "npix < 0");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(y, npix, pol, st));
    if (nt == 0 || npix == 0) return CM2_OK;
    return with_pol(pol, [&](auto P) { return launch_tod(k_pointing_apply_t<P>, tod_blocks(nt), 0, st, pix, c, s, nt, d, y); });
}

static int check_blocks(const double *wblk, int64_t nblocks, int64_t blocksize, const int64_t *blk_start) {
    if (wblk == nullptr) return CM2_OK;
    if (nblocks <= 0) return set_error(CM2_ERR_ARG, "nblocks must be > 0 when weights are given");
    if (blk_start == nullptr && blocksize <= 0) return set_error(CM2_ERR_ARG, "blocksize must be > 0");
    return CM2_OK;
}

static int g_white_stage_wpix = 0;

/* > 0 selects the shared-memory-staged scatter of the fused white A-matvec with a window of that many pixels
 * per warp tile (pixels crossed in 2..6 samples; tools/pattern_probe.py) */
extern "C" int cm2_amatvec_white_set_stage(int wpix) {
    CM2_REQUIRE(wpix >= 0 && wpix <= 1024, "stage window must be 0..1024 pixels");
    g_white_stage_wpix = wpix;
    return CM2_OK;
}

extern "C" int cm2_amatvec_white(const int32_t *pix, const uint64_t *pix_packed, const double *c, const double *s,
                                 int64_t nt, int pol, const double *wblk, int64_t nblocks, int64_t blocksize,
                                 const int64_t *blk_start, const double *x, double *y, int64_t npix, int64_t nstreams,
                                 cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    rc = check_blocks(wblk, nblocks, blocksize, blk_start);
    if (rc) return rc;
    CM2_REQUIRE(npix >= 0, "npix < 0");
    CM2_REQUIRE(aligned(pix_packed, 8), "pix_packed must be 8-byte aligned");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(y, npix, pol, st));
    if (nt == 0 || npix == 0) return CM2_OK;
    const BlockW bw = make_blockw(wblk, nblocks, blocksize, blk_start);
    const TileOrder ord = make_order(nt, nstreams);
    if (g_white_stage_wpix > 0) {
        CM2_REQUIRE(pix_packed == nullptr, "the staged scatter reads int32 pixels only");
        const int wpix = g_white_stage_wpix;
        const size_t smem = sizeof(double) * (size_t)(BLOCK / 32) * pol * wpix;
        return with_pol(pol, [&](auto P) {
            return launch_tod(k_amatvec_white_staged<P>, tod_blocks(nt), smem, st, pix, c, s, nt, bw, ord, x, y, wpix);
        });
    }
    if (wblk != nullptr && blk_start == nullptr && blocksize == 1) {      // one weight per sample, streamed
        CM2_REQUIRE(nblocks >= nt && aligned(wblk, 32), "per-sample weights: nt values, 32-byte aligned");
        CM2_REQUIRE(pix_packed == nullptr, "per-sample weights read int32 pixels only");
        return with_pol(pol, [&](auto P) {
            return launch_tod(k_amatvec_white<P, false, true>, tod_blocks(nt), 0, st, pix, c, s, nt, bw, ord, x, y,
                              (const uint64_t *)nullptr);
        });
    }
    return with_pol(pol, [&](auto P) {
        auto kern = ord.S > 1 ? (pix_packed ? k_amatvec_white<P, true, false, true> : k_amatvec_white<P, true>)
                              : (pix_packed ? k_amatvec_white<P, false, false, true> : k_amatvec_white<P, false>);
        return launch_tod(kern, tod_blocks(nt), 0, st, pix, c, s, nt, bw, ord, x, y, pix_packed);
    });
}

/* the packed pixel stream of pix (format at PK_ESCAPE) and its number of escape lanes */
extern "C" int cm2_pack_pointing(const int32_t *pix, int64_t nt, uint64_t *packed, int64_t *nescape, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0, "nt < 0");
    CM2_REQUIRE(nescape != nullptr && (nt == 0 || (pix != nullptr && packed != nullptr)), "NULL argument");
    CM2_REQUIRE(aligned(pix, 32) && aligned(packed, 8), "pix must be 32-byte and packed 8-byte aligned");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(nescape, 1, 1, st));
    if (nt == 0) return CM2_OK;
    return launch_tod(k_pack_pointing, tod_blocks(nt), 0, st, pix, nt, packed, reinterpret_cast<unsigned long long *>(nescape));
}

template <int POL, int NLAG>
static int launch_amatvec_toeplitz(const int32_t *pix, const double *c, const double *s, int64_t nt, const ToepW &tw,
                                   const double *x, double *y, cudaStream_t st) {
    constexpr int VAL = TILE - 2 * ((NLAG + K - 1) / K) * K;
    return launch_tod(k_amatvec_toeplitz<POL, NLAG>, tod_blocks(nt, VAL), 0, st, pix, c, s, nt, tw, x, y);
}

template <int POL>
static int dispatch_amatvec_toeplitz(const int32_t *pix, const double *c, const double *s, int64_t nt, const ToepW &tw,
                                     const double *x, double *y, cudaStream_t st) {
    const int nlag = tw.nband - 1;
    if (nlag <= 2) return launch_amatvec_toeplitz<POL, 2>(pix, c, s, nt, tw, x, y, st);
    if (nlag <= 4) return launch_amatvec_toeplitz<POL, 4>(pix, c, s, nt, tw, x, y, st);
    return launch_amatvec_toeplitz<POL, 8>(pix, c, s, nt, tw, x, y, st);
}

extern "C" int cm2_amatvec_toeplitz_max_band(void) { return 9; }

extern "C" int cm2_amatvec_toeplitz(const int32_t *pix, const double *c, const double *s, int64_t nt, int pol,
                                    const double *band, int nband, int64_t nblocks, int64_t blocksize,
                                    const int64_t *blk_start, const double *x, double *y, int64_t npix,
                                    cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    CM2_REQUIRE(band != nullptr && nband >= 1, "band required");
    rc = check_blocks(band, nblocks, blocksize, blk_start);
    if (rc) return rc;
    CM2_REQUIRE(blk_start != nullptr || nblocks - 1 <= nt / blocksize, "equal blocks past nt: (nblocks-1)*blocksize > nt");
    if (nband >cm2_amatvec_toeplitz_max_band())
        return set_error(CM2_ERR_UNSUPPORTED, "fused Toeplitz A-matvec: nband=%d, bands of up to %d coefficients are supported",
                         nband, cm2_amatvec_toeplitz_max_band());
    CM2_REQUIRE(npix >= 0, "npix < 0");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(y, npix, pol, st));
    if (nt == 0 || npix == 0) return CM2_OK;
    const ToepW tw{band, nband, make_blockw(nullptr, nblocks, blocksize, blk_start)};
    return with_pol(pol, [&](auto P) { return dispatch_amatvec_toeplitz<P>(pix, c, s, nt, tw, x, y, st); });
}

extern "C" int cm2_weights_moments(const int32_t *pix, const double *c, const double *s, const double *w,
                                   const double *wblk, int64_t nblocks, int64_t blocksize, const int64_t *blk_start,
                                   int64_t nt, int pol, double *mom, int64_t npix, cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    rc = check_blocks(wblk, nblocks, blocksize, blk_start);
    if (rc) return rc;
    CM2_REQUIRE(aligned(w, 32), "w must be 32-byte aligned");
    CM2_REQUIRE(npix >= 0, "npix < 0");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(mom, npix, 6, st));
    if (nt == 0 || npix == 0) return CM2_OK;
    const BlockW bw = make_blockw(wblk, nblocks, blocksize, blk_start);
    return with_pol(pol, [&](auto P) { return launch_tod(k_moments<P>, tod_blocks(nt), 0, st, pix, c, s, w, bw, nt, mom); });
}

extern "C" int cm2_hits_i64(const int32_t *pix, int64_t nt, int64_t npix, int64_t *hits, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0 && npix >= 0, "negative size");
    CM2_REQUIRE(aligned(pix, 32), "pix must be 32-byte aligned");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(hits, npix, 1, st));
    if (nt == 0 || npix == 0) return CM2_OK;
    return launch_tod(k_hits, tod_blocks(nt), 0, st, pix, nt, reinterpret_cast<unsigned long long *>(hits));
}

extern "C" int cm2_amatvec_filter(const int32_t *pix, const double *c, const double *s, int64_t nt, int pol,
                                  const int64_t *seg_start, const int64_t *seg_end, int64_t nseg, const double *x,
                                  double *y, int64_t npix, cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    CM2_REQUIRE(npix >= 0 && nseg >= 0, "negative size");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(y, npix, pol, st));
    if (nt == 0 || npix == 0 || nseg == 0) return CM2_OK;
    const size_t smem = sizeof(double) * SEG_SMEM;
    return with_pol(pol, [&](auto P) {
        return launch_tod(k_amatvec_filter<P>, nseg, smem, st, pix, c, s, nt, seg_start, seg_end, nseg, x, y);
    });
}

extern "C" int cm2_amatvec_filter_mu(const int32_t *pix, const double *c, const double *s, int64_t nt, int pol,
                                     const int64_t *seg_start, const int64_t *seg_end, const double *seg_mu,
                                     const int32_t *tile_seg, const uint8_t *tile_flag, int64_t nseg, const double *x,
                                     double *y, int64_t npix, int64_t nstreams, cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    CM2_REQUIRE(npix >= 0 && nseg >= 0, "negative size");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(y, npix, pol, st));
    if (nt == 0 || npix == 0 || nseg == 0) return CM2_OK;
    SegInfo sg{seg_start, seg_end, seg_mu, tile_seg, tile_flag, nseg};
    const TileOrder ord = make_order(nt, nstreams);
    return with_pol(pol, [&](auto P) {
        return launch_tod(k_amatvec_filter_mu<P>, tod_blocks(nt), 0, st, pix, c, s, nt, sg, ord, x, y);
    });
}

extern "C" int cm2_pointing_filter_mu(const int32_t *pix, const double *c, const double *s, int64_t nt, int pol,
                                      const int64_t *seg_start, const int64_t *seg_end, const double *seg_mu,
                                      const int32_t *tile_seg, const uint8_t *tile_flag, int64_t nseg, const double *x,
                                      double *d, cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    CM2_REQUIRE(nseg >= 0, "negative size");
    CM2_REQUIRE(aligned(d, 32), "d must be 32-byte aligned");
    if (nt == 0) return CM2_OK;
    cudaStream_t st = as_stream(stream);
    if (nseg == 0) {
        CM2_CUDA(zero_fill(d, nt, 1, st));
        return CM2_OK;
    }
    SegInfo sg{seg_start, seg_end, seg_mu, tile_seg, tile_flag, nseg};
    return with_pol(pol, [&](auto P) { return launch_tod(k_pointing_filter_mu<P>, tod_blocks(nt), 0, st, pix, c, s, nt, sg, x, d); });
}

/* single-TOD-pass P^T F_K P given the per-subscan Legendre coefficients (cm2_filter_poly_seg_coef);
 * accumulate != 0 adds to y instead of overwriting it */
extern "C" int cm2_amatvec_filter_poly_mu(const int32_t *pix, const double *c, const double *s, int64_t nt, int pol,
                                          const int64_t *seg_start, const int64_t *seg_end, const double *seg_coef,
                                          const int32_t *tile_seg, const uint8_t *tile_flag, int64_t nseg, int poly_order,
                                          const double *x, double *y, int64_t npix, int accumulate, int64_t nstreams,
                                          cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    CM2_REQUIRE(npix >= 0 && nseg >= 0, "negative size");
    if (poly_order < 1 || poly_order > 4)
        return set_error(CM2_ERR_UNSUPPORTED, "run-table Legendre A-matvec: poly_order=%d, orders 1..4 are supported", poly_order);
    cudaStream_t st = as_stream(stream);
    if (!accumulate) CM2_CUDA(zero_fill(y, npix, pol, st));
    if (nt == 0 || npix == 0 || nseg == 0) return CM2_OK;
    SegPoly sg{seg_start, seg_end, seg_coef, tile_seg, tile_flag, nseg};
    const int nk = poly_order + 1;
    const TileOrder ord = make_order(nt, nstreams);
    return with_pol(pol, [&](auto P) {
        return with_nk(nk, [&](auto NK) {
            return launch_tod(k_amatvec_filter_poly_mu<P, NK>, tod_blocks(nt), 0, st, pix, c, s, nt, sg, ord, x, y);
        });
    });
}

/* fused P^T F_K P, Legendre subscan filter of order 1..4 */
extern "C" int cm2_amatvec_filter_poly_max_order(void) { return 4; }

extern "C" int cm2_amatvec_filter_poly(const int32_t *pix, const double *c, const double *s, int64_t nt, int pol,
                                       const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                                       int64_t max_seg_len, int poly_order, const double *x, double *y, int64_t npix,
                                       cm2_stream_t stream) {
    int rc = check_tod(pix, c, s, nt, pol);
    if (rc) return rc;
    CM2_REQUIRE(npix >= 0 && nseg >= 0 && max_seg_len >= 0, "negative size");
    if (poly_order < 1 || poly_order > 4)
        return set_error(CM2_ERR_UNSUPPORTED, "fused Legendre A-matvec: poly_order=%d, orders 1..4 are supported", poly_order);
    // window: every tile the longest subscan can touch
    const int64_t cap = (max_seg_len / TILE + 2) * TILE;
    if (cap * 12 > 200 * 1024)
        return set_error(CM2_ERR_UNSUPPORTED, "fused Legendre A-matvec: subscan of %lld samples exceeds the shared-memory window",
                         (long long)max_seg_len);
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(y, npix, pol, st));
    if (nt == 0 || npix == 0 || nseg == 0) return CM2_OK;
    const int nk = poly_order + 1;
    return with_pol(pol, [&](auto P) {
        return with_nk(nk, [&](auto NK) {
            return launch_tod(k_amatvec_filter_poly<P, NK>, nseg, (size_t)cap * 12, st, pix, c, s, nt, seg_start, seg_end,
                              nseg, x, y, (int)cap);
        });
    });
}
