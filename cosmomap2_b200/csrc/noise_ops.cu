// cosmomap2_b200 -- time-domain noise operators N^-1 and the subscan offset filter F (sm_100a).
//
//   cm2_noise_white_apply     per-block scalar weight        (linearoperators.py:676-683, 606-617)
//   cm2_noise_toeplitz_apply  banded symmetric Toeplitz/block (ToeplitzLO.mult :582-595)
//   cm2_filter_offset_apply   subscan offset removal          (FilterLO.mult :129-168)
#include "cm2_common.cuh"

namespace cm2 {

constexpr int NB = 256;

__device__ __forceinline__ int64_t find_block(const int64_t *__restrict__ start, int64_t nblocks, int64_t blocksize, int64_t t) {
    if (start == nullptr) {
        int64_t b = t / blocksize;
        return b < nblocks ? b : nblocks - 1;
    }
    return last_le(start, nblocks, t);
}

// each thread: 4 consecutive samples (256-bit load/store); the block index is looked up once
__global__ void __launch_bounds__(NB) k_white(const double *__restrict__ w, int64_t nblocks, int64_t blocksize,
                                              const int64_t *__restrict__ start, const double *__restrict__ d,
                                              double *__restrict__ out, int64_t nt) {
    const int64_t nchunk = (nt + 3) / 4;
    for (int64_t ch = (int64_t)blockIdx.x * NB + threadIdx.x; ch < nchunk; ch += (int64_t)gridDim.x * NB) {
        const int64_t t0 = ch * 4;
        const int64_t b0 = find_block(start, nblocks, blocksize, t0);
        const int64_t bend = start ? start[b0 + 1] : (b0 + 1) * blocksize;
        if (t0 + 4 <= nt && t0 + 4 <= bend) {
            const double wb = __ldg(w + b0);
            D4 v = ld_stream_d4(d + t0);
#pragma unroll
            for (int j = 0; j < 4; ++j) v.v[j] *= wb;
            st_stream_d4(out + t0, v);
        } else {
            for (int j = 0; j < 4 && t0 + j < nt; ++j) {
                const int64_t b = find_block(start, nblocks, blocksize, t0 + j);
                out[t0 + j] = __ldg(w + b) * d[t0 + j];
            }
        }
    }
}

// ---- banded Toeplitz ---------------------------------------------------------------------------
// One CTA computes TT consecutive outputs of one noise block.  The input window
// [j0-(L-1), j0+TT+(L-1)) (zero outside the block: the reference's non-circulant boundary) and
// the band a[0..L) are staged in shared memory; each thread owns R consecutive outputs and slides
// two register windows over the lags, so one lag costs 2 shared loads + 1 broadcast for 2R flops.
//   y_j = a_0 v_j + sum_{k=1}^{L-1} a_k (v_{j-k} + v_{j+k})
constexpr int TR = 4;                    // outputs per thread
constexpr int TT = NB * TR;              // outputs per CTA tile (1024)

__global__ void __launch_bounds__(NB) k_toeplitz(const double *__restrict__ band, int L, int64_t nblocks, int64_t blocksize,
                                                 const int64_t *__restrict__ start, const int64_t *__restrict__ tile_first,
                                                 const double *__restrict__ d, double *__restrict__ out, int64_t nt) {
    extern __shared__ double sm[];
    double *sa = sm;            // L band values
    double *sv = sm + L;        // TT + 2(L-1) window
    const int H = L - 1;
    const int64_t ntiles = tile_first[nblocks];
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        // tile -> (block b, offset within block): tile_first[b] = first tile index of block b
        const int64_t b = last_le(tile_first, nblocks, tile);
        const int64_t bs = start ? start[b] : b * blocksize;
        const int64_t be = start ? start[b + 1] : (b + 1 == nblocks ? nt : (b + 1) * blocksize);
        const int64_t j0 = bs + (tile - tile_first[b]) * TT;   // first output of this tile (global index)
        __syncthreads();
        for (int k = threadIdx.x; k < L; k += NB) sa[k] = band[(int64_t)b * L + k];
        const int W = TT + 2 * H;
        for (int i = threadIdx.x; i < W; i += NB) {
            const int64_t t = j0 - H + i;
            sv[i] = (t >= bs && t < be) ? d[t] : 0.0;
        }
        __syncthreads();
        const int o0 = threadIdx.x * TR;        // first output of this thread within the tile
        double acc[TR], lw[TR], rw[TR];
#pragma unroll
        for (int r = 0; r < TR; ++r) {
            const double v = sv[H + o0 + r];
            acc[r] = sa[0] * v;
            lw[r] = v;   // window of v_{j-k}, k = 0
            rw[r] = v;   // window of v_{j+k}, k = 0
        }
        for (int k = 1; k < L; ++k) {
            // slide: left window moves one sample down, right window one sample up
#pragma unroll
            for (int r = TR - 1; r > 0; --r) lw[r] = lw[r - 1];
            lw[0] = sv[H + o0 - k];
#pragma unroll
            for (int r = 0; r < TR - 1; ++r) rw[r] = rw[r + 1];
            rw[TR - 1] = sv[H + o0 + TR - 1 + k];
            const double ak = sa[k];
#pragma unroll
            for (int r = 0; r < TR; ++r) acc[r] = fma(ak, lw[r] + rw[r], acc[r]);
        }
#pragma unroll
        for (int r = 0; r < TR; ++r) {
            const int64_t t = j0 + o0 + r;
            if (t < be) out[t] = acc[r];
        }
    }
}

__global__ void k_tile_first(int64_t nblocks, int64_t blocksize, const int64_t *__restrict__ start, int64_t nt,
                             int64_t *__restrict__ tile_first) {
    // single thread: prefix of per-block tile counts (nblocks is small: detectors x CES)
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int64_t acc = 0;
        for (int64_t b = 0; b < nblocks; ++b) {
            tile_first[b] = acc;
            const int64_t bs = start ? start[b] : b * blocksize;
            const int64_t be = start ? start[b + 1] : (b + 1 == nblocks ? nt : (b + 1) * blocksize);
            acc += (be - bs + TT - 1) / TT;
        }
        tile_first[nblocks] = acc;
    }
}

// ---- subscan offset filter -----------------------------------------------------------------------
// one CTA per segment: masked mean (deterministic tree), then out = d - mean over the segment
__global__ void __launch_bounds__(NB) k_filter_offset(const int32_t *__restrict__ pix, const int64_t *__restrict__ seg_start,
                                                      const int64_t *__restrict__ seg_end, int64_t nseg,
                                                      const double *__restrict__ d, double *__restrict__ out) {
    __shared__ double red[32];
    __shared__ double s_mean;
    __shared__ int s_skip;
    for (int64_t k = blockIdx.x; k < nseg; k += gridDim.x) {
        const int64_t a = seg_start[k], b = seg_end[k];
        double sum = 0.0, cnt = 0.0;
        for (int64_t t = a + threadIdx.x; t < b; t += NB) {
            if (pix[t] != -1) { sum += d[t]; cnt += 1.0; }
        }
        const double tsum = block_sum(sum, red);
        const double tcnt = block_sum(cnt, red);
        if (threadIdx.x == 0) {
            s_skip = !(tcnt > 0.0);
            s_mean = tcnt > 0.0 ? tsum / tcnt : 0.0;
            if (isinf(s_mean) || isnan(s_mean)) s_skip = 1;
        }
        __syncthreads();
        if (!s_skip) {
            const double mu = s_mean;
            for (int64_t t = a + threadIdx.x; t < b; t += NB) out[t] = d[t] - mu;
        }
        __syncthreads();
    }
}

}  // namespace cm2

using namespace cm2;

extern "C" int cm2_noise_white_apply(const double *wblk, int64_t nblocks, int64_t blocksize, const int64_t *blk_start,
                                     const double *d, double *out, int64_t nt, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0 && nblocks > 0, "bad sizes");
    CM2_REQUIRE(blk_start != nullptr || blocksize > 0, "blocksize must be > 0");
    CM2_REQUIRE(aligned(d, 32) && aligned(out, 32), "TOD vectors must be 32-byte aligned");
    if (nt == 0) return CM2_OK;
    return launch(k_white, capped_grid(cdiv(cdiv(nt, 4), NB), 8), NB, 0, as_stream(stream), wblk, nblocks, blocksize,
                  blk_start, d, out, nt);
}

extern "C" int64_t cm2_toeplitz_scratch_bytes(int64_t nblocks) { return (nblocks + 1) * (int64_t)sizeof(int64_t); }

extern "C" int cm2_noise_toeplitz_apply(const double *band, int nband, int64_t nblocks, int64_t blocksize,
                                        const int64_t *blk_start, const double *d, double *out, int64_t nt,
                                        void *scratch, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0 && nblocks > 0 && nband >= 1, "bad sizes");
    CM2_REQUIRE(blk_start != nullptr || blocksize > 0, "blocksize must be > 0");
    CM2_REQUIRE(blk_start != nullptr || nblocks - 1 <= nt / blocksize, "equal blocks past nt: (nblocks-1)*blocksize > nt");
    CM2_REQUIRE(scratch != nullptr, "scratch (cm2_toeplitz_scratch_bytes) required");
    CM2_REQUIRE(d != out, "in-place Toeplitz apply is not supported");
    if (nt == 0) return CM2_OK;
    const size_t smem = sizeof(double) * ((size_t)nband + TT + 2 * (size_t)(nband - 1));
    if (smem > 227 * 1024)
        return set_error(CM2_ERR_UNSUPPORTED, "Toeplitz band of %d lags needs %zu B of shared memory (max 227 kB)", nband, smem);
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(cudaFuncSetAttribute(k_toeplitz, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t *tile_first = reinterpret_cast<int64_t *>(scratch);
    k_tile_first<<<1, 1, 0, st>>>(nblocks, blocksize, blk_start, nt, tile_first);
    CM2_LAUNCHED();
    // upper bound of the tile count without reading the device prefix back
    const int64_t ntiles_ub = nt / TT + nblocks + 1;
    // the exact tile count is tile_first[nblocks], read on the device; at NB threads no more than 8 CTAs fit on an SM
    return launch(k_toeplitz, persistent_grid(k_toeplitz, NB, smem, ntiles_ub), NB, smem, st, band, nband, nblocks,
                  blocksize, blk_start, tile_first, d, out, nt);
}

extern "C" int cm2_filter_offset_apply(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                                       const double *d, double *out, int64_t nt, cm2_stream_t stream) {
    CM2_REQUIRE(nt >= 0 && nseg >= 0, "bad sizes");
    CM2_REQUIRE(d != out, "in-place filtering is not supported");
    cudaStream_t st = as_stream(stream);
    CM2_CUDA(zero_fill(out, nt, 1, st));
    if (nt == 0 || nseg == 0) return CM2_OK;
    return launch(k_filter_offset, capped_grid(nseg, 8), NB, 0, st, pix, seg_start, seg_end, nseg, d, out);
}
