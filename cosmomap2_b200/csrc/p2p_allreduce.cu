// cosmomap2_b200 -- map-domain all-reduce over NVLink peer memory (sm_100a, one process per GPU).
//
// After the local A-matvec every rank holds its own contribution y_g (npix*pol fp64, 12 MB at
// configs[1]).  One kernel per rank does the whole exchange over NVSwitch peer mappings:
//   1. start barrier (per CTA, flags in peer memory): every peer's y_g is complete;
//   2. rank r reduces ITS slice of the vector from all peers' buffers (peer loads, fixed rank order
//      -> deterministic, and every element is summed by exactly one rank, so all ranks end with
//      bit-identical q) and writes the sum straight into every peer's output buffer (peer stores);
//   3. end barrier: all slices of my output buffer have landed.
// Traffic per GPU: (G-1)/G * n * 8 B in and the same out, versus 2x that for a ring; latency is two
// flag round trips instead of NCCL's launch + protocol latency (the payload is small: the TOD stays
// local, only the pixel-domain vector is exchanged).
//
// Buffers and flags are torch CUDA allocations shared through CUDA IPC (torch plumbing); this file
// only sees pointer tables.  Spin waits carry a wall-clock timeout (%globaltimer, 20 s by default)
// and raise an error word instead of hanging the device.
#include "cm2_common.cuh"

namespace cm2 {

constexpr int AR_MAX_WORLD = 8;
constexpr int AR_MAX_BLOCKS = 148;
constexpr int AR_THREADS = 512;

struct ARSignals {
    unsigned int start[AR_MAX_BLOCKS][AR_MAX_WORLD];
    unsigned int end[AR_MAX_BLOCKS][AR_MAX_WORLD];
    unsigned int error;   // generation of the first wait that timed out (0 = none), sticky
    unsigned int abort;   // local: stop waiting
};

struct ARPtrs {
    const double *send[AR_MAX_WORLD];
    double *recv[AR_MAX_WORLD];
    ARSignals *sig[AR_MAX_WORLD];
};

__device__ __forceinline__ void st_flag(unsigned int *p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_flag(const unsigned int *p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ long long now_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// which = 0: start flags, 1: end flags.  Flags carry the generation of the call; the compare is
// monotone and wrap-safe (a flag that has already moved on to a later generation still satisfies the
// wait), and a wait that times out raises `error` (first generation that failed, sticky) and `abort`,
// which makes every later wait of this rank fall through at once: the rank never hangs and never
// spends more than one timeout in total; the host reads `error` (P2PAllReduce.error) and all ranks
// switch to NCCL together (distributed.py).
__device__ __forceinline__ void peer_barrier(const ARPtrs &P, int rank, int world, unsigned int gen, int which,
                                             long long timeout_ns) {
    __syncthreads();
    if ((int)threadIdx.x < world) {
        const int t = threadIdx.x;
        ARSignals *peer = P.sig[t];
        ARSignals *self = P.sig[rank];
        unsigned int *dst = which == 0 ? &peer->start[blockIdx.x][rank] : &peer->end[blockIdx.x][rank];
        const unsigned int *src = which == 0 ? &self->start[blockIdx.x][t] : &self->end[blockIdx.x][t];
        st_flag(dst, gen);
        if ((int)(ld_flag(src) - gen) < 0) {
            const long long t0 = now_ns();
            unsigned int polls = 0;
            while ((int)(ld_flag(src) - gen) < 0) {
                if ((++polls & 255u) != 0) continue;
                if (*((volatile unsigned int *)&self->abort) != 0) break;
                if (now_ns() - t0 > timeout_ns) {          // give up loudly instead of hanging
                    atomicCAS(&self->error, 0u, gen);
                    *((volatile unsigned int *)&self->abort) = 1u;
                    break;
                }
            }
        }
    }
    __syncthreads();
}

// WORLD and UNROLL are compile-time so that WORLD*UNROLL 16-byte peer loads per thread are in
// flight without spilling (NVLink load latency is ~2-3 us: the exchange is latency-bound unless
// enough loads are outstanding).
template <int WORLD, int UNROLL>
__global__ void __launch_bounds__(AR_THREADS) k_allreduce_p2p(ARPtrs P, int rank, int64_t n, unsigned int gen,
                                                                  long long timeout_ns) {
    peer_barrier(P, rank, WORLD, gen, 0, timeout_ns);
    const int64_t n2 = n / 2;   // my slice, in units of double2
    const int64_t lo = n2 * rank / WORLD, hi = n2 * (rank + 1) / WORLD;
    const int64_t stride = (int64_t)gridDim.x * AR_THREADS;
    for (int64_t i0 = lo + (int64_t)blockIdx.x * AR_THREADS + threadIdx.x; i0 < hi; i0 += stride * UNROLL) {
        double2 v[UNROLL][WORLD];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int64_t i = i0 + u * stride;
#pragma unroll
            for (int g = 0; g < WORLD; ++g)
                if (i < hi) v[u][g] = reinterpret_cast<const double2 *>(P.send[g])[i];
        }
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
            const int64_t i = i0 + u * stride;
            if (i < hi) {
                double2 s = v[u][0];
#pragma unroll
                for (int g = 1; g < WORLD; ++g) { s.x += v[u][g].x; s.y += v[u][g].y; }   // fixed rank order
#pragma unroll
                for (int g = 0; g < WORLD; ++g) reinterpret_cast<double2 *>(P.recv[g])[i] = s;
            }
        }
    }
    if ((n & 1) && rank == WORLD - 1 && blockIdx.x == 0 && threadIdx.x == 0) {   // odd tail element
        double s = 0.0;
        for (int g = 0; g < WORLD; ++g) s += P.send[g][n - 1];
        for (int g = 0; g < WORLD; ++g) P.recv[g][n - 1] = s;
    }
    __threadfence_system();
    peer_barrier(P, rank, WORLD, gen, 1, timeout_ns);
}

static long long g_ar_timeout_ns = 20000000000LL;   // 20 s

template <int WORLD, int UNROLL>
static void launch_ar(const ARPtrs &P, int rank, int64_t n, unsigned int gen, int grid, cudaStream_t st) {
    k_allreduce_p2p<WORLD, UNROLL><<<grid, AR_THREADS, 0, st>>>(P, rank, n, gen, g_ar_timeout_ns);
}

}  // namespace cm2

using namespace cm2;

/* timeout of the peer-flag waits in seconds (default 20); returns the previous value */
extern "C" double cm2_allreduce_p2p_set_timeout(double seconds) {
    const double old = 1e-9 * (double)g_ar_timeout_ns;
    if (seconds > 0.0) g_ar_timeout_ns = (long long)(seconds * 1e9);
    return old;
}

extern "C" int64_t cm2_allreduce_p2p_signal_bytes(void) { return (int64_t)sizeof(ARSignals); }

extern "C" int cm2_allreduce_p2p(const void *const *send_ptrs_host, void *const *recv_ptrs_host,
                                 void *const *signal_ptrs_host, int rank, int world, int64_t n, uint32_t generation,
                                 cm2_stream_t stream) {
    CM2_REQUIRE(world >= 1 && world <= AR_MAX_WORLD && rank >= 0 && rank < world, "bad rank/world");
    CM2_REQUIRE(n >= 0, "n < 0");
    CM2_REQUIRE(generation != 0, "generation must be non-zero");
    ARPtrs P;
    for (int g = 0; g < AR_MAX_WORLD; ++g) {
        P.send[g] = g < world ? reinterpret_cast<const double *>(send_ptrs_host[g]) : nullptr;
        P.recv[g] = g < world ? reinterpret_cast<double *>(recv_ptrs_host[g]) : nullptr;
        P.sig[g] = g < world ? reinterpret_cast<ARSignals *>(signal_ptrs_host[g]) : nullptr;
        if (g < world) CM2_REQUIRE(aligned(P.send[g], 16) && aligned(P.recv[g], 16), "buffers must be 16-byte aligned");
    }
    const int grid = capped_grid(cdiv(cdiv(n / 2, world), AR_THREADS), 1, AR_MAX_BLOCKS);
    // every rank must launch the SAME grid (per-CTA barriers): it depends only on n and world
    cudaStream_t st = as_stream(stream);
    switch (world) {
        case 1: launch_ar<1, 4>(P, rank, n, generation, grid, st); break;
        case 2: launch_ar<2, 8>(P, rank, n, generation, grid, st); break;
        case 3: launch_ar<3, 4>(P, rank, n, generation, grid, st); break;
        case 4: launch_ar<4, 4>(P, rank, n, generation, grid, st); break;
        case 5: launch_ar<5, 2>(P, rank, n, generation, grid, st); break;
        case 6: launch_ar<6, 2>(P, rank, n, generation, grid, st); break;
        case 7: launch_ar<7, 2>(P, rank, n, generation, grid, st); break;
        default: launch_ar<8, 2>(P, rank, n, generation, grid, st); break;
    }
    CM2_LAUNCHED();
    return CM2_OK;
}

extern "C" int cm2_enable_peer_access(int peer_device) {
    int dev = 0;
    CM2_CUDA(cudaGetDevice(&dev));
    if (peer_device == dev) return CM2_OK;
    int can = 0;
    CM2_CUDA(cudaDeviceCanAccessPeer(&can, dev, peer_device));
    if (!can) return set_error(CM2_ERR_UNSUPPORTED, "device %d cannot access peer %d", dev, peer_device);
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return CM2_OK;
    }
    CM2_CUDA(e);
    return CM2_OK;
}
