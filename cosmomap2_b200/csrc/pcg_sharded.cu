// cosmomap2_b200 -- the pixel-domain tail of an M_BD PCG iteration FUSED with the map exchange, over
// NVLink peer memory (sm_100a, one process per GPU).  SURVEY section 8(e): reduce-scatter -> pixel-
// sharded M_BD / CG work -> all-gather, as ONE kernel per iteration instead of all-reduce + replicated
// vector work.
//
// Every rank g holds its local A p in y_g (n doubles, written by the fused TOD kernel straight into
// this peer-visible buffer) and a full copy of the search direction p.  Rank g owns the pixel slice
// [pix_lo[g], pix_lo[g+1]) of x, r, z, q and of the M_BD blocks.  One launch of k_pcg_bd_sharded:
//
//   start barrier         every peer's y is complete (flags in peer memory)
//   phase 1 (my slice)    q = sum_g y_g  by peer LOADS in fixed rank order   (the reduce-scatter)
//                         partial p.q  -> exchange of one double per rank     (flag-guarded peer stores)
//   phase 2 (my slice)    alpha = rho / p.q ; x += alpha p ; r -= alpha q ; z = M_BD r
//                         partials r.z, |r|^2 -> exchange of two doubles per rank
//   phase 3 (my slice)    beta = rho'/rho ; p = z + beta p  written into EVERY rank's p by peer
//                         STORES                                              (the all-gather)
//   end barrier           all slices of my p have landed: the next TOD pass may read it
//
// SciPy's recurrence and exit rule (scipy/_isolve/iterative.py:405-431; call sites
// src/test_BD_precond_onto_real_data.py:47, src/test_M2_precond_onto_real_data.py:117) as in vecops.cu;
// the same 16-double scalar workspace, kept on every rank.  All ranks sum the per-rank partials in
// rank order, so alpha, beta, |r| and the `done` flag are bit-identical everywhere and no rank ever
// disagrees about stopping.  Within a rank the CTA partials are summed in CTA order by the last CTA
// to arrive (ticket), so there is no grid-wide barrier at all: the launch is cooperative only to
// guarantee that all CTAs are co-resident (they wait on flags written by each other).
//
// Flags carry a monotonically increasing generation and are compared wrap-safe with >=, so a rank that
// is late never misses a flag that has moved on.  Every wait has a timeout (wall clock, %globaltimer):
// the rank that times out raises `abort`, all its waits fall through, the kernel finishes (with
// garbage), marks the solve as failed in scal[9] and done in scal[7]; the host sees it in the scalar
// snapshot it reads anyway, all ranks agree on the failure over NCCL and redo the solve with the
// NCCL all-reduce (distributed.py).
//
// Emulation on ONE GPU (tests): nvirt = world virtual ranks in one cooperative launch, CTA group v
// acting as rank v on its own buffers -- the same code path, flags and all, without NVLink.
#include <cstring>

#include "cm2_common.cuh"

namespace cm2 {

constexpr int SH_MAX_WORLD = 8;
constexpr int SH_THREADS = 256;
constexpr int SH_MAXP = 1024;      // max CTAs per rank

struct ShardSignals {
    unsigned int start[2][SH_MAX_WORLD];        // [generation parity][source rank]
    unsigned int end[2][SH_MAX_WORLD];
    unsigned int sflag[2][2][SH_MAX_WORLD];     // [parity][exchange][source rank]
    double sval[2][2][SH_MAX_WORLD][2];
    unsigned int ticket[4];                     // local: CTAs of this rank that finished a phase
    unsigned int error;                         // generation of the first wait that timed out (0 = none)
    unsigned int abort;                         // local: a wait timed out, stop waiting
};

struct ShardArgs {
    // peer-visible, indexed by rank
    const double *y[SH_MAX_WORLD];
    double *p[SH_MAX_WORLD];
    ShardSignals *sig[SH_MAX_WORLD];
    // private to a rank (filled for the ranks this launch plays: one, or all when emulating)
    double *x[SH_MAX_WORLD], *r[SH_MAX_WORLD], *z[SH_MAX_WORLD], *q[SH_MAX_WORLD];
    const double *inv[SH_MAX_WORLD];            // M_BD blocks of the rank's pixel slice
    const double *b[SH_MAX_WORLD];              // reset: right-hand side, the rank's slice
    double *scal[SH_MAX_WORLD];
    double *part[SH_MAX_WORLD];                 // 2 * SH_MAXP doubles
    int64_t pix_lo[SH_MAX_WORLD + 1];
    int world, rank0, nvirt;
    unsigned int gen;
    double atol, rtol;
    long long timeout_ns;
};

__device__ __forceinline__ void sh_st_release(unsigned int *p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int sh_ld_acquire(const unsigned int *p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void sh_st_f64(double *p, double v) {
    asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ double sh_ld_f64(const double *p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ long long sh_now_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// wait until *flag has reached generation gen (wrap-safe); false if the wait was abandoned
__device__ __noinline__ bool sh_wait_ge(const unsigned int *flag, unsigned int gen, ShardSignals *me, long long timeout_ns) {
    if ((int)(sh_ld_acquire(flag) - gen) >= 0) return true;
    const long long t0 = sh_now_ns();
    unsigned int polls = 0;
    while ((int)(sh_ld_acquire(flag) - gen) < 0) {
        if ((++polls & 255u) == 0) {
            if (*((volatile unsigned int *)&me->abort) != 0) return false;
            if (sh_now_ns() - t0 > timeout_ns) {
                atomicCAS(&me->error, 0u, gen);
                *((volatile unsigned int *)&me->abort) = 1u;
                __threadfence();
                return false;
            }
        }
    }
    return true;
}

// Sum of NV per-CTA partials over the CTAs of this rank (CTA order, by the last CTA to arrive) and then
// over the ranks (rank order, by every CTA of every rank): bit-identical totals everywhere.
// v is valid in warp 0; tot is returned to all threads.  Block-wide: all threads must call.
template <int NV>
__device__ __forceinline__ void sh_exchange_sum(const ShardArgs &a, int rank, int cta, int cpr, int ex, const double (&v)[NV],
                                                double (&tot)[NV], double *red, double *sm) {
    __shared__ int s_last;
    ShardSignals *me = a.sig[rank];
    double *part = a.part[rank];
    const int par = a.gen & 1;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < NV; ++k) part[k * SH_MAXP + cta] = v[k];
        __threadfence();
        s_last = atomicAdd(&me->ticket[ex], 1u) == (unsigned)(cpr - 1);
    }
    __syncthreads();
    if (s_last) {                      // block-uniform
        __threadfence();
        double t[NV];
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            double s = 0.0;
            for (int i = threadIdx.x; i < cpr; i += SH_THREADS) s += ((volatile double *)part)[k * SH_MAXP + i];
            t[k] = block_sum(s, red);  // valid in all lanes of warp 0
        }
        if ((int)threadIdx.x < a.world) {
            ShardSignals *peer = a.sig[threadIdx.x];
#pragma unroll
            for (int k = 0; k < NV; ++k) sh_st_f64(&peer->sval[par][ex][rank][k], t[k]);
            sh_st_release(&peer->sflag[par][ex][rank], a.gen);
        }
        if (threadIdx.x == 0) me->ticket[ex] = 0;
    }
    if ((int)threadIdx.x < a.world) {
        sh_wait_ge(&me->sflag[par][ex][threadIdx.x], a.gen, me, a.timeout_ns);
#pragma unroll
        for (int k = 0; k < NV; ++k) sm[2 * threadIdx.x + k] = sh_ld_f64(&me->sval[par][ex][threadIdx.x][k]);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        double s = 0.0;
        for (int g = 0; g < a.world; ++g) s += sm[2 * g + k];
        tot[k] = s;
    }
    __syncthreads();
}

template <int POL, bool RESET>
__global__ void __launch_bounds__(SH_THREADS) k_pcg_bd_sharded(const ShardArgs a) {
    __shared__ double red[32];
    __shared__ double sm[2 * SH_MAX_WORLD];
    __shared__ int s_last_end;
    const int cpr = gridDim.x / a.nvirt;
    const int v = blockIdx.x / cpr, cta = blockIdx.x - v * cpr;
    const int rank = a.rank0 + v;
    double *scal = a.scal[rank];
    if (!RESET && scal[7] != 0.0) return;        // identical on every rank: nobody posts, nobody waits
    ShardSignals *me = a.sig[rank];
    const unsigned int gen = a.gen;
    const int par = gen & 1;
    const int64_t plo = a.pix_lo[rank], npl = a.pix_lo[rank + 1] - plo;
    const int64_t elo = POL * plo, ne = POL * npl, n2 = ne >> 1;
    const int64_t tid = (int64_t)cta * SH_THREADS + threadIdx.x, stride = (int64_t)cpr * SH_THREADS;
    double *x = a.x[rank], *r = a.r[rank], *z = a.z[rank], *q = a.q[rank];
    const double *inv = a.inv[rank];
    double *pme = a.p[rank] + elo;               // my slice of my copy of p (elo is even: 16-byte aligned)

    // ---- start barrier: every peer has finished the TOD pass that wrote its y ----------------------
    if (cta == 0 && (int)threadIdx.x < a.world) sh_st_release(&a.sig[threadIdx.x]->start[par][rank], gen);
    if ((int)threadIdx.x < a.world) sh_wait_ge(&me->start[par][threadIdx.x], gen, me, a.timeout_ns);
    __syncthreads();

    double rho = 0.0, alpha = 0.0, pq = 0.0;
    if constexpr (!RESET) {
        rho = scal[0];
        // ---- phase 1: q = sum over ranks of y (peer loads, fixed order), p.q --------------------------
        double s[1] = {0.0};
        constexpr int U = 2;
        for (int64_t i0 = tid; i0 < n2; i0 += stride * U) {
            double2 acc[U];
#pragma unroll
            for (int u = 0; u < U; ++u) acc[u] = make_double2(0.0, 0.0);
            double2 yv[U][SH_MAX_WORLD];
#pragma unroll
            for (int g = 0; g < SH_MAX_WORLD; ++g) {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int64_t i = i0 + u * stride;
                    if (g < a.world && i < n2) yv[u][g] = reinterpret_cast<const double2 *>(a.y[g] + elo)[i];
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t i = i0 + u * stride;
                if (i < n2) {
#pragma unroll
                    for (int g = 0; g < SH_MAX_WORLD; ++g)
                        if (g < a.world) { acc[u].x += yv[u][g].x; acc[u].y += yv[u][g].y; }
                    reinterpret_cast<double2 *>(q)[i] = acc[u];
                    const double2 pp = reinterpret_cast<const double2 *>(pme)[i];
                    s[0] = fma(pp.x, acc[u].x, s[0]);
                    s[0] = fma(pp.y, acc[u].y, s[0]);
                }
            }
        }
        if ((ne & 1) && tid == 0) {              // odd tail element (only the last rank can have one)
            double acc = 0.0;
            for (int g = 0; g < a.world; ++g) acc += a.y[g][elo + ne - 1];
            q[ne - 1] = acc;
            s[0] = fma(pme[ne - 1], acc, s[0]);
        }
        s[0] = block_sum(s[0], red);
        double tot[1];
        sh_exchange_sum<1>(a, rank, cta, cpr, 0, s, tot, red, sm);
        pq = tot[0];
        alpha = rho / pq;
    }

    // ---- phase 2: x, r, z = M_BD r on my pixels; r.z and |r|^2 --------------------------------------
    double s2[2] = {0.0, 0.0};
    for (int64_t j = tid; j < npl; j += stride) {
        double rv[POL], zv[POL];
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            const int64_t i = POL * j + k;
            if constexpr (RESET) {
                rv[k] = a.b[rank][i];
                x[i] = 0.0;
            } else {
                x[i] = fma(alpha, pme[i], x[i]);
                rv[k] = fma(-alpha, q[i], r[i]);
            }
            r[i] = rv[k];
        }
        bd_z<POL>(inv, j, rv, zv);
#pragma unroll
        for (int k = 0; k < POL; ++k) {
            z[POL * j + k] = zv[k];
            s2[0] = fma(rv[k], zv[k], s2[0]);
            s2[1] = fma(rv[k], rv[k], s2[1]);
        }
    }
    s2[0] = block_sum(s2[0], red);
    s2[1] = block_sum(s2[1], red);
    double tot2[2];
    sh_exchange_sum<2>(a, rank, cta, cpr, 1, s2, tot2, red, sm);
    const double rho_new = tot2[0], rr = tot2[1];
    const double beta = RESET ? 0.0 : rho_new / rho;

    // ---- phase 3: next search direction, written into every rank's p (peer stores) ------------------
    for (int64_t i = tid; i < n2; i += stride) {
        double2 zz = reinterpret_cast<const double2 *>(z)[i];
        if constexpr (!RESET) {
            const double2 pp = reinterpret_cast<const double2 *>(pme)[i];
            zz.x = fma(beta, pp.x, zz.x);
            zz.y = fma(beta, pp.y, zz.y);
        }
#pragma unroll
        for (int g = 0; g < SH_MAX_WORLD; ++g)
            if (g < a.world) reinterpret_cast<double2 *>(a.p[g] + elo)[i] = zz;
    }
    if ((ne & 1) && tid == 0) {
        double zz = z[ne - 1];
        if constexpr (!RESET) zz = fma(beta, pme[ne - 1], zz);
        for (int g = 0; g < a.world; ++g) a.p[g][elo + ne - 1] = zz;
    }
    // ---- end barrier: my stores have landed everywhere, and everybody's have landed here ------------
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last_end = atomicAdd(&me->ticket[2], 1u) == (unsigned)(cpr - 1);
    }
    __syncthreads();
    if (s_last_end) {
        __threadfence_system();
        if ((int)threadIdx.x < a.world) sh_st_release(&a.sig[threadIdx.x]->end[par][rank], gen);
        if (threadIdx.x == 0) me->ticket[2] = 0;
    }
    if ((int)threadIdx.x < a.world) sh_wait_ge(&me->end[par][threadIdx.x], gen, me, a.timeout_ns);
    __syncthreads();

    if (cta == 0 && threadIdx.x == 0) {
        const bool failed = *((volatile unsigned int *)&me->abort) != 0;
        if constexpr (RESET) {
            const double atol = fmax(a.atol, a.rtol * sqrt(rr));      // SciPy: atol = max(atol, rtol * ||b||)
            scal[0] = rho_new; scal[1] = 0.0; scal[2] = 0.0; scal[4] = 0.0; scal[5] = 0.0;
            scal[3] = rr;
            scal[6] = atol;
            scal[7] = (sqrt(rr) < atol || rr == 0.0 || failed) ? 1.0 : 0.0;   // b = 0: x = 0 is the answer
            scal[8] = 0.0;
            scal[9] = failed ? (double)me->error : 0.0;
            scal[10] = rr;                                            // ||b||^2 for the caller
        } else {
            scal[1] = rho;
            scal[0] = rho_new;
            scal[2] = pq;
            scal[3] = rr;
            scal[4] = alpha;
            scal[5] = beta;
            scal[8] += 1.0;
            scal[7] = (sqrt(rr) < scal[6] || failed) ? 1.0 : 0.0;
            if (failed) scal[9] = (double)me->error;
        }
    }
}

template <int POL, bool RESET>
static int launch_sharded(const ShardArgs &a, cudaStream_t st) {
    auto kern = k_pcg_bd_sharded<POL, RESET>;
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, SH_THREADS, 0);
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 4) per_sm = 4;
    int64_t total = (int64_t)sm_count() * per_sm;         // all CTAs co-resident
    int64_t cpr = total / a.nvirt;
    if (cpr > SH_MAXP) cpr = SH_MAXP;
    int64_t maxpix = 1;
    for (int v = 0; v < a.nvirt; ++v) {
        const int64_t np = a.pix_lo[a.rank0 + v + 1] - a.pix_lo[a.rank0 + v];
        if (np > maxpix) maxpix = np;
    }
    const int64_t need = (maxpix + SH_THREADS - 1) / SH_THREADS;
    if (need < cpr) cpr = need;
    if (cpr < 1) return set_error(CM2_ERR_UNSUPPORTED, "sharded PCG: %d virtual ranks do not fit on this device", a.nvirt);
    void *args[] = {(void *)&a};
    cudaError_t e = cudaLaunchCooperativeKernel((const void *)kern, dim3((unsigned)(cpr * a.nvirt)), dim3(SH_THREADS), args, 0, st);
    if (e != cudaSuccess) {
        cudaGetLastError();                               // do not leave the error for the next launch check
        return set_error(CM2_ERR_CUDA, "cm2_pcg_bd_sharded: %s", cudaGetErrorString(e));
    }
    count_launch();
    return CM2_OK;
}

}  // namespace cm2

using namespace cm2;

extern "C" int64_t cm2_pcg_sharded_signal_bytes(void) { return (int64_t)sizeof(ShardSignals); }
extern "C" int64_t cm2_pcg_sharded_work_doubles(void) { return 2 * SH_MAXP; }

// tables: HOST arrays with `world` entries of DEVICE pointers.  y/p/sig: every rank's peer-visible
// buffers (mapped into this process).  x/r/z/q/inv/b/scal/part: private buffers, entries
// [rank0, rank0 + nvirt) are used (nvirt = 1: a real rank; nvirt = world: one-GPU emulation).
extern "C" int cm2_pcg_bd_sharded(int reset, int pol, int world, int rank0, int nvirt, const int64_t *pix_lo_host,
                                  const void *const *y_tab, void *const *p_tab, void *const *sig_tab, void *const *x_tab,
                                  void *const *r_tab, void *const *z_tab, void *const *q_tab, const void *const *inv_tab,
                                  const void *const *b_tab, void *const *scal_tab, void *const *part_tab,
                                  uint32_t generation, double atol, double rtol, double timeout_s, cm2_stream_t stream) {
    CM2_REQUIRE(pol >= 1 && pol <= 3, "bad pol");
    CM2_REQUIRE(world >= 1 && world <= SH_MAX_WORLD, "world must be 1..8");
    CM2_REQUIRE(nvirt == 1 || (nvirt == world && rank0 == 0), "nvirt must be 1, or world with rank0 = 0");
    CM2_REQUIRE(rank0 >= 0 && rank0 + nvirt <= world, "bad rank");
    CM2_REQUIRE(generation != 0, "generation must be non-zero");
    ShardArgs a;
    memset(&a, 0, sizeof(a));
    for (int g = 0; g <= world; ++g) {
        a.pix_lo[g] = pix_lo_host[g];
        if (g > 0) CM2_REQUIRE(a.pix_lo[g] >= a.pix_lo[g - 1], "pix_lo must be non-decreasing");
        if (g < world) CM2_REQUIRE(((a.pix_lo[g] * pol) & 1) == 0, "slice offsets must be even (16-byte aligned)");
    }
    for (int g = 0; g < world; ++g) {
        a.y[g] = reinterpret_cast<const double *>(y_tab[g]);
        a.p[g] = reinterpret_cast<double *>(p_tab[g]);
        a.sig[g] = reinterpret_cast<ShardSignals *>(sig_tab[g]);
        CM2_REQUIRE(aligned(a.y[g], 16) && aligned(a.p[g], 16) && aligned(a.sig[g], 8), "peer buffers must be 16-byte aligned");
    }
    for (int g = rank0; g < rank0 + nvirt; ++g) {
        a.x[g] = reinterpret_cast<double *>(x_tab[g]);
        a.r[g] = reinterpret_cast<double *>(r_tab[g]);
        a.z[g] = reinterpret_cast<double *>(z_tab[g]);
        a.q[g] = reinterpret_cast<double *>(q_tab[g]);
        a.inv[g] = reinterpret_cast<const double *>(inv_tab[g]);
        a.b[g] = b_tab ? reinterpret_cast<const double *>(b_tab[g]) : nullptr;
        a.scal[g] = reinterpret_cast<double *>(scal_tab[g]);
        a.part[g] = reinterpret_cast<double *>(part_tab[g]);
        CM2_REQUIRE(aligned(a.z[g], 16) && aligned(a.q[g], 16) && aligned(a.inv[g], 16), "z, q and the M_BD blocks must be 16-byte aligned");
        if (reset) CM2_REQUIRE(a.b[g] != nullptr, "reset needs b");
    }
    a.world = world;
    a.rank0 = rank0;
    a.nvirt = nvirt;
    a.gen = generation;
    a.atol = atol;
    a.rtol = rtol;
    a.timeout_ns = (long long)(timeout_s * 1e9);
    cudaStream_t st = as_stream(stream);
    return with_pol(pol, [&](auto P) { return reset ? launch_sharded<P, true>(a, st) : launch_sharded<P, false>(a, st); });
}
