/*
 * cosmomap2_b200 -- C ABI of the B200-native map-making hot path.
 *
 * The reference (giuspugl/COSMOMAP2) has no C ABI: its inner loops are C++ snippets JIT-compiled
 * by weave.inline from Python.  Each entry point below replaces one of those loops (or the
 * NumPy/BLAS code next to it); the reference site is cited as file:line relative to the
 * reference tree.  INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every data pointer is a DEVICE pointer (HBM) unless the
 *     name ends in _host; the library never owns caller buffers;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on that stream;
 *   - return value: 0 = ok, negative = error (cm2_last_error() gives the text); nothing throws;
 *   - maps are interleaved per pixel ([I0,Q0,U0,I1,...] for pol=3, [Q0,U0,...] for pol=2),
 *     fp64; pixel indices are int32, -1 = flagged sample (skipped everywhere);
 *   - TOD vectors are CES-major, detector-major, time-minor (linearoperators.py:134-140).
 */
#ifndef COSMOMAP2_B200_H
#define COSMOMAP2_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CM2_OK 0
#define CM2_ERR_ARG (-1)
#define CM2_ERR_CUDA (-2)
#define CM2_ERR_UNSUPPORTED (-3)

typedef void *cm2_stream_t;

/* ---- library ------------------------------------------------------------------------- */
int cm2_version(void);
const char *cm2_last_error(void);
/* SM count, L2 bytes and compute capability (major*10+minor) of the current device */
int cm2_device_info(int *sm_count, int64_t *l2_bytes, int *cc);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
int64_t cm2_launch_count(void);

/* ---- a1/a2: pointing operator (interfaces/linearoperators.py:356-526) -------------------- */
/* d[t] = x[p] | x[2p]c+x[2p+1]s | x[3p]+x[3p+1]c+x[3p+2]s ; flagged -> 0   (:368-375,424-430,483-489) */
int cm2_pointing_apply(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                       int64_t nt, int pol, const double *x, double *d, cm2_stream_t stream);
/* y = P^T d, y zero-filled first (:394-401, 447-454, 509-517); warp-aggregated atomics */
int cm2_pointing_apply_t(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                         int64_t nt, int pol, const double *d, double *y, int64_t npix,
                         cm2_stream_t stream);
/* deterministic P^T d: samples visited in pixel-sorted order (perm = stable argsort of pix with
 * the flagged samples removed, rowptr[npix+1] = first entry of each pixel); one warp per pixel,
 * fixed summation order, no atomics */
int cm2_pointing_apply_t_sorted(const int64_t *rowptr, const int32_t *perm,
                                const double *cos2phi, const double *sin2phi, int pol,
                                const double *d, double *y, int64_t npix, cm2_stream_t stream);
/* integer hit counts, bit-exact (tests/test_matrix_vector_product.py:9-23) */
int cm2_hits_i64(const int32_t *pix, int64_t nt, int64_t npix, int64_t *hits,
                 cm2_stream_t stream);

/* ---- a6/a7: ProcessTimeSamples (utilities/process_ces.py:58-555) -------------------------- */
/* cos2phi = cos(2 phi), sin2phi = sin(2 phi)   (:493-494) */
int cm2_angles(const double *phi, int64_t nt, double *cos2phi, double *sin2phi,
               cm2_stream_t stream);
/* narrow caller pixels (int64 host convention) to the device int32 layout and back */
int cm2_pix_narrow(const int64_t *pix64, int64_t nt, int32_t *pix32, cm2_stream_t stream);
int cm2_pix_widen(const int32_t *pix32, int64_t nt, int64_t *pix64, cm2_stream_t stream);
/* weighted per-pixel moments, interleaved mom[npix][6] = {h, c, s, c2, cs, s2} (the upper
 * triangle of [[h,c,s],[c,c2,cs],[s,cs,s2]]); mom zero-filled first.  Weights: per-sample `w`
 * (the reference's w=N.diag), else per-block `wblk` as in cm2_noise_white_apply, else (both
 * NULL) unit weights   (:480-486, 505-513, 527-538, 125-189) */
int cm2_weights_moments(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                        const double *w, const double *wblk, int64_t nblocks, int64_t blocksize,
                        const int64_t *blk_start, int64_t nt, int pol, double *mom, int64_t npix,
                        cm2_stream_t stream);
/* the same moments in the reference's own summation order (one thread per pixel, samples in time
 * order through the stable pixel-sorted permutation, serial association, no FMA): bit-identical to
 * the serial loops on the same inputs.  rowptr[npix+1], perm[nvalid] as for
 * cm2_pointing_apply_t_sorted. */
int cm2_weights_moments_sorted(const int64_t *rowptr, const int32_t *perm, const double *cos2phi,
                               const double *sin2phi, const double *w, const double *wblk,
                               int64_t nblocks, int64_t blocksize, const int64_t *blk_start,
                               int pol, double *mom, int64_t npix, cm2_stream_t stream);
/* good-pixel flags (:491, 544-555): pol=1 h>0; pol=2 cond<=thr; pol=3 cond<=thr && h>2 */
int cm2_weights_mask(const double *mom, int64_t npix, int pol, double threshold_cond,
                     int32_t *good, cm2_stream_t stream);
/* exclusive scan of good[] -> old2new (-1 where dropped); *npix_new_dev receives the count.
 * scratch: at least cm2_scan_scratch_bytes(npix) bytes   (replaces the O(Nold*Nmask) search :192-349) */
int64_t cm2_scan_scratch_bytes(int64_t n);
int cm2_weights_old2new(const int32_t *good, int64_t npix, int32_t *old2new,
                        int64_t *npix_new_dev, void *scratch, cm2_stream_t stream);
/* compact per-pixel rows: dst[old2new[j]][0..width) = src[j][0..width) for kept j (fp64 rows) */
int cm2_compact_rows_f64(const double *src, const int32_t *old2new, int64_t npix, int width,
                         double *dst, cm2_stream_t stream);
int cm2_compact_rows_i64(const int64_t *src, const int32_t *old2new, int64_t npix, int width,
                         int64_t *dst, cm2_stream_t stream);
/* pix[t] = old2new[pix[t]] in place, flagged stay -1   (:411-417) */
int cm2_relabel(int32_t *pix, int64_t nt, const int32_t *old2new, cm2_stream_t stream);

/* ---- a8/a9: block-diagonal preconditioner (interfaces/linearoperators.py:700-859) --------- */
/* inv[npix][6] = upper triangle of the per-pixel inverse block (or zeros where masked:
 * pol=1 h<=0, pol=2/3 |det|<=1e-5), from mom[npix][6]   (:789-801, 820-826) */
int cm2_bd_build(const double *mom, int64_t npix, int pol, double *inv, cm2_stream_t stream);
/* y = M_BD x with the packed inverse blocks   (:796-806, 822-831) */
int cm2_bd_apply(const double *inv, int64_t npix, int pol, const double *x, double *y,
                 cm2_stream_t stream);
/* y = (P^T diag(N^-1) P) x, the forward per-pixel block   (:728-746) */
int cm2_bdfwd_apply(const double *mom, int64_t npix, int pol, const double *x, double *y,
                    cm2_stream_t stream);

/* ---- a3/a4/a5: noise operators ------------------------------------------------------------ */
/* Noise blocks (here, for the Toeplitz entry points below and cm2_amatvec_toeplitz):
 *  - blk_start == NULL: equal blocks, block b = [b*blocksize, (b+1)*blocksize) and the last block
 *    [(nblocks-1)*blocksize, nt), which also takes the remainder past nblocks*blocksize.  The Toeplitz
 *    entry points refuse (nblocks-1)*blocksize > nt with CM2_ERR_ARG.
 *  - else block b = [blk_start[b], blk_start[b+1]) with blk_start[0] = 0, blk_start non-decreasing
 *    and blk_start[nblocks] = nt; empty blocks are allowed.  This is not checked on the device.
 * white: out[t] = w[block(t)] * d[t]   (linearoperators.py:676-683, blkop.py:178-208,
 * WeightingLO :606-617).  in-place allowed (out == d). */
int cm2_noise_white_apply(const double *wblk, int64_t nblocks, int64_t blocksize,
                          const int64_t *blk_start, const double *d, double *out, int64_t nt,
                          cm2_stream_t stream);
/* banded symmetric Toeplitz per block, zero boundaries (ToeplitzLO.mult :582-595):
 * band[b*nband + k] = a_k of block b; blocks as above */
int64_t cm2_toeplitz_scratch_bytes(int64_t nblocks);
int cm2_noise_toeplitz_apply(const double *band, int nband, int64_t nblocks, int64_t blocksize,
                             const int64_t *blk_start, const double *d, double *out, int64_t nt,
                             void *scratch, cm2_stream_t stream);
/* same operator by overlap-save FFT in shared memory (for wide bands: 2(2 nband - 1) flop/sample of
 * the direct form become ~150).  coef[nblocks][2][M] complex fp64, M = cm2_toeplitz_fft_points():
 * the packed transfer function C1, C2 of each block's band, stored at the bit-reversed position of
 * each frequency (see csrc/toeplitz_fft.cu), built on the host.  Requires 2 (nband-1) < M.  scratch: cm2_toeplitz_fft_scratch_bytes(nblocks) bytes; pass
 * init != 0 on the first call with a given scratch (twiddle tables).
 * pair = 1: windows of 4M = 32768 samples on clusters of two CTAs (one 2M-point packed transform split by a
 * radix-2 stage: even frequencies in CTA 0, odd ones in CTA 1, joined over distributed shared memory), which
 * leaves 75 % of a window alias-free at 4096 coefficients instead of 50 % and admits bands of up to 8192
 * coefficients (2 (nband-1) < 2M); coef is then
 * [nblocks][2 (CTA c)][2][M] with entry p of CTA c = C[2 brev(p) + c] of the 2M-point transform. */
int cm2_toeplitz_fft_points(void);
int64_t cm2_toeplitz_fft_scratch_bytes(int64_t nblocks);
int cm2_noise_toeplitz_fft_apply(const double *coef, int nband, int64_t nblocks, int64_t blocksize,
                                 const int64_t *blk_start, const double *d, double *out,
                                 int64_t nt, void *scratch, int init, int pair, cm2_stream_t stream);
/* Welch periodogram sums per noise block (blocks as above), for estimating N^-1 from the data.  With
 * M = cm2_toeplitz_fft_points() and NF = 2M: block b of n_b samples holds floor((n_b - NF)/M) + 1 windows
 * of NF samples at hop M from its first sample if n_b >= NF, none otherwise; samples past the last full
 * window are not used.  In window w, x_t = h_t m_t d_t with the periodic Hann window h_t = sin^2(pi t/NF)
 * and m_t = 0 where pix[t] < 0 (pix may be NULL: no mask).  A flagged sample is selected away, so NaN in a
 * flagged d never reaches the result; nothing is detrended.  Outputs, for k = 0..M:
 *   psd[b][k] = S_b(k) = sum_w |X_w(k)|^2  (X_w the NF-point DFT of window w's x),
 *   wsum[b]   = W_b    = sum_w sum_t (h_t m_t)^2,
 * 0 for a block without windows.  S_b / W_b is the pooled one-sided-range estimate of the two-sided PSD
 * (without flags: scipy.signal.welch(window='hann', nperseg=NF, noverlap=M, detrend=False,
 * return_onesided=False)[:M+1]).  Deterministic: a repeated call gives the same bits, whatever the
 * alignment of d and pix.  scratch: cm2_noise_psd_scratch_bytes(nblocks) bytes for the current device,
 * 16-byte aligned; pass init != 0 on the first call with a given scratch (twiddle and window tables). */
int64_t cm2_noise_psd_scratch_bytes(int64_t nblocks);
int cm2_noise_psd(const double *d, const int32_t *pix /* NULL: no mask */, int64_t nblocks, int64_t blocksize,
                  const int64_t *blk_start, int64_t nt, double *psd /* [nblocks][M+1] */, double *wsum /* [nblocks] */,
                  void *scratch, int init, cm2_stream_t stream);
/* subscan offset filter (FilterLO.mult :129-168): out = 0; for each segment [seg_start[k],
 * seg_end[k]): mu = mean of d over unflagged samples; skipped if none; out = d - mu */
int cm2_filter_offset_apply(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end,
                            int64_t nseg, const double *d, double *out, int64_t nt,
                            cm2_stream_t stream);

/* ---- fused A-matvecs (no TOD temporary) ---------------------------------------------------- */
/* y = P^T diag(w) P x   (the composition P.T*N*P at tests/test_toeplitz_vector_multiplication.py:28)
 * nstreams (here and in the other single-pass A-matvecs): order in which the TOD is walked.  <= 1: time
 * order.  S > 1: the TOD is treated as S equally long timelines (detectors; the reference's layout is
 * detector-major, interfaces/linearoperators.py:134-140) that are walked round-robin, tile by tile, so that
 * all detectors are processed at the same scan time and the map rows they share stay in L2 -- for maps larger
 * than L2 (nside >= 1024 patches), where time order makes every detector timeline a pass over the whole map.
 * The result is the same sum in a different order of the atomic adds.
 * pix_packed: NULL, or the packed stream of pix from cm2_pack_pointing; the pass then reads 1 byte of pixel id
 * per sample instead of 4 (17 instead of 20 B/sample) and pix only for escape lanes.  Not with per-sample
 * weights (blocksize 1) or the staged scatter (cm2_amatvec_white_set_stage), which read pix. */
int cm2_amatvec_white(const int32_t *pix, const uint64_t *pix_packed, const double *cos2phi,
                      const double *sin2phi, int64_t nt, int pol, const double *wblk, int64_t nblocks,
                      int64_t blocksize, const int64_t *blk_start, const double *x, double *y,
                      int64_t npix, int64_t nstreams, cm2_stream_t stream);
/* packed[(nt + 7) / 8] = pix at one byte per sample, one 64-bit word per 8 samples t0 .. t0+7 (t0 = 8 l).  With
 * lo = the signed bits 0..31 of a word:
 *   lo >= 0   b0 = lo, b1 = b0 + (int16) bits 32..47, codes = bits 48..63; sample j has pixel
 *             (code_j & 2 ? b1 : b0) + (code_j & 1), code_j = (codes >> 2j) & 3;
 *   lo == -1  all 8 samples are flagged (-1); bits 32..63 are zero;
 *   lo == -2  escape: read the 8 pixels from pix (mixed flagged and unflagged samples, pixels the two bases do
 *             not cover, and the last word when nt % 8 != 0).
 * *nescape = the number of escape words.  pix 32-byte aligned. */
int cm2_pack_pointing(const int32_t *pix, int64_t nt, uint64_t *packed, int64_t *nescape, cm2_stream_t stream);
/* Scatter variant of cm2_amatvec_white: wpix > 0 stages the scatter of every warp tile whose pixels span fewer
 * than wpix pixels through a shared-memory window and flushes it with coalesced REDs (pixels crossed in few
 * samples: 1-4 samples per pixel crossing); 0 = run compression in registers + warp merge (the default). */
int cm2_amatvec_white_set_stage(int wpix);
/* y = P^T F P x with the offset filter (src/test_M2_precond_onto_real_data.py:86) */
int cm2_amatvec_filter(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                       int64_t nt, int pol, const int64_t *seg_start, const int64_t *seg_end,
                       int64_t nseg, const double *x, double *y, int64_t npix,
                       cm2_stream_t stream);

/* Single-TOD-pass P^T F P x (csrc/filter_runs.cu): u_k = P^T 1_k of every subscan is kept
 * run-compressed -- run_pix[nruns], run_mom[nruns][3] = {n, sum cos, sum sin}, per segment seg_first,
 * seg_nruns.  Build: runs_mark (flags[nt] at run starts, pix_masked[nt] = pix inside segments else
 * -1) -> exclusive scan of flags (cm2_weights_old2new) -> runs_fill.  Apply: seg_mean
 * (mu_k = u_k.x / n_k over the run table) -> amatvec_filter_mu: y = P^T (P x - mu_seg) over the
 * unflagged samples inside segments in one TOD pass.  Segments must be sorted and non-overlapping;
 * tile_seg[ceil(nt/256)] = first segment whose end lies beyond sample 256*tile; tile_flag = 0 (tile
 * in a gap), 1 (tile inside segment tile_seg) or 2 (a boundary falls inside the tile). */
int cm2_filter_runs_mark(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end,
                         int64_t nseg, int64_t nt, int32_t *flags, int32_t *pix_masked,
                         cm2_stream_t stream);
int cm2_filter_runs_fill(const int32_t *pix_masked, const double *cos2phi, const double *sin2phi,
                         int pol, const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                         const int32_t *runidx, int32_t *run_pix, double *run_mom,
                         int64_t *seg_first, int32_t *seg_nruns, cm2_stream_t stream);
int cm2_filter_seg_mean(const int32_t *run_pix, const double *run_mom, const int64_t *seg_first,
                        const int32_t *seg_nruns, int64_t nseg, int pol, const double *x,
                        double *mu, cm2_stream_t stream);
int cm2_amatvec_filter_mu(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                          int64_t nt, int pol, const int64_t *seg_start, const int64_t *seg_end,
                          const double *seg_mu, const int32_t *tile_seg, const uint8_t *tile_flag,
                          int64_t nseg, const double *x, double *y, int64_t npix, int64_t nstreams,
                          cm2_stream_t stream);

/* Single-TOD-pass P^T F_K P x for the Legendre filter, poly_order 1..4 (FilterLO.polyfilter
 * interfaces/linearoperators.py:170-204 inside the composition of src/test_M2_precond_onto_real_data.py:37-41;
 * csrc/filter_runs.cu).  The fitted polynomial of a subscan is sum_k c_k L_k(x_t) with c = W S, S the
 * Legendre moments of the unflagged samples and W fixed by the pointing.  Set-up: poly_gram (per subscan
 * W[nk*nk] and info = {unflagged samples, smallest pivot of the scaled Cholesky factor of the Gram matrix;
 * 1 without flags, 0 for a subscan the reference skips}; the caller keeps the well-conditioned subscans),
 * runs_mark + scan as for the offset filter, poly_runs_fill (run_mom[nruns][3*nk] = sums of L_k, L_k cos,
 * L_k sin over each run).  Apply: poly_seg_coef (coef[nseg][nk] = W S from the run table), then
 * amatvec_filter_poly_mu: y (+)= P^T (P x - polynomial) in one TOD pass; tile tables as for
 * cm2_amatvec_filter_mu.  Experimental: not selected by default (DESIGN.md section 10). */
int cm2_filter_poly_gram(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end,
                         int64_t nseg, int poly_order, double *W, double *info, cm2_stream_t stream);
int cm2_filter_poly_runs_fill(const int32_t *pix_masked, const double *cos2phi, const double *sin2phi,
                              int pol, const int64_t *seg_start, const int64_t *seg_end, int64_t nseg,
                              int poly_order, const int32_t *runidx, int32_t *run_pix, double *run_mom,
                              int64_t *seg_first, int32_t *seg_nruns, cm2_stream_t stream);
int cm2_filter_poly_seg_coef(const int32_t *run_pix, const double *run_mom, const int64_t *seg_first,
                             const int32_t *seg_nruns, int64_t nseg, int pol, int poly_order,
                             const double *W, const double *x, double *coef, cm2_stream_t stream);
int cm2_amatvec_filter_poly_mu(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                               int64_t nt, int pol, const int64_t *seg_start, const int64_t *seg_end,
                               const double *seg_coef, const int32_t *tile_seg, const uint8_t *tile_flag,
                               int64_t nseg, int poly_order, const double *x, double *y, int64_t npix,
                               int accumulate, int64_t nstreams, cm2_stream_t stream);

/* d = F P x for the offset filter in one TOD pass (the first two factors of a chain such as
 * P.T*F*N*F*P): d_t = (P x)_t - mu_seg(t) inside subscans -- flagged samples included, as
 * FilterLO.mult does (interfaces/linearoperators.py:165) -- and 0 in the gaps; seg_mu from
 * cm2_filter_seg_mean, tile tables as for cm2_amatvec_filter_mu. */
int cm2_pointing_filter_mu(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                           int64_t nt, int pol, const int64_t *seg_start, const int64_t *seg_end,
                           const double *seg_mu, const int32_t *tile_seg, const uint8_t *tile_flag,
                           int64_t nseg, const double *x, double *d, cm2_stream_t stream);

/* y = P^T T P x with T = the banded symmetric Toeplitz blocks of BlockLO(offdiag=True)
 * (ToeplitzLO.mult interfaces/linearoperators.py:582-595 applied per block, :672-674; the composition
 * A = P.T*N*P of tests/test_2level_preconditioner.py:16-29, tests/test_coarse_operator.py:15-26):
 * one TOD pass, no time-domain temporary.  band[nblocks][nband] = a_0 .. a_{nband-1} per block,
 * nband <= cm2_amatvec_toeplitz_max_band(); noise blocks as for cm2_noise_toeplitz_apply. */
int cm2_amatvec_toeplitz_max_band(void);
int cm2_amatvec_toeplitz(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                         int64_t nt, int pol, const double *band, int nband, int64_t nblocks,
                         int64_t blocksize, const int64_t *blk_start, const double *x, double *y,
                         int64_t npix, cm2_stream_t stream);

/* ---- a10/a11/a13: deflation, coarse operator, two-level preconditioner ---------------------- */
/* Z is n x r, column-major (column i at Z + i*ldz), as DeflationLO stores columns (:1058-1062).
 * `work`: cm2_defl_work_doubles(r) doubles of device scratch. */
int64_t cm2_defl_work_doubles(int r);
/* out[i] = Z[:,i] . x  (DeflationLO.rmult :1056); for ncols_x > 1: out = Z^T X, r x ncols_x
 * column-major (used for E = Z^T (A Z), CoarseLO :1019).  Deterministic reduction. */
int cm2_defl_zt_apply(const double *Z, int64_t n, int r, int64_t ldz, const double *X,
                      int ncols_x, int64_t ldx, double *out, double *work, cm2_stream_t stream);
/* y = beta*y0 + alpha * Z c  (DeflationLO.mult :1047-1050); y0 may be NULL */
int cm2_defl_z_apply(const double *Z, int64_t n, int r, int64_t ldz, const double *c,
                     double alpha, double beta, const double *y0, double *y,
                     cm2_stream_t stream);
/* c = Einv (r x r, column-major, device) * v  (CoarseLO.mult_eig :984) */
int cm2_coarse_apply(const double *Einv, int r, const double *v, double *c,
                     cm2_stream_t stream);
/* fused two-level apply (src/test_M2_precond_onto_real_data.py:109-112):
 *   c = Einv Z^T v ;  y = M_BD (v - AZ c) + Z c    (reads Z twice, AZ once) */
int cm2_m2_apply(const double *Z, const double *AZ, int64_t n, int r, int64_t ld,
                 const double *Einv, const double *bd_inv, int64_t npix, int pol,
                 const double *v, double *y, double *work, cm2_stream_t stream);
/* The same apply for a SUBDOMAIN coarse space (column k of Z = intensity indicator of the pixels of band k, as built
 * by cosmomap2_b200.scan_coarse_space): band[npix] = the pixel's column (-1: none), azb[npix][pol][3] = the entries of
 * A Z in columns band-1, band, band+1 (cyclic) -- A z_k lives on band k and its neighbours.  172 B per IQU pixel
 * instead of 3 r doubles per map element; pol = 1 or 3, 3 <= r <= 64; work as for cm2_m2_apply. */
int cm2_m2_banded_apply(const int32_t *band, const double *azb, int r, const double *Einv,
                        const double *bd_inv, int64_t npix, int pol, const double *v, double *y,
                        double *work, cm2_stream_t stream);

/* ---- a11 / a12: the dense tall-skinny contractions on the fp64 tensor cores (DMMA m8n8k4) ----------
 * Tall matrices are column-major with a leading dimension (every column contiguous).
 *   gram   : out (r1 x r2, column-major, ldo) = X^T Y, X: n x r1 (ldx), Y: n x r2 (ldy); ONE pass over X
 *            and Y per 32 x 32 panel of out.  E = Z^T (A Z): CoarseLO.__init__ -> dgemm(Z, Az.T),
 *            interfaces/linearoperators.py:1019, utilities/linear_algebra_funcs.py:16-29.
 *            work: cm2_dense_gram_work_doubles() doubles.
 *   combine: Z (n x r, ldz) = V (n x m, ldv) U (m x r, ldu); Z must not overlap V.  Ritz vectors
 *            V[:, :m] U (kp.utils.ritz, interfaces/deflationlib.py:204-219), build_Z (:140-184), and
 *            the thick restart of cosmomap2_b200.eigsh. */
int64_t cm2_dense_gram_work_doubles(void);
int cm2_dense_gram(const double *X, int64_t ldx, int r1, const double *Y, int64_t ldy, int r2,
                   int64_t n, double *out, int64_t ldo, double *work, cm2_stream_t stream);
int cm2_dense_combine(const double *V, int64_t ldv, int64_t n, int m, const double *U, int64_t ldu,
                      int r, double *Z, int64_t ldz, cm2_stream_t stream);

/* ---- a14: PCG vector work (scipy _isolve/iterative.py:405-431) ------------------------------- */
/* out[0] = a.b */
int cm2_dot(const double *a, const double *b, int64_t n, double *out, cm2_stream_t stream);
/* y = alpha*x + beta*y  (alpha, beta host scalars) */
int cm2_axpby(double alpha, const double *x, double beta, double *y, int64_t n,
              cm2_stream_t stream);
/* Device-scalar PCG.  scal[] is a 16-double device workspace:
 *   [0]=rho [1]=rho_prev [2]=p.q [3]=|r|^2 [4]=alpha [5]=beta [6]=atol
 *   [7]=done flag (||r||_2 < atol, SciPy's exit test) [8]=iterations completed [9..15] spare
 * Every update below is a no-op once the done flag is set, so the host may queue iterations
 * ahead of reading the flag and x still stops at exactly SciPy's iteration.
 * reset: |r|^2, atol, done flag, counters (call after r = b - A x0) */
int cm2_pcg_reset(const double *r, int64_t n, double *scal, double atol, cm2_stream_t stream);
/* rho = r.z ; beta = rho/rho_prev (0 on the first iteration) ; p = z + beta p */
int cm2_pcg_update_p(const double *r, const double *z, double *p, int64_t n, double *scal,
                     cm2_stream_t stream);
/* pq = p.q ; alpha = rho/pq ; x += alpha p ; r -= alpha q ; |r|^2 ; rho_prev = rho ; flags */
int cm2_pcg_update_xr(const double *p, const double *q, double *x, double *r, int64_t n,
                      double *scal, cm2_stream_t stream);
/* M = M_BD fast path (the preconditioner is pixel-local, so z = M r and rho = r.z ride in the
 * kernel that updates r):
 *   bd_reset   : z = M r ; rho = r.z ; |r|^2 ; atol ; flags.  With b, x non-NULL the x0 = 0 start
 *                of the solve happens in the same pass (r = b, x = 0) and rtol > 0 folds SciPy's
 *                atol = max(atol, rtol ||b||) in on the device; pass both NULL otherwise
 *   bd_update_p: p = z + beta p
 *   bd_update  : pq ; alpha ; x += alpha p ; r -= alpha q ; z = M r ; rho' ; beta' ; |r|^2 ; flags
 *   bd_iter    : bd_update followed by the NEXT iteration's p = z + beta' p, all in ONE cooperative
 *                launch (two grid barriers); with it an iteration is  q = A p ; bd_iter.  bd_reset's
 *                p0, when non-NULL, receives the first search direction p = z.
 * z is scratch of the M_BD path: bd_iter, and bd_reset with b, x and p0 all non-NULL, keep it on chip
 * and may leave the buffer unwritten; bd_update writes it for bd_update_p.  bd_iter holds its
 * pixels' p on chip between its grid barriers up to cm2_pcg_bd_iter_max_npix(pol) pixels and runs a
 * one-thread-per-pixel kernel above that, or when p, q, x or r is not 16-byte aligned. */
int cm2_pcg_bd_reset(const double *bd_inv, int64_t npix, int pol, double *r, double *z,
                     double *scal, double atol, double rtol, const double *b, double *x, double *p0,
                     cm2_stream_t stream);
int cm2_pcg_bd_update_p(const double *z, double *p, int64_t n, double *scal, cm2_stream_t stream);
int cm2_pcg_bd_update(const double *bd_inv, int64_t npix, int pol, const double *p,
                      const double *q, double *x, double *r, double *z, double *scal,
                      cm2_stream_t stream);
int cm2_pcg_bd_iter(const double *bd_inv, int64_t npix, int pol, double *p, const double *q,
                    double *x, double *r, double *z, double *scal, cm2_stream_t stream);
/* test hook: on != 0 makes cm2_pcg_bd_iter ask for more CTAs than can be co-resident, so that the
 * cooperative launch is refused like on a GPU that does not grant them; returns the previous value */
int cm2_pcg_bd_iter_refuse(int on);
/* the largest npix for which cm2_pcg_bd_iter runs its on-chip (tiled) kernel on the current device */
int64_t cm2_pcg_bd_iter_max_npix(int pol);
/* development/test hook: on != 0 makes cm2_pcg_bd_reset and cm2_pcg_bd_iter run the
 * one-thread-per-pixel kernels at every npix (the large-npix path); returns the previous value */
int cm2_pcg_bd_tail_strided(int on);

/* ---- (f) next rows: the other time-domain filters and the map output step ----------------------
 * Subscan filter of polynomial order 0..cm2_filter_poly_max_order(), one CTA per subscan with the
 * subscan staged in shared memory (d and pix read once, out written once; 20 B/sample).
 *   poly_order = 0: FilterLO.mult (linearoperators.py:129-168), same result as
 *                   cm2_filter_offset_apply: mean over samples with pix != -1, subtracted from every
 *                   sample of the subscan; subscans without unflagged samples and the gaps stay 0.
 *   poly_order > 0: FilterLO.polyfilter (:170-204): unflagged = pix >= 0; subscans with
 *                   <= poly_order unflagged samples stay 0; without flags p = sum_k (b_k.d) b_k with
 *                   b_k = L_k(x)/||L_k(x)||, x = linspace(-1,1,len) (get_legendre_polynomials,
 *                   utilities/linear_algebra_funcs.py:47-59); with flags the least-squares
 *                   polynomial over the unflagged samples (the reference's QR, :190-194);
 *                   out = d - p on unflagged samples, 0 on flagged ones.
 * max_seg_len = longest subscan (sizes the shared-memory window); sorted != 0 promises
 * seg_start[k] >= seg_end[k-1] for all k (then no memset of `out` is issued). */
int cm2_filter_poly_max_order(void);
/* Two variants exist: (A) one CTA per subscan staged by ordinary loads (any subscan length) and
 * (B) persistent CTAs with the subscans streamed through a ring of shared-memory stages by the TMA
 * engine (cp.async.bulk + mbarrier), used when two stages of the longest subscan fit (<= ~8 500
 * samples).  cm2_filter_poly_set_tma(0) forces (A) (tests, measurements); returns the old setting. */
int cm2_filter_poly_set_tma(int on);
int cm2_filter_poly_apply(const int32_t *pix, const int64_t *seg_start, const int64_t *seg_end,
                          int64_t nseg, int64_t max_seg_len, int poly_order, int sorted,
                          const double *d, double *out, int64_t nt, cm2_stream_t stream);
/* fused y = P^T F_K P x for the Legendre filter of order 1..cm2_amatvec_filter_poly_max_order()
 * (the composition at src/test_M2_precond_onto_real_data.py:37-41), no TOD temporary; segments as
 * above, flags taken from pix.  CM2_ERR_UNSUPPORTED if the longest subscan exceeds the
 * shared-memory window (~16 000 samples) or the order is out of range. */
int cm2_amatvec_filter_poly_max_order(void);
int cm2_amatvec_filter_poly(const int32_t *pix, const double *cos2phi, const double *sin2phi,
                            int64_t nt, int pol, const int64_t *seg_start, const int64_t *seg_end,
                            int64_t nseg, int64_t max_seg_len, int poly_order, const double *x,
                            double *y, int64_t npix, cm2_stream_t stream);
/* GroundFilterLO.mult (linearoperators.py:24-61): out = v - G (G^T G)^-1 G^T v, G = pol-1 pointing
 * onto ground bins (ground[t] in [0,nbins), -1 = flagged), (G^T G)^-1 = 1/hits where hits > 0
 * (counts_in_groundbins :26-46 -> cm2_hits_i64).  bins[nbins] is scratch (receives G^T v). */
int cm2_ground_filter_apply(const int32_t *ground, int64_t nt, int64_t nbins, const int64_t *hits,
                            const double *v, double *bins, double *out, cm2_stream_t stream);
/* second half alone, out = v - bins[g]/hits[g]: for a TOD sharded over GPUs the bin sums
 * (cm2_pointing_apply_t with pol = 1) and the hits are summed over ranks in between */
int cm2_ground_filter_sub(const int32_t *ground, int64_t nt, int64_t nbins, const int64_t *hits,
                          const double *bins, const double *v, double *out, cm2_stream_t stream);
/* reorganize_map (utilities/healpy_functions.py:50-105): out[k][obspix[p]] = map[pol*p + k] for
 * k < pol, zero elsewhere; out is pol arrays of healpix_npix = 12 nside^2 values, back to back. */
int cm2_reorganize_map(const double *map, const int64_t *obspix, int64_t npix, int pol,
                       int64_t healpix_npix, double *out, cm2_stream_t stream);

/* ---- (e) multi-GPU: map-domain all-reduce over NVLink peer memory ------------------------------
 * One process per GPU.  send/recv/signal tables are HOST arrays of `world` DEVICE pointers (entry g
 * = rank g's buffer mapped into this process through CUDA IPC; signal buffers are
 * cm2_allreduce_p2p_signal_bytes() bytes, zero-initialised once).  recv[rank] receives
 * sum_g send[g][0..n) (fixed rank order, bit-identical on every rank).  `generation` must be the
 * same non-zero, strictly increasing value on every rank for every call.  All ranks must call. */
int64_t cm2_allreduce_p2p_signal_bytes(void);
int cm2_allreduce_p2p(const void *const *send_ptrs_host, void *const *recv_ptrs_host,
                      void *const *signal_ptrs_host, int rank, int world, int64_t n,
                      uint32_t generation, cm2_stream_t stream);
int cm2_enable_peer_access(int peer_device);
/* timeout of the peer-flag waits of cm2_allreduce_p2p in seconds (default 20; <= 0 only queries);
 * returns the previous value.  A wait that times out never hangs: the error word at
 * signal + cm2_allreduce_p2p_signal_bytes() - 8 (uint32) receives the generation that failed. */
double cm2_allreduce_p2p_set_timeout(double seconds);

/* ---- (e) multi-GPU: the M_BD PCG tail fused with the map exchange (SURVEY 8e: reduce-scatter ->
 * pixel-sharded M_BD / CG vector work -> all-gather), ONE cooperative kernel per iteration over NVLink
 * peer memory.  Replaces, per iteration, scipy's cg loop body (scipy/_isolve/iterative.py:405-431)
 * around  q = A p  (call sites src/test_BD_precond_onto_real_data.py:47,
 * src/test_M2_precond_onto_real_data.py:117) for A = sum_g P_g^T N_g^-1 P_g sharded by detector
 * (layout linearoperators.py:134-167):
 *   reset != 0 : r = b, x = 0, z = M r, p = z (sent to every rank), rho, |r|^2,
 *                atol_eff = max(atol, rtol*||b||); scal[10] = ||b||^2
 *   reset == 0 : q = sum_g y_g on this rank's pixel slice (peer loads), p.q, alpha, x, r, z = M r,
 *                rho', |r|^2, beta, p = z + beta p sent to every rank (peer stores), flags
 * Rank g owns pixels [pix_lo[g], pix_lo[g+1]); pix_lo[g]*pol must be even.  Tables are HOST arrays of
 * `world` DEVICE pointers: y / p / sig = every rank's peer-visible buffers (n doubles, n doubles,
 * cm2_pcg_sharded_signal_bytes() zero-initialised bytes) mapped into this process; x / r / z / q
 * (slice length), inv (6 doubles per slice pixel), b (slice of the right-hand side, reset only), scal
 * (16 doubles, layout as above; [9] = generation of a timed-out wait, 0 = none) and part
 * (cm2_pcg_sharded_work_doubles()) are private: entries [rank0, rank0 + nvirt) are used.  nvirt = 1
 * is a real rank; nvirt = world with rank0 = 0 plays all ranks in one launch on one GPU (tests).
 * `generation`: the same non-zero, strictly increasing value on every rank for every call. */
int64_t cm2_pcg_sharded_signal_bytes(void);
int64_t cm2_pcg_sharded_work_doubles(void);
int cm2_pcg_bd_sharded(int reset, int pol, int world, int rank0, int nvirt,
                       const int64_t *pix_lo_host, const void *const *y_tab, void *const *p_tab,
                       void *const *sig_tab, void *const *x_tab, void *const *r_tab,
                       void *const *z_tab, void *const *q_tab, const void *const *inv_tab,
                       const void *const *b_tab, void *const *scal_tab, void *const *part_tab,
                       uint32_t generation, double atol, double rtol, double timeout_s,
                       cm2_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* COSMOMAP2_B200_H */
