"""
The noise model from the data: per-detector Welch PSD on the GPU, and the N^-1 Toeplitz bands for
``BlockLO(blocksize, bands, offdiag=True)`` (DESIGN.md section 4c), noise simulations with that model
(section 4d), and the noise model from the map residual d - P x (section 4e).

    freqs, psd = noise_psd(d, blocksize, pix=pix)     # cm2_noise_psd: one pass over the TOD on the device
    bands = inverse_noise_bands(psd, nband)            # host, NumPy: nblocks x (M+1) values
    N = BlockLO(blocksize, bands, offdiag=True)
    Mbd_weights = [t[0] for t in bands]
    n = simulate_noise(noise_sim_bands(psd, nband), blocksize, seed, realization)   # on the device

The PSD of ``d`` includes the sky, which is strongest at the scan frequencies.  Estimate the noise from the
residual of a first solve and solve again (section 4e); the residual is formed inside the PSD pass:

    x0 = solve with N0 = BlockLO(blocksize, inverse_noise_bands(noise_psd(d, blocksize, pix=pix)[1], nband), True)
    freqs, psd = noise_psd(d, blocksize, P=P, x=x0)    # PSD of d - P x0, masked by P's own pixel table
    x1 = solve with N1 = BlockLO(blocksize, inverse_noise_bands(psd, nband), offdiag=True)

Noise blocks are BlockLO's partition: ``blocksize`` an int (equal blocks, the remainder past
``nblocks * blocksize`` in the last one, nblocks = len(d) // blocksize) or one size per block.
``BlockLO(blocksize, bands)`` with an int spans exactly ``nblocks * blocksize`` samples: when the int
does not divide len(d), pass the per-block sizes (the last one with the remainder) to BlockLO, or to
both functions.

The TOD is sharded across ranks by detector and a noise block never straddles detectors, so every
rank estimates its own blocks from its own data: there is no collective and no ``comm`` argument.
"""
import numpy as np
import torch

from . import _device as dv
from .linearoperators import SparseLO, _block_starts, _Blocks, _ToeplitzFFT


def _points():
    return int(dv.call("cm2_toeplitz_fft_points"))


def _block_edges(nt, blocksize):
    if np.ndim(blocksize):
        edges = _block_starts(blocksize, len(blocksize))
        if int(edges[-1]) != nt:
            raise ValueError("block sizes add up to %d samples, the TOD has %d" % (int(edges[-1]), nt))
        return edges, 0
    bs = int(blocksize)
    if bs <= 0:
        raise ValueError("blocksize must be > 0")
    nb = max(nt // bs, 1)
    return np.r_[np.arange(nb, dtype=np.int64) * bs, nt], bs


def noise_psd(d, blocksize, pix=None, P=None, x=None):
    """Welch PSD of every noise block of the TOD ``d`` (host array or device tensor), computed on the GPU, or of the
    map residual ``d - P x`` when a pointing ``P`` and a map ``x`` are given.

    Windows of NF = 2M = 16384 samples (M = ``cm2_toeplitz_fft_points()``) at hop M (50 % overlap) from
    each block's first sample; samples past the last full window are not used.  Each window is tapered
    with the periodic Hann window and masked where ``pix < 0`` (``pix``: the pointing with -1 for flagged
    samples -- ``P.pairs``, raw ``pixs`` or a device int32 tensor; None: nothing flagged).  A flagged
    sample is selected away, so NaN in flagged ``d`` does not reach the result.  Nothing is detrended:
    pass ``F d`` for filtered data, or ``d - P x`` for a residual.

    ``psd[b] = sum_w |X_w|^2 / sum_w sum_t (h_t m_t)^2`` over block b's windows, k = 0..M: a pooled
    estimate in which a window with many flags counts less.  Without flags this is
    ``scipy.signal.welch(d_b, fs=1, window='hann', nperseg=NF, noverlap=M, detrend=False,
    return_onesided=False)[1][:M+1]``.  Returns ``(freqs, psd)``: cycles per sample, shape (M+1,), and
    shape (nblocks, M+1).  Raises ValueError for a block shorter than one window or with every window
    sample flagged.  With an int ``blocksize`` that does not divide len(d) the last block holds the
    remainder; give BlockLO the same partition as per-block sizes.

    Residual (``cm2_noise_psd_residual``): with ``P`` a ``SparseLO`` and ``x`` its map (host or device,
    ``P.pol * P.ncols`` float64 values), the samples are ``r_t = d_t - (P x)_t``, formed inside the PSD pass: no
    residual TOD is written.  The mask is ``P``'s own pixel table, so samples whose pixel ProcessTimeSamples dropped
    are masked too.  The result is bit for bit ``noise_psd(d - P.mult(x), blocksize, pix=<P's pixel table>)``.  The
    two-pass estimate: solve with bands from ``noise_psd(d, ...)``, then estimate again from
    ``noise_psd(d, ..., P=P, x=x0)`` and solve with the new bands (DESIGN.md section 4e).  Raises ValueError for
    ``pix`` together with ``P``, only one of ``P`` and ``x``, a ``P`` that is not a ``SparseLO`` (composite operators
    are not accepted), ``len(d) != P.nrows`` or a wrong length of ``x``.
    """
    nt = int(d.numel() if dv.is_dev(d) else np.size(d))
    if P is not None and pix is not None:
        raise ValueError("pass pix or P, not both: the residual is masked by P's own pixel table")
    if (P is None) != (x is None):
        raise ValueError("a residual needs both P and x")
    if P is not None:
        if not isinstance(P, SparseLO):
            raise ValueError("P must be a SparseLO pointing operator, got %s" % type(P).__name__)
        if nt != P.nrows:
            raise ValueError("d has %d samples, P has %d rows" % (nt, P.nrows))
        nx = int(x.numel() if dv.is_dev(x) else np.size(x))
        if nx != P.pol * P.ncols:
            raise ValueError("x has %d values, P needs pol * ncols = %d" % (nx, P.pol * P.ncols))
    M = _points()
    NF = 2 * M
    edges, bs = _block_edges(nt, blocksize)
    nb = len(edges) - 1
    short = np.flatnonzero(np.diff(edges) < NF)
    if short.size:
        b = int(short[0])
        raise ValueError("noise block %d has %d samples: fewer than one window of %d"
                         % (b, int(edges[b + 1] - edges[b]), NF))
    dd = dv.to_dev_f64(d).reshape(-1)
    pp = None
    if pix is not None:
        pp = dv.pix_to_dev(pix)
        if pp.numel() != nt:
            raise ValueError("pix has %d samples, d has %d" % (pp.numel(), nt))
    start = None if bs else dv.to_dev(edges, torch.int64)
    scratch = torch.empty(int(dv.call("cm2_noise_psd_scratch_bytes", nb)) // 8 + 2, dtype=torch.float64,
                          device=dd.device)
    S = torch.empty(nb * (M + 1), dtype=torch.float64, device=dd.device)
    W = torch.empty(nb, dtype=torch.float64, device=dd.device)
    if P is None:
        dv.call("cm2_noise_psd", dv.ptr(dd), dv.ptr(pp), nb, bs, dv.ptr(start), nt, dv.ptr(S), dv.ptr(W),
                dv.ptr(scratch), 1, dv.stream())
    else:
        xx = dv.to_dev_f64(x).reshape(-1)
        dv.call("cm2_noise_psd_residual", dv.ptr(dd), dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev),
                P.pol, dv.ptr(xx), nb, bs, dv.ptr(start), nt, dv.ptr(S), dv.ptr(W), dv.ptr(scratch), 1, dv.stream())
    S = dv.to_host(S).reshape(nb, M + 1)
    W = dv.to_host(W)
    empty = np.flatnonzero(~(W > 0))
    if empty.size:
        raise ValueError("noise block %d: every window sample is flagged" % int(empty[0]))
    return np.arange(M + 1) / float(NF), S / W[:, None]


def inverse_noise_bands(psd, nband):
    """N^-1 Toeplitz bands from the PSDs of ``noise_psd`` (host, NumPy), one per block:

        c_b = irfft(1 / psd_b, NF)[:nband],   t_b[j] = c_b[j] (1 - j / nband),   1 <= nband <= M.

    The Bartlett lag taper has a non-negative transform, so the Toeplitz symbol of every band is positive
    for any positive PSD: N^-1 is positive definite and P^T N^-1 P symmetric positive (semi)definite,
    whatever the data.  ``nband = 1`` gives t_b[0] = mean of 1/psd_b over the full circle of NF
    frequencies: the white weight, usable in ``BlockLO(blocksize, t)``.  Pass the result straight to
    ``BlockLO(blocksize, bands, offdiag=True)``; the M_BD weights are ``[t[0] for t in bands]``.
    Raises ValueError when a block's PSD has a value <= 0 or not finite.
    """
    return _tapered_bands(psd, nband, lambda p: 1.0 / p)


def _tapered_bands(psd, nband, symbol):
    """t_b[j] = c_b[j] (1 - j / nband), c_b = irfft(symbol(psd_b), NF)[:nband]: the Bartlett lag taper shared by
    the N^-1 bands and the simulation bands."""
    psd = np.atleast_2d(np.asarray(psd, dtype=np.float64))
    M = psd.shape[1] - 1
    nband = int(nband)
    if M < 1 or not 1 <= nband <= M:
        raise ValueError("nband must be in [1, %d], got %d" % (M, nband))
    for b in range(psd.shape[0]):
        if not np.all(np.isfinite(psd[b]) & (psd[b] > 0)):
            raise ValueError("noise block %d: the PSD has a value <= 0 or not finite" % b)
    c = np.fft.irfft(symbol(psd), 2 * M, axis=1)[:, :nband]
    t = c * (1.0 - np.arange(nband) / float(nband))
    return [t[b].copy() for b in range(psd.shape[0])]


def noise_sim_bands(psd, nband):
    """Simulation bands from the PSDs of ``noise_psd`` (host, NumPy), one per block, for ``simulate_noise``:

        c_b = irfft(sqrt(psd_b), NF)[:nband],   t_b[j] = c_b[j] (1 - j / nband),   1 <= nband <= M.

    The Bartlett lag taper of ``inverse_noise_bands`` keeps the symbol smooth, so truncation makes no Gibbs
    notches.  Noise drawn with band t_b has exactly the PSD |sum_{|j|<nband} t_b[|j|] e^{-2 pi i f j}|^2; at
    nband = M that is psd_b smoothed by the Fejer kernel, and nothing below the resolution 1/NF of the estimate
    is invented.  ``nband = 1`` gives white noise of amplitude mean(sqrt(psd_b)) over the full circle of NF
    frequencies.  Raises ValueError when a block's PSD has a value <= 0 or not finite.
    """
    return _tapered_bands(psd, nband, np.sqrt)


# Bands of at least this many coefficients are simulated on 32768-sample windows on 2-CTA clusters: only those that one
# CTA's window cannot hold.  Unlike the apply (TOEPLITZ_FFT_PAIR_MIN_BAND), each CTA of a cluster generates both halves
# of its window, twice the generator work per output.  Measured per 1e8 samples on a B200, one-CTA / cluster windows:
# 1.29 / 2.17 ms at 1 coefficient, 1.34 / 2.18 at 256, 2.41 / 2.78 at 4096 (DESIGN.md section 4d).
NOISE_SIM_PAIR_MIN_BAND = 4097


class NoiseSimulator(object):
    """The device tables of ``simulate_noise`` for one set of bands and blocks, kept for many draws (a Monte Carlo):
    ``NoiseSimulator(bands, blocksize)(seed, realization=0, block_ids=None, add_to=None)``."""

    def __init__(self, bands, blocksize):
        bands = [np.atleast_1d(np.asarray(a, dtype=np.float64)) for a in bands]
        nb = len(bands)
        if nb == 0:
            raise ValueError("no noise blocks")
        L = max(len(a) for a in bands)
        band = np.zeros((nb, L))
        for i, a in enumerate(bands):
            band[i, :len(a)] = a
        self._fft = _ToeplitzFFT(band, L, pair=L >= NOISE_SIM_PAIR_MIN_BAND)
        if not self._fft.ok:
            raise ValueError("bands of %d coefficients: at most %d can be simulated" % (L, _points()))
        self.nband, self.nblocks = L, nb
        self._blk = _Blocks(_block_starts(blocksize, nb))
        self.nt = self._blk.nt

    def __call__(self, seed, realization=0, block_ids=None, add_to=None):
        ids = None
        if block_ids is not None:
            ids = np.asarray(block_ids, dtype=np.int64).reshape(-1)
            if ids.size != self.nblocks or np.any(ids < 0) or np.any(ids >= 1 << 32):
                raise ValueError("block_ids: one id in [0, 2^32) per noise block")
            ids = dv.to_dev(ids, torch.int64)
        seed, realization = int(seed), int(realization)
        if not 0 <= seed < 1 << 64 or not 0 <= realization < 1 << 32:
            raise ValueError("seed must be in [0, 2^64) and realization in [0, 2^32)")
        fft = self._fft
        if add_to is None:
            out = torch.empty(self.nt, dtype=torch.float64, device=fft.coef.device)
        else:
            out = add_to
            if not (isinstance(out, torch.Tensor) and out.is_cuda and out.device == fft.coef.device
                    and out.dtype == torch.float64 and out.is_contiguous()):
                raise ValueError("add_to must be a contiguous float64 tensor on %s" % fft.coef.device)
            if out.numel() != self.nt:
                raise ValueError("add_to has %d samples, the noise blocks %d" % (out.numel(), self.nt))
        nb, bs, startp = self._blk.args()
        dv.call("cm2_noise_simulate", dv.ptr(fft.coef), self.nband, nb, bs, startp, dv.ptr(ids), seed, realization,
                dv.ptr(out), self.nt, int(add_to is not None), dv.ptr(fft.scratch), fft.init, fft.pair, dv.stream())
        fft.init = 0
        return out


def simulate_noise(bands, blocksize, seed, realization=0, block_ids=None, add_to=None):
    """Gaussian noise with the band ``bands[b]`` in noise block b, drawn on the GPU (``cm2_noise_simulate``):

        n_t = sum_{|k|<L} h_b[|k|] w_b(t - k - s_b),   s_b <= t < e_b,

    with w_b a unit Gaussian stream (Philox4x32-10 and Box-Muller, DESIGN.md section 4d) keyed on
    ``(seed, realization, block_ids[b])`` and defined past the block edges, so the noise is stationary up to them.
    A sample depends on that key and its offset in the block only: the same detector gets the same noise however
    the TOD is split over calls or ranks.  Sharded use: each rank passes the global ids of its own blocks
    (default ``range(len(bands))``).  The blocks are BlockLO's partition ``_block_starts(blocksize, len(bands))``,
    so ``BlockLO(blocksize, bands)`` and the simulation agree; bands of different lengths are zero-padded.  Use
    ``noise_sim_bands(psd, nband)`` for bands with the PSD of ``noise_psd``; bands of up to M = 8192 coefficients.
    Returns a new float64 device tensor, or adds the noise in place to ``add_to`` (d = P m + n without a second
    TOD buffer), which must have exactly the partition's number of samples, and returns it.  For many draws with
    the same bands, keep a ``NoiseSimulator``.
    """
    return NoiseSimulator(bands, blocksize)(seed, realization, block_ids, add_to)


def baseline_prior_bands(psd, L, nband, white=None):
    """``(weights, bands)`` of a destriper with a noise prior (``Destriper``, DESIGN.md section 4f) from the PSDs of
    ``noise_psd`` (host, NumPy), for baselines of ``L`` samples.  For each block b:

    1. the white level sigma2_b = ``white[b]``, by default the median of psd_b over the bins k >= M/2;
    2. the correlated part C_b = max(psd_b - sigma2_b, 0);
    3. the spectral density of the baseline means, S_b(F) = (1/L) sum_{m=0}^{L-1} C_b(f_m) K_L(f_m) with
       f_m = (F + m)/L folded into [-1/2, 1/2] and K_L(f) = [sin(pi L f) / (L sin(pi f))]^2, on F_k = k/(2M),
       k = 0..M, with C_b interpolated linearly in |f|;
    4. bands = the Bartlett-tapered coefficients of 1/S_b (as ``inverse_noise_bands``), so the prior's Toeplitz
       symbol is positive; ``weights[b]`` = 1/sigma2_b.

    The densities are two-sided, with their integral over [-1/2, 1/2] the variance, as ``noise_psd``'s.  Pass
    ``weights`` to ``BlockLO(blocksize, weights)`` and ``bands`` as the ``prior``.  Raises ValueError for nband
    outside [1, M], L < 1, a wrong length of ``white`` and a block whose S_b is not positive somewhere (a PSD with
    no correlated part, for instance).
    """
    psd = np.atleast_2d(np.asarray(psd, dtype=np.float64))
    nb, M = psd.shape[0], psd.shape[1] - 1
    L, nband = int(L), int(nband)
    if M < 1 or not 1 <= nband <= M:
        raise ValueError("nband must be in [1, %d], got %d" % (M, nband))
    if L < 1:
        raise ValueError("the baseline length must be >= 1 sample, got %d" % L)
    k = np.arange(M + 1)
    if white is None:
        sigma2 = np.median(psd[:, k >= M / 2.0], axis=1)
    else:
        sigma2 = np.asarray(white, dtype=np.float64).reshape(-1)
        if sigma2.size != nb:
            raise ValueError("white has %d values, psd has %d blocks" % (sigma2.size, nb))
    if not np.all(np.isfinite(sigma2) & (sigma2 > 0)):
        raise ValueError("the white level must be positive and finite in every block")
    C = np.maximum(psd - sigma2[:, None], 0.0)
    f = k / (2.0 * M)                                   # the PSD bins and the baseline frequencies F_k alike
    S = np.zeros((nb, M + 1))
    step = max(1, (1 << 22) // (M + 1))                 # aliases per chunk: bounded temporaries for long baselines
    for m0 in range(0, L, step):
        fm = (f[:, None] + np.arange(m0, min(L, m0 + step))[None, :]) / L
        fm -= np.round(fm)
        sf = np.sin(np.pi * fm)
        tiny = np.abs(sf) < 1e-300
        K = np.where(tiny, 1.0, np.sin(np.pi * L * fm) / (L * np.where(tiny, 1.0, sf))) ** 2
        af = np.abs(fm).reshape(-1)
        for b in range(nb):
            S[b] += (np.interp(af, f, C[b]).reshape(K.shape) * K).sum(axis=1)
    S /= L
    for b in range(nb):
        if not np.all(np.isfinite(S[b]) & (S[b] > 0)):
            raise ValueError("noise block %d: the baseline spectrum is not positive everywhere (no correlated noise "
                             "at some frequency): no prior can be formed" % b)
    return 1.0 / sigma2, _tapered_bands(S, nband, lambda s: 1.0 / s)
