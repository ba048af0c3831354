"""
The noise model from the data: per-detector Welch PSD on the GPU, and the N^-1 Toeplitz bands for
``BlockLO(blocksize, bands, offdiag=True)`` (DESIGN.md section 4c).

    freqs, psd = noise_psd(d, blocksize, pix=pix)     # cm2_noise_psd: one pass over the TOD on the device
    bands = inverse_noise_bands(psd, nband)            # host, NumPy: nblocks x (M+1) values
    N = BlockLO(blocksize, bands, offdiag=True)
    Mbd_weights = [t[0] for t in bands]

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
from .linearoperators import _block_starts


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


def noise_psd(d, blocksize, pix=None):
    """Welch PSD of every noise block of the TOD ``d`` (host array or device tensor), computed on the GPU.

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
    """
    nt = int(d.numel() if dv.is_dev(d) else np.size(d))
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
    dv.call("cm2_noise_psd", dv.ptr(dd), dv.ptr(pp), nb, bs, dv.ptr(start), nt, dv.ptr(S), dv.ptr(W),
            dv.ptr(scratch), 1, dv.stream())
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
    psd = np.atleast_2d(np.asarray(psd, dtype=np.float64))
    M = psd.shape[1] - 1
    nband = int(nband)
    if M < 1 or not 1 <= nband <= M:
        raise ValueError("nband must be in [1, %d], got %d" % (M, nband))
    for b in range(psd.shape[0]):
        if not np.all(np.isfinite(psd[b]) & (psd[b] > 0)):
            raise ValueError("noise block %d: the PSD has a value <= 0 or not finite" % b)
    c = np.fft.irfft(1.0 / psd, 2 * M, axis=1)[:, :nband]
    t = c * (1.0 - np.arange(nband) / float(nband))
    return [t[b].copy() for b in range(psd.shape[0])]
