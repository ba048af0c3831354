"""
Drop-in operator classes for the map-making hot path, with the names, constructor signatures and
attributes of the reference's ``interfaces/linearoperators.py`` / ``interfaces/blkop.py``.

Every ``mult``/``rmult`` below is a CUDA kernel behind the C ABI (include/cosmomap2_b200.h); the
classes only own device buffers and describe the launch.  There is no CPU path.
"""
import numpy as np
import torch
from scipy.linalg import eigh, lu_factor, lu_solve

from . import _device as dv
from . import linop as lp
from .process_ces import BlockWeights, ProcessTimeSamples  # noqa: F401


def _stream():
    return dv.stream()


# =============================================================================================
# pointing
# =============================================================================================
class SparseLO(lp.LinearOperator):
    """Pointing operator P (nt x pol*npix) and P^T -- interfaces/linearoperators.py:326-557.

    ``SparseLO(n, m, pix_samples, pol=1, angle_processed=None)``; attributes ``ncols, nrows, pol,
    pairs, cos, sin, maptype``.  The device image of ``pix_samples`` is taken at construction
    (the reference aliases the caller's array, :531).
    """

    def __init__(self, n, m, pix_samples, pol=1, angle_processed=None):
        dv.require_cuda()
        self.ncols = int(n)
        self.nrows = int(m)
        self.pol = pol
        self.pairs = pix_samples
        if pol not in (1, 2, 3):
            raise RuntimeError("No valid polarization key set!\t=>\tpol=%d \n \
                                    Possible values are pol=%d(I),%d(QU), %d(IQU)." % (pol, 1, 2, 3))
        if len(pix_samples) != self.nrows:
            raise lp.ShapeError("pix_samples must have one pixel per time sample")
        self._angles = angle_processed
        self._pix_dev = dv.pix_to_dev(pix_samples)
        self._cos_dev = self._sin_dev = None
        if pol > 1:
            c = getattr(angle_processed, "_cos_dev", None)
            if c is not None:
                self._cos_dev, self._sin_dev = angle_processed._cos_dev, angle_processed._sin_dev
            else:
                self._cos_dev = dv.to_dev_f64(angle_processed.cos)
                self._sin_dev = dv.to_dev_f64(angle_processed.sin)
        self._sorted = None
        self.__runcase = {1: "I", 2: "QU", 3: "IQU"}[pol]
        super(SparseLO, self).__init__(nargin=self.pol * self.ncols, nargout=self.nrows, matvec=self.mult,
                                       rmatvec=self.rmult, symmetric=False, device=True)

    # reference attribute names; host copies are made on demand
    @property
    def cos(self):
        return self._angles.cos

    @property
    def sin(self):
        return self._angles.sin

    @property
    def maptype(self):
        return self.__runcase

    def mult(self, v):                                    # :356-384, 411-438, 463-497
        d = dv.empty_f64(self.nrows)
        dv.call("cm2_pointing_apply", dv.ptr(self._pix_dev), dv.ptr(self._cos_dev), dv.ptr(self._sin_dev),
                self.nrows, self.pol, dv.ptr(v), dv.ptr(d), _stream())
        return d

    mult_qu = mult_iqu = mult

    def rmult(self, v):                                   # :385-410, 439-462, 498-526
        y = dv.out_f64(self.ncols * self.pol)
        dv.call("cm2_pointing_apply_t", dv.ptr(self._pix_dev), dv.ptr(self._cos_dev), dv.ptr(self._sin_dev),
                self.nrows, self.pol, dv.ptr(v), dv.ptr(y), self.ncols, _stream())
        return y

    rmult_qu = rmult_iqu = rmult

    # -- deterministic transpose (pixel-sorted, no atomics) ---------------------------------------
    def build_sorted(self):
        """Stable argsort of the samples by pixel (flagged dropped) for ``rmult_sorted``."""
        if self._sorted is None:
            pix = self._pix_dev
            order = torch.sort(pix, stable=True).indices            # one-off set-up
            nflag = int((pix < 0).sum().item())
            perm = order[nflag:].to(torch.int32).contiguous()
            counts = torch.bincount(pix[pix >= 0].to(torch.int64), minlength=self.ncols)
            rowptr = torch.zeros(self.ncols + 1, dtype=torch.int64, device=pix.device)
            rowptr[1:] = torch.cumsum(counts, 0)
            self._sorted = (rowptr, perm)
        return self._sorted

    def rmult_sorted(self, v):
        rowptr, perm = self.build_sorted()
        v = dv.to_dev_f64(v)
        y = dv.empty_f64(self.ncols * self.pol)
        dv.call("cm2_pointing_apply_t_sorted", dv.ptr(rowptr), dv.ptr(perm), dv.ptr(self._cos_dev),
                dv.ptr(self._sin_dev), self.pol, dv.ptr(v), dv.ptr(y), self.ncols, _stream())
        return y

    def run_statistics(self):
        """(mean run length, contiguity): the mean number of consecutive samples on the same pixel (flagged
        samples excluded) and the fraction of pixel changes that go to the neighbouring pixel index (a sweep along
        a pixel row) -- what the fused A-matvecs use to choose their scatter (registers / staged through shared
        memory / pixel-sorted pointing).  One chunked pass over the pixels at first use."""
        if getattr(self, "_run_stats", None) is None:
            pix, nt = self._pix_dev, self.nrows
            starts = good = near = 0
            step = 1 << 27
            for a in range(0, nt, step):
                b = min(a + step, nt)
                cur = pix[a:b]
                prev = pix[a - 1:b - 1] if a > 0 else torch.cat([cur[:1] - 2, cur[:-1]])
                ok = cur >= 0
                change = (cur != prev) & ok
                starts += int(change.sum().item())
                near += int((change & ((cur - prev).abs() == 1)).sum().item())
                good += int(ok.sum().item())
            self._run_stats = (good / max(starts, 1), near / max(starts, 1))
        return self._run_stats

    def mean_run_length(self):
        return self.run_statistics()[0]

    def hits(self):
        out = torch.empty(max(self.ncols, 1), dtype=torch.int64, device=self._pix_dev.device)
        dv.call("cm2_hits_i64", dv.ptr(self._pix_dev), self.nrows, self.ncols, dv.ptr(out), _stream())
        return dv.to_host(out[:self.ncols])


# =============================================================================================
# noise
# =============================================================================================
def _block_starts(blocksize, nblocks):
    if np.ndim(blocksize):
        sizes = np.asarray(blocksize, dtype=np.int64)
        if len(sizes) != nblocks:
            raise ValueError("need one block size per noise value")
    else:
        sizes = np.full(nblocks, int(blocksize), dtype=np.int64)
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


class _Blocks(object):
    """Device description of the block partition of the TOD."""

    def __init__(self, starts):
        self.starts = np.asarray(starts, dtype=np.int64)
        self.n = len(self.starts) - 1
        sizes = np.diff(self.starts)
        self.blocksize = int(sizes[0]) if self.n and np.all(sizes == sizes[0]) else 0
        self.nt = int(self.starts[-1])
        self._dev = None

    def args(self):
        """(nblocks, blocksize, blk_start_ptr)"""
        if self.blocksize == 0 and self._dev is None:
            self._dev = dv.to_dev(self.starts, torch.int64)
        return self.n, self.blocksize, dv.ptr(self._dev)


class ToeplitzLO(lp.LinearOperator):
    """Symmetric banded Toeplitz block, zero boundaries -- interfaces/linearoperators.py:560-602."""

    def __init__(self, a, size):
        self.array = a
        self._blocks = _Blocks([0, int(size)])
        self._band_dev = None
        super(ToeplitzLO, self).__init__(nargin=size, nargout=size, matvec=self.mult, symmetric=True,
                                         device=True)

    def mult(self, v):                                    # :582-595
        if self._band_dev is None:
            band = np.atleast_1d(np.asarray(self.array, dtype=np.float64))
            self._band_dev = dv.to_dev_f64(band)
            self._fft = _ToeplitzFFT(band, len(band)) if len(band) >= TOEPLITZ_FFT_MIN_BAND else None
        return _toeplitz_apply(self._band_dev, self._band_dev.numel(), self._blocks, v, self._fft)


TOEPLITZ_FFT_MIN_BAND = 48     # bands at least this wide go through the overlap-save FFT kernel (measured
                               # crossover at 1e8 samples: direct 64 lags 2.29 ms, FFT 1.5 ms for any band <= 256)


# Bands of at least this many coefficients use 32768-sample windows on 2-CTA clusters (1.5x fewer window points per
# output at 4096 coefficients, paid for by the join over distributed shared memory and a second read of the window).
# Measured per 1e8 samples, one-CTA windows / cluster windows: 1.14 / 1.42 ms at 2048 coefficients, 1.46 / 1.43 at 3000,
# 1.63 / 1.54 at 4096; beyond 4096 one CTA cannot hold the band at all (before: the direct kernel, ~50x slower there).
TOEPLITZ_FFT_PAIR_MIN_BAND = 3000


def _bit_reverse(M):
    k = np.arange(M)
    bits = int(np.log2(M))
    brev = np.zeros(M, dtype=np.int64)
    for bit in range(bits):
        brev |= ((k >> bit) & 1) << (bits - 1 - bit)
    return brev


def _packed_transfer(a, nband, M):
    """C1, C2 (natural frequency order, 1/M folded in) of the M-point packed transform of a 2M-sample window."""
    NF = 2 * M
    hc = np.zeros(NF)
    hc[:nband] = a
    if nband > 1:
        hc[NF - nband + 1:] = a[1:][::-1]
    H = np.fft.fft(hc).real                      # real and even: the band is symmetric
    w = np.exp(-2j * np.pi * np.arange(M) / NF)
    Hs, Hd = 0.5 * (H[:M] + H[M:]), 0.5 * (H[:M] - H[M:])
    return (Hs + 1j * Hd * np.conj(w)) / M, (Hd * w + 1j * Hs) / M


def toeplitz_fft_tables(band_host, nband, M, pair=False):
    """Packed transfer functions C1, C2 of cm2_noise_toeplitz_fft_apply for every noise block (host, NumPy), 1/M
    folded in, stored at the position the kernel keeps each frequency at (spectra stay bit-reversed in place).
    ``pair=False``: [nblocks][2][M] for windows of 2M samples, table[p] = C[brev(p)].
    ``pair=True``: [nblocks][2 (CTA)][2][M] for windows of 4M samples on a 2-CTA cluster: CTA c holds the
    frequencies 2k' + c of the 2M-point transform at position brev(k').  See csrc/toeplitz_fft.cu."""
    band_host = np.asarray(band_host, dtype=np.float64).reshape(-1, nband)
    nb = band_host.shape[0]
    brev = _bit_reverse(M)
    if not pair:
        coef = np.empty((nb, 2, M), dtype=np.complex128)
        for b in range(nb):
            C1, C2 = _packed_transfer(band_host[b], nband, M)
            coef[b, 0] = C1[brev]                    # table[position] = C[brev(position)]
            coef[b, 1] = C2[brev]
        return coef
    coef = np.empty((nb, 2, 2, M), dtype=np.complex128)
    for b in range(nb):
        C1, C2 = _packed_transfer(band_host[b], nband, 2 * M)
        for c in range(2):
            coef[b, c, 0] = C1[2 * brev + c]
            coef[b, c, 1] = C2[2 * brev + c]
    return coef


class _ToeplitzFFT(object):
    """Host-built packed transfer functions + device scratch for cm2_noise_toeplitz_fft_apply."""

    def __init__(self, band_host, nband):
        M = int(dv.call("cm2_toeplitz_fft_points"))
        self.pair = 1 if nband >= TOEPLITZ_FFT_PAIR_MIN_BAND else 0
        self.ok = 2 * (nband - 1) < (2 * M if self.pair else M)
        if not self.ok:
            return
        coef = toeplitz_fft_tables(band_host, nband, M, pair=bool(self.pair))
        nb = coef.shape[0]
        self.coef = dv.to_dev_f64(coef.view(np.float64).reshape(-1))
        self.scratch = torch.empty(int(dv.call("cm2_toeplitz_fft_scratch_bytes", nb)) // 8 + 2, dtype=torch.float64,
                                   device=self.coef.device)
        self.init = 1
        self.nband = int(nband)

    def apply(self, blocks, v):
        out = torch.empty_like(v)
        nb, bs, startp = blocks.args()
        dv.call("cm2_noise_toeplitz_fft_apply", dv.ptr(self.coef), self.nband, nb, bs, startp, dv.ptr(v), dv.ptr(out),
                v.numel(), dv.ptr(self.scratch), self.init, self.pair, _stream())
        self.init = 0
        return out


def _toeplitz_apply(band_dev, nband, blocks, v, fft=None):
    if fft is not None and fft.ok:
        return fft.apply(blocks, v)
    out = torch.empty_like(v)
    nb, bs, startp = blocks.args()
    scratch = torch.empty(nb + 1, dtype=torch.int64, device=v.device)
    dv.call("cm2_noise_toeplitz_apply", dv.ptr(band_dev), int(nband), nb, bs, startp, dv.ptr(v), dv.ptr(out),
            v.numel(), dv.ptr(scratch), _stream())
    return out


class WeightingLO(lp.LinearOperator):
    """Per-(CES, detector) scalar weight -- interfaces/linearoperators.py:604-625.
    The reference scales ``d`` IN PLACE and returns it (:613); so does this."""

    def __init__(self, bolos_per_ces, samples_per_bolopair, weights):
        self.ndet_pairs = bolos_per_ces
        self.nsample_per_pair = samples_per_bolopair
        self.size = int(np.sum([i * j for i, j in zip(samples_per_bolopair, bolos_per_ces)]))
        self.weights = np.asarray(weights, dtype=np.float64)
        sizes = np.concatenate([np.full(int(b), int(ns)) for b, ns in zip(bolos_per_ces, samples_per_bolopair)])
        self._blocks = _Blocks(np.concatenate([[0], np.cumsum(sizes)]))
        self._w_dev = None
        super(WeightingLO, self).__init__(nargin=self.size, nargout=self.size, matvec=self.mult,
                                          symmetric=True, device=True)

    def mult(self, d):
        if self._w_dev is None:
            self._w_dev = dv.to_dev_f64(self.weights[:self._blocks.n])
        nb, bs, startp = self._blocks.args()
        dv.call("cm2_noise_white_apply", dv.ptr(self._w_dev), nb, bs, startp, dv.ptr(d), dv.ptr(d), d.numel(),
                _stream())
        return d

    def matvec(self, x):
        if isinstance(x, np.ndarray) and x.ndim == 1 and x.dtype == np.float64:
            y = super(WeightingLO, self).matvec(x)
            x[...] = y                                     # in-place semantics of the reference
            return x
        return super(WeightingLO, self).matvec(x)


class BlockDiagonalLinearOperator(lp.LinearOperator):
    """Generic block-diagonal of operators -- interfaces/blkop.py:140-242 (kept for API
    compatibility; BlockLO overrides the application with single-launch kernels)."""

    def __init__(self, blocks, **kwargs):
        try:
            for block in blocks:
                block.shape
        except (TypeError, AttributeError):
            raise ValueError("blocks should be a flattened list of operators")
        self._blocks_list = blocks
        nargin = sum(b.shape[-1] for b in blocks)
        nargout = sum(b.shape[0] for b in blocks)
        symmetric = all(b.symmetric for b in blocks)
        kwargs.pop("symmetric", None)
        super(BlockDiagonalLinearOperator, self).__init__(
            nargin, nargout, symmetric=symmetric, matvec=lambda x: self._blk_apply(x, False),
            rmatvec=lambda x: self._blk_apply(x, True), device=True, **kwargs)

    def _blk_apply(self, x, transpose):
        outs = []
        c0 = 0
        for B in self._blocks_list:
            op = B.T if transpose else B
            c1 = c0 + op.shape[-1]
            outs.append(op._apply(dv.to_dev_f64(x[c0:c1])))
            c0 = c1
        return torch.cat(outs)

    @property
    def blocks(self):
        return self._blocks_list

    def __getitem__(self, idx):
        blks = self._blocks_list[idx]
        if isinstance(idx, slice):
            return BlockDiagonalLinearOperator(blks)
        return blks


class BlockLO(BlockDiagonalLinearOperator):
    """N^-1 as a block-diagonal operator -- interfaces/linearoperators.py:627-697.

    ``BlockLO(blocksize, t, offdiag=False)``; attributes ``blocklist, diag, covnoise, isoffdiag,
    blocksize``.  ``offdiag=False``: block i is ``t[i]`` times the identity and ``diag`` is the
    per-sample weight vector (a lazy ``BlockWeights``).  ``offdiag=True``: block i is the banded
    Toeplitz of ``t[i]``.  ``blocksize`` may be a list of per-block sizes (the intent of
    tests/test_toeplitz_vector_multiplication.py:12).  One kernel launch applies all blocks.
    """

    def __init__(self, blocksize, t, offdiag=False):
        self.__isoffdiag = offdiag
        self.blocksize = blocksize
        self.covnoise = t
        nb = len(t)
        self._blk = _Blocks(_block_starts(blocksize, nb))
        self._blocklist = None
        if offdiag:
            bands = [np.atleast_1d(np.asarray(a, dtype=np.float64)) for a in t]
            self._nband = max(len(a) for a in bands)
            band = np.zeros((nb, self._nband))
            for i, a in enumerate(bands):
                band[i, :len(a)] = a
            self._band_host = band
            self._band_dev = None
            self.diag = bands[0].copy()                  # linearoperators.py:673 (sic: t[0] only)
        else:
            self._w_host = np.asarray([float(v) for v in t], dtype=np.float64)
            self._w_dev = None
            self.diag = BlockWeights(self._w_host, self._blk.starts)
        nt = self._blk.nt
        lp.LinearOperator.__init__(self, nt, nt, matvec=self._apply_all, rmatvec=self._apply_all,
                                   symmetric=True, device=True)

    @property
    def isoffdiag(self):
        return self.__isoffdiag

    @property
    def blocklist(self):
        if self._blocklist is None:
            sizes = np.diff(self._blk.starts)
            if self.isoffdiag:
                self._blocklist = [ToeplitzLO(a, int(sz)) for a, sz in zip(self.covnoise, sizes)]
            else:
                self._blocklist = [lp.DiagonalOperator(np.full(int(sz), v)) for v, sz in zip(self._w_host, sizes)]
        return self._blocklist

    @property
    def blocks(self):
        return self.blocklist

    _blocks_list = property(lambda self: self.blocklist)

    def weights_dev(self):
        if self._w_dev is None:
            self._w_dev = dv.to_dev_f64(self._w_host)
        return self._w_dev

    def _toeplitz_state(self):
        """Device band and (for wide bands) the overlap-save FFT tables, built at first use."""
        if self._band_dev is None:
            self._band_dev = dv.to_dev_f64(self._band_host.reshape(-1))
            self._fft = (_ToeplitzFFT(self._band_host, self._nband)
                         if self._nband >= TOEPLITZ_FFT_MIN_BAND else None)
        return self._fft

    def _apply_all(self, x):
        if x.numel() != self._blk.nt:
            raise lp.ShapeError("Multiplying with vector of wrong shape.")
        nb, bs, startp = self._blk.args()
        if self.isoffdiag:
            self._toeplitz_state()
            return _toeplitz_apply(self._band_dev, self._nband, self._blk, x, self._fft)
        out = torch.empty_like(x)
        dv.call("cm2_noise_white_apply", dv.ptr(self.weights_dev()), nb, bs, startp, dv.ptr(x), dv.ptr(out),
                x.numel(), _stream())
        return out


def flatten_subscans(subscans, tstart, nsamples, nbolos):
    """The reference's (CES, detector, subscan) triple loop (linearoperators.py:134-140, 167) as one
    sorted list of segments [start, end) in the CES-major, detector-major, time-minor TOD."""
    starts, ends = [], []
    offset = 0
    for subsc, ts, ns, nb in zip(subscans, tstart, nsamples, nbolos):
        subsc = np.asarray(subsc, dtype=np.int64)
        ts = np.asarray(ts, dtype=np.int64)
        det0 = offset + int(ns) * np.arange(int(nb), dtype=np.int64)       # :139
        s = (det0[:, None] + ts[None, :]).reshape(-1)
        starts.append(s)
        ends.append(s + np.tile(subsc, int(nb)))
        offset += int(nb) * int(ns)
    if not starts:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    return np.concatenate(starts), np.concatenate(ends)


FILTER_STAGED = True        # subscan staged in shared memory (cm2_filter_poly_apply) also for poly_order = 0


class _NoPool(object):
    """Stand-in for the ``multiprocessing.Pool`` the reference keeps in ``FilterLO.procs`` when
    ``poly_order > 0`` (linearoperators.py:280): scripts that close / terminate it keep working."""

    def __init__(self, npool):
        self._processes = npool

    def close(self):
        pass

    terminate = join = close


class FilterLO(lp.LinearOperator):
    """Subscan filter -- interfaces/linearoperators.py:94-322.

    ``poly_order = 0``: offset removal (``mult`` :129-168).  ``poly_order > 0``: Legendre polynomials
    up to that order (``polyfilter`` :170-204; the reference's ``multiprocessing.Pool`` of ``npool``
    workers, :246-261, 286-322, is a CPU implementation detail -- ``npool`` is accepted and ignored).
    Same constructor; the (CES, detector, subscan) triple loop of the reference is flattened at
    construction into one list of segments [start, end) and ONE kernel launch applies them all.
    """

    def __init__(self, size, subscan_nsample, samples_per_bolopair, bolos_per_ces, pix_samples,
                 poly_order=0, npool=4):
        dv.require_cuda()
        self.n = size
        self.nsamples = samples_per_bolopair
        self.nbolos = bolos_per_ces
        self.subscans = subscan_nsample[0]
        self.tstart = subscan_nsample[1]
        if not (type(self.nsamples) is list):
            self.nsamples = [self.nsamples]
            self.nbolos = [self.nbolos]
            self.subscans = [self.subscans]
            self.tstart = [self.tstart]
        self.pixels = pix_samples
        self.poly_order = int(poly_order)
        if self.poly_order < 0:
            raise ValueError("poly_order must be >= 0")
        max_order = int(dv.call("cm2_filter_poly_max_order"))
        if self.poly_order > max_order:
            raise NotImplementedError("poly_order=%d: the device filter supports orders 0..%d"
                                      % (self.poly_order, max_order))
        self._seg_start_host, self._seg_end_host = flatten_subscans(self.subscans, self.tstart, self.nsamples,
                                                                    self.nbolos)
        ss, se = self._seg_start_host, self._seg_end_host
        if len(se) and (se.max() > size or ss.min() < 0):
            raise lp.ShapeError("subscan table exceeds the TOD size")
        self._seg_start = dv.to_dev(ss, torch.int64)
        self._seg_end = dv.to_dev(se, torch.int64)
        self.nseg = len(ss)
        self._max_seg_len = int((se - ss).max()) if self.nseg else 0
        # sorted, non-overlapping, non-negative lengths: the kernel then writes every output sample itself
        self._sorted = bool(self.nseg == 0 or (np.all(se >= ss) and np.all(ss[1:] >= se[:-1])))
        self._pix_dev = dv.pix_to_dev(pix_samples)
        self._legendres = None
        if self.poly_order > 0:
            self.procs = _NoPool(npool)
        matvec = self.mult if self.poly_order == 0 else self.polyfilter
        super(FilterLO, self).__init__(nargin=size, nargout=size, matvec=matvec, symmetric=False,
                                       device=True)

    def _staged(self, d):
        out = torch.empty_like(d)
        dv.call("cm2_filter_poly_apply", dv.ptr(self._pix_dev), dv.ptr(self._seg_start), dv.ptr(self._seg_end),
                self.nseg, self._max_seg_len, self.poly_order, int(self._sorted), dv.ptr(d), dv.ptr(out),
                d.numel(), _stream())
        return out

    def mult(self, d):                                    # :129-168
        if FILTER_STAGED:
            return self._staged(d)
        out = torch.empty_like(d)
        dv.call("cm2_filter_offset_apply", dv.ptr(self._pix_dev), dv.ptr(self._seg_start), dv.ptr(self._seg_end),
                self.nseg, dv.ptr(d), dv.ptr(out), d.numel(), _stream())
        return out

    def polyfilter(self, d):                              # :170-204
        return self._staged(d)

    polyfilter_multithreads = polyfilter                  # :246-261

    def compute_legendres(self):                          # :206-213 (host tables; the kernel evaluates
        from .utilities import get_legendre_polynomials   # the recurrence on the fly and never reads them)
        sizes = []
        for array in self.subscans:
            for i in array:
                if int(i) not in sizes:
                    sizes.append(int(i))
        self._legendres = {size: get_legendre_polynomials(self.poly_order, size) for size in sizes}

    @property
    def legendres(self):
        if self._legendres is None:
            self.compute_legendres()
        return self._legendres


# =============================================================================================
# fused A-matvecs: the factor chains [P.T, P], [P.T, N_white, P], [P.T, F, P] collapse to one
# kernel without a TOD temporary
# =============================================================================================
TOD_INTERLEAVE_MIN_MAP_BYTES = 100e6   # x and y together; measured: 61 MB (nside 1024 patch) is faster in time order (2.26 vs 2.39 ms per 5e8 samples), 246 MB (nside 2048) interleaved (4.00 vs 4.40 ms per 1e9)


def _tod_streams(P, samples_per_timeline):
    """``nstreams`` of the single-pass A-matvecs (include/cosmomap2_b200.h): the number of detector timelines
    when x and y together are too large to stay in L2 next to the TOD stream, else 1 (time order)."""
    ns = int(samples_per_timeline or 0)
    if ns <= 0 or 2 * 8 * P.pol * P.ncols < TOD_INTERLEAVE_MIN_MAP_BYTES:
        return 1
    k = P.nrows // ns
    return int(k) if k > 1 and k * ns == P.nrows else 1


def _filter_timeline(F):
    """Samples per detector timeline of a FilterLO (its ``samples_per_bolopair``: a number, or one per CES)."""
    ns = np.atleast_1d(np.asarray(F.nsamples)).astype(np.int64)
    return int(ns[0]) if ns.size and np.all(ns == ns[0]) else 0


WHITE_STAGE_RUN_RANGE = (3.0, 6.0)   # mean run length for which the staged scatter wins (measured, tools/pattern_probe.py)
WHITE_STAGE_MIN_CONTIGUITY = 0.9     # ... on sweeps along pixel rows only (a tilted scan changes row at most pixel changes)
WHITE_STAGE_WINDOW = 288             # pixels per warp tile
WHITE_SORT_BELOW_RUN = 3.0           # below: the white A-matvec runs over a pixel-sorted copy of the pointing
WHITE_PACK_BELOW_RUN = 16.0          # register scatter in time order along pixel rows with shorter runs: packed pixel
                                     # stream (measured, tools/pack_probe.py: faster at 8 samples per pixel crossing,
                                     # slower at 32, on a tilted scan and in the detector-interleaved order)


class _FusedWhiteA(lp.LinearOperator):
    """``P^T diag(w) P`` in one pass over the TOD (cm2_amatvec_white).  The scatter is chosen from the pointing
    (SparseLO.mean_run_length, at first use):

    * runs of >= 6 samples (a raster scan at the usual sampling), or sweeps that do not follow pixel rows: run
      compression in registers + warp merge;
    * runs of 3-6 samples along pixel rows: the same pass with the scatter staged through a shared-memory window
      and flushed with coalesced REDs (cm2_amatvec_white_set_stage; 0.55 -> 0.46 ms per 1e8 samples at 4 samples
      per pixel);
    * shorter (1-2 samples per pixel crossing, or the random pointing of the reference's tests,
      utilities/utilities_functions.py:111-122): one atomic and one gather per sample and component would bound
      the pass (0.96 / 1.83 / 2.2 ms per 1e8 samples at 2 / 1 samples per pixel / random); white noise has no
      time-domain structure, so the pass runs over a copy of the pointing SORTED BY PIXEL with per-sample
      weights instead (28 B/sample, every pixel one run: 0.45 ms).  Set-up: one stable sort; memory: a second
      copy of the pointing.

    In time order, for runs of fewer than 16 samples along pixel rows (configs[1]: 8), the register scatter reads the
    pixel ids from a packed stream built at first use (cm2_pack_pointing: two base pixels and a 2-bit code per sample,
    1 byte per sample instead of 4; lanes it cannot encode read the int32 ids), 17 instead of 20 B/sample.  It lives
    as long as the operator: nt bytes of device memory (100 MB per 1e8 samples)."""

    def __init__(self, P, N):
        self.P, self.N = P, N
        n = P.pol * P.ncols
        bs = N._blk.blocksize if N is not None else 0
        self._streams = _tod_streams(P, bs)
        self._mode = None
        self._sorted = None
        self._packed = None
        self.nescape = 0
        super(_FusedWhiteA, self).__init__(n, n, matvec=self._run, symmetric=True, device=True)

    def _choose(self):
        run, contig = self.P.run_statistics()
        if run < WHITE_SORT_BELOW_RUN and self.P.nrows > 0:
            self._mode = "sorted"
            self._build_sorted()
        elif WHITE_STAGE_RUN_RANGE[0] <= run < WHITE_STAGE_RUN_RANGE[1] and contig >= WHITE_STAGE_MIN_CONTIGUITY:
            self._mode = "staged"
        else:
            self._mode = "registers"
            if self._streams == 1 and run < WHITE_PACK_BELOW_RUN and contig >= WHITE_STAGE_MIN_CONTIGUITY:
                self._build_packed()

    def _build_packed(self):
        P = self.P
        self._packed = torch.empty(max((P.nrows + 7) // 8, 1), dtype=torch.int64, device=P._pix_dev.device)
        nesc = torch.empty(1, dtype=torch.int64, device=P._pix_dev.device)
        dv.call("cm2_pack_pointing", dv.ptr(P._pix_dev), P.nrows, dv.ptr(self._packed), dv.ptr(nesc), _stream())
        self.nescape = int(nesc.item())

    def tod_bytes(self):
        """Bytes of TOD one apply reads: 20 per sample, or with the packed pixel stream 17 per sample plus the
        32 bytes of int32 ids of every escape lane."""
        if self._mode is None:
            self._choose()
        if self._packed is not None:
            return 17 * self.P.nrows + 32 * self.nescape
        return 20 * self.P.nrows

    def _build_sorted(self):
        P, N = self.P, self.N
        order = torch.sort(P._pix_dev, stable=True).indices                  # one-off set-up (flagged first)
        nflag = int((P._pix_dev < 0).sum().item())
        order = order[nflag:]
        nts = int(order.numel())
        pad = (-nts) % 8                                                      # keep 32-byte alignment rules simple
        pix = torch.full((nts + pad,), -1, dtype=torch.int32, device=order.device)
        pix[:nts] = P._pix_dev[order]
        cs = sn = None
        if P.pol > 1:
            cs, sn = dv.zeros_f64(nts + pad), dv.zeros_f64(nts + pad)
            cs[:nts] = P._cos_dev[order]
            sn[:nts] = P._sin_dev[order]
        w = None
        if N is not None:
            starts = dv.to_dev(N._blk.starts, torch.int64)
            blk = torch.bucketize(order, starts[1:], right=True)
            w = dv.zeros_f64(nts + pad)
            w[:nts] = N.weights_dev()[blk]
        self._sorted = (pix, cs, sn, w, nts + pad)

    def _run(self, x):
        P = self.P
        if self._mode is None:
            self._choose()
        y = dv.out_f64(P.ncols * P.pol)
        if self._mode == "sorted":
            pix, cs, sn, w, nts = self._sorted
            dv.call("cm2_amatvec_white", dv.ptr(pix), None, dv.ptr(cs), dv.ptr(sn), nts, P.pol,
                    dv.ptr(w) if w is not None else None, nts if w is not None else 0, 1, None, dv.ptr(x), dv.ptr(y),
                    P.ncols, 1, _stream())
            return y
        if self.N is None:
            w, nb, bs, startp = None, 0, 0, None
        else:
            w = dv.ptr(self.N.weights_dev())
            nb, bs, startp = self.N._blk.args()
        if self._mode == "staged":
            dv.call("cm2_amatvec_white_set_stage", WHITE_STAGE_WINDOW)
        try:
            dv.call("cm2_amatvec_white", dv.ptr(P._pix_dev), dv.ptr(self._packed),
                    dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows, P.pol, w, nb, bs, startp, dv.ptr(x), dv.ptr(y),
                    P.ncols, self._streams, _stream())
        finally:
            if self._mode == "staged":
                dv.call("cm2_amatvec_white_set_stage", 0)
        return y


FILTER_RUN_TABLE = True     # single-TOD-pass P^T F P through the run-compressed u_k table


def _tile_tables(seg_start, seg_end, nseg, nt):
    """Per 256-sample tile of the TOD: the first segment whose end lies beyond the tile's first sample
    (int32) and a flag -- 0 = the tile lies in a gap, 1 = inside that segment, 2 = a boundary falls inside."""
    dev = seg_start.device
    ntiles = (nt + 255) // 256
    tile_t0 = torch.arange(ntiles, dtype=torch.int64, device=dev) * 256
    tile_seg = torch.searchsorted(seg_end, tile_t0, right=True)
    kk = torch.clamp(tile_seg, max=nseg - 1)
    a, b = seg_start[kk], seg_end[kk]
    t1 = torch.clamp(tile_t0 + 256, max=nt)
    inside = (tile_seg < nseg) & (a <= tile_t0) & (t1 <= b)
    outside = (tile_seg >= nseg) | (a >= t1)
    tile_flag = torch.full((ntiles,), 2, dtype=torch.uint8, device=dev)
    tile_flag[inside] = 1
    tile_flag[outside] = 0
    return tile_seg.to(torch.int32), tile_flag


def _build_filter_runs(P, F):
    """Run-compressed table of u_k = P^T 1_k per subscan + the per-tile subscan lookup (csrc/filter_runs.cu),
    built on the device; False when the subscans are unsorted or the pointing has no runs."""
    nt, st = P.nrows, _stream()
    dev = P._pix_dev.device
    ss, se = F._seg_start_host, F._seg_end_host
    if F.nseg == 0 or np.any(ss[1:] < se[:-1]):
        return False                                    # unsorted / overlapping subscans
    flags = torch.empty(max(nt, 1), dtype=torch.int32, device=dev)
    pixm = torch.empty(max(nt, 1), dtype=torch.int32, device=dev)
    dv.call("cm2_filter_runs_mark", dv.ptr(P._pix_dev), dv.ptr(F._seg_start), dv.ptr(F._seg_end), F.nseg, nt,
            dv.ptr(flags), dv.ptr(pixm), st)
    runidx = torch.empty(max(nt, 1), dtype=torch.int32, device=dev)
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    scratch = torch.empty(int(dv.call("cm2_scan_scratch_bytes", nt)) // 8 + 1, dtype=torch.int64, device=dev)
    dv.call("cm2_weights_old2new", dv.ptr(flags), nt, dv.ptr(runidx), dv.ptr(count), dv.ptr(scratch), st)
    nruns = int(count.item())
    del flags, scratch
    if nruns == 0 or 2 * nruns > nt:
        return False
    run_pix = torch.empty(nruns, dtype=torch.int32, device=dev)
    run_mom = torch.empty(3 * nruns, dtype=torch.float64, device=dev)
    seg_first = torch.empty(max(F.nseg, 1), dtype=torch.int64, device=dev)
    seg_nruns = torch.empty(max(F.nseg, 1), dtype=torch.int32, device=dev)
    dv.call("cm2_filter_runs_fill", dv.ptr(pixm), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.pol,
            dv.ptr(F._seg_start), dv.ptr(F._seg_end), F.nseg, dv.ptr(runidx), dv.ptr(run_pix), dv.ptr(run_mom),
            dv.ptr(seg_first), dv.ptr(seg_nruns), st)
    del pixm, runidx
    tile_seg, tile_flag = _tile_tables(F._seg_start, F._seg_end, F.nseg, nt)
    mu = torch.empty(max(F.nseg, 1), dtype=torch.float64, device=dev)
    return dict(run_pix=run_pix, run_mom=run_mom, seg_first=seg_first, seg_nruns=seg_nruns, nruns=nruns,
                tile_seg=tile_seg, tile_flag=tile_flag, mu=mu)


def _filter_runs(P, F):
    """The table of _build_filter_runs, built once per (P, F) pair and shared by the fused operators."""
    if not FILTER_RUN_TABLE:
        return False
    cache = F.__dict__.setdefault("_run_tables", {})
    key = (id(P), P._pix_dev.data_ptr())
    if key not in cache:
        cache[key] = _build_filter_runs(P, F)
    return cache[key]


class _FusedFilterA(lp.LinearOperator):
    """P^T F P as one operator.  Default: the subscan means from the run-compressed table of
    u_k = P^T 1_k (csrc/filter_runs.cu), then ONE fused gather/scatter pass over the TOD; the table
    is built on the device at first use and is used when the segments are sorted and the scan has
    runs (>= 2 samples per run on average).  Otherwise: the two-pass kernel cm2_amatvec_filter."""

    def __init__(self, P, F):
        self.P, self.F = P, F
        self._runs = None
        n = P.pol * P.ncols
        super(_FusedFilterA, self).__init__(n, n, matvec=self._run, symmetric=True, device=True)

    def _run(self, x):
        P, F = self.P, self.F
        y = dv.out_f64(P.ncols * P.pol)
        if self._runs is None:
            self._runs = _filter_runs(P, F)
        rt = self._runs
        if rt:
            dv.call("cm2_filter_seg_mean", dv.ptr(rt["run_pix"]), dv.ptr(rt["run_mom"]), dv.ptr(rt["seg_first"]),
                    dv.ptr(rt["seg_nruns"]), F.nseg, P.pol, dv.ptr(x), dv.ptr(rt["mu"]), _stream())
            dv.call("cm2_amatvec_filter_mu", dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows,
                    P.pol, dv.ptr(F._seg_start), dv.ptr(F._seg_end), dv.ptr(rt["mu"]), dv.ptr(rt["tile_seg"]),
                    dv.ptr(rt["tile_flag"]), F.nseg, dv.ptr(x), dv.ptr(y), P.ncols,
                    _tod_streams(P, _filter_timeline(F)), _stream())
            return y
        dv.call("cm2_amatvec_filter", dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows, P.pol,
                dv.ptr(F._seg_start), dv.ptr(F._seg_end), F.nseg, dv.ptr(x), dv.ptr(y), P.ncols, _stream())
        return y


FILTER_POLY_RUN_TABLE = True      # single-TOD-pass P^T F_K P through a Legendre run table (order 1: 0.61 vs 0.79 ms per 1e8 samples)
POLY_RUN_MIN_PIVOT = 0.02         # subscans whose scaled Gram matrix has a smaller Cholesky pivot keep the per-subscan kernel


def _build_poly_runs(P, F):
    """Set-up of the single-pass Legendre A-matvec (csrc/filter_runs.cu): per subscan W (c = W S) and its
    conditioning; the subscans the reference filters and whose Gram matrix is well conditioned ('easy')
    get a run table of Legendre-weighted sums and tile tables; ill-conditioned ones ('hard': most of the
    subscan flagged) stay with the per-subscan kernel; the others contribute nothing (the reference skips
    them).  False when the path does not apply."""
    order = F.poly_order
    nk = order + 1
    if not (1 <= order <= 4 and F._sorted and F.nseg > 0):
        return False
    nt, st = P.nrows, _stream()
    dev = P._pix_dev.device
    ss, se = F._seg_start_host, F._seg_end_host
    W_all = torch.empty(F.nseg * nk * nk, dtype=torch.float64, device=dev)
    info = torch.empty(2 * F.nseg, dtype=torch.float64, device=dev)
    dv.call("cm2_filter_poly_gram", dv.ptr(P._pix_dev), dv.ptr(F._seg_start), dv.ptr(F._seg_end), F.nseg, order,
            dv.ptr(W_all), dv.ptr(info), st)
    info_h = dv.to_host(info).reshape(-1, 2)
    cnt, piv = info_h[:, 0], info_h[:, 1]
    alive = cnt > order
    easy = alive & ((cnt == (se - ss)) | (piv >= POLY_RUN_MIN_PIVOT))
    hard = alive & ~easy
    ie, ih = np.nonzero(easy)[0], np.nonzero(hard)[0]
    ne = len(ie)
    if ne == 0:
        return False
    seg_start = dv.to_dev(ss[ie], torch.int64)
    seg_end = dv.to_dev(se[ie], torch.int64)
    W = W_all.view(F.nseg, nk * nk)[dv.to_dev(ie, torch.int64)].contiguous().view(-1)
    del W_all, info
    flags = torch.empty(max(nt, 1), dtype=torch.int32, device=dev)
    pixm = torch.empty(max(nt, 1), dtype=torch.int32, device=dev)
    dv.call("cm2_filter_runs_mark", dv.ptr(P._pix_dev), dv.ptr(seg_start), dv.ptr(seg_end), ne, nt,
            dv.ptr(flags), dv.ptr(pixm), st)
    runidx = torch.empty(max(nt, 1), dtype=torch.int32, device=dev)
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    scratch = torch.empty(int(dv.call("cm2_scan_scratch_bytes", nt)) // 8 + 1, dtype=torch.int64, device=dev)
    dv.call("cm2_weights_old2new", dv.ptr(flags), nt, dv.ptr(runidx), dv.ptr(count), dv.ptr(scratch), st)
    nruns = int(count.item())
    del flags, scratch
    if nruns == 0 or 2 * nruns > nt:
        return False
    run_pix = torch.empty(nruns, dtype=torch.int32, device=dev)
    run_mom = torch.empty(3 * nk * nruns, dtype=torch.float64, device=dev)
    seg_first = torch.empty(ne, dtype=torch.int64, device=dev)
    seg_nruns = torch.empty(ne, dtype=torch.int32, device=dev)
    dv.call("cm2_filter_poly_runs_fill", dv.ptr(pixm), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.pol,
            dv.ptr(seg_start), dv.ptr(seg_end), ne, order, dv.ptr(runidx), dv.ptr(run_pix), dv.ptr(run_mom),
            dv.ptr(seg_first), dv.ptr(seg_nruns), st)
    del pixm, runidx
    tile_seg, tile_flag = _tile_tables(seg_start, seg_end, ne, nt)
    rt = dict(nseg=ne, seg_start=seg_start, seg_end=seg_end, W=W, run_pix=run_pix, run_mom=run_mom,
              seg_first=seg_first, seg_nruns=seg_nruns, nruns=nruns, tile_seg=tile_seg, tile_flag=tile_flag,
              coef=torch.empty(ne * nk, dtype=torch.float64, device=dev), nhard=len(ih))
    if len(ih):
        rt["hard_start"] = dv.to_dev(ss[ih], torch.int64)
        rt["hard_end"] = dv.to_dev(se[ih], torch.int64)
        rt["hard_maxlen"] = int((se[ih] - ss[ih]).max())
    return rt


class _FusedPolyFilterA(lp.LinearOperator):
    """P^T F_K P for the Legendre filter (poly_order 1..4) as one kernel: one CTA per subscan, the
    subscan's P x kept in shared memory between the moment pass and the scatter pass.  With
    ``FILTER_POLY_RUN_TABLE`` (experimental) the well-conditioned subscans go through the single-TOD-pass
    scheme of the offset filter instead: coefficients from a Legendre run table, then one streaming pass."""

    def __init__(self, P, F):
        self.P, self.F = P, F
        self._runs = None
        n = P.pol * P.ncols
        super(_FusedPolyFilterA, self).__init__(n, n, matvec=self._run, symmetric=True, device=True)

    @staticmethod
    def supported(P, F):
        return (1 <= F.poly_order <= int(dv.call("cm2_amatvec_filter_poly_max_order")) and F._sorted
                and (F._max_seg_len // 256 + 2) * 256 * 12 <= 200 * 1024)

    def _per_subscan(self, seg_start, seg_end, nseg, max_len, x, y):
        P, F = self.P, self.F
        dv.call("cm2_amatvec_filter_poly", dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows,
                P.pol, dv.ptr(seg_start), dv.ptr(seg_end), nseg, max_len, F.poly_order, dv.ptr(x),
                dv.ptr(y), P.ncols, _stream())
        return y

    def _run(self, x):
        P, F = self.P, self.F
        y = dv.out_f64(P.ncols * P.pol)
        if self._runs is None:
            self._runs = _build_poly_runs(P, F) if FILTER_POLY_RUN_TABLE else False
        rt = self._runs
        if not rt:
            return self._per_subscan(F._seg_start, F._seg_end, F.nseg, F._max_seg_len, x, y)
        dv.call("cm2_filter_poly_seg_coef", dv.ptr(rt["run_pix"]), dv.ptr(rt["run_mom"]), dv.ptr(rt["seg_first"]),
                dv.ptr(rt["seg_nruns"]), rt["nseg"], P.pol, F.poly_order, dv.ptr(rt["W"]), dv.ptr(x),
                dv.ptr(rt["coef"]), _stream())
        dv.call("cm2_amatvec_filter_poly_mu", dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows,
                P.pol, dv.ptr(rt["seg_start"]), dv.ptr(rt["seg_end"]), dv.ptr(rt["coef"]), dv.ptr(rt["tile_seg"]),
                dv.ptr(rt["tile_flag"]), rt["nseg"], F.poly_order, dv.ptr(x), dv.ptr(y), P.ncols, 0,
                _tod_streams(P, _filter_timeline(F)), _stream())
        if rt["nhard"]:
            y2 = self._per_subscan(rt["hard_start"], rt["hard_end"], rt["nhard"], rt["hard_maxlen"], x,
                                   dv.empty_f64(P.ncols * P.pol))
            dv.call("cm2_axpby", 1.0, dv.ptr(y2), 1.0, dv.ptr(y), y.numel(), _stream())
        return y


class _FusedFilterP(lp.LinearOperator):
    """F P (offset filter) as one TOD pass: the subscan means of P x come from the run table, so
    d = P x - mu_seg is written directly (the head of chains such as P.T*F*N*F*P).  Falls back to the
    two operators when the run table cannot be used (unsorted subscans, run-free pointing)."""

    def __init__(self, P, F):
        self.P, self.F = P, F
        self._runs = None
        super(_FusedFilterP, self).__init__(P.pol * P.ncols, P.nrows, matvec=self._run, symmetric=False, device=True)

    def _run(self, x):
        P, F = self.P, self.F
        if self._runs is None:
            self._runs = _filter_runs(P, F)
        rt = self._runs
        if not rt:
            return F._apply(P._apply(x))
        d = dv.empty_f64(P.nrows)
        dv.call("cm2_filter_seg_mean", dv.ptr(rt["run_pix"]), dv.ptr(rt["run_mom"]), dv.ptr(rt["seg_first"]),
                dv.ptr(rt["seg_nruns"]), F.nseg, P.pol, dv.ptr(x), dv.ptr(rt["mu"]), _stream())
        dv.call("cm2_pointing_filter_mu", dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows, P.pol,
                dv.ptr(F._seg_start), dv.ptr(F._seg_end), dv.ptr(rt["mu"]), dv.ptr(rt["tile_seg"]),
                dv.ptr(rt["tile_flag"]), F.nseg, dv.ptr(x), dv.ptr(d), _stream())
        return d


class _FusedToeplitzA(lp.LinearOperator):
    """P^T N P for a short-band Toeplitz N = BlockLO(offdiag=True) (the reference tests' composition,
    tests/test_2level_preconditioner.py:16-29) as ONE kernel without a TOD temporary."""

    def __init__(self, P, N):
        self.P, self.N = P, N
        n = P.pol * P.ncols
        super(_FusedToeplitzA, self).__init__(n, n, matvec=self._run, symmetric=True, device=True)

    @staticmethod
    def supported(P, N):
        return (N.isoffdiag and N.shape[0] == P.nrows
                and N._nband <= int(dv.call("cm2_amatvec_toeplitz_max_band")))

    def _run(self, x):
        P, N = self.P, self.N
        y = dv.out_f64(P.ncols * P.pol)
        if N._band_dev is None:
            N._band_dev = dv.to_dev_f64(N._band_host.reshape(-1))
            N._fft = None
        nb, bs, startp = N._blk.args()
        dv.call("cm2_amatvec_toeplitz", dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows, P.pol,
                dv.ptr(N._band_dev), int(N._nband), nb, bs, startp, dv.ptr(x), dv.ptr(y), P.ncols, _stream())
        return y


def _is_pt(op):
    return getattr(op, "_adjoint_of", None) is not None and isinstance(op._adjoint_of, SparseLO)


fusion_enabled = True
FUSE_TOEPLITZ_A = True      # [P.T, N_toeplitz (<= 9 coefficients), P] -> cm2_amatvec_toeplitz
FUSE_FILTER_P = True        # [F_offset, P] -> cm2_pointing_filter_mu


@lp.register_fuser
def _fuse_pointing(factors):
    if not fusion_enabled:
        return None
    n = len(factors)
    for i in range(n):
        if not _is_pt(factors[i]):
            continue
        P = factors[i]._adjoint_of
        # [P.T, P]
        if i + 1 < n and factors[i + 1] is P:
            return factors[:i] + [_FusedWhiteA(P, None)] + factors[i + 2:]
        if i + 2 < n and factors[i + 2] is P:
            mid = factors[i + 1]
            if isinstance(mid, BlockLO) and not mid.isoffdiag and mid.shape[0] == P.nrows:
                return factors[:i] + [_FusedWhiteA(P, mid)] + factors[i + 3:]
            if FUSE_TOEPLITZ_A and isinstance(mid, BlockLO) and _FusedToeplitzA.supported(P, mid):
                return factors[:i] + [_FusedToeplitzA(P, mid)] + factors[i + 3:]
            if (isinstance(mid, FilterLO) and mid.shape[0] == P.nrows
                    and mid._pix_dev.data_ptr() == P._pix_dev.data_ptr()):
                if mid.poly_order == 0:
                    return factors[:i] + [_FusedFilterA(P, mid)] + factors[i + 3:]
                if _FusedPolyFilterA.supported(P, mid):
                    return factors[:i] + [_FusedPolyFilterA(P, mid)] + factors[i + 3:]
    return None


@lp.register_fuser
def _fuse_filter_pointing(factors):
    """[..., F, P] with the offset filter and no P.T in front of it (that case is one kernel, above):
    F P becomes one TOD pass."""
    if not (fusion_enabled and FUSE_FILTER_P):
        return None
    for i in range(len(factors) - 1):
        F, P = factors[i], factors[i + 1]
        if (isinstance(F, FilterLO) and isinstance(P, SparseLO) and F.poly_order == 0 and F._sorted and F.nseg > 0
                and F.shape[0] == P.nrows and F._pix_dev.data_ptr() == P._pix_dev.data_ptr()):
            return factors[:i] + [_FusedFilterP(P, F)] + factors[i + 2:]
    return None


# =============================================================================================
# block-diagonal preconditioner
# =============================================================================================
def _moments_from(CES, n, pol):
    """Device [n][6] moment table {h,c,s,c2,cs,s2} from a ProcessTimeSamples (device-resident)
    or from any object exposing the reference's attribute arrays."""
    mom = getattr(CES, "_mom_dev", None)
    if mom is not None and getattr(CES, "pol", pol) == pol and mom.numel() >= 6 * n:
        return mom
    tab = np.zeros((max(n, 1), 6))
    if pol in (1, 3):
        tab[:n, 0] = np.asarray(CES.counts)[:n]
    if pol == 3:
        tab[:n, 1] = np.asarray(CES.cosine)[:n]
        tab[:n, 2] = np.asarray(CES.sine)[:n]
    if pol in (2, 3):
        tab[:n, 3] = np.asarray(CES.cos2)[:n]
        tab[:n, 4] = np.asarray(CES.sincos)[:n]
        tab[:n, 5] = np.asarray(CES.sin2)[:n]
    return dv.to_dev_f64(tab.reshape(-1))


class _PixelBlockLO(lp.LinearOperator):
    def _attrs_from(self, CES, n, pol):
        self.size = pol * n
        self.pixels = np.arange(n)
        self.pol = pol
        self._n = int(n)
        self._ces = CES
        self._mom_dev = _moments_from(CES, n, pol)

    # reference attribute names (linearoperators.py:717-726, 847-856)
    counts = property(lambda self: self._ces.counts)
    sin2 = property(lambda self: self._ces.sin2)
    cos2 = property(lambda self: self._ces.cos2)
    sincos = property(lambda self: self._ces.sincos)
    cos = property(lambda self: self._ces.cosine)
    sin = property(lambda self: self._ces.sine)


class BlockDiagonalLO(_PixelBlockLO):
    """Explicit P^T diag(N^-1) P, one small block per pixel -- linearoperators.py:700-746."""

    def __init__(self, CES, n, pol=1):
        dv.require_cuda()
        self._attrs_from(CES, n, pol)
        super(BlockDiagonalLO, self).__init__(nargin=self.size, nargout=self.size, matvec=self.mult,
                                              symmetric=True, device=True)

    def mult(self, x):
        y = torch.empty_like(x)
        dv.call("cm2_bdfwd_apply", dv.ptr(self._mom_dev), self._n, self.pol, dv.ptr(x), dv.ptr(y), _stream())
        return y


class BlockDiagonalPreconditionerLO(_PixelBlockLO):
    """M_BD = (P^T diag(N^-1) P)^-1, closed-form per-pixel inverse -- linearoperators.py:749-859.
    The inverse blocks are computed once at construction (the reference recomputes the determinant
    and the mask at every call, :792-795) with the same absolute threshold |det| > 1e-5."""

    def __init__(self, CES, n, pol=1):
        dv.require_cuda()
        self._attrs_from(CES, n, pol)
        self._inv_dev = torch.empty(max(self._n, 1) * 6, dtype=torch.float64, device=self._mom_dev.device)
        dv.call("cm2_bd_build", dv.ptr(self._mom_dev), self._n, pol, dv.ptr(self._inv_dev), _stream())
        super(BlockDiagonalPreconditionerLO, self).__init__(nargin=self.size, nargout=self.size,
                                                            matvec=self.mult, symmetric=True, device=True)

    def mult(self, x):                                    # :775-841
        y = torch.empty_like(x)
        dv.call("cm2_bd_apply", dv.ptr(self._inv_dev), self._n, self.pol, dv.ptr(x), dv.ptr(y), _stream())
        return y


class GroundFilterLO(lp.LinearOperator):
    """Ground-template filter I - G (G^T G)^-1 G^T -- interfaces/linearoperators.py:24-61.

    ``GroundFilterLO(ground)``: ``ground[t]`` = azimuth bin of sample t (-1 = flagged).  Attributes
    ``nbins, n, Pg`` as in the reference; ``mult`` is two kernels (bin sums by the run-aggregating
    pol-1 scatter, then the subtraction) instead of the three-operator chain ``G*invGtG*G.T``.

    ``comm=True`` (or a process group): the TOD is sharded over GPUs by detector while the ground
    template is common to all detectors, so the number of bins, the hits and -- at every application --
    the bin sums are summed over the ranks (two tiny all-reduces; ``Pg`` then is the local part only).
    """

    def counts_in_groundbins(self, g):                    # :26-46
        gd = g if (isinstance(g, torch.Tensor) and g.is_cuda and g.dtype == torch.int32) else dv.pix_to_dev(g)
        hits = torch.empty(max(self.nbins, 1), dtype=torch.int64, device=gd.device)
        dv.call("cm2_hits_i64", dv.ptr(gd), gd.numel(), self.nbins, dv.ptr(hits), _stream())
        if self._group is not None:
            from . import distributed
            distributed.all_reduce_sum_(hits, self._group_arg)
        self._hits_dev = hits
        return dv.to_host(hits[:self.nbins]).astype(np.float64)

    def mult(self, v):                                    # :48-49
        out = torch.empty_like(v)
        if self._group is None:
            dv.call("cm2_ground_filter_apply", dv.ptr(self._g_dev), self.n, self.nbins, dv.ptr(self._hits_dev),
                    dv.ptr(v), dv.ptr(self._bins), dv.ptr(out), _stream())
            return out
        from . import distributed
        dv.call("cm2_pointing_apply_t", dv.ptr(self._g_dev), None, None, self.n, 1, dv.ptr(v), dv.ptr(self._bins),
                self.nbins, _stream())
        distributed.all_reduce_sum_(self._bins, self._group_arg)
        dv.call("cm2_ground_filter_sub", dv.ptr(self._g_dev), self.n, self.nbins, dv.ptr(self._hits_dev),
                dv.ptr(self._bins), dv.ptr(v), dv.ptr(out), _stream())
        return out

    def __init__(self, ground, comm=None):                # :51-61
        dv.require_cuda()
        from . import distributed
        self._group_arg = None if comm is True else comm
        self._group = comm if (comm is not None and comm is not False and distributed.is_distributed(self._group_arg)) \
            else None
        self.n = len(ground)
        self._g_dev = dv.pix_to_dev(ground)
        if isinstance(ground, torch.Tensor):
            self.nbins = int(ground.max().item()) + 1 if self.n else 0
        else:
            self.nbins = int(np.max(ground)) + 1 if self.n else 0
        self.nbins = max(self.nbins, 0)
        if self._group is not None:                       # every rank works on the same bins
            nb = torch.tensor([self.nbins], dtype=torch.int64, device=self._g_dev.device)
            torch.distributed.all_reduce(nb, op=torch.distributed.ReduceOp.MAX, group=self._group_arg)
            self.nbins = int(nb.item())
        counts = self.counts_in_groundbins(self._g_dev)
        self._bins = dv.empty_f64(max(self.nbins, 1))
        G = SparseLO(self.nbins, self.n, self._g_dev)
        G.counts = counts
        invGtG = BlockDiagonalPreconditionerLO(G, self.nbins)
        self.Pg = (G * invGtG * G.T)
        super(GroundFilterLO, self).__init__(nargin=self.n, nargout=self.n, matvec=self.mult,
                                             symmetric=True, device=True)


class InverseLO(lp.LinearOperator):
    """A solver wrapped as the operator A^-1 -- interfaces/linearoperators.py:861-941."""

    def mult(self, x):
        y, info = self.method(self.A, x, M=self.preconditioner)
        self.isconverged(info)
        return y

    def isconverged(self, info):
        self.__converged = info
        return info == 0

    def __init__(self, A, method=None, preconditioner=None):
        super(InverseLO, self).__init__(nargin=A.shape[0], nargout=A.shape[1], matvec=self.mult,
                                        symmetric=True, device=True)
        self.A = A
        self.__method = method
        self.__preconditioner = preconditioner
        self.__converged = None

    method = property(lambda self: self.__method)
    converged = property(lambda self: self.__converged)
    preconditioner = property(lambda self: self.__preconditioner)


# =============================================================================================
# deflation / coarse operator / two-level preconditioner
# =============================================================================================
def _columns_dev(z):
    """n x r matrix (NumPy, np.matrix or CUDA tensor) -> (r, n) row-contiguous CUDA tensor, i.e.
    column-major n x r with ld = n, as the kernels read it."""
    if isinstance(z, torch.Tensor):
        return dv.to_dev_f64(z.t())
    return dv.to_dev_f64(np.ascontiguousarray(np.asarray(z, dtype=np.float64).T))


class DeflationLO(lp.LinearOperator):
    """Z y and Z^T x -- interfaces/linearoperators.py:1029-1065."""

    def __init__(self, z):
        dv.require_cuda()
        self.nrows, self.ncols = z.shape
        self._z_host = None if isinstance(z, torch.Tensor) else np.asarray(z)
        self._zt = _columns_dev(z)
        self._work = dv.empty_f64(int(dv.call("cm2_defl_work_doubles", int(self.ncols))))
        super(DeflationLO, self).__init__(nargin=self.ncols, nargout=self.nrows, matvec=self.mult,
                                          rmatvec=self.rmult, symmetric=False, device=True)

    @property
    def z(self):
        src = self._z_host if self._z_host is not None else dv.to_host(self._zt).T
        return [src[:, j] for j in range(self.ncols)]

    def mult(self, x):                                    # :1041-1050
        y = dv.empty_f64(self.nrows)
        dv.call("cm2_defl_z_apply", dv.ptr(self._zt), self.nrows, self.ncols, self.nrows, dv.ptr(x), 1.0, 0.0,
                None, dv.ptr(y), _stream())
        return y

    def rmult(self, x):                                   # :1051-1056
        out = dv.empty_f64(self.ncols)
        dv.call("cm2_defl_zt_apply", dv.ptr(self._zt), self.nrows, self.ncols, self.nrows, dv.ptr(x), 1,
                self.nrows, dv.ptr(out), dv.ptr(self._work), _stream())
        return out


class CoarseLO(lp.LinearOperator):
    """E = Z^T A Z and the action of E^-1 -- interfaces/linearoperators.py:946-1027.

    E (r x r) is accumulated on the device from Z and AZ; its r x r factorisation (LU, or eigh with
    eigenvalues |lambda/lambda_max| < 1e-6 discarded, :994-1015) is host LAPACK, and the resulting
    r x r inverse is applied on the device.
    """

    def __init__(self, Z, Az, r, apply="LU"):
        dv.require_cuda()
        zt = _columns_dev(Z)
        azt = _columns_dev(Az)
        n = zt.shape[1]
        from . import dense
        self.E = dv.to_host(dense.gram(zt[:r], azt[:r])).copy()   # E = Z^T (A Z), one pass over Z and AZ (DMMA)
        self.r = int(r)
        self.apply = apply
        if apply == "eig":
            self.setting_inverse_w_eigenvalues(self.E)
        elif apply == "LU":
            self._lu = lu_factor(self.E, check_finite=False)
            self.invE = lu_solve(self._lu, np.eye(self.r), check_finite=False)
        else:
            raise ValueError("apply must be 'LU' or 'eig'")
        self._einv_dev = dv.to_dev_f64(np.asfortranarray(self.invE).reshape(-1, order="F"))
        super(CoarseLO, self).__init__(nargin=r, nargout=r, matvec=self.mult, symmetric=True, device=True)

    def setting_inverse_w_eigenvalues(self, E):            # :986-1015
        eigenvals, W = eigh(E)
        lambda_max = max(eigenvals)
        diags = eigenvals * 0.
        nondegenerate = np.where(abs(eigenvals / lambda_max) > 1.e-6)[0]
        self.ndiscarded = len(eigenvals) - len(nondegenerate)
        diags[nondegenerate] = 1. / eigenvals[nondegenerate]
        self.invE = (W * diags[None, :]).dot(W.T)

    def mult(self, v):                                    # :969-984
        c = dv.empty_f64(self.r)
        dv.call("cm2_coarse_apply", dv.ptr(self._einv_dev), self.r, dv.ptr(v), dv.ptr(c), _stream())
        return c

    mult_eig = mult


M2_BANDED = True     # use the banded form of the two-level apply when Z is a subdomain (indicator) coarse space


def _banded_coarse_space(Zd, AZd, pol):
    """If ``Z`` is a subdomain coarse space -- every column the intensity indicator of a set of pixels, every pixel in
    at most one column (deflationlib.scan_coarse_space) -- and ``A Z`` is confined to each column's own band and its two
    cyclic neighbours, return ``(band, azb)``: band[npix] int32 (-1: pixel in no column) and azb[npix][pol][3], the
    entries of AZ in columns band-1, band, band+1.  ``None`` otherwise (checked exactly, entry by entry: nothing is
    dropped)."""
    zt, azt = Zd._zt, AZd._zt                       # (r, n), row k = column k
    r, n = zt.shape
    if pol not in (1, 3) or r < 3 or r > 64 or n % pol or azt.shape != zt.shape or Zd.nrows != n:
        return None
    npix = n // pol
    zi = zt[:, 0::pol]                               # (r, npix) intensity rows
    ones = zi == 1.0
    if not bool(((zi == 0.0) | ones).all().item()):
        return None
    cnt = ones.sum(dim=0)
    if int(cnt.max().item()) > 1:
        return None
    if pol == 3 and (bool((zt[:, 1::3] != 0).any().item()) or bool((zt[:, 2::3] != 0).any().item())):
        return None
    band = torch.where(cnt > 0, ones.to(torch.int8).argmax(dim=0), torch.full_like(cnt, -1)).to(torch.int32)
    del zi, ones
    bl = band.to(torch.int64)
    bsafe = torch.clamp(bl, min=0)
    azb = torch.zeros((npix, pol, 3), dtype=torch.float64, device=zt.device)
    nnz_kept = 0
    for k in range(pol):
        ak = azt[:, k::pol]                                                   # (r, npix)
        for o in range(3):
            col = torch.remainder(bsafe + (o - 1), r)
            vals = ak.gather(0, col.unsqueeze(0)).squeeze(0)
            vals = torch.where(bl >= 0, vals, torch.zeros_like(vals))
            azb[:, k, o] = vals
            nnz_kept += int((vals != 0).sum().item())
    nnz_all = int((azt != 0).sum().item())
    if nnz_kept != nnz_all:                          # some entry of AZ lies outside the three bands (or on an unbanded pixel)
        return None
    return band.contiguous(), azb.contiguous()


class TwoLevelPreconditionerLO(lp.LinearOperator):
    """M_2lvl = M_BD (I - AZ E^-1 Z^T) + Z E^-1 Z^T as ONE fused apply.

    The reference composes it with operator algebra (src/test_M2_precond_onto_real_data.py:109-112),
    which evaluates ``E*Zd.T*v`` twice; the algebraic composition still works with the classes
    above, and ``_fuse_two_level`` below rewrites it into this operator.  When ``Z`` is a subdomain coarse space
    (one non-zero per pixel, ``A Z`` banded: ``_banded_coarse_space``) the apply reads the band index and three
    entries of AZ per map element instead of 3 r doubles (cm2_m2_banded_apply).
    """

    def __init__(self, Mbd, Zd, AZd, E):
        self.Mbd, self.Zd, self.AZd, self.E = Mbd, Zd, AZd, E
        n = Zd.nrows
        self._work = dv.empty_f64(int(dv.call("cm2_defl_work_doubles", int(Zd.ncols))))
        self._banded = _banded_coarse_space(Zd, AZd, Mbd.pol) if M2_BANDED else None
        super(TwoLevelPreconditionerLO, self).__init__(n, n, matvec=self.mult, symmetric=True, device=True)

    def mult(self, v):
        Zd, M = self.Zd, self.Mbd
        y = torch.empty_like(v)
        if self._banded is not None:
            band, azb = self._banded
            dv.call("cm2_m2_banded_apply", dv.ptr(band), dv.ptr(azb), Zd.ncols, dv.ptr(self.E._einv_dev), dv.ptr(M._inv_dev),
                    M._n, M.pol, dv.ptr(v), dv.ptr(y), dv.ptr(self._work), _stream())
            return y
        dv.call("cm2_m2_apply", dv.ptr(Zd._zt), dv.ptr(self.AZd._zt), Zd.nrows, Zd.ncols, Zd.nrows,
                dv.ptr(self.E._einv_dev), dv.ptr(M._inv_dev), M._n, M.pol, dv.ptr(v), dv.ptr(y),
                dv.ptr(self._work), _stream())
        return y


def _is_zt(op, Zd=None):
    z = getattr(op, "_adjoint_of", None)
    return isinstance(z, DeflationLO) and (Zd is None or z is Zd)


@lp.register_sum_fuser
def _fuse_two_level(sum_op):
    """Recognise  Mbd*(I - AZd*E*Zd.T) + Zd*E*Zd.T  (src/test_M2_precond_onto_real_data.py:109-112)."""
    if not fusion_enabled or sum_op.sign != 1.0:
        return None
    a, b = sum_op.a, sum_op.b
    if not (isinstance(a, lp._ProductLO) and isinstance(b, lp._ProductLO)):
        return None
    fb = b.factors
    if not (len(fb) == 3 and isinstance(fb[0], DeflationLO) and isinstance(fb[1], CoarseLO) and _is_zt(fb[2], fb[0])):
        return None
    Zd, E = fb[0], fb[1]
    fa = a.factors
    if not (len(fa) == 2 and isinstance(fa[0], BlockDiagonalPreconditionerLO) and isinstance(fa[1], lp._SumLO)):
        return None
    R = fa[1]
    if not (R.sign == -1.0 and isinstance(R.a, lp.IdentityOperator) and isinstance(R.b, lp._ProductLO)):
        return None
    fr = R.b.factors
    if not (len(fr) == 3 and isinstance(fr[0], DeflationLO) and fr[1] is E and _is_zt(fr[2], Zd)):
        return None
    if fr[0].nrows != Zd.nrows or fr[0].ncols != Zd.ncols or fa[0].size != Zd.nrows:
        return None
    return TwoLevelPreconditionerLO(fa[0], Zd, fr[0], E)
