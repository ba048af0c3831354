"""
Destriping with a noise prior (DESIGN.md section 4f): the noise is white noise W^-1 plus offsets a_j on baselines of
L samples with covariance C_a, and the offsets are solved for in baseline space,

    (F^T W Z F + C_a^-1) a = F^T W Z d,     x = M_BD P^T W (d - F a),     Z = I - P M_BD P^T W,

with F spreading a_j over the unflagged samples of baseline j and M_BD the block-diagonal preconditioner built by
ProcessTimeSamples with the same white weights W.  By Woodbury, x is the GLS map for N = W^-1 + F C_a F^T.  The
operator runs over the run-compressed table of u_j = P^T 1_j (csrc/destripe.cu) and never passes over the TOD; the
right-hand side takes the TOD once per solve.

    weights, prior = baseline_prior_bands(noise_psd(d, ns, pix=pix)[1], L, nband)
    N = BlockLO(ns, weights)
    pts = ProcessTimeSamples(pix, npix, pol=pol, phi=phi, w=N.diag)
    x, a, info = destripe(d, P, N, BlockDiagonalPreconditionerLO(pts, P.ncols, pol), L, prior, rtol=1e-8)

Without a prior, the system of pol 1 and 3 is singular along "the same offset on every baseline", which is the I
monopole: CG from a = 0 converges on this consistent system and the map is defined up to the I monopole (compare maps
after ``subtract_offset``).  Not covered: several GPUs (the scatter would need a map all-reduce and CG a baseline-domain
one), per-sample weights, a Toeplitz W and a two-level preconditioner for the baseline system.
"""
import numpy as np
import torch

from . import _device as dv
from . import linop as lp
from .linearoperators import BlockDiagonalPreconditionerLO, BlockLO, SparseLO, _build_run_table
from .pcg import cg


def _baselines(starts, L):
    """[start, end) of the baselines of every noise block [starts[b], starts[b+1]) and the count per block"""
    sizes = np.diff(starts)
    per_block = -(-sizes // L)
    blk = np.repeat(np.arange(len(sizes)), per_block)
    first = np.concatenate([[0], np.cumsum(per_block)])[:-1]
    s = starts[:-1][blk] + L * (np.arange(len(blk)) - first[blk])
    e = np.minimum(s + L, starts[1:][blk])
    return s.astype(np.int64), e.astype(np.int64), per_block.astype(np.int64), blk


class Destriper(object):
    """The destriper system of ``(P, N, Mbd)`` with baselines of ``baseline`` samples (module docstring).

    ``N``: white ``BlockLO(blocksize, w)`` over the TOD; baseline j of block b covers [s_b + jL, min(s_b + (j+1)L, e_b)).
    ``Mbd``: ``BlockDiagonalPreconditionerLO`` built with ``w=N.diag``.  ``prior``: None (no prior) or one symmetric
    positive definite Toeplitz band per noise block for C_a^-1 on that block's baselines -- the bands of
    ``baseline_prior_bands`` or any others.  Attributes:

    - ``A``: the symmetric device operator F^T W Z F + C_a^-1 on baseline vectors (``nbase`` values);
    - ``M``: the Jacobi preconditioner 1 / (w_b n_j + t_b[0]), 0 where that sum is 0 (a baseline without an
      unflagged sample);
    - ``rhs(d)``, ``solve(d, rtol, maxiter, residuals) -> (a, info)`` through ``cg``, ``map(d, a) -> x``.

    ``d`` is a host array or a device tensor of ``P.nrows`` values, finite on flagged samples too (P^T W d reads
    them).  Raises ValueError for an ``N`` that is not white, ``P`` that is not a ``SparseLO``, ``L < 1``, a prior of the wrong block
    count and an ``Mbd`` or ``N`` of the wrong size.
    """

    def __init__(self, P, N, Mbd, baseline, prior=None):
        if not isinstance(P, SparseLO):
            raise ValueError("P must be a SparseLO pointing operator, got %s" % type(P).__name__)
        if not isinstance(N, BlockLO) or N.isoffdiag:
            raise ValueError("N must be a white BlockLO(blocksize, w) (offdiag=False)")
        if N.shape[0] != P.nrows:
            raise ValueError("N spans %d samples, P has %d rows" % (N.shape[0], P.nrows))
        if not isinstance(Mbd, BlockDiagonalPreconditionerLO) or Mbd.pol != P.pol or Mbd._n != P.ncols:
            raise ValueError("Mbd must be the BlockDiagonalPreconditionerLO of P's pixels and pol")
        L = int(baseline)
        if L < 1:
            raise ValueError("the baseline length must be >= 1 sample, got %d" % L)
        nblocks = N._blk.n
        if prior is not None and len(prior) != nblocks:
            raise ValueError("prior has %d bands, N has %d noise blocks" % (len(prior), nblocks))
        self.P, self.N, self.Mbd, self.L = P, N, Mbd, L
        s, e, self.nbase_per_block, blk = _baselines(N._blk.starts, L)
        self.nbase = nb = len(s)
        self._start, self._end = dv.to_dev(s, torch.int64), dv.to_dev(e, torch.int64)
        self._bw = dv.to_dev_f64(N._w_host[blk])
        rt = _build_run_table(P, self._start, self._end, nb, need_runs=False)
        if not rt:
            raise ValueError("no unflagged sample: nothing to destripe")
        self._runs = rt
        # lanes per baseline: the power of two in 4..32 nearest above the mean runs per baseline
        self._group = int(min(32, max(4, 1 << int(np.ceil(np.log2(max(rt["nruns"] / max(nb, 1), 1.0)))))))
        self._m = dv.empty_f64(P.pol * P.ncols)
        self._y = dv.empty_f64(P.pol * P.ncols)
        self.prior = None
        t0 = np.zeros(nblocks)
        if prior is not None:
            bands = [np.atleast_1d(np.asarray(t, dtype=np.float64)) for t in prior]
            if any(t.ndim != 1 or t.size == 0 for t in bands):
                raise ValueError("each prior band must be a non-empty 1-d array")
            self.prior = BlockLO([int(v) for v in self.nbase_per_block], bands, offdiag=True)
            t0 = np.array([t[0] for t in bands])
        # w_b n_j: the dot with a = 1 and m = 0
        diag = dv.empty_f64(nb)
        self._m.zero_()
        self._dot(torch.ones(nb, dtype=torch.float64, device=diag.device), self._m, None, diag)
        diag += dv.to_dev_f64(t0[blk])
        self._jacobi = torch.where(diag > 0, 1.0 / torch.where(diag > 0, diag, torch.ones_like(diag)),
                                   torch.zeros_like(diag))
        self.A = lp.LinearOperator(nb, nb, matvec=self._apply, symmetric=True, device=True)
        self.M = lp.LinearOperator(nb, nb, matvec=self._precondition, symmetric=True, device=True)

    def run_table_bytes(self):
        """Bytes of run table one apply reads per pass: run_pix (4) and run_mom (24) per run."""
        return 28 * self._runs["nruns"]

    # ---- kernels ----------------------------------------------------------------------------------------------------
    def _tables(self):
        rt = self._runs
        return (dv.ptr(rt["run_pix"]), dv.ptr(rt["run_mom"]), dv.ptr(rt["seg_first"]), dv.ptr(rt["seg_nruns"]),
                self.nbase, self.P.pol, self._group)

    def _scatter(self, c, alpha, y, accumulate):
        dv.call("cm2_destripe_scatter", *self._tables(), dv.ptr(c), dv.ptr(self._bw), float(alpha), dv.ptr(y),
                self.P.ncols, int(accumulate), dv.stream())

    def _dot(self, a, m, add, out):
        dv.call("cm2_destripe_dot", *self._tables(), dv.ptr(self._bw), dv.ptr(a), dv.ptr(m), dv.ptr(add), dv.ptr(out),
                dv.stream())

    def _bd(self, y, out):
        dv.call("cm2_bd_apply", dv.ptr(self.Mbd._inv_dev), self.Mbd._n, self.Mbd.pol, dv.ptr(y), dv.ptr(out),
                dv.stream())

    def _apply(self, a):
        self._scatter(a, 1.0, self._y, False)                          # y = P^T W F a
        self._bd(self._y, self._m)                                     # m = M_BD y
        add = self.prior._apply_all(a) if self.prior is not None else None
        out = dv.empty_f64(self.nbase)
        self._dot(a, self._m, add, out)                                # F^T W F a - F^T W P m + C_a^-1 a
        return out

    def _precondition(self, r):
        out = torch.empty_like(r)
        dv.call("cm2_noise_white_apply", dv.ptr(self._jacobi), self.nbase, 1, None, dv.ptr(r), dv.ptr(out),
                self.nbase, dv.stream())
        return out

    def _tod(self, d):
        n = int(d.numel() if dv.is_dev(d) else np.size(d))
        if n != self.P.nrows:
            raise ValueError("d has %d samples, P has %d rows" % (n, self.P.nrows))
        return dv.to_dev_f64(d).reshape(-1)

    def _ptwd(self, dd):
        """P^T W d"""
        return self.P.rmult(self.N._apply_all(dd))

    # ---- public -----------------------------------------------------------------------------------------------------
    def rhs(self, d):
        """F^T W Z d = F^T W d - F^T W P M_BD P^T W d, a device vector of ``nbase`` values."""
        dd = self._tod(d)
        self._bd(self._ptwd(dd), self._m)
        fwd = dv.empty_f64(self.nbase)
        dv.call("cm2_destripe_tod_sums", dv.ptr(self.P._pix_dev), dv.ptr(dd), dv.ptr(self._start), dv.ptr(self._end),
                self.nbase, dv.ptr(self._bw), dv.ptr(fwd), dv.stream())
        out = dv.empty_f64(self.nbase)
        self._dot(None, self._m, fwd, out)
        return out

    def solve(self, d, rtol=1e-8, maxiter=None, residuals=None):
        """(a, info): the baseline offsets (device) by ``cg(A, rhs(d), M=M)`` from a = 0."""
        return cg(self.A, self.rhs(d), rtol=rtol, maxiter=maxiter, M=self.M, residuals=residuals)

    def map(self, d, a):
        """x = M_BD P^T W (d - F a), a device map of ``P.pol * P.ncols`` values."""
        y = self._ptwd(self._tod(d))
        self._scatter(dv.to_dev_f64(a).reshape(-1), -1.0, y, True)
        x = dv.empty_f64(y.numel())
        self._bd(y, x)
        return x


def destripe(d, P, N, Mbd, baseline, prior=None, **cg_kw):
    """``(x, a, info)``: the destriped map, the baseline offsets and cg's info for ``Destriper(P, N, Mbd, baseline,
    prior)``; ``cg_kw`` go to ``Destriper.solve`` (rtol, maxiter, residuals).  Host ``d`` gives host results, a device
    tensor device results."""
    D = Destriper(P, N, Mbd, baseline, prior)
    a, info = D.solve(d, **cg_kw)
    x = D.map(d, a)
    if not dv.is_dev(d):
        return dv.to_host(x), dv.to_host(a), info
    return x, a, info
