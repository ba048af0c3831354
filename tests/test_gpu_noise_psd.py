"""cm2_noise_psd (k_noise_psd + k_psd_sum, csrc/toeplitz_fft.cu) and the noise model built on it (cosmomap2_b200/noise.py).

1. The per-block sums against the long-double reference of the definition (test_noise_host.welch_sums), called through
   the C ABI with sentinel-guarded outputs.  Bounds, u = 2^-53, per block b with n_win windows:
     sum_k |S_b(k) - ref| <= (2 * 8 log2 M + n_win + 4) u NF sum_w ||x_w||^2
   (the transform's normwise error 8 log2(M) u ||X||, as in test_gpu_toeplitz_reference.py, enters |X|^2 twice; n_win
   the summation over windows; 4 the taper product, the packed-real split and the squaring; NF ||x_w||^2 = ||X_w||^2)
     |W_b - ref_h| <= (17 + n_slots) u W_b,   ref_h = W_b from the kernel's own Hann table h_t
   (all terms are positive, so relative errors add: 1 for each product (h m)^2, 3 for the pairwise sum of a group of
   8, 2 for the thread's compensated run sum, 1 for adding its compensation, 10 for block_sum's two 5-level shuffle
   trees, n_slots - 1 for k_psd_sum adding the block's (CTA, block) slots)
     |h_t - sin^2(pi t / NF)| <= 9 u sin^2   (CUDA's double sinpi is within 2 ulp, i.e. 4 u; squared and rounded)
2. Without flags, noise_psd equals scipy.signal.welch to 1e-12 relative.
3. A repeated call gives the same bits, and so do calls on copies of the inputs 8 (d) and 4 (pix) bytes off alignment.
4. Statistics: the estimate from synthetic.one_over_f_noise agrees with its analytic PSD in octave-averaged bins.
5. End to end: GLS with the estimated bands converges and maps the sky better than the white-weighted solve.
"""
import zlib

import numpy as np
import pytest
import scipy.signal

from test_gpu_tod_reference import LD, U, Guarded, sm_count
from test_noise_host import M, NF, hann, welch_sums

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def cm():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import cosmomap2_b200
    assert int(cosmomap2_b200._cabi.lib.cm2_toeplitz_fft_points()) == M
    return cosmomap2_b200


def _dv():
    from cosmomap2_b200 import _device as dv
    return dv


# ---- layouts and masks -----------------------------------------------------------------------------------------------

def layout(name):
    """(nt, nblocks, blocksize, edges or None)"""
    if name == "equal":
        bs = NF + 2 * M
        return 3 * bs, 3, bs, None
    if name == "remainder":
        bs = NF + M
        return 3 * bs + M + 5, 3, bs, None
    if name == "starts":            # odd starts (8 bytes off 16-byte alignment), blocks without a window, NF + kM +- 1
        lens = [3, NF, NF + M + 1, NF - 1, NF + 2 * M, 0, NF + 5 * M - 1, 5, NF + 3 * M]
        return sum(lens), len(lens), 0, np.r_[0, np.cumsum(lens)]
    if name == "many":              # more windows than CTAs: >= 3 trips per CTA
        nw = max(3 * sm_count() // 4 + 2, 8)
        bs = NF + (nw - 1) * M
        return 4 * bs, 4, bs, None
    raise KeyError(name)


def edges_of(nt, nb, bs, edges):
    return edges if edges is not None else np.r_[np.arange(nb) * bs, nt]


def make_mask(kind, nt, edges, rng):
    if kind == "none":
        return None
    pix = rng.integers(0, 1000, nt).astype(np.int32)
    if kind in ("turnarounds", "nan"):
        period = 5000
        pix[(np.arange(nt) % period) < 600] = -1
    if kind == "window":             # one fully flagged window (the second of the first block that has two)
        b = int(np.flatnonzero(np.diff(edges) >= NF + M)[0])
        pix[edges[b] + M:edges[b] + M + NF] = -1
    return pix


def run_psd(cm, d, pix, nt, nb, bs, edges, d_shift=0, p_shift=0):
    """cm2_noise_psd on device copies of d / pix placed d_shift doubles / p_shift ints into their buffers."""
    import torch
    dv = _dv()
    dbuf = torch.zeros(nt + 4, dtype=torch.float64, device="cuda")
    dbuf[d_shift:d_shift + nt] = torch.from_numpy(np.ascontiguousarray(d)).cuda()
    pptr = None
    if pix is not None:
        pbuf = torch.zeros(nt + 8, dtype=torch.int32, device="cuda")
        pbuf[p_shift:p_shift + nt] = torch.from_numpy(pix).cuda()
        pptr = pbuf.data_ptr() + 4 * p_shift
    start = None if edges is None else dv.to_dev(np.asarray(edges, dtype=np.int64), torch.int64)
    S, W = Guarded(nb * (M + 1), torch.float64), Guarded(nb, torch.float64)
    scratch = torch.empty(int(dv.call("cm2_noise_psd_scratch_bytes", nb)) // 8 + 2, dtype=torch.float64, device="cuda")
    rc = cm._cabi.lib.cm2_noise_psd(dbuf.data_ptr() + 8 * d_shift, pptr, nb, bs, dv.ptr(start), nt, S.ptr(), W.ptr(),
                                    scratch.data_ptr(), 1, dv.stream())
    assert rc == 0, cm._cabi.last_error()
    torch.cuda.synchronize()
    run_psd.hann = scratch[4 * M:4 * M + NF].cpu().numpy()     # the Hann table: after the 2M complex twiddles
    return S.result("psd").reshape(nb, M + 1), W.result("wsum")


def slots_per_block(nt, edges):
    """(CTA, block) runs that k_psd_sum adds for each block: CTA c takes windows [c per, (c+1) per)"""
    n = np.diff(edges)
    nw = np.where(n >= NF, (n - NF) // M + 1, 0)
    wf = np.r_[0, np.cumsum(nw)]
    grid = max(min(sm_count(), nt // M + 1), 1)
    per = max(-(-int(wf[-1]) // grid), 1)
    return [((wf[b + 1] - 1) // per - wf[b] // per + 1) if nw[b] else 0 for b in range(len(n))]


def check_hann(h):
    exact = hann()
    err = np.abs(h.astype(LD) - exact)
    assert np.all(err <= 9 * LD(U) * exact), "Hann table: %.3g u relative" % float(np.max(err[1:] / exact[1:]) / U)


def check_sums(S, W, Sref, Wref, edges, what, nt):
    """Wref from the kernel's own Hann table (run_psd.hann), Sref from the exact one"""
    worst_s = worst_w = 0.0
    slots = slots_per_block(nt, edges)
    for b in range(len(edges) - 1):
        n = int(edges[b + 1] - edges[b])
        nwin = (n - NF) // M + 1 if n >= NF else 0
        if nwin == 0:
            assert np.all(S[b] == 0.0) and W[b] == 0.0, "%s: block %d has no window but nonzero sums" % (what, b)
            continue
        energy = Sref[b, 0] + Sref[b, M] + 2 * np.sum(Sref[b, 1:M])          # = NF sum_w ||x_w||^2
        bound = (2 * 8 * np.log2(M) + nwin + 4) * LD(U) * energy
        err = np.sum(np.abs(S[b].astype(LD) - Sref[b]))
        assert np.all(np.isfinite(S[b])) and err <= bound, "%s: block %d: sum |dS| %.3g > bound %.3g" % (what, b, err, bound)
        werr = abs(LD(W[b]) - Wref[b])
        wbound = (17 + slots[b]) * LD(U) * Wref[b]
        assert werr <= wbound, "%s: block %d: |dW| = %.3g u W > %d u W" % (what, b, werr / (U * Wref[b]), 17 + slots[b])
        worst_s, worst_w = max(worst_s, float(err / bound)), max(worst_w, float(werr / (LD(U) * Wref[b])))
    return worst_s, worst_w


# ---- 1. sums against the long-double reference -----------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("mask", ["none", "turnarounds", "window", "nan"])
@pytest.mark.parametrize("lay", ["equal", "remainder", "starts"])
def test_psd_sums_against_long_double(cm, lay, mask):
    rng = np.random.default_rng(zlib.crc32((lay + mask).encode()))
    nt, nb, bs, edges = layout(lay)
    e = edges_of(nt, nb, bs, edges)
    d = rng.standard_normal(nt) * rng.uniform(0.5, 2.0) + 0.3
    pix = make_mask(mask, nt, e, rng)
    dd = d.copy()
    if mask == "nan":
        dd[pix < 0] = np.nan
    S, W = run_psd(cm, dd, pix, nt, nb, bs, edges)
    check_hann(run_psd.hann)
    Sref, _ = welch_sums(d, e, pix)
    _, Wref = welch_sums(d, e, pix, h=run_psd.hann)
    check_sums(S, W, Sref, Wref, e, "%s/%s" % (lay, mask), nt)


@gpu
def test_psd_sums_many_trips_per_cta(cm):
    rng = np.random.default_rng(17)
    nt, nb, bs, edges = layout("many")
    e = edges_of(nt, nb, bs, edges)
    d = rng.standard_normal(nt)
    pix = make_mask("nan", nt, e, rng)
    dd = d.copy()
    dd[pix < 0] = np.nan
    S, W = run_psd(cm, dd, pix, nt, nb, bs, edges, d_shift=1, p_shift=1)
    Sref, _ = welch_sums(d, e, pix)
    _, Wref = welch_sums(d, e, pix, h=run_psd.hann)
    assert max(slots_per_block(nt, e)) >= 2
    check_sums(S, W, Sref, Wref, e, "many", nt)


# ---- 2. scipy.signal.welch -------------------------------------------------------------------------------------------

@gpu
def test_unflagged_equals_scipy_welch(cm):
    rng = np.random.default_rng(21)
    lens = [NF, NF + M + 1, NF + 6 * M - 1, NF + 4 * M]
    e = np.r_[0, np.cumsum(lens)]
    d = 1.5 * rng.standard_normal(e[-1]) - 0.2
    freqs, P = cm.noise_psd(d, lens)
    assert P.shape == (len(lens), M + 1)
    np.testing.assert_array_equal(freqs, np.arange(M + 1) / NF)
    for b in range(len(lens)):
        _, ref = scipy.signal.welch(d[e[b]:e[b + 1]], fs=1.0, window="hann", nperseg=NF, noverlap=M, detrend=False,
                                    scaling="density", return_onesided=False)
        rel = float(np.max(np.abs(P[b] - ref[:M + 1]) / ref[:M + 1]))
        assert rel < 1e-12, "block %d: %.3g" % (b, rel)
    # the same with the device tensor and an all-unflagged pixel stream
    import torch
    _, P2 = cm.noise_psd(torch.from_numpy(d).cuda(), lens, pix=np.zeros(d.size, dtype=np.int64))
    np.testing.assert_array_equal(P, P2)


# ---- 3. determinism --------------------------------------------------------------------------------------------------

@gpu
def test_bit_identical_repeats_and_alignments(cm):
    rng = np.random.default_rng(31)
    for lay in ("starts", "many"):
        nt, nb, bs, edges = layout(lay)
        e = edges_of(nt, nb, bs, edges)
        d = rng.standard_normal(nt)
        pix = make_mask("turnarounds", nt, e, rng)
        ref = run_psd(cm, d, pix, nt, nb, bs, edges)
        for ds, ps in ((0, 0), (1, 1), (1, 0), (0, 1), (2, 3)):
            got = run_psd(cm, d, pix, nt, nb, bs, edges, d_shift=ds, p_shift=ps)
            assert np.array_equal(got[0].view(np.int64), ref[0].view(np.int64)), "%s: psd differs at shift %r" % (lay, (ds, ps))
            assert np.array_equal(got[1].view(np.int64), ref[1].view(np.int64)), "%s: wsum differs at shift %r" % (lay, (ds, ps))


# ---- 4. statistics ---------------------------------------------------------------------------------------------------

@gpu
def test_one_over_f_statistics(cm):
    """Octave-averaged estimate / analytic PSD within 6 sigma + the window bias.  The estimate of one bin over n_win
    Hann windows at 50 % overlap has relative variance (1 + 2 rho^2) / n_win, rho^2 = 1/6 the squared correlation of
    overlapping windows; K adjacent bins of one window are correlated by 2/3 (neighbour) and 1/6 (next), so the mean of K
    bins has relative variance 1.33 * 1.94 / (n_win K).  The window's spectral second moment (~1 bin^2) biases a
    power law P ~ k^-alpha by at most alpha (alpha+1)/2 / k^2 relative (<= 2 / k_lo^2 here)."""
    from cosmomap2_b200 import synthetic
    ns, ndet, sigma, fknee, alpha = 1 << 21, 2, 1.5, 2e-3, 1.5
    d = synthetic.one_over_f_noise(ns, ndet, sigma, fknee, alpha, seed=5)
    freqs, P = cm.noise_psd(d, ns)
    nwin = (ns - NF) // M + 1
    analytic = sigma ** 2 * (1.0 + (fknee / freqs[1:]) ** alpha)
    for b in range(ndet):
        for j in range(3, 13):                       # bins [2^j, 2^(j+1)), 8 .. 8191
            k0, k1 = 1 << j, min(1 << (j + 1), M)
            K = k1 - k0
            ratio = np.mean(P[b, k0:k1]) / np.mean(analytic[k0 - 1:k1 - 1])
            tol = 6.0 * np.sqrt(1.33 * 1.94 / (nwin * K)) + 2.0 / k0 ** 2
            assert abs(ratio - 1.0) < tol, "detector %d, bins [%d, %d): ratio %.4f, tol %.4f" % (b, k0, k1, ratio, tol)


# ---- 5. end to end ---------------------------------------------------------------------------------------------------

def e2e_scenario(seed=11):
    """Raster scan of 4 detectors x 2^17 samples over 800 pixels (I only), sky ~ N(0, 1), 1/f noise with
    fknee = 0.05 cycles/sample and alpha = 1.  Rehearsed on the CPU with the oracle's P and Toeplitz operators and
    scipy's Welch estimate: map rms error GLS / white-weighted = 0.967 (seed 11) and 0.981 (seed 12)."""
    from cosmomap2_b200 import synthetic
    ndet, ns = 4, 1 << 17
    sc = synthetic.raster_scan(ndet * ns, nside=32, ndet=ndet, nx=40, ny=20, samples_per_pixel=6.0, seed=seed,
                               with_data=False)
    sky = np.random.default_rng(seed + 1).standard_normal(sc.npix_full)
    noise = synthetic.one_over_f_noise(ns, ndet, 1.0, 0.05, 1.0, seed + 2)
    return sc, sky, sky[sc.pix.astype(np.int64)] + noise


@gpu
def test_gls_with_estimated_bands_beats_white_weights(cm):
    sc, sky, d = e2e_scenario()
    ns = sc.ns
    _, P = cm.noise_psd(d, ns)
    bands = cm.inverse_noise_bands(P, 512)
    weights = [t[0] for t in bands]
    obs = np.unique(sc.pix[sc.pix >= 0])
    err = {}
    for name, N in (("gls", cm.BlockLO(ns, bands, offdiag=True)), ("white", cm.BlockLO(ns, weights))):
        pix = sc.pix.astype(np.int64)
        pts = cm.ProcessTimeSamples(pix, sc.npix_full, pol=1, w=cm.BlockLO(ns, weights).diag)
        npix, obspix = pts.get_new_pixel
        assert npix == obs.size and np.array_equal(np.asarray(obspix)[:npix], obs)
        Pt = cm.SparseLO(npix, sc.nt, pix, pol=1, angle_processed=pts)
        A = Pt.T * N * Pt
        b = Pt.T * (N * d)
        x, info = cm.cg(A, b, M=cm.BlockDiagonalPreconditionerLO(pts, npix, pol=1), rtol=1e-8, maxiter=500)
        assert info == 0, "%s: cg info %d" % (name, info)
        r = np.asarray(x) - sky[obs]
        err[name] = float(np.sqrt(np.mean((r - r.mean()) ** 2)))
    assert err["gls"] < 0.99 * err["white"], err
