"""cm2_noise_simulate (k_toeplitz_fft with the NoiseWindow source, DESIGN.md section 4d) against the host
transcription of its definition, called through the C ABI so that the test picks one-CTA or cluster windows.

Reference: per noise block, the stream w_b is regenerated on the host (tests/test_noise_sim_host.py, Philox4x32-10
in integers, Box-Muller in long double) over [-HD, nw S - HD + NF) -- every window input, past both block edges -- and
convolved with the block's band in long double (band_apply of test_gpu_toeplitz_reference.py).

Bound per window w, normwise over its outputs (u = 2^-53):
    ||y_w - ref_w||_2 <= 8 log2(N) u max|H_b| ||w_window||_2  +  sqrt(n_w) (|h_0| + 2 sum_{k>0} |h_k|) 8 u rho_w
The first term is check_fft's bound for the transform of exact inputs.  The second is the generator's: each device
sample differs from the exact w by at most 8 u rho (rho = sqrt(-2 ln u1) of its pair, rho_w the largest in the
window), and each output sums the band against 2L - 1 such samples; sqrt(n_w) turns the per-output bound into a 2-norm.
The 8 u rho: u1 and u2 are exact.  CUDA's double log is within 1 ulp, so -2 ln u1 is within 2u relative (x(-2) is
exact); sqrt halves that and adds 0.5 ulp: rho within 2u relative.  sincospi is within 2 ulp of cos / sin (2 pi u2),
i.e. 4u absolute since |cos|, |sin| <= 1.  The product rho cos adds 0.5 ulp <= u rho.  Together
|dw| <= rho (2u + 4u + u) + O(u^2) <= 8 u rho.
"""
import numpy as np
import pytest

from test_gpu_tod_reference import LD, SENTINEL, U, Guarded, sm_count
from test_gpu_toeplitz_reference import (CM2_ERR_ARG, Layout, band_apply, checked, fft_geometry, fft_points,
                                         make_bands, noise_layout, written)
from test_noise_sim_host import noise_stream

gpu = pytest.mark.gpu
SEED = 0x123456789ABCDEF


@pytest.fixture(scope="module")
def cm():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import cosmomap2_b200
    return cosmomap2_b200


def _dv():
    from cosmomap2_b200 import _device as dv
    return dv


def _lib():
    from cosmomap2_b200 import _cabi
    return _cabi.lib


class Sim:
    """The device tables of one band set and one window mode, and the raw C ABI call."""

    def __init__(self, bands, pair):
        import torch
        from cosmomap2_b200 import linearoperators as lo
        dv = _dv()
        self.bands, self.L, self.pair = bands, bands.shape[1], pair
        coef = lo.toeplitz_fft_tables(bands, self.L, fft_points(), pair=bool(pair))
        self.coef = dv.to_dev_f64(coef.view(np.float64).reshape(-1))
        self.stride = coef[0].nbytes
        self.scratch = torch.empty(int(dv.call("cm2_toeplitz_fft_scratch_bytes", len(bands))) // 8 + 2,
                                   dtype=torch.float64, device="cuda")

    def __call__(self, nb, bs, start, out, nt, seed=SEED, realization=0, ids=None, add=0, block=0, L=None,
                 coef_off=0, scratch_off=0):
        dv = _dv()
        return _lib().cm2_noise_simulate(self.coef.data_ptr() + block * self.stride + coef_off, L or self.L, nb, bs,
                                         start, dv.ptr(ids), seed, realization, out, nt, add,
                                         self.scratch.data_ptr() + scratch_off, 1, self.pair, dv.stream())

    def run(self, lay, **kw):
        y = Guarded(lay.nt)
        what = "sim pair=%d L=%d %r" % (self.pair, self.L, lay)
        checked(self(*lay.args(), y.ptr(), lay.nt, **kw), what)
        return written(y.result(what), what)


def check_sim(y, sim, lay, seed=SEED, realization=0, ids=None):
    L, bands = sim.L, sim.bands
    NF, HD, S = fft_geometry(L, sim.pair)
    logn = np.log2(NF // 2)
    worst = 0.0
    for b, (s, e) in enumerate(lay.bounds()):
        n = e - s
        if n == 0:
            continue
        nw = -(-n // S)
        w, rho = noise_stream(seed, realization, b if ids is None else int(ids[b]), -HD, nw * S - HD + NF)
        ref = band_apply(w, bands[b])[HD:HD + n]
        err2 = np.asarray((y[s:e].astype(LD) - ref) ** 2, dtype=np.float64)
        err_w = np.sqrt(np.bincount(np.arange(n) // S, weights=err2, minlength=nw))
        wf = w.astype(np.float64)
        cs = np.r_[0.0, np.cumsum(wf ** 2)]
        w0 = np.arange(nw) * S                                    # window inputs at [w0, w0 + NF) of the stream
        v_w = np.sqrt(cs[w0 + NF] - cs[w0])
        rho_w = np.array([rho[i:i + NF].max() for i in w0])
        n_w = np.minimum(S, n - np.arange(nw) * S)
        hc = np.zeros(NF)
        hc[:L] = bands[b]
        if L > 1:
            hc[NF - L + 1:] = bands[b][1:][::-1]
        h1 = abs(bands[b][0]) + 2 * np.sum(np.abs(bands[b][1:]))
        bound = 8 * logn * U * np.max(np.abs(np.fft.rfft(hc))) * v_w + np.sqrt(n_w) * h1 * 8 * U * rho_w
        bad = np.flatnonzero(~(err_w <= bound))
        assert bad.size == 0, "pair=%d L=%d %r block %d [%d, %d): %d windows beyond the bound, first %d: %.3g > %.3g" % (
            sim.pair, L, lay, b, s, e, bad.size, bad[0], err_w[bad[0]], bound[bad[0]])
        worst = max(worst, float(np.max(err_w / bound)))
    return worst


def _case(L, pair, layout, trips, seed):
    rng = np.random.default_rng(seed)
    S = fft_geometry(L, pair)[2]
    grid = (sm_count() // 2 if pair else sm_count()) if trips else 1
    lay = noise_layout(layout, S, L, grid * S, rng)
    return lay, make_bands(lay.nb, L, rng)


CASES = ([(L, 0, lay, False) for L in (1, 2, 48, 2047, 4096) for lay in ("equal", "remainder", "ragged")] +
         [(L, 1, lay, False) for L in (3000, 4096, 8192) for lay in ("equal", "remainder", "ragged")] +
         [(48, 0, "ragged", True), (4096, 1, "ragged", True)])


@gpu
@pytest.mark.parametrize("L,pair,layout,trips", CASES)
def test_sim_against_reference_stream(cm, L, pair, layout, trips):
    """Every output written, nothing outside the guards, every window within the bound of the module docstring.
    The ragged layouts hold empty, 1-sample, odd-start and shorter-than-band blocks; `trips` runs >= 3 windows per
    CTA (cluster)."""
    lay, bands = _case(L, pair, layout, trips, seed=L + 7 * pair)
    sim = Sim(bands, pair)
    y = sim.run(lay)
    worst = check_sim(y, sim, lay)
    if trips:
        S = fft_geometry(L, pair)[2]
        nwin = sum(-(-(e - s) // S) for s, e in lay.bounds())
        assert nwin >= 3 * (sm_count() // 2 if pair else sm_count()), "fewer than 3 trips"
    print("sim pair=%d L=%d %r: largest error / bound %.3g" % (pair, L, lay, worst))


@gpu
@pytest.mark.parametrize("L,pair", [(48, 0), (4096, 1)])
def test_sim_bit_exact(cm, L, pair):
    """Repeated calls, out 8 bytes off 16-byte alignment, the blocks split over two calls with block_ids, and add
    mode against x + n: all the same bits."""
    import torch
    dv = _dv()
    lay, bands = _case(L, pair, "ragged", False, seed=100 + L)
    sim = Sim(bands, pair)
    y = sim.run(lay)
    assert np.array_equal(sim.run(lay).view(np.int64), y.view(np.int64)), "repeated call differs"
    ys = Guarded(lay.nt, shift=1)
    checked(sim(*lay.args(), ys.ptr(), lay.nt), "shifted out")
    assert np.array_equal(ys.result("shifted out").view(np.int64), y.view(np.int64)), "out 8 bytes off: differs"
    # blocks [0, k) with the default ids, then [k, nb) with ids k.. on their own sub-TOD
    k = lay.nb // 2
    st = lay.edges
    yb = Guarded(lay.nt)
    lo = torch.from_numpy(st[:k + 1].copy()).cuda()
    hi = torch.from_numpy((st[k:] - st[k]).copy()).cuda()
    ids = torch.arange(k, lay.nb, dtype=torch.int64, device="cuda")
    checked(sim(k, 0, dv.ptr(lo), yb.ptr(), int(st[k])), "first half")
    checked(sim(lay.nb - k, 0, dv.ptr(hi), yb.ptr() + 8 * int(st[k]), int(st[-1] - st[k]), ids=ids, block=k),
            "second half")
    yb = yb.result("split")
    assert np.array_equal(yb.view(np.int64), y.view(np.int64)), "split over two calls with block_ids: differs"
    # add mode
    x = np.random.default_rng(5).standard_normal(lay.nt)
    for shift in (0, 1):                          # 16-byte read-modify-write stores, and the 8-byte ones
        ya = Guarded(lay.nt, shift=shift)
        ya.view.copy_(torch.from_numpy(x))
        checked(sim(*lay.args(), ya.ptr(), lay.nt, add=1), "add")
        assert np.array_equal(ya.result("add").view(np.int64), (x + y).view(np.int64)), \
            "add mode, out shifted by %d words: differs from x + n" % shift


@gpu
def test_sim_streams_independent(cm):
    """White band [1]: streams for another seed, realization or block id are uncorrelated within 5 / sqrt(n), and
    each has unit variance."""
    nt = 1 << 21
    sim = Sim(np.array([[1.0, 0.0]]), 0)
    lay = Layout("one", nt, 1, nt)
    import torch
    base = sim.run(lay)
    others = [sim.run(lay, seed=SEED + 1), sim.run(lay, realization=1),
              sim.run(lay, ids=torch.tensor([1], dtype=torch.int64, device="cuda"))]
    tol = 5 / np.sqrt(nt)
    assert abs(np.mean(base ** 2) - 1) < 5 * np.sqrt(2.0 / nt)
    for i, o in enumerate(others):
        assert abs(np.mean(o ** 2) - 1) < 5 * np.sqrt(2.0 / nt)
        c = np.mean(base * o)
        assert abs(c) < tol, "stream %d: correlation %.3g beyond %.3g" % (i, c, tol)
    assert abs(np.mean(base[1:] * base[:-1])) < tol


@gpu
def test_sim_psd_round_trip(cm):
    """noise_psd of a simulation with bands from an estimated 1/f PSD at nband = M against the exact expected Welch
    mean sum_tau r_tau (h*h)_tau e^{-2 pi i k tau / NF} / sum h^2 (r the simulation's autocovariance, h the Hann
    window), averaged over 64-bin bands, within 5 sigma of the Welch variance."""
    from cosmomap2_b200 import noise_psd, noise_sim_bands, simulate_noise, synthetic
    M = fft_points()
    NF = 2 * M
    x = synthetic.one_over_f_noise(64 * M, 1, 1.0, 0.02, 1.5, seed=3)
    _, psd = noise_psd(x, 64 * M)
    t = noise_sim_bands(psd, M)[0]
    n = 401 * M
    K = (n - NF) // M + 1
    y = simulate_noise([t], n, seed=11)
    _, p = noise_psd(y, n)
    hs = np.r_[t[::-1], t[1:]]                                     # the two-sided filter
    m = 1 << 16
    r = np.fft.irfft(np.abs(np.fft.rfft(hs, m)) ** 2, m)           # autocovariance of unit white noise through hs
    h = np.sin(np.pi * np.arange(NF) / NF) ** 2
    hh = np.fft.irfft(np.abs(np.fft.rfft(h, 2 * NF)) ** 2, 2 * NF)   # (h * h)_tau, tau mod 2 NF
    g = np.zeros(2 * NF)
    tau = np.arange(-(NF - 1), NF)
    g[tau % (2 * NF)] = r[tau % m] * hh[tau % (2 * NF)]
    expect = np.fft.fft(g).real[0::2][:M + 1] / np.sum(h ** 2)
    nbin = 64
    nbands = (M - 1) // nbin
    sl = slice(1, 1 + nbands * nbin)
    got_b = p[0][sl].reshape(nbands, nbin).mean(axis=1)
    exp_b = expect[sl].reshape(nbands, nbin)
    # Welch variance of a band mean: E[P]^2 / K per bin, times 1.06 for the 50 % overlap of Hann windows and
    # 1 + 2 (4/9) + 2 (1/36) = 1.94 for the correlation of neighbouring Hann bins: 2.2 in all
    sigma = np.sqrt(2.2 * np.sum(exp_b ** 2, axis=1) / K) / nbin
    z = (got_b - exp_b.mean(axis=1)) / sigma
    assert np.max(np.abs(z)) < 5, "band %d: %.2f sigma" % (int(np.argmax(np.abs(z))), float(np.max(np.abs(z))))


@gpu
def test_sim_map_domain_white(cm):
    """White bands [1 / sqrt(w_b)] and K = 64 realizations of the binned map M_BD P^T W n: the per-pixel variance
    averages to diag((P^T W P)^-1) = 1 / sum_{t in p} w_t, within the chi^2 spread."""
    import cosmomap2_b200 as cmm
    from cosmomap2_b200 import synthetic
    sc = synthetic.raster_scan(400000, nside=64, ndet=4, nx=80, ny=40, samples_per_pixel=6.0, seed=2)
    pix = sc.pix.astype(np.int64)
    N = cmm.BlockLO(sc.ns, sc.weights)
    pts = cmm.ProcessTimeSamples(pix, sc.npix_full, pol=1, w=N.diag)
    npix = pts.get_new_pixel[0]
    P = cmm.SparseLO(npix, sc.nt, pix, pol=1, angle_processed=pts)
    Mbd = cmm.BlockDiagonalPreconditionerLO(pts, npix, pol=1)
    sizes = np.diff(np.r_[0, np.cumsum(np.broadcast_to(sc.ns, (len(sc.weights),)))])
    wt = np.repeat(np.asarray(sc.weights, dtype=np.float64), sizes)
    ok = pix >= 0
    diag = 1.0 / np.bincount(pix[ok], weights=wt[ok], minlength=npix)
    sim = cmm.NoiseSimulator([[1.0 / np.sqrt(w)] for w in sc.weights], sc.ns)
    K = 64
    acc = np.zeros(npix)
    for k in range(K):
        n = sim(7, realization=k).cpu().numpy()
        m = Mbd * (P.T * (N * n))
        acc += np.asarray(m) ** 2
    ratio = acc / K / diag
    spread = np.sqrt(2.0 / (K * npix))
    assert abs(ratio.mean() - 1) < 5 * spread, "mean variance ratio %.4f, chi^2 spread %.4f" % (ratio.mean(), spread)


@gpu
def test_sim_argument_checks(cm):
    import torch
    dv = _dv()
    M = fft_points()
    for L, pair in ((M // 2 + 1, 0), (M + 1, 1)):
        sim = Sim(np.ones((1, L)), pair)
        y = Guarded(100)
        assert sim(1, 100, None, y.ptr(), 100) == CM2_ERR_ARG, "L=%d pair=%d accepted" % (L, pair)
        y.result("refused")
    sim = Sim(np.ones((2, 8)), 0)
    y = Guarded(100)
    assert sim(2, 50, None, y.ptr(), 100, coef_off=8) == CM2_ERR_ARG, "misaligned coef accepted"
    assert sim(2, 50, None, y.ptr(), 100, scratch_off=8) == CM2_ERR_ARG, "misaligned scratch accepted"
    assert sim(2, 101, None, y.ptr(), 100) == CM2_ERR_ARG, "(nblocks-1) blocksize > nt accepted"
    assert sim(1, 50, None, y.ptr(), 0) == 0, "nt = 0 refused"
    assert _lib().cm2_noise_simulate(sim.coef.data_ptr(), 8, 1, 50, None, None, 1, 0, None, 0, 0,
                                     sim.scratch.data_ptr(), 1, 0, dv.stream()) == 0, "nt = 0 with out = NULL refused"
    assert np.all(y.buf.cpu().numpy() == SENTINEL), "a refused call or nt = 0 wrote"
    # the Python layer
    from cosmomap2_b200 import simulate_noise
    with pytest.raises(ValueError):
        simulate_noise([np.ones(M + 1)], 1000, 1)
    with pytest.raises(ValueError):
        simulate_noise([np.ones(4)] * 2, 1000, 1, add_to=torch.zeros(1999, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        simulate_noise([np.ones(4)] * 2, 1000, 1, block_ids=[0, -1])
    for bad in (torch.zeros(2000, dtype=torch.float64), torch.zeros(2000, dtype=torch.float32, device="cuda")):
        with pytest.raises(ValueError, match="add_to"):
            simulate_noise([np.ones(4)] * 2, 1000, 1, add_to=bad)        # a host tensor, a float32 tensor
    x0 = torch.linspace(-3.0, 5.0, 2000, dtype=torch.float64, device="cuda")
    x = x0.clone()
    n = simulate_noise([np.ones(4)] * 2, 1000, 1)
    assert simulate_noise([np.ones(4)] * 2, 1000, 1, add_to=x) is x
    assert torch.equal(x, x0 + n)
    # the apply still refuses d == out, NULL included
    kern = Sim(np.ones((1, 8)), 0)
    assert _lib().cm2_noise_toeplitz_fft_apply(kern.coef.data_ptr(), 8, 1, 100, None, None, None, 100,
                                               kern.scratch.data_ptr(), 1, 0, dv.stream()) == CM2_ERR_ARG
