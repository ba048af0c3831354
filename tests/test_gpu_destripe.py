"""The destriper with a noise prior (cosmomap2_b200/destripe.py, csrc/destripe.cu, DESIGN.md section 4f) against dense
NumPy references, for pol 1, 2 and 3 on scans with flagged turnarounds, noise blocks of different sizes, a baseline
length that divides none of them and a flagged stretch longer than a baseline (baselines with no unflagged sample).

The dense references use the M_BD the library built (its packed inverse blocks read back), not an exact inverse, so
that Z = I - P M_BD P^T W is the same matrix on both sides.
"""
import numpy as np
import pytest

gpu = pytest.mark.gpu

SIZES = [1301, 977, 1650]          # noise blocks (detectors); L = 37 divides none of them
L = 37
NPIX = 70
WEIGHTS = [1.0, 2.5, 0.6]


@pytest.fixture(scope="module")
def cm():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import cosmomap2_b200
    return cosmomap2_b200


def _prior_bands(nband=6):
    """SPD bands per block: a decaying positive-definite sequence (symbol > 0) of different scales"""
    out = []
    for b, scale in enumerate((0.3, 1.0, 3.0)):
        t = scale * 0.5 ** np.arange(nband + b)
        t[0] += scale
        out.append(t)
    return out


def make_case(cm, pol, seed=0):
    rng = np.random.default_rng(seed + 10 * pol)
    nt = sum(SIZES)
    t = np.arange(nt)
    # a back-and-forth sweep with 1..6 samples per pixel, turnarounds flagged, one stretch of 3 L flagged
    run = rng.integers(1, 7, nt // 2 + 1)
    pix = np.repeat(np.arange(run.size) % (2 * NPIX), run)[:nt]
    pix = np.where(pix < NPIX, pix, 2 * NPIX - 1 - pix).astype(np.int64)
    pix[(t % 400) < 25] = -1
    pix[1400:1400 + 3 * L] = -1
    phi = rng.uniform(0, np.pi, nt)
    N = cm.BlockLO(SIZES, WEIGHTS)
    pts = cm.ProcessTimeSamples(pix, NPIX, pol=pol, phi=phi, w=N.diag)
    npix, _ = pts.get_new_pixel
    P = cm.SparseLO(npix, nt, pix, pol=pol, angle_processed=pts)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
    return P, N, Mbd


def dense(cm, P, N, Mbd, prior):
    """(P, W, M_BD, F, C_a^-1, baselines) as dense matrices from the operators' own device tables"""
    pol, npix, nt = P.pol, P.ncols, P.nrows
    pp = P._pix_dev.cpu().numpy()
    c = P._cos_dev.cpu().numpy() if pol > 1 else np.ones(nt)
    s = P._sin_dev.cpu().numpy() if pol > 1 else np.zeros(nt)
    Pd = np.zeros((nt, pol * npix))
    ok = np.flatnonzero(pp >= 0)
    cols = {1: [np.ones(nt)], 2: [c, s], 3: [np.ones(nt), c, s]}[pol]
    for k, v in enumerate(cols):
        Pd[ok, pol * pp[ok] + k] = v[ok]
    edges = np.r_[0, np.cumsum(SIZES)]
    w = np.repeat(WEIGHTS, SIZES)
    inv = Mbd._inv_dev.cpu().numpy().reshape(-1, 6)[:npix]
    Md = np.zeros((pol * npix, pol * npix))
    for j in range(npix):
        a00, a01, a02, a11, a12, a22 = inv[j]
        blk = {1: [[a00]], 2: [[a11, a12], [a12, a22]], 3: [[a00, a01, a02], [a01, a11, a12], [a02, a12, a22]]}[pol]
        Md[pol * j:pol * j + pol, pol * j:pol * j + pol] = blk
    starts, ends, nper = [], [], []
    for b in range(len(SIZES)):
        st = np.arange(edges[b], edges[b + 1], L)
        starts.append(st)
        ends.append(np.minimum(st + L, edges[b + 1]))
        nper.append(st.size)
    starts, ends = np.concatenate(starts), np.concatenate(ends)
    nbase = starts.size
    Fd = np.zeros((nt, nbase))
    for j in range(nbase):
        tt = np.arange(starts[j], ends[j])
        Fd[tt[pp[tt] >= 0], j] = 1.0
    Cinv = np.zeros((nbase, nbase))
    if prior is not None:
        o = 0
        for b, n in enumerate(nper):
            band = np.zeros(n)
            k = min(n, len(prior[b]))
            band[:k] = prior[b][:k]
            i = np.arange(n)
            Cinv[o:o + n, o:o + n] = band[np.abs(i[:, None] - i[None, :])]
            o += n
    return Pd, w, Md, Fd, Cinv, (starts, ends)


def dense_A(Pd, w, Md, Fd, Cinv):
    WF = w[:, None] * Fd
    PtWF = Pd.T @ WF
    return Fd.T @ WF - PtWF.T @ Md @ PtWF + Cinv, (np.abs(Fd).T @ np.abs(WF), np.abs(PtWF).T @ np.abs(Md) @ np.abs(PtWF),
                                                   np.abs(Cinv))


@gpu
@pytest.mark.parametrize("pol", [1, 2, 3])
@pytest.mark.parametrize("with_prior", [False, True])
def test_apply_matches_dense(cm, pol, with_prior):
    import torch
    P, N, Mbd = make_case(cm, pol)
    prior = _prior_bands() if with_prior else None
    D = cm.Destriper(P, N, Mbd, L, prior)
    Pd, w, Md, Fd, Cinv, (starts, ends) = dense(cm, P, N, Mbd, prior)
    assert D.nbase == Fd.shape[1]
    assert np.any(Fd.sum(axis=0) == 0), "the case must have a baseline with no unflagged sample"
    A, mags = dense_A(Pd, w, Md, Fd, Cinv)
    rng = np.random.default_rng(1)
    for _ in range(3):
        a = rng.standard_normal(D.nbase)
        got = D.A.matvec(a)
        # every term is a sum of at most a few thousand products: 1e-12 of the magnitudes is > 100 roundings each
        scale = max(float(np.max(m @ np.abs(a))) for m in mags)
        assert np.max(np.abs(got - A @ a)) <= 1e-12 * scale
    # the scatter alone equals P.T*(W*(F a)) with F a a TOD spread over the baselines by the white-noise kernel
    a = rng.standard_normal(D.nbase)
    y = torch.empty(P.pol * P.ncols, dtype=torch.float64, device="cuda")
    D._scatter(torch.from_numpy(a).cuda(), 1.0, y, False)
    Fa = cm.BlockLO(list(ends - starts), list(a)).matvec(np.ones(P.nrows))
    ref = P.T * (N * Fa)
    np.testing.assert_allclose(y.cpu().numpy(), ref, rtol=0, atol=1e-13 * np.max(np.abs(ref)))
    # the Jacobi preconditioner
    diag = np.diag(Fd.T @ (w[:, None] * Fd)) + np.diag(Cinv)
    want = np.where(diag > 0, 1.0 / np.where(diag > 0, diag, 1.0), 0.0)
    np.testing.assert_allclose(D.M.matvec(np.ones(D.nbase)), want, rtol=1e-15, atol=0)


@gpu
@pytest.mark.parametrize("pol", [1, 2, 3])
def test_symmetric_and_deterministic(cm, pol):
    import torch
    P, N, Mbd = make_case(cm, pol, seed=3)
    D = cm.Destriper(P, N, Mbd, L, _prior_bands())
    rng = np.random.default_rng(2)
    a, b = rng.standard_normal(D.nbase), rng.standard_normal(D.nbase)
    Aa, Ab = D.A.matvec(a), D.A.matvec(b)
    lhs, rhs = a @ Ab, b @ Aa
    assert abs(lhs - rhs) <= 1e-13 * (np.abs(a) @ np.abs(Ab) + np.abs(b) @ np.abs(Aa))
    m = torch.from_numpy(rng.standard_normal(P.pol * P.ncols)).cuda()
    ad = torch.from_numpy(a).cuda()
    outs = []
    for _ in range(3):
        o = torch.empty(D.nbase, dtype=torch.float64, device="cuda")
        D._dot(ad, m, None, o)
        outs.append(o.cpu().numpy())
    assert all(np.array_equal(outs[0].view(np.int64), o.view(np.int64)) for o in outs[1:])


@gpu
@pytest.mark.parametrize("pol", [1, 2, 3])
def test_solved_map_is_the_gls_map(cm, pol):
    """With a prior, x = M_BD P^T W (d - F a) is the GLS map for N = W^-1 + F C_a F^T (Woodbury), where M_BD is the
    exact inverse of P^T W P (checked first).  Bound: CG stops at ||A (a - a*)|| <= rtol ||b||, so
    ||a - a*|| <= rtol ||b|| / lambda_min(A) and ||x - x*|| <= ||M_BD P^T W F||_2 ||a - a*||; the dense GLS solve adds
    at most cond(P^T N^-1 P) * 1e-14 relative (a few hundred roundings of its factorisation)."""
    P, N, Mbd = make_case(cm, pol, seed=5)
    prior = _prior_bands()
    Pd, w, Md, Fd, Cinv, _ = dense(cm, P, N, Mbd, prior)
    PtWP = Pd.T @ (w[:, None] * Pd)
    assert np.max(np.abs(Md @ PtWP - np.eye(PtWP.shape[0]))) < 1e-10
    rng = np.random.default_rng(7)
    d = Pd @ rng.standard_normal(Pd.shape[1]) + Fd @ rng.standard_normal(Fd.shape[1]) + rng.standard_normal(P.nrows)
    rtol = 1e-12
    D = cm.Destriper(P, N, Mbd, L, prior)
    a, info = D.solve(d, rtol=rtol, maxiter=5000)
    assert info == 0
    x = D.map(d, a).cpu().numpy()
    A, _ = dense_A(Pd, w, Md, Fd, Cinv)
    b = D.rhs(d).cpu().numpy()
    WF = w[:, None] * Fd
    Ninv = np.diag(w) - WF @ np.linalg.solve(Cinv + Fd.T @ WF, WF.T)
    G = Pd.T @ Ninv @ Pd
    xs = np.linalg.solve(G, Pd.T @ Ninv @ d)
    lam = np.linalg.eigvalsh(A)
    assert lam[0] > 0
    bound = np.linalg.norm(Md @ Pd.T @ WF, 2) * rtol * np.linalg.norm(b) / lam[0] + np.linalg.cond(G) * 1e-14 * np.linalg.norm(xs)
    assert np.linalg.norm(x - xs) <= bound, (np.linalg.norm(x - xs), bound)


@gpu
@pytest.mark.parametrize("pol", [1, 2, 3])
def test_no_prior_is_the_offset_filter_map(cm, pol):
    """Without a prior the map is that of P.T*F*N*F*P with FilterLO subscans equal to the baselines (up to the I
    monopole for pol 1 and 3).  Both are solved to rtol 1e-12; the small systems here have condition numbers below
    1e4, so 1e-7 of the map is far above what the two solves leave."""
    P, N, Mbd = make_case(cm, pol, seed=9)
    _, _, _, _, _, (starts, ends) = dense(cm, P, N, Mbd, None)
    rng = np.random.default_rng(8)
    d = rng.standard_normal(P.nrows) + np.repeat(rng.standard_normal(starts.size) * 3, ends - starts)
    x, a, info = cm.destripe(d, P, N, Mbd, L, rtol=1e-12, maxiter=5000)
    assert info == 0
    F = cm.FilterLO(P.nrows, [list(ends - starts), list(starts)], P.nrows, 1, P._pix_dev.cpu().numpy().astype(np.int64))
    xf, info = cm.cg(P.T * F * N * F * P, P.T * F * N * F * d, M=Mbd, rtol=1e-12, maxiter=5000)
    assert info == 0
    obs = np.arange(P.ncols)
    if pol in (1, 3):
        x, xf = x.reshape(-1, pol), np.asarray(xf).reshape(-1, pol)
        x[:, 0] -= x[:, 0].mean()
        xf[:, 0] -= xf[:, 0].mean()
    assert np.max(np.abs(np.ravel(x) - np.ravel(xf))) <= 1e-7 * np.max(np.abs(xf)), obs.size


@gpu
def test_destriped_map_beats_white_map(cm):
    """1/f noise drawn by simulate_noise plus an I sky on a raster with flagged turnarounds; the prior comes from
    noise_psd of the data.  The noise is steep (alpha = 2), so most of its power lies below the baseline frequency
    1/L, where the offsets model it.  The destriped map has the lower rms error, as Toeplitz GLS does in
    test_gpu_noise_psd."""
    import torch
    from cosmomap2_b200 import synthetic
    ndet, ns = 4, 1 << 17
    sc = synthetic.raster_scan(ndet * ns, nside=32, ndet=ndet, nx=40, ny=20, samples_per_pixel=6.0, seed=11,
                               with_data=False, flag_turnarounds=True)
    sky = np.random.default_rng(12).standard_normal(sc.npix_full)
    M = int(cm._cabi.lib.cm2_toeplitz_fft_points())
    f = np.arange(M + 1) / (2.0 * M)
    model = 1.0 + (0.02 / np.maximum(f, 0.5 / M)) ** 2
    n = cm.simulate_noise(cm.noise_sim_bands(np.tile(model, (ndet, 1)), 4096), ns, seed=13).cpu().numpy()
    good = sc.pix >= 0
    d = np.where(good, sky[np.where(good, sc.pix, 0)] + n, 0.0)
    _, psd = cm.noise_psd(d, ns, pix=sc.pix)
    weights, prior = cm.baseline_prior_bands(psd, 16, 256)
    N = cm.BlockLO(ns, list(weights))
    pix = sc.pix.astype(np.int64)
    pts = cm.ProcessTimeSamples(pix, sc.npix_full, pol=1, w=N.diag)
    npix, obspix = pts.get_new_pixel
    P = cm.SparseLO(npix, sc.nt, pix, pol=1, angle_processed=pts)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=1)
    truth = sky[np.asarray(obspix)[:npix]]
    xw, info = cm.cg(P.T * N * P, P.T * (N * d), M=Mbd, rtol=1e-8, maxiter=500)
    assert info == 0
    xd, a, info = cm.destripe(torch.from_numpy(d).cuda(), P, N, Mbd, 16, prior, rtol=1e-8, maxiter=2000)
    assert info == 0

    def err(x):
        r = np.asarray(x.cpu() if torch.is_tensor(x) else x) - truth
        return float(np.sqrt(np.mean((r - r.mean()) ** 2)))

    print("map rms error: destriped %.4f, white %.4f" % (err(xd), err(xw)))
    assert err(xd) < 0.99 * err(xw), (err(xd), err(xw))


@gpu
def test_value_errors(cm):
    P, N, Mbd = make_case(cm, 3)
    with pytest.raises(ValueError, match="white"):
        cm.Destriper(P, cm.BlockLO(SIZES, _prior_bands(), offdiag=True), Mbd, L)
    with pytest.raises(ValueError, match="SparseLO"):
        cm.Destriper(P.T * P, N, Mbd, L)
    with pytest.raises(ValueError, match="baseline length"):
        cm.Destriper(P, N, Mbd, 0)
    with pytest.raises(ValueError, match="noise blocks"):
        cm.Destriper(P, N, Mbd, L, _prior_bands()[:2])
    D = cm.Destriper(P, N, Mbd, L)
    with pytest.raises(ValueError, match="samples"):
        D.solve(np.zeros(P.nrows + 1))
    with pytest.raises(ValueError, match="samples"):
        cm.destripe(np.zeros(P.nrows - 1), P, N, Mbd, L)
