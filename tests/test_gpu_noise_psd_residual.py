"""cm2_noise_psd_residual (k_noise_psd<Residual<POL>>, csrc/toeplitz_fft.cu) and noise_psd(d, bs, P=P, x=x): the Welch
PSD of the map residual r = d - P x, formed inside the PSD pass.

1. Bit-identity with the unfused path: the fused sums equal cm2_noise_psd on d - P.mult(x) (a torch subtraction) with
   P's pixel table, for pol 1, 2, 3, the block layouts of test_gpu_noise_psd.py, masks none / turnarounds / NaN in
   flagged d, d 8 bytes off 16-byte alignment and repeated calls.
2. Against long double: r = d - P x in np.longdouble, then test_noise_host.welch_sums.  The bound of
   test_gpu_noise_psd.py (its docstring) plus the residual's own rounding: the kernel forms fl(d_t - fl((P x)_t)), so
     |r^_t - r_t| <= e_t = (|d_t| + 3 A_t) u,   A_t = |x_0| + |x_1 c_t| + |x_2 s_t|  (the magnitudes of P x's terms)
   (at most 2 roundings of the projection, relative to A_t >= |(P x)_t|, and one of the subtraction).  Carried through
   one window w of exact input x_w = h m r and perturbation dx_w (|dx_w| <= e_w = h m e elementwise), Parseval gives
     sum_k | |X_w + dX_w|^2 - |X_w|^2 | <= 2 ||X_w|| ||dX_w|| + ||dX_w||^2 <= NF (2 ||x_w|| ||e_w|| + ||e_w||^2),
   added over the block's windows.  W_b does not depend on the samples: the bound of test_gpu_noise_psd.py.  The
   scratch is a sentinel-guarded buffer, and the "many" layout runs several trips per CTA.
3. Exact sky: with d = P x_true + n (rounded once) and x = x_true, the sums equal those of n within the bound of 2 with
   e_t = (2 |d_t| + 4 A_t) u (d's own rounding and that of the host projection added).
4. The sky bias goes away (test_residual_pass_removes_sky_bias).
5. Argument checks: the C-ABI refusals, nt = 0 writes nothing, and the ValueErrors of noise_psd.
"""
import types
import zlib

import numpy as np
import pytest

from test_gpu_noise_psd import edges_of, layout, slots_per_block
from test_gpu_tod_reference import LD, SENTINEL, U, Guarded
from test_noise_host import M, NF, welch_sums

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def cm():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    assert np.finfo(np.longdouble).eps <= 2.0 ** -63, "the reference needs an extended-precision long double"
    import cosmomap2_b200
    assert int(cosmomap2_b200._cabi.lib.cm2_toeplitz_fft_points()) == M
    return cosmomap2_b200


def _dv():
    from cosmomap2_b200 import _device as dv
    return dv


# ---- inputs -----------------------------------------------------------------------------------------------------------

NPIX = 3000


def make_inputs(pol, nt, mask, rng):
    """(d, pix, cos, sin, x): pixel ids in [0, NPIX), flagged turnarounds (-1), NaN in flagged d for mask 'nan'"""
    pix = rng.integers(0, NPIX, nt).astype(np.int32)
    if mask in ("turnarounds", "nan"):
        pix[(np.arange(nt) % 5000) < 600] = -1
    phi = rng.uniform(0, 2 * np.pi, nt)
    c, s = np.cos(2 * phi), np.sin(2 * phi)
    x = rng.standard_normal(pol * NPIX) * np.tile([10.0, 1.0, 1.0][:pol], NPIX)
    d = rng.standard_normal(nt) * 3.0 + 0.5
    if mask == "nan":
        d[pix < 0] = np.nan
    return d, pix, c, s, x


def pointing(cm, pol, pix, c, s):
    """SparseLO over NPIX pixels with the given table and angles"""
    ang = types.SimpleNamespace(cos=c, sin=s) if pol > 1 else None
    return cm.SparseLO(NPIX, pix.size, pix, pol=pol, angle_processed=ang)


def exact_residual(d, pix, c, s, x, pol):
    """r = d - P x and A = sum of |terms of P x| in long double; 0 where pix < 0"""
    good = pix >= 0
    p = np.where(good, pix, 0).astype(np.int64)
    xv = np.asarray(x, dtype=LD).reshape(-1, pol)[p]
    cl, sl = np.asarray(c, dtype=LD), np.asarray(s, dtype=LD)
    if pol == 1:
        terms = [xv[:, 0]]
    elif pol == 2:
        terms = [xv[:, 0] * cl, xv[:, 1] * sl]
    else:
        terms = [xv[:, 0], xv[:, 1] * cl, xv[:, 2] * sl]
    px = sum(terms)
    A = sum(np.abs(t) for t in terms)
    dl = np.where(good, np.asarray(d, dtype=LD), LD(0))
    return np.where(good, dl - px, LD(0)), np.where(good, A, LD(0)), np.where(good, px, LD(0))


# ---- calls ------------------------------------------------------------------------------------------------------------

def _dev_copy(a, shift, dtype):
    import torch
    buf = torch.zeros(a.size + 4, dtype=dtype, device="cuda")
    buf[shift:shift + a.size] = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return buf, buf.data_ptr() + buf.element_size() * shift


def run_fused(cm, P, d, x, nt, nb, bs, edges, d_shift=0):
    """cm2_noise_psd_residual with d d_shift doubles into its buffer; outputs and scratch sentinel-guarded"""
    import torch
    dv = _dv()
    _keep, dptr = _dev_copy(d, d_shift, torch.float64)
    xd = dv.to_dev_f64(x)
    start = None if edges is None else dv.to_dev(np.asarray(edges, dtype=np.int64), torch.int64)
    S, W = Guarded(nb * (M + 1), torch.float64), Guarded(nb, torch.float64)
    scratch = Guarded(int(dv.call("cm2_noise_psd_scratch_bytes", nb)) // 8, torch.float64)
    rc = cm._cabi.lib.cm2_noise_psd_residual(dptr, dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.pol,
                                             dv.ptr(xd), nb, bs, dv.ptr(start), nt, S.ptr(), W.ptr(), scratch.ptr(), 1,
                                             dv.stream())
    assert rc == 0, cm._cabi.last_error()
    torch.cuda.synchronize()
    scr = scratch.result("scratch")
    run_fused.hann = scr[4 * M:4 * M + NF]
    return S.result("psd").reshape(nb, M + 1), W.result("wsum")


def run_unfused(cm, P, d, x, nt, nb, bs, edges):
    """cm2_noise_psd on r = d - P.mult(x) (torch), masked with P's pixel table"""
    import torch
    dv = _dv()
    r = (torch.from_numpy(np.ascontiguousarray(d)).cuda() - P.mult(dv.to_dev_f64(x))).contiguous()
    start = None if edges is None else dv.to_dev(np.asarray(edges, dtype=np.int64), torch.int64)
    S = torch.empty(nb * (M + 1), dtype=torch.float64, device="cuda")
    W = torch.empty(nb, dtype=torch.float64, device="cuda")
    scratch = torch.empty(int(dv.call("cm2_noise_psd_scratch_bytes", nb)) // 8 + 2, dtype=torch.float64, device="cuda")
    dv.call("cm2_noise_psd", dv.ptr(r), dv.ptr(P._pix_dev), nb, bs, dv.ptr(start), nt, dv.ptr(S), dv.ptr(W),
            dv.ptr(scratch), 1, dv.stream())
    torch.cuda.synchronize()
    return S.cpu().numpy().reshape(nb, M + 1), W.cpu().numpy()


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


# ---- 1. bit-identity with the unfused path ----------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("mask", ["none", "turnarounds", "nan"])
@pytest.mark.parametrize("lay", ["equal", "remainder", "starts"])
@pytest.mark.parametrize("pol", [1, 2, 3])
def test_fused_equals_unfused_bits(cm, pol, lay, mask):
    rng = np.random.default_rng(zlib.crc32(("%d%s%s" % (pol, lay, mask)).encode()))
    nt, nb, bs, edges = layout(lay)
    d, pix, c, s, x = make_inputs(pol, nt, mask, rng)
    P = pointing(cm, pol, pix, c, s)
    ref = run_unfused(cm, P, d, x, nt, nb, bs, edges)
    assert np.all(np.isfinite(ref[0])) and np.all(ref[1] >= 0)
    for shift in (0, 1, 0):                   # aligned, 8 bytes off 16-byte alignment, and a repeat
        got = run_fused(cm, P, d, x, nt, nb, bs, edges, d_shift=shift)
        assert same_bits(got[0], ref[0]), "psd differs from the unfused path (d shift %d)" % shift
        assert same_bits(got[1], ref[1]), "wsum differs from the unfused path (d shift %d)" % shift
    if edges is None:                         # the Python entry point (every block has windows): the sums, divided
        _, psd = cm.noise_psd(d, bs, P=P, x=x)
        assert same_bits(psd, ref[0] / ref[1][:, None])


# ---- 2. / 3. against long double --------------------------------------------------------------------------------------

def check_residual_sums(S, W, r, e, edges, pix, nt, what):
    """S, W against welch_sums of the exact residual r, with the per-sample perturbation bound e (module docstring)"""
    Sref, _ = welch_sums(r, edges, pix)
    _, Wref = welch_sums(r, edges, pix, h=run_fused.hann)
    h = np.asarray(run_fused.hann, dtype=LD)
    slots = slots_per_block(nt, edges)
    worst = 0.0
    for b in range(len(edges) - 1):
        n = int(edges[b + 1] - edges[b])
        nwin = (n - NF) // M + 1 if n >= NF else 0
        if nwin == 0:
            assert np.all(S[b] == 0.0) and W[b] == 0.0, "%s: block %d has no window but nonzero sums" % (what, b)
            continue
        energy = Sref[b, 0] + Sref[b, M] + 2 * np.sum(Sref[b, 1:M])          # = NF sum_w ||x_w||^2
        extra = LD(0)
        for w in range(nwin):
            t0 = int(edges[b]) + w * M
            hm = np.where(pix[t0:t0 + NF] >= 0, h, LD(0))
            xn = np.sqrt(np.sum((hm * r[t0:t0 + NF]) ** 2))
            en = np.sqrt(np.sum((hm * e[t0:t0 + NF]) ** 2))
            extra += NF * (2 * xn * en + en * en)
        bound = (2 * 8 * np.log2(M) + nwin + 4) * LD(U) * energy + extra
        err = np.sum(np.abs(S[b].astype(LD) - Sref[b]))
        assert np.all(np.isfinite(S[b])) and err <= bound, "%s: block %d: sum |dS| %.3g > bound %.3g" % (what, b, err, bound)
        werr = abs(LD(W[b]) - Wref[b])
        assert werr <= (17 + slots[b]) * LD(U) * Wref[b], "%s: block %d: |dW| = %.3g u W" % (what, b, werr / (U * Wref[b]))
        worst = max(worst, float(err / bound))
    return worst


@gpu
@pytest.mark.parametrize("lay", ["remainder", "starts", "many"])
@pytest.mark.parametrize("pol", [1, 2, 3])
def test_residual_sums_against_long_double(cm, pol, lay):
    rng = np.random.default_rng(zlib.crc32(("ld%d%s" % (pol, lay)).encode()))
    nt, nb, bs, edges = layout(lay)
    e_ = edges_of(nt, nb, bs, edges)
    d, pix, c, s, x = make_inputs(pol, nt, "nan", rng)
    P = pointing(cm, pol, pix, c, s)
    S, W = run_fused(cm, P, d, x, nt, nb, bs, edges, d_shift=1 if lay == "many" else 0)
    if lay == "many":
        assert max(slots_per_block(nt, e_)) >= 2
    r, A, _ = exact_residual(d, pix, c, s, x, pol)
    dl = np.where(pix >= 0, np.abs(np.nan_to_num(d)).astype(LD), LD(0))
    check_residual_sums(S, W, r, (dl + 3 * A) * LD(U), e_, pix, nt, "pol %d / %s" % (pol, lay))


@gpu
@pytest.mark.parametrize("pol", [1, 3])
def test_exact_sky_recovers_the_noise(cm, pol):
    rng = np.random.default_rng(40 + pol)
    nt, nb, bs, edges = layout("remainder")
    e_ = edges_of(nt, nb, bs, edges)
    _, pix, c, s, x = make_inputs(pol, nt, "turnarounds", rng)
    n = rng.standard_normal(nt)
    _, A, px = exact_residual(np.zeros(nt), pix, c, s, x, pol)
    d = px.astype(np.float64) + n                    # d = P x_true + n, rounded
    P = pointing(cm, pol, pix, c, s)
    S, W = run_fused(cm, P, d, x, nt, nb, bs, edges)
    nl = np.where(pix >= 0, n.astype(LD), LD(0))
    check_residual_sums(S, W, nl, (2 * np.abs(d).astype(LD) + 4 * A) * LD(U), e_, pix, nt, "exact sky, pol %d" % pol)


# ---- 4. the sky bias goes away ----------------------------------------------------------------------------------------

def bias_scenario(seed=11):
    """e2e_scenario of test_gpu_noise_psd.py with a sky 8x brighter: 4 detectors x 2^17 samples of a raster scan over
    800 pixels (I only), sky ~ 8 N(0, 1) (rms 8.25, 5.7x the noise rms of 1.45), 1/f noise with sigma 1,
    fknee = 0.05 cycles/sample and alpha = 1.  One sweep is 240 samples, so the scan fundamental is NF / 480 = bin 34.
    Rehearsed on the CPU with the oracle's P, BlockLO and Toeplitz operators, scipy.signal.welch and 512-coefficient
    bands, seed 11 (seed 12):
      pass 0, psd(d) / psd(n): median over bins and detectors 2.08 (1.85); at bins 34, 68, 102: 216, 292, 279
        (195, 389, 316); median over bins below 0.1 cycles/sample 9.98 (7.89)
      pass 1, psd(d - P x0) / psd(n): median 0.9998 (0.9998), every bin within [0.76, 1.72] ([0.66, 1.49])
      map rms error: GLS pass 1 / GLS pass 0 = 0.947 (0.970), GLS pass 1 / white (pass-0 weights) = 0.965 (0.978)"""
    from cosmomap2_b200 import synthetic
    ndet, ns = 4, 1 << 17
    sc = synthetic.raster_scan(ndet * ns, nside=32, ndet=ndet, nx=40, ny=20, samples_per_pixel=6.0, seed=seed,
                               with_data=False)
    sky = 8.0 * np.random.default_rng(seed + 1).standard_normal(sc.npix_full)
    noise = synthetic.one_over_f_noise(ns, ndet, 1.0, 0.05, 1.0, seed + 2)
    return sc, sky, noise, sky[sc.pix.astype(np.int64)] + noise


@gpu
def test_residual_pass_removes_sky_bias(cm):
    sc, sky, noise, d = bias_scenario()
    ns = sc.ns
    obs = np.unique(sc.pix[sc.pix >= 0])
    _, Pn = cm.noise_psd(noise, ns)

    def solve(bands, white):
        weights = [t[0] for t in bands]
        N = cm.BlockLO(ns, weights) if white else cm.BlockLO(ns, bands, offdiag=True)
        pix = sc.pix.astype(np.int64)
        pts = cm.ProcessTimeSamples(pix, sc.npix_full, pol=1, w=cm.BlockLO(ns, weights).diag)
        npix, obspix = pts.get_new_pixel
        assert npix == obs.size and np.array_equal(np.asarray(obspix)[:npix], obs)
        P = cm.SparseLO(npix, sc.nt, pix, pol=1, angle_processed=pts)
        x, info = cm.cg(P.T * N * P, P.T * (N * d), M=cm.BlockDiagonalPreconditionerLO(pts, npix, pol=1), rtol=1e-8,
                        maxiter=500)
        assert info == 0, "cg info %d" % info
        r = np.asarray(x) - sky[obs]
        return P, x, float(np.sqrt(np.mean((r - r.mean()) ** 2)))

    _, P0 = cm.noise_psd(d, ns)
    q0 = P0 / Pn
    assert np.median(q0[:, 34]) > 50, "pass 0 at the scan fundamental: %.1f" % np.median(q0[:, 34])
    assert np.median(q0[:, 1:NF // 10]) > 4, "pass 0 below 0.1 cycles/sample: %.2f" % np.median(q0[:, 1:NF // 10])
    b0 = cm.inverse_noise_bands(P0, 512)
    Pt, x0, e0 = solve(b0, False)
    _, _, ew = solve(b0, True)
    _, P1 = cm.noise_psd(d, ns, P=Pt, x=x0)
    q1 = P1 / Pn
    assert abs(np.median(q1) - 1.0) < 0.02, "pass 1 median %.4f" % np.median(q1)
    assert 0.5 < q1.min() and q1.max() < 2.0, "pass 1 bins in [%.3f, %.3f]" % (q1.min(), q1.max())
    _, _, e1 = solve(cm.inverse_noise_bands(P1, 512), False)
    assert e1 < 0.99 * e0 and e1 < 0.99 * ew, {"gls pass 0": e0, "gls pass 1": e1, "white": ew}


# ---- 5. argument checks -----------------------------------------------------------------------------------------------

@gpu
def test_cabi_refusals_and_empty_tod(cm):
    import torch
    dv = _dv()
    lib = cm._cabi.lib
    nt = NF
    rng = np.random.default_rng(5)
    d, pix, c, s, x = make_inputs(3, nt, "turnarounds", rng)
    dd, pd, cd, sd, xd = (dv.to_dev_f64(d), dv.pix_to_dev(pix), dv.to_dev_f64(c), dv.to_dev_f64(s), dv.to_dev_f64(x))
    S, W = Guarded(M + 1, torch.float64), Guarded(1, torch.float64)
    scratch = torch.empty(int(dv.call("cm2_noise_psd_scratch_bytes", 1)) // 8 + 2, dtype=torch.float64, device="cuda")

    def call(d_=dd, p_=pd, c_=cd, s_=sd, pol=3, x_=xd, n=nt):
        ptr = lambda t: None if t is None else t.data_ptr()
        return lib.cm2_noise_psd_residual(ptr(d_), ptr(p_), ptr(c_), ptr(s_), pol, ptr(x_), 1, max(n, 1), None, n,
                                          S.ptr(), W.ptr(), scratch.data_ptr(), 1, dv.stream())

    refusals = {"d NULL": dict(d_=None), "pix NULL": dict(p_=None), "x NULL": dict(x_=None), "pol 0": dict(pol=0),
                "pol 4": dict(pol=4), "cos NULL, pol 2": dict(c_=None, pol=2), "sin NULL, pol 2": dict(s_=None, pol=2),
                "cos NULL, pol 3": dict(c_=None), "sin NULL, pol 3": dict(s_=None)}
    for what, kw in refusals.items():
        assert call(**kw) == -1, what                 # CM2_ERR_ARG
        assert "cm2_noise_psd_residual" in cm._cabi.last_error(), what
    torch.cuda.synchronize()
    untouched = lambda g: bool((g.buf == SENTINEL).all().item())
    assert untouched(S) and untouched(W), "a refused call wrote its outputs"
    assert call(n=0) == 0 and call(n=0, d_=dd, c_=None, s_=None, pol=1) == 0
    torch.cuda.synchronize()
    assert untouched(S) and untouched(W), "nt = 0 wrote its outputs"
    assert call(c_=None, s_=None, pol=1) == 0, "pol 1 does not need the angles"
    torch.cuda.synchronize()
    assert np.all(np.isfinite(S.result("psd"))) and W.result("wsum")[0] > 0


@gpu
def test_noise_psd_value_errors(cm):
    rng = np.random.default_rng(6)
    nt = 2 * NF
    d, pix, c, s, x = make_inputs(2, nt, "turnarounds", rng)
    P = pointing(cm, 2, pix, c, s)
    with pytest.raises(ValueError, match="not both"):
        cm.noise_psd(d, NF, pix=pix, P=P, x=x)
    with pytest.raises(ValueError, match="both P and x"):
        cm.noise_psd(d, NF, P=P)
    with pytest.raises(ValueError, match="both P and x"):
        cm.noise_psd(d, NF, x=x)
    with pytest.raises(ValueError, match="SparseLO"):
        cm.noise_psd(d, NF, P=P.T * P, x=x)
    with pytest.raises(ValueError, match="SparseLO"):
        cm.noise_psd(d, NF, P=cm.BlockLO(NF, [1.0, 1.0]), x=x)
    with pytest.raises(ValueError, match="x has"):
        cm.noise_psd(d, NF, P=P, x=x[:-1])
    with pytest.raises(ValueError, match="x has"):
        cm.noise_psd(d, NF, P=P, x=np.r_[x, x[:2]])
    with pytest.raises(ValueError, match="rows"):
        cm.noise_psd(d[:-1], NF, P=P, x=x)
    # a device map is accepted, and gives the host map's result
    import torch
    _, a = cm.noise_psd(d, NF, P=P, x=x)
    _, b = cm.noise_psd(torch.from_numpy(d).cuda(), NF, P=P, x=torch.from_numpy(x).cuda())
    assert same_bits(a, b)
