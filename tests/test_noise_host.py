"""CPU-only: the definition of the noise estimate (cosmomap2_b200/noise.py, cm2_noise_psd) and the host step that turns
PSDs into N^-1 bands.

    welch_sums   the per-block sums S_b(k), W_b of the definition in np.longdouble, the reference the GPU tests use
    bands        c_b = irfft(1/P_b, NF)[:nband] with the Bartlett lag taper: a positive Toeplitz symbol for any P_b > 0
"""
import numpy as np
import pytest
import scipy.signal

LD = np.longdouble
M = 8192                     # cm2_toeplitz_fft_points()
NF = 2 * M


def windows_of(n):
    return (n - NF) // M + 1 if n >= NF else 0


def hann(M=M):
    """h_t = sin^2(pi t / 2M), t < 2M, in long double: pi in long double (np.pi, a double, is off by 1e-16, which is
    1e-12 relative to sin near t = 2M) and the argument folded to [0, pi/2]"""
    t = np.arange(2 * M)
    return np.sin(4 * np.arctan(LD(1)) * np.minimum(t, 2 * M - t).astype(LD) / LD(2 * M)) ** 2


def welch_sums(d, edges, pix=None, M=M, h=None):
    """S[b][k] = sum_w |X_w(k)|^2 (k = 0..M) and W[b] = sum_w sum_t (h_t m_t)^2 per noise block [edges[b], edges[b+1]),
    in long double: windows of 2M samples at hop M from the block's first sample, x_t = h_t m_t d_t, h_t = sin^2(pi t/2M)
    (or the given table), m_t = [pix_t >= 0], flagged samples selected away (NaN there does not propagate)."""
    NF = 2 * M
    h = hann(M) if h is None else np.asarray(h, dtype=LD)
    nb = len(edges) - 1
    S = np.zeros((nb, M + 1), dtype=LD)
    W = np.zeros(nb, dtype=LD)
    for b in range(nb):
        s, e = int(edges[b]), int(edges[b + 1])
        nw = (e - s - NF) // M + 1 if e - s >= NF else 0
        if nw == 0:
            continue
        t0 = s + M * np.arange(nw)
        idx = t0[:, None] + np.arange(NF)[None, :]
        hm = np.broadcast_to(h, idx.shape) if pix is None else np.where(pix[idx] >= 0, h, LD(0))
        x = np.where(hm > 0, hm * np.asarray(d, dtype=LD)[idx], LD(0))
        X = np.fft.rfft(x, axis=1)
        S[b] = np.sum(X.real ** 2 + X.imag ** 2, axis=0)
        W[b] = np.sum(hm ** 2)
    return S, W


def test_long_double_definition_is_scipy_welch():
    """Without flags S_b / W_b is scipy.signal.welch(hann, 50 % overlap, no detrend, two-sided)[:M+1], per block."""
    assert np.finfo(LD).eps <= 2.0 ** -63, "the reference needs an extended-precision long double"
    rng = np.random.default_rng(3)
    lens = [NF, NF + M, NF + 3 * M - 1, NF + 2 * M + 1]
    edges = np.r_[0, np.cumsum(lens)]
    d = rng.standard_normal(edges[-1]) * 2.0 + 0.5
    S, W = welch_sums(d, edges)
    for b, (s, e) in enumerate(zip(edges[:-1], edges[1:])):
        _, P = scipy.signal.welch(d[s:e], fs=1.0, window="hann", nperseg=NF, noverlap=M, detrend=False,
                                  scaling="density", return_onesided=False)
        got = (S[b] / W[b]).astype(np.float64)
        rel = np.max(np.abs(got - P[:M + 1]) / P[:M + 1])
        assert rel < 1e-12, "block %d: %.3g" % (b, rel)
        assert windows_of(e - s) == (e - s - NF) // M + 1


def test_flagged_nan_is_selected_away():
    rng = np.random.default_rng(4)
    d = rng.standard_normal(2 * NF)
    pix = np.zeros(d.size, dtype=np.int32)
    pix[100:3000] = -1
    d2 = d.copy()
    d2[100:3000] = np.nan
    S1, W1 = welch_sums(d, [0, d.size], pix)
    S2, W2 = welch_sums(d2, [0, d.size], pix)
    assert np.array_equal(S1, S2) and np.array_equal(W1, W2) and np.all(np.isfinite(S2))


def _symbol(t, nomega=1 << 16):
    """f(omega) = t_0 + 2 sum_j t_j cos(j omega) on a dense grid of [0, pi]"""
    c = np.zeros(2 * nomega)
    c[:len(t)] = t
    c[2 * nomega - len(t) + 1:] = t[1:][::-1]
    return np.fft.rfft(c).real


def _one_over_f_psd(fknee, alpha, sigma=1.0):
    f = np.arange(M + 1) / NF
    P = np.empty(M + 1)
    P[1:] = sigma ** 2 * (1.0 + (fknee / f[1:]) ** alpha)
    P[0] = P[1]
    return P


def test_bartlett_band_has_a_positive_symbol():
    from cosmomap2_b200.noise import inverse_noise_bands
    rng = np.random.default_rng(5)
    psds = [np.exp(rng.normal(0.0, 2.0, M + 1)) for _ in range(4)]
    psds += [rng.uniform(1e-6, 1.0, M + 1), _one_over_f_psd(1e-2, 2.0), _one_over_f_psd(0.05, 3.0),
             _one_over_f_psd(1e-3, 1.0, 0.1)]
    for nband in (2, 3, 17, 64, 1000, 4096, M):
        bands = inverse_noise_bands(np.array(psds), nband)
        for i, t in enumerate(bands):
            assert t.shape == (nband,)
            f = _symbol(t)
            assert np.min(f) > 0.0, "PSD %d, nband %d: symbol min %.3g" % (i, nband, np.min(f))


def test_one_coefficient_is_the_mean_inverse_psd():
    from cosmomap2_b200.noise import inverse_noise_bands
    rng = np.random.default_rng(6)
    P = rng.uniform(0.5, 3.0, (3, M + 1))
    t = inverse_noise_bands(P, 1)
    for b in range(3):
        full = np.r_[P[b], P[b, 1:M][::-1]]                # the two-sided circle of NF frequencies
        assert t[b].shape == (1,)
        assert t[b][0] == pytest.approx(np.mean(1.0 / full), rel=1e-14)


def test_bands_match_the_definition():
    from cosmomap2_b200.noise import inverse_noise_bands
    rng = np.random.default_rng(7)
    P = rng.uniform(0.5, 3.0, (2, M + 1))
    nband = 300
    t = inverse_noise_bands(P, nband)
    for b in range(2):
        full = np.r_[P[b], P[b, 1:M][::-1]]
        c = np.real(np.fft.ifft(1.0 / full))[:nband]
        np.testing.assert_allclose(t[b], c * (1.0 - np.arange(nband) / nband), rtol=0, atol=1e-15 * np.max(1 / P))


def test_value_errors():
    from cosmomap2_b200.noise import inverse_noise_bands, noise_psd
    P = np.ones((3, M + 1))
    for bad, what in ((0.0, "zero"), (-1.0, "negative"), (np.nan, "NaN"), (np.inf, "inf")):
        Q = P.copy()
        Q[2, 17] = bad
        with pytest.raises(ValueError, match="block 2"):
            inverse_noise_bands(Q, 10)
    for nband in (0, M + 1):
        with pytest.raises(ValueError):
            inverse_noise_bands(P, nband)
    d = np.zeros(3 * NF)
    with pytest.raises(ValueError, match="block 1 "):             # blocks of NF, NF - 1, NF + 1 samples
        noise_psd(d, [NF, NF - 1, NF + 1])
    with pytest.raises(ValueError, match="block 0 "):
        noise_psd(d[:NF - 1], NF)
    with pytest.raises(ValueError):                                # sizes not adding up to the TOD
        noise_psd(d, [NF, NF])
