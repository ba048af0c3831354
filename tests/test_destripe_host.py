"""CPU-only: the destriper's prior from the PSD, ``baseline_prior_bands`` (cosmomap2_b200/noise.py, DESIGN.md
section 4f).

    S_b(F) = (1/L) sum_{m<L} C_b(f_m) K_L(f_m),  f_m = (F + m)/L folded into [-1/2, 1/2],  K_L = [sin(pi L f)/(L sin pi f)]^2
    bands  = the Bartlett-tapered coefficients of 1/S_b,  weights = 1/sigma2_b
"""
import numpy as np
import pytest

M = 8192                     # cm2_toeplitz_fft_points()
NF = 2 * M
F = np.arange(M + 1) / NF


def _symbol(t, nomega=1 << 16):
    """t_0 + 2 sum_j t_j cos(j omega) on a dense grid of [0, pi]"""
    c = np.zeros(2 * nomega)
    c[:len(t)] = t
    c[2 * nomega - len(t) + 1:] = t[1:][::-1]
    return np.fft.rfft(c).real


def _one_over_f(fknee, alpha, sigma2=1.0):
    P = np.empty(M + 1)
    P[1:] = sigma2 * (1.0 + (fknee / F[1:]) ** alpha)
    P[0] = P[1]
    return P


def _direct_S(C, L, Cfun=None):
    """The aliased sum by a plain loop over the aliases and frequencies: C interpolated linearly in |f| (or the
    analytic Cfun), K_L from its definition with K_L(0) = 1."""
    S = np.zeros(M + 1)
    for m in range(L):
        f = (F + m) / L
        f = f - np.round(f)
        with np.errstate(invalid="ignore", divide="ignore"):
            K = (np.sin(np.pi * L * f) / (L * np.sin(np.pi * f))) ** 2
        K[f == 0] = 1.0
        c = Cfun(np.abs(f)) if Cfun is not None else np.interp(np.abs(f), F, C)
        S += c * K
    return S / L


def _bands_of(S, nband):
    c = np.fft.irfft(1.0 / S, NF)[:nband]
    return c * (1.0 - np.arange(nband) / nband)


@pytest.mark.parametrize("L", [2, 7, 100, 1000])
def test_matches_the_direct_evaluation(L):
    from cosmomap2_b200.noise import baseline_prior_bands
    psd = np.vstack([_one_over_f(0.05, 1.0), _one_over_f(0.01, 2.0, 2.5)])
    nband = 64
    w, bands = baseline_prior_bands(psd, L, nband)
    for b in range(2):
        sigma2 = np.median(psd[b, np.arange(M + 1) >= M / 2])
        assert w[b] == pytest.approx(1.0 / sigma2, rel=1e-15)
        S = _direct_S(np.maximum(psd[b] - sigma2, 0.0), L)
        ref = _bands_of(S, nband)
        np.testing.assert_allclose(bands[b], ref, rtol=0, atol=1e-12 * np.max(np.abs(ref)))


def test_explicit_white_level():
    from cosmomap2_b200.noise import baseline_prior_bands
    psd = _one_over_f(0.05, 1.5)[None, :]
    w, bands = baseline_prior_bands(psd, 50, 32, white=[0.9])
    assert w[0] == pytest.approx(1 / 0.9, rel=1e-15)
    ref = _bands_of(_direct_S(psd[0] - 0.9, 50), 32)
    np.testing.assert_allclose(bands[0], ref, rtol=0, atol=1e-12 * np.max(np.abs(ref)))


@pytest.mark.parametrize("nband", [1, 2, 17, 256, 4096])
def test_symbol_is_positive(nband):
    from cosmomap2_b200.noise import baseline_prior_bands
    psd = np.vstack([_one_over_f(0.05, 1.0), _one_over_f(1e-3, 2.0), _one_over_f(0.2, 3.0, 0.1)])
    for L in (10, 300):
        _, bands = baseline_prior_bands(psd, L, nband)
        for b, t in enumerate(bands):
            assert t.shape == (nband,)
            assert np.min(_symbol(t)) > 0.0, "block %d, L %d, nband %d" % (b, L, nband)


def test_analytic_aliased_sums():
    """Two power laws with an exact answer.  C = c (exponent 0): the mean of L white samples of variance c is white
    across baselines with variance c/L, so S = c/L at every F (sum_m K_L(f_m) = L).  C = c |f| (exponent 1): linear
    interpolation is exact, so S equals the aliased sum of the analytic C at the exact alias frequencies."""
    from cosmomap2_b200.noise import baseline_prior_bands
    nband = M
    for L in (1, 4, 33, 200):
        _, bands = baseline_prior_bands(np.full((1, M + 1), 1.0 + 3.0), L, nband, white=[1.0])
        t = bands[0]
        assert t[0] == pytest.approx(L / 3.0, rel=1e-12)
        assert np.max(np.abs(t[1:])) <= 1e-12 * t[0]
        if L == 1:                           # C(0) = 0 and no alias: S(0) = 0, no prior
            with pytest.raises(ValueError, match="noise block 0"):
                baseline_prior_bands((1.0 + 5.0 * F)[None, :], L, 128, white=[1.0])
            continue
        _, bands = baseline_prior_bands((1.0 + 5.0 * F)[None, :], L, 128, white=[1.0])
        ref = _bands_of(_direct_S(None, L, Cfun=lambda f: 5.0 * f), 128)
        np.testing.assert_allclose(bands[0], ref, rtol=0, atol=1e-12 * np.max(np.abs(ref)))


def test_value_errors():
    from cosmomap2_b200.noise import baseline_prior_bands
    white_only = np.ones((2, M + 1))
    with pytest.raises(ValueError, match="noise block 0"):
        baseline_prior_bands(white_only, 10, 8)
    mixed = np.vstack([_one_over_f(0.05, 1.0), np.ones(M + 1)])
    with pytest.raises(ValueError, match="noise block 1"):
        baseline_prior_bands(mixed, 10, 8)
    psd = _one_over_f(0.05, 1.0)[None, :]
    for nband in (0, -1, M + 1):
        with pytest.raises(ValueError, match="nband"):
            baseline_prior_bands(psd, 10, nband)
    with pytest.raises(ValueError, match="baseline length"):
        baseline_prior_bands(psd, 0, 8)
    with pytest.raises(ValueError, match="white"):
        baseline_prior_bands(psd, 10, 8, white=[1.0, 1.0])
