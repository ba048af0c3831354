"""Host side of the noise simulation (DESIGN.md section 4d): a NumPy transcription of the generator -- Philox4x32-10
and the Box-Muller mapping of cm2_noise_simulate -- that the GPU tests regenerate the stream with, checked here against
the Random123 known-answer vectors, and noise_sim_bands against its definition.  No GPU needed."""
import numpy as np
import pytest

LD = np.longdouble
PI_LD = LD("3.141592653589793238462643383279502884")
M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 on arrays: ctr (4, n) and key (2, n) of 32-bit words held in uint64; returns (4, n)."""
    c = [np.asarray(x, dtype=np.uint64) & MASK for x in ctr]
    k0, k1 = (np.asarray(x, dtype=np.uint64) & MASK for x in key)
    for r in range(10):
        if r:
            k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
        p0, p1 = M0 * c[0], M1 * c[2]              # < 2^64: exact in uint64
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & MASK, p1 & MASK, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & MASK,
             p0 & MASK]
    return np.array(c)


def uniforms(x):
    """(u1, u2) from Philox output words: a = (x0:x1) >> 11, c = (x2:x3) >> 11, u1 = (a + 1) 2^-53, u2 = c 2^-53."""
    a = ((x[0] << np.uint64(32)) | x[1]) >> np.uint64(11)
    c = ((x[2] << np.uint64(32)) | x[3]) >> np.uint64(11)
    return (a + np.uint64(1)).astype(np.float64) * 2.0 ** -53, c.astype(np.float64) * 2.0 ** -53


def noise_stream(seed, realization, block_id, r0, r1):
    """w(r) for r0 <= r < r1 (r0 even) in long double, and rho = sqrt(-2 ln u1) of each sample's pair."""
    assert r0 % 2 == 0
    p = np.arange(r0 // 2, -(-r1 // 2), dtype=np.int64)
    pu = p.view(np.uint64)
    n = p.size
    x = philox4x32_10([pu & MASK, pu >> np.uint64(32), np.full(n, block_id), np.full(n, realization)],
                      [np.full(n, seed & 0xFFFFFFFF), np.full(n, seed >> 32)])
    u1, u2 = uniforms(x)
    rho = np.sqrt(LD(-2) * np.log(u1.astype(LD)))
    ang = LD(2) * PI_LD * u2.astype(LD)
    w = np.empty(2 * n, dtype=LD)
    w[0::2], w[1::2] = rho * np.cos(ang), rho * np.sin(ang)
    rr = np.repeat(rho, 2)
    return w[:r1 - r0], np.asarray(rr[:r1 - r0], dtype=np.float64)


KAT = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
       ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
       ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]


@pytest.mark.parametrize("ctr,key,out", KAT)
def test_philox_known_answers(ctr, key, out):
    got = philox4x32_10([[c] for c in ctr], [[k] for k in key])[:, 0]
    assert [int(v) for v in got] == list(out)


def test_uniform_mapping():
    """u1 in (0, 1] and u2 in [0, 1), both exact: the extremes and one pattern per bit position."""
    x = np.array([[0, 0xffffffff, 0x80000000, 0], [0, 0xffffffff, 0, 0x800],
                  [0, 0xffffffff, 0x80000000, 0], [0, 0xffffffff, 0, 0x7ff]], dtype=np.uint64)
    u1, u2 = uniforms(x)
    assert u1.tolist() == [2.0 ** -53, 1.0, 0.5 + 2.0 ** -53, 2.0 ** -53 + 2.0 ** -53]
    assert u2.tolist() == [0.0, 1.0 - 2.0 ** -53, 0.5, 0.0]
    rng = np.random.default_rng(3)
    w = rng.integers(0, 1 << 32, size=(4, 1000), dtype=np.uint64)
    u1, u2 = uniforms(w)
    a = (w[0] * np.uint64(1 << 32) + w[1]) >> np.uint64(11)
    assert np.all(u1 * 2.0 ** 53 == (a + np.uint64(1)).astype(np.float64))
    assert np.all((u1 > 0) & (u1 <= 1) & (u2 >= 0) & (u2 < 1))


def test_stream_pairs_and_moments():
    """Samples 2p and 2p+1 come from one call; a window starting at an odd pair regenerates the same samples; the
    stream has unit variance and no lag-1 correlation within 5 / sqrt(n)."""
    w, rho = noise_stream(7, 2, 5, -64, 40000)
    w2, _ = noise_stream(7, 2, 5, -10, 100)
    assert np.array_equal(w[54:54 + 110], w2)
    assert np.allclose(rho[0::2] ** 2, (w[0::2] ** 2 + w[1::2] ** 2).astype(np.float64), rtol=1e-15)
    x = w.astype(np.float64)
    n = x.size
    assert abs(x.mean()) < 5 / np.sqrt(n)
    assert abs(x.var() - 1) < 5 * np.sqrt(2.0 / n)
    assert abs(np.mean(x[1:] * x[:-1])) < 5 / np.sqrt(n)


def _noise():
    from cosmomap2_b200 import noise
    return noise


def _psd(nb, M, rng):
    f = np.arange(M + 1) / (2.0 * M)
    return np.array([(1 + (0.01 / np.maximum(f, 0.5 / M)) ** (1 + rng.random())) * (0.5 + rng.random())
                     for _ in range(nb)])


@pytest.mark.parametrize("M,nband", [(64, 1), (64, 7), (64, 64), (8192, 1), (8192, 4096), (8192, 8192)])
def test_noise_sim_bands_formula(M, nband):
    noise = _noise()
    rng = np.random.default_rng(M + nband)
    psd = _psd(3, M, rng)
    t = noise.noise_sim_bands(psd, nband)
    assert len(t) == 3 and all(x.shape == (nband,) for x in t)
    NF = 2 * M
    for b in range(3):
        s = np.sqrt(psd[b])
        sym = np.r_[s, s[1:M][::-1]]                      # the full circle of NF frequencies
        j = np.arange(nband)
        c = np.array([np.sum(sym * np.cos(2 * np.pi * np.arange(NF) * jj / NF)) / NF for jj in j])
        ref = c * (1 - j / nband)
        assert np.allclose(t[b], ref, rtol=0, atol=1e-13 * np.max(s))
        if nband == 1:
            assert t[b][0] == pytest.approx(np.mean(sym), rel=1e-14)


def test_noise_sim_bands_shapes_and_refusals():
    noise = _noise()
    psd = _psd(2, 64, np.random.default_rng(1))
    assert len(noise.noise_sim_bands(psd[0], 4)) == 1                 # one PSD: one band
    for nband in (0, 65):
        with pytest.raises(ValueError):
            noise.noise_sim_bands(psd, nband)
    for bad in (0.0, -1.0, np.nan, np.inf):
        p = psd.copy()
        p[1, 5] = bad
        with pytest.raises(ValueError, match="block 1"):
            noise.noise_sim_bands(p, 4)


def test_inverse_bands_unchanged_by_the_shared_helper():
    """inverse_noise_bands through the shared helper: the same bits as its formula written out."""
    noise = _noise()
    psd = _psd(3, 8192, np.random.default_rng(2))
    for nband in (1, 48, 4096):
        t = noise.inverse_noise_bands(psd, nband)
        c = np.fft.irfft(1.0 / psd, 2 * 8192, axis=1)[:, :nband]
        ref = c * (1.0 - np.arange(nband) / float(nband))
        for b in range(3):
            assert np.array_equal(t[b], ref[b])
