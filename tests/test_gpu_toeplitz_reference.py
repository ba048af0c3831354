"""The banded Toeplitz noise kernels against an extended-precision reference, called through the C ABI so that every
instantiation (direct or FFT, one-CTA or 2-CTA-cluster windows, the NLAG of the fused kernel) is chosen here and not
by the planner's band thresholds in linearoperators.py.

    cm2_noise_toeplitz_apply       k_toeplitz, the direct kernel: persistent CTAs over 1024-sample tiles
    cm2_noise_toeplitz_fft_apply   k_toeplitz_fft<512>, <1024> (CM2_FFT_THREADS=1024) and <512, true>: persistent
                                   CTAs (clusters) over overlap-save windows of 2M (4M) samples
    cm2_amatvec_toeplitz           k_amatvec_toeplitz<POL, NLAG>: y = P^T T P x in one TOD pass

All three walk their tiles or windows in trips over a persistent grid, so each runs here at >= 3 trips as well as at
one, on block layouts with empty blocks, 1-sample blocks, blocks shorter than the band, blocks of k S and k S +- 1
samples (S = outputs per window), odd block starts, equal blocks with and without a remainder, and a different band
per block.

Reference: y_b = T_b v_b per noise block (zero boundaries), by overlap-save np.fft in np.longdouble (NumPy >= 2
transforms long double in long double; checked against np.convolve below).  Bounds, u = 2^-53:
  direct, per element:      |y_j - ref_j| <= (L + 2) u sum_k |a_k| (|v_{j-k}| + |v_{j+k}|)   (one FMA per lag)
  FFT, per window, normwise: ||y_w - ref_w||_2 <= 8 log2(N) u max_k |H_b(k)| ||v_w||_2, N the complex transform
                            length, H_b the DFT of block b's circularly arranged band, v_w the window's input
  fused, per pixel component: (n_i + 2 NLAG + 6) u S_i, S_i the sum over the pixel's samples of
                            |f_t| sum_k |a_k| (|Px|_{t-k} + |Px|_{t+k}), |Px|_s = |x_0| + |x_1 c_s| + |x_2 s_s|
The noise kernels are deterministic per output: a multi-block call must equal, bit for bit, one call per block on
that block's data and band (at most one window or tile per CTA there), and the same call on inputs and outputs 8 bytes
off 16-byte alignment.  Every output sits in a sentinel-guarded buffer: nothing may be written outside it, and every
output sample must be written.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from test_gpu_tod_reference import (LD, SENTINEL, U, Guarded, Tod, check_map, make_map, projection, scatter_ref,
                                    sm_count)

gpu = pytest.mark.gpu
CM2_ERR_ARG, CM2_ERR_UNSUPPORTED = -1, -3
TILE_DIRECT = 1024                # k_toeplitz outputs per CTA tile
SMEM_PER_SM = 228 * 1024          # B200 shared memory per SM (1 kB of it reserved per CTA)


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


# ---- the reference ---------------------------------------------------------------------------------------------------

def band_apply(v, a):
    """T v for one block in long double: y_j = sum_{|k| < L} a_|k| v_{j-k}, v = 0 outside the block (overlap-save)."""
    v, a = np.asarray(v, dtype=LD), np.asarray(a, dtype=LD)
    n, L = v.size, a.size
    H = L - 1
    if n == 0 or H == 0:
        return a[0] * v
    F = min(1 << (n + 2 * H - 1).bit_length(), max(1 << (4 * H).bit_length(), 1 << 15))
    C = F - 2 * H                                     # outputs per chunk
    nch = -(-n // C)
    pad = np.zeros(nch * C + 2 * H, dtype=LD)
    pad[H:H + n] = v
    X = np.lib.stride_tricks.sliding_window_view(pad, F)[::C]
    hc = np.zeros(F, dtype=LD)
    hc[:L] = a
    hc[F - H:] = a[1:][::-1]
    Hf = np.fft.rfft(hc)
    y = np.empty(nch * C, dtype=LD)
    for i in range(0, nch, 64):
        Y = np.fft.irfft(np.fft.rfft(X[i:i + 64], axis=1) * Hf, F, axis=1)
        y[i * C:(i + Y.shape[0]) * C] = Y[:, H:H + C].ravel()
    return y[:n]


def test_reference_matches_convolve():
    """The long-double overlap-save reference against long-double np.convolve, with one and several chunks."""
    assert np.finfo(np.longdouble).eps <= 2.0 ** -63, "the reference needs an extended-precision long double"
    rng = np.random.default_rng(0)
    for n, L in ((1, 1), (1, 5), (7, 3), (100, 300), (4000, 300), (40000, 47), (40000, 600), (3000, 9344)):
        v = rng.standard_normal(n).astype(LD)
        a = rng.standard_normal(L).astype(LD)
        full = np.convolve(v, np.concatenate([a[1:][::-1], a]))          # index j + L - 1 holds y_j
        ref = full[L - 1:L - 1 + n]
        got = band_apply(v, a)
        scale = np.convolve(np.abs(v), np.abs(np.concatenate([a[1:][::-1], a])))[L - 1:L - 1 + n]
        rel = float(np.max(np.abs(got - ref) / scale))
        assert rel < 2.0 ** -58, "n=%d L=%d: %.3g relative to sum |a| |v|" % (n, L, rel)


# ---- block layouts ---------------------------------------------------------------------------------------------------

class Layout:
    """Noise blocks of the C ABI: equal blocks of `bs` (the last one up to nt) or blk_start boundaries."""

    def __init__(self, name, nt, nb, bs=0, start=None):
        self.name, self.nt, self.nb, self.bs = name, int(nt), int(nb), int(bs)
        self.start = None if start is None else np.asarray(start, dtype=np.int64)
        self.edges = self.start if start is not None else np.r_[np.arange(self.nb) * self.bs, self.nt]
        assert self.edges[0] == 0 and self.edges[-1] == self.nt and np.all(np.diff(self.edges) >= 0)
        self._dev = None

    def bounds(self):
        return list(zip(self.edges[:-1].tolist(), self.edges[1:].tolist()))

    def block_id(self):
        return np.repeat(np.arange(self.nb), np.diff(self.edges))

    def args(self):
        import torch
        if self.start is not None and self._dev is None:
            self._dev = _dv().to_dev(self.start, torch.int64)
        return self.nb, self.bs, _dv().ptr(self._dev)

    def __repr__(self):
        return "%s(nt=%d, %d blocks)" % (self.name, self.nt, self.nb)


def noise_layout(name, S, L, cap, rng):
    """Layouts of >= 3 trips for a kernel with S outputs per window (tile) and `cap` = S * (windows per trip): every
    block holds at most cap samples, so that one call per block runs at most one window per CTA."""
    B = cap // 2 + 7
    if name == "equal":
        return Layout(name, 7 * B, 7, B)
    if name == "remainder":
        return Layout(name, 7 * B + B // 2 + 3, 7, B)
    lens = [0, 1, 1, 0, max(L // 2, 1), 3, S, S - 1, S + 1, 0, 2 * S + 1, 2 * S - 1, 2 * S, 7, max(L - 1, 2), 1]
    while sum(lens) < 3 * cap:
        lens.append(int(rng.integers(cap // 2, cap + 1)) if rng.random() < 0.6 else
                    int(rng.choice([1, 2, 5, L, S - 1, S + 1, 3 * S])))
    lens += [int(rng.integers(1, S)), 0]
    return Layout(name, sum(lens), len(lens), start=np.r_[0, np.cumsum(lens)])


def make_bands(nb, L, rng):
    """A different band per block: a_0 in [1, 2], a_1 .. a_{L-1} random of size 1 / sqrt(L), either sign."""
    a = rng.standard_normal((nb, L)) / np.sqrt(L) * (0.5 + 0.5 * rng.random((nb, 1)))
    a[:, 0] = 1.0 + rng.random(nb)
    return a


def make_tod(nt, rng):
    """Random signs and magnitudes in [0.5, 1.5], so that the per-element bound sum |a| |v| never vanishes."""
    return np.where(rng.random(nt) < 0.5, -1.0, 1.0) * rng.uniform(0.5, 1.5, nt)


# ---- the noise kernels -----------------------------------------------------------------------------------------------

def fft_points():
    return int(_dv().call("cm2_toeplitz_fft_points"))


def fft_geometry(L, pair):
    """(window samples, head HD, outputs per window S) as in toeplitz_fft.cu"""
    NF = (4 if pair else 2) * fft_points()
    HD = (L - 1) + ((L - 1) & 1)
    return NF, HD, (NF - HD - (L - 1)) & ~1


class NoiseKernel:
    """One kernel instantiation and the device image of its per-block operator: the bands (direct) or the packed
    transfer tables (FFT)."""

    def __init__(self, L, pair, bands):
        from cosmomap2_b200 import linearoperators as lo
        dv = _dv()
        self.L, self.pair = L, pair
        if pair is None:
            self.op = dv.to_dev_f64(bands.ravel())
            self.stride = 8 * L
        else:
            coef = lo.toeplitz_fft_tables(bands, L, fft_points(), pair=bool(pair))
            self.op = dv.to_dev_f64(coef.view(np.float64).reshape(-1))
            self.stride = coef[0].nbytes

    def __call__(self, nb, bs, start, d, out, nt, block=0):
        """The C ABI call on raw pointers; `block` selects the block's band / table.  Returns the status."""
        import torch
        dv = _dv()
        op = self.op.data_ptr() + block * self.stride
        if self.pair is None:
            scratch = torch.empty(nb + 1, dtype=torch.int64, device="cuda")
            return _lib().cm2_noise_toeplitz_apply(op, self.L, nb, bs, start, d, out, nt, dv.ptr(scratch), dv.stream())
        scratch = torch.empty(int(dv.call("cm2_toeplitz_fft_scratch_bytes", nb)) // 8 + 2, dtype=torch.float64,
                              device="cuda")
        return _lib().cm2_noise_toeplitz_fft_apply(op, self.L, nb, bs, start, d, out, nt, dv.ptr(scratch), 1,
                                                   self.pair, dv.stream())

    def name(self):
        return "direct" if self.pair is None else "FFT pair=%d" % self.pair


def checked(rc, what):
    assert rc == 0, "%s failed (%d): %s" % (what, rc, _cabi_error())


def _cabi_error():
    from cosmomap2_b200 import _cabi
    return _cabi.last_error()


def written(out, what):
    unwritten = np.flatnonzero(out.view(np.int64) == SENTINEL)
    assert unwritten.size == 0, "%s: %d outputs not written, first at %d" % (what, unwritten.size, unwritten[0])
    return out


def check_direct(y, v, bands, lay, what):
    L = bands.shape[1]
    worst = 0.0
    for b, (s, e) in enumerate(lay.bounds()):
        if e == s:
            continue
        ref = band_apply(v[s:e], bands[b])
        bound = (L + 2) * LD(U) * band_apply(np.abs(v[s:e]), np.abs(bands[b]))
        err = np.abs(y[s:e].astype(LD) - ref)
        bad = np.flatnonzero(~(err <= bound))
        assert bad.size == 0, "%s: block %d [%d, %d): %d outputs beyond the bound, first t=%d: got %r ref %r bound %.3g" % (
            what, b, s, e, bad.size, s + bad[0], y[s + bad[0]], float(ref[bad[0]]), float(bound[bad[0]]))
        worst = max(worst, float(np.max(err / bound)))
    return worst


def check_fft(y, v, bands, lay, pair, what):
    L = bands.shape[1]
    NF, HD, S = fft_geometry(L, pair)
    logn = np.log2(NF // 2)
    worst = 0.0
    for b, (s, e) in enumerate(lay.bounds()):
        if e == s:
            continue
        n = e - s
        ref = band_apply(v[s:e], bands[b])
        err2 = np.asarray((y[s:e].astype(LD) - ref) ** 2, dtype=np.float64)
        nw = -(-n // S)
        err_w = np.sqrt(np.bincount(np.arange(n) // S, weights=err2, minlength=nw))
        cs = np.r_[0.0, np.cumsum(v[s:e] ** 2)]
        w0 = np.arange(nw) * S - HD                                  # first input sample of each window
        v_w = np.sqrt(np.maximum(cs[np.clip(w0 + NF, 0, n)] - cs[np.clip(w0, 0, n)], 0.0))
        hc = np.zeros(NF)
        hc[:L] = bands[b]
        if L > 1:
            hc[NF - L + 1:] = bands[b][1:][::-1]
        bound = 8 * logn * U * np.max(np.abs(np.fft.rfft(hc))) * v_w
        bad = np.flatnonzero(~(err_w <= bound))
        assert bad.size == 0, "%s: block %d [%d, %d): %d windows beyond the bound, first window %d: %.3g > %.3g" % (
            what, b, s, e, bad.size, bad[0], err_w[bad[0]], bound[bad[0]])
        worst = max(worst, float(np.max(err_w / bound)))
    return worst


def run_noise(kern, lay, v, alignments):
    """The multi-block call (aligned, and for each shift in `alignments` with d and out 8 bytes off 16-byte alignment)
    and one call per block; returns the aligned result after checking that all of them agree bit for bit."""
    import torch
    dv = _dv()
    nt = lay.nt
    d = torch.empty(nt + 1, dtype=torch.float64, device="cuda")
    d[:nt] = torch.from_numpy(v).cuda()
    d1 = torch.empty(nt + 1, dtype=torch.float64, device="cuda")
    d1[1:] = d[:nt]
    what = "%s L=%d %r" % (kern.name(), kern.L, lay)
    y = Guarded(nt)
    checked(kern(*lay.args(), dv.ptr(d), y.ptr(), nt), what)
    y = written(y.result(what), what)
    for dshift, oshift in alignments:
        ys = Guarded(nt, shift=oshift)
        checked(kern(*lay.args(), dv.ptr(d1[1:] if dshift else d), ys.ptr(), nt), what)
        ys = ys.result(what)
        assert np.array_equal(ys.view(np.int64), y.view(np.int64)), \
            "%s: d shifted by %d, out by %d words: not bit-identical to the aligned call" % (what, dshift, oshift)
    yb = Guarded(nt)
    for b, (s, e) in enumerate(lay.bounds()):
        if e > s:
            checked(kern(1, e - s, None, dv.ptr(d) + 8 * s, yb.ptr() + 8 * s, e - s, block=b), what + " block %d" % b)
    yb = yb.result(what + " per block")
    diff = np.flatnonzero(yb.view(np.int64) != y.view(np.int64))
    assert diff.size == 0, "%s: %d outputs differ from the per-block calls, first t=%d (%r vs %r)" % (
        what, diff.size, diff[0], y[diff[0]], yb[diff[0]])
    return y


def check_noise(L, pair, layout, seed):
    rng = np.random.default_rng(seed)
    sm = sm_count()
    if pair is None:
        S = TILE_DIRECT
        smem = 8 * (L + TILE_DIRECT + 2 * (L - 1))
        grid = sm * max(1, min(8, SMEM_PER_SM // (smem + 1024)))       # at most 8 CTAs of 256 threads per SM
    else:
        S = fft_geometry(L, pair)[2]
        grid = sm // 2 if pair else sm
    lay = noise_layout(layout, S, L, grid * S, rng)
    bands = make_bands(lay.nb, L, rng)
    v = make_tod(lay.nt, rng)
    kern = NoiseKernel(L, pair, bands)
    y = run_noise(kern, lay, v, [] if pair is None else [(1, 1), (1, 0), (0, 1)])
    nwin = sum(-(-(e - s) // S) for s, e in lay.bounds())
    assert nwin >= 3 * grid, "fewer than 3 trips"
    if pair is None:
        worst = check_direct(y, v, bands, lay, "direct L=%d %r" % (L, lay))
    else:
        worst = check_fft(y, v, bands, lay, pair, "FFT pair=%d L=%d %r" % (pair, L, lay))
    print("%s L=%d %r: %d windows / tiles on a grid of %d, largest error / bound %.3g" % (
        kern.name(), L, lay, nwin, grid, worst))


LAYOUTS = ["equal", "remainder", "ragged"]


@gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("L", [3000, 4096, 6000, 8192])
def test_fft_cluster_windows(cm, L, layout):
    """k_toeplitz_fft<512, true> at >= 3 windows per 2-CTA cluster: the split-phase join barrier between windows."""
    check_noise(L, 1, layout, seed=L)


@gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("L", [1, 2, 48, 200, 2047, 4096])
def test_fft_one_cta_windows(cm, L, layout):
    """k_toeplitz_fft<512> (or <1024> under CM2_FFT_THREADS=1024) at >= 3 windows per CTA."""
    check_noise(L, 0, layout, seed=L + 1)


@gpu
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("L", [1, 2, 16, 47, 4096, 8192, 9344])
def test_direct_tiles(cm, L, layout):
    """k_toeplitz at >= 3 trips of its persistent grid; bands up to the 227 kB shared-memory limit (9344)."""
    check_noise(L, None, layout, seed=L + 2)


@gpu
def test_fft_1024_threads(cm):
    """The one-CTA window cases with CM2_FFT_THREADS=1024 (read once per process: a fresh interpreter)."""
    env = dict(os.environ, CM2_FFT_THREADS="1024", PYTHONDONTWRITEBYTECODE="1")
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-s",
                        os.path.abspath(__file__), "-k", "test_fft_one_cta_windows or test_fft_threads_in_use"],
                       cwd=os.path.dirname(here), env=env, capture_output=True, text=True)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-3000:]
    assert " passed" in r.stdout and "skipped" not in r.stdout.splitlines()[-1]


@gpu
def test_fft_threads_in_use(cm):
    """The one-CTA FFT kernel that runs is the instantiation CM2_FFT_THREADS selects (512 unless it is 1024)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    threads = 1024 if os.environ.get("CM2_FFT_THREADS") == "1024" else 512
    rng = np.random.default_rng(5)
    lay = Layout("one", 40000, 1, 40000)
    kern = NoiseKernel(200, 0, make_bands(1, 200, rng))
    d = _dv().to_dev_f64(make_tod(lay.nt, rng))
    y = Guarded(lay.nt)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        checked(kern(*lay.args(), d.data_ptr(), y.ptr(), lay.nt), "FFT")
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "k_toeplitz_fft" in e.name}
    assert names and all("k_toeplitz_fft<%d, false>" % threads in n or "k_toeplitz_fftILi%dELb0E" % threads in n
                         for n in names), names


# ---- small cases and argument checks of the noise kernels ------------------------------------------------------------

@gpu
@pytest.mark.parametrize("kind", ["direct", "fft0", "fft1"])
def test_noise_small_blocks(cm, kind):
    """One trip or less: 1-sample equal blocks, blocksize 2..7 with remainders, one block shorter than the band."""
    pair = {"direct": None, "fft0": 0, "fft1": 1}[kind]
    rng = np.random.default_rng(len(kind))
    for L in (1, 2, 5, 48, 301) + ((3001,) if pair == 1 else ()):
        for nt, bs in ((1, 1), (2, 1), (13, 5), (100, 7), (299, 300), (1000, 2), (5003, 4999), (20001, 1700)):
            nb = max(nt // bs, 1)
            if pair is not None and nb > 64:
                continue                                 # 256 / 512 kB of transfer tables per block
            lay = Layout("bs%d" % bs, nt, nb, bs)
            bands = make_bands(nb, L, rng)
            v = make_tod(nt, rng)
            kern = NoiseKernel(L, pair, bands)
            y = run_noise(kern, lay, v, [] if pair is None else [(1, 1)])
            what = "%s L=%d %r" % (kern.name(), L, lay)
            check_direct(y, v, bands, lay, what) if pair is None else check_fft(y, v, bands, lay, pair, what)


def _status(kern, nb, bs, start, nt, n_alloc, same=False, writes=False):
    """Status of one call on 32-byte aligned inputs of n_alloc elements and a guarded output, which must stay untouched
    unless the call `writes`."""
    dv = _dv()
    d = dv.to_dev_f64(np.ones(max(n_alloc, 1)))
    y = Guarded(max(n_alloc, 1))
    rc = kern(nb, bs, start, dv.ptr(d), dv.ptr(d) if same else y.ptr(), nt)
    out = y.result("refused call")
    assert writes or np.all(out.view(np.int64) == SENTINEL), "a refused or empty call wrote its output"
    return rc


@gpu
def test_noise_argument_checks(cm):
    rng = np.random.default_rng(3)
    M = fft_points()
    # band widths: the FFT windows take 2 (L - 1) < M (one CTA) and < 2 M (clusters); the direct kernel 227 kB
    assert _status(NoiseKernel(M // 2 + 1, 0, make_bands(1, M // 2 + 1, rng)), 1, 100, None, 100, 100) == CM2_ERR_ARG
    assert _status(NoiseKernel(M + 1, 1, make_bands(1, M + 1, rng)), 1, 100, None, 100, 100) == CM2_ERR_ARG
    assert _status(NoiseKernel(9345, None, make_bands(1, 9345, rng)), 1, 100, None, 100, 100) == CM2_ERR_UNSUPPORTED
    for pair in (None, 0, 1):
        kern = NoiseKernel(5, pair, make_bands(3, 5, rng))
        assert _status(kern, 1, 100, None, 100, 100, same=True) == CM2_ERR_ARG           # in place
        assert _status(kern, 1, 7, None, 0, 0) == 0                                    # nt = 0: nothing written
        # equal blocks past nt: (nblocks - 1) blocksize > nt.  Without the check the call would read and write
        # d / out up to 2000, which still lies inside the 3000 elements here
        assert _status(kern, 3, 1000, None, 1500, 3000) == CM2_ERR_ARG, kern.name()
        assert _status(kern, 3, 750, None, 1500, 3000, writes=True) == 0               # (nblocks - 1) bs == nt


# ---- the fused P^T T P ---------------------------------------------------------------------------------------------

VAL = 240                         # k_amatvec_toeplitz outputs per warp tile (256 minus one 8-sample halo lane each side)


def fused_layout(name, nt, nband, rng):
    """Blocks for the fused kernel: equal (with or without a remainder), blocksize 1..7 (every lane straddles a
    boundary), and boundaries on lane, halo and tile edges with empty, 1-sample and shorter-than-band blocks."""
    if name == "one":
        return Layout(name, nt, 1, max(nt, 1))
    if name.startswith("bs"):
        bs = int(name[2:])
        return Layout(name, nt, max(nt // bs, 1), bs)
    if name == "equal":
        bs = next(b for b in (24003, 2403, 243, 81, 27, 9, 3, 1) if nt % b == 0)
        return Layout(name, nt, nt // bs, bs)
    if name == "remainder":
        bs = 24011 if nt > 50000 else max(nt // 3, 1) + 1 if nt > 3 else 1
        return Layout(name, nt, max(nt // bs, 1), bs)
    assert name == "ragged"
    tiles = rng.integers(0, nt // VAL + 1, 4 + nt // 4000)
    offs = np.array([0, 1, -1, 7, -7, 8, -8, 9, -9, 16, -16, 17, -17])
    e = [(VAL * tiles[:, None] + offs[None, :]).ravel(), 8 * rng.integers(0, nt // 8 + 1, 4 + nt // 4000),
         rng.integers(0, nt + 1, 8 + nt // 4000), [0, 1, 2, 2, 3, 8, 8, 9, 8 + nband // 2, nt // 2, nt // 2]]
    e = np.clip(np.concatenate(e), 0, nt)
    start = np.sort(np.r_[0, e, nt, nt])
    return Layout(name, nt, start.size - 1, start=start)


def fused_ref(tod, pol, x, bands, lay):
    """P^T T P x per touched pixel in long double, and its bound (n_i + 2 NLAG + 6) u S_i."""
    nlag = bands.shape[1] - 1
    good = tod.pix >= 0
    px = np.zeros(tod.nt, dtype=LD)
    apx = np.zeros(tod.nt, dtype=LD)
    px[good], apx[good] = projection(x.reshape(-1, pol)[tod.pix[good]], tod.c[good].astype(LD), tod.s[good].astype(LD),
                                     pol)
    bid = lay.block_id()
    a0 = bands[bid, 0].astype(LD)
    z, az = a0 * px, np.abs(a0) * apx
    for k in range(1, nlag + 1):
        if k >= tod.nt:
            break
        same = bid[k:] == bid[:-k]
        ak = bands[bid, k].astype(LD)
        for shift, src in ((slice(k, None), slice(None, -k)), (slice(None, -k), slice(k, None))):
            z[shift] += np.where(same, ak[shift] * px[src], 0)
            az[shift] += np.where(same, np.abs(ak[shift]) * apx[src], 0)
    zo, azo = z[tod.order], az[tod.order]
    ref, bound = scatter_ref(tod, [(zo * f, azo * np.abs(f)) for f in tod.factors(pol)])
    return ref, bound * ((tod.cnt + 2 * nlag + 6) / (tod.cnt + 4))[:, None]


def check_fused(tod, pol, nband, lay, seed, xkinds=("positive", "normal")):
    dv = _dv()
    rng = np.random.default_rng(seed)
    bands = make_bands(lay.nb, nband, rng)
    band_d = dv.to_dev_f64(bands.ravel())
    for xk in xkinds:
        x = make_map(xk, pol, tod.npix, rng)
        y = Guarded(pol * tod.npix)
        checked(_lib().cm2_amatvec_toeplitz(dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), tod.nt, pol,
                                            dv.ptr(band_d), nband, *lay.args(), dv.ptr(dv.to_dev_f64(x)), y.ptr(),
                                            tod.npix, dv.stream()), "cm2_amatvec_toeplitz")
        ref, bound = fused_ref(tod, pol, x, bands, lay)
        check_map(y.result("cm2_amatvec_toeplitz"), pol, 0, ref, bound, tod,
                  "P^T T P pol=%d nband=%d %r x=%s" % (pol, nband, lay, xk))


NBANDS = [1, 2, 3, 4, 5, 8, 9]    # every NLAG instantiation (2, 4, 8), and bands shorter than NLAG + 1
FUSED_LAYOUTS = ["one", "equal", "remainder", "ragged", "bs1", "bs2", "bs3", "bs5", "bs7"]


@gpu
@pytest.mark.parametrize("nt", [1, 7, 8, 9, 239, 240, 241, 255, 257, 481, 2049, 20011])
def test_fused_toeplitz_small(cm, nt):
    for i, pattern in enumerate(("seams", "flags", "random", "reappear")):
        tod = Tod.zoo(pattern, nt, seed=i)
        for pol in (1, 2, 3):
            rng = np.random.default_rng(100 * i + pol)
            for j, name in enumerate(FUSED_LAYOUTS):
                check_fused(tod, pol, NBANDS[(i + j + pol) % len(NBANDS)], fused_layout(name, nt, 9, rng), seed=j)
            lay = fused_layout("ragged", nt, 9, rng)
            for nband in NBANDS:
                check_fused(tod, pol, nband, lay, seed=nband)


def nt_fused_trips():
    """>= 3 trips of tod_blocks(nt, 240) for every instantiation: 73..128 registers per thread leave at most 3 CTAs
    of 8 warps per SM (4 assumed here); nt % 8 != 0.  3 410 437 samples on 148 SMs."""
    return 3 * sm_count() * 4 * 8 * VAL + 1237


TRIPS_FUSED = [("raster", 3, 9, "ragged"), ("raster", 1, 3, "remainder"), ("seams", 2, 5, "equal"),
               ("flags", 3, 2, "ragged"), ("tilted", 3, 8, "remainder"), ("random", 2, 4, "ragged"),
               ("single", 1, 1, "equal"), ("reappear", 3, 9, "bs7"), ("packed_edges", 1, 8, "bs3"),
               ("descending", 2, 9, "remainder"), ("raster", 2, 5, "bs1")]


@gpu
@pytest.mark.parametrize("pattern,pol,nband,layout", TRIPS_FUSED)
def test_fused_toeplitz_trips(cm, pattern, pol, nband, layout):
    """k_amatvec_toeplitz at >= 3 trips: the run scatter carried across trips, the halo lanes at every tile seam."""
    nt = nt_fused_trips()
    if layout == "equal":
        nt -= nt % 24003
    rng = np.random.default_rng(nband)
    check_fused(Tod.zoo(pattern, nt, seed=pol), pol, nband, fused_layout(layout, nt, nband, rng), seed=pol,
                xkinds=("positive", "normal") if pattern == "raster" else ("normal",))


@gpu
@pytest.mark.parametrize("nband", [2, 5, 9])
def test_fused_toeplitz_remainder_block(cm, nband):
    """Equal blocks whose last one takes nt - nblocks * blocksize extra samples: those samples couple to their right
    neighbours as well as their left ones (a symmetric T), as in the noise kernels."""
    nt = 8 * 1000 + 517
    lay = Layout("remainder", nt, 8, 1000)
    check_fused(Tod.zoo("random", nt, seed=nband), 3, nband, lay, seed=nband)


@gpu
def test_fused_toeplitz_blocks_past_nt_refused(cm):
    """(nblocks - 1) blocksize > nt is refused before anything is written (y is zero-filled only after the checks)."""
    dv = _dv()
    tod = Tod.zoo("random", 3000, seed=1)
    band = dv.to_dev_f64(np.ones(3 * 3))
    x = dv.to_dev_f64(np.ones(tod.npix))
    y = Guarded(tod.npix)
    rc = _lib().cm2_amatvec_toeplitz(dv.ptr(tod.d_pix), None, None, 1500, 1, dv.ptr(band), 3, 3, 1000, None,
                                     dv.ptr(x), y.ptr(), tod.npix, dv.stream())
    assert rc == CM2_ERR_ARG
    assert np.all(y.result("refused call").view(np.int64) == SENTINEL)
