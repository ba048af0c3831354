"""The TOD-pass kernels of csrc/tod_pass.cu against an extended-precision reference, called through the C ABI so that
every kernel instantiation is chosen here and not by the planner in linearoperators.py.

The kernels are persistent: each warp walks tiles of 256 samples, one trip over the grid after the other, and carries
state from one trip to the next (the open runs of the register scatter, the prefetched packed word, the staged window,
the next tiles' subscan lookups).  So every kernel runs here at a size of several trips as well as at small sizes, on
a zoo of pointings aimed at the branches of the run compression, the warp merge and the packed stream.

Reference: every output is computed in ``np.longdouble`` (80-bit on x86-64, IEEE quad on aarch64) from the same fp64
inputs, with the kernels' association of the terms.  Scatters sort the samples by pixel (stable) and reduce with
``np.add.reduceat``.

Tolerance: a first-order bound per output element instead of a relative error scaled by the largest entry, so that an
error in a pixel with few hits or in a cancelling Q / U component cannot hide behind the largest I entry.  For a
scatter output i (pixel, component) with n_i contributing samples

    |y_i - ref_i| <= (n_i + 4) * 2^-53 * S_i,      S_i = sum_j |term_ij|   (in long double).

A term is a product of fp64 roundings (up to 4: the two FMAs of the projection, the weight, cos / sin), and n_i - 1
additions combine the n_i terms in whatever order the fp64 atomics, the shared-memory adds and the warp merge take.
|term_ij| counts the magnitudes of its parts, |w| (|x_0| + |x_1 c| + |x_2 s|) |f| for the A-matvec terms, because the
projection's rounding is relative to those and not to its (possibly cancelling) value.  Outputs without a contributing
sample must be exactly 0, and nothing may be written outside the output: y, d, mom and hits are views 32 bytes into
larger buffers filled with a sentinel bit pattern, which is checked after every call.
"""
import copy
import ctypes
import time
from types import SimpleNamespace

import numpy as np
import pytest

import golden_cases as gc

pytestmark = pytest.mark.gpu

LD = np.longdouble
U = 2.0 ** -53
SENTINEL = 0x7ff4deadbeefcafe     # a signalling-NaN bit pattern: no kernel writes it
GUARD_HI = 4096                   # int64 / fp64 sentinel words after an output (4 = 32 bytes before it)
SMALL_NT = [1, 7, 8, 9, 255, 256, 257, 2047, 2049]


@pytest.fixture(scope="module")
def cm():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    assert np.finfo(np.longdouble).eps <= 2.0 ** -63, "the reference needs an extended-precision long double"
    import cosmomap2_b200
    yield cosmomap2_b200
    # cm2_amatvec_white_set_stage is process-global: the tests below restore 0, and the packed stream is refused
    # by the staged scatter, so a call with it succeeds only when the stage is off
    from cosmomap2_b200 import _device as dv
    pix = torch.zeros(8, dtype=torch.int32, device="cuda")
    packed = torch.zeros(1, dtype=torch.int64, device="cuda")
    xy = torch.zeros(2, dtype=torch.float64, device="cuda")
    dv.call("cm2_amatvec_white", dv.ptr(pix), dv.ptr(packed), None, None, 8, 1, None, 0, 0, None, dv.ptr(xy[:1]),
            dv.ptr(xy[1:]), 1, 1, dv.stream())


def _dv():
    from cosmomap2_b200 import _device as dv
    return dv


def sm_count():
    sm, l2, cc = ctypes.c_int(), ctypes.c_int64(), ctypes.c_int()
    _dv().call("cm2_device_info", ctypes.byref(sm), ctypes.byref(l2), ctypes.byref(cc))
    return sm.value


def nt_trips():
    """At least 3 trips over the grid for every TOD kernel, whatever its occupancy (at most 8 CTAs of 8 warps per SM
    of 256-sample tiles), and nt % 8 != 0.  7 274 733 samples on 148 SMs."""
    return 3 * sm_count() * 8 * 8 * 256 + 1237


class Guarded:
    """An n-element output at 32 bytes (+ 8 * shift) into a buffer of sentinel words."""

    def __init__(self, n, dtype=None, shift=0):
        import torch
        self.n, self.lo = int(n), 4 + shift
        self.buf = torch.full((self.lo + self.n + GUARD_HI,), SENTINEL, dtype=torch.int64, device="cuda")
        self.view = self.buf[self.lo:self.lo + self.n]
        if dtype is not torch.int64:
            self.view = self.view.view(torch.float64)

    def ptr(self):
        return self.view.data_ptr()

    def result(self, what):
        b = self.buf
        ok = bool((b[:self.lo] == SENTINEL).all().item()) and bool((b[self.lo + self.n:] == SENTINEL).all().item())
        assert ok, "%s: wrote outside its output" % what
        return self.view.cpu().numpy()


# ---- the pointing zoo: generators of int32 pixel ids (-1 = flagged) and the number of pixels -------------------

SEAM_RUNS = np.array([8] * 32 + [16] * 16 + [256, 257, 256, 1, 8, 8, 7, 16, 256, 257, 1, 7, 7, 8, 16, 255, 257, 9, 8,
                                             256, 256])


def zoo_single(nt, rng, sm):
    """One pixel for the whole TOD: one run over every lane, tile and trip, every RED to one address."""
    return np.full(nt, 5, dtype=np.int32), 9


def zoo_seams(nt, rng, sm):
    """Runs of exactly 8, 16, 256 and 257 samples, aligned to lanes and tiles and shifted by 1 and 7 samples."""
    lens = np.tile(SEAM_RUNS, nt // int(SEAM_RUNS.sum()) + 1)
    ids = (np.arange(lens.size) * 37) % 4093                 # neighbouring runs always differ
    return np.repeat(ids, lens)[:nt].astype(np.int32), 4093


def zoo_reappear(nt, rng, sm):
    """Pixels that come back inside a lane (ABAB, AABBA), a pixel running through several single-run lanes, and the
    same pixel on both sides of an all-flagged lane and of an all-flagged tile.  Periods of 3 tiles."""
    A, B, C, F, R = 0, 1, 2, -1, -2
    t1 = [A, B] * 4 + [A, A, B, B, A, B, B, A] + [C] * 24 + [F] * 8 + [C] * 8 + [C, C, A, A, C, C, A, A]
    t1 += [R] * (256 - 8 - len(t1)) + [C] * 8
    t3 = [C] * 8 + [R] * 240 + [A, B, A, B, A, A, B, B]
    period = np.array(t1 + [F] * 256 + t3)
    reps = nt // period.size + 1
    pix = np.tile(period, reps).reshape(reps, -1)
    rnd = rng.integers(0, 3, pix.shape)
    pix = np.where(pix == R, rnd, pix)
    base = (3 * np.arange(reps) % 999)[:, None]
    return np.where(pix >= 0, pix + base, -1).ravel()[:nt].astype(np.int32), 1002


def zoo_flags(nt, rng, sm):
    """Runs of 5 samples with -1 at the first / last sample of lanes, of tiles and of the TOD; fully flagged lanes,
    tiles, and one fully flagged trip of the kernels that run 2 CTAs per SM."""
    t = np.arange(nt)
    pix = ((t // 5) % 3001).astype(np.int32)
    lane, tile, j, k = t // 8, t // 256, t % 8, t % 256
    m = ((j == 0) & (lane % 13 == 3)) | ((j == 7) & (lane % 13 == 7)) | (((k == 0) | (k == 255)) & (tile % 5 == 1))
    m |= (lane % 17 == 5) | (tile % 11 == 4)
    trip = sm * 2 * 8 * 256
    if nt > 2 * trip:
        m[trip:2 * trip] = True
    if nt:
        m[0] = m[-1] = True
    pix[m] = -1
    return pix, 3001


def zoo_all_flagged(nt, rng, sm):
    return np.full(nt, -1, dtype=np.int32), 4


def zoo_descending(nt, rng, sm):
    """Pixel ids that decrease along time (the packer's b0 is a later sample of the lane): runs of 3 samples down a
    row of 97 pixels, then a jump back by 204 ids to the next row."""
    r = np.arange(nt, dtype=np.int64) // 3
    row, col = r // 97, r % 97
    top = 300 * (int(row[-1]) + 2) if nt else 1
    return (top - (row * 300 + col)).astype(np.int32), top + 1


PACKED_LANES = np.array([
    [0, 0, 1, 1, 2, 2, 3, 3],                                # base delta 2, code 3 (b1 + 1)
    [0, 32766, 32767, 0, 1, 32767, 1, 0],                    # delta 32766 with code 3
    [32767, 32768, 0, 1, 0, 32768, 1, 32767],                # delta 32767 (the largest that fits) with code 3
    [0, 1, 32768, 32769, 0, 1, 32768, 32769],                # delta 32768: escape
    [-1] * 8,                                                # all flagged
    [0, -1, 0, 0, 1, -1, 1, 0],                              # mixed flags: escape
    [0, 5, 10, 0, 5, 10, 0, 0],                              # three clusters: escape
    [32767, 32767, 32766, 0, 0, 1, 32766, 1],                # descending inside the lane
    [5] * 8,                                                 # one run
])


def zoo_packed_edges(nt, rng, sm):
    """Lanes at the edges of the packed format, in random order, so that flagged lanes sit next to escape lanes."""
    nl = (nt + 7) // 8
    lanes = PACKED_LANES[rng.integers(0, len(PACKED_LANES), nl)]
    base = rng.integers(0, 5000, nl)[:, None]
    return np.where(lanes >= 0, lanes + base, -1).ravel()[:nt].astype(np.int32), 5000 + 32770


def zoo_random(nt, rng, sm):
    """Run-free pointing: every sample an independent pixel."""
    return rng.integers(0, 200000, nt).astype(np.int32), 200000


def _scan(nt, tilt):
    from cosmomap2_b200 import workloads
    ndet = 16
    _, _, pix, _, _, _, _ = workloads.make_scan(-(-max(nt, ndet) // ndet) * ndet, nside=512, nx=1000, ny=500,
                                                ndet=ndet, spp=8.0, seed=11, tilt_deg=tilt)
    pix = pix[:nt].cpu().numpy()
    return pix, int(pix.max()) + 3


def zoo_raster(nt, rng, sm):
    return _scan(nt, 0.0)


def zoo_tilted(nt, rng, sm):
    return _scan(nt, 30.0)


ZOO = {f.__name__[4:]: f for f in (zoo_single, zoo_seams, zoo_reappear, zoo_flags, zoo_all_flagged, zoo_descending,
                                   zoo_packed_edges, zoo_random, zoo_raster, zoo_tilted)}
ADVERSARIAL = ["single", "seams", "reappear", "flags", "all_flagged", "descending", "packed_edges", "random"]


class Tod:
    """A pointing with random angles, on the host and on the device, and its pixel-sorted unflagged samples."""

    def __init__(self, pix, npix, seed=0):
        dv = _dv()
        rng = np.random.default_rng(seed)
        self.pix = np.ascontiguousarray(pix, dtype=np.int32)
        self.nt, self.npix = self.pix.size, int(npix)
        phi = rng.uniform(0.0, 2 * np.pi, self.nt)
        self.c, self.s = np.cos(2 * phi), np.sin(2 * phi)
        order = np.argsort(self.pix, kind="stable")
        self._index(order[self.pix[order] >= 0])
        self.d_pix = dv.to_dev(self.pix if self.nt else np.full(8, -1, np.int32))
        self.d_c = dv.to_dev_f64(self.c if self.nt else np.zeros(8))
        self.d_s = dv.to_dev_f64(self.s if self.nt else np.zeros(8))
        self._packed = None

    def _index(self, order):
        """order: the contributing samples, sorted by pixel (stable)."""
        self.order = order
        self.ps = self.pix[order].astype(np.int64)
        self.starts = np.flatnonzero(np.r_[True, self.ps[1:] != self.ps[:-1]]) if self.ps.size else \
            np.zeros(0, dtype=np.int64)
        self.upix = self.ps[self.starts]
        self.cnt = np.diff(np.r_[self.starts, self.ps.size]).astype(np.int64)
        self.cs, self.ss = self.c[order].astype(LD), self.s[order].astype(LD)

    def restricted(self, keep):
        """The same pointing, with only the unflagged samples where keep[t] holds contributing."""
        sub = copy.copy(self)
        sub._index(self.order[keep[self.order]])
        return sub

    @classmethod
    def zoo(cls, name, nt, seed=0):
        pix, npix = ZOO[name](nt, np.random.default_rng(seed + 1), sm_count())
        return cls(pix, npix, seed)

    def packed(self):
        import torch
        dv = _dv()
        if self._packed is None:
            self._packed = torch.empty(max((self.nt + 7) // 8, 1), dtype=torch.int64, device="cuda")
            nesc = torch.empty(1, dtype=torch.int64, device="cuda")
            dv.call("cm2_pack_pointing", dv.ptr(self.d_pix), self.nt, dv.ptr(self._packed), dv.ptr(nesc), dv.stream())
        return self._packed

    def factors(self, pol):
        """cos / sin factors of the components a sample adds to (pixel-sorted order)."""
        one = np.ones(self.ps.size, dtype=LD)
        return [one] if pol == 1 else [self.cs, self.ss] if pol == 2 else [one, self.cs, self.ss]


def projection(rows, c, s, pol):
    """P x of samples with x rows `rows` and angles c, s, and the magnitude its rounding is relative to."""
    X = rows.astype(LD)
    if pol == 1:
        return X[:, 0], np.abs(X[:, 0])
    if pol == 2:
        a, b = X[:, 0] * c, X[:, 1] * s
        return a + b, np.abs(a) + np.abs(b)
    a, b, e = X[:, 0], X[:, 1] * c, X[:, 2] * s
    return a + b + e, np.abs(a) + np.abs(b) + np.abs(e)


def scatter_ref(tod, comps):
    """Per touched pixel (tod.upix) the sums of the terms in comps [(term, |term|), ...] over its samples, and the
    bound (n_i + 4) 2^-53 S_i of each."""
    ref = np.zeros((tod.upix.size, len(comps)), dtype=LD)
    bound = np.zeros_like(ref)
    if tod.upix.size:
        for k, (t, a) in enumerate(comps):
            ref[:, k] = np.add.reduceat(t, tod.starts)
            bound[:, k] = (tod.cnt + 4) * LD(U) * np.add.reduceat(a, tod.starts)
    return ref, bound


def check_map(y, width, offset, ref, bound, tod, what):
    """y[npix * width]: the components offset .. offset + ncomp of the touched pixels within the bound, every other
    entry exactly 0."""
    y = np.array(y).reshape(-1, width)
    assert y.shape[0] == tod.npix
    got = y[tod.upix, offset:offset + ref.shape[1]]
    err = np.abs(got.astype(LD) - ref)
    bad = np.argwhere(~(err <= bound))
    assert bad.size == 0, "%s: %d outputs beyond the bound; pixel %d comp %d: got %r ref %r bound %.3g" % (
        what, bad.shape[0], tod.upix[bad[0, 0]], offset + bad[0, 1], got[bad[0, 0], bad[0, 1]],
        float(ref[bad[0, 0], bad[0, 1]]), float(bound[bad[0, 0], bad[0, 1]]))
    rest = y.copy()
    rest[tod.upix, offset:offset + ref.shape[1]] = 0.0
    stray = np.argwhere(rest != 0)
    assert stray.size == 0, "%s: %d outputs without samples are nonzero, first at pixel %d comp %d" % (
        what, stray.shape[0], stray[0, 0], stray[0, 1])


def make_map(kind, pol, npix, rng):
    """'positive': I in [1, 2] and Q, U in [-0.5, 0.5], so that with weights in [0.5, 1.5] every I term is >= 0.14 and
    one lost, doubled or misrouted sample is far beyond the bound.  'normal': standard normal, for cancellation."""
    if kind == "normal":
        return rng.standard_normal(pol * npix)
    x = rng.uniform(-0.5, 0.5, (npix, pol))
    if pol != 2:
        x[:, 0] = rng.uniform(1.0, 2.0, npix)
    return x.ravel()


class Weighting:
    """Noise weights of cm2_amatvec_white / cm2_weights_moments: unit, equal blocks, ragged blocks (zero-length blocks,
    boundaries at lane and tile edges and inside lanes) and one weight per sample; w_t is the weight of each sample."""

    def __init__(self, kind, nt, rng):
        import torch
        dv = _dv()
        self.kind, self.nb, self.bs, start, wblk = kind, 0, 0, None, None
        t = np.arange(nt)
        if kind == "unit":
            self.w_t = np.ones(nt)
        elif kind in ("blk7", "blk1001"):
            self.bs = int(kind[3:])
            self.nb = max(-(-nt // self.bs), 1)
            wblk = rng.uniform(0.5, 1.5, self.nb)
            self.w_t = wblk[np.minimum(t // self.bs, self.nb - 1)]
        elif kind == "ragged":
            edges = [0, 0, 1, 7, 8, 8, 255, 256, 264, 512, 513, 2048, nt, nt]
            edges += list(rng.integers(0, nt + 1, 6 + nt // 3000)) + list(8 * rng.integers(0, nt // 8 + 1, 6 + nt // 3000))
            edges += list(256 * rng.integers(0, nt // 256 + 1, 6 + nt // 30000))
            start = np.sort(np.clip(np.array(edges, dtype=np.int64), 0, nt))
            self.nb = start.size - 1
            wblk = rng.uniform(0.5, 1.5, self.nb)
            self.w_t = wblk[np.searchsorted(start[:self.nb], t, side="right") - 1]
        elif kind == "sample":
            self.bs, self.nb = 1, max(nt, 1)
            wblk = rng.uniform(0.5, 1.5, self.nb)
            self.w_t = wblk[:nt]
        else:
            raise KeyError(kind)
        self.d_wblk = None if wblk is None else dv.to_dev_f64(wblk)
        self.d_start = None if start is None else dv.to_dev(start, torch.int64)

    def args(self):
        dv = _dv()
        return dv.ptr(self.d_wblk), self.nb, self.bs, dv.ptr(self.d_start)


# ---- cm2_amatvec_white ---------------------------------------------------------------------------------------------

def white_ref(tod, pol, x, w_t):
    proj, ap = projection(x.reshape(-1, pol)[tod.ps], tod.cs, tod.ss, pol)
    w = w_t[tod.order].astype(LD)
    v, av = w * proj, np.abs(w) * ap
    return scatter_ref(tod, [(v * f, av * np.abs(f)) for f in tod.factors(pol)])


def white_variants(tod, wt):
    """(name, nstreams, packed, stage wpix) of every kernel path of cm2_amatvec_white for this input."""
    if wt.kind == "sample":
        return [("per-sample weights", 1, False, 0)]
    ntiles = -(-tod.nt // 256)
    S = next((S for S in (7, 5, 3, 6, 9, 11, 13, 2) if ntiles >= 4 * S and ntiles % S), None)
    vs = [("time order", 1, False, 0), ("packed", 1, True, 0)]
    if S:
        vs += [("interleaved S=%d (short last stream)" % S, S, False, 0), ("packed interleaved S=%d" % S, S, True, 0),
               ("staged 32 interleaved S=%d" % S, S, False, 32)]
    if ntiles // 4 + 1 >= 2:
        vs.append(("S=%d > ntiles/4 (time order)" % (ntiles // 4 + 1), ntiles // 4 + 1, False, 0))
    vs += [("staged %d" % wp, 1, False, wp) for wp in (1, 32, 288, 1024)]
    return vs


def run_white(tod, pol, wt, x_d, nstreams, packed, stage):
    dv = _dv()
    y = Guarded(pol * tod.npix)
    if stage:
        dv.call("cm2_amatvec_white_set_stage", stage)
    try:
        dv.call("cm2_amatvec_white", dv.ptr(tod.d_pix), dv.ptr(tod.packed()) if packed else None, dv.ptr(tod.d_c),
                dv.ptr(tod.d_s), tod.nt, pol, *wt.args(), dv.ptr(x_d), y.ptr(), tod.npix, nstreams, dv.stream())
    finally:
        if stage:
            dv.call("cm2_amatvec_white_set_stage", 0)
    return y.result("cm2_amatvec_white")


def check_white(tod, pol, wkind, xkinds, seed):
    dv = _dv()
    rng = np.random.default_rng(seed)
    wt = Weighting(wkind, tod.nt, rng)
    for xk in xkinds:
        x = make_map(xk, pol, tod.npix, rng)
        x_d = dv.to_dev_f64(x)
        ref, bound = white_ref(tod, pol, x, wt.w_t)
        for name, S, packed, stage in white_variants(tod, wt):
            y = run_white(tod, pol, wt, x_d, S, packed, stage)
            check_map(y, pol, 0, ref, bound, tod, "nt=%d pol=%d weights=%s x=%s %s" % (tod.nt, pol, wkind, xk, name))


@pytest.mark.parametrize("nt", SMALL_NT)
def test_white_amatvec_small(cm, nt):
    """Every path of cm2_amatvec_white on every adversarial pointing at sizes around a lane and a tile."""
    for i, name in enumerate(ADVERSARIAL):
        tod = Tod.zoo(name, nt, seed=i)
        for pol in (1, 2, 3):
            for wkind in ("unit", "blk7", "blk1001", "ragged", "sample"):
                xk = ("positive", "normal") if wkind in ("unit", "ragged") else ("positive",)
                check_white(tod, pol, wkind, xk, seed=100 * i + 10 * pol + len(wkind))


TRIPS_WHITE = [("raster", 3, "unit"), ("raster", 1, "blk1001"), ("raster", 2, "ragged"), ("raster", 3, "sample"),
               ("seams", 3, "blk7"), ("reappear", 2, "ragged"), ("flags", 3, "blk1001"), ("single", 3, "unit"),
               ("descending", 1, "blk7"), ("packed_edges", 3, "ragged"), ("tilted", 3, "blk1001"),
               ("random", 2, "sample"), ("flags", 1, "sample")]


@pytest.mark.parametrize("pattern,pol,wkind", TRIPS_WHITE)
def test_white_amatvec_trips(cm, pattern, pol, wkind):
    """Every path of cm2_amatvec_white at >= 3 trips over the grid: the prefetched packed word, the in-loop flush of
    the staged window, the run state carried from trip to trip and the short last stream of the interleaved order."""
    tod = Tod.zoo(pattern, nt_trips(), seed=7)
    check_white(tod, pol, wkind, ("positive", "normal") if pattern in ("raster", "seams") else ("positive",), seed=pol)


# ---- P x, P^T d (atomic and pixel-sorted), the moments, the hit counts ---------------------------------------------

def check_tod_kernels(tod, pol, seed):
    import torch
    dv = _dv()
    rng = np.random.default_rng(seed)
    st = dv.stream()
    good = tod.pix >= 0
    for xk in ("positive", "normal"):
        x = make_map(xk, pol, tod.npix, rng)
        x_d = dv.to_dev_f64(x)
        d = Guarded(tod.nt)
        dv.call("cm2_pointing_apply", dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), tod.nt, pol, dv.ptr(x_d),
                d.ptr(), st)
        d = d.result("cm2_pointing_apply")
        proj, ap = projection(x.reshape(-1, pol)[tod.pix[good]], tod.c[good].astype(LD), tod.s[good].astype(LD), pol)
        err = np.abs(d[good].astype(LD) - proj)
        assert np.all(err <= 3 * LD(U) * ap), "P x pol=%d x=%s: max excess %r" % (pol, xk, float(np.max(err - 3 * LD(U) * ap)))
        assert np.all(d[~good] == 0.0), "P x: flagged samples not 0"

    dvec = rng.standard_normal(max(tod.nt, 1))
    dd = dv.to_dev_f64(dvec)
    dl = dvec[tod.order].astype(LD)
    ref, bound = scatter_ref(tod, [(dl * f, np.abs(dl * f)) for f in tod.factors(pol)])
    y = Guarded(pol * tod.npix)
    dv.call("cm2_pointing_apply_t", dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), tod.nt, pol, dv.ptr(dd),
            y.ptr(), tod.npix, st)
    check_map(y.result("cm2_pointing_apply_t"), pol, 0, ref, bound, tod, "P^T d pol=%d" % pol)

    rowptr = np.zeros(tod.npix + 1, dtype=np.int64)
    rowptr[1:] = np.cumsum(np.bincount(tod.ps, minlength=tod.npix))
    perm = dv.to_dev(np.r_[tod.order, 0].astype(np.int32))
    rp = dv.to_dev(rowptr)
    ys = []
    for _ in range(2):
        y = Guarded(pol * tod.npix)
        dv.call("cm2_pointing_apply_t_sorted", dv.ptr(rp), dv.ptr(perm), dv.ptr(tod.d_c), dv.ptr(tod.d_s), pol,
                dv.ptr(dd), y.ptr(), tod.npix, st)
        ys.append(y.result("cm2_pointing_apply_t_sorted"))
    check_map(ys[0], pol, 0, ref, bound, tod, "sorted P^T d pol=%d" % pol)
    assert np.array_equal(ys[0].view(np.int64), ys[1].view(np.int64)), "sorted P^T d is not deterministic"

    hits = Guarded(tod.npix, torch.int64)
    dv.call("cm2_hits_i64", dv.ptr(tod.d_pix), tod.nt, tod.npix, hits.ptr(), st)
    gc.exact(hits.result("cm2_hits_i64"), np.bincount(tod.ps, minlength=tod.npix), what="hits")

    for mode in ("w", "wblk", "ragged", "none"):
        wt = Weighting({"w": "sample", "wblk": "blk1001" if tod.nt > 100000 else "blk7", "ragged": "ragged",
                        "none": "unit"}[mode], tod.nt, rng)
        w_dev = wt.d_wblk if mode == "w" else None
        args = (None, 0, 0, None) if mode in ("w", "none") else wt.args()
        mom = Guarded(6 * tod.npix)
        dv.call("cm2_weights_moments", dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), dv.ptr(w_dev), *args,
                tod.nt, pol, mom.ptr(), tod.npix, st)
        w = wt.w_t[tod.order].astype(LD)
        c, s = tod.cs, tod.ss
        terms = {1: [w], 2: [(w * c) * c, (w * s) * c, (w * s) * s],
                 3: [w, w * c, w * s, (w * c) * c, (w * s) * c, (w * s) * s]}[pol]
        ref, bound = scatter_ref(tod, [(t, np.abs(t)) for t in terms])
        check_map(mom.result("cm2_weights_moments"), 6, 3 if pol == 2 else 0, ref, bound, tod,
                  "moments pol=%d weights=%s" % (pol, mode))


@pytest.mark.parametrize("nt", SMALL_NT)
def test_tod_kernels_small(cm, nt):
    for i, name in enumerate(ADVERSARIAL):
        tod = Tod.zoo(name, nt, seed=i)
        for pol in (1, 2, 3):
            check_tod_kernels(tod, pol, seed=10 * i + pol)


@pytest.mark.parametrize("pattern,pol", [("raster", 3), ("tilted", 2), ("flags", 3), ("single", 1), ("reappear", 2),
                                         ("packed_edges", 3), ("random", 3)])
def test_tod_kernels_trips(cm, pattern, pol):
    check_tod_kernels(Tod.zoo(pattern, nt_trips(), seed=3), pol, seed=pol)


# ---- subscan filters: the offset filter through the run table, the Legendre run-table kernel ------------------------

def subscan_layout(nt, rng):
    """Sorted, non-overlapping subscans [start, end): boundaries at tile and lane edges and inside lanes, two subscans
    inside one lane, subscans shorter than a lane, gaps of exactly one tile and of several tiles, the first subscan
    at 0 and the last one ending at nt."""
    segs = [(0, 768), (768, 776), (1001, 1003), (1004, 1007), (1010, 1015), (1016, 2048), (2051, 2056), (2056, 2403),
            (2403, 5120), (5376, 6000), (6000 + 256 * 9, 9000)]
    t = 9000
    while True:
        gap = int(rng.choice([0, 0, 1, 5, 256, 3 * 256, 1000]))
        a = t + gap
        if rng.random() < 0.3:
            a = -(-a // 256) * 256
        elif rng.random() < 0.3:
            a = -(-a // 8) * 8
        n = int(rng.choice([1, 3, 8, 256, 257, 999])) if rng.random() < 0.3 else int(rng.integers(1000, 30000))
        if a + n >= nt - 100:
            break
        segs.append((a, a + n))
        t = a + n
    segs.append((t + 7, nt))
    ss, se = np.array(segs, dtype=np.int64).T
    return ss, se


def filter_tables(tod, pol, ss, se):
    import torch
    from cosmomap2_b200 import linearoperators as lo
    dv = _dv()
    P = SimpleNamespace(_pix_dev=tod.d_pix, _cos_dev=tod.d_c, _sin_dev=tod.d_s, nrows=tod.nt, pol=pol)
    F = SimpleNamespace(_seg_start_host=ss, _seg_end_host=se, nseg=ss.size, _seg_start=dv.to_dev(ss, torch.int64),
                        _seg_end=dv.to_dev(se, torch.int64))
    rt = lo._filter_runs(P, F)
    assert rt, "the run table was not built"
    return F, rt


def run_table_ref(pix, c, s, ss, se, pol):
    """The offset run table as the header defines it: a run starts at an unflagged sample of a segment that is the
    segment's first sample or follows a different pixel, and lasts while the pixel repeats inside the segment; runs
    are numbered in sample order.  The cos / sin sums add the run's samples one by one from 0.0 in sample order."""
    nt = pix.size
    seg = np.full(nt, -1)
    for k, (a, b) in enumerate(zip(ss, se)):
        seg[a:b] = k
    t = np.arange(nt)
    first = np.where(seg >= 0, ss[np.maximum(seg, 0)], -1)
    starts = np.flatnonzero((seg >= 0) & (pix >= 0) & ((t == first) | (np.r_[-1, pix[:-1]] != pix)))
    change = np.r_[np.flatnonzero(pix[1:] != pix[:-1]) + 1, nt]
    ends = np.minimum(change[np.searchsorted(change, starts, side="right")], se[seg[starts]])
    lens = ends - starts
    csum, ssum = np.zeros(starts.size), np.zeros(starts.size)
    if pol > 1:
        for i in range(int(lens.max(initial=0))):
            m = lens > i
            csum[m] += c[starts[m] + i]
            ssum[m] += s[starts[m] + i]
    mom = np.stack([lens.astype(np.float64), csum, ssum], axis=1).ravel()
    nruns = np.bincount(seg[starts], minlength=ss.size).astype(np.int32)
    seg_first = np.where(nruns > 0, np.searchsorted(seg[starts], np.arange(ss.size)), 0)
    return pix[starts], mom, seg_first, nruns


@pytest.mark.parametrize("pol", [1, 2, 3])
def test_filter_run_table_bits(cm, pol):
    """The offset run table of _build_run_table (cm2_filter_runs_mark, the scan, cm2_filter_runs_fill) equals its
    host reference bit for bit, on flagged raster pointing with a fully flagged subscan, adjacent subscans and
    subscans that cut runs."""
    import torch
    from cosmomap2_b200 import linearoperators as lo
    dv = _dv()
    nt = (1 << 20) + 1237
    rng = np.random.default_rng(10 + pol)
    pix, npix = ZOO["raster"](nt, rng, sm_count())
    pix = pix.copy()
    pix[rng.random(nt) < 0.01] = -1
    ss, se = subscan_layout(nt, rng)
    pix[ss[ss.size // 2]:se[ss.size // 2]] = -1
    tod = Tod(pix, npix, seed=pol)
    P = SimpleNamespace(_pix_dev=tod.d_pix, _cos_dev=tod.d_c, _sin_dev=tod.d_s, nrows=nt, pol=pol)
    rt = lo._build_run_table(P, dv.to_dev(ss, torch.int64), dv.to_dev(se, torch.int64), ss.size, need_runs=True)
    assert rt, "the run table was not built"
    run_pix, mom, seg_first, seg_nruns = run_table_ref(pix, tod.c, tod.s, ss, se, pol)
    assert rt["nruns"] == run_pix.size
    assert np.array_equal(rt["run_pix"].cpu().numpy(), run_pix)
    assert np.array_equal(rt["run_mom"].cpu().numpy().view(np.int64), mom.view(np.int64)), "run moments"
    assert np.array_equal(rt["seg_first"].cpu().numpy()[:ss.size], seg_first)
    assert np.array_equal(rt["seg_nruns"].cpu().numpy()[:ss.size], seg_nruns)


@pytest.mark.parametrize("pol", [1, 2, 3])
def test_filter_mu_trips(cm, pol):
    """cm2_filter_seg_mean + cm2_amatvec_filter_mu (time order and interleaved) and cm2_pointing_filter_mu at >= 3
    trips, against the filter built from its definition in long double:
      mu_k = mean of (P x)_t over the unflagged samples of subscan k (0 without any);
      y = sum over the unflagged samples inside subscans of ((P x)_t - mu_k) (1, c, s);
      d_t = (P x)_t - mu_k inside subscans (flagged samples included, with (P x)_t = 0), exactly 0 in the gaps.
    Bounds: the mean is a sum over the subscan's n_k samples (run sums, then the runs), so
    |dmu_k| <= (n_k + 8) 2^-53 A_k / n_k + 2^-53 |mu_k| with A_k = sum |x_0| + |x_1 c| + |x_2 s|.  A sample term has
    the projection's magnitude plus |mu_k| and carries dmu_k:  |y_i - ref_i| <= (n_i + 4) 2^-53 S_i + sum_j |f_ij|
    dmu_k(j), and |d_t - ref_t| <= 3 2^-53 (|P x|_t + |mu_k|) + dmu_k."""
    import torch
    dv = _dv()
    nt = nt_trips()
    rng = np.random.default_rng(pol)
    pix, npix = ZOO["raster"](nt, rng, sm_count())
    pix = pix.copy()
    pix[rng.random(nt) < 0.01] = -1
    ss, se = subscan_layout(nt, rng)
    full = ss.size // 2                                          # one fully flagged subscan
    pix[ss[full]:se[full]] = -1
    pix[ss[3]:se[3]] = -1
    tod = Tod(pix, npix, seed=pol)
    F, rt = filter_tables(tod, pol, ss, se)
    assert int(rt["tile_flag"].eq(0).sum()) > 0 and int(rt["tile_flag"].eq(2).sum()) > 0
    t = np.arange(nt)
    k = np.searchsorted(se, t, side="right")
    inside = (k < ss.size) & (t >= ss[np.minimum(k, ss.size - 1)])
    good = pix >= 0
    st = dv.stream()
    for xk in ("positive", "normal"):
        x = make_map(xk, pol, npix, rng)
        x_d = dv.to_dev_f64(x)
        proj = np.zeros(nt, dtype=LD)
        ap = np.zeros(nt, dtype=LD)
        proj[good], ap[good] = projection(x.reshape(-1, pol)[pix[good]], tod.c[good].astype(LD),
                                          tod.s[good].astype(LD), pol)
        use = inside & good
        n_k = np.bincount(k[use], minlength=ss.size)
        sum_k = np.zeros(ss.size, dtype=LD)
        abs_k = np.zeros(ss.size, dtype=LD)
        np.add.at(sum_k, k[use], proj[use])
        np.add.at(abs_k, k[use], ap[use])
        nz = np.maximum(n_k, 1)
        mu = np.where(n_k > 0, sum_k / nz, 0)
        dmu = np.where(n_k > 0, (n_k + 8) * LD(U) * abs_k / nz + LD(U) * np.abs(mu), 0)
        mu_d = torch.empty(ss.size, dtype=torch.float64, device="cuda")
        dv.call("cm2_filter_seg_mean", dv.ptr(rt["run_pix"]), dv.ptr(rt["run_mom"]), dv.ptr(rt["seg_first"]),
                dv.ptr(rt["seg_nruns"]), F.nseg, pol, dv.ptr(x_d), dv.ptr(mu_d), st)
        mu_h = mu_d.cpu().numpy()
        assert np.all(np.abs(mu_h.astype(LD) - mu) <= dmu), "subscan means"
        assert np.all(mu_h[n_k == 0] == 0.0)

        # y: the scatter of ((P x)_t - mu_k) (1, c, s) over the unflagged samples inside subscans
        sub = tod.restricted(inside)
        ks = k[sub.order]
        v = proj[sub.order] - mu[ks]
        av = ap[sub.order] + np.abs(mu[ks])
        ref, bound = scatter_ref(sub, [(v * f, av * np.abs(f)) for f in sub.factors(pol)])
        if sub.upix.size:
            bound += np.stack([np.add.reduceat(np.abs(f) * dmu[ks], sub.starts) for f in sub.factors(pol)], axis=1)
        ntiles = -(-nt // 256)
        S = next(S for S in (7, 5, 3, 6, 9) if ntiles % S)
        for nstreams in (1, S):
            y = Guarded(pol * npix)
            dv.call("cm2_amatvec_filter_mu", dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), nt, pol,
                    dv.ptr(F._seg_start), dv.ptr(F._seg_end), dv.ptr(mu_d), dv.ptr(rt["tile_seg"]),
                    dv.ptr(rt["tile_flag"]), F.nseg, dv.ptr(x_d), y.ptr(), npix, nstreams, st)
            check_map(y.result("cm2_amatvec_filter_mu"), pol, 0, ref, bound, sub,
                      "P^T F P pol=%d x=%s nstreams=%d" % (pol, xk, nstreams))

        d = Guarded(nt)
        dv.call("cm2_pointing_filter_mu", dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), nt, pol,
                dv.ptr(F._seg_start), dv.ptr(F._seg_end), dv.ptr(mu_d), dv.ptr(rt["tile_seg"]), dv.ptr(rt["tile_flag"]),
                F.nseg, dv.ptr(x_d), d.ptr(), st)
        d = d.result("cm2_pointing_filter_mu")
        kk = np.minimum(k, ss.size - 1)
        dref = proj - mu[kk]
        dbound = 3 * LD(U) * (ap + np.abs(mu[kk])) + dmu[kk]
        err = np.abs(d.astype(LD) - dref)
        bad = np.flatnonzero(inside & ~(err <= dbound))
        assert bad.size == 0, "F P x pol=%d x=%s: %d samples beyond the bound, first t=%d" % (pol, xk, bad.size, bad[0])
        assert np.all(d[~inside] == 0.0), "F P x: gap samples not 0"


@pytest.mark.parametrize("order", [1, 2])
def test_filter_poly_mu_trips(cm, order):
    """cm2_amatvec_filter_poly_mu (the Legendre run-table kernel) in time order and detector-interleaved at >= 3 trips,
    both against the oracle's chain P^T (F (P x)).  The oracle takes about 1.5 s at this size on a CPU."""
    import oracle
    from cosmomap2_b200 import linearoperators as lo, synthetic
    dv = _dv()
    ndet = 16
    sc = synthetic.raster_scan(-(-nt_trips() // ndet) * ndet, nside=512, ndet=ndet, nx=1000, ny=500,
                               samples_per_pixel=8.0, seed=order, flag_turnarounds=True, with_data=False)
    sc.pix[np.random.default_rng(order).random(sc.nt) < 0.003] = -1          # flags inside subscans too
    res = {}
    t0 = time.perf_counter()
    for name, impl in (("oracle", oracle), ("gpu", cm)):
        pix = sc.pix.astype(np.int64)
        pts = impl.ProcessTimeSamples(pix, sc.npix_full, pol=3, phi=sc.phi)
        npix = pts.get_new_pixel[0]
        P = impl.SparseLO(npix, sc.nt, pix, pol=3, angle_processed=pts)
        F = impl.FilterLO(sc.nt, [sc.sub_len, sc.sub_start], sc.ns, sc.ndet, pix, poly_order=order)
        x = np.random.default_rng(4).standard_normal(3 * npix)
        if name == "oracle":
            res[name] = P.T * (F * (P * x))
            print("oracle P^T F P x, poly_order %d, %d samples: %.2f s" % (order, sc.nt, time.perf_counter() - t0))
            continue
        rt = lo._build_poly_runs(P, F)
        assert rt and rt["nhard"] == 0
        x_d = dv.to_dev_f64(x)
        dv.call("cm2_filter_poly_seg_coef", dv.ptr(rt["run_pix"]), dv.ptr(rt["run_mom"]), dv.ptr(rt["seg_first"]),
                dv.ptr(rt["seg_nruns"]), rt["nseg"], 3, order, dv.ptr(rt["W"]), dv.ptr(x_d), dv.ptr(rt["coef"]),
                dv.stream())
        for nstreams in (1, ndet):
            y = Guarded(3 * npix)
            dv.call("cm2_amatvec_filter_poly_mu", dv.ptr(P._pix_dev), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), sc.nt, 3,
                    dv.ptr(rt["seg_start"]), dv.ptr(rt["seg_end"]), dv.ptr(rt["coef"]), dv.ptr(rt["tile_seg"]),
                    dv.ptr(rt["tile_flag"]), rt["nseg"], order, dv.ptr(x_d), y.ptr(), npix, 0, nstreams, dv.stream())
            res[nstreams] = y.result("cm2_amatvec_filter_poly_mu")
    gc.close(res[1], res["oracle"], what="time order vs oracle")
    gc.close(res[ndet], res["oracle"], what="interleaved vs oracle")
    gc.close(res[ndet], res[1], what="interleaved vs time order")


# ---- pixel ids whose pol * p and 6 * p offsets do not fit int32 -----------------------------------------------------

def test_pixel_ids_past_int32_offsets(cm):
    """POL = 3 and npix = 7.2e8 + 5: pixel ids above 2^31 / 3 (the map offsets 3 p) and 2^31 / 6 (the moment offsets
    6 p), next to ids near 0.  The white A-matvec (int32 ids and packed), P, P^T, the hits and the moments against
    the reference on the touched outputs; every other output must stay exactly 0 (checked on the device)."""
    import torch
    dv = _dv()
    if torch.cuda.mem_get_info()[0] < 90e9:
        pytest.skip("needs 90 GB of free device memory (x, y, mom and the hit counts take about 75 GB)")
    npix, pol, nt = 720_000_005, 3, (1 << 20) + 3
    rng = np.random.default_rng(9)
    # raster-like runs of 1..9 samples, half of them near the top of the range, half near 0; flags between
    runs = rng.integers(1, 10, nt)
    rid = np.repeat(np.arange(nt), runs)[:nt]
    hi = (rid // 64) % 2 == 1
    pix = np.where(hi, npix - 1 - rid % 5000, rid % 5000).astype(np.int32)
    pix[rng.random(nt) < 0.01] = -1
    assert 3 * int(pix.max()) >= 2 ** 31 and 6 * int(pix.max()) >= 2 ** 31
    tod = Tod(pix, npix, seed=9)
    st = dv.stream()

    def dev_rows(t, width, comps, offset=0):
        idx = torch.from_numpy(tod.upix).cuda()
        rows = t.view(-1, width)[idx][:, offset:offset + comps].cpu().numpy()
        t.view(-1, width)[idx] = 0
        nz = int(torch.count_nonzero(t).item())
        assert nz == 0, "%d outputs without samples are nonzero" % nz
        return rows

    def check_rows(rows, ref, bound, what):
        assert np.all(np.abs(rows.astype(LD) - ref) <= bound), what

    x_d = torch.rand(pol * npix, dtype=torch.float64, device="cuda") - 0.5
    xr = x_d.view(-1, pol)[torch.from_numpy(tod.ps).cuda()].cpu().numpy()
    proj, ap = projection(xr, tod.cs, tod.ss, pol)
    wt = Weighting("blk1001", nt, rng)
    w = wt.w_t[tod.order].astype(LD)
    ref, bound = scatter_ref(tod, [(w * proj * f, w * ap * np.abs(f)) for f in tod.factors(pol)])
    y = torch.empty(pol * npix, dtype=torch.float64, device="cuda")
    for packed in (False, True):
        dv.call("cm2_amatvec_white", dv.ptr(tod.d_pix), dv.ptr(tod.packed()) if packed else None, dv.ptr(tod.d_c),
                dv.ptr(tod.d_s), nt, pol, *wt.args(), dv.ptr(x_d), dv.ptr(y), npix, 1, st)
        check_rows(dev_rows(y, pol, pol), ref, bound, "A x, packed=%s" % packed)

    d = Guarded(nt)
    dv.call("cm2_pointing_apply", dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), nt, pol, dv.ptr(x_d), d.ptr(),
            st)
    d = d.result("cm2_pointing_apply")
    dref = np.zeros(nt, dtype=LD)
    dabs = np.zeros(nt, dtype=LD)
    dref[tod.order], dabs[tod.order] = proj, ap
    assert np.all(np.abs(d.astype(LD) - dref) <= 3 * LD(U) * dabs), "P x"

    dl = d[tod.order].astype(LD)
    dv.call("cm2_pointing_apply_t", dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), nt, pol,
            dv.ptr(dv.to_dev_f64(d)), dv.ptr(y), npix, st)
    ref, bound = scatter_ref(tod, [(dl * f, np.abs(dl * f)) for f in tod.factors(pol)])
    check_rows(dev_rows(y, pol, pol), ref, bound, "P^T d")
    del y, x_d

    hits = torch.empty(npix, dtype=torch.int64, device="cuda")
    dv.call("cm2_hits_i64", dv.ptr(tod.d_pix), nt, npix, dv.ptr(hits), st)
    gc.exact(dev_rows(hits, 1, 1)[:, 0], tod.cnt, what="hits")
    del hits

    mom = torch.empty(6 * npix, dtype=torch.float64, device="cuda")
    dv.call("cm2_weights_moments", dv.ptr(tod.d_pix), dv.ptr(tod.d_c), dv.ptr(tod.d_s), None, *wt.args(), nt, pol,
            dv.ptr(mom), npix, st)
    c, s = tod.cs, tod.ss
    terms = [w, w * c, w * s, (w * c) * c, (w * s) * c, (w * s) * s]
    ref, bound = scatter_ref(tod, [(t, np.abs(t)) for t in terms])
    check_rows(dev_rows(mom, 6, 6), ref, bound, "moments")
