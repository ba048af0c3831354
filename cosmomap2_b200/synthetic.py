"""
Seeded synthetic scans for the configurations of BASELINE.json (SURVEY.md section 8(d)).  NumPy
only: it produces INPUTS (pixel indices, polarisation angles, data, subscan tables, noise
weights) for both the CUDA path and the CPU oracle; nothing here is timed.

Geometry: a rectangular sky patch of ``nx x ny`` pixels inside the equatorial belt of a
RING-ordered HEALPix map of the given ``nside`` -- one patch row is a run of consecutive pixel
indices on one iso-latitude ring, rows are ``4*nside`` apart.  Every detector sweeps the patch
back and forth at constant speed (``samples_per_pixel`` samples per pixel crossing, as a
constant-elevation scan does) while the patch drifts in the cross-scan direction; detectors are
offset from each other on the focal plane.  The polarisation angle is the reference's HWP ramp
(utilities/utilities_functions.py:99-107) plus a per-detector offset.  The TOD is
detector-major, time-minor, like the reference's CES layout (linearoperators.py:134-140).
"""
import numpy as np


class Scan(object):
    """Container: pix (int32, HEALPix ids), phi, d, per-detector weights, subscan table."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def raster_scan(nt, nside=512, ndet=64, nx=1000, ny=500, samples_per_pixel=8.0, seed=0,
                flag_turnarounds=False, turnaround_frac=0.05, sigma=1.0, with_data=True,
                sky_seed=1234, hwp_jitter=1e-3):
    """Raster scan of ``ndet`` detectors x ``nt // ndet`` samples over an ``nx x ny`` patch."""
    rng = np.random.default_rng(seed)
    ns = nt // ndet
    nt = ns * ndet
    npix_full = 12 * nside * nside
    ring = 4 * nside
    iy0 = 2 * nside - ny // 2            # centred on the equator: rings of constant length 4*nside
    ix0 = ring // 2 - nx // 2
    sweep = int(round(nx * samples_per_pixel))            # samples per one-way sweep (incl. turnaround)
    t = np.arange(ns, dtype=np.int64)
    isw = t // sweep
    frac = (t - isw * sweep) / float(sweep)
    # scanning portion of a sweep; the rest is the turnaround
    ta = turnaround_frac if flag_turnarounds else 0.0
    u = np.clip((frac - ta / 2) / (1.0 - ta), 0.0, 1.0 - 1e-12)
    xpos = np.where(isw % 2 == 0, u, 1.0 - 1e-12 - u) * nx
    nsweeps = int(isw[-1]) + 1
    pix = np.empty(nt, dtype=np.int32)
    phi = np.empty(nt, dtype=np.float64)
    weights = rng.uniform(0.5, 1.5, size=ndet)
    det_dx = rng.uniform(-0.02, 0.02, size=ndet) * nx
    det_dy = rng.uniform(-0.05, 0.05, size=ndet) * ny
    theta0 = rng.uniform(0, np.pi, size=ndet)
    for b in range(ndet):
        # cross-scan drift: the whole patch height is crossed once per detector timeline
        ypos = (t / float(ns)) * ny + det_dy[b]
        ix = np.mod(np.floor(xpos + det_dx[b]).astype(np.int64), nx)
        iy = np.mod(np.floor(ypos).astype(np.int64), ny)
        p = (iy0 + iy) * ring + (ix0 + ix)
        if flag_turnarounds:
            p = np.where((frac < ta / 2) | (frac >= 1.0 - ta / 2), -1, p)
        pix[b * ns:(b + 1) * ns] = p
        # HWP ramp + encoder jitter.  Without jitter a pixel hit over whole HWP periods has an
        # exactly isotropic QU block and the reference's condition-number mask evaluates
        # sqrt(tr^2/4 - det) on +-1e-17: NaN or not depending on rounding (DESIGN.md section 7).
        phi[b * ns:(b + 1) * ns] = theta0[b] + 2 * np.pi * 2.5 / 200. * t + hwp_jitter * rng.standard_normal(ns)
    # subscan table shared by all detectors (reference: subscans[ces], tstart[ces])
    s0 = int(np.ceil(ta / 2 * sweep))
    s1 = int(np.ceil((1.0 - ta / 2) * sweep))             # offsets with ta/2 <= frac < 1 - ta/2
    sub_start = (np.arange(nsweeps, dtype=np.int64) * sweep + s0)
    sub_len = np.full(nsweeps, s1 - s0, dtype=np.int64)
    keep = sub_start < ns                                  # the last sweep may be cut by the timeline's end
    sub_start, sub_len = sub_start[keep], np.minimum(sub_len[keep], ns - sub_start[keep])
    scan = Scan(nt=nt, ndet=ndet, ns=ns, nside=nside, npix_full=npix_full, pix=pix, phi=phi,
                weights=weights, sub_len=sub_len, sub_start=sub_start, nx=nx, ny=ny,
                samples_per_pixel=samples_per_pixel, seed=seed)
    if with_data:
        scan.d = simulate_data(scan, sigma=sigma, rng=rng, sky_seed=sky_seed)
    return scan


def simulate_data(scan, sigma=1.0, rng=None, sky_seed=1234):
    """d = P sky + white noise of per-detector variance sigma^2 / w_det (flagged samples: noise only)."""
    rng = np.random.default_rng(7) if rng is None else rng
    sky = np.random.default_rng(sky_seed)
    # smooth-ish random IQU sky on the patch, indexed by the full-sky pixel id through a hash-free
    # table on the patch bounding box
    ring = 4 * scan.nside
    good = scan.pix >= 0
    p = scan.pix[good].astype(np.int64)
    iy = p // ring
    ix = p - iy * ring
    iy -= iy.min()
    ix -= ix.min()
    ny, nx = int(iy.max()) + 1, int(ix.max()) + 1
    I = 100.0 * sky.standard_normal((ny, nx))
    Q = 10.0 * sky.standard_normal((ny, nx))
    U = 10.0 * sky.standard_normal((ny, nx))
    d = np.zeros(scan.nt)
    ph = scan.phi[good]
    d[good] = I[iy, ix] + Q[iy, ix] * np.cos(2 * ph) + U[iy, ix] * np.sin(2 * ph)
    wsamp = np.repeat(scan.weights, scan.ns)
    d += sigma * rng.standard_normal(scan.nt) / np.sqrt(wsamp)
    return d


def config_c1(seed=0):
    """C1 stand-in for the absent real CES (data/20131011_092136.hdf5): 4 detector pairs,
    nt ~ 6.26e6 (data/profile_pol.dat:113), nside 128, turnarounds flagged."""
    return raster_scan(6258942 // 4 * 4, nside=128, ndet=4, nx=160, ny=120, samples_per_pixel=12.0,
                       seed=seed, flag_turnarounds=True)


def config_c2(nt=100000000, seed=0, with_data=True):
    """C2: raster scan, 1e8 samples, IQU nside 512, 64 white-noise blocks (one per detector)."""
    return raster_scan(nt, nside=512, ndet=64, nx=1000, ny=500, samples_per_pixel=8.0, seed=seed,
                       with_data=with_data)


def toeplitz_bands(ndet, nband, seed=0, eps=0.3, alpha=1.5):
    """Per-detector symmetric bands a_0 = 1, a_k = -eps k^-alpha / zeta-ish norm: SPD, diagonally
    dominant (SURVEY.md section 8(d), C3)."""
    rng = np.random.default_rng(seed)
    k = np.arange(1, nband, dtype=np.float64)
    base = k ** (-alpha)
    base /= 2.0 * base.sum() if nband > 1 else 1.0
    bands = []
    for _ in range(ndet):
        a = np.empty(nband)
        a[0] = 1.0 + 0.1 * rng.random()
        a[1:] = -eps * (1.0 + 0.1 * rng.random()) * base
        bands.append(a)
    return bands


def one_over_f_noise(ns, ndet, sigma, fknee, alpha, seed):
    """Seeded 1/f noise, detector-major (ndet timelines of ns samples): per detector, white noise shaped in
    Fourier space to the PSD P(f) = sigma^2 (1 + (fknee / |f|)^alpha), f in cycles per sample (periodic over the
    timeline; the mean mode keeps the white level sigma^2)."""
    rng = np.random.default_rng(seed)
    f = np.fft.rfftfreq(int(ns))
    gain = np.full(f.shape, float(sigma))
    gain[1:] *= np.sqrt(1.0 + (float(fknee) / f[1:]) ** float(alpha))
    out = np.empty(int(ns) * int(ndet))
    for b in range(int(ndet)):
        out[b * ns:(b + 1) * ns] = np.fft.irfft(np.fft.rfft(rng.standard_normal(int(ns))) * gain, int(ns))
    return out
