#!/usr/bin/env python
"""
Map-making with a noise model estimated twice: first from the data, then from the residual of the first map.

    pass 0:  psd = noise_psd(d, ns, pix=pix)              -> bands -> x0 = solve(P^T N0^-1 P, P^T N0^-1 d)
    pass 1:  psd = noise_psd(d, ns, P=P0, x=x0)           -> bands -> x1 = solve(P^T N1^-1 P, P^T N1^-1 d)

The PSD of d holds the sky as well as the noise, and a scanning experiment puts the sky at the scan frequencies,
where the 1/f model matters; the residual d - P x0 leaves the noise.  Pass 1 forms the residual inside the PSD pass
(cm2_noise_psd_residual), with no TOD-sized temporary.  The data: a raster scan with flagged turnarounds, an IQU sky
well above the noise, and 1/f noise P(f) = sigma^2 (1 + (fknee/|f|)^alpha) from synthetic.one_over_f_noise.

Prints one JSON line per pass: the PSD time, the median and max over bins and detectors of psd / noise_psd(n) (n the
known noise, same mask), the CG iterations and the rms map error against the sky (mean of each Stokes component
removed).

    python examples/solve_iterated_noise.py --ns 2097152 --ndet 8 --nband 4096
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ns", type=int, default=1 << 21, help="samples per detector")
    ap.add_argument("--ndet", type=int, default=8)
    ap.add_argument("--nband", type=int, default=4096, help="N^-1 coefficients per detector (<= 8192)")
    ap.add_argument("--sigma", type=float, default=1.0)
    ap.add_argument("--fknee", type=float, default=0.05, help="cycles per sample")
    ap.add_argument("--alpha", type=float, default=1.0)
    ap.add_argument("--sky", type=float, nargs=3, default=[20.0, 2.0, 2.0], help="rms of the I, Q, U sky")
    ap.add_argument("--nside", type=int, default=128)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--rtol", type=float, default=1e-8)
    args = ap.parse_args()
    import cosmomap2_b200 as cm
    from cosmomap2_b200 import synthetic
    pol, ns, ndet = 3, args.ns, args.ndet
    sc = synthetic.raster_scan(ns * ndet, nside=args.nside, ndet=ndet, nx=160, ny=80, samples_per_pixel=8.0,
                               seed=args.seed, with_data=False, flag_turnarounds=True)
    rng = np.random.default_rng(args.seed + 1)
    sky = rng.standard_normal((sc.npix_full, 3)) * args.sky
    good = sc.pix >= 0
    p = np.where(good, sc.pix, 0)
    n = synthetic.one_over_f_noise(ns, ndet, args.sigma, args.fknee, args.alpha, args.seed + 2)
    d = sky[p, 0] + sky[p, 1] * np.cos(2 * sc.phi) + sky[p, 2] * np.sin(2 * sc.phi) + n
    d[~good] = np.nan                                  # flagged samples: never read by the estimates or the solves
    d_dev = torch.from_numpy(d).cuda()
    pix_dev = torch.from_numpy(sc.pix).cuda()
    _, psd_n = cm.noise_psd(torch.from_numpy(n).cuda(), ns, pix=pix_dev)     # the known noise's estimate
    d0 = np.where(good, d, 0.0)

    def timed_psd(**kw):
        cm.noise_psd(d_dev, ns, **kw)                  # first call: module load, tables
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        psd = cm.noise_psd(d_dev, ns, **kw)[1]
        return psd, time.perf_counter() - t0

    base = {"ns": ns, "ndet": ndet, "nt": sc.nt, "nband": args.nband, "fknee": args.fknee, "alpha": args.alpha,
            "sky_rms_IQU": list(args.sky), "flagged_fraction": float(1 - good.mean())}
    psd, psd_s = timed_psd(pix=pix_dev)
    for it in (0, 1):
        if it == 1:
            psd, psd_s = timed_psd(P=P, x=x)          # the residual of the pass-0 map, P's own pixel table
        q = psd / psd_n
        bands = cm.inverse_noise_bands(psd, args.nband)
        weights = [t[0] for t in bands]
        pix = sc.pix.astype(np.int64)
        pts = cm.ProcessTimeSamples(pix, sc.npix_full, pol=pol, phi=sc.phi, w=cm.BlockLO(ns, weights).diag)
        npix, obspix = pts.get_new_pixel
        P = cm.SparseLO(npix, sc.nt, pix, pol=pol, angle_processed=pts)
        N = cm.BlockLO(ns, bands, offdiag=True)
        A = P.T * N * P
        b = P.T * (N * d0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = []
        x, info = cm.cg(A, b, M=cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol), rtol=args.rtol, maxiter=1000,
                        residuals=res)
        torch.cuda.synchronize()
        solve_s = time.perf_counter() - t0
        xh = np.asarray(x.cpu() if torch.is_tensor(x) else x).reshape(-1, pol)
        r = xh - sky[np.asarray(obspix)[:npix]]        # the solved pixels' ids, in the order of the solution
        r -= r.mean(axis=0)
        out = dict(base, **{"pass": it, "psd_source": "d" if it == 0 else "d - P x0", "psd_seconds": psd_s,
                            "psd_over_noise_median": float(np.median(q)), "psd_over_noise_max": float(np.max(q)),
                            "info": int(info), "iterations": len(res) - 1 if info == 0 else len(res),
                            "solve_seconds": solve_s, "npix": int(npix),
                            "map_rms_error_IQU": [float(v) for v in np.sqrt(np.mean(r ** 2, axis=0))]})
        print(json.dumps(out))


if __name__ == "__main__":
    main()
