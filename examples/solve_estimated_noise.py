#!/usr/bin/env python
"""
Map-making with a noise model estimated from the data itself:

    freqs, psd = noise_psd(d, ns, pix=pix)           # per-detector Welch PSD on the GPU
    bands = inverse_noise_bands(psd, nband)           # N^-1 Toeplitz bands (host)
    A = P^T N^-1 P,  N^-1 = BlockLO(ns, bands, offdiag=True),  M_BD from the weights t[0]

on a raster scan of an IQU sky with white plus 1/f noise, P(f) = sigma^2 (1 + (fknee/|f|)^alpha), and the
same solve with the white weights t[0] alone for comparison.  Prints one JSON line: PSD and band times,
CG iterations, and the rms map error against the true sky (mean of each Stokes component removed) of both.

    python examples/solve_estimated_noise.py --ns 2097152 --ndet 8 --nband 4096
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
    sky = rng.standard_normal((sc.npix_full, 3)) * [10.0, 1.0, 1.0]
    good = sc.pix >= 0
    p = np.where(good, sc.pix, 0)
    d = sky[p, 0] + sky[p, 1] * np.cos(2 * sc.phi) + sky[p, 2] * np.sin(2 * sc.phi)
    d += synthetic.one_over_f_noise(ns, ndet, args.sigma, args.fknee, args.alpha, args.seed + 2)
    d[~good] = np.nan                                  # flagged samples: never read by the estimate or the solve
    d_dev = torch.from_numpy(d).cuda()
    pix_dev = torch.from_numpy(sc.pix).cuda()

    cm.noise_psd(d_dev, ns, pix=pix_dev)               # first call: module load, tables
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    freqs, psd = cm.noise_psd(d_dev, ns, pix=pix_dev)
    psd_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    bands = cm.inverse_noise_bands(psd, args.nband)
    band_s = time.perf_counter() - t0
    weights = [t[0] for t in bands]

    d0 = np.where(good, d, 0.0)
    out = {"ns": ns, "ndet": ndet, "nt": sc.nt, "nband": args.nband, "fknee": args.fknee, "alpha": args.alpha,
           "flagged_fraction": float(1 - good.mean()), "psd_seconds": psd_s, "bands_seconds": band_s}
    for name, N in (("gls", cm.BlockLO(ns, bands, offdiag=True)), ("white", cm.BlockLO(ns, weights))):
        pix = sc.pix.astype(np.int64)
        pts = cm.ProcessTimeSamples(pix, sc.npix_full, pol=pol, phi=sc.phi, w=cm.BlockLO(ns, weights).diag)
        npix, obspix = pts.get_new_pixel
        P = cm.SparseLO(npix, sc.nt, pix, pol=pol, angle_processed=pts)
        A = P.T * N * P
        b = P.T * (N * d0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = []
        x, info = cm.cg(A, b, M=cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol), rtol=args.rtol, maxiter=1000,
                        residuals=res)
        torch.cuda.synchronize()
        x = np.asarray(x.cpu() if torch.is_tensor(x) else x).reshape(-1, pol)
        r = x - sky[np.asarray(obspix)[:npix]]          # the solved pixels' ids, in the order of the solution
        r -= r.mean(axis=0)
        out[name] = {"info": int(info), "iterations": len(res) - 1 if info == 0 else len(res),
                     "solve_seconds": time.perf_counter() - t0, "npix": int(npix),
                     "map_rms_error_IQU": [float(v) for v in np.sqrt(np.mean(r ** 2, axis=0))]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
