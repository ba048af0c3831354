#!/usr/bin/env python
"""
Destriping with a noise prior against the white-weight map and Toeplitz GLS, on the data of solve_iterated_noise.py:
a raster scan with flagged turnarounds, an IQU sky well above the noise and 1/f noise
P(f) = sigma^2 (1 + (fknee/|f|)^alpha).

    white        cg(P^T W P, P^T W d), W = 1/sigma2 per detector from the PSD estimate
    destripe     destripe(d, P, N, M_BD, L) without a prior (map up to the I monopole)
    destripe     with the prior baseline_prior_bands(noise_psd(d), L, nband), at two baseline lengths
    gls          cg(P^T N^-1 P, P^T N^-1 d), N^-1 = inverse_noise_bands(noise_psd(d), nband)

Prints one JSON line per case: the CG iterations, the solve time (device synchronised; set-up such as the run table
excluded and reported apart) and the rms map error against the sky per Stokes component (mean of each removed).

    python examples/solve_destriped.py --ns 2097152 --ndet 8 --nband 4096 --baselines 64 512
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
    ap.add_argument("--nband", type=int, default=4096, help="N^-1 coefficients per detector for GLS (<= 8192)")
    ap.add_argument("--prior-nband", type=int, default=256, help="prior coefficients per detector")
    ap.add_argument("--baselines", type=int, nargs=2, default=[64, 512], help="two baseline lengths in samples")
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
    d = np.where(good, d, 0.0)
    d_dev = torch.from_numpy(d).cuda()
    _, psd = cm.noise_psd(d_dev, ns, pix=torch.from_numpy(sc.pix).cuda())
    bands = cm.inverse_noise_bands(psd, args.nband)
    weights = cm.baseline_prior_bands(psd, args.baselines[0], args.prior_nband)[0]
    N = cm.BlockLO(ns, list(weights))
    pix = sc.pix.astype(np.int64)
    pts = cm.ProcessTimeSamples(pix, sc.npix_full, pol=pol, phi=sc.phi, w=N.diag)
    npix, obspix = pts.get_new_pixel
    P = cm.SparseLO(npix, sc.nt, pix, pol=pol, angle_processed=pts)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
    truth = sky[np.asarray(obspix)[:npix]]
    base = {"ns": ns, "ndet": ndet, "nt": sc.nt, "npix": int(npix), "fknee": args.fknee, "alpha": args.alpha,
            "sky_rms_IQU": list(args.sky), "flagged_fraction": float(1 - good.mean()), "rtol": args.rtol,
            "gpu": torch.cuda.get_device_name()}

    def report(case, x, info, iters, solve_s, **extra):
        r = (x.cpu().numpy() if torch.is_tensor(x) else np.asarray(x)).reshape(-1, pol) - truth
        r -= r.mean(axis=0)
        out = dict(base, case=case, info=int(info), iterations=iters, solve_seconds=solve_s,
                   map_rms_error_IQU=[float(v) for v in np.sqrt(np.mean(r ** 2, axis=0))], **extra)
        print(json.dumps(out), flush=True)

    def timed_cg(A, b, M):
        cm.cg(A, b, M=M, rtol=args.rtol, maxiter=3)            # warm-up: modules, tables, solver state
        torch.cuda.synchronize()
        res = []
        t0 = time.perf_counter()
        x, info = cm.cg(A, b, M=M, rtol=args.rtol, maxiter=5000, residuals=res)
        torch.cuda.synchronize()
        return x, info, (len(res) - 1 if info == 0 else len(res)), time.perf_counter() - t0

    x, info, it, s = timed_cg(P.T * N * P, P.T * (N * d_dev), Mbd)
    report("white", x, info, it, s)
    for L, with_prior in ((args.baselines[0], False), (args.baselines[0], True), (args.baselines[1], True)):
        prior = cm.baseline_prior_bands(psd, L, args.prior_nband)[1] if with_prior else None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        D = cm.Destriper(P, N, Mbd, L, prior)
        torch.cuda.synchronize()
        setup_s = time.perf_counter() - t0
        D.solve(d_dev, rtol=args.rtol, maxiter=3)
        torch.cuda.synchronize()
        res = []
        t0 = time.perf_counter()
        a, info = D.solve(d_dev, rtol=args.rtol, maxiter=5000, residuals=res)
        x = D.map(d_dev, a)
        torch.cuda.synchronize()
        report("destripe_prior" if with_prior else "destripe_no_prior", x, info,
               len(res) - 1 if info == 0 else len(res), time.perf_counter() - t0, baseline=L, nbase=D.nbase,
               nruns=D._runs["nruns"], setup_seconds=setup_s)
    x, info, it, s = timed_cg(P.T * cm.BlockLO(ns, bands, offdiag=True) * P,
                              P.T * (cm.BlockLO(ns, bands, offdiag=True) * d_dev), Mbd)
    report("gls_toeplitz", x, info, it, s, nband=args.nband)


if __name__ == "__main__":
    main()
