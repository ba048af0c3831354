#!/usr/bin/env python
"""
Noise Monte Carlo with the noise model estimated from the data:

    freqs, psd = noise_psd(d, ns, pix=pix)                 # per-detector Welch PSD on the GPU
    sim = NoiseSimulator(noise_sim_bands(psd, nband), ns)   # bands with that PSD, device tables kept
    for k in range(K):  n_k = sim(seed, realization=k)      # one noise-only TOD per realization, on the device
                        solve A m_k = P^T N^-1 n_k          # the same GLS A and M_BD for every realization

on a raster scan with white plus 1/f noise.  The per-pixel rms of the K noise-only maps is the Monte Carlo estimate of
the map noise.  Prints one JSON line: the per-realization time of the simulation, the right-hand side and the solve,
and a summary (median and quartiles) of the per-pixel MC noise rms of I, Q and U.

    python examples/noise_monte_carlo.py --ns 2097152 --ndet 8 --nband 4096 --K 8
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
    ap.add_argument("--nband", type=int, default=4096, help="N^-1 and simulation coefficients per detector (<= 8192)")
    ap.add_argument("--K", type=int, default=8, help="noise realizations")
    ap.add_argument("--fknee", type=float, default=0.05, help="cycles per sample")
    ap.add_argument("--alpha", type=float, default=1.0)
    ap.add_argument("--nside", type=int, default=128)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--rtol", type=float, default=1e-6)
    args = ap.parse_args()
    import cosmomap2_b200 as cm
    from cosmomap2_b200 import synthetic
    pol, ns, ndet = 3, args.ns, args.ndet
    sc = synthetic.raster_scan(ns * ndet, nside=args.nside, ndet=ndet, nx=160, ny=80, samples_per_pixel=8.0,
                               seed=args.seed, with_data=False)
    d = synthetic.one_over_f_noise(ns, ndet, 1.0, args.fknee, args.alpha, args.seed + 2)
    _, psd = cm.noise_psd(d, ns)
    N = cm.BlockLO(ns, cm.inverse_noise_bands(psd, args.nband), offdiag=True)
    weights = [t[0] for t in N.covnoise]
    sim = cm.NoiseSimulator(cm.noise_sim_bands(psd, args.nband), ns)

    pix = sc.pix.astype(np.int64)
    pts = cm.ProcessTimeSamples(pix, sc.npix_full, pol=pol, phi=sc.phi, w=cm.BlockLO(ns, weights).diag)
    npix = pts.get_new_pixel[0]
    P = cm.SparseLO(npix, sc.nt, pix, pol=pol, angle_processed=pts)
    A = P.T * N * P
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)

    t_sim, t_rhs, t_solve, iters = [], [], [], []
    maps = []
    for k in range(args.K + 1):                       # realization 0 also warms up every kernel and table
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = sim(args.seed, realization=k)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        b = P.T * (N * n)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        res = []
        x, info = cm.cg(A, b, M=Mbd, rtol=args.rtol, maxiter=1000, residuals=res)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        if k == 0:
            continue
        t_sim.append(t1 - t0)
        t_rhs.append(t2 - t1)
        t_solve.append(t3 - t2)
        iters.append(len(res) - 1 if info == 0 else len(res))
        maps.append(np.asarray(x.cpu() if torch.is_tensor(x) else x).reshape(-1, pol))
    rms = np.sqrt(np.mean(np.square(maps), axis=0))               # per pixel and Stokes component
    q = np.percentile(rms, [25, 50, 75], axis=0)
    out = {"ns": ns, "ndet": ndet, "nt": sc.nt, "nband": args.nband, "K": args.K, "npix": int(npix),
           "sim_ms": 1e3 * float(np.median(t_sim)), "rhs_ms": 1e3 * float(np.median(t_rhs)),
           "solve_ms": 1e3 * float(np.median(t_solve)), "cg_iterations": iters,
           "mc_rms_IQU_q25_median_q75": [[float(v) for v in q[:, c]] for c in range(pol)],
           "card": torch.cuda.get_device_name()}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
