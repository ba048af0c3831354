#!/usr/bin/env python
"""Time the destriper (cosmomap2_b200.Destriper) against the white and Toeplitz A-matvecs, with CUDA events.

    python tools/destripe_probe.py [--out profiles/destripe_probe.json] [--baseline 100] [--windows 3]

Cases: configs[1]'s raster (1e8 samples, 64 detectors, IQU nside 512), the same with run-free (uniform random)
pointing, and configs[2]'s share (1.25e8 samples, 8 detectors, Toeplitz bands of 4096 coefficients).  Per case:
one apply of Destriper.A (with a prior of 64 coefficients), of the fused white P^T W P and of P^T N^-1 P with the
Toeplitz bands, each timed in event windows of at least 0.3 s, the three alternated window by window; then the
full solves to rtol 1e-6 (destriper with the prior, white M_BD PCG, Toeplitz M_BD PCG) on d = P sky + 1/f-like
noise.  Byte floor of an apply: run_pix (4 B) + run_mom (24 B) per run, read twice (scatter and dot), at 7.7 TB/s.
The run table of a raster of 1e8 samples (~1.3e7 runs, 0.35 GB) is larger than L2 only a few times over, so part of
the second read may come from L2; the run-free table (1e8 runs, 2.8 GB) is not.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "unknown"


def window_ms(fn, min_s=0.3):
    """ms per call over one event window of at least min_s seconds"""
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    reps = max(3, int(np.ceil(min_s / max(time.perf_counter() - t0, 1e-6))))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, reps


def run_case(cm, name, nt, ndet, nband, random, L, windows, rtol, maxiter):
    from cosmomap2_b200 import synthetic, workloads
    nside, nx, ny, pol = 512, 1000, 500, 3
    if random:
        pix, phi, g = workloads.random_pointing(nt, nside, nx, ny, seed=0)
        ns = nt // ndet
    else:
        nt, ns, pix, phi, _l, _s, g = workloads.make_scan(nt, nside, nx, ny, ndet, 8.0, seed=0)
    bands = synthetic.toeplitz_bands(ndet, nband, seed=100)
    Nt = cm.BlockLO(ns, bands, offdiag=True)
    N = cm.BlockLO(ns, [a[0] for a in bands])
    pts = cm.ProcessTimeSamples(pix, 12 * nside ** 2, obspix=np.arange(12 * nside ** 2), pol=pol, phi=phi, w=N.diag)
    del phi
    npix = pts.get_new_pixel[0]
    P = cm.SparseLO(npix, nt, pts._pix_dev, pol=pol, angle_processed=pts)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
    prior = [1.0 * 0.7 ** np.arange(64) + np.r_[1.0, np.zeros(63)] for _ in range(ndet)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    D = cm.Destriper(P, N, Mbd, L, prior)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    Aw, At = P.T * N * P, P.T * Nt * P
    gen = torch.Generator(device="cuda").manual_seed(5)
    a = torch.randn(D.nbase, dtype=torch.float64, device="cuda", generator=gen)
    x = torch.randn(pol * npix, dtype=torch.float64, device="cuda", generator=gen)
    fns = {"destripe_A": lambda: D.A._apply(a), "white_PtWP": lambda: Aw._apply(x), "toeplitz_PtNP": lambda: At._apply(x)}
    times = {k: [] for k in fns}
    for _ in range(windows):
        for k, fn in fns.items():
            times[k].append(window_ms(fn)[0])
    floor_ms = 2 * D.run_table_bytes() / HBM_BYTES_PER_S * 1e3
    out = {"case": name, "nt": nt, "ndet": ndet, "pol": pol, "npix": int(npix), "random_pointing": random,
           "baseline": L, "nbase": D.nbase, "nruns": D._runs["nruns"], "runs_per_baseline": D._runs["nruns"] / D.nbase,
           "lanes_per_baseline": D._group, "toeplitz_nband": nband, "prior_nband": 64, "destriper_setup_s": setup_s,
           "apply_ms_median": {k: float(np.median(v)) for k, v in times.items()},
           "apply_ms_windows": times, "destripe_A_byte_floor_ms": floor_ms,
           "destripe_A_share_of_byte_floor": floor_ms / float(np.median(times["destripe_A"]))}
    print(json.dumps(out), flush=True)
    # full solves on d = P sky + noise (white plus a random offset per baseline)
    sky = torch.randn(pol * npix, dtype=torch.float64, device="cuda", generator=gen)
    d = P._apply(sky)
    d += torch.randn(nt, dtype=torch.float64, device="cuda", generator=gen)
    d += torch.repeat_interleave(torch.randn(D.nbase, dtype=torch.float64, device="cuda", generator=gen),
                                 D._end - D._start)
    solves = {}
    for k, run in (("destripe", lambda: D.solve(d, rtol=rtol, maxiter=maxiter)),
                   ("white", None), ("toeplitz", None)):
        res = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if k == "destripe":
            av, info = D.solve(d, rtol=rtol, maxiter=maxiter, residuals=res)
            D.map(d, av)
        else:
            Nk = N if k == "white" else Nt
            b = P.T._apply(Nk._apply(d))
            _, info = cm.cg(Aw if k == "white" else At, b, M=Mbd, rtol=rtol, maxiter=maxiter, residuals=res)
        torch.cuda.synchronize()
        s = time.perf_counter() - t0
        its = len(res) - 1 if info == 0 else len(res)
        solves[k] = {"seconds": s, "iterations": its, "info": int(info), "ms_per_iteration": 1e3 * s / max(its, 1)}
    out2 = {"case": name, "rtol": rtol, "maxiter": maxiter, "solves": solves}
    print(json.dumps(out2), flush=True)
    out.update(out2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--baseline", type=int, default=100)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--maxiter", type=int, default=300)
    args = ap.parse_args()
    import cosmomap2_b200 as cm
    res = {"card_name_power_limit_max_sm_clock": card(), "torch": torch.__version__, "cases": []}
    print(json.dumps(res), flush=True)
    for name, nt, ndet, nband, random in (("configs[1] raster", 100_000_000, 64, 4096, False),
                                          ("configs[1] run-free random pointing", 100_000_000, 64, 4096, True),
                                          ("configs[2] share", 125_000_000, 8, 4096, False)):
        res["cases"].append(run_case(cm, name, nt, ndet, nband, random, args.baseline, args.windows, args.rtol,
                                     args.maxiter))
        torch.cuda.empty_cache()
    res["card_after"] = card()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
