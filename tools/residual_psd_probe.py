#!/usr/bin/env python
"""Time the Welch PSD of a map residual d - P x three ways with CUDA events, and record the device memory each path
needs.

    python tools/residual_psd_probe.py [--out profiles/residual_psd_probe.json] [--reps 50] [--windows 5]

Data: 1e8 samples in 64 noise blocks (one per detector) of synthetic.config_c2's raster scan at nside 512, its pixel
ids compacted to the observed pixels (as ProcessTimeSamples does), pol 1 and 3, without and with flagged turnarounds
(5 % of each sweep).  Per case, these are timed in alternating event windows of --reps calls each:
  fused    cm2_noise_psd_residual: what noise_psd(d, bs, P=P, x=x) launches
  unfused  P.mult(x) (cm2_pointing_apply into a new TOD tensor), a torch subtraction, then cm2_noise_psd with P's
           pixel table: what noise_psd(d - P.mult(x), bs, pix=...) launches
  plain    cm2_noise_psd(d) without a mask, and with P's pixel table
The median, min and max per call are reported.  The TOD (800 MB per vector) is larger than L2, so every call streams it
from HBM; the map (pol x 8 B x ~0.5 M pixels) stays in L2.  HBM floors at 7.7 TB/s: fused 12 B/sample (d, pix) + 16
for cos / sin at pol 3; unfused 4 + 16 + 8 (P x) + 8 + 8 + 8 (subtraction) + 8 + 4 (PSD) = 64 B/sample at pol 3 (48
at pol 1).  Memory: torch.cuda.max_memory_allocated over one call of noise_psd through each path, above what was
allocated before it.
"""
import argparse
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--nt", type=int, default=100_000_000)
    args = ap.parse_args()
    import cosmomap2_b200 as cm
    from cosmomap2_b200 import _cabi, _device as dv, synthetic
    M = int(dv.call("cm2_toeplitz_fft_points"))
    res = {"card": card(), "torch": torch.__version__, "cases": []}
    nb = 64
    sc = synthetic.config_c2(nt=args.nt, with_data=False)
    nt, bs = sc.nt, sc.ns
    raw = torch.from_numpy(sc.pix).cuda()
    uniq, inv = torch.unique(raw, return_inverse=True)
    pix_all = inv.to(torch.int32)
    npix = int(uniq.numel())
    # flagged turnarounds: the first and last 2.5 % of every sweep, as raster_scan(flag_turnarounds=True) does
    sweep = int(round(sc.nx * sc.samples_per_pixel))
    frac = (torch.arange(nt, device="cuda") % bs % sweep).double() / sweep
    pix_flag = torch.where((frac < 0.025) | (frac >= 0.975), torch.full_like(pix_all, -1), pix_all)
    phi = torch.from_numpy(sc.phi).cuda()
    ang = types.SimpleNamespace(_cos_dev=torch.cos(2 * phi), _sin_dev=torch.sin(2 * phi))
    del phi, raw, inv, frac
    g = torch.Generator(device="cuda").manual_seed(3)
    d = torch.randn(nt, dtype=torch.float64, device="cuda", generator=g)
    scratch = torch.empty(int(dv.call("cm2_noise_psd_scratch_bytes", nb)) // 8 + 2, dtype=torch.float64, device="cuda")
    S = torch.empty(nb * (M + 1), dtype=torch.float64, device="cuda")
    W = torch.empty(nb, dtype=torch.float64, device="cuda")
    res.update({"nt": nt, "nblocks": nb, "blocksize": bs, "nside": sc.nside, "npix_observed": npix,
                "flagged_fraction": float((pix_flag < 0).double().mean().item())})
    for pol in (1, 3):
        x = torch.randn(pol * npix, dtype=torch.float64, device="cuda", generator=g)
        for flags in (False, True):
            pix = pix_flag if flags else pix_all
            P = cm.SparseLO(npix, nt, pix, pol=pol, angle_processed=ang if pol > 1 else None)

            def psd(dd, p):
                dv.call("cm2_noise_psd", dv.ptr(dd), dv.ptr(p), nb, bs, None, nt, dv.ptr(S), dv.ptr(W), dv.ptr(scratch),
                        0, dv.stream())

            calls = {
                "fused": lambda: dv.call("cm2_noise_psd_residual", dv.ptr(d), dv.ptr(P._pix_dev), dv.ptr(P._cos_dev),
                                         dv.ptr(P._sin_dev), pol, dv.ptr(x), nb, bs, None, nt, dv.ptr(S), dv.ptr(W),
                                         dv.ptr(scratch), 0, dv.stream()),
                "unfused": lambda: psd(d - P.mult(x), P._pix_dev),
                "plain_unmasked": lambda: psd(d, None),
                "plain_masked": lambda: psd(d, P._pix_dev),
            }
            dv.call("cm2_noise_psd", dv.ptr(d), None, nb, bs, None, nt, dv.ptr(S), dv.ptr(W), dv.ptr(scratch), 1,
                    dv.stream())                        # the twiddle and window tables in the scratch
            for f in calls.values():
                f()
                f()
            torch.cuda.synchronize()
            # the fused and unfused sums agree bit for bit
            calls["fused"]()
            a = S.clone(), W.clone()
            calls["unfused"]()
            same = bool(torch.equal(a[0], S) and torch.equal(a[1], W))
            times = {k: [] for k in calls}
            for _ in range(args.windows):
                for k, f in calls.items():
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(args.reps):
                        f()
                    e1.record()
                    torch.cuda.synchronize()
                    times[k].append(e0.elapsed_time(e1) / args.reps)
            # device memory of one noise_psd call through each path
            mem = {}
            for k, f in (("fused", lambda: cm.noise_psd(d, bs, P=P, x=x)),
                         ("unfused", lambda: cm.noise_psd(d - P.mult(x), bs, pix=P._pix_dev))):
                torch.cuda.synchronize()
                torch.cuda.empty_cache()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                f()
                torch.cuda.synchronize()
                mem[k] = torch.cuda.max_memory_allocated() - base
            floors = {"fused": 12 + (16 if pol > 1 else 0), "unfused": 48 + (16 if pol > 1 else 0),
                      "plain_unmasked": 8, "plain_masked": 12}
            case = {"pol": pol, "flags": flags, "fused_equals_unfused_bits": same,
                    "peak_extra_bytes_noise_psd": mem}
            for k in calls:
                ms = float(np.median(times[k]))
                floor_ms = floors[k] * nt / HBM_BYTES_PER_S * 1e3
                case[k] = {"ms": ms, "ms_min": min(times[k]), "ms_max": max(times[k]), "ms_per_window": times[k],
                           "ms_per_1e8_samples": ms * 1e8 / nt, "hbm_floor_B_per_sample": floors[k],
                           "hbm_floor_ms": floor_ms, "share_of_hbm_floor": floor_ms / ms}
            case["calls_per_window"] = args.reps
            res["cases"].append(case)
            print(json.dumps({"pol": pol, "flags": flags, "same_bits": same, "mem": mem,
                              **{k: round(case[k]["ms"], 4) for k in calls}}), flush=True)
            del P
        del x
    res["launches"] = _cabi.launch_count()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
