#!/usr/bin/env python
"""Time cm2_noise_simulate (cosmomap2_b200.simulate_noise: Philox / Box-Muller noise generated inside the overlap-save
windows) with CUDA events, against torch.randn + cm2_noise_toeplitz_fft_apply at the same sizes and window mode, and
the host generator synthetic.one_over_f_noise.

    python tools/noise_sim_probe.py [--out profiles/r06_noise_sim_probe.json] [--reps 100] [--windows 5]

Cases: 1e8 samples in 64 noise blocks, nband in {1, 256, 4096, 8192}, one-CTA windows (up to 4096 coefficients) and
2-CTA cluster windows, the plain write and the add mode (out += n).  Each case is timed in `--windows` event windows of
`--reps` calls, alternating the simulation and the randn + apply pair window by window; the median, min and max per
call are reported.  The output (800 MB) is larger than L2.  HBM floor: 8 B/sample written (16 with add: read and
write) at 7.7 TB/s, 0.10 / 0.21 ms per 1e8 samples; randn + apply moves 8 + 16 B/sample.  The host arm is
one_over_f_noise at 1e7 samples (one timeline) on the host.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r06_noise_sim_probe.json")
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--nt", type=int, default=100_000_000)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe needs a GPU"
    from cosmomap2_b200 import _device as dv, synthetic
    from cosmomap2_b200 import linearoperators as lo

    nt, nb = args.nt, 64
    bs = nt // nb
    M = int(dv.call("cm2_toeplitz_fft_points"))
    rng = np.random.default_rng(0)
    out = torch.empty(nt, dtype=torch.float64, device="cuda")
    white = torch.empty(nt, dtype=torch.float64, device="cuda")
    y = torch.empty(nt, dtype=torch.float64, device="cuda")
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1)
    scratch = torch.empty(int(dv.call("cm2_toeplitz_fft_scratch_bytes", nb)) // 8 + 2, dtype=torch.float64,
                          device="cuda")
    result = {"card": card(), "nt": nt, "nblocks": nb, "reps": args.reps, "windows": args.windows, "cases": []}
    for L in (1, 256, 4096, 8192):
        bands = rng.standard_normal((nb, L)) / np.sqrt(L)
        bands[:, 0] = 1.0
        for pair in (0, 1):
            if not pair and 2 * (L - 1) >= M:
                continue
            coef = dv.to_dev_f64(lo.toeplitz_fft_tables(bands, L, M, pair=bool(pair)).view(np.float64).reshape(-1))
            dv.call("cm2_noise_toeplitz_fft_apply", dv.ptr(coef), L, nb, bs, None, dv.ptr(white), dv.ptr(y), nt,
                    dv.ptr(scratch), 1, pair, dv.stream())
            for add in (0, 1):
                def sim(r, add=add, pair=pair, coef=coef, L=L):
                    dv.call("cm2_noise_simulate", dv.ptr(coef), L, nb, bs, None, None, 7, r, dv.ptr(out), nt, add,
                            dv.ptr(scratch), 0, pair, dv.stream())

                def ref(pair=pair, coef=coef, L=L):
                    torch.randn(nt, dtype=torch.float64, device="cuda", generator=gen, out=white)
                    dv.call("cm2_noise_toeplitz_fft_apply", dv.ptr(coef), L, nb, bs, None, dv.ptr(white), dv.ptr(y), nt,
                            dv.ptr(scratch), 0, pair, dv.stream())

                for _ in range(3):
                    sim(0)
                    ref()
                torch.cuda.synchronize()
                t_sim, t_ref = [], []
                for w in range(args.windows):
                    for arm, acc in ((sim, t_sim), (ref, t_ref)) if w % 2 == 0 else ((ref, t_ref), (sim, t_sim)):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        for r in range(args.reps):
                            arm(r) if arm is sim else arm()
                        e1.record()
                        e1.synchronize()
                        acc.append(e0.elapsed_time(e1) / args.reps)
                floor = (16 if add else 8) * nt / HBM_BYTES_PER_S * 1e3
                case = {"nband": L, "pair": pair, "add": add,
                        "sim_ms": float(np.median(t_sim)), "sim_ms_min": min(t_sim), "sim_ms_max": max(t_sim),
                        "randn_apply_ms": float(np.median(t_ref)), "randn_apply_ms_min": min(t_ref),
                        "randn_apply_ms_max": max(t_ref),
                        "sim_ms_per_1e8": float(np.median(t_sim)) * 1e8 / nt,
                        "hbm_floor_ms": floor, "share_of_hbm_floor": floor / float(np.median(t_sim))}
                result["cases"].append(case)
                print(json.dumps(case), flush=True)
            del coef
    n_host = 10_000_000
    t0 = time.perf_counter()
    synthetic.one_over_f_noise(n_host, 1, 1.0, 0.05, 1.0, seed=0)
    th = time.perf_counter() - t0
    result["host_one_over_f_noise"] = {"samples": n_host, "s": th, "s_per_1e8": th * 1e8 / n_host}
    print(json.dumps(result["host_one_over_f_noise"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("card:", result["card"])


if __name__ == "__main__":
    main()
