#!/usr/bin/env python
"""Per-kernel device time of bench.py's step loop (configs[1] at N = 1: start() + step_async() + tick()) under
torch.profiler.  Usage: python tools/prof_step.py [--nt 100000000] [--steps 50] [--out profiles/step_kernels.json]

Writes, per kernel name, the number of launches and the device time per step (mean over the profiled steps), the
sum over kernels and the wall time per step of the same loop timed with CUDA events and the profiler off."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmomap2_b200 as cm  # noqa: E402
from cosmomap2_b200 import synthetic, _device as dv  # noqa: E402
from cosmomap2_b200.pcg import make_solver  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nt", type=int, default=100000000)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "step_kernels.json"))
    args = ap.parse_args()
    pol = 3
    sc = synthetic.config_c2(nt=args.nt, seed=0)
    N = cm.BlockLO(sc.ns, sc.weights)
    pts = cm.ProcessTimeSamples(sc.pix, sc.npix_full, pol=pol, phi=sc.phi, w=N.diag)
    npix = pts.get_new_pixel[0]
    P = cm.SparseLO(npix, sc.nt, sc.pix, pol=pol, angle_processed=pts)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
    A = P.T * N * P
    b = P.T._apply(N._apply(dv.to_dev_f64(sc.d)))
    sc.d = None
    solver = make_solver(A, Mbd, pol * npix)

    def one_step():
        solver.start(b)
        solver.step_async()
        solver.tick()

    for _ in range(20):
        one_step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        one_step()
    e1.record()
    torch.cuda.synchronize()
    ms_per_step = e0.elapsed_time(e1) / args.steps

    acts = [torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        for _ in range(args.steps):
            one_step()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.events():
        # device-side activity only (kernels, memsets, copies); CPU-side rows would count the same time again
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        k = kernels.setdefault(ev.name, {"launches_per_step": 0.0, "us_per_step": 0.0})
        k["launches_per_step"] += 1.0 / args.steps
        k["us_per_step"] += ev.time_range.elapsed_us() / args.steps
    out = {"gpu": gpu_info(), "nt": sc.nt, "npix": int(npix), "steps": args.steps,
           "ms_per_step_events_profiler_off": ms_per_step,
           "kernel_us_per_step_sum": sum(v["us_per_step"] for v in kernels.values()),
           "kernels": dict(sorted(kernels.items(), key=lambda kv: -kv[1]["us_per_step"]))}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
