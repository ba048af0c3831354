#!/usr/bin/env python
"""Time cm2_noise_psd (the per-block Welch sums of cosmomap2_b200.noise_psd) with CUDA events, next to
scipy.signal.welch on the host cores on the same data.

    python tools/noise_probe.py [--out profiles/noise_probe.json] [--reps 200] [--windows 5]

Cases: 1e8 samples in 64 noise blocks, and configs[2]'s per-GPU share (1.25e8 samples, 8 blocks), each
without and with a pixel mask.  The TOD (800 MB+) is larger than L2, so every timed call streams it from
HBM.  Each case is timed in `--windows` event windows of `--reps` calls (about 0.4 s each), alternating the
masked and unmasked calls window by window; the median, min and max per call are reported.  HBM floor: 8 B
of d + 4 B of pix per sample = 12 B/sample (8 without a mask) at 7.7 TB/s.  The host arm is
scipy.signal.welch on one core, and on every core of the process: blocks on a thread pool, the rest of the
cores as scipy.fft workers.
"""
import argparse
import concurrent.futures
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.fft
import scipy.signal
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
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--windows", type=int, default=5)
    args = ap.parse_args()
    from cosmomap2_b200 import _cabi, _device as dv
    M = int(dv.call("cm2_toeplitz_fft_points"))
    NF = 2 * M
    res = {"card": card(), "torch": torch.__version__, "host_cores": len(os.sched_getaffinity(0)), "cases": []}
    g = torch.Generator(device="cuda").manual_seed(3)
    for nt, nb in ((100_000_000, 64), (125_000_000, 8)):
        bs = nt // nb
        d = torch.randn(nt, dtype=torch.float64, device="cuda", generator=g)
        pix = torch.randint(0, 1 << 20, (nt,), dtype=torch.int32, device="cuda", generator=g)
        pix[torch.arange(nt, device="cuda") % 5000 < 300] = -1
        scratch = torch.empty(int(dv.call("cm2_noise_psd_scratch_bytes", nb)) // 8 + 2, dtype=torch.float64,
                              device="cuda")
        S = torch.empty(nb * (M + 1), dtype=torch.float64, device="cuda")
        W = torch.empty(nb, dtype=torch.float64, device="cuda")
        nwin = nb * ((bs - NF) // M + 1)
        calls = {}
        for masked in (False, True):
            p = dv.ptr(pix) if masked else None

            def call(init=0, p=p):
                dv.call("cm2_noise_psd", dv.ptr(d), p, nb, bs, None, nt, dv.ptr(S), dv.ptr(W), dv.ptr(scratch), init,
                        dv.stream())
            call(1)
            call()
            calls[masked] = call
        torch.cuda.synchronize()
        times = {False: [], True: []}
        for _ in range(args.windows):
            for masked in (False, True):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    calls[masked]()
                e1.record()
                torch.cuda.synchronize()
                times[masked].append(e0.elapsed_time(e1) / args.reps)
        for masked in (False, True):
            ms = float(np.median(times[masked]))
            bps = 12.0 if masked else 8.0
            floor_ms = bps * nt / HBM_BYTES_PER_S * 1e3
            res["cases"].append({"nt": nt, "nblocks": nb, "masked": masked, "windows": nwin, "ms": ms,
                                 "ms_min": min(times[masked]), "ms_max": max(times[masked]),
                                 "ms_per_window_of_calls": times[masked], "calls_per_window": args.reps,
                                 "ms_per_1e8_samples": ms * 1e8 / nt, "samples_per_s": nt / (ms * 1e-3),
                                 "hbm_floor_B_per_sample": bps, "hbm_floor_ms": floor_ms,
                                 "share_of_hbm_floor": floor_ms / ms})
            print(json.dumps(res["cases"][-1]), flush=True)
        # the host estimate of the same (unmasked) data, one block after the other, on one core and on all of them
        dh = dv.to_host(d)
        dv.call("cm2_noise_psd", dv.ptr(d), None, nb, bs, None, nt, dv.ptr(S), dv.ptr(W), dv.ptr(scratch), 0,
                dv.stream())
        Pg = dv.to_host(S).reshape(nb, M + 1) / dv.to_host(W)[:, None]
        gpu_ms = [c["ms"] for c in res["cases"] if c["nt"] == nt and not c["masked"]][0]
        def host_block(b, workers):
            seg = dh[b * bs:(b + 1) * bs if b + 1 < nb else nt]
            with scipy.fft.set_workers(workers):
                return scipy.signal.welch(seg, fs=1.0, window="hann", nperseg=NF, noverlap=M, detrend=False,
                                          return_onesided=False)[1][:M + 1]
        for cores in (1, res["host_cores"]):
            t0 = time.perf_counter()
            if cores == 1:
                Ph = np.array([host_block(b, 1) for b in range(nb)])
            else:     # blocks on a thread pool (NumPy and pocketfft release the GIL), FFT workers for the rest
                with concurrent.futures.ThreadPoolExecutor(min(cores, nb)) as ex:
                    Ph = np.array(list(ex.map(lambda b: host_block(b, max(1, cores // nb)), range(nb))))
            host_s = time.perf_counter() - t0
            res["cases"].append({"nt": nt, "nblocks": nb, "host_cores_used": cores, "host_scipy_welch_s": host_s,
                                 "host_samples_per_s": nt / host_s, "gpu_speedup": host_s / (gpu_ms * 1e-3),
                                 "max_rel_diff_gpu_vs_scipy": float(np.max(np.abs(Pg - Ph) / Ph))})
            print(json.dumps(res["cases"][-1]), flush=True)
        del d, pix, S, W, scratch, dh
        torch.cuda.empty_cache()
    res["launches"] = _cabi.launch_count()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "host_cores": res["host_cores"]}))


if __name__ == "__main__":
    main()
