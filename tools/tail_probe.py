#!/usr/bin/env python
"""Device time of the M_BD PCG tail (cm2_pcg_bd_reset's x0 = 0 start with p0, cm2_pcg_bd_iter) at the pixel counts of
configs[1], [3], [4], for the coalesced tiled kernels and for the one-thread-per-pixel kernels side by side, plus the
generic-M updates (development tool).  Usage: python tools/tail_probe.py [out.json]

Algorithmic bytes per pixel (POL = 3): the tiled start reads b, inv and writes r, x, p (144 B; the strided one also
writes z: 168 B); the tiled iteration reads p, q, x, r, inv and writes x, r, p (216 B; the strided one reads p and q
twice, p a third time, and writes and re-reads z: 336 B).  Above cm2_pcg_bd_iter_max_npix(3) the library's iteration
IS the strided kernel."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmomap2_b200 as cm  # noqa: E402,F401
from cosmomap2_b200 import workloads, _device as dv  # noqa: E402

BYTES = {"strided": {"reset": 168.0, "iter": 336.0}, "tiled": {"reset": 144.0, "iter": 216.0}}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except Exception:
        return None


def main():
    lines = [{"gpu": gpu_info(), "bd_iter_max_npix_pol3": dv.call("cm2_pcg_bd_iter_max_npix", 3)}]
    print(json.dumps(lines[0]), flush=True)
    st = dv.stream
    for npix in (500000, 1280000, 5120000):
        n = 3 * npix
        g = torch.Generator(device="cuda").manual_seed(1)
        inv = torch.rand(6 * npix, dtype=torch.float64, device="cuda", generator=g) + 0.5
        p, q, x, r, z, b = (torch.randn(n, dtype=torch.float64, device="cuda", generator=g) for _ in range(6))
        scal = dv.zeros_f64(16)

        def reset():
            dv.call("cm2_pcg_bd_reset", dv.ptr(inv), npix, 3, dv.ptr(r), dv.ptr(z), dv.ptr(scal), 0.0, 0.0, dv.ptr(b),
                    dv.ptr(x), dv.ptr(p), st())

        def it():
            dv.call("cm2_pcg_bd_iter", dv.ptr(inv), npix, 3, dv.ptr(p), dv.ptr(q), dv.ptr(x), dv.ptr(r), dv.ptr(z),
                    dv.ptr(scal), st())

        def upd():
            dv.call("cm2_pcg_update_p", dv.ptr(r), dv.ptr(z), dv.ptr(p), n, dv.ptr(scal), st())
            dv.call("cm2_pcg_update_xr", dv.ptr(p), dv.ptr(q), dv.ptr(x), dv.ptr(r), n, dv.ptr(scal), st())

        out = {"npix": npix, "bd_iter_path": "tiled" if npix <= lines[0]["bd_iter_max_npix_pol3"] else "strided"}
        # alternate the two variants three times; report every repetition's time
        for rep in range(3):
            for kind in ("strided", "tiled"):
                old = dv.call("cm2_pcg_bd_tail_strided", 1 if kind == "strided" else 0)
                try:
                    reset()
                    scal[7] = 0.0          # atol = 0: the iteration never raises `done` by itself
                    out.setdefault("bd_reset_ms_" + kind, []).append(workloads.time_device(reset, 50))
                    reset()
                    scal[7] = 0.0
                    out.setdefault("bd_iter_ms_" + kind, []).append(workloads.time_device(it, 50))
                finally:
                    dv.call("cm2_pcg_bd_tail_strided", old)
        for kind in ("strided", "tiled"):
            for op in ("reset", "iter"):
                t = min(out["bd_%s_ms_%s" % (op, kind)])
                # above the on-chip bound the library's iteration is the strided kernel: count what actually ran
                ran = "strided" if op == "iter" and out["bd_iter_path"] == "strided" else kind
                out["bd_%s_bytes_%s" % (op, kind)] = BYTES[ran][op] * npix
                out["bd_%s_GBs_%s" % (op, kind)] = BYTES[ran][op] * npix / t / 1e6
        out["generic_update_p_plus_xr_ms"] = workloads.time_device(upd, 50)
        lines.append(out)
        print(json.dumps(out), flush=True)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
