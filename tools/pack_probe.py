#!/usr/bin/env python
"""Fused white A-matvec (cm2_amatvec_white) over the int32 pixel ids vs over the packed pixel stream
(cm2_pack_pointing), on the same operator and inputs.  Usage: python tools/pack_probe.py [out.json] [--quick]

Patterns: configs[1] (1e8 samples, IQU nside 512, time order), the benchmark's sensitivity patterns that take the
register scatter (5e7 samples: 8 and 32 samples per pixel crossing, a scan tilted 30 degrees at 8), and configs[4]'s
detector-interleaved order (1e9 samples, nside 2048).  Per pattern: kernel time of both (CUDA events, the two
alternated in rounds after a >= 0.5 s warm-up of each), the bytes each reads (int32: 20 B/sample; packed:
17 B/sample + 32 B per escape lane; both + 48 B/pixel for x and y) and the GB/s they give, the escape fraction,
and max|y_packed - y_int32| / max|y_int32|."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cosmomap2_b200 as cm  # noqa: E402
from cosmomap2_b200 import synthetic, workloads, linearoperators as lo, _device as dv  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else None
    except Exception:
        return None


def probe(name, P, N, rounds=5, iters=20):
    A = P.T * N * P
    x = torch.randn(P.pol * P.ncols, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    A._apply(x)                                        # plans the fused operator and builds the packed stream
    f = [op for op in A.planned() if isinstance(op, lo._FusedWhiteA)][0]
    assert f._mode == "registers", (name, f._mode)
    selected = f._packed is not None
    if not selected:
        f._build_packed()                              # the packed stream is measured where the operator does not plan it
    nb, bs, startp = N._blk.args()
    y = {k: dv.zeros_f64(P.pol * P.ncols) for k in ("int32", "packed")}

    def run(kind):
        dv.call("cm2_amatvec_white", dv.ptr(P._pix_dev), dv.ptr(f._packed) if kind == "packed" else None,
                dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows, P.pol, dv.ptr(N.weights_dev()), nb, bs, startp,
                dv.ptr(x), dv.ptr(y[kind]), P.ncols, f._streams, dv.stream())

    for kind in ("int32", "packed"):
        t0 = time.time()
        while time.time() - t0 < 0.5:
            run(kind)
            torch.cuda.synchronize()
    ms = {"int32": [], "packed": []}
    for _ in range(rounds):
        for kind in ("int32", "packed"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                run(kind)
            e1.record()
            torch.cuda.synchronize()
            ms[kind].append(e0.elapsed_time(e1) / iters)
    yi, yp = y["int32"], y["packed"]
    nt, npix = P.nrows, P.ncols
    nlanes = (nt + 7) // 8
    nbytes = {"int32": 20.0 * nt + 48.0 * npix, "packed": float(f.tod_bytes()) + 48.0 * npix}
    row = {"pattern": name, "nt": int(nt), "npix": int(npix), "nstreams": int(f._streams), "packed_selected": selected,
           "escape_lanes": int(f.nescape), "escape_fraction": f.nescape / max(nlanes, 1),
           "max_rel_dy": float((yp - yi).abs().max() / yi.abs().max())}
    for kind in ("int32", "packed"):
        m = float(np.mean(ms[kind]))
        row[kind] = {"ms": m, "ms_rounds": ms[kind], "bytes": nbytes[kind], "GBs": nbytes[kind] / m / 1e6}
    row["packed_vs_int32_time"] = row["packed"]["ms"] / row["int32"]["ms"]
    print(json.dumps(row), flush=True)
    del A, f, x, y
    return row


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    quick = "--quick" in sys.argv
    out = {"gpu": gpu_info(), "patterns": []}
    print(json.dumps({"gpu": out["gpu"]}), flush=True)
    pol = 3

    sc = synthetic.config_c2(nt=int(1e6 if quick else 1e8), seed=0, with_data=False)
    N = cm.BlockLO(sc.ns, sc.weights)
    pts = cm.ProcessTimeSamples(sc.pix, sc.npix_full, pol=pol, phi=sc.phi, w=N.diag)
    P = cm.SparseLO(pts.get_new_pixel[0], sc.nt, sc.pix, pol=pol, angle_processed=pts)
    out["patterns"].append(probe("configs[1]", P, N))
    del sc, N, pts, P
    torch.cuda.empty_cache()

    nside, nx, ny, ndet = 512, 1000, 500, 64
    for name, spp, tilt in (("spp=8", 8.0, 0.0), ("spp=32", 32.0, 0.0), ("tilt30 spp=8", 8.0, 30.0)):
        nt, ns, pix, phi, _a, _b, _g = workloads.make_scan(int(5e5 if quick else 5e7), nside, nx, ny, ndet, spp, seed=0,
                                                           turnaround=0.0, tilt_deg=tilt)
        N = cm.BlockLO(ns, 0.5 + np.random.default_rng(0).random(ndet))
        pts = cm.ProcessTimeSamples(pix, 12 * nside ** 2, obspix=np.arange(12 * nside ** 2), pol=pol, phi=phi, w=N.diag)
        P = cm.SparseLO(pts.get_new_pixel[0], nt, pts._pix_dev, pol=pol, angle_processed=pts)
        out["patterns"].append(probe("sensitivity " + name, P, N))
        del pix, phi, N, pts, P
        torch.cuda.empty_cache()

    nside = 2048
    nt, ns, pix, phi, _a, _b, g = workloads.make_scan(int(1e6 if quick else 1e9), nside, 3200, 1600, 64, 8.0, seed=0,
                                                      turnaround=0.0)
    w = 0.5 + torch.rand(64, generator=g, device="cuda", dtype=torch.float64).cpu().numpy()
    N = cm.BlockLO(ns, w)
    pts = cm.ProcessTimeSamples(pix, 12 * nside ** 2, obspix=np.arange(12 * nside ** 2), pol=pol, phi=phi, w=N.diag)
    del phi
    P = cm.SparseLO(pts.get_new_pixel[0], nt, pts._pix_dev, pol=pol, angle_processed=pts)
    out["patterns"].append(probe("configs[4]", P, N, rounds=3, iters=5))

    if args:
        os.makedirs(os.path.dirname(os.path.abspath(args[0])), exist_ok=True)
        with open(args[0], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
