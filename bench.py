#!/usr/bin/env python
"""
bench.py -- BASELINE.json's metric on BASELINE.json's configuration.

    metric   : TOD samples/s per PCG iteration (one A apply + one M apply + the CG vector work)
    workload : configs[1] -- synthetic raster scan, 1e8 samples per GPU, IQU nside=512, white noise
               (64 detector blocks), block-diagonal-preconditioned PCG on A = P^T N^-1 P
    N GPUs   : weak scaling -- every rank owns its own 64 detectors x 1e8/64 samples of the same sky
               patch; per iteration one local TOD pass + one kernel that fuses the map exchange over
               NVLink peer memory with the pixel-sharded M_BD / CG vector work (csrc/pcg_sharded.cu)

    python bench.py --gpus N --steps K --warmup W        (torchrun launches it for N > 1)
    python bench.py --impl reference ...                  (CPU arm: the oracle port on host cores)

A step = one full PCG iteration from a fresh residual (r <- b, x <- 0, then z = M r, rho, p, q = A p,
alpha, x, r, ||r||).  White noise with the weights fed to M_BD makes M_BD A = I, so the solve
converges in ONE iteration (the reference expects exactly that,
src/test_BD_precond_onto_real_data.py:52); iterating on the converged residual would only process
rounding noise until it underflows, hence the restart -- the work per step is the full iteration.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "tod_samples_per_s_per_pcg_iter"
UNIT = "samples/s"


_json_out = None


def claim_stdout():
    """Keep stdout to the ONE JSON line of the contract: the real stdout is set aside for it and file
    descriptor 1 is pointed at stderr, so banners that libraries print to stdout (NCCL prints its
    version there when NCCL_DEBUG is VERSION or WARN) cannot get in front of it."""
    global _json_out
    if _json_out is None:
        sys.stdout.flush()
        _json_out = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    claim_stdout()
    _json_out.write(json.dumps(line) + "\n")
    _json_out.flush()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nt", type=int, default=100000000, help="TOD samples per GPU (configs[1]: 1e8)")
    ap.add_argument("--cpu-nt", type=int, default=30000000, help="samples of the bounded CPU-baseline sample")
    ap.add_argument("--cpu-iters", type=int, default=10)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip the `secondary` block (configs[2], configs[3], configs[4] on this run's GPUs)")
    ap.add_argument("--secondary-timeout", type=float, default=420.0,
                    help="seconds after which the line is printed without the unfinished part of `secondary`")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --nt samples per GPU (default, the contract); strong: --nt samples in total")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (the PCG iterate x) as "
                         "DIR/<name>.npy in float64, so that two builds can be compared on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write every array as ``out_dir/<name>.npy`` in float64."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    # x has 3 entries per observed pixel of the fixed 1000 x 500 patch: at most 12 MB
    assert total <= DUMP_LIMIT_BYTES, "outputs of %d bytes exceed the %d-byte dump limit" % (total, DUMP_LIMIT_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port (plain-C twin of the reference's weave loops + SciPy's cg), host cores
# ---------------------------------------------------------------------------------------------
def cpu_pcg_throughput(nt, iters, warmup=1, seed=0):
    """samples/s per PCG iteration of the oracle on a bounded sample of the same workload."""
    import importlib.util
    import scipy.sparse.linalg as spla
    import oracle
    from oracle import cloops
    # the workload generator is plain NumPy: load it by path so that the CPU arm never imports the
    # package (which maps the CUDA library) -- nothing of the product may be on the reference arm's path
    spec = importlib.util.spec_from_file_location("cm2_synthetic", os.path.join(ROOT, "cosmomap2_b200", "synthetic.py"))
    synthetic = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(synthetic)
    cloops.build()
    sc = synthetic.config_c2(nt=nt, seed=seed)
    pix = sc.pix.astype(np.int64)
    N = oracle.BlockLO(sc.ns, sc.weights)
    pts = oracle.ProcessTimeSamples(pix, sc.npix_full, pol=3, phi=sc.phi, w=N.diag)
    npix = pts.get_new_pixel[0]
    P = oracle.SparseLO(npix, sc.nt, pix, pol=3, angle_processed=pts)
    Mbd = oracle.BlockDiagonalPreconditionerLO(pts, npix, pol=3)
    A = P.T * N * P
    b = P.T * (N * sc.d)
    for _ in range(warmup):
        spla.cg(A, b, M=Mbd, rtol=1e-30, maxiter=1)
    t0 = time.perf_counter()
    for _ in range(iters):
        spla.cg(A, b, M=Mbd, rtol=1e-30, maxiter=1)        # one full iteration from a fresh residual
    dt = time.perf_counter() - t0
    return sc.nt * iters / dt, dt / iters, sc.nt, npix


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    v, t_iter, nt, npix = cpu_pcg_throughput(args.cpu_nt, max(args.steps, 1), warmup=max(args.warmup, 0))
    sample = ("oracle port (C twin of the weave loops, gcc -O3, + scipy.sparse.linalg.cg) on %d of the "
              "1e8 samples/GPU of configs[1] (same generator, same patch), %d timed iterations"
              % (nt, max(args.steps, 1)))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_iter, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[1]: raster scan, IQU nside=512, white noise, M_BD PCG (bounded sample)",
                   "nt_sample": nt, "npix_observed": int(npix), "pol": 3},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample,
                         "host_cores_available": os.cpu_count(),
                         "note": "the reference's loops are serial (weave.inline, no omp pragma): 1 thread"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
class ClockSampler(object):
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if ts < t0 or ts > t1:
                continue
            parts = [p.strip() for p in line.split(",")]
            try:
                sm.append(float(parts[0]))
                smax = float(parts[1])
            except Exception:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def run_sensitivity(nt=50000000):
    """Pointing-pattern sensitivity of the dominant kernel (the fused white A-matvec through the drop-in operators,
    which choose the scatter from the pointing): samples per pixel crossing 1..32, a scan tilted 30 degrees against
    the pixel rows, and the random pointing of the reference's tests (utilities/utilities_functions.py:111-122);
    IQU nside 512, 64 white-noise blocks, device-generated, CUDA events, inputs far larger than L2."""
    import gc
    import torch
    import cosmomap2_b200 as cm
    from cosmomap2_b200 import workloads, linearoperators as lo
    peak, _src = workloads._peak()
    nside, nx, ny, ndet, pol = 512, 1000, 500, 64, 3
    rows = []
    cases = [("spp=%g" % s, dict(spp=s)) for s in (1.0, 2.0, 4.0, 8.0, 32.0)]
    cases += [("tilt30 spp=8", dict(spp=8.0, tilt_deg=30.0)), ("random (pairs_gen)", None)]
    for name, kw in cases:
        if kw is None:
            pix, phi, g = workloads.random_pointing(nt, nside, nx, ny, seed=0)
            ntt, ns = nt, nt // ndet
        else:
            ntt, ns, pix, phi, _a, _b, g = workloads.make_scan(nt, nside, nx, ny, ndet, kw["spp"], seed=0, turnaround=0.0,
                                                               tilt_deg=kw.get("tilt_deg", 0.0))
        N = cm.BlockLO(ns, 0.5 + np.random.default_rng(0).random(ndet))
        pts = cm.ProcessTimeSamples(pix, 12 * nside ** 2, obspix=np.arange(12 * nside ** 2), pol=pol, phi=phi, w=N.diag)
        del phi
        npix = pts.get_new_pixel[0]
        P = cm.SparseLO(npix, ntt, pts._pix_dev, pol=pol, angle_processed=pts)
        A = P.T * N * P
        x = torch.randn(pol * npix, dtype=torch.float64, device="cuda", generator=g)
        A._apply(x)
        ms = workloads.time_device(lambda: A._apply(x), 20, warmup=3)
        fused = [f for f in A.planned() if isinstance(f, lo._FusedWhiteA)]
        alg = 20.0 * ntt + 48.0 * npix
        rows.append({"pattern": name, "nt": int(ntt), "mean_run_length": P.mean_run_length(),
                     "scatter": fused[0]._mode if fused else None, "kernel_ms": ms, "GBs": alg / ms / 1e6,
                     "frac": alg / ms / 1e6 / peak})
        del P, A, N, pts, pix, x
        gc.collect()
        torch.cuda.empty_cache()
    return {"kernel": "cm2_amatvec_white through P.T*N*P (scatter chosen from SparseLO.mean_run_length)",
            "algorithmic_bytes": "20 B/sample + 48 B/pixel for every pattern (the pixel-sorted path really reads 28 B/sample)",
            "patterns": rows}


def run_secondary(world, rank, out):
    """configs[2], configs[3] and configs[4] on this run's GPUs (cosmomap2_b200/workloads.py, the functions behind
    examples/solve_correlated.py and examples/solve_two_level.py): per-GPU shares of the named sizes, so that
    N = 8 runs them at exactly 1e9, 4e9 and 8e9 samples.  Results go into ``out`` as they complete."""
    import gc
    import torch
    from cosmomap2_b200 import workloads

    def run(key, fn, **kw):
        t0 = time.time()
        try:
            res = fn(**kw)
            res["wall_seconds_incl_setup"] = time.time() - t0
            out[key] = res
        except Exception as e:                      # noqa: BLE001 -- the headline line must still be printed
            out[key] = {"error": "%s: %s" % (type(e).__name__, e)}
        gc.collect()
        torch.cuda.empty_cache()

    # configs[2]: 1e9 samples / 64 detectors over 8 GPUs = 1.25e8 samples, 8 detectors per GPU
    run("configs[2]", workloads.correlated, nt=1.25e8, ndet=8, nband=4096, nside=512, nx=1000, ny=500, rtol=1e-6,
        maxiter=300, time_iters=10, symmetry=False, two_level_r=32)
    # configs[3]: 4e9 samples over 8 GPUs = 5e8 per GPU, nside 1024, r = 32
    run("configs[3]", workloads.two_level, nt=5e8, nside=1024, nx=1600, ny=800, ndet=64, r=32, coarse="scan", smooth=2,
        rtol=1e-8, maxiter=2000)
    # configs[4]: 8e9 samples in total when they fit (N >= 4: strong scaling), else 1e9 per GPU; nside 2048
    nt4 = 8e9 / world if world >= 4 else 1e9
    run("configs[4]", workloads.white, nt=nt4, nside=2048, nx=3200, ny=1600, ndet=64, steps=20)
    if "error" not in out["configs[4]"]:
        out["configs[4]"]["scaling"] = "strong (8e9 samples in total)" if world >= 4 else "1e9 samples per GPU (8e9 do not fit %d GPU)" % world


def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        claim_stdout()                                 # NCCL's version banner goes to stderr
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import cosmomap2_b200 as cm
    from cosmomap2_b200 import synthetic, _cabi, distributed
    from cosmomap2_b200.pcg import make_solver
    from cosmomap2_b200 import _device as dv

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs: this rank's detectors of configs[1] -----------------------------------------------
    pol = 3
    nt_rank = args.nt if args.scaling == "weak" else max(args.nt // world, 64 * 256)
    sc = synthetic.config_c2(nt=nt_rank, seed=rank)
    nt = sc.nt
    N = cm.BlockLO(sc.ns, sc.weights)
    pix = sc.pix                                     # int32 HEALPix ids, relabelled in place
    pts = cm.ProcessTimeSamples(pix, sc.npix_full, pol=pol, phi=sc.phi, w=N.diag, comm=(True if world > 1 else None))
    npix = pts.get_new_pixel[0]
    n = pol * npix
    P = cm.SparseLO(npix, nt, pix, pol=pol, angle_processed=pts)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
    A_local = P.T * N * P                              # planned as ONE fused kernel (cm2_amatvec_white)
    a_events = []

    class Timed(cm.lp.LinearOperator):                 # CUDA events around the local fused kernel only
        def __init__(self, op):
            self.op = op
            super(Timed, self).__init__(op.nargin, op.nargout, matvec=self._run, symmetric=True, device=True)
            self.record = False

        def _run(self, x):
            if not self.record:
                return self.op._apply(x)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            y = self.op._apply(x)
            e1.record()
            a_events.append((e0, e1))
            return y

    A_timed = Timed(A_local)
    A = distributed.AllReduceLO(A_timed) if world > 1 else A_timed
    d_dev = dv.to_dev_f64(sc.d)
    b = P.T._apply(N._apply(d_dev))
    if world > 1:
        distributed.all_reduce_sum_(b)
    del d_dev
    sc.d = None
    torch.cuda.synchronize()

    # ---- correctness gate (not timed): the solve converges, A x = b ---------------------------------
    res = []
    x_sol, info = cm.cg(A, b, M=Mbd, rtol=1e-10, maxiter=20, residuals=res)
    relres = float(torch.linalg.norm(b - A._apply(x_sol)) / torch.linalg.norm(b))
    check = {"cg_info": int(info), "cg_iterations": len(res) - 1 if info == 0 else len(res), "relres": relres}
    del x_sol

    # ---- device-resident timing -----------------------------------------------------------------------
    # N = 1: pcg.PCG (A apply + one cooperative kernel for the pixel-domain tail); N > 1: the pixel-sharded
    # solver (distributed.ShardedPCG: local TOD pass + ONE kernel fusing reduce-scatter, M_BD, CG vector work
    # and all-gather over NVLink peer memory), NCCL all-reduce + replicated tail if peer memory is unavailable
    solver = make_solver(A, Mbd, n)
    sharded = isinstance(solver, distributed.ShardedPCG)

    def one_step():
        solver.start(b)            # r <- b, x <- 0, z = M r, rho, ||r||^2 (device)
        solver.step_async()        # p, q = A p, alpha, x, r, z, rho, ||r||, exit test (device)
        solver.tick()              # the solve loop's one-iteration-late 128-byte read of the scalars

    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()
    if world > 1 and getattr(A, "_p2p", None) is not None:
        # the peer-memory exchange must never have timed out; if it did on any rank, every rank
        # falls back to NCCL for the measurement (and says so in `config.parallelism`)
        bad = (sharded and solver.failed()) or A._p2p.error() != 0
        if distributed.agree_failed(bad):
            sys.stderr.write("[bench] peer-memory exchange timed out on some rank: falling back to NCCL\n")
            A.disable_p2p("timeout during warm-up")
            solver = make_solver(A, Mbd, n)
            sharded = False
            for _ in range(3):
                one_step()
            barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if world > 1:
        # rank 0 has just spent a fork + exec on the clock sampler: without this barrier every other rank's first
        # timed step would wait for it inside the peer exchange (0.7 ms at N = 8: +0.03 ms per step over 20 steps)
        for _ in range(2):
            one_step()
        barrier()
    launches0 = _cabi.launch_count()
    A_timed.record = True
    t_wall0 = time.time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        one_step()
    ev1.record()
    barrier()
    A_timed.record = False
    launches = _cabi.launch_count() - launches0
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = world * nt * args.steps / (ms * 1e-3)
    t_a_ms = float(np.mean([e0.elapsed_time(e1) for e0, e1 in a_events]))
    assert bool(torch.isfinite(solver.x).all().item()), "PCG state is not finite"
    x_last = None
    if args.dump_outputs:
        # the last timed step's iterate, copied on the device now (the steps below overwrite the solver state) and
        # written to disk once the headline measurements are done.  ||r|| after the step is not dumped: M_BD A = I makes it
        # rounding noise that differs from run to run.
        x_last = solver.gather_x() if sharded else solver.x.clone()

    # keep the GPU under the same load for ~1.5 s so that nvidia-smi sees the clocks of this loop.  Every
    # rank runs the SAME number of extra steps (each one contains a peer exchange: a per-rank wall-clock
    # bound would leave unmatched exchanges behind), derived from the measured step time.
    n_extra = int(min(20000, max(20, 1.5e3 / max(ms_per_step, 1e-3))))
    for _ in range(n_extra):
        one_step()
    barrier()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    if clocks is not None:
        clocks["window"] = "timed loop + 1.5 s repeat of the same loop"

    # ---- end to end through the public API with HOST buffers: x, info = cm.cg(A, b_host, M=Mbd, maxiter=1)
    # per step: b (pinned host) -> HBM, one full PCG iteration (same step as above), x -> host
    b_host = dv.pinned_array(n)
    b_host[...] = dv.to_host(b)
    e2e_steps = max(1, min(args.e2e_steps, args.steps))
    gather = "shard" if sharded else "all"   # sharded: every rank moves only ITS pixel slice of b and x over PCIe
    for _ in range(4):                 # warm-up, results kept alive exactly as in the timed loop
        x_h, _info = cm.cg(A, b_host, M=Mbd, rtol=1e-30, maxiter=1, gather=gather)
    barrier()
    t0 = time.perf_counter()
    per = []
    for _ in range(e2e_steps):
        t00 = time.perf_counter()
        x_h, _info = cm.cg(A, b_host, M=Mbd, rtol=1e-30, maxiter=1, gather=gather)
        per.append(time.perf_counter() - t00)
    barrier()
    dt = time.perf_counter() - t0
    if os.environ.get("CM2_BENCH_DEBUG"):
        sys.stderr.write("e2e per-step ms: %s\n" % ["%.2f" % (1e3 * v) for v in per])
    tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_value = world * nt * e2e_steps / float(tt.item())
    assert np.all(np.isfinite(x_h))

    # the reference's own driver: SciPy's cg over the drop-in operators (host vectors both ways at
    # every A and M apply; SciPy's NumPy vector updates on the host)
    import scipy.sparse.linalg as spla
    spla.cg(A, b_host, M=Mbd, rtol=1e-30, maxiter=1)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        spla.cg(A, b_host, M=Mbd, rtol=1e-30, maxiter=1)
    barrier()
    dts = time.perf_counter() - t0
    tt = torch.tensor([dts], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_scipy = world * nt * e2e_steps / float(tt.item())

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        alg_bytes = 20.0 * nt + 48.0 * npix
        achieved = alg_bytes / (t_a_ms * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "amatvec_white_traffic.json")))["dram_bytes_per_launch"]
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[1]: synthetic raster scan, 1e8 samples/GPU, IQU nside=512, white noise "
                                   "(64 detector blocks), M_BD PCG on A=P^T N^-1 P",
                       "nt_per_gpu": nt, "npix_observed": int(npix), "pol": pol, "nside": 512,
                       "samples_per_pixel_crossing": sc.samples_per_pixel,
                       "step": "one PCG iteration from a fresh residual (A apply + M_BD apply + CG vector work + ||r|| readback)",
                       "l2": "inputs (2.0 GB TOD per pass) larger than L2 (126 MB); no flush needed",
                       "parallelism": (("tod sharded by detector x%d; per iteration one local k_amatvec_white + ONE kernel "
                                        "k_pcg_bd_sharded over NVLink peer memory (reduce-scatter of A p by peer loads, "
                                        "pixel-sharded M_BD + CG vector work, all-gather of p by peer stores; 3 doubles of "
                                        "scalars exchanged by flag-guarded peer stores); no NCCL call in the iteration" % world)
                                       if sharded else
                                       ("tod sharded by detector x%d, map all-reduce (%s), replicated pixel-domain tail"
                                        % (world, "own kernel over NVLink peer memory" if getattr(A, "_p2p", None) is not None
                                           else "NCCL"))) if world > 1 else "single GPU",
                       "check": check},
            "roofline": {"bound": "hbm", "kernel": "k_amatvec_white<3> (cm2_amatvec_white)", "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one committed `ncu --set full` capture of "
                                           "this kernel on this workload (profiles/amatvec_white_traffic.json), not measured in this run",
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                         "kernel_ms": t_a_ms, "frac_of_8TBs_spec": achieved / 8000.0,
                         "bracket": "CUDA events around the cm2_amatvec_white call on its stream, averaged over the timed steps: "
                                    "the kernel plus the cudaMemsetAsync of the 12 MB output map in front of it (3-4 us)"},
            "e2e": {"value": e2e_value, "unit": UNIT,
                    "h2d_bytes_per_step": 8 * n if (sharded or world == 1) else 8 * n * world,
                    "d2h_bytes_per_step": (8 * n if (sharded or world == 1) else 8 * n * world) + 128 * world,
                    "bytes_are": "job totals over all ranks" + ("; every rank moves only its 1/%d pixel slice of b and x" % world
                                                                 if sharded else ""),
                    "steps": e2e_steps,
                    "path": "x, info = cosmomap2_b200.cg(A, b_host, M=Mbd, maxiter=1%s): b from pinned host memory, one full "
                            "PCG iteration (the same step as `value`), x back to the host" % (', gather="shard"' if sharded else ""),
                    "scipy_driver": {"value": e2e_scipy, "unit": UNIT, "h2d_bytes_per_step": 2 * 8 * n,
                                     "d2h_bytes_per_step": 2 * 8 * n,
                                     "path": "scipy.sparse.linalg.cg(A, b_host, M=Mbd, maxiter=1) over the drop-in operators: "
                                             "host ndarrays cross PCIe at every A and M apply, SciPy's vector updates run on the host"}},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            v, t_iter, nt_cpu, _np = cpu_pcg_throughput(args.cpu_nt, args.cpu_iters)
            line["cpu_baseline"] = {
                "value": v, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": "oracle port (C twin of the reference's weave loops, gcc -O3, + scipy cg) on %d samples of the "
                          "same workload generator, %d iterations, %.2f s/iteration" % (nt_cpu, args.cpu_iters, t_iter),
                "host_cores_available": os.cpu_count()}
    else:
        line = None
    if x_last is not None and rank == 0:
        dump_outputs(args.dump_outputs, {"x": dv.to_host(x_last)})
    failed_primary = world > 1 and ((sharded and solver.failed()) or (getattr(A, "_p2p", None) is not None and A._p2p.error() != 0))
    if not args.no_secondary and not failed_primary:
        # the other configurations, on the same GPUs, after the headline measurement.  A watchdog prints the line
        # with whatever has completed if a part hangs (every rank exits then).
        secondary = {"note": "per-GPU shares of configs[2] (1e9 samples / 8), configs[3] (4e9 / 8) and configs[4]; device-generated "
                             "synthetic scans; solve times are wall clock around cosmomap2_b200.cg, kernel times CUDA events, max over ranks"}
        if line is not None:
            line["secondary"] = secondary

        def watchdog():
            if line is not None:
                secondary["error"] = "timeout after %.0f s: unfinished parts are missing" % args.secondary_timeout
                emit(line)
            os._exit(0)
        timer = threading.Timer(args.secondary_timeout, watchdog)
        timer.daemon = True
        timer.start()
        if world == 1:
            try:
                secondary["sensitivity"] = run_sensitivity()
            except Exception as e:                      # noqa: BLE001
                secondary["sensitivity"] = {"error": "%s: %s" % (type(e).__name__, e)}
            try:
                # configs[0], the reference's own CPU-runnable case, on the GPU and (the checker, on the host cores)
                # through the oracle: the one place besides cpu_baseline where bench.py runs oracle/
                import oracle
                from oracle import cloops
                from cosmomap2_b200 import workloads
                cloops.build()
                secondary["configs[0]"] = workloads.real_ces_script(cpu_oracle=oracle)
            except Exception as e:                      # noqa: BLE001
                secondary["configs[0]"] = {"error": "%s: %s" % (type(e).__name__, e)}
        run_secondary(world, rank, secondary)
        timer.cancel()
    if line is not None:
        emit(line)
    if world > 1:
        if sharded and solver.failed():
            raise RuntimeError("sharded PCG: a peer-flag wait timed out during the benchmark")
        A.check()
        A.close()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
