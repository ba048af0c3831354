"""
The configurations of BASELINE.json beyond configs[1] as callable workloads, shared by ``examples/`` (the
command-line drivers) and ``bench.py`` (the ``secondary`` block of the bench line):

    correlated()   configs[2]: A = P^T F N^-1 F P, banded-Toeplitz noise (4096 coefficients) + subscan
                   offset filter, M_BD PCG               (linearoperators.py:582-595, :129-168)
    two_level()    configs[3]: A = P^T F P, M_BD against M_2lvl (deflation space r = 32, coarse E solve),
                   nside 1024                            (src/test_M2_precond_onto_real_data.py:54-122)
    white()        configs[4]: the white-noise A-matvec and the full M_BD PCG iteration at nside 2048

Every function builds ONE rank's share on the device (the pointing is generated there: inputs only),
runs under torch.distributed when it is initialised (TOD sharded by detector, map-domain sums through
``distributed.AllReduceLO``) and returns a JSON-able dict.  Device times are CUDA events on the launching
stream, max over ranks.
"""
import time

import numpy as np
import torch
import torch.distributed as dist


def _world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def _max_over_ranks(v):
    t = torch.tensor([float(v)], dtype=torch.float64, device="cuda")
    if _world()[0] > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _barrier():
    torch.cuda.synchronize()
    if _world()[0] > 1:
        dist.barrier()
        torch.cuda.synchronize()


def time_device(fn, iters, warmup=3):
    """Mean device time of ``fn()`` in ms (CUDA events on the current stream, max over ranks)."""
    for _ in range(warmup):
        fn()
    _barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return _max_over_ranks(e0.elapsed_time(e1) / iters)


def make_scan(nt, nside, nx, ny, ndet, spp, seed, turnaround=0.05, tilt_deg=0.0):
    """Raster scan of ``ndet`` detectors over an nx x ny patch of a RING-ordered HEALPix map, generated on the
    device: constant-speed sweeps (``spp`` samples per pixel crossing) with flagged turnarounds (-1), a slow
    cross-scan drift over the detector timeline, per-detector focal-plane offsets, the reference's HWP ramp
    (utilities/utilities_functions.py:99-107) plus encoder jitter.  Returns
    (nt, ns, pix int32, phi fp64, sub_len, sub_start, generator).  ``tilt_deg`` turns the sweep direction against
    the pixel rows (iso-latitude rings) by that angle: the sweep then changes row every 1 / tan(tilt) pixels."""
    dev = torch.device("cuda")
    ns = nt // ndet
    nt = ns * ndet
    ring = 4 * nside
    sweep = int(nx * spp / (1.0 - turnaround))
    t = torch.arange(ns, dtype=torch.int64, device=dev)
    isw = t // sweep
    frac = (t - isw * sweep).to(torch.float64) / sweep
    u = torch.clamp((frac - turnaround / 2) / (1.0 - turnaround), 0.0, 1.0 - 1e-12)
    xpos = torch.where(isw % 2 == 0, u, 1.0 - 1e-12 - u) * nx
    inside = (frac >= turnaround / 2) & (frac < 1.0 - turnaround / 2)
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    pix = torch.empty(nt, dtype=torch.int32, device=dev)
    phi = torch.empty(nt, dtype=torch.float64, device=dev)
    for b in range(ndet):
        dx = (torch.rand(1, generator=g, device=dev).item() - 0.5) * 0.04 * nx
        dy = (torch.rand(1, generator=g, device=dev).item() - 0.5) * 0.1 * ny
        ix = torch.remainder(torch.floor(xpos + dx).to(torch.int64), nx)
        ypos = t.to(torch.float64) / ns * ny + dy
        if tilt_deg:
            ypos = ypos + float(np.tan(np.radians(tilt_deg))) * xpos
        iy = torch.remainder(torch.floor(ypos).to(torch.int64), ny)
        p = ((2 * nside - ny // 2 + iy) * ring + (ring // 2 - nx // 2 + ix)).to(torch.int32)
        pix[b * ns:(b + 1) * ns] = torch.where(inside, p, torch.full_like(p, -1))
        phi[b * ns:(b + 1) * ns] = 3.0 * torch.rand(1, generator=g, device=dev).item() + \
            2 * np.pi * 2.5 / 200. * t.to(torch.float64) + 1e-3 * torch.randn(ns, generator=g, device=dev, dtype=torch.float64)
    nsweeps = int(ns // sweep)
    s0 = int(np.ceil(turnaround / 2 * sweep))
    s1 = int(np.ceil((1 - turnaround / 2) * sweep))
    sub_start = np.arange(nsweeps, dtype=np.int64) * sweep + s0
    sub_len = np.full(nsweeps, s1 - s0, dtype=np.int64)
    return nt, ns, pix, phi, sub_len, sub_start, g


def random_pointing(nt, nside, nx, ny, seed):
    """The reference tests' pointing (utilities/utilities_functions.py:111-122 ``pairs_gen``: every sample an
    independent uniform pixel), over the same nx x ny patch, on the device."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    ring = 4 * nside
    ix = torch.randint(0, nx, (nt,), generator=g, device="cuda")
    iy = torch.randint(0, ny, (nt,), generator=g, device="cuda")
    pix = ((2 * nside - ny // 2 + iy) * ring + (ring // 2 - nx // 2 + ix)).to(torch.int32)
    phi = 3.0 * torch.rand(nt, generator=g, device="cuda", dtype=torch.float64)
    return pix, phi, g


def _peak():
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    try:
        return float(json.load(open(os.path.join(root, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s"


def _roofline(kernel, alg_bytes, ms, note=None):
    peak, src = _peak()
    ach = alg_bytes / (ms * 1e-3) / 1e9
    out = {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
           "frac_of_8TBs_spec": ach / 8000.0, "algorithmic_bytes_per_launch": float(alg_bytes), "kernel_ms": ms,
           "peak_source": src, "traffic": None}
    if note:
        out["note"] = note
    return out


def _solve(cm, A, b, M, rtol, maxiter):
    res = []
    _barrier()
    t0 = time.perf_counter()
    x, info = cm.cg(A, b, M=M, rtol=rtol, maxiter=maxiter, residuals=res)
    torch.cuda.synchronize()
    dt = _max_over_ranks(time.perf_counter() - t0)
    its = len(res) - 1 if info == 0 else len(res)
    rel = float(torch.linalg.norm(b - A._apply(x)) / torch.linalg.norm(b))
    return x, res, dict(info=int(info), iterations=its, seconds=dt, ms_per_iteration=1e3 * dt / max(its, 1),
                        true_relres=rel, rtol=rtol)


def _close(A):
    if _world()[0] > 1 and hasattr(A, "close"):
        A.close()


# -------------------------------------------------------------------------------------------------------
def real_ces_script(cpu_oracle=None, seed=0):
    """configs[0]: the reference's real-data script (src/test_BD_precond_onto_real_data.py:8-61) on the stand-in for
    its absent CES file (synthetic.config_c1: 4 detector pairs, 6.26e6 samples, IQU nside 128, flagged turnarounds):
    ProcessTimeSamples -> SparseLO -> BlockDiagonalPreconditionerLO -> A = P^T P -> cg(tol=1e-3, maxiter=10), host
    arrays in and out, timed as a whole.  ``cpu_oracle``: the oracle module (bench.py passes it; the product never
    imports it) to run the same script on the host cores for the comparison."""
    import scipy.sparse.linalg as spla
    import cosmomap2_b200 as cm
    from cosmomap2_b200 import synthetic
    sc = synthetic.config_c1(seed=seed)
    pol = 3

    def script(impl, solver):
        pix = sc.pix.astype(np.int64)
        t0 = time.perf_counter()
        pts = impl.ProcessTimeSamples(pix, sc.npix_full, pol=pol, phi=sc.phi)
        npix = pts.get_new_pixel[0]
        P = impl.SparseLO(npix, sc.nt, pix, pol=pol, angle_processed=pts)
        Mbd = impl.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
        A = P.T * P
        b = P.T * sc.d
        t1 = time.perf_counter()
        res = []
        x, info = solver(A, b, M=Mbd, rtol=1e-3, maxiter=10, callback=lambda xk: res.append(0))
        if impl is cm:
            torch.cuda.synchronize()
        t2 = time.perf_counter()
        return dict(npix=int(npix), x=np.asarray(x), info=int(info), iterations=len(res), setup_seconds=t1 - t0,
                    solve_seconds=t2 - t1)

    script(cm, cm.cg)                                   # first use: kernel load, allocator warm-up
    g = script(cm, cm.cg)
    out = {"config": "configs[0] stand-in: 4 detector pairs, %d samples, IQU nside 128, A = P^T P, cg(tol=1e-3, maxiter=10)" % sc.nt,
           "nt": int(sc.nt), "npix": g["npix"], "info": g["info"], "iterations": g["iterations"],
           "gpu_setup_seconds": g["setup_seconds"], "gpu_solve_seconds": g["solve_seconds"],
           "samples_per_s_per_pcg_iter": sc.nt * max(g["iterations"], 1) / g["solve_seconds"]}
    if cpu_oracle is not None:
        c = script(cpu_oracle, spla.cg)
        out.update({"cpu_oracle_setup_seconds": c["setup_seconds"], "cpu_oracle_solve_seconds": c["solve_seconds"],
                    "cpu_iterations": c["iterations"], "npix_equal": c["npix"] == g["npix"],
                    "x_rel_diff": float(np.max(np.abs(c["x"] - g["x"])) / np.max(np.abs(c["x"]))),
                    "speedup_whole_script": (c["setup_seconds"] + c["solve_seconds"]) / (g["setup_seconds"] + g["solve_seconds"])})
    return out


def correlated(nt=1.25e8, ndet=8, nband=4096, nside=512, nx=1000, ny=500, rtol=1e-6, maxiter=300, time_iters=20,
               symmetry=True, two_level_r=0):
    """configs[2], one rank's share: ``ndet`` detectors x nt/ndet samples, one symmetric banded Toeplitz block of
    ``nband`` coefficients per detector, subscan offset filter; M_BD built with the weights a_0 (the reference
    feeds ``N.diag`` to ProcessTimeSamples, src/test_BD_precond_onto_real_data.py:78-80)."""
    import cosmomap2_b200 as cm
    from cosmomap2_b200 import distributed, synthetic
    world, rank = _world()
    pol = 3
    nt, ns, pix, phi, sub_len, sub_start, g = make_scan(int(nt), nside, nx, ny, ndet, 8.0, seed=rank)
    npix_full = 12 * nside ** 2
    bands = synthetic.toeplitz_bands(ndet, nband, seed=100 + rank)
    N = cm.BlockLO(ns, bands, offdiag=True)
    Nw = cm.BlockLO(ns, [a[0] for a in bands])             # the diagonal of N^-1: the weights of M_BD
    pts = cm.ProcessTimeSamples(pix, npix_full, obspix=np.arange(npix_full), pol=pol, phi=phi, w=Nw.diag,
                                comm=(True if world > 1 else None))
    del phi
    npix = pts.get_new_pixel[0]
    n = pol * npix
    P = cm.SparseLO(npix, nt, pts._pix_dev, pol=pol, angle_processed=pts)
    F = cm.FilterLO(nt, [sub_len, sub_start], ns, ndet, pts._pix_dev)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
    A_local = P.T * F * N * F * P
    A = distributed.AllReduceLO(A_local) if world > 1 else A_local
    sky = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(99))
    d = P._apply(sky)
    d += 0.5 * torch.randn(nt, dtype=torch.float64, device="cuda", generator=g)
    b = P.T._apply(F._apply(N._apply(F._apply(d))))
    if world > 1:
        distributed.all_reduce_sum_(b)
    torch.cuda.synchronize()

    t0 = time.perf_counter()
    A._apply(b)                        # first use: run table of F P, plan, work buffers (set-up, not the solve)
    torch.cuda.synchronize()
    first_apply = time.perf_counter() - t0
    x, res, cg = _solve(cm, A, b, Mbd, rtol, maxiter)
    cg["first_A_apply_seconds_not_in_solve"] = first_apply
    cg["residual_first_last"] = [float(res[0]), float(res[-1])] if len(res) else None
    out = {"config": "configs[2]: Toeplitz noise (%d coefficients) + subscan offset filter, M_BD PCG" % nband,
           "world": world, "nt_total": nt * world, "nt_per_gpu": nt, "ndet_per_gpu": ndet, "npix": int(npix),
           "nside": nside, "nseg_per_gpu": F.nseg, "nband": nband,
           "plan": [type(f).__name__ for f in A_local.planned()], "cg": cg,
           "samples_per_s_per_pcg_iter": nt * world / (cg["seconds"] / max(cg["iterations"], 1))}
    if two_level_r:
        try:
            # beyond the named configuration (M_BD PCG): the same solve with M_2lvl on the scan coarse space -- the slow
            # modes of P^T F N F P are those of the offset filter, whatever N is
            _barrier()
            t0 = time.perf_counter()
            r2 = int(two_level_r)
            Zt = cm.scan_coarse_space(P, r2, ns, A=A, Mbd=Mbd, smooth=2)
            AZt = cm.coarse_products(A, Zt, pol)
            E = cm.CoarseLO(Zt.t(), AZt.t(), r2, apply="eig")
            Zd, AZd = cm.DeflationLO(Zt.t()), cm.DeflationLO(AZt.t())
            del Zt, AZt
            M2 = Mbd * (cm.lp.IdentityOperator(n) - AZd * E * Zd.T) + Zd * E * Zd.T
            M2._apply(b)
            torch.cuda.synchronize()
            build = _max_over_ranks(time.perf_counter() - t0)
            x2, _res2, cg2 = _solve(cm, A, b, M2, rtol, maxiter)
            cg2.update(r=r2, build_seconds=build)
            ax1, ax2 = A._apply(x), A._apply(x2)
            cg2["Ax_agreement"] = float(torch.linalg.norm(ax1 - ax2) / torch.linalg.norm(ax1))
            cg2["build_plus_solve_vs_M_BD_solve"] = (build + cg2["seconds"]) / cg["seconds"]
            out["M_2lvl_scan_space"] = cg2
            del M2, Zd, AZd, E, x2
        except Exception as e:                      # noqa: BLE001 -- the named configuration (M_BD) stands
            out["M_2lvl_scan_space"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if symmetry:
        # symmetry of the composed operator (F and N symmetric): <u, A v> = <v, A u>
        u = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(7))
        v = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
        Av, Au = A._apply(v), A._apply(u)
        uav, vau = float(torch.dot(u, Av)), float(torch.dot(v, Au))
        sym_scale = float(torch.linalg.norm(u) * torch.linalg.norm(Av))
        out["symmetry"] = {"u_Av": uav, "v_Au": vau, "rel": abs(uav - vau) / max(abs(uav), 1e-300),
                           "rel_to_norms": abs(uav - vau) / max(sym_scale, 1e-300)}
    # device time of the A apply alone and of its dominant kernel (the Toeplitz noise operator)
    a_ms = time_device(lambda: A._apply(x), time_iters)
    al_ms = time_device(lambda: A_local._apply(x), time_iters)
    n_ms = time_device(lambda: N._apply(d), time_iters)
    del d
    out.update({"A_apply_ms": a_ms, "A_local_apply_ms": al_ms, "A_apply_samples_per_s": nt * world / (a_ms * 1e-3),
                "roofline": _roofline("k_toeplitz_fft (cm2_noise_toeplitz_apply, %d coefficients)" % nband, 16.0 * nt, n_ms,
                                      "16 B/sample is the HBM floor the contract asks for; the kernel is bound by the fp64 and "
                                      "shared-memory pipes of its in-CTA FFT (ncu, profiles/r02_fft_ncu.txt: fp64 pipe 46 %, "
                                      "L1/shared-memory data pipe 57 % busy, DRAM 10 %; ~150 flop/sample instead of the 16 382 of "
                                      "the direct form; DESIGN sections 4, 4b)"),
                "roofline_A_apply": _roofline("A_local = P^T F N F P (%d kernels)" % len(A_local.planned()),
                                              20.0 * nt + 48.0 * npix, al_ms,
                                              "against the ideal-fusion 20 B/sample + 48 B/pixel of SURVEY 8(d)"),
                "hbm_GB": torch.cuda.max_memory_allocated() / 1e9})
    _close(A)
    return out


# -------------------------------------------------------------------------------------------------------
def two_level(nt=5e8, nside=1024, nx=1600, ny=800, ndet=64, r=32, coarse="scan", smooth=2, arnoldi=300, rtol=1e-8,
              maxiter=2000, shard_m2=False, poly_order=0, time_iters=10):
    """configs[3], one rank's share: offset-filtered map-making (P^T F P) x = P^T F d, first with M_BD, then with
    M_2lvl = M_BD (I - A Z E^-1 Z^T) + Z E^-1 Z^T (src/test_M2_precond_onto_real_data.py:109-112).  ``coarse``:
    'scan' = a-priori subdomain space from the scan order (deflationlib.scan_coarse_space), 'ritz' = the
    reference's recipe (run_krypy_arnoldi -> find_ritz_eigenvalues, :54-100)."""
    import cosmomap2_b200 as cm
    from cosmomap2_b200 import distributed, _device as dv
    world, rank = _world()
    pol = 3
    nt, ns, pix, phi, sub_len, sub_start, g = make_scan(int(nt), nside, nx, ny, ndet, 8.0, seed=rank)
    npix_full = 12 * nside ** 2
    pts = cm.ProcessTimeSamples(pix, npix_full, obspix=np.arange(npix_full), pol=pol, phi=phi,
                                comm=(True if world > 1 else None))
    del phi
    npix = pts.get_new_pixel[0]
    n = pol * npix
    P = cm.SparseLO(npix, nt, pts._pix_dev, pol=pol, angle_processed=pts)
    F = cm.FilterLO(nt, [sub_len, sub_start], ns, ndet, pts._pix_dev, poly_order=poly_order)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
    A_local = P.T * F * P
    A = distributed.AllReduceLO(A_local) if world > 1 else A_local
    # data: a random sky (same on every rank) seen through P, plus white noise
    sky = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(99))
    d = P._apply(sky)
    d += 0.5 * torch.randn(nt, dtype=torch.float64, device="cuda", generator=g)
    b = P.T._apply(F._apply(d))
    if world > 1:
        distributed.all_reduce_sum_(b)
    del d
    torch.cuda.synchronize()

    out = {"config": "configs[3]: A = P^T F P (subscan filter order %d), M_BD vs M_2lvl (r = %d, coarse space '%s')"
                     % (poly_order, r, coarse),
           "world": world, "nt_total": nt * world, "nt_per_gpu": nt, "npix": int(npix), "nside": nside,
           "nseg_per_gpu": F.nseg, "poly_order": poly_order, "shard_m2": bool(shard_m2 and world > 1)}
    t0 = time.perf_counter()
    A._apply(b)                        # first use: run table of P^T F P, plan, work buffers (set-up, not the solve)
    torch.cuda.synchronize()
    out["first_A_apply_seconds_not_in_solve"] = time.perf_counter() - t0
    x_bd, _res, out["M_BD"] = _solve(cm, A, b, Mbd, rtol, maxiter)

    # ---- deflation space ---------------------------------------------------------------------------
    _barrier()
    t0 = time.perf_counter()
    if coarse == "scan":
        Zt = cm.scan_coarse_space(P, r, ns, A=A, Mbd=Mbd, smooth=smooth)          # (r, n), rows = columns of Z
        m, theta, thr = 0, np.zeros(1), 0.0
    else:
        V, H, m = cm.run_krypy_arnoldi(A, torch.ones(n, dtype=torch.float64, device="cuda"), Mbd, 1e-5,
                                       maxiter=arnoldi, ortho="dmgs")
        theta = np.sort(np.linalg.eigvalsh(H[:H.shape[1], :]))
        r = min(r, len(theta) - 1)
        thr = 0.5 * (theta[r - 1] + theta[r])
        Z, r, _th = cm.find_ritz_eigenvalues(H, V, threshold=thr, eigenvalues=True)
        Zt = Z.t().contiguous()
        del V, Z
    AZt = cm.coarse_products(A, Zt, pol) if coarse == "scan" else torch.stack([A._apply(Zt[i]) for i in range(r)])
    E = cm.CoarseLO(Zt.t(), AZt.t(), r, apply="eig")
    Zd, AZd = cm.DeflationLO(Zt.t()), cm.DeflationLO(AZt.t())
    del Zt, AZt
    if shard_m2 and world > 1:
        M2 = distributed.ShardedTwoLevelPreconditionerLO(Mbd, Zd, AZd, E)
    else:
        M2 = Mbd * (cm.lp.IdentityOperator(n) - AZd * E * Zd.T) + Zd * E * Zd.T  # fused at first use
    M2._apply(b)                      # first use (fusion, work buffers, kernel load) belongs to the build
    torch.cuda.synchronize()
    out["deflation"] = dict(kind=coarse, arnoldi_steps=int(m), r=int(r), ritz_min=float(theta[0]), ritz_cut=float(thr),
                            ritz_max=float(theta[-1]), discarded_E_modes=int(getattr(E, "ndiscarded", 0)),
                            build_seconds=_max_over_ranks(time.perf_counter() - t0))
    x_m2, _res, out["M_2lvl"] = _solve(cm, A, b, M2, rtol, maxiter)
    out["iteration_ratio"] = out["M_2lvl"]["iterations"] / max(out["M_BD"]["iterations"], 1)
    out["build_plus_solve_vs_M_BD_solve"] = (out["deflation"]["build_seconds"] + out["M_2lvl"]["seconds"]) / out["M_BD"]["seconds"]
    # the two solutions agree where A sees them (P^T F P has the per-subscan-offset null space)
    ax1, ax2 = A._apply(x_bd), A._apply(x_m2)
    out["Ax_agreement"] = float(torch.linalg.norm(ax1 - ax2) / torch.linalg.norm(ax1))
    for k in ("M_BD", "M_2lvl"):
        out[k]["samples_per_s_per_pcg_iter"] = nt * world / (out[k]["ms_per_iteration"] * 1e-3)
    al_ms = time_device(lambda: A_local._apply(x_bd), time_iters)
    m2_ms = time_device(lambda: M2._apply(x_bd), time_iters)
    out["A_local_apply_ms"] = al_ms
    out["M_2lvl_apply_ms"] = m2_ms
    out["roofline"] = _roofline("k_seg_mean + k_amatvec_filter_mu (P^T F P, cm2_amatvec_filter_mu)" if poly_order == 0
                                else "P^T F_K P (Legendre order %d)" % poly_order, 20.0 * nt + 48.0 * npix, al_ms,
                                note=("DRAM traffic of the pair measured by ncu at 1e8 samples, 8 samples per pixel crossing "
                                      "(profiles/r02_filter_mu_ncu.txt): 2.41 GB against 2.024 GB algorithmic -- k_amatvec_filter_mu "
                                      "reads 1.00x its 20 B/sample, the rest is the run table of k_seg_mean (28 B per run); "
                                      "not measured at this size, hence traffic = null") if poly_order == 0 else None)
    out["hbm_GB"] = torch.cuda.max_memory_allocated() / 1e9
    _close(A)
    return out


# -------------------------------------------------------------------------------------------------------
def white(nt=1e9, nside=2048, nx=3200, ny=1600, ndet=64, steps=30):
    """configs[4], one rank's share: white noise, nside 2048 patch; device time of the fused A-matvec and of one
    full M_BD PCG iteration from a fresh residual (the step bench.py times on configs[1])."""
    import cosmomap2_b200 as cm
    from cosmomap2_b200 import distributed
    from cosmomap2_b200.pcg import make_solver
    world, rank = _world()
    pol = 3
    nt, ns, pix, phi, _sl, _ss, g = make_scan(int(nt), nside, nx, ny, ndet, 8.0, seed=rank, turnaround=0.0)
    npix_full = 12 * nside ** 2
    w = 0.5 + torch.rand(ndet, generator=g, device="cuda", dtype=torch.float64).cpu().numpy()
    N = cm.BlockLO(ns, w)
    pts = cm.ProcessTimeSamples(pix, npix_full, obspix=np.arange(npix_full), pol=pol, phi=phi, w=N.diag,
                                comm=(True if world > 1 else None))
    del phi
    npix = pts.get_new_pixel[0]
    n = pol * npix
    P = cm.SparseLO(npix, nt, pts._pix_dev, pol=pol, angle_processed=pts)
    Mbd = cm.BlockDiagonalPreconditionerLO(pts, npix, pol=pol)
    A_local = P.T * N * P
    A = distributed.AllReduceLO(A_local) if world > 1 else A_local
    b = torch.randn(n, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    b = A._apply(b)
    x, info = cm.cg(A, b, M=Mbd, rtol=1e-10, maxiter=20)
    relres = float(torch.linalg.norm(b - A._apply(x)) / torch.linalg.norm(b))
    solver = make_solver(A, Mbd, n)

    def one_step():
        solver.start(b)
        solver.step_async()
        solver.tick()
    it_ms = time_device(one_step, steps)
    al_ms = time_device(lambda: A_local._apply(x), steps)
    from cosmomap2_b200 import linearoperators as lo
    fused = [f for f in A_local.planned() if isinstance(f, lo._FusedWhiteA)]
    tod_bytes = fused[0].tod_bytes() if fused else 20.0 * nt     # 17 B/sample + escape lanes with the packed pixel stream
    out = {"config": "configs[4]: white noise, IQU nside=%d, M_BD PCG" % nside, "world": world, "nt_total": nt * world,
           "nt_per_gpu": nt, "npix": int(npix), "nside": nside, "cg_info": int(info), "relres": relres,
           "ms_per_pcg_iteration": it_ms, "samples_per_s_per_pcg_iter": nt * world / (it_ms * 1e-3),
           "A_local_apply_ms": al_ms,
           "roofline": _roofline("k_amatvec_white<3> (cm2_amatvec_white)", tod_bytes + 48.0 * npix, al_ms),
           "solver": type(solver).__name__, "hbm_GB": torch.cuda.max_memory_allocated() / 1e9}
    _close(A)
    return out
