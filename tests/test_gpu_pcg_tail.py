"""GPU: the coalesced M_BD PCG tail (tiled k_bd_reset / k_bd_iter, vecops.cu) against the three-kernel
tail (cm2_pcg_bd_update + cm2_pcg_bd_update_p) and against the one-thread-per-pixel kernels, over 12
iterations of the same seeded system.  The tiled kernels sum p.q, r.z and |r|^2 in another order, so
the iterates agree to rounding (1e-12 relative), not bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ITERS = 12


@pytest.fixture(scope="module")
def dv():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import cosmomap2_b200  # noqa: F401
    from cosmomap2_b200 import _device
    return _device


def _system(npix, pol, seed, b_zero=False):
    """SPD per-pixel inverse blocks (upper triangles), A = diag(c) + (shift by one pixel, both ways) / 4, b."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = pol * npix
    inv = torch.zeros(npix, 6, dtype=torch.float64, device="cuda")
    inv[:, [0, 3, 5]] = 0.5 + 0.5 * torch.rand(npix, 3, dtype=torch.float64, device="cuda", generator=g)
    inv[:, [1, 2, 4]] = 0.1 * (torch.rand(npix, 3, dtype=torch.float64, device="cuda", generator=g) - 0.5)
    c = 1.5 + torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    b = torch.zeros(n, dtype=torch.float64, device="cuda") if b_zero else \
        torch.randn(n, dtype=torch.float64, device="cuda", generator=g)

    def apply_a(v):
        return c * v + 0.25 * (torch.roll(v, pol) + torch.roll(v, -pol))
    return inv.reshape(-1).contiguous(), apply_a, b


def _solve(dv, npix, pol, path, seed=3, b_zero=False, iters=ITERS):
    """path: 'auto' (the library's choice), 'strided' (one thread per pixel at every npix) or 'three'
    (the three-kernel tail).  Returns x, r, p, the scalars and the ||r||^2 history."""
    import torch
    inv, apply_a, b = _system(npix, pol, seed, b_zero)
    n = pol * npix
    x, r, p, z = (torch.full((n,), np.nan, dtype=torch.float64, device="cuda") for _ in range(4))
    scal = dv.zeros_f64(16)
    st = dv.stream()
    old = dv.call("cm2_pcg_bd_tail_strided", 1 if path != "auto" else 0)
    try:
        dv.call("cm2_pcg_bd_reset", dv.ptr(inv), npix, pol, dv.ptr(r), dv.ptr(z), dv.ptr(scal), 0.0, 0.0, dv.ptr(b),
                dv.ptr(x), dv.ptr(p), st)
        hist = [scal[3].item()]
        for _ in range(iters):
            q = apply_a(p)
            if path == "three":
                dv.call("cm2_pcg_bd_update", dv.ptr(inv), npix, pol, dv.ptr(p), dv.ptr(q), dv.ptr(x), dv.ptr(r), dv.ptr(z),
                        dv.ptr(scal), st)
                dv.call("cm2_pcg_bd_update_p", dv.ptr(z), dv.ptr(p), n, dv.ptr(scal), st)
            else:
                dv.call("cm2_pcg_bd_iter", dv.ptr(inv), npix, pol, dv.ptr(p), dv.ptr(q), dv.ptr(x), dv.ptr(r), dv.ptr(z),
                        dv.ptr(scal), st)
            hist.append(scal[3].item())
    finally:
        dv.call("cm2_pcg_bd_tail_strided", old)
    torch.cuda.synchronize()
    return {"x": x.cpu().numpy(), "r": r.cpu().numpy(), "p": p.cpu().numpy(), "scal": scal.cpu().numpy(),
            "hist": np.array(hist), "bnorm": float(torch.linalg.norm(b))}


def _close(a, b, what):
    scale = max(np.max(np.abs(b)), 1e-300)
    err = np.max(np.abs(a - b)) / scale
    assert np.all(np.isfinite(a)), what
    assert err <= 1e-12, "%s: max|d| / max|ref| = %.3e" % (what, err)


def _compare(new, ref):
    for k in ("x", "r", "p"):
        _close(new[k], ref[k], k)
    bn2 = ref["bnorm"] ** 2
    assert np.max(np.abs(new["hist"] - ref["hist"])) <= 1e-12 * bn2, "||r||^2 history"
    assert new["scal"][8] == ref["scal"][8] == ITERS
    assert new["scal"][7] == ref["scal"][7]


@pytest.mark.parametrize("pol", [1, 2, 3])
@pytest.mark.parametrize("npix", [37, 1037, 100003])
def test_tiled_tail_equals_three_kernel_tail(dv, pol, npix):
    """npix smaller than one warp tile and than the grid, not a multiple of the tile, and a grid-filling size."""
    _compare(_solve(dv, npix, pol, "auto"), _solve(dv, npix, pol, "three"))


@pytest.mark.parametrize("pol", [1, 3])
def test_both_sides_of_the_on_chip_bound(dv, pol):
    """At the bound the tiled kernel runs; one pixel above it cm2_pcg_bd_iter is the one-thread-per-pixel kernel."""
    bound = dv.call("cm2_pcg_bd_iter_max_npix", pol)
    assert bound >= 64
    for npix in (bound, bound + 1):
        new = _solve(dv, npix, pol, "auto", iters=4)
        ref = _solve(dv, npix, pol, "three", iters=4)
        for k in ("x", "r", "p"):
            _close(new[k], ref[k], "%s at npix = bound%s" % (k, "" if npix == bound else " + 1"))


def test_partial_last_tile_with_several_tiles_per_warp(dv):
    """Just below the bound every warp holds several tiles and the last tile is partial."""
    bound = dv.call("cm2_pcg_bd_iter_max_npix", 2)
    npix = bound - 37
    new = _solve(dv, npix, 2, "auto", iters=4)
    ref = _solve(dv, npix, 2, "three", iters=4)
    for k in ("x", "r", "p"):
        _close(new[k], ref[k], k)


@pytest.mark.parametrize("pol", [1, 3])
def test_misaligned_vectors_take_the_strided_kernels(dv, pol):
    """Vectors that start 8 bytes past a 16-byte boundary: the start and the iteration fall back to the one-thread-
    per-pixel kernels and give what aligned vectors give."""
    import torch
    npix = 1037
    n = pol * npix
    inv, apply_a, b = _system(npix, pol, 7)
    out = {}
    for off in (0, 1):
        bufs = [torch.zeros(n + 2, dtype=torch.float64, device="cuda") for _ in range(5)]
        x, r, p, z, bb = (t[off:off + n] for t in bufs)
        bb.copy_(b)
        scal = dv.zeros_f64(16)
        st = dv.stream()
        dv.call("cm2_pcg_bd_reset", dv.ptr(inv), npix, pol, dv.ptr(r), dv.ptr(z), dv.ptr(scal), 0.0, 0.0, dv.ptr(bb),
                dv.ptr(x), dv.ptr(p), st)
        for _ in range(4):
            q = apply_a(p)
            dv.call("cm2_pcg_bd_iter", dv.ptr(inv), npix, pol, dv.ptr(p), dv.ptr(q), dv.ptr(x), dv.ptr(r), dv.ptr(z),
                    dv.ptr(scal), st)
        torch.cuda.synchronize()
        assert scal[8].item() == 4
        out[off] = [v.cpu().numpy() for v in (x, r, p)]
    for name, a, c in zip("xrp", out[1], out[0]):
        _close(a, c, name)


def test_max_npix_covers_the_flagship_size(dv):
    """configs[1] (5e5 IQU pixels on one GPU) runs the on-chip kernel on a B200."""
    import torch
    if torch.cuda.get_device_properties(0).multi_processor_count < 148:
        pytest.skip("not a B200-sized device")
    assert dv.call("cm2_pcg_bd_iter_max_npix", 3) >= 500000


@pytest.mark.parametrize("pol", [1, 3])
def test_zero_rhs_start(dv, pol):
    """b = 0: x = r = p0 = 0 and the done flag up, as the one-thread-per-pixel start; later launches are no-ops."""
    npix = 1037
    new = _solve(dv, npix, pol, "auto", b_zero=True, iters=2)
    old = _solve(dv, npix, pol, "strided", b_zero=True, iters=2)
    for k in ("x", "r", "p"):
        assert np.array_equal(new[k], np.zeros(pol * npix)), k
    assert np.array_equal(new["scal"], old["scal"])
    assert new["scal"][7] == 1.0 and new["scal"][8] == 0.0


@pytest.mark.parametrize("path", ["auto", "strided"])
@pytest.mark.parametrize("pol", [2, 3])
def test_launch_after_done_changes_nothing(dv, pol, path):
    import torch
    npix = 5000
    inv, apply_a, b = _system(npix, pol, 5)
    n = pol * npix
    x, r, p, z = (torch.empty(n, dtype=torch.float64, device="cuda") for _ in range(4))
    scal = dv.zeros_f64(16)
    st = dv.stream()
    old = dv.call("cm2_pcg_bd_tail_strided", 1 if path == "strided" else 0)
    try:
        dv.call("cm2_pcg_bd_reset", dv.ptr(inv), npix, pol, dv.ptr(r), dv.ptr(z), dv.ptr(scal), 0.0, 0.0, dv.ptr(b),
                dv.ptr(x), dv.ptr(p), st)
        for _ in range(3):
            q = apply_a(p)
            dv.call("cm2_pcg_bd_iter", dv.ptr(inv), npix, pol, dv.ptr(p), dv.ptr(q), dv.ptr(x), dv.ptr(r), dv.ptr(z),
                    dv.ptr(scal), st)
        scal[7] = 1.0
        before = [v.clone() for v in (x, r, p, scal)]
        q = apply_a(p)
        dv.call("cm2_pcg_bd_iter", dv.ptr(inv), npix, pol, dv.ptr(p), dv.ptr(q), dv.ptr(x), dv.ptr(r), dv.ptr(z),
                dv.ptr(scal), st)
        torch.cuda.synchronize()
    finally:
        dv.call("cm2_pcg_bd_tail_strided", old)
    for name, v0, v1 in zip(("x", "r", "p", "scal"), before, (x, r, p, scal)):
        assert torch.equal(v0, v1), name
