"""The packed pixel stream of the fused white A-matvec (cm2_pack_pointing): it decodes to the int32 pointing bit
for bit, it escapes exactly the lanes the two-base format cannot hold, and the A-matvec over it gives the result of
the A-matvec over the int32 ids."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cm():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import cosmomap2_b200
    return cosmomap2_b200


def decode(words, pix):
    """The pixels of the packed stream `words` by the format rules (include/cosmomap2_b200.h); escape lanes from pix."""
    nt = pix.size
    w = words.view(np.uint64)
    assert w.size == (nt + 7) // 8
    lo = (w & np.uint64(0xffffffff)).astype(np.uint32).view(np.int32).astype(np.int64)
    assert np.all(lo >= -2)
    delta = ((w >> np.uint64(32)) & np.uint64(0xffff)).astype(np.uint16).view(np.int16).astype(np.int64)
    codes = (w >> np.uint64(48)).astype(np.int64)
    code = (codes[:, None] >> (2 * np.arange(8))) & 3
    b0 = lo[:, None]
    out = np.where(code & 2, b0 + delta[:, None], b0) + (code & 1)
    out[lo == -1] = -1
    esc = lo == -2
    padded = np.full(w.size * 8, -7, dtype=np.int64)
    padded[:nt] = pix
    out[esc] = padded.reshape(-1, 8)[esc]
    return out.ravel()[:nt], int(esc.sum())


def numpy_escapes(pix):
    """Lanes of 8 samples that the two-base format cannot hold, plus a last lane of fewer than 8 samples."""
    nt = pix.size
    q = pix[:nt // 8 * 8].reshape(-1, 8).astype(np.int64)
    big = np.iinfo(np.int64).max
    b0 = q.min(axis=1, initial=big)[:, None]
    b1 = np.where(q - b0 > 1, q, big).min(axis=1, initial=big)[:, None]
    b1 = np.where(b1 == big, b0, b1)
    fits = (((q - b0) <= 1) | ((q - b1) <= 1)).all(axis=1) & ((b1 - b0)[:, 0] <= 32767)
    all_flagged = (q == -1).all(axis=1)
    esc = ~all_flagged & ((q < 0).any(axis=1) | ~fits)
    return int(esc.sum()) + int(nt % 8 != 0)


def pack(pix):
    import torch
    from cosmomap2_b200 import _device as dv
    nt = pix.size
    pd = torch.from_numpy(np.ascontiguousarray(pix, dtype=np.int32)).cuda()
    packed = torch.full((max((nt + 7) // 8, 1),), 0x5a5a5a5a, dtype=torch.int64, device="cuda")
    nesc = torch.full((1,), -5, dtype=torch.int64, device="cuda")
    dv.call("cm2_pack_pointing", dv.ptr(pd) if nt else None, nt, dv.ptr(packed) if nt else None, dv.ptr(nesc), dv.stream())
    torch.cuda.synchronize()
    return packed.cpu().numpy()[:(nt + 7) // 8], int(nesc.item())


def compact(pix):
    """Observed pixels relabelled 0..npix-1 in id order (as ProcessTimeSamples does), flagged samples kept at -1."""
    out = np.full(pix.size, -1, dtype=np.int32)
    good = pix >= 0
    out[good] = np.unique(pix[good], return_inverse=True)[1]
    return out


def _raster(nt, **kw):
    from cosmomap2_b200 import synthetic
    return synthetic.raster_scan(nt, nside=512, ndet=kw.pop("ndet", 64), nx=1000, ny=500, samples_per_pixel=8.0,
                                 seed=kw.pop("seed", 0), with_data=False, **kw)


def _case(name):
    rng = np.random.default_rng(17)
    if name == "raster":                     # configs[1] at small nt
        return compact(_raster(64 * 4096).pix)
    if name == "odd_nt":                     # nt not a multiple of 8 or of 256
        return compact(_raster(64 * 4099 + 5).pix)
    if name == "flags":                      # flagged turnarounds and isolated flags
        pix = _raster(16 * 8000, ndet=16, flag_turnarounds=True).pix.copy()
        pix[rng.random(pix.size) < 0.003] = -1
        return compact(pix)
    if name == "detector_blocks":            # 1001 samples per detector: lanes straddle the block boundaries
        from cosmomap2_b200 import synthetic
        return compact(synthetic.raster_scan(40 * 1001, nside=64, ndet=40, nx=90, ny=5, seed=5, with_data=False).pix)
    if name == "row_jump":                   # deltas of 32767 fit the int16 field, 32768 and more escape
        lanes = [[5, 5, 6, 6, 5 + d, 5 + d, 6 + d, 6 + d] for d in (2, 1000, 32767, 32768, 40000, 1 << 30)]
        lanes += [[7 + d, 7 + d, 8 + d, 7, 7, 8, 8 + d, 8] for d in (32767, 32768)]
        return np.array(lanes * 40, dtype=np.int32).ravel()
    if name == "descending":                 # ids fall along time: b0 is a later sample of the lane; backward row jumps
        r = np.arange(40 * 1024) // 3
        return (10 ** 6 - (r // 97) * 300 - r % 97).astype(np.int32)
    if name == "code3_edges":                # delta 2 and 32766 / 32767 with code 3 (b1 + 1), and 32768 (escape)
        lanes = [[0, 0, 1, 1, 2, 2, 3, 3], [0, 32766, 32767, 0, 1, 32767, 1, 0],
                 [32767, 32768, 0, 1, 0, 32768, 1, 32767], [32767, 32767, 32766, 0, 0, 1, 32766, 1],
                 [0, 1, 32768, 32769, 0, 1, 32768, 32769]]
        return (np.array(lanes * 40, dtype=np.int32) + 100).ravel()
    if name == "flagged_by_escapes":         # all-flagged lanes next to escape lanes (mixed flags, three clusters)
        lanes = [[-1] * 8, [4, -1, 4, 4, 5, -1, 5, 4], [-1] * 8, [0, 5, 10, 0, 5, 10, 0, 0], [-1] * 8, [7] * 8]
        order = np.random.default_rng(5).integers(0, len(lanes), 4000)
        return np.array(lanes, dtype=np.int32)[order].ravel()
    if name == "random":                     # mostly escape lanes
        return rng.integers(0, 3 * 10 ** 6, 50021).astype(np.int32)
    if name == "short":
        return np.array([3, 3, 4, -1, 9], dtype=np.int32)
    if name == "empty":
        return np.zeros(0, dtype=np.int32)
    raise KeyError(name)


@pytest.mark.parametrize("case", ["raster", "odd_nt", "flags", "detector_blocks", "row_jump", "descending", "code3_edges",
                                  "flagged_by_escapes", "random", "short", "empty"])
def test_pack_round_trip(cm, case):
    pix = _case(case)
    words, nesc = pack(pix)
    dec, nesc_words = decode(words, pix)
    assert np.array_equal(dec, pix.astype(np.int64))
    assert nesc == nesc_words == numpy_escapes(pix)
    if case == "row_jump":
        lo = (words & 0xffffffff).astype(np.uint32).view(np.int32)
        assert list(lo[:8]) == [5, 5, 5, -2, -2, -2, 7, -2]
    if case == "raster":
        assert nesc < 1e-3 * words.size
    if case in ("descending", "code3_edges"):
        lo = (words & 0xffffffff).astype(np.uint32).view(np.int32)
        delta = ((words >> 32) & 0xffff).astype(np.uint16).view(np.int16)
        if case == "descending":
            assert np.all(np.diff(lo[lo >= 0]) <= 0) and np.count_nonzero(lo >= 0) > 0.99 * lo.size
        else:
            assert list(lo[:5]) == [100, 100, 100, 100, -2] and list(delta[:4]) == [2, 32766, 32767, 32766]
    if case == "random":
        assert nesc > 0.9 * words.size


def _operator(cm, sc, pol):
    pix = compact(sc.pix).astype(np.int64)
    N = cm.BlockLO(sc.ns, sc.weights)
    pts = cm.ProcessTimeSamples(pix, int(pix.max()) + 1, pol=pol, phi=sc.phi, w=N.diag)
    npix = pts.get_new_pixel[0]
    P = cm.SparseLO(npix, sc.nt, pix, pol=pol, angle_processed=pts)
    return P, N, npix


@pytest.mark.parametrize("pol", [1, 2, 3])
@pytest.mark.parametrize("interleaved", [False, True])
def test_packed_amatvec_matches_int32(cm, pol, interleaved):
    """cm2_amatvec_white over the packed stream vs over the int32 ids: the same sums up to the order of the fp64
    atomics, with flags, noise blocks of 2001 samples (not a multiple of 8) and nt % 8 != 0."""
    import torch
    from cosmomap2_b200 import _device as dv
    from cosmomap2_b200 import synthetic
    sc = synthetic.raster_scan(47 * 2001, nside=256, ndet=47, nx=300, ny=8, samples_per_pixel=8.0, seed=5,
                               flag_turnarounds=True, with_data=False)
    sc.pix[np.random.default_rng(3).random(sc.nt) < 0.003] = -1
    P, N, npix = _operator(cm, sc, pol)
    pixh = dv.to_host(P._pix_dev).astype(np.int32)
    packed = torch.empty((P.nrows + 7) // 8, dtype=torch.int64, device="cuda")
    nesc = torch.empty(1, dtype=torch.int64, device="cuda")
    dv.call("cm2_pack_pointing", dv.ptr(P._pix_dev), P.nrows, dv.ptr(packed), dv.ptr(nesc), dv.stream())
    assert int(nesc.item()) == numpy_escapes(pixh)
    x = torch.from_numpy(np.random.default_rng(4).standard_normal(pol * npix)).cuda()
    nb, bs, startp = N._blk.args()
    ys = []
    for pk in (None, packed):
        y = torch.empty(pol * npix, dtype=torch.float64, device="cuda")
        dv.call("cm2_amatvec_white", dv.ptr(P._pix_dev), dv.ptr(pk), dv.ptr(P._cos_dev), dv.ptr(P._sin_dev), P.nrows,
                pol, dv.ptr(N.weights_dev()), nb, bs, startp, dv.ptr(x), dv.ptr(y), npix, sc.ndet if interleaved else 1,
                dv.stream())
        ys.append(y.cpu().numpy())
    ref = ys[0]
    assert np.max(np.abs(ref)) > 0
    assert np.max(np.abs(ys[1] - ref)) <= 1e-14 * np.max(np.abs(ref))


@pytest.mark.parametrize("spp, mode", [(8.0, "registers"), (4.0, "staged"), (1.0, "sorted")])
def test_packed_stream_selection(cm, spp, mode, monkeypatch):
    """The register scatter plans the packed stream at first use; the staged and pixel-sorted scatters read int32."""
    from cosmomap2_b200 import _device as dv
    from cosmomap2_b200 import linearoperators as lo
    from cosmomap2_b200 import synthetic
    monkeypatch.setattr(lo, "WHITE_STAGE_MIN_CONTIGUITY", 0.5)
    sc = synthetic.raster_scan(6 * 40003, nside=64, ndet=6, nx=90, ny=50, samples_per_pixel=spp, seed=7,
                               with_data=False)
    P, N, npix = _operator(cm, sc, 3)
    A = P.T * N * P
    A * np.ones(3 * npix)
    fused = [f for f in A.planned() if isinstance(f, lo._FusedWhiteA)]
    assert len(fused) == 1 and fused[0]._mode == mode
    if mode == "registers":
        assert fused[0]._packed is not None
        assert fused[0].nescape == numpy_escapes(dv.to_host(P._pix_dev))
        assert fused[0].tod_bytes() == 17 * P.nrows + 32 * fused[0].nescape
    else:
        assert fused[0]._packed is None
        assert fused[0].tod_bytes() == 20 * P.nrows
