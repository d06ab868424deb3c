"""GPU parity of the Carrington ("fa") search (K4/K5) against oracle/carrington.py."""
import numpy as np
import pytest

from conftest import load_pair

pytestmark = pytest.mark.gpu
R_TOL = 1e-6

GRID = dict(lonlims=(248.0, 252.0), latlims=(-4.0, 0.0), shape=(120, 100))
LAGS = dict(lag_crval1=np.arange(20, 29, 2.0), lag_crval2=np.arange(2, 11, 2.0), lag_cdelt1=[0], lag_cdelt2=[0],
            lag_crota=[0])


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _both(pair, lags, grid, **kw):
    from euispice_coreg_b200.hdrshift import Alignment
    from oracle.carrington import CarringtonSearch
    a = Alignment(pair[0], pair[1], parallelism=True, **lags, **kw)
    gpu = a.align_using_carrington(method="correlation", return_type="corr", **grid)
    dl, hl, ds, hs = load_pair(*pair[:2])
    okw = {("order" if k == "reprojection_order" else k): v for k, v in kw.items()}
    s = CarringtonSearch(dl, hl, ds, hs, **lags, **grid, **okw)
    return gpu, s.cube(), a, s


def _assert_parity(gpu, ref):
    assert gpu.shape == ref.shape
    assert np.array_equal(np.isnan(gpu), np.isnan(ref))
    err = np.nanmax(np.abs(gpu - ref))
    assert err <= R_TOL, err
    assert np.unravel_index(np.nanargmax(gpu), gpu.shape) == np.unravel_index(np.nanargmax(ref), ref.shape)
    return err


def test_carrington_large_image_projection_matches_oracle(torch_cuda, toy_pair):
    gpu, ref, a, s = _both(toy_pair, dict(LAGS, lag_crval1=[24.0], lag_crval2=[6.0]), GRID)
    got = a.engine.ref.cpu().numpy()
    assert got.shape == s.data_large.shape == (100, 120) and got.dtype == np.float64
    assert np.array_equal(np.isnan(got), np.isnan(s.data_large))
    # device atan vs libm atan differ by <= 1 ulp in the coordinates -> ~1e-12 relative in the samples
    assert np.nanmax(np.abs(got - s.data_large) / np.abs(s.data_large)) < 1e-10


def test_carrington_cube_parity(torch_cuda, toy_pair):
    gpu, ref, a, _ = _both(toy_pair, LAGS, GRID)
    err = _assert_parity(gpu, ref)
    assert err < 1e-9
    i, j = np.unravel_index(np.nanargmax(gpu), gpu.shape)[:2]
    assert (LAGS["lag_crval1"][i], LAGS["lag_crval2"][j]) == (24.0, 6.0)


def test_carrington_cube_parity_rotation_lags_thresholds_grid_beyond_fov(torch_cuda, toy_pair):
    """CROTA lags (one plane pair per value), masked small pixels, and a grid much larger than the small FOV
    (most Carrington pixels fall outside the small image)."""
    lags = dict(LAGS, lag_crota=[-0.4, 0.0, 0.6])
    grid = dict(lonlims=(244.0, 256.0), latlims=(-8.0, 4.0), shape=(150, 130))
    gpu, ref, _, _ = _both(toy_pair, lags, grid, small_fov_value_min=80.0, small_fov_value_max=1500.0)
    _assert_parity(gpu, ref)


@pytest.mark.parametrize("order", [1, 3])
def test_carrington_orders(torch_cuda, toy_pair, order):
    gpu, ref, _, _ = _both(toy_pair, dict(LAGS, lag_crval1=[22.0, 24.0], lag_crval2=[6.0, 8.0]), GRID,
                           reprojection_order=order)
    _assert_parity(gpu, ref)


def test_carrington_size_deg_grid_and_results_object(torch_cuda, toy_pair):
    from euispice_coreg_b200.hdrshift import Alignment
    a = Alignment(toy_pair[0], toy_pair[1], parallelism=True, **LAGS)
    res = a.align_using_carrington(size_deg_carrington=(4.0, 4.0))
    assert a.shape == [96, 96] and res.corr.shape == (5, 5, 1, 1, 1, 1)
    assert abs(res.shift_arcsec[0] - 24.0) < 1.0 and abs(res.shift_arcsec[1] - 6.0) < 1.0
    with pytest.raises(ValueError):
        Alignment(toy_pair[0], toy_pair[1], **LAGS).align_using_carrington(lonlims=(1, 2))


def test_window_kernel_staging_paths_give_the_same_bits(torch_cuda, toy_pair, monkeypatch):
    """The Carrington kernel stages the reachable part of the small image in shared memory with one TMA tile load per
    (tile, lag chunk); COREG_NO_TMA=1 makes the block copy the window itself (what happens for images whose row pitch
    is not a multiple of 16 bytes). Same arithmetic, same accumulation order: the cubes are bit-identical. The toy
    pair's small image is float32; the float64 instantiation and the copy's own triggers (unaligned pitch or base)
    are driven in test_gpu_carrington_window.py."""
    from euispice_coreg_b200.hdrshift import Alignment, engine
    lags = dict(LAGS, lag_crval1=np.arange(10, 38, 1.0), lag_crval2=np.arange(-6, 18, 1.0))
    grid = dict(lonlims=(246.0, 254.0), latlims=(-6.0, 2.0), shape=(150, 170))

    def run():
        a = Alignment(toy_pair[0], toy_pair[1], parallelism=True, **lags)
        return a.align_using_carrington(method="correlation", return_type="corr", **grid), a

    tma, a = run()
    assert a.engine.small.dtype == torch_cuda.float32
    monkeypatch.setenv("COREG_NO_TMA", "1")
    copy, _ = run()
    monkeypatch.delenv("COREG_NO_TMA")
    assert np.array_equal(tma, copy, equal_nan=True)
    # lags handed over in flat order instead of detector-plane patches: chunks whose window does not fit the box read
    # global memory -- the same samples, the same sums
    eng = a.engine
    d1, d2, _, _, _ = engine.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
    roll = a.hdr_small["CROTA"]
    planes = eng.carrington_planes(a.hdr_small, float(a.lag_solar_r[0]), a.lonlims, a.latlims, a.shape)
    x0, y0 = eng.carrington_offset(a.hdr_small, a.crval1_ref + d1, a.crval2_ref + d2, roll)
    flat = eng.search(np.stack([x0, y0], axis=1), planes=planes)
    assert np.array_equal(flat, tma.ravel(), equal_nan=True)
    from oracle.carrington import CarringtonSearch
    dl, hl, ds, hs = load_pair(*toy_pair[:2])
    s = CarringtonSearch(dl, hl, ds, hs, **lags, **grid)
    sel = [(0, 0), (14, 12), (27, 23), (5, 20)]
    for i, j in sel:
        assert abs(tma[i, j, 0, 0, 0, 0] - s.step(lags["lag_crval1"][i], lags["lag_crval2"][j], 0.0, 0.0, 0.0)) < 1e-9


def test_window_kernel_far_apart_lags_take_the_global_path(torch_cuda, toy_pair):
    """Lags 30 arcsec apart: no shared-memory window holds a 16 x 16 patch of them, every chunk falls back to global
    loads. Parity against the oracle all the same."""
    lags = dict(LAGS, lag_crval1=np.arange(-36, 85, 30.0), lag_crval2=np.arange(-54, 67, 30.0))
    gpu, ref, _, _ = _both(toy_pair, lags, dict(lonlims=(244.0, 256.0), latlims=(-8.0, 4.0), shape=(130, 90)))
    assert _assert_parity(gpu, ref) < 1e-9


def test_carrington_host_buffer_entry_point_matches_public_api(torch_cuda, toy_pair):
    """coreg_carrington_search_host (the call a non-Python host makes at the seam `alignment.py:237`): host images,
    per-header constants and the (x0, y0) offsets of the CRVAL lags in, cube out -- the same bits as the public API
    (it orders the lags into detector-plane patches by itself)."""
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200.hdrshift import Alignment, engine
    lags = dict(LAGS, lag_crval1=np.arange(10, 38, 1.0), lag_crval2=np.arange(-6, 18, 1.0))
    grid = dict(lonlims=(246.0, 254.0), latlims=(-6.0, 2.0), shape=(150, 170))
    a = Alignment(toy_pair[0], toy_pair[1], parallelism=True, **lags)
    cube = a.align_using_carrington(method="correlation", return_type="corr", **grid)
    dl, hl, ds, hs = load_pair(*toy_pair[:2])
    E = engine.LagSearchEngine
    r_sun = float(a.lag_solar_r[0])
    hdr_l, hdr_s = a.hdr_large, a.hdr_small        # with the PCi_j / CROTA checks applied
    roll_l = hdr_l["CROTA"] if "CROTA" in hdr_l else hdr_l["CROTA2"]
    roll_s = hdr_s["CROTA"] if "CROTA" in hdr_s else hdr_s["CROTA2"]
    d1, d2, _, _, _ = engine.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
    x0, y0 = E.carrington_offset(hdr_s, a.crval1_ref + d1, a.crval2_ref + d2, roll_s)
    corr, nvalid = _ext.carrington_search_host(
        dl, E.carrington_struct(hdr_l, r_sun), E.carrington_offset(hdr_l, hdr_l["CRVAL1"], hdr_l["CRVAL2"], roll_l), ds,
        E.carrington_struct(hdr_s, r_sun), E.carrington_vectors(grid["lonlims"], grid["latlims"], grid["shape"],
                                                                hdr_l["CRLN_OBS"]),
        E.carrington_vectors(grid["lonlims"], grid["latlims"], grid["shape"], hdr_s["CRLN_OBS"]),
        np.stack([x0, y0], axis=1))
    assert np.array_equal(corr.reshape(cube.shape), cube, equal_nan=True)
    assert np.array_equal(nvalid.reshape(a.nvalid.shape), a.nvalid)
