"""Per-block correlation cubes of the Carrington searches (`align_using_carrington(..., local_block=...)`) on the device:
parity with the oracle's block cubes on the window kernel, the generic kernel and the "sunpy" path, the global cube
left bit-identical, a planted latitude-dependent shift, and frame sequences."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from conftest import load_pair  # noqa: E402
from test_carrington_local_blocks import carrington_block_cube, with_observers  # noqa: E402  (CPU oracle, shared)

pytestmark = pytest.mark.gpu
R_TOL = 1e-6

# ragged Carrington grid: 150 longitude x 130 latitude samples (no side a multiple of 32 or 64), larger than the FOV
RAGGED = dict(lonlims=(246.0, 254.0), latlims=(-6.0, 2.0), shape=(150, 130))
# two CROTA lags (two plane pairs) and a CDELT2 lag the reference cannot evaluate (0.0 in every block)
LAGS = dict(lag_crval1=[20.0, 22.0, 24.0, 26.0], lag_crval2=[4.0, 6.0, 8.0], lag_cdelt1=[0.0], lag_cdelt2=[0.0, 0.5],
            lag_crota=[0.0, 0.5])
SUNPY_LAGS = dict(LAGS, lag_cdelt2=[0.0])


@pytest.fixture(scope="module")
def pairs(toy_pair, tmp_path_factory):
    """The toy pair (float32 small image), its float64 copy, a copy with NaN holes and -32762 pixels, and a copy with
    the observer keywords of the "sunpy" path."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from euispice_coreg_b200._compat import fits_lite
    d = tmp_path_factory.mktemp("car_blocks")
    hd = fits_lite.open(toy_pair[1])[0]

    def write(data, name):
        p = str(d / name)
        fits_lite.writeto(p, [fits_lite.PrimaryHDU(data, hd.header.copy())], overwrite=True)
        return p

    holes = np.array(hd.data, dtype=np.float32)
    holes[10:30, 50:70] = np.nan
    holes[60:66, :] = np.nan
    holes[40:44, 5:90:3] = -32762.0
    holes[::7, 3] = np.nan
    return {"f32": toy_pair[:2], "f64": (toy_pair[0], write(np.array(hd.data, dtype=np.float64), "f64.fits")),
            "holes": (toy_pair[0], write(holes, "holes.fits")), "sunpy": with_observers(toy_pair, d)}


def _run(pair, block, lags, method="fa", grid=RAGGED, **kw):
    from euispice_coreg_b200.hdrshift import Alignment
    a = Alignment(pair[0], pair[1], parallelism=True, **lags, **kw)
    cube = a.align_using_carrington(return_type="corr", method_carrington_reprojection=method, local_block=block,
                                    **({} if method == "sunpy" else grid))
    return a, cube


def _oracle(pair, block, lags, method="fa", grid=RAGGED, **kw):
    dl, hl, ds, hs = load_pair(*pair)
    if method == "sunpy":
        from oracle.surface_reproject import SurfaceSearch
        s = SurfaceSearch(dl, hl, ds, hs, **lags)
    else:
        from oracle.carrington import CarringtonSearch
        okw = {("order" if k == "reprojection_order" else k): v for k, v in kw.items() if k != "strict_arithmetic"}
        s = CarringtonSearch(dl, hl, ds, hs, **lags, **grid, **okw)
    return carrington_block_cube(s, block, counts=True)


# (pair, block, lag grid, method, Alignment keywords, kernel)
CASES = [
    ("f32", 64, LAGS, "fa", {}, "window, float32"),
    ("f64", (128, 64), LAGS, "fa", {}, "window, float64"),
    ("f32", (192, 64), LAGS, "fa", {}, "window, longitude bands"),
    ("f64", (64, 192), LAGS, "fa", {}, "window, latitude bands"),
    ("holes", 64, LAGS, "fa", {}, "window, NaN holes and -32762"),
    ("f32", 64, LAGS, "fa", {"reprojection_order": 1}, "generic, order 1"),
    ("f64", (128, 64), LAGS, "fa", {"reprojection_order": 3}, "generic, order 3"),
    ("holes", 64, LAGS, "fa", {"strict_arithmetic": True}, "generic, strict arithmetic"),
    ("sunpy", 64, SUNPY_LAGS, "sunpy", {}, "sunpy"),
    ("sunpy", (64, 192), SUNPY_LAGS, "sunpy", {}, "sunpy, latitude bands"),
]


def _assert_block_parity(a, cube, ref, ref_n, block):
    loc = a.local
    assert loc.corr.shape == ref.shape and loc.nvalid.shape == ref_n.shape
    assert np.array_equal(np.isnan(loc.corr), np.isnan(ref))
    assert np.nanmax(np.abs(loc.corr - ref)) <= R_TOL
    assert np.array_equal(loc.nvalid, ref_n)
    assert np.array_equal(loc.nvalid.sum(axis=(0, 1)), a.nvalid)
    gny, gnx = a.engine.ref.shape
    from euispice_coreg_b200.hdrshift.engine import region_bounds
    rows, cols = (block, block) if np.isscalar(block) else block
    assert np.array_equal(loc.bounds, region_bounds(gny, gnx, (rows, cols)))
    for i in range(ref.shape[0]):
        for j in range(ref.shape[1]):
            if np.isfinite(ref[i, j]).any():
                assert tuple(loc.max_index[i, j]) == np.unravel_index(np.nanargmax(ref[i, j]), ref.shape[2:]), (i, j)


@pytest.mark.parametrize("case", CASES, ids=[c[-1] for c in CASES])
def test_block_cubes_match_oracle(pairs, case):
    name, block, lags, method, kw, _ = case
    a, cube = _run(pairs[name], block, lags, method, **kw)
    if method == "fa":
        assert a.engine.ref.shape == (130, 150)
    ref, ref_n = _oracle(pairs[name], block, lags, method, **kw)
    _assert_block_parity(a, cube, ref, ref_n, block)
    if method == "fa":      # CDELT2 lags: 0.0 in every block, as in the cube
        assert (a.local.corr[:, :, :, :, :, 1] == 0.0).all() and (a.local.nvalid[:, :, :, :, :, 1] == 0).all()
    # most blocks of a grid wider than the FOV see nothing: NaN with count 0
    if name != "sunpy":
        empty = (a.local.nvalid == 0).all(axis=tuple(range(2, a.local.nvalid.ndim)))
        assert empty.any() and np.isnan(a.local.corr[empty][..., 0, 0, 0, :]).all()


def test_window_kernel_staging_without_tma_matches_oracle(pairs, monkeypatch):
    monkeypatch.setenv("COREG_NO_TMA", "1")
    a, cube = _run(pairs["f32"], 64, LAGS)
    ref, ref_n = _oracle(pairs["f32"], 64, LAGS)
    _assert_block_parity(a, cube, ref, ref_n, 64)


# 768 lags: three 16 x 16 patches of the window kernel's lag order, three launches of 256 when the workspace is capped
SPLIT = dict(lag_crval1=np.arange(0.0, 48.0), lag_crval2=np.arange(-2.0, 14.0), lag_cdelt1=[0.0], lag_cdelt2=[0.0],
             lag_crota=[0.0])


@pytest.mark.parametrize("variant", [("fa", {}), ("fa", {"reprojection_order": 1}), ("sunpy", {})],
                         ids=["window", "generic", "sunpy"])
def test_global_cube_unchanged_and_one_block_is_the_global_cube(pairs, variant, monkeypatch):
    from euispice_coreg_b200.hdrshift.engine import LagSearchEngine
    method, kw = variant
    p = pairs["sunpy" if method == "sunpy" else "f32"]
    a_none, cube_none = _run(p, None, SPLIT, method, **kw)
    assert a_none.local is None
    a_b, cube_b = _run(p, 64, SPLIT, method, **kw)
    assert np.array_equal(cube_b.view(np.uint64), cube_none.view(np.uint64))
    assert np.array_equal(a_b.nvalid, a_none.nvalid)
    assert np.array_equal(a_b.local.nvalid.sum(axis=(0, 1)), a_none.nvalid)
    a_one, _ = _run(p, 4096, SPLIT, method, **kw)
    assert a_one.local.corr.shape[:2] == (1, 1)
    assert np.array_equal(a_one.local.corr[0, 0].view(np.uint64), cube_none.view(np.uint64))
    assert np.array_equal(a_one.local.nvalid[0, 0], a_none.nvalid)
    # three or more launches: each lag's block values depend on its own records only
    monkeypatch.setattr(LagSearchEngine, "max_workspace_bytes", 1)
    a_split, cube_split = _run(p, 64, SPLIT, method, **kw)
    assert a_split.engine.last_launches >= 3 * 3
    assert np.array_equal(cube_split.view(np.uint64), cube_none.view(np.uint64))
    assert np.array_equal(a_split.local.corr.view(np.uint64), a_b.local.corr.view(np.uint64))
    assert np.array_equal(a_split.local.nvalid, a_b.local.nvalid)


def test_results_object_carries_the_block_cubes(pairs):
    from euispice_coreg_b200.hdrshift import Alignment, AlignmentResults
    lags = dict(LAGS, lag_cdelt2=[0.0], lag_crota=[0.0])
    a = Alignment(*pairs["f32"], parallelism=True, **lags)
    res = a.align_using_carrington(local_block=(64, 192), **RAGGED)
    plain = Alignment(*pairs["f32"], parallelism=True, **lags).align_using_carrington(**RAGGED)
    assert not hasattr(plain, "local") and a.local_block is None
    assert np.array_equal(res.corr, plain.corr, equal_nan=True) and res.shift_arcsec == plain.shift_arcsec
    loc = res.local
    assert loc is a.local and loc.corr.shape == (3, 1) + res.corr.shape
    i = int(np.argmax(loc.nvalid.reshape(3, -1).sum(axis=1)))
    r = loc.results(i, 0)
    assert isinstance(r, AlignmentResults) and r.max_index == tuple(loc.max_index[i, 0])


def test_planted_latitude_dependent_shift(tmp_path):
    """The southern and northern halves of the small image come from renderings whose true pointings differ by 4 arcsec
    in each axis, under one header: each latitude band of the Carrington grid finds its own correction."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    from oracle.carrington import CarringtonTransform
    spec = small_spec(256, 400, true_crval=(-12.0, 8.0), true_shift=(6.0, 4.0))
    p_large, p_a, _ = make_pair(str(tmp_path), spec, tag="a")
    _, p_b, _ = make_pair(str(tmp_path), small_spec(256, 400, true_crval=(-12.0, 8.0), true_shift=(6.0, 4.0),
                                                     jitter=(4.0, -4.0)), tag="b", write_large=False)
    a, b = fits_lite.open(p_a)[0], fits_lite.open(p_b)[0]
    grid = dict(lonlims=(249.2, 250.8), latlims=(-2.9, -1.3), shape=(128, 128))
    # detector row of the boundary between the two latitude bands (grid rows 63 | 64), from the small header
    t = CarringtonTransform(dict(a.header.items()), radius_correction=1.004)
    _, ys = t(*np.meshgrid(np.linspace(*grid["lonlims"], grid["shape"][0], dtype=np.float32),
                           np.linspace(*grid["latlims"], grid["shape"][1], dtype=np.float32)))
    assert ys.shape == (128, 128) and ((ys > 2) & (ys < 253)).all()      # the grid lies inside the small image
    cut = int(round(0.5 * (np.median(ys[63]) + np.median(ys[64]))))
    south_low = np.median(ys[:64]) < cut
    img = np.array(a.data)
    img[cut:] = b.data[cut:]
    p = str(tmp_path / "stitched.fits")
    fits_lite.writeto(p, [fits_lite.PrimaryHDU(np.ascontiguousarray(img, dtype=np.float32), a.header.copy())],
                      overwrite=True)
    lags = dict(lag_crval1=np.arange(2, 15, 1.0), lag_crval2=np.arange(-4, 9, 1.0), lag_cdelt1=[0.0],
                lag_cdelt2=[0.0], lag_crota=[0.0])
    al, _ = _run((p_large, p), (64, 128), lags, grid=grid)
    loc = al.local
    assert loc.corr.shape[:2] == (2, 1)
    found = [(lags["lag_crval1"][loc.max_index[i, 0][0]], lags["lag_crval2"][loc.max_index[i, 0][1]]) for i in (0, 1)]
    want = [(6.0, 4.0), (10.0, 0.0)] if south_low else [(10.0, 0.0), (6.0, 4.0)]
    assert found == want, (found, cut, south_low)


# ------------------------------------------------------------------------------------------------ frame sequences
SEQ_LAGS = dict(lag_crval1=np.arange(18, 31, 2.0), lag_crval2=np.arange(0, 13, 2.0), lag_cdelt1=[0], lag_cdelt2=[0],
                lag_crota=[0.0, 0.5], small_fov_value_min=80.0)
SEQ_GRID = dict(lonlims=(244.0, 256.0), latlims=(-8.0, 4.0), shape=(150, 130))


@pytest.fixture(scope="module")
def frames(tmp_path_factory):
    """{"fa" / "sunpy": (reference path, [frame paths])}: jittered renderings of one sky."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from euispice_coreg_b200._synth.scene import make_pair, master_scene, small_spec
    d = tmp_path_factory.mktemp("seqcar_blocks")
    sky = master_scene(small_spec(96, 160, true_crval=(-12.0, 8.0)))
    p_large, paths, obs = None, [], []
    for i, jit in enumerate([(0.0, 0.0), (1.3, -0.8), (-2.1, 0.4)]):
        spec = small_spec(96, 160, true_crval=(-12.0, 8.0), jitter=jit, noise_seed=400 + i,
                          date=f"2022-03-17T09:5{i}:45.000")
        pl, ps, _ = make_pair(str(d), spec, tag=f"c{i}", sky=sky, write_large=(i == 0))
        p_large = p_large or pl
        paths.append(ps)
        obs.append(with_observers((p_large, ps), d, tag=f"o{i}"))
    return {"fa": (p_large, paths), "sunpy": (obs[0][0], [o[1] for o in obs])}


@pytest.mark.parametrize("n_frames", [1, 3])
@pytest.mark.parametrize("method", ["fa", "sunpy"])
def test_sequence_blocks_equal_per_pair_alignment(frames, method, n_frames):
    from euispice_coreg_b200.hdrshift import Alignment, SequenceAlignment
    p_large, paths = frames[method]
    grid = SEQ_GRID if method == "fa" else {}
    seq = SequenceAlignment(p_large, paths[:n_frames], **SEQ_LAGS)
    res = seq.align_using_carrington(method_carrington_reprojection=method, local_block=64, **grid)
    assert len(res) == n_frames
    for p, r in zip(paths, res):
        one = Alignment(p_large, p, parallelism=True, **SEQ_LAGS).align_using_carrington(
            method_carrington_reprojection=method, local_block=64, **grid)
        assert np.array_equal(r.corr, one.corr, equal_nan=True)
        assert r.local.corr.shape == one.local.corr.shape
        assert np.array_equal(r.local.corr.view(np.uint64), one.local.corr.view(np.uint64))
        assert np.array_equal(r.local.nvalid, one.local.nvalid)
        assert np.array_equal(r.local.bounds, one.local.bounds)
        assert np.array_equal(r.local.max_index, one.local.max_index)
