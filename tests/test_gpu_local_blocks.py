"""Per-block correlation cubes (`Alignment(..., local_block=...)`) on the device: parity with the oracle's block cubes
for both lag kernels, the global cube left bit-identical, a planted local shift, and SPICE column bands.
Lag grids here leave out the lag (0, 0, 0, 0, 0): its border-membership knife-edge (README) weighs far more in a small
block than in the whole grid."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_local_blocks import block_cube  # noqa: E402  (the block-cube oracle, shared with the CPU tests)

pytestmark = pytest.mark.gpu
R_TOL = 1e-6


def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _load(path):
    from euispice_coreg_b200._compat import fits_lite
    h = fits_lite.open(path)[0]
    return h.data, dict(h.header.items())


def _write_small(p_small, data, hdr, out):
    from euispice_coreg_b200._compat import fits_lite
    fits_lite.writeto(out, [fits_lite.PrimaryHDU(np.ascontiguousarray(data, dtype=np.float32), hdr)], overwrite=True)
    return out


@pytest.fixture(scope="module")
def pairs(tmp_path_factory):
    """96^2 and 256^2 pairs, the ragged 150 x 70 cut, and the 96^2 image with NaN holes."""
    _need_gpu()
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    d = tmp_path_factory.mktemp("local_blocks")
    out = {}
    out["p96"] = make_pair(str(d), small_spec(96, 160, true_crval=(-12.0, 8.0)), tag="p96")[:2]
    out["p256"] = make_pair(str(d), small_spec(256, 400, true_crval=(-12.0, 8.0)), tag="p256")[:2]
    p_large, p_small, _ = make_pair(str(d), small_spec(160, 200, true_crval=(-12.0, 8.0)), tag="rect")
    hd = fits_lite.open(p_small)[0]
    h = hd.header.copy()
    h["NAXIS1"], h["NAXIS2"] = 150, 70
    h["CRPIX1"] = h["CRPIX1"] - 5
    h["CRPIX2"] = h["CRPIX2"] - 10
    out["rect"] = (p_large, _write_small(p_small, hd.data[10:80, 5:155], h, str(d / "rect_cut.fits")))
    data, hdr = _load(out["p96"][1])
    holes = np.array(data, dtype=np.float32)
    holes[10:30, 50:70] = np.nan           # a hole inside one block
    holes[60:66, :] = np.nan               # a band across a block edge
    holes[::7, 3] = np.nan
    out["holes"] = (out["p96"][0], _write_small(None, holes, fits_lite.open(out["p96"][1])[0].header.copy(),
                                                str(d / "holes.fits")))
    return out


SHIFT = dict(lag_crval1=np.arange(19, 30, 2.0), lag_crval2=np.arange(1, 12, 2.0), lag_cdelt1=[0.0], lag_cdelt2=[0.0],
             lag_crota=[0.0])
ROTATED = dict(lag_crval1=np.arange(20, 29, 2.0), lag_crval2=np.arange(2, 11, 2.0), lag_cdelt1=[0.0], lag_cdelt2=[0.0],
               lag_crota=[-0.6, 0.6])


def _run(p_large, p_small, block, lags, **kw):
    from euispice_coreg_b200.hdrshift import Alignment
    a = Alignment(p_large, p_small, parallelism=True, local_block=block, **lags, **kw)
    cube = a.align_using_helioprojective(return_type="corr")
    return a, cube


def _oracle(p_large, p_small, block, lags, **kw):
    from oracle.hpc import HpcSearch
    dl, hl = _load(p_large)
    ds, hs = _load(p_small)
    return block_cube(HpcSearch(dl, hl, ds, hs, **lags, **kw), block)


def _assert_block_parity(gpu, ref):
    assert gpu.shape == ref.shape
    assert np.array_equal(np.isnan(gpu), np.isnan(ref))
    assert np.nanmax(np.abs(gpu - ref)) <= R_TOL
    for i in range(gpu.shape[0]):
        for j in range(gpu.shape[1]):
            if np.isfinite(ref[i, j]).any():
                assert np.nanargmax(gpu[i, j]) == np.nanargmax(ref[i, j]), (i, j)


# (pair, block, lag grid, Alignment keywords, oracle keywords, kernel)
CASES = [
    ("p96", 64, SHIFT, {}, {}, "rolling, pure shifts"),
    ("p96", (64, 128), ROTATED, {}, {}, "rolling, rotated lags"),
    ("p96", 64, SHIFT, {"reprojection_order": 1}, {"order": 1}, "generic, order 1"),
    ("p96", 64, ROTATED, {"reprojection_order": 3}, {"order": 3}, "generic, order 3"),
    ("p96", 64, SHIFT, {"strict_arithmetic": True}, {}, "generic, strict arithmetic"),
    ("p256", 64, SHIFT, {}, {}, "rolling, 256^2"),
    ("p256", (128, 64), ROTATED, {"reprojection_order": 1}, {"order": 1}, "generic, 256^2"),
    ("rect", 64, dict(SHIFT, lag_cdelt2=[0.0, 0.5]), {}, {}, "rolling, ragged grid, dead lags"),
    ("rect", (64, 128), SHIFT, {"reprojection_order": 3}, {"order": 3}, "generic, ragged grid"),
    ("holes", 64, SHIFT, {}, {}, "rolling, NaN holes"),
    ("holes", 64, ROTATED, {"reprojection_order": 1}, {"order": 1}, "generic, NaN holes"),
]


@pytest.mark.parametrize("case", CASES, ids=[c[-1] for c in CASES])
def test_block_cubes_match_oracle(pairs, case):
    name, block, lags, kw, okw, _ = case
    a, cube = _run(*pairs[name], block, lags, **kw)
    ref = _oracle(*pairs[name], block, lags, **okw)
    loc = a.local
    _assert_block_parity(loc.corr, ref)
    ny, nx = _load(pairs[name][1])[0].shape
    from euispice_coreg_b200.hdrshift.engine import region_bounds
    rows, cols = (block, block) if np.isscalar(block) else block
    assert np.array_equal(loc.bounds, region_bounds(ny, nx, (rows, cols)))
    assert loc.corr.shape[:2] == loc.bounds.shape[:2] == loc.nvalid.shape[:2]
    assert np.array_equal(loc.nvalid.sum(axis=(0, 1)), a.nvalid)
    if "dead" in case[-1]:
        assert (loc.corr[:, :, :, :, :, 1] == 0.0).all()
    for i in range(ref.shape[0]):
        for j in range(ref.shape[1]):
            if np.isfinite(ref[i, j]).any():
                assert tuple(loc.max_index[i, j]) == np.unravel_index(np.nanargmax(ref[i, j]), ref.shape[2:])


@pytest.mark.parametrize("kw", [{}, {"reprojection_order": 1}], ids=["rolling", "generic"])
def test_global_cube_unchanged_and_one_block_is_the_global_cube(pairs, kw, monkeypatch):
    from euispice_coreg_b200.hdrshift.engine import LagSearchEngine
    lags = dict(ROTATED, lag_crval1=np.arange(11, 31, 1.0), lag_crval2=np.arange(-4, 16, 1.0))   # 800 lags
    p = pairs["p256"]
    a_none, cube_none = _run(*p, None, lags, **kw)
    assert a_none.local is None
    a_b, cube_b = _run(*p, 64, lags, **kw)
    assert np.array_equal(cube_b.view(np.uint64), cube_none.view(np.uint64))
    assert np.array_equal(a_b.nvalid, a_none.nvalid)
    assert np.array_equal(a_b.local.nvalid.sum(axis=(0, 1)), a_none.nvalid)
    a_one, cube_one = _run(*p, 4096, lags, **kw)
    assert a_one.local.corr.shape[:2] == (1, 1)
    assert np.array_equal(a_one.local.corr[0, 0].view(np.uint64), cube_none.view(np.uint64))
    assert np.array_equal(a_one.local.nvalid[0, 0], a_none.nvalid)
    # lags split over several launches (256 per launch): each lag's block values depend on its own records only
    monkeypatch.setattr(LagSearchEngine, "max_workspace_bytes", 1)
    a_split, cube_split = _run(*p, 64, lags, **kw)
    assert a_split.engine.last_launches == 4 * 3
    assert np.array_equal(cube_split.view(np.uint64), cube_none.view(np.uint64))
    assert np.array_equal(a_split.local.corr.view(np.uint64), a_b.local.corr.view(np.uint64))
    assert np.array_equal(a_split.local.nvalid, a_b.local.nvalid)


def test_results_object_carries_the_block_cubes(pairs):
    from euispice_coreg_b200.hdrshift import Alignment, AlignmentResults
    p = pairs["p96"]
    res = Alignment(*p, parallelism=True, local_block=64, **SHIFT).align_using_helioprojective()
    plain = Alignment(*p, parallelism=True, **SHIFT).align_using_helioprojective()
    assert not hasattr(plain, "local")
    assert np.array_equal(res.corr, plain.corr) and res.shift_arcsec == plain.shift_arcsec
    loc = res.local
    assert loc.corr.shape == (2, 2) + res.corr.shape
    r00 = loc.results(0, 0)
    assert isinstance(r00, AlignmentResults) and np.array_equal(r00.corr, loc.corr[0, 0], equal_nan=True)
    assert r00.max_index == tuple(loc.max_index[0, 0])
    assert np.array_equal(r00.parameters_alignment["lag_crval1"][0], SHIFT["lag_crval1"])


def test_planted_local_shift(tmp_path):
    """Left half of one rendering, right half of another whose true pointing is 4 arcsec away, under one header: the
    two blocks find the two planted corrections."""
    _need_gpu()
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    spec = small_spec(256, 400, true_crval=(-12.0, 8.0), true_shift=(6.0, 4.0))
    p_large, p_a, _ = make_pair(str(tmp_path), spec, tag="a")
    _, p_b, _ = make_pair(str(tmp_path), small_spec(256, 400, true_crval=(-12.0, 8.0), true_shift=(6.0, 4.0),
                                                     jitter=(4.0, -4.0)), tag="b", write_large=False)
    a, b = fits_lite.open(p_a)[0], fits_lite.open(p_b)[0]
    img = np.array(a.data)
    img[:, 128:] = b.data[:, 128:]
    p = _write_small(None, img, a.header.copy(), str(tmp_path / "stitched.fits"))
    lags = dict(lag_crval1=np.arange(2, 15, 1.0), lag_crval2=np.arange(-4, 9, 1.0), lag_cdelt1=[0.0],
                lag_cdelt2=[0.0], lag_crota=[0.0])
    al, cube = _run(p_large, p, (256, 128), lags)
    loc = al.local
    assert loc.corr.shape[:2] == (1, 2)
    found = [(lags["lag_crval1"][loc.max_index[0, j][0]], lags["lag_crval2"][loc.max_index[0, j][1]]) for j in (0, 1)]
    assert found == [(6.0, 4.0), (10.0, 0.0)], found
    # the block cubes' sub-lag fits sit near the planted corrections too
    for j, want in ((0, (6.0, 4.0)), (1, (10.0, 0.0))):
        s = loc.results(0, j).shift_arcsec
        assert abs(s[0] - want[0]) < 1.0 and abs(s[1] - want[1]) < 1.0, (j, s)


def test_spice_column_bands_match_oracle(tmp_path):
    """A 192-slit-position raster cut into three bands of 64 positions (one block row covering the raster height)."""
    _need_gpu()
    from euispice_coreg_b200._synth.spice import make_spice_case, small_spice_spec
    from euispice_coreg_b200.hdrshift import AlignmentSpice
    from oracle.hpc import HpcSearch
    from oracle.synras import spice_l2_image
    p_spice, imagers, spec = make_spice_case(str(tmp_path), small_spice_spec(n_x=192, large_n=256, nbin2=8, pxbeg2=192),
                                             tag="bands")
    lags = dict(lag_crval1=np.arange(-14, -1, 2.0), lag_crval2=np.arange(6, 19, 2.0), lag_cdelt1=[0], lag_cdelt2=[0],
                lag_crota=[0])
    d4, h4 = _load(p_spice)
    img, hdr = spice_l2_image(d4, h4)
    assert img.shape == (spec.n_y, 192)
    rows = -(-spec.n_y // 64) * 64
    a = AlignmentSpice(imagers[0], p_spice, parallelism=True, small_fov_window=0, large_fov_window=-1,
                       local_block=(rows, 64), **lags)
    res = a.align_using_helioprojective()
    loc = res.local
    assert loc.corr.shape[:2] == (1, 3)
    assert loc.bounds[0, :, 2:].tolist() == [[0, 64], [64, 128], [128, 192]]
    dl, hl = _load(imagers[0])
    ref = block_cube(HpcSearch(dl, hl, img, hdr, **lags), (rows, 64))
    _assert_block_parity(loc.corr, ref)
    assert np.array_equal(loc.nvalid.sum(axis=(0, 1)), a.nvalid)
