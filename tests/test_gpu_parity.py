"""GPU parity tests: CUDA path (through the C ABI) vs the CPU oracle on the same seeded inputs.

Bars (north_star): every correlation coefficient within 1e-6 absolute of the oracle (observed ~1e-13),
arg-max lag tuple identical, NaN pattern identical; the one-shot resampling kernels are bit-exact against
scipy's map_coordinates.
"""
import numpy as np
import pytest
from scipy.ndimage import map_coordinates

from conftest import load_pair

pytestmark = pytest.mark.gpu

R_TOL = 1e-6  # tolerance stated by BASELINE.json north_star
# what the two arithmetic modes of the homography kernel actually deliver against the oracle (both far inside R_TOL):
# "fp64" (the default) repeats the reference's FP64 tap arithmetic (FMA-contracted); "mixed" (opt-in, small images that
# hold float32 values) evaluates the spline in FP32 on the pivot-centred image and reproduces the reference's float32
# store on the uncentred value; lags its error model cannot vouch for to 1e-7 are redone in FP64
OBSERVED = {"fp64": 1e-10, "mixed": 5e-8}
ARITH = pytest.mark.parametrize("arithmetic", ["fp64", "mixed"])


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from euispice_coreg_b200 import _ext
    _ext.load()
    return torch


def _hdr(crval=(-100.0, 50.0), crota=3.0, unit="arcsec", n=(200, 120), cdelt=0.492):
    rho = np.deg2rad(crota)
    return {"NAXIS1": n[0], "NAXIS2": n[1], "CTYPE1": "HPLN-TAN", "CTYPE2": "HPLT-TAN", "CUNIT1": unit,
            "CUNIT2": unit, "CRPIX1": (n[0] + 1) / 2, "CRPIX2": (n[1] + 1) / 2, "CDELT1": cdelt, "CDELT2": cdelt,
            "CRVAL1": crval[0], "CRVAL2": crval[1], "PC1_1": np.cos(rho), "PC1_2": -np.sin(rho),
            "PC2_1": np.sin(rho), "PC2_2": np.cos(rho), "LONPOLE": 180.0, "CROTA": crota}


@pytest.mark.parametrize("unit,crval,cdelt", [("arcsec", (-100.0, 50.0), 0.492), ("deg", (0.3, -0.2), 4.44 / 3600),
                                              ("arcsec", (2000.0, -1500.0), 4.44)])
def test_k3_pixel_to_world_matches_oracle(torch_cuda, unit, crval, cdelt):
    from euispice_coreg_b200.utils.Util import AlignEUIUtil
    from oracle import wcs_tan
    h = _hdr(crval=crval, unit=unit, cdelt=cdelt)
    lng, lat = AlignEUIUtil.extract_EUI_coordinates(h, dsun=False)
    lng_o, lat_o = wcs_tan.extract_coordinates(h)
    assert lng.shape == (120, 200)
    assert np.max(np.abs(lng - lng_o)) < 1e-11 and np.max(np.abs(lat - lat_o)) < 1e-11


def test_world_to_pixel_matches_oracle(torch_cuda):
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._compat.wcs import TanWcs
    from oracle import wcs_tan
    h = _hdr()
    lng_o, lat_o = wcs_tan.extract_coordinates(h)
    for shift, crota in (((30.0, -20.0), 3.0), ((-5.0, 7.5), 3.75)):
        h2 = _hdr(crval=(-100.0 + shift[0], 50.0 + shift[1]), crota=crota)
        x_o, y_o = wcs_tan.WcsTan(h2).world_to_pixel(lng_o, lat_o)
        x, y = _ext.tan_world2pix(TanWcs.from_header(h2), torch_cuda.from_numpy(lng_o).cuda(),
                                  torch_cuda.from_numpy(lat_o).cuda())
        assert np.max(np.abs(x.cpu().numpy() - x_o)) < 1e-9 and np.max(np.abs(y.cpu().numpy() - y_o)) < 1e-9


@pytest.mark.parametrize("order", [0, 1, 2, 3])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_fused_cut_equals_the_three_kernels_bit_for_bit(torch_cuda, order, dtype):
    """`coreg_hpc_cut` (one kernel: world grid -> large-image coordinates -> window origin -> spline sample -> float32)
    against tan_pix2world -> tan_world2pix -> origin subtraction -> map_coordinates, which are pinned one by one above and
    below: same bits, NaN pattern included (part of the small grid lies outside the large image), for the whole image
    and for an uploaded window of it; and against the oracle's `_create_submap_of_large_data`."""
    torch = torch_cuda
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._compat.wcs import TanWcs
    hs = _hdr(crval=(-100.0, 50.0), crota=3.0, n=(200, 120), cdelt=0.492)
    hl = _hdr(crval=(-80.0, 30.0), crota=-1.5, n=(96, 80), cdelt=1.1)      # covers most, not all, of the small grid
    ws, wl = TanWcs.from_header(hs), TanWcs.from_header(hl)
    rng = np.random.default_rng(7)
    large = rng.normal(500.0, 300.0, (80, 96)).astype(dtype)
    large[10, 20] = np.nan
    for x0, y0 in ((0, 0), (7, 5)):
        d_large = torch.from_numpy(np.ascontiguousarray(large[y0:, x0:])).cuda()
        lng, lat = _ext.tan_pix2world(ws, ws.naxis1, ws.naxis2, True)
        x, y = _ext.tan_world2pix(wl, lng, lat)
        x -= float(x0)
        y -= float(y0)
        ref3 = _ext.map_coordinates(d_large, y, x, order, float("nan"), torch.float32).cpu().numpy()
        ref1 = _ext.hpc_cut(ws, wl, d_large, (x0, y0), order).cpu().numpy()
        assert ref1.shape == (120, 200) and ref1.dtype == np.float32
        assert np.isnan(ref1).any() and np.isfinite(ref1).sum() > 0.3 * ref1.size
        assert np.array_equal(ref1.view(np.uint32), ref3.view(np.uint32))
    if order == 0:
        return      # nearest pixel: a coordinate 1e-10 pixel from a half-integer may pick the neighbour
    from oracle import wcs_tan
    xo, yo = wcs_tan.extract_coordinates_pixels(hs, hl)
    want = map_coordinates(large, [yo, xo], order=order, mode="constant", cval=np.nan, prefilter=False).astype(np.float32)
    got = _ext.hpc_cut(ws, wl, torch.from_numpy(large).cuda(), (0, 0), order).cpu().numpy()
    both = np.isfinite(want) & np.isfinite(got)
    assert (np.isfinite(want) != np.isfinite(got)).sum() <= 4          # closed-bound membership of border pixels
    assert np.max(np.abs(want[both] - got[both])) <= 1e-3              # coordinates agree to ~1e-10 pixel


@pytest.mark.parametrize("order", [0, 1, 2, 3])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_map_coordinates_bit_exact_vs_scipy(torch_cuda, order, dtype):
    """interpol2d drop-in (utils/Util.py:82-104): integer/half-integer/border/NaN coordinates included."""
    from euispice_coreg_b200.utils.Util import AlignCommonUtil
    rng = np.random.default_rng(order * 7 + 1)
    img = rng.lognormal(5, 1, (37, 53)).astype(dtype)
    img[5, 7] = np.nan
    n = 30000
    y = rng.uniform(-3, 40, n)
    x = rng.uniform(-3, 56, n)
    y[:8] = [0.0, 36.0, 36.0000001, -1e-12, 0.5, 35.5, np.nan, 18.0]
    x[:8] = [0.0, 52.0, 3.0, 4.0, 51.5, 0.5, 2.0, np.nan]
    for out_dtype in (np.float32, np.float64):
        ref = np.empty(n, dtype=out_dtype)
        map_coordinates(img, np.stack((y, x)), order=order, mode="constant", cval=-7.5, output=ref, prefilter=False)
        dst = np.zeros(n, dtype=out_dtype)
        AlignCommonUtil.interpol2d(img, x=x, y=y, fill=-7.5, order=order, dst=dst)
        assert np.array_equal(ref, dst, equal_nan=True)
    # tiny images: every tap mirrored
    tiny = rng.normal(size=(2, 3)).astype(dtype)
    yy, xx = rng.uniform(0, 1, 500), rng.uniform(0, 2, 500)
    ref = map_coordinates(tiny, np.stack((yy, xx)), order=order, mode="constant", cval=0.0, prefilter=False)
    assert np.array_equal(ref, AlignCommonUtil.interpol2d(tiny, x=xx, y=yy, fill=0.0, order=order))


def _gpu_cube(pair, **kw):
    from euispice_coreg_b200.hdrshift import Alignment
    a = Alignment(pair[0], pair[1], parallelism=True, **kw)
    return a.align_using_helioprojective(return_type="corr"), a


def _oracle_cube(pair, **kw):
    from oracle.hpc import HpcSearch
    dl, hl, ds, hs = load_pair(*pair[:2])
    kw = dict(kw)
    kw["order"] = kw.pop("reprojection_order", 2)
    kw["cdelt_mode"] = kw.pop("cdelt_semantics", "reference")
    kw.pop("strict_arithmetic", None)
    kw.pop("arithmetic", None)
    s = HpcSearch(dl, hl, ds, hs, **kw)
    return s.cube(), s


def _assert_parity(gpu, ref, tol=R_TOL):
    assert gpu.shape == ref.shape and gpu.dtype == np.float64
    assert np.array_equal(np.isnan(gpu), np.isnan(ref))
    err = np.nanmax(np.abs(gpu - ref))
    assert err <= tol, err
    assert np.unravel_index(np.nanargmax(gpu), gpu.shape) == np.unravel_index(np.nanargmax(ref), ref.shape)
    return err


LAGS = dict(lag_crval1=np.arange(20, 29, 2.0), lag_crval2=np.arange(2, 11, 2.0), lag_cdelt1=[0], lag_cdelt2=[0],
            lag_crota=[0])


@ARITH
def test_hpc_cube_parity_basic(torch_cuda, toy_pair, arithmetic):
    gpu, a = _gpu_cube(toy_pair, arithmetic=arithmetic, **LAGS)
    assert (a.engine.small32 is not None) == (arithmetic == "mixed")   # the toy files are BITPIX -32
    ref, s = _oracle_cube(toy_pair, **LAGS)
    err = _assert_parity(gpu, ref)
    assert err < OBSERVED[arithmetic]
    i, j = np.unravel_index(np.nanargmax(gpu), gpu.shape)[:2]
    assert (LAGS["lag_crval1"][i], LAGS["lag_crval2"][j]) == (24.0, 6.0)
    # the one-time cut of the large image (K2): same NaN pattern; the coordinates come from device trig (<= 1e-11 px
    # from the oracle's) so a float32 rounding may flip in a rare pixel, never more than one float32 ulp
    k2, k2o = a.engine.ref.cpu().numpy(), s.data_large
    assert np.array_equal(np.isnan(k2), np.isnan(k2o)) and np.mean(k2 == k2o) > 0.999
    assert np.nanmax(np.abs(k2 - k2o) / np.abs(k2o)) < 1.3e-7


@pytest.mark.parametrize("order", [1, 2, 3])
def test_hpc_cube_parity_orders_rotation_thresholds(torch_cuda, toy_pair, order):
    kw = dict(LAGS, lag_crota=[-0.5, 0.0, 0.75], reprojection_order=order, small_fov_value_min=80.0,
              small_fov_value_max=1500.0)
    gpu, _ = _gpu_cube(toy_pair, **kw)
    ref, _ = _oracle_cube(toy_pair, **kw)
    _assert_parity(gpu, ref)


def test_hpc_cube_parity_ragged_tiles_and_large_shifts(torch_cuda, toy_rect_pair):
    """150x70 grid (partial 64x32 tiles) and lags that push most of the small image out of bounds."""
    kw = dict(lag_crval1=np.array([-150.0, -60.0, 24.0, 90.0, 400.0]), lag_crval2=np.array([-80.0, 6.0, 70.0]),
              lag_cdelt1=None, lag_cdelt2=None, lag_crota=None)
    gpu, a = _gpu_cube(toy_rect_pair, **kw)
    ref, _ = _oracle_cube(toy_rect_pair, **kw)
    _assert_parity(gpu, ref)
    assert np.isnan(gpu[4]).all()            # shifted completely off the image: empty selection -> NaN
    assert a.nvalid[4].max() == 0


def test_hpc_cube_fov_limits_and_remove_fov_limits(torch_cuda, toy_pair):
    """fov_limits: the small image is first re-sampled onto a regular, unrotated lon / lat grid inside the limits
    (alignment.py:1082-1127, non-square selection: the reference's NAXIS1 / CRPIX1 quirk included); the search runs
    on that image and header."""
    from euispice_coreg_b200.hdrshift import Alignment
    from oracle.hpc import HpcSearch
    fov = [[-80.0, 10.0], [-40.0, 45.0]]
    a = Alignment(toy_pair[0], toy_pair[1], parallelism=True, **LAGS)
    gpu = a.align_using_helioprojective(return_type="corr", fov_limits=fov)
    dl, hl, ds, hs = load_pair(*toy_pair[:2])
    s = HpcSearch(dl, hl, ds, hs, fov_limits=fov, **LAGS)
    assert a.hdr_small["NAXIS1"] == s.hdr_small["NAXIS1"] != a.hdr_small["NAXIS2"] and a.hdr_small["CROTA"] == 0.0
    for k in ("CRVAL1", "CRVAL2", "CDELT1", "CDELT2", "CRPIX1", "CRPIX2"):
        assert abs(a.hdr_small[k] - s.hdr_small[k]) < 1e-7, k   # device vs numpy trig: ~1e-12 deg
    _assert_parity(gpu, s.cube())
    i, j = np.unravel_index(np.nanargmax(gpu), gpu.shape)[:2]
    assert (LAGS["lag_crval1"][i], LAGS["lag_crval2"][j]) == (24.0, 6.0)


def test_hpc_cube_cdelt_semantics(torch_cuda, toy_pair):
    kw = dict(lag_crval1=[22.0, 24.0], lag_crval2=[6.0], lag_cdelt1=[0.0, 0.004], lag_cdelt2=[0.0, -0.003],
              lag_crota=[0.0, 0.3])
    for sem in ("reference", "intended"):
        gpu, _ = _gpu_cube(toy_pair, cdelt_semantics=sem, **kw)
        ref, _ = _oracle_cube(toy_pair, cdelt_semantics=sem, **kw)
        _assert_parity(gpu, ref)
    assert np.all(gpu != 0.0)


def test_hpc_cube_deg_units(torch_cuda, toy_pair, tmp_path):
    """Headers in degrees: lags given in arcsec are converted like alignment.py:819-837."""
    from euispice_coreg_b200._compat import fits_lite
    paths = []
    for p in toy_pair[:2]:
        h = fits_lite.open(p)[0]
        hdr = h.header.copy()
        for k in ("CRVAL1", "CRVAL2", "CDELT1", "CDELT2"):
            hdr[k] = hdr[k] / 3600.0
        hdr["CUNIT1"] = hdr["CUNIT2"] = "deg"
        q = str(tmp_path / ("deg_" + p.split("/")[-1]))
        fits_lite.writeto(q, [fits_lite.PrimaryHDU(h.data, hdr)], overwrite=True)
        paths.append(q)
    gpu, _ = _gpu_cube(paths, **LAGS)
    ref, _ = _oracle_cube(paths, **LAGS)
    _assert_parity(gpu, ref)
    i, j = np.unravel_index(np.nanargmax(gpu), gpu.shape)[:2]
    assert (LAGS["lag_crval1"][i], LAGS["lag_crval2"][j]) == (24.0, 6.0)


def test_strict_arithmetic_mode(torch_cuda, toy_pair):
    """scipy's exact tap arithmetic; the default FMA mode differs from it by far less than the tolerance."""
    gpu, _ = _gpu_cube(toy_pair, strict_arithmetic=True, **LAGS)
    fma, _ = _gpu_cube(toy_pair, arithmetic="fp64", **LAGS)
    # homography kernel with FMA arithmetic vs strict = generic kernel, scipy operation order
    assert np.nanmax(np.abs(gpu - fma)) < 1e-10
    dflt, a = _gpu_cube(toy_pair, **LAGS)       # the default is the reference's arithmetic: everything in FP64
    assert a.engine.arithmetic == "fp64" and a.engine.small32 is None and np.array_equal(dflt, fma)
    mixed, a = _gpu_cube(toy_pair, arithmetic="mixed", **LAGS)      # opt-in: FP64 projection, FP32 spline
    assert a.engine.arithmetic == "mixed" and a.engine.small32 is not None
    assert np.nanmax(np.abs(gpu - mixed)) < OBSERVED["mixed"]
    ref, _ = _oracle_cube(toy_pair, **LAGS)
    _assert_parity(gpu, ref)


def test_mixed_arithmetic_needs_float32_headroom(torch_cuda, toy_pair):
    """The float32 segment sums of the mixed kernel square pixel values: an image in units that push them towards the
    ends of the float32 range is searched by the all-FP64 kernel, whatever was requested. Scaling by 2^-70 is exact
    in binary floating point and r is scale-invariant, so that cube equals the all-FP64 cube of the original image
    bit for bit."""
    from euispice_coreg_b200.hdrshift import engine
    f64, _ = _gpu_cube(toy_pair, arithmetic="fp64", **LAGS)
    mixed, a = _gpu_cube(toy_pair, arithmetic="mixed", **LAGS)
    eng = a.engine
    assert eng._mixed_applies() and not np.array_equal(mixed, f64)
    d = engine.flat_lag_grid(LAGS["lag_crval1"], LAGS["lag_crval2"], [0.0], [0.0], [0.0])
    table, _ = eng.hpc_lag_table(a.hdr_small, a, *d)
    small = eng.small.cpu().numpy()
    eng.set_small(small * 2.0 ** -70)          # ~1e-19: float32 values still, but their squares are not
    assert eng.small32 is not None and not eng._mixed_applies()
    assert np.array_equal(eng.search(table), f64.ravel())
    eng.set_small(small)
    assert eng._mixed_applies() and np.array_equal(eng.search(table), mixed.ravel())


def _rewrite_small(pair, out_dir, tag, fn):
    """The pair with its small image's pixel values transformed by `fn` (float64 -> float64), stored as float32."""
    import os
    from euispice_coreg_b200._compat import fits_lite
    hd = fits_lite.open(pair[1])[0]
    data = fn(np.asarray(hd.data, dtype=np.float64)).astype(np.float32)
    p = os.path.join(str(out_dir), f"{tag}_small.fits")
    fits_lite.writeto(p, [fits_lite.PrimaryHDU(data, hd.header.copy())], overwrite=True)
    return pair[0], p


HARD_IMAGES = {
    # un-subtracted background: mean 3e4, sigma 1 -- one float32 ulp of a PIXEL VALUE is 2e-3 sigma
    "low_contrast": lambda d: 3e4 + (d - d.mean()) / d.std(),
    # six decades of dynamic range, 0.1 ... 1e5
    "six_decades": lambda d: 10.0 ** (6.0 * (d - d.min()) / (d.max() - d.min()) - 1.0),
    # mean 1e7, sigma 1: the float32 grid of the samples is as coarse as the signal
    "quantised": lambda d: 1e7 + (d - d.mean()) / d.std(),
}


@pytest.mark.parametrize("kind", sorted(HARD_IMAGES))
@ARITH
def test_hard_images_stay_inside_the_contract(torch_cuda, toy_pair, tmp_path, kind, arithmetic):
    """Images built to break a float32 spline: every r within 1e-6 of the oracle in BOTH arithmetic modes. The mixed
    kernel centres the image on its pivot and reproduces the reference's float32 store, so its error scales with the
    deviation from the pivot, not with the pixel value; where its per-lag error model (a 4-sigma bound, loose for a
    9216-pixel toy) cannot vouch for 1e-7 the lag is re-evaluated in FP64 and carries the FP64 kernel's bits."""
    pair = _rewrite_small(toy_pair, tmp_path, kind, HARD_IMAGES[kind])
    gpu, a = _gpu_cube(pair, arithmetic=arithmetic, **LAGS)
    ref, _ = _oracle_cube(pair, **LAGS)
    err = _assert_parity(gpu, ref)
    assert err < 1e-9 if arithmetic == "fp64" else err <= R_TOL
    if arithmetic == "mixed":
        assert a.engine.small32 is not None
        f64, _ = _gpu_cube(pair, arithmetic="fp64", **LAGS)
        flagged = a.engine.flagged_lags
        if kind in ("low_contrast", "quantised"):
            assert flagged == gpu.size and np.array_equal(gpu, f64)     # guard tripped everywhere: FP64 bits
        else:
            assert flagged == 0 and not np.array_equal(gpu, f64) and np.nanmax(np.abs(gpu - f64)) < 1e-7


def test_mixed_kernel_on_low_contrast_image_at_full_size(torch_cuda, config1_pair, tmp_path):
    """BASELINE configs[0] with the small image rescaled to mean 3e4, sigma 1 (float32 ulp of a pixel value = 2e-3
    sigma): with 4e6 samples per lag the mixed kernel's error model stays under 1e-7, no lag is flagged, and the whole
    3600-lag cube agrees with the all-FP64 kernel to 1e-7 -- whose own distance to the oracle is checked on a
    bounded sample of lags."""
    import os
    import bench
    from euispice_coreg_b200.hdrshift import Alignment
    from oracle.hpc import HpcSearch, cube_multiprocess
    pair = _rewrite_small(config1_pair, tmp_path, "cfg1_low_contrast", HARD_IMAGES["low_contrast"])
    cubes = {}
    for arith in ("fp64", "mixed"):
        a = Alignment(pair[0], pair[1], parallelism=True, arithmetic=arith, **bench.LAGS)
        cubes[arith] = a.align_using_helioprojective(return_type="corr").ravel()
        assert a.engine.flagged_lags == 0 and (a.engine.small32 is not None) == (arith == "mixed")
    d = np.abs(cubes["mixed"] - cubes["fp64"])
    assert np.nanmax(d) < 1e-7, np.nanmax(d)
    assert int(np.nanargmax(cubes["mixed"])) == int(np.nanargmax(cubes["fp64"])) == 54 * 60 + 36
    dl, hl, ds, hs = load_pair(*pair)
    sel = np.array([0, 3599, 54 * 60 + 36, 1000, 2500, 59])
    ref = cube_multiprocess(HpcSearch(dl, hl, ds, hs, **bench.LAGS), max(1, min(len(sel), len(os.sched_getaffinity(0)))),
                            sel)
    assert np.max(np.abs(cubes["fp64"][sel] - ref)) < 1e-9
    assert np.max(np.abs(cubes["mixed"][sel] - ref)) <= 1e-7


def test_host_buffer_entry_point_matches_device_path(torch_cuda, toy_pair):
    """coreg_hpc_search_host (the non-Python caller's entry) == the torch-plumbed path, bit for bit."""
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._compat.wcs import TanWcs
    from euispice_coreg_b200.hdrshift import engine
    gpu, a = _gpu_cube(toy_pair, arithmetic="fp64", **LAGS)
    dl, hl, ds, hs = load_pair(*toy_pair[:2])
    d = engine.flat_lag_grid(LAGS["lag_crval1"], LAGS["lag_crval2"], [0.0], [0.0], [0.0])
    w_small = TanWcs.from_header(a.hdr_small)
    table, _ = engine.tan_wcs_table(a.hdr_small, a, *d)
    flags = _ext.make_flags(variant=1)    # 16 rows per thread: what the engine launches for a pure CRVAL lag grid
    corr, nvalid = _ext.hpc_search_host(dl.astype(np.float64), TanWcs.from_header(hl), ds.astype(np.float64), w_small,
                                        table, flags=flags)
    assert np.array_equal(corr.reshape(gpu.shape), gpu)
    assert np.array_equal(nvalid.reshape(a.nvalid.shape), a.nvalid)
    # float32 payloads (what FITS BITPIX -32 files hold) go up as they are: same bits
    assert dl.dtype == np.float32 and ds.dtype == np.float32
    corr32, _ = _ext.hpc_search_host(dl, TanWcs.from_header(hl), ds, w_small, table, flags=flags)
    assert np.array_equal(corr32, corr)
    # the generic kernel from the same candidate headers (lag constants derived on the device)
    corr_g, nv_g = _ext.hpc_search_host(dl, TanWcs.from_header(hl), ds, w_small, table,
                                        flags=_ext.make_flags(no_fast=True))
    assert np.nanmax(np.abs(corr_g - corr)) < 1e-11 and np.array_equal(nv_g, nvalid)
    # mixed arithmetic through the same entry (COREG_FLAG_MIXED, float32 payload; 16 rows per thread is what the
    # engine launches for pure CRVAL lags) == the torch-plumbed default path, bit for bit
    gpu_m, a_m = _gpu_cube(toy_pair, arithmetic="mixed", **LAGS)
    corr_m, nv_m = _ext.hpc_search_host(dl, TanWcs.from_header(hl), ds, w_small, table,
                                        flags=_ext.make_flags(variant=1) | _ext.FLAG_MIXED)
    assert np.array_equal(corr_m.reshape(gpu_m.shape), gpu_m) and np.array_equal(nv_m, nvalid)
    assert not np.array_equal(corr_m, corr) and np.nanmax(np.abs(corr_m - corr)) < OBSERVED["mixed"]
    # a float64 payload has no float32 twin on this entry: the flag is ignored, FP64 kernel
    corr_d, _ = _ext.hpc_search_host(dl, TanWcs.from_header(hl), ds.astype(np.float64), w_small, table,
                                     flags=flags | _ext.FLAG_MIXED)
    assert np.array_equal(corr_d, corr)


def test_multi_device_host_entry_point_gives_the_same_cube(torch_cuda, toy_pair):
    """coreg_hpc_search_host_multi: one host thread per listed device, contiguous slices of the lag list, slices
    gathered in the host buffer. Listing the one GPU of the test box three times exercises the slicing and the
    threads; the cube has the bits of the single-device entry (it does for any device list)."""
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._compat.wcs import TanWcs
    from euispice_coreg_b200.hdrshift import engine
    gpu, a = _gpu_cube(toy_pair, arithmetic="fp64", **LAGS)
    dl, hl, ds, hs = load_pair(*toy_pair[:2])
    d = engine.flat_lag_grid(LAGS["lag_crval1"], LAGS["lag_crval2"], [0.0], [0.0], [0.0])
    w_small = TanWcs.from_header(a.hdr_small)
    table, _ = engine.tan_wcs_table(a.hdr_small, a, *d)
    flags = _ext.make_flags(variant=1)
    one, nv_one = _ext.hpc_search_host(dl, TanWcs.from_header(hl), ds, w_small, table, flags=flags)
    n_dev = torch_cuda.cuda.device_count()
    for devices in ([0, 0, 0], list(range(n_dev)), [0] * 30):      # 30 devices for 25 lags: empty slices
        corr, nvalid = _ext.hpc_search_host_multi(devices, dl, TanWcs.from_header(hl), ds, w_small, table, flags=flags)
        assert np.array_equal(corr, one, equal_nan=True) and np.array_equal(nvalid, nv_one)
    assert np.array_equal(one.reshape(gpu.shape), gpu)
    with pytest.raises(_ext.CoregLibraryError):
        _ext.hpc_search_host_multi([99], dl, TanWcs.from_header(hl), ds, w_small, table, flags=flags)


def test_results_and_written_header_match_oracle_cube(torch_cuda, toy_pair, tmp_path):
    """Parity policy of SURVEY 8c(iii): both cubes through the same host post-processing."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.hdrshift import Alignment, AlignmentResults
    a = Alignment(toy_pair[0], toy_pair[1], parallelism=True, **LAGS)
    res = a.align_using_helioprojective()
    ref, _ = _oracle_cube(toy_pair, **LAGS)
    res_o = AlignmentResults(corr=ref, lag_crval1=LAGS["lag_crval1"], lag_crval2=LAGS["lag_crval2"], lag_cdelt1=[0],
                             lag_cdelt2=[0], lag_crota=[0], unit_lag="arcsec", image_to_align_path=toy_pair[1],
                             image_to_align_window=-1)
    assert res.max_index == res_o.max_index
    assert np.max(np.abs(np.array(res.shift_arcsec) - np.array(res_o.shift_arcsec))) <= 1e-6
    out = str(tmp_path / "l3.fits")
    out_o = str(tmp_path / "l3_o.fits")
    res.write_corrected_fits([-1], out)
    res_o.write_corrected_fits([-1], out_o)
    h, ho = fits_lite.open(out)[0].header, fits_lite.open(out_o)[0].header
    for k in ("CRVAL1", "CRVAL2", "CDELT1", "CDELT2", "PC1_1", "PC1_2", "PC2_1", "PC2_2", "CROTA"):
        assert abs(h[k] - ho[k]) <= 1e-6, k
    h0 = fits_lite.open(toy_pair[1])[0].header
    assert abs(h["CRVAL1"] - h0["CRVAL1"] - 24.0) < 0.5 and abs(h["CRVAL2"] - h0["CRVAL2"] - 6.0) < 0.5
    # arg-max-lag header (the ValueError fallback of AlignmentResults.py:323-341) is bit-exact by construction
    assert LAGS["lag_crval1"][res.max_index[0]] == LAGS["lag_crval1"][res_o.max_index[0]]


@ARITH
def test_determinism_and_lag_sharding_invariance(torch_cuda, toy_pair, arithmetic):
    """Same bits run to run, and the same bits whether the lag list is evaluated whole or in slices
    (what makes the cube independent of the GPU count)."""
    from euispice_coreg_b200.hdrshift import engine
    gpu, a = _gpu_cube(toy_pair, arithmetic=arithmetic, **LAGS)
    gpu2, _ = _gpu_cube(toy_pair, arithmetic=arithmetic, **LAGS)
    assert np.array_equal(gpu, gpu2)
    eng = a.engine
    d = engine.flat_lag_grid(LAGS["lag_crval1"], LAGS["lag_crval2"], [0.0], [0.0], [0.0])
    table, _ = eng.hpc_lag_table(a.hdr_small, a, *d)
    assert table.shape[1] == 11     # candidate-header rows: the homography kernel is the default path
    parts = [eng.search(table[lo:hi]) for lo, hi in ((0, 7), (7, 8), (8, 25))]
    assert np.array_equal(np.concatenate(parts), gpu.ravel())
    # the generic kernel (separate world-coordinate planes + trig per lag) agrees far inside the tolerance
    eng_g = engine.LagSearchEngine(order=2, no_fast=True)
    eng_g.set_small(eng.small.cpu().numpy())
    eng_g.ref, eng_g.frame, eng_g.grid_wcs, eng_g.pivots = eng.ref, "hpc", eng.grid_wcs, eng.pivots
    eng_g.alpha_ref_deg, eng_g.delta_ref_deg = eng.alpha_ref_deg, eng.delta_ref_deg
    table_g, _ = eng_g.hpc_lag_table(a.hdr_small, a, *d)
    assert table_g.shape[1] == 10
    assert np.nanmax(np.abs(eng_g.search(table_g) - gpu.ravel())) < (1e-11 if arithmetic == "fp64" else OBSERVED["mixed"])


_CFG1_REF = {}


@ARITH
def test_config1_full_size_bounded_sample_vs_oracle(torch_cuda, config1_pair, arithmetic):
    """BASELINE.json configs[0] at full size (2048^2 vs 3072^2, 60x60 CRVAL lags): the whole GPU cube through the
    public API against the oracle on a bounded sample of lags (the oracle needs ~5 s per lag per core).

    The lag (0, 0) is the known knife edge (DESIGN.md section 4): the candidate header equals the grid's own header,
    every pixel maps onto itself to ~1e-11 px, and whether the four border rows / columns pass map_coordinates'
    closed bound [0, n-1] is decided by the last bits of the pixel->world->pixel round trip -- in the reference too.
    There only the membership of border pixels may differ: |dr| < 1e-3 and at most two border rows + columns."""
    import os
    import bench
    from euispice_coreg_b200.hdrshift import Alignment
    from oracle.hpc import HpcSearch, cube_multiprocess
    pl, ps = config1_pair
    a = Alignment(pl, ps, parallelism=True, arithmetic=arithmetic, **bench.LAGS)
    cube = a.align_using_helioprojective(return_type="corr")
    assert cube.shape == (60, 60, 1, 1, 1, 1)
    assert (a.engine.small32 is not None) == (arithmetic == "mixed")
    gpu = cube.ravel()
    nvalid = a.nvalid.ravel()
    dl, hl, ds, hs = load_pair(pl, ps)
    search = HpcSearch(dl, hl, ds, hs, **bench.LAGS)
    zero = 30 * 60 + 30
    sel = np.array([0, 59, 3540, 3599, 54 * 60 + 36, 1000, 2500, zero])   # corners, the peak (24, 6), interior, (0, 0)
    assert bench.LAGS["lag_crval1"][30] == 0.0
    cores = max(1, min(len(sel), len(os.sched_getaffinity(0))))
    if "ref" not in _CFG1_REF:       # the oracle sample is the slow part: once for both arithmetic modes
        _CFG1_REF["ref"] = cube_multiprocess(search, cores, sel)
    ref = _CFG1_REF["ref"]
    err = np.abs(gpu[sel] - ref)
    assert np.all(err[:-1] <= R_TOL), err
    assert err[:-1].max() < OBSERVED[arithmetic]
    assert err[-1] < 1e-3 and 2048 * 2048 - nvalid[zero] <= 2 * (2048 + 2048)
    assert int(np.nanargmax(gpu)) == 54 * 60 + 36


@pytest.fixture(scope="module")
def wide_pair(tmp_path_factory):
    """A wide-field toy pair (small image 96 px x 300 arcsec = 8 deg): shifts of degrees make the projective
    denominator of the homography leave the ranges of the two reciprocal series."""
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    d = tmp_path_factory.mktemp("wide")
    spec = small_spec(96, 160, small_cdelt=300.0, true_crval=(-3000.0, 2000.0), true_shift=(2400.0, 600.0))
    return make_pair(str(d), spec, tag="wide")


@ARITH
def test_hpc_cube_parity_all_three_reciprocal_modes(torch_cuda, wide_pair, arithmetic):
    """Per lag the rolling kernel picks 1 + e + e^2 (|e| <= 2^-18), the three-factor product (|e| <= 2^-7) or a true
    division from the exact range of e = 1 - D over the grid. One cube that needs all three, against the oracle."""
    import torch
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200.hdrshift import engine
    # (no exact (0, 0, 0) lag: that one is the closed-bound knife edge of DESIGN.md section 4)
    kw = dict(lag_crval1=np.array([0.5, 3.0, 600.0, 2400.0, 9000.0, 30000.0]), lag_crval2=np.array([0.0, 600.0, -20000.0]),
              lag_cdelt1=None, lag_cdelt2=None, lag_crota=[0.0, 2.0])
    gpu, a = _gpu_cube(wide_pair, arithmetic=arithmetic, **kw)
    ref, _ = _oracle_cube(wide_pair, **kw)
    _assert_parity(gpu, ref)
    # which series each lag got: e_max of the device-built homographies
    d = engine.flat_lag_grid(kw["lag_crval1"], kw["lag_crval2"], [0.0], [0.0], kw["lag_crota"])
    table, _ = a.engine.hpc_lag_table(a.hdr_small, a, *d)
    emax = _ext.homography_emax(a.engine.grid_wcs, torch.from_numpy(table).cuda(), a.engine.ref.shape[1],
                                a.engine.ref.shape[0]).cpu().numpy()
    modes = np.where(emax <= 2.0 ** -18, 0, np.where(emax <= 2.0 ** -7, 1, 2))
    assert set(modes.tolist()) == {0, 1, 2}, (emax.min(), emax.max())
    # and the generic kernel (per-lag trig, true division everywhere) agrees with all of them
    gen, _ = _gpu_cube(wide_pair, strict_arithmetic=True, **kw)
    assert np.nanmax(np.abs(gen - gpu)) < (1e-9 if arithmetic == "fp64" else OBSERVED["mixed"])


def test_small_image_with_holes_and_all_nan(torch_cuda, toy_pair, tmp_path):
    """NaN holes in the small image (segments with a non-finite sample leave the rolling path) and the
    reference's ValueError when the thresholds mask everything (alignment.py:656)."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.hdrshift import Alignment
    hd = fits_lite.open(toy_pair[1])[0]
    data = hd.data.copy()
    rng = np.random.default_rng(5)
    data[rng.integers(0, data.shape[0], 40), rng.integers(0, data.shape[1], 40)] = np.nan
    data[30:34, 10:50] = np.inf
    p = str(tmp_path / "holes_small.fits")
    fits_lite.writeto(p, [fits_lite.PrimaryHDU(data, hd.header)], overwrite=True)
    pair = (toy_pair[0], p)
    gpu, _ = _gpu_cube(pair, **LAGS)
    ref, _ = _oracle_cube(pair, **LAGS)
    _assert_parity(gpu, ref)
    with pytest.raises(ValueError):
        Alignment(toy_pair[0], toy_pair[1], small_fov_value_min=1e30, **LAGS).align_using_helioprojective()


def test_single_lag_and_tiny_images(torch_cuda, tmp_path):
    """One lag; images too small for the fast kernels (2 x 3 pixels) fall back to the generic kernel."""
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    one = dict(lag_crval1=[24.0], lag_crval2=[6.0], lag_cdelt1=[0], lag_cdelt2=[0], lag_crota=[0])
    pair = make_pair(str(tmp_path), small_spec(40, 64, true_crval=(-12.0, 8.0)), tag="one")
    gpu, _ = _gpu_cube(pair, **one)
    ref, _ = _oracle_cube(pair, **one)
    assert gpu.shape == (1, 1, 1, 1, 1, 1) and abs(gpu.item() - ref.item()) <= R_TOL


def test_config1_full_size_properties(torch_cuda, config1_pair):
    """Size-independent properties at BASELINE's full size (2048^2, 3600 lags), where the oracle is too slow to
    check every lag: (1) the cube does not depend on how the lag list is sliced or ordered (bitwise); (2) Pearson's
    r is invariant under a positive affine map of the small image -- scaling by 2 is exact in binary floating
    point, so the cube must not change by a single bit; a general map moves it only by rounding; (3) every r lies
    in [-1, 1] and the number of valid pixels decreases away from the zero lag."""
    import bench
    from euispice_coreg_b200._compat.wcs import TanWcs
    from euispice_coreg_b200.hdrshift import Alignment, engine
    pl, ps = config1_pair
    a = Alignment(pl, ps, parallelism=True, **bench.LAGS)
    cube = a.align_using_helioprojective(return_type="corr").ravel()
    eng = a.engine
    d = engine.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
    table, _ = eng.hpc_lag_table(a.hdr_small, a, *d)
    # (1) slices and a permutation
    parts = [eng.search(table[lo:hi]) for lo, hi in ((0, 1), (1, 1237), (1237, 3600))]
    assert np.array_equal(np.concatenate(parts), cube)
    perm = np.random.default_rng(0).permutation(table.shape[0])
    assert np.array_equal(eng.search(table[perm]), cube[perm])
    # (3)
    assert np.all(np.abs(cube) <= 1.0)
    nv = a.nvalid.reshape(60, 60)
    assert nv[30, 30] == nv.max() and nv[0, 0] < nv[15, 15] < nv[30, 30]
    # (2)
    small = eng.small.clone()
    piv = eng.pivots.clone()
    eng.set_small((small * 2.0).cpu().numpy())
    assert np.array_equal(eng.search(table), cube)
    eng.set_small((small * 3.0 + 100.0).cpu().numpy())
    # (3 a + 100 is not a float32 image any more: this search runs the all-FP64 kernel, `cube` came from the mixed
    # one -- rounding of the map + the difference between the two arithmetic modes, ~1e-9)
    assert np.max(np.abs(eng.search(table) - cube)) < 1e-8
    eng.small, eng.pivots = small, piv


def test_coarse_to_fine_search_equals_dense_where_evaluated(torch_cuda, toy_pair):
    """lag_search="coarse_to_fine" (SURVEY 8f-3): same arg-max and same fitted shift as the dense search from a
    fraction of the lags; every evaluated entry has the dense cube's bits, the rest is NaN."""
    from euispice_coreg_b200.hdrshift import Alignment
    lags = dict(lag_crval1=np.arange(4, 45, 1.0), lag_crval2=np.arange(-14, 27, 1.0), lag_cdelt1=[0], lag_cdelt2=[0],
                lag_crota=[0.0, 0.5])
    dense = Alignment(toy_pair[0], toy_pair[1], parallelism=True, **lags)
    rd = dense.align_using_helioprojective()
    c2f = Alignment(toy_pair[0], toy_pair[1], parallelism=True, lag_search="coarse_to_fine", **lags)
    rc = c2f.align_using_helioprojective()
    ev = ~np.isnan(rc.corr)
    assert c2f.lags_evaluated == ev.sum() < 0.35 * rd.corr.size and dense.lags_evaluated == rd.corr.size
    assert np.array_equal(rc.corr[ev], rd.corr[ev])
    assert rc.max_index == rd.max_index and rc.shift_arcsec == rd.shift_arcsec
    with pytest.raises(ValueError):
        Alignment(toy_pair[0], toy_pair[1], lag_search="pyramid", **lags)


def test_adaptive_segment_rotated_rescaled_lags_with_holes(torch_cuda, tmp_path):
    """Rotated / rescaled candidate headers make column segments drift off the one-row-per-row lattice; a warp with such a
    lane takes the rolling kernel's ADAPTIVE segment (every pixel its own floors, csrc/coreg_lag_roll.cu). A grid large
    enough to have interior warps (448 x 448: the toy pairs are all rim), NaN holes in the small image (an adaptive
    segment that meets a non-finite sample is redone pixel by pixel), against the oracle; and against the kernel flavour
    WITHOUT the adaptive code (variant 1), which evaluates the same lags by the per-pixel rules."""
    import torch
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    from euispice_coreg_b200.hdrshift import engine
    pair = make_pair(str(tmp_path), small_spec(448, 512, true_crval=(-12.0, 8.0), master_n=1024), tag="adapt")
    hd = fits_lite.open(pair[1])[0]
    data = hd.data.copy()
    rng = np.random.default_rng(11)
    data[rng.integers(0, 448, 25), rng.integers(0, 448, 25)] = np.nan
    p = str(tmp_path / "adapt_holes_small.fits")
    fits_lite.writeto(p, [fits_lite.PrimaryHDU(data, hd.header)], overwrite=True)
    pair = (pair[0], p)
    cd = float(hd.header["CDELT1"])
    kw = dict(lag_crval1=np.array([22.0, 24.0, 27.0]), lag_crval2=np.array([6.0]), lag_crota=[-0.4, 0.3],
              lag_cdelt1=[-0.016 * cd, 0.009 * cd], lag_cdelt2=[-0.012 * cd, 0.015 * cd], cdelt_semantics="intended")
    gpu, a = _gpu_cube(pair, **kw)
    assert gpu.size == 24 and not a.engine.pure_shift_hint
    ref, _ = _oracle_cube(pair, **kw)
    err = _assert_parity(gpu, ref)
    assert err < OBSERVED["fp64"]
    # the same lags through the flavour without the adaptive segment, and through the generic kernel
    d = engine.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
    table, _ = a.engine.hpc_lag_table(a.hdr_small, a, *d, "intended")
    c0, n0 = a.engine.search(table, return_nvalid=True)
    assert np.array_equal(c0, gpu.ravel())
    a.engine.variant, a.engine.flags = 1, _ext.make_flags(variant=1)
    c1, n1 = a.engine.search(table, return_nvalid=True)
    # (the float32 store of every sample hides the different FP64 operation order of the two paths: the cubes usually
    # agree to the last bit)
    assert np.array_equal(n0, n1) and np.max(np.abs(c0 - c1)) < 1e-12
    gen, _ = _gpu_cube(pair, strict_arithmetic=True, **kw)
    assert np.nanmax(np.abs(gen - gpu)) < 1e-9
