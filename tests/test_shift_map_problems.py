"""Host side of the per-block shift maps: `gaussian_fit_problems` poses exactly the fits `AlignmentResults._compute_shift`
hands to scipy's `curve_fit`, and predicts which of them `curve_fit` refuses; the shift map of blocks that need no fit;
the C entry's argument checks; the argument checks of `SequenceAlignment.align_using_helioprojective(local_block=...)`.
No device needed."""
import ctypes
import importlib
import warnings

import numpy as np
import pytest

AR = importlib.import_module("euispice_coreg_b200.hdrshift.AlignmentResults")   # the module, not the class

FAILED = ("Gaussian fitting failed", "Cannot compute shift")


def _lags(shape):
    n1, n2, n3, n4, n5 = shape[:5]
    return dict(lag_crval1=np.linspace(-10, 10, n1), lag_crval2=np.linspace(5, 17, n2), lag_cdelt1=np.arange(n3) * 0.1,
                lag_cdelt2=np.arange(n4) * 0.2, lag_crota=np.arange(n5) * 0.5, unit_lag="arcsec")


def _host_fit(monkeypatch, cube):
    """AlignmentResults of one cube with curve_fit recorded -> (results, record or None, warned)."""
    calls = []
    real = AR.curve_fit

    def spy(f, xdata, ydata, p0, bounds):
        calls.append(dict(xdata=xdata, ydata=ydata, p0=p0, bounds=bounds))
        return real(f=f, xdata=xdata, ydata=ydata, p0=p0, bounds=bounds)

    monkeypatch.setattr(AR, "curve_fit", spy)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        res = AR.AlignmentResults(corr=cube, **_lags(cube.shape))
    warned = any(str(m.message).strip().startswith(FAILED) for m in w)
    assert len(calls) <= 1
    return res, (calls[0] if calls else None), warned


def _peak_cube(shape, peak, seed=0, value=0.9):
    """A Gaussian bump at `peak` in its CRVAL plane over a low noisy floor, with the maximum `value` at `peak`."""
    rng = np.random.default_rng(seed)
    cube = rng.uniform(0.0, 0.05, shape) + value - 0.6
    i, j = np.meshgrid(np.arange(shape[0]), np.arange(shape[1]), indexing="ij")
    plane = (slice(None), slice(None)) + tuple(peak[2:])
    cube[plane] += 0.5 * np.exp(-((i - peak[0] - 0.3) ** 2 + (j - peak[1] + 0.2) ** 2) / (2 * 1.6 ** 2))
    cube[peak] = value
    return cube


def _cases():
    out = []
    n1, n2 = 6, 7
    for i in (0, 1, n1 - 2, n1 - 1):
        for j in (0, 1, n2 - 2, n2 - 1):
            out.append((f"peak {i},{j}", _peak_cube((n1, n2, 1, 1, 1, 1), (i, j, 0, 0, 0, 0), seed=i * 10 + j)))
    out.append(("2x2", _peak_cube((2, 2, 1, 1, 1, 1), (1, 0, 0, 0, 0, 0))))
    out.append(("2x2 at 0", _peak_cube((2, 2, 1, 1, 1, 1), (0, 0, 0, 0, 0, 0))))
    out.append(("3x60", _peak_cube((3, 60, 1, 1, 1, 1), (1, 31, 0, 0, 0, 0))))
    out.append(("3x60 edge", _peak_cube((3, 60, 1, 1, 1, 1), (0, 59, 0, 0, 0, 0))))
    nan_nb = _peak_cube((6, 6, 1, 1, 1, 1), (3, 3, 0, 0, 0, 0))
    nan_nb[4, 2] = np.nan
    out.append(("NaN neighbour", nan_nb))
    far_nan = _peak_cube((8, 8, 1, 1, 1, 1), (5, 5, 0, 0, 0, 0))
    far_nan[0, 0] = np.nan              # outside the 5 x 5 window: the fit still runs
    out.append(("NaN outside the window", far_nan))
    wrap_nan = _peak_cube((8, 8, 1, 1, 1, 1), (0, 3, 0, 0, 0, 0))
    wrap_nan[6, 3] = np.nan             # read through the -2 wrap of the peak at row 0
    out.append(("NaN behind the wrap", wrap_nan))
    out.append(("all negative", _peak_cube((6, 6, 1, 1, 1, 1), (2, 2, 0, 0, 0, 0), value=-0.01)))
    out.append(("CDELT / CROTA axes", _peak_cube((7, 6, 3, 2, 4, 1), (3, 2, 2, 1, 3, 0))))
    out.append(("CDELT / CROTA axes, edge", _peak_cube((7, 6, 2, 3, 2, 1), (6, 0, 1, 2, 1, 0))))
    hpc = np.repeat(_peak_cube((20, 20, 1, 1, 1, 1), (9, 11, 0, 0, 0, 0)), 2, axis=5)
    out.append(("solar radius repeated", hpc))
    return out


@pytest.mark.parametrize("name,cube", _cases(), ids=[c[0] for c in _cases()])
def test_problems_are_the_fits_compute_shift_poses(monkeypatch, name, cube):
    res, rec, warned = _host_fit(monkeypatch, cube)
    mi = np.asarray(res.max_index)
    prob = AR.gaussian_fit_problems(cube, mi)
    npts = int(prob.npts[0])
    assert rec is not None and npts >= 4
    x, y = rec["xdata"]
    assert np.array_equal(x, prob.points[0, :npts, 0]) and np.array_equal(y, prob.points[0, :npts, 1])
    assert np.array_equal(prob.ix[0, :npts], x.astype(np.int64))
    assert (prob.points[0, npts:] == 0).all()
    n_r = cube.shape[5]
    if n_r == 1:
        assert np.array_equal(rec["ydata"], prob.points[0, :npts, 2], equal_nan=True)
    else:
        assert rec["ydata"].size == npts * n_r
        assert np.array_equal(rec["ydata"].reshape(npts, n_r)[:, 0], prob.points[0, :npts, 2], equal_nan=True)
    assert np.array_equal(np.asarray(rec["p0"], dtype=np.float64), prob.p0[0])
    assert np.array_equal(np.concatenate([np.asarray(b, dtype=np.float64) for b in rec["bounds"]]), prob.bounds[0])
    # the maximum is listed twice, and offsets of -2 keep their coordinate
    assert (x[0], y[0]) == (mi[0], mi[1]) and ((x == mi[0]) & (y == mi[1])).sum() == 2
    assert (prob.decision[0] == AR.FIT) == (not warned)
    assert prob.decision[0] in (AR.FIT, AR.ARGMAX_FALLBACK)
    if name in ("NaN neighbour", "NaN behind the wrap", "all negative", "solar radius repeated"):
        assert prob.decision[0] == AR.ARGMAX_FALLBACK
    if name.startswith("peak 0") or name in ("2x2 at 0", "3x60 edge"):
        assert (prob.points[0, :npts, 0] == -2).any() or (prob.points[0, :npts, 1] == -2).any()


@pytest.mark.parametrize("shape", [(1, 1), (1, 3), (3, 1)])
def test_a_lag_axis_of_one_raises_as_compute_shift_does(monkeypatch, shape):
    cube = _peak_cube(shape + (1, 1, 1, 1), (0, 0, 0, 0, 0, 0))
    with pytest.raises(IndexError):
        _host_fit(monkeypatch, cube)
    mi = np.zeros(6, dtype=np.int64)
    with pytest.raises(IndexError):
        AR.gaussian_fit_problems(cube, mi)


def test_a_stack_gives_each_cube_its_own_problem():
    cases = [c for _, c in _cases() if c.shape == (6, 6, 1, 1, 1, 1)]
    stack = np.stack(cases).reshape((len(cases) // 1, 1) + cases[0].shape)
    mi = np.array([np.unravel_index(np.nanargmax(c), c.shape) for c in cases]).reshape(len(cases), 1, 6)
    mi[0, 0] = -1               # a block that is NaN at every lag
    stack[0, 0] = np.nan
    both = AR.gaussian_fit_problems(stack, mi)
    assert both.decision.shape == (len(cases),) and both.decision[0] == AR.NO_MAXIMUM and both.npts[0] == 0
    for k in range(1, len(cases)):
        one = AR.gaussian_fit_problems(cases[k], mi[k, 0])
        for f in ("ix", "iy", "npts", "p0", "bounds", "decision"):
            assert np.array_equal(getattr(both, f)[k], getattr(one, f)[0]), f
        assert np.array_equal(both.points[k], one.points[0], equal_nan=True)


def _local(corr):
    nb = corr.shape[:2]
    return AR.LocalAlignmentResults(corr, np.ones(corr.shape[:-1], dtype=np.int64), np.zeros(nb + (4,), np.int64),
                                    **_lags(corr.shape[2:]), image_to_align_path=None, image_to_align_window=None,
                                    reference_image_path=None, reference_image_window=None)


def test_shift_map_of_blocks_without_a_fit_needs_no_device():
    """Fallback and empty blocks are decided on the host: no launch, the arg-max lags of `results(i, j)`, NaN."""
    shape = (6, 6, 2, 1, 3, 1)
    corr = np.stack([np.stack([_peak_cube(shape, (2, 3, 1, 0, 2, 0), seed=1, value=-0.01),
                               _peak_cube(shape, (0, 5, 0, 0, 1, 0), seed=2)])])
    corr[0, 1, 1, 4, 0, 0, 1, 0] = np.nan       # a NaN in the fit set of block (0, 1)
    corr = np.concatenate([corr, np.full_like(corr, np.nan)])
    loc = _local(corr)
    assert loc.fit_status.dtype == np.int8
    assert loc.fit_status.tolist() == [[AR.ARGMAX_FALLBACK] * 2, [AR.NO_MAXIMUM] * 2]
    for j in range(2):
        r = loc.results(0, j)
        assert np.array_equal(loc.shift_arcsec[0, j], np.array(r.shift_arcsec, dtype=np.float64))
        assert np.array_equal(loc.shift_pixels[0, j], np.array(r.shift_pixels, dtype=np.float64))
    assert np.isnan(loc.shift_arcsec[1]).all() and np.isnan(loc.shift_pixels[1]).all()


def test_shift_map_with_fits_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from euispice_coreg_b200 import _ext
    loc = _local(_peak_cube((8, 8, 1, 1, 1, 1), (4, 4, 0, 0, 0, 0))[None, None])
    with pytest.raises(_ext.CoregLibraryError):
        loc.shift_arcsec


def test_fit_entry_rejects_bad_arguments_without_a_device():
    from euispice_coreg_b200 import _ext
    lib = _ext.load()
    fake, null = ctypes.c_void_p(0x1000), None
    rc = lib.coreg_gauss2d_fit(fake, fake, fake, fake, -1, fake, fake, fake, fake, null)
    assert rc == -1 and "n_problems" in lib.coreg_last_error().decode()
    rc = lib.coreg_gauss2d_fit(fake, null, fake, fake, 4, fake, fake, fake, fake, null)
    assert rc == -1 and "null pointer" in lib.coreg_last_error().decode()
    assert lib.coreg_gauss2d_fit(fake, fake, fake, fake, 0, fake, fake, fake, fake, null) == 0   # nothing to launch


def test_sequence_helioprojective_blocks_are_checked_before_any_device_work(monkeypatch):
    from euispice_coreg_b200.hdrshift import SequenceAlignment
    lags = dict(lag_crval1=[0.0, 1.0], lag_crval2=[0.0, 1.0])
    seq = SequenceAlignment("missing_large.fits", ["missing_small.fits"], **lags)
    with pytest.raises(ValueError, match='return_type="AlignmentResults"'):
        seq.align_using_helioprojective(return_type="corr", local_block=64)
    with pytest.raises(ValueError, match="multiples of 64"):
        seq.align_using_helioprojective(local_block=(64, 96))
    with pytest.raises(ValueError, match="FP64"):
        SequenceAlignment("missing_large.fits", ["missing_small.fits"], arithmetic="mixed",
                          **lags).align_using_helioprojective(local_block=64)
    monkeypatch.setenv("COREG_ARITHMETIC", "mixed")
    with pytest.raises(ValueError, match="FP64"):
        seq.align_using_helioprojective(local_block=64)
