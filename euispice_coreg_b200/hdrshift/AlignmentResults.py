"""`AlignmentResults` -- host post-processing of the correlation cube, same API and arithmetic as the
reference's `hdrshift/AlignmentResults.py:25-341`: arg-max (first occurrence, C order), a bounded
2-D Gaussian `curve_fit` on the <= 5x5 neighbourhood of the maximum in the (CRVAL1, CRVAL2) plane, and
linear interpolation of the fitted sub-index centre back into the lag arrays. The whole-grid fit is
numpy/scipy, pinned by the reference's own golden cube (`hdrshift/test/test_AlignmentResults.py:35-126,
172-173`); the shift maps of `LocalAlignmentResults` pose the same fits (`gaussian_fit_problems`) and run them
in one batched device launch (`coreg_gauss2d_fit`).
"""
from __future__ import annotations

import warnings

import numpy as np
from scipy.optimize import curve_fit

from .._compat import units
from ..utils.Util import AlignCommonUtil, _fits


def twoD_Gaussian(xy, amplitude, xo, yo, sigma_x, sigma_y, offset):
    x, y = xy
    x0 = float(xo)
    y0 = float(yo)
    g = offset + amplitude * np.exp(
        -((((x - x0) ** 2) / (2 * sigma_x ** 2)) + (((y - y0) ** 2) / (2 * sigma_y ** 2))))
    return g.ravel()


_NEIGHBOURS = [(ii, jj) for ii in (-2, -1, 0, 1, 2) for jj in (-2, -1, 0, 1, 2)]
# the fit set: the maximum, then the 5 x 5 neighbourhood in C order (the maximum is listed twice)
_FIT_OFFSETS = np.array([(0, 0)] + _NEIGHBOURS, dtype=np.int64)
FIT_MAX_POINTS = len(_FIT_OFFSETS)      # 26

# decisions of `gaussian_fit_problems`, and the values of `LocalAlignmentResults.fit_status`
FIT, ARGMAX_FALLBACK, NO_MAXIMUM, NOT_CONVERGED = 0, 1, 2, 3


def _lag_parameters(lag_crval1, lag_crval2, lag_cdelt1, lag_cdelt2, lag_crota, unit_lag):
    """(parameters_alignment, parameters_alignment_arcsec) of `AlignmentResults`: missing lag arrays read [0]; (value
    array, unit) pairs stand in for astropy quantities."""
    zero = lambda v: np.array([0]) if v is None else v  # noqa: E731
    lag_crval1, lag_crval2 = zero(lag_crval1), zero(lag_crval2)
    lag_cdelt1, lag_cdelt2, lag_crota = zero(lag_cdelt1), zero(lag_cdelt2), zero(lag_crota)
    as_arr = lambda v: np.asarray(v, dtype=np.float64)  # noqa: E731
    native = {
        "lag_crval1": (as_arr(lag_crval1), unit_lag), "lag_crval2": (as_arr(lag_crval2), unit_lag),
        "lag_cdelt1": (as_arr(lag_cdelt1), unit_lag), "lag_cdelt2": (as_arr(lag_cdelt2), unit_lag),
        "lag_crota": (as_arr(lag_crota), "deg"),
    }
    arcsec = {
        "lag_crval1": units.convert(as_arr(lag_crval1), unit_lag, "arcsec"),
        "lag_crval2": units.convert(as_arr(lag_crval2), unit_lag, "arcsec"),
        "lag_cdelt1": units.convert(as_arr(lag_cdelt1), unit_lag, "arcsec"),
        "lag_cdelt2": units.convert(as_arr(lag_cdelt2), unit_lag, "arcsec"),
        "lag_crota": as_arr(lag_crota),
    }
    return native, arcsec


class GaussianFitProblems:
    """The sub-lag fits of a stack of cubes, as `AlignmentResults._compute_shift` poses them (`gaussian_fit_problems`).

    ix, iy    [n, 26] int64: lag indices of the fit points (the first npts of each row; -2 stays -2 and its value is
              read at the far edge, as Python indexing does)
    points    [n, 26, 3] float64: (x, y, value) of each point at solar-radius index 0; zeros past npts
    npts      [n] int32
    p0        [n, 6], bounds [n, 12] (lo then hi) float64
    decision  [n] int8: FIT, ARGMAX_FALLBACK (curve_fit would raise the ValueError `_compute_shift` catches, or fewer
              than 4 points) or NO_MAXIMUM (max_index -1: NaN at every lag)
    """

    def __init__(self, ix, iy, points, npts, p0, bounds, decision):
        self.ix, self.iy, self.points, self.npts = ix, iy, points, npts
        self.p0, self.bounds, self.decision = p0, bounds, decision


def gaussian_fit_problems(corr, max_index):
    """Point selection, start and bounds of the sub-lag Gaussian fit of each cube, and what `_compute_shift` does with
    it. corr: [..., n_crval1, n_crval2, n_cdelt1, n_cdelt2, n_crota, n_solar_r]; max_index: [..., 6] (the cube index of
    each maximum, -1 for a cube without one). The fit slice is corr[:, :, i_cdelt1, i_cdelt2, i_crota] at the maximum's
    indices; the points are the maximum, then its 5 x 5 neighbours in C order whose indices are neither -1 nor past the
    end (so -2 is kept: its value wraps to the far edge, its coordinate stays -2.0); p0 = (value at the maximum, i0, i1,
    1, 1, 0.9). A fit is predicted to fail, as scipy's `curve_fit` does with a ValueError, when a point value is not
    finite, when the maximum is negative (p0 outside the amplitude bounds [0, 10]) or when the cube has more than one
    solar-radius plane (ydata then holds n_r values per point). A -2 on a lag axis of length 1 raises the IndexError
    `_compute_shift` raises there."""
    corr = np.asarray(corr)
    n1, n2, n_r = corr.shape[-6], corr.shape[-5], corr.shape[-1]
    cubes = corr.reshape((-1,) + corr.shape[-6:])
    mi = np.asarray(max_index, dtype=np.int64).reshape(-1, 6)
    n = cubes.shape[0]
    has = mi[:, 0] >= 0
    x = mi[:, :1] + _FIT_OFFSETS[:, 0]
    y = mi[:, 1:2] + _FIT_OFFSETS[:, 1]
    keep = (x != -1) & (x < n1) & (y != -1) & (y < n2)
    keep[:, 0] = True
    keep &= has[:, None]
    order = np.argsort(~keep, axis=1, kind="stable")      # kept points first, in fit-set order
    x, y, keep = (np.take_along_axis(a, order, axis=1) for a in (x, y, keep))
    npts = keep.sum(axis=1).astype(np.int32)
    decision = np.where(has, np.where(npts < 4, ARGMAX_FALLBACK, FIT), NO_MAXIMUM).astype(np.int8)
    fitting = decision == FIT
    if (fitting[:, None] & keep & ((x < -n1) | (y < -n2))).any():
        raise IndexError(f"index -2 is out of bounds for a lag axis of size {min(n1, n2)}")
    x = np.where(keep, x, 0)
    y = np.where(keep, y, 0)
    rows = np.arange(n)[:, None]
    at = np.where(has[:, None], mi, 0)
    vals = cubes[rows, x, y, at[:, 2:3], at[:, 3:4], at[:, 4:5], 0]
    vals = np.where(keep, vals, 0.0)
    points = np.stack([x.astype(np.float64), y.astype(np.float64), vals], axis=-1)
    peak = cubes[np.arange(n), at[:, 0], at[:, 1], at[:, 2], at[:, 3], at[:, 4], 0].astype(np.float64)
    i0, i1 = at[:, 0].astype(np.float64), at[:, 1].astype(np.float64)
    one = np.ones(n)
    p0 = np.stack([peak, i0, i1, one, one, 0.9 * one], axis=-1)
    bounds = np.stack([0 * one, i0 - 5, i1 - 5, 0 * one, 0 * one, -10 * one,
                       10 * one, i0 + 5, i1 + 5, 1000 * one, 1000 * one, 10 * one], axis=-1)
    fails = (n_r > 1) | ~np.isfinite(np.where(keep, vals, 0.0)).all(axis=1) | (peak < 0)
    decision[fitting & fails] = ARGMAX_FALLBACK
    return GaussianFitProblems(x, y, points, npts, p0, bounds, decision)


class AlignmentResults:

    def __init__(self, corr, lag_crval1, lag_crval2, lag_cdelt1, lag_cdelt2, lag_crota, unit_lag: str,
                 image_to_align_path: str = None, image_to_align_window=None, reference_image_path: str = None,
                 reference_image_window: int = None):
        self.max_index = np.unravel_index(np.nanargmax(corr), corr.shape)
        self.corr = corr
        self.parameters_alignment, self.parameters_alignment_arcsec = _lag_parameters(
            lag_crval1, lag_crval2, lag_cdelt1, lag_cdelt2, lag_crota, unit_lag)
        self.image_to_align_path = image_to_align_path
        self.image_to_align_window = image_to_align_window
        self.reference_image_path = reference_image_path
        self.reference_image_window = reference_image_window
        self.unit_lag = unit_lag
        self.shift_pixels = None
        self.shift_arcsec = None
        self._compute_shift()

    # ------------------------------------------------------------------ plotting (delegated, lazy)
    def plot_correlation(self, path_save_figure: str = None, show=False, fig=None, ax=None):
        from ..plot.plot import PlotFunctions
        return PlotFunctions.plot_correlation(
            corr=self.corr, show=show, path_save_figure=path_save_figure, fig=fig, ax=ax, shift=self.shift_arcsec,
            unit_to_plot=self.unit_lag, lag_dx_label=f"CRVAL1 [{self.unit_lag}]",
            lag_dy_label=f"CRVAL2 [{self.unit_lag}]", **self.parameters_alignment_arcsec)

    def plot_co_alignment(self, path_save_figure: str = None, show=False, lonlims=None, latlims=None, **kwargs):
        from ..plot.plot import PlotFunctions
        return PlotFunctions.plot_co_alignment(
            reference_image_path=self.reference_image_path, reference_image_window=self.reference_image_window,
            image_to_align_path=self.image_to_align_path, image_to_align_window=self.image_to_align_window,
            path_save_figure=path_save_figure, shift_arcsec=self.shift_arcsec, show=show,
            unit_to_plot=self.unit_lag, lonlims=lonlims, latlims=latlims, **kwargs)

    # ------------------------------------------------------------------ writing
    def write_corrected_fits(self, window_list_to_apply_shift: list, path_to_l3_output: str,
                             path_to_l2_input: str = None):
        """FITS copy with corrected pointing keywords in the selected windows (`AlignmentResults.py:149-176`)."""
        if path_to_l2_input is None:
            if self.image_to_align_path is None:
                raise ValueError("Please provide a path_to_l2_input parameter")
            path_to_l2_input = self.image_to_align_path
        AlignCommonUtil.write_corrected_fits(
            corr=self.corr, path_to_l2_input=path_to_l2_input, path_to_l3_output=path_to_l3_output,
            window_list_to_apply_shift=window_list_to_apply_shift, shift_arcsec=self.shift_arcsec)

    def savefig(self, filename: str):
        raise NotImplementedError

    def saveyaml(self, filename: str, window: str, path_to_l2_input: str = None):
        raise NotImplementedError

    def return_corrected_header(self, window, path_to_l2_input: str = None):
        """Header of `window` with the corrected pointing (`AlignmentResults.py:187-214`)."""
        if path_to_l2_input is None:
            if self.image_to_align_path is None:
                raise ValueError("Please provide a path_to_l2_input parameter")
            path_to_l2_input = self.image_to_align_path
        with _fits().open(path_to_l2_input) as hdul:
            header = hdul[window].header.copy()
            AlignCommonUtil.correct_pointing_header(
                header, lag_crval1=self.shift_arcsec[0], lag_crval2=self.shift_arcsec[1],
                lag_cdelt1=self.shift_arcsec[2], lag_cdelt2=self.shift_arcsec[3], lag_crota=self.shift_arcsec[4])
        return header

    # ------------------------------------------------------------------ sub-lag peak
    def _argmax_shift(self):
        mi = self.max_index
        pa = self.parameters_alignment_arcsec
        self.shift_pixels = (mi[0], mi[1], mi[2], mi[3], mi[4])
        self.shift_arcsec = (pa["lag_crval1"][mi[0]], pa["lag_crval2"][mi[1]], pa["lag_cdelt1"][mi[2]],
                             pa["lag_cdelt2"][mi[3]], pa["lag_crota"][mi[4]])

    def _compute_shift(self, method="fitting_gaussian"):
        """`AlignmentResults.py:218-341`, with the fit set of `gaussian_fit_problems`. Quirks kept: the maximum is listed
        twice in the fit set, an offset of -2 below index 0 wraps around (only -1 is excluded), and solar-radius index
        0 is used."""
        mi = self.max_index
        corr2d = self.corr[:, :, mi[2], mi[3], mi[4]]
        if method != "fitting_gaussian":
            raise NotImplementedError
        prob = gaussian_fit_problems(self.corr, np.asarray(mi))
        npts = int(prob.npts[0])
        px, py = prob.ix[0, :npts], prob.iy[0, :npts]
        if npts < 4:
            warnings.warn(" Cannot compute shift with Gaussian fitting: not enough points")
            self._argmax_shift()
            return None
        A = (np.float64(px), np.float64(py))
        B = np.float64(corr2d[px, py].ravel())
        p0 = tuple(np.float64(v) for v in prob.p0[0])
        bounds = ([np.float64(v) for v in prob.bounds[0, :6]], [np.float64(v) for v in prob.bounds[0, 6:]])
        try:
            popt, _ = curve_fit(f=twoD_Gaussian, xdata=A, ydata=B, p0=p0, bounds=bounds)
        except ValueError:
            warnings.warn("Gaussian fitting failed, setting shift params as the pixel of the maximal correlation")
            self._argmax_shift()
            return None
        pa = self.parameters_alignment_arcsec
        lag_x, lag_y = pa["lag_crval1"], pa["lag_crval2"]
        shift_x = np.interp(popt[1], np.arange(len(lag_x)), lag_x)
        shift_y = np.interp(popt[2], np.arange(len(lag_y)), lag_y)
        self.shift_pixels = (popt[1], popt[2], mi[2], mi[3], mi[4])
        self.shift_arcsec = (shift_x, shift_y, pa["lag_cdelt1"][mi[2]], pa["lag_cdelt2"][mi[3]],
                             pa["lag_crota"][mi[4]])
        return True

    def __str__(self):
        s = self.shift_arcsec
        return (f"\n Shift : \n x = {s[0]} '' \n y = {s[1]} '' \n dx = {s[2]} '' "
                f"\n dy = {s[3]} '' \n dcrot = {s[4]} deg")

    __repr__ = __str__


class LocalAlignmentResults:
    """Per-block correlation cubes of one helioprojective search (`Alignment(..., local_block=...)`): the common grid
    cut into blocks from pixel (0, 0), the last block row and column taking whatever remains.

    corr       [nby, nbx, n_crval1, n_crval2, n_cdelt1, n_cdelt2, n_crota, n_solar_r] float64: Pearson r of each block's
               pixels; NaN where a block has no valid pixel pair under a lag, 0.0 for lags the reference cannot
               evaluate (as in the global cube)
    nvalid     [nby, nbx, n_crval1, ..., n_crota] int64: valid pixel pairs per block and lag (they sum to the global count)
    bounds     [nby, nbx, 4] int64: (row0, row1, col0, col1) of each block on the common grid
    max_index  [nby, nbx, 6] int64: the cube index of each block's maximum (first occurrence, C order, NaN ignored), -1
               for a block that is NaN at every lag

    The shift map, computed for all blocks together on first access (one batched fit on the CUDA device,
    `coreg_gauss2d_fit`; no CPU fallback):
    shift_pixels  [nby, nbx, 5] float64: the sub-lag indices of `results(i, j).shift_pixels`
    shift_arcsec  [nby, nbx, 5] float64: the shifts of `results(i, j).shift_arcsec`, in the same units
    fit_status    [nby, nbx] int8: FIT (0, fitted), ARGMAX_FALLBACK (1: the arg-max lags, as `results(i, j)` falls back
                  to them), NO_MAXIMUM (2) or NOT_CONVERGED (3); the shifts of the last two read NaN
    """

    def __init__(self, corr, nvalid, bounds, **results_kwargs):
        self.corr = corr
        self.nvalid = nvalid
        self.bounds = bounds
        self.max_index = np.full(corr.shape[:2] + (corr.ndim - 2,), -1, dtype=np.int64)
        flat = corr.reshape(corr.shape[:2] + (-1,))
        some = ~np.isnan(flat).all(axis=-1)
        if some.any():
            self.max_index[some] = np.stack(np.unravel_index(np.nanargmax(flat[some], axis=-1), corr.shape[2:]), -1)
        self._results_kwargs = results_kwargs
        self._shift = None

    def results(self, i, j):
        """`AlignmentResults` of block (i, j): its arg-max and Gaussian sub-lag fit, as for the whole grid."""
        return AlignmentResults(corr=self.corr[i, j], **self._results_kwargs)

    @property
    def shift_pixels(self):
        return self._shift_map()[0]

    @property
    def shift_arcsec(self):
        return self._shift_map()[1]

    @property
    def fit_status(self):
        return self._shift_map()[2]

    def _shift_map(self):
        if self._shift is None:
            self._shift = self._fit_blocks()
        return self._shift

    def _fit_blocks(self):
        """The fits of `results(i, j)` for every block at once: the problems gathered on the host, the fits of the
        blocks that get one in one device launch, the fitted sub-indices interpolated into the lag arrays as
        `_compute_shift` does."""
        from .. import _ext
        nb = self.corr.shape[:2]
        prob = gaussian_fit_problems(self.corr, self.max_index)
        status = prob.decision.copy()
        fit = np.flatnonzero(status == FIT)
        mi = self.max_index.reshape(-1, 6)
        pix = mi[:, :5].astype(np.float64)
        if fit.size:
            import torch
            _ext.load()
            if not torch.cuda.is_available():
                raise _ext.CoregLibraryError("no CUDA device: the peak fits have no CPU fallback")
            dev = torch.device("cuda", torch.cuda.current_device())
            up = lambda a: torch.from_numpy(np.ascontiguousarray(a[fit])).to(dev)  # noqa: E731
            popt, _, _, st = _ext.gauss2d_fit(up(prob.points), up(prob.npts), up(prob.p0), up(prob.bounds))
            popt, st = popt.cpu().numpy(), st.cpu().numpy()
            pix[fit, 0], pix[fit, 1] = popt[:, 1], popt[:, 2]
            status[fit[st != _ext.FIT_CONVERGED]] = NOT_CONVERGED
        kw = self._results_kwargs
        _, pa = _lag_parameters(kw.get("lag_crval1"), kw.get("lag_crval2"), kw.get("lag_cdelt1"), kw.get("lag_cdelt2"),
                                kw.get("lag_crota"), kw["unit_lag"])
        at = np.maximum(mi, 0)
        arcsec = np.stack([pa["lag_crval1"][at[:, 0]], pa["lag_crval2"][at[:, 1]], pa["lag_cdelt1"][at[:, 2]],
                           pa["lag_cdelt2"][at[:, 3]], pa["lag_crota"][at[:, 4]]], axis=-1)
        fitted = status == FIT
        lag_x, lag_y = pa["lag_crval1"], pa["lag_crval2"]
        arcsec[fitted, 0] = np.interp(pix[fitted, 0], np.arange(len(lag_x)), lag_x)
        arcsec[fitted, 1] = np.interp(pix[fitted, 1], np.arange(len(lag_y)), lag_y)
        lost = (status == NO_MAXIMUM) | (status == NOT_CONVERGED)
        pix[lost] = np.nan
        arcsec[lost] = np.nan
        return pix.reshape(nb + (5,)), arcsec.reshape(nb + (5,)), status.reshape(nb)
