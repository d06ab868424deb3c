"""`AlignmentResults` -- host post-processing of the correlation cube, same API and arithmetic as the
reference's `hdrshift/AlignmentResults.py:25-341`: arg-max (first occurrence, C order), a bounded
2-D Gaussian `curve_fit` on the <= 5x5 neighbourhood of the maximum in the (CRVAL1, CRVAL2) plane, and
linear interpolation of the fitted sub-index centre back into the lag arrays. Pure numpy/scipy: this
part is not on the device path (SURVEY.md section 8a, last rows) and is pinned by the reference's own
golden cube (`hdrshift/test/test_AlignmentResults.py:35-126, 172-173`).
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


class AlignmentResults:

    def __init__(self, corr, lag_crval1, lag_crval2, lag_cdelt1, lag_cdelt2, lag_crota, unit_lag: str,
                 image_to_align_path: str = None, image_to_align_window=None, reference_image_path: str = None,
                 reference_image_window: int = None):
        zero = lambda v: np.array([0]) if v is None else v  # noqa: E731
        lag_crval1, lag_crval2 = zero(lag_crval1), zero(lag_crval2)
        lag_cdelt1, lag_cdelt2, lag_crota = zero(lag_cdelt1), zero(lag_cdelt2), zero(lag_crota)
        self.max_index = np.unravel_index(np.nanargmax(corr), corr.shape)
        self.corr = corr
        as_arr = lambda v: np.asarray(v, dtype=np.float64)  # noqa: E731
        # (value array, unit) pairs stand in for astropy quantities
        self.parameters_alignment = {
            "lag_crval1": (as_arr(lag_crval1), unit_lag), "lag_crval2": (as_arr(lag_crval2), unit_lag),
            "lag_cdelt1": (as_arr(lag_cdelt1), unit_lag), "lag_cdelt2": (as_arr(lag_cdelt2), unit_lag),
            "lag_crota": (as_arr(lag_crota), "deg"),
        }
        self.parameters_alignment_arcsec = {
            "lag_crval1": units.convert(as_arr(lag_crval1), unit_lag, "arcsec"),
            "lag_crval2": units.convert(as_arr(lag_crval2), unit_lag, "arcsec"),
            "lag_cdelt1": units.convert(as_arr(lag_cdelt1), unit_lag, "arcsec"),
            "lag_cdelt2": units.convert(as_arr(lag_cdelt2), unit_lag, "arcsec"),
            "lag_crota": as_arr(lag_crota),
        }
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
        """`AlignmentResults.py:218-341`. Quirks kept: the maximum is listed twice in the fit set, an offset of
        -2 below index 0 wraps around (only -1 is excluded), and solar-radius index 0 is used."""
        mi = self.max_index
        corr2d = self.corr[:, :, mi[2], mi[3], mi[4]]
        px, py = [mi[0]], [mi[1]]
        lenx, leny = corr2d.shape[0], corr2d.shape[1]
        for ii, jj in _NEIGHBOURS:
            x, y = mi[0] + ii, mi[1] + jj
            if (x != -1) and (x < lenx) and (y != -1) and (y < leny):
                px.append(x)
                py.append(y)
        if method != "fitting_gaussian":
            raise NotImplementedError
        if len(px) < 4:
            warnings.warn(" Cannot compute shift with Gaussian fitting: not enough points")
            self._argmax_shift()
            return None
        A = (np.float64(px), np.float64(py))
        B = np.float64(corr2d[px, py].ravel())
        p0 = (np.float64(corr2d[mi[0], mi[1]][0]), np.float64(mi[0]), np.float64(mi[1]), np.float64(1),
              np.float64(1), np.float64(0.9))
        bounds = ([np.float64(0), np.float64(mi[0] - 5), np.float64(mi[1] - 5), np.float64(0), np.float64(0),
                   np.float64(-10)],
                  [np.float64(10), np.float64(mi[0] + 5), np.float64(mi[1] + 5), np.float64(1000), np.float64(1000),
                   np.float64(10)])
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

    def results(self, i, j):
        """`AlignmentResults` of block (i, j): its arg-max and Gaussian sub-lag fit, as for the whole grid."""
        return AlignmentResults(corr=self.corr[i, j], **self._results_kwargs)
