"""`Alignment` -- same public API as the reference's `hdrshift/alignment.py`, B200 engine underneath.

Public signatures mirror `hdrshift/alignment.py:47-55, 144-148, 263-269`. What changes is everything
below `_find_best_header_parameters` (`:613-797`): instead of forking `counts_cpu_max` workers that each
rebuild two WCS objects, call scipy and numba per lag, the lag grid is turned into a table of per-lag
constants and evaluated by the fused CUDA kernels of `csrc/coreg_lag_*.cu` (see `engine.py`).

Semantics follow the reference's `parallelism=True` branch (the contract of SURVEY.md section 0):
the common grid of the helioprojective search is the UNSHIFTED small grid. `parallelism`,
`counts_cpu_max` and `display_progress_bar` are accepted and ignored. Never-evaluated lags (the ones
that kill the reference's worker, App. B1) are reported as 0.0 exactly like the reference's cube.
"""
from __future__ import annotations

import copy
import os
import warnings

import numpy as np

from .._compat import fits_lite, units
from .._compat.wcs import CarWcs, TanWcs
from ..utils import Util
from . import engine as _engine
from .AlignmentResults import AlignmentResults, LocalAlignmentResults


def _open_fits(path):
    return Util._fits().open(path)


class _Refs:
    pass


class Alignment:

    def __init__(self, large_fov_known_pointing: str, small_fov_to_correct: str, lag_crval1: np.array,
                 lag_crval2: np.array, lag_cdelt1: object, lag_cdelt2: object, lag_crota: object,
                 lag_solar_r: object = None,
                 small_fov_value_min: object = None,
                 parallelism: object = False, display_progress_bar: bool = False,
                 small_fov_value_max: object = None, counts_cpu_max: int = 40, large_fov_window: object = -1,
                 small_fov_window: object = -1,
                 path_save_figure: str = None, reprojection_order=2, force_crota_0=False,
                 unit_lag="arcsec", cdelt_semantics="reference", strict_arithmetic=False, lag_search="dense",
                 coarse_stride=None, arithmetic=None, local_block=None):
        """Same parameters as the reference (`hdrshift/alignment.py:47-83`). Additions:

        arithmetic: "fp64" (default): every sample is evaluated in FP64 like the reference does (scipy accumulates in
            double, `utils/Util.py:98-102`) and then rounded to float32 (`alignment.py:1024`); |dr| ~ 1e-13 against
            the reference's operation order. "mixed" (opt-in, helioprojective order-2 search of a small image that
            holds float32 values, e.g. a BITPIX -32 file): projection in FP64, spline and per-segment sums in FP32 on
            the image centred on its pivot, the float32 store reproduced on the uncentred value; a per-lag error
            model (checked on the device) sends any lag that cannot be trusted to 1e-7 back through the FP64
            kernel. None: the COREG_ARITHMETIC environment variable, else "fp64".

        cdelt_semantics: "reference" reproduces the reference's handling of CDELT lags (a CDELT1 lag only
            rebuilds PCi_j, a non-zero CDELT2 lag leaves 0.0 in the cube because the reference's worker dies,
            SURVEY App. B1); "intended" applies CDELTi = ref + lag before the PCi_j rebuild.
        strict_arithmetic: evaluate the spline weights / tap sums in scipy's exact operation order (separate
            multiply and add) instead of fused multiply-add; per-sample bit-faithful, ~1e-15 in r, slower.
        lag_search: "dense" (default) evaluates every lag like the reference. "coarse_to_fine" (helioprojective frame)
            evaluates the CRVAL1 x CRVAL2 plane on a sub-lattice of stride `coarse_stride` first (all CDELT / CROTA
            lags), then densely in a window around the best coarse lag, re-centring while the maximum sits on the
            window's edge; lags that were not evaluated are NaN in the cube. Every evaluated entry is bit-identical
            to the dense cube's; the arg-max is the dense one whenever the correlation peak is wider than the
            stride (default stride: the large image's pixel size in lag steps, at least 2).
        local_block: None (default) or the block size (rows, cols) -- or one int for square blocks -- in pixels of the
            common grid, each a positive multiple of 64. `align_using_helioprojective` then also returns, from the same
            pass of the lag kernels, one correlation cube per block of the common grid (blocks from pixel (0, 0), the
            last block row and column taking whatever remains): `.local`, a `LocalAlignmentResults`, on this object and
            on the returned `AlignmentResults`. A shift that changes across the field (pointing drift along a SPICE
            raster, a roll or plate-scale error) shows up as block maxima that differ. Not with
            lag_search="coarse_to_fine" (its windows follow the global maximum), mixed arithmetic, or the Carrington
            entry points (`align_using_carrington` takes its blocks as an argument of the call, on the grid it
            defines).
        """
        self.large_fov_known_pointing = large_fov_known_pointing
        self.small_fov_to_correct = small_fov_to_correct
        self.lag_crval1 = lag_crval1
        self.lag_crval2 = lag_crval2
        self.lag_cdelt1 = lag_cdelt1
        self.lag_cdelt2 = lag_cdelt2
        self.lag_crota = lag_crota
        self.lag_solar_r = lag_solar_r
        self.unit_lag = unit_lag
        self.unit_lag_input = copy.deepcopy(unit_lag)

        self.lonlims = None
        self.latlims = None
        self.shape = None
        self.reference_date = None
        self.parallelism = parallelism            # accepted, ignored: the GPU path is always "parallel"
        self.small_fov_window = small_fov_window
        self.large_fov_window = large_fov_window

        self.crval1_ref = None
        self.crval2_ref = None
        self.crota_ref = None
        self.cdelt1_ref = None
        self.cdelt2_ref = None
        self.data_large = None
        self.counts = counts_cpu_max              # accepted, ignored
        self.data_small = None
        self.hdr_small = None
        self.hdr_large = None
        self.method = None
        self.small_fov_value_min = small_fov_value_min
        self.small_fov_value_max = small_fov_value_max
        self.path_save_figure = path_save_figure
        self.display_progress_bar = display_progress_bar
        self.force_crota_0 = force_crota_0
        self.method_carrington_reprojection = None
        self.use_pcij = not ((lag_crota is None) and (lag_cdelt1 is None) and (lag_cdelt2 is None))
        self.order = reprojection_order
        self.lon_ctype = None
        self.lat_ctype = None
        self.use_sunpy = False
        self.cdelt_semantics = cdelt_semantics
        self.strict_arithmetic = strict_arithmetic
        self.arithmetic = arithmetic
        if lag_search not in ("dense", "coarse_to_fine"):
            raise ValueError("lag_search must be 'dense' or 'coarse_to_fine'")
        self.lag_search = lag_search
        self.coarse_stride = coarse_stride
        self.local_block = None if local_block is None else _engine.local_block_shape(local_block)
        self.local = None
        if self.local_block is not None:
            if lag_search != "dense":
                raise ValueError("local_block needs lag_search='dense' (the coarse-to-fine windows follow the global "
                                 "maximum)")
            if arithmetic == "mixed":
                raise ValueError("local_block needs all-FP64 arithmetic (the mixed kernel's per-lag guard is "
                                 "calibrated on whole-grid moments)")
        self.lags_evaluated = None
        self.engine = None
        self.nvalid = None
        for lag_name in ("lag_crval1", "lag_crval2", "lag_crota", "lag_cdelt1", "lag_cdelt2"):
            if getattr(self, lag_name) is None:
                setattr(self, lag_name, np.array([0.0]))

    # ------------------------------------------------------------------------------------------------
    # public entry points
    # ------------------------------------------------------------------------------------------------
    def align_using_helioprojective(self, method: str = 'correlation', return_type: str = 'AlignmentResults',
                                    fov_limits=None, remove_fov_limits=None):
        """Co-alignment in the helioprojective frame (`hdrshift/alignment.py:263-342`)."""
        self.lonlims = None
        self.latlims = None
        self.shape = None
        self.reference_date = None
        self.method = method
        self.coordinate_frame = "final_helioprojective"
        self.lon_ctype = "HPLN-TAN"
        self.lat_ctype = "HPLT-TAN"
        self.ang2pipi = True
        masking = (self.small_fov_value_min is not None or self.small_fov_value_max is not None
                   or fov_limits is not None or remove_fov_limits is not None)
        self._load_pair(lazy=True, host_masking=masking)
        results = self._find_best_header_parameters(fov_limits=fov_limits, remove_fov_limits=remove_fov_limits)
        return self._wrap_results(results, return_type)

    def align_using_carrington(self, lonlims=None, latlims=None, size_deg_carrington=None, shape=None,
                               reference_date=None, method='correlation', method_carrington_reprojection="fa",
                               return_type='AlignmentResults', local_block=None):
        """Co-alignment on a user Carrington grid (`hdrshift/alignment.py:144-261`). method_carrington_reprojection:
        "fa" (`_carrington_transform_fa`, the default) or "sunpy" (`_carrington_transform_sunpy`, `:939-985`: no grid
        arguments needed; the search runs on the small image's own grid after a solar-surface reprojection of the large
        image -- a restatement of sunpy / reproject's published algorithm, `_surface_search`).

        local_block: None (default) or the block size (rows, cols) -- or one int for square blocks --, each a positive
        multiple of 64, in pixels of the grid the search runs on: with "fa" the Carrington grid of this call (rows =
        latitude samples, shape[1] of them; columns = longitude samples, shape[0] of them; both on the `linspace` grid
        of lonlims / latlims), with "sunpy" the small image's own grid. The search then also returns one correlation
        cube per block from the same pass of the lag kernel (`.local`, a `LocalAlignmentResults`, on this object and on
        the returned `AlignmentResults`), e.g. latitude bands that see the longitude shift the rigid "fa" rotation
        leaves. It applies to this call only; the constructor's `local_block` is refused here."""
        self._refuse_local_block("align_using_carrington")
        block = None if local_block is None else _engine.local_block_shape(local_block)
        self.method = method
        self.coordinate_frame = "final_carrington"
        self.lon_ctype = "HPLN-TAN"
        self.lat_ctype = "HPLT-TAN"
        self.ang2pipi = True
        self.method_carrington_reprojection = method_carrington_reprojection
        if method_carrington_reprojection not in ("fa", "sunpy"):
            raise ValueError("method_carrington_reprojection must be either 'fa' or 'sunpy")
        self._load_pair()
        if method_carrington_reprojection == "sunpy":
            # (the reference reads no grid argument on this path: alignment.py:198-231 is the "fa" branch)
            self.lonlims = self.latlims = self.shape = self.reference_date = None
            results = self._find_best_header_parameters(carrington_block=block)
            return self._wrap_results(results, return_type)
        if reference_date is None:
            if "DATE-AVG" not in self.hdr_large:
                raise ValueError(
                    "Either provide a reference date manualy or the reference file header must have a DATE-AVG keyword.")
            self.reference_date = self.hdr_large["DATE-AVG"]
        else:
            self.reference_date = reference_date
        if (lonlims is None) and (latlims is None) & (size_deg_carrington is not None):
            crln, crlt = self.hdr_small["CRLN_OBS"], self.hdr_small["CRLT_OBS"]
            self.lonlims = [crln - 0.5 * size_deg_carrington[0], crln + 0.5 * size_deg_carrington[0]]
            self.latlims = [crlt - 0.5 * size_deg_carrington[1], crlt + 0.5 * size_deg_carrington[1]]
            self.shape = [self.hdr_small["NAXIS1"], self.hdr_small["NAXIS2"]]
        elif (lonlims is not None) and (latlims is not None) & (shape is not None):
            self.lonlims = lonlims
            self.latlims = latlims
            self.shape = shape
        else:
            raise ValueError("either set lonlims as None, or not. no in between.")
        if self.shape[0] * self.shape[1] > 25000000:
            warnings.warn(f"shape parameter is shape={shape}, which is very large."
                          "Computational time might significantly increase")
        results = self._find_best_header_parameters(carrington_block=block)
        return self._wrap_results(results, return_type)

    def align_using_initial_carrington(self, method='correlation', return_type='AlignmentResults'):
        """Co-alignment of two images that already are Carrington maps, CTYPE CRLN-CAR / CRLT-CAR
        (`hdrshift/alignment.py:344-399`): the helioprojective search with the plate-carree projection, both images
        rounded to float32 when read (`:373, 387`), lags converted to header units without longitude wrapping
        (`:388, 831-837`), and -- unlike the other two entry points -- the lag arrays handed to `AlignmentResults`
        as they are (`:392-399`)."""
        self._refuse_local_block("align_using_initial_carrington")
        self.lonlims = None
        self.latlims = None
        self.shape = None
        self.reference_date = None
        self.method = method
        self.coordinate_frame = "initial_carrington"
        self.lon_ctype = "CRLN-CAR"
        self.lat_ctype = "CRLT-CAR"
        self.ang2pipi = False
        f_large = self._open_large()
        f_small = self._open_small()
        self.data_large = np.array(f_large[self.large_fov_window].data, dtype="float32")
        self.hdr_large = f_large[self.large_fov_window].header.copy()
        self.hdr_small = f_small[self.small_fov_window].header.copy()
        self._check_ant_create_pcij_matrix(self.hdr_small)
        self._check_ant_create_pcij_matrix(self.hdr_large)
        self.data_small = np.array(f_small[self.small_fov_window].data, dtype="float32")
        f_large.close()
        f_small.close()
        results = self._find_best_header_parameters(ang2pipi=False)
        if return_type == "corr":
            return results
        if return_type == "AlignmentResults":
            return AlignmentResults(corr=results, lag_crval1=self.lag_crval1, lag_crval2=self.lag_crval2,
                                    lag_cdelt1=self.lag_cdelt1, lag_cdelt2=self.lag_cdelt2, lag_crota=self.lag_crota,
                                    unit_lag=self.unit_lag, image_to_align_path=self.small_fov_to_correct,
                                    image_to_align_window=self.small_fov_window,
                                    reference_image_path=self.large_fov_known_pointing,
                                    reference_image_window=self.large_fov_window)
        return results

    def _refuse_local_block(self, entry):
        if getattr(self, "local_block", None) is not None:
            raise ValueError(f"local_block is implemented for align_using_helioprojective only, not {entry}")

    # ------------------------------------------------------------------------------------------------
    # host preparation (mirrors alignment.py:299-316, 580-611, 799-887)
    # ------------------------------------------------------------------------------------------------
    def _open_large(self):
        return _open_fits(self.large_fov_known_pointing)

    def _open_small(self):
        return _open_fits(self.small_fov_to_correct)

    def _load_pair(self, lazy=False, host_masking=True):
        """Open both files, copy the headers, check / create the PCi_j matrices and take the images.
        lazy=True (helioprojective frame): the large image stays in its memory-mapped file -- the engine converts and
        uploads only the window the small grid can reach -- and, when no host-side masking will touch it
        (host_masking=False) and the file holds float32 (BITPIX -32), the small image is handed over as stored
        (big-endian) for a byte swap on the device. The reference widens both images to float64 on the host
        (alignment.py:299-316); float32 payloads are kept as they are here (float32 -> float64 is exact)."""
        f_large = self._open_large()
        f_small = self._open_small()
        h_large, h_small = f_large[self.large_fov_window], f_small[self.small_fov_window]
        if lazy and hasattr(h_large, "read_window") and h_large.shape is not None and len(h_large.shape) == 2:
            self.data_large = h_large
        else:
            self.data_large = self._float_image(h_large.data)
        self.hdr_large = h_large.header.copy()
        self.hdr_small = h_small.header.copy()
        self._check_ant_create_pcij_matrix(self.hdr_small)
        self._check_ant_create_pcij_matrix(self.hdr_large)
        raw = h_small.raw_big_endian() if (lazy and not host_masking and hasattr(h_small, "raw_big_endian")) else None
        if raw is not None and raw.dtype == np.dtype(">f4") and raw.ndim == 2:
            self.data_small = raw
        else:
            self.data_small = self._float_image(h_small.data)
        f_large.close()
        f_small.close()

    @staticmethod
    def _float_image(data):
        data = np.asarray(data)
        if data.dtype in (np.float32, np.float64) and data.dtype.isnative:
            return np.array(data)      # private, writable copy
        return np.array(data, dtype=np.float64)

    def _wrap_results(self, results, return_type):
        if return_type == "corr":
            self._wrap_local()
            return results
        if return_type == "AlignmentResults":
            conv = lambda v: units.convert(units.ang2pipi(v, self.unit_lag), self.unit_lag, self.unit_lag_input)  # noqa: E731
            self.lag_crval1 = conv(self.lag_crval1)
            self.lag_crval2 = conv(self.lag_crval2)
            self.lag_cdelt1 = conv(self.lag_cdelt1)
            self.lag_cdelt2 = conv(self.lag_cdelt2)
            self.unit_lag = self.unit_lag_input
            res = AlignmentResults(corr=results, **self._results_kwargs())
            if self._wrap_local() is not None:
                res.local = self.local
            return res
        self._wrap_local()
        return results

    def _results_kwargs(self):
        """Everything but the cube that `AlignmentResults` takes, with the lag arrays as they stand (header units
        after a search, the caller's units once `_wrap_results` has converted them back)."""
        return dict(lag_crval1=self.lag_crval1, lag_crval2=self.lag_crval2, lag_cdelt1=self.lag_cdelt1,
                    lag_cdelt2=self.lag_cdelt2, lag_crota=self.lag_crota, unit_lag=self.unit_lag,
                    image_to_align_path=self.small_fov_to_correct, image_to_align_window=self.small_fov_window,
                    reference_image_path=self.large_fov_known_pointing, reference_image_window=self.large_fov_window)

    def _wrap_local(self):
        """`LocalAlignmentResults` of the per-block cubes the last search left (None without `local_block`)."""
        raw = getattr(self, "_local_raw", None)
        if raw is not None:
            self._local_raw = None
            self.local = LocalAlignmentResults(*raw, **self._results_kwargs())
        return getattr(self, "local", None)

    def _check_ant_create_pcij_matrix(self, hdr):
        """`alignment.py:580-611`."""
        if "PC1_1" not in hdr:
            warnings.warn("PCi_j matrix not found in header of the FITS file to align. Adding it to the header.")
            if "CROTA" in hdr:
                crot = hdr["CROTA"]
            elif "CROTA2" in hdr:
                crot = hdr["CROTA2"]
            elif self.force_crota_0:
                crot = 0.0
                hdr["CROTA"] = 0.0
            else:
                raise ValueError("No, CROTA, CROTA2 or PCi_j matrix in your FITS file. If want to force a CROTA=0, "
                                 "please set the force_crota_0 to True when initializing Alignment ")
            rho = np.deg2rad(crot)
            lam = hdr["CDELT2"] / hdr["CDELT1"]
            hdr["PC1_1"] = float(np.cos(rho))
            hdr["PC2_2"] = float(np.cos(rho))
            hdr["PC1_2"] = float(-lam * np.sin(rho))
            hdr["PC2_1"] = float((1 / lam) * np.sin(rho))
        if hdr["PC1_1"] >= 1.0:
            warnings.warn(f'hdr["PC1_1"]={hdr["PC1_1"]}, setting to  1.0.')
            hdr["PC1_1"] = 1.0
            hdr["PC2_2"] = 1.0
            hdr["PC1_2"] = 0.0
            hdr["PC2_1"] = 0.0
            hdr["CROTA"] = 0.0
        if "CROTA" not in hdr:
            s = -np.sign(hdr["PC1_2"]) + (hdr["PC1_2"] == 0)
            hdr["CROTA"] = float(s * np.rad2deg(np.arccos(hdr["PC1_1"])))

    def _set_initial_header_values(self, ang2pipi):
        """`alignment.py:799-842`."""
        self.crval1_ref = self.hdr_small['CRVAL1']
        self.crval2_ref = self.hdr_small['CRVAL2']
        if 'CROTA' in self.hdr_small:
            self.crota_ref = self.hdr_small['CROTA']
        elif 'CROTA2' in self.hdr_small:
            self.crota_ref = self.hdr_small['CROTA2']
        else:
            s = -np.sign(self.hdr_small['PC1_2']) + (self.hdr_small['PC1_2'] == 0)
            self.crota_ref = float(np.rad2deg(np.arccos(self.hdr_small['PC1_1'])) * s)
            self.hdr_small["CROTA"] = float(np.rad2deg(np.arccos(self.hdr_small['PC1_1'])))
        self.cdelt1_ref = self.hdr_small['CDELT1']
        self.cdelt2_ref = self.hdr_small['CDELT2']
        self.unit1 = self.hdr_small["CUNIT1"]
        self.unit2 = self.hdr_small["CUNIT2"]
        if self.unit_lag in self.unit1:
            pass
        else:
            warnings.warn("Units of headers in deg: Modyfying inputs units to deg.")
            conv = _engine.lag_unit_to_header_unit
            self.lag_crval1 = conv(self.lag_crval1, self.unit_lag, self.unit1, ang2pipi)
            self.lag_crval2 = conv(self.lag_crval2, self.unit_lag, self.unit2, ang2pipi)
            self.lag_cdelt1 = conv(self.lag_cdelt1, self.unit_lag, self.unit1, ang2pipi)
            self.lag_cdelt2 = conv(self.lag_cdelt2, self.unit_lag, self.unit2, ang2pipi)
            self.unit_lag = self.unit1
        if self.unit1 != self.unit2:
            raise ValueError("CUNIT1 and CUNIT2 must be equal")
        if self.lag_solar_r is None:
            self.lag_solar_r = np.array([1.004])

    def _set_threshold_minmax_to_nan(self):
        """`alignment.py:876-887`."""
        if self.small_fov_value_min is None and self.small_fov_value_max is None:
            return
        self.data_small = self.data_small.astype(np.float64)   # compare in float64 like the reference
        c1 = np.ones(self.data_small.shape, dtype=bool)
        c2 = np.ones(self.data_small.shape, dtype=bool)
        with np.errstate(invalid="ignore"):
            if self.small_fov_value_min is not None:
                c1[np.abs(self.data_small) < self.small_fov_value_min] = False
            if self.small_fov_value_max is not None:
                c2[np.abs(self.data_small) > self.small_fov_value_max] = False
        self.data_small[np.logical_not(np.logical_and(c1, c2))] = np.nan

    def _set_remove_fov_limits_to_nan(self, remove_fov_limits):
        """`alignment.py:862-874`; limits are [[lonmin, lonmax], [latmin, latmax]] in arcsec (plain numbers or
        astropy quantities)."""
        lon, lat = Util.AlignEUIUtil.extract_EUI_coordinates(self.hdr_small, dsun=False)
        lims = []
        for pair in remove_fov_limits:
            v, unit = units.strip(pair, "arcsec")
            lims.append(units.convert(np.asarray(v, dtype=np.float64), unit, "deg"))
        lonl, latl = lims
        mask = (lon >= lonl[0]) & (lon <= lonl[1]) & (lat >= latl[0]) & (lat <= latl[1])
        self.data_small[mask] = np.nan

    def _set_removed_values_to_nan_in_datasmall(self, fov_limits, remove_fov_limits):
        """`alignment.py:844-861`."""
        self._set_threshold_minmax_to_nan()
        if remove_fov_limits is not None:
            self._set_remove_fov_limits_to_nan(remove_fov_limits)
        if fov_limits is not None:
            self._select_fov_in_small_data(fov_limits)

    def _limits_deg(self, limits):
        out = []
        for pair in limits:
            v, unit = units.strip(pair, "arcsec")
            out.append(units.convert(np.asarray(v, dtype=np.float64), unit, "deg"))
        return out

    def _select_fov_in_small_data(self, fov_limits):
        """`alignment.py:1082-1127`: the small image re-sampled (order `reprojection_order`, NaN fill, float64) onto a
        regular, unrotated lon / lat grid inside `fov_limits` = [[lonmin, lonmax], [latmin, latmax]] (arcsec numbers
        or astropy quantities); the search then runs on that image and its new header. Kept as the reference has it,
        including NAXIS1 / CRPIX1 taken from the grid's ROW count (only matters for non-square selections)."""
        from .. import _ext
        torch = _engine._torch()
        lonlims, latlims = self._limits_deg(fov_limits)
        lon, lat = Util.AlignEUIUtil.extract_EUI_coordinates(self.hdr_small, dsun=False)
        long, latg, dlon, dlat = Util.PlotFits.build_regular_grid(lon, lat, lonlims=lonlims, latlims=latlims)
        if long.size == 0:
            raise ValueError("fov_limits select no pixel of the small image")
        mid = [long.shape[0] // 2, long.shape[1] // 2]
        hdrg = self.hdr_small.copy()
        hdrg["CRVAL1"] = float(units.convert(long[mid[0], mid[1]], "deg", hdrg["CUNIT1"]))
        hdrg["CRVAL2"] = float(units.convert(latg[mid[0], mid[1]], "deg", hdrg["CUNIT2"]))
        hdrg["CRPIX1"] = mid[0] + 1
        hdrg["CRPIX2"] = mid[1] + 1
        hdrg["CDELT1"] = float(units.convert(dlon, "deg", hdrg["CUNIT1"]))
        hdrg["CDELT2"] = float(units.convert(dlat, "deg", hdrg["CUNIT2"]))
        hdrg["PC1_1"], hdrg["PC2_2"], hdrg["PC1_2"], hdrg["PC2_1"] = 1.0, 1.0, 0.0, 0.0
        hdrg["CROTA"] = 0.0
        hdrg["CROTA2"] = 0.0
        hdrg["NAXIS1"] = long.shape[0]
        hdrg["NAXIS2"] = long.shape[1]
        # _extract_coordinates_pixels(hdrg -> hdr_small) + interpol2d, on the device
        lng_d, lat_d = Util.AlignEUIUtil.extract_EUI_coordinates(hdrg, dsun=False, as_device=True)
        xg, yg = _ext.tan_world2pix(TanWcs.from_header(self.hdr_small), lng_d, lat_d)
        img = torch.from_numpy(np.ascontiguousarray(_engine.LagSearchEngine._native_float(self.data_small))).to(xg.device)
        out = _ext.map_coordinates(img, yg, xg, self.order, float("nan"), torch.float64)
        self.data_small = out.cpu().numpy()
        self.hdr_small = hdrg

    # ------------------------------------------------------------------------------------------------
    # the seam: lag grid -> correlation cube
    # ------------------------------------------------------------------------------------------------
    def _find_best_header_parameters(self, ang2pipi: bool = True, fov_limits=None, remove_fov_limits=None,
                                     carrington_block=None):
        """Correlation cube float64 [n_crval1, n_crval2, n_cdelt1, n_cdelt2, n_crota, n_solar_r]
        (`alignment.py:613-797`, parallel branch). carrington_block: the (rows, cols) blocks of
        `align_using_carrington(local_block=...)` (the helioprojective search reads `self.local_block`)."""
        if self.method != 'correlation':
            raise NotImplementedError("only method='correlation' is on the device path")
        self.local = self._local_raw = None
        if getattr(self, "local_block", None) is not None and \
                (getattr(self, "arithmetic", None) or os.environ.get("COREG_ARITHMETIC")) == "mixed":
            raise ValueError("local_block needs all-FP64 arithmetic (COREG_ARITHMETIC=mixed is set)")
        self._set_removed_values_to_nan_in_datasmall(fov_limits=fov_limits, remove_fov_limits=remove_fov_limits)
        self._set_initial_header_values(ang2pipi)
        if self.unit_lag != self.hdr_small["CUNIT1"] or self.unit_lag != self.hdr_small["CUNIT2"]:
            raise ValueError("lag.unit and cUNIT are not the same")
        shape5 = (len(self.lag_crval1), len(self.lag_crval2), len(self.lag_cdelt1), len(self.lag_cdelt2),
                  len(self.lag_crota))
        d1, d2, d3, d4, d5 = _engine.flat_lag_grid(self.lag_crval1, self.lag_crval2, self.lag_cdelt1,
                                                   self.lag_cdelt2, self.lag_crota)
        refs = _Refs()
        refs.crval1_ref, refs.crval2_ref, refs.crota_ref = self.crval1_ref, self.crval2_ref, self.crota_ref
        refs.cdelt1_ref, refs.cdelt2_ref = self.cdelt1_ref, self.cdelt2_ref

        # small-image storage on the device: float64 for the helioprojective kernels (FP64-issue bound: no per-tap
        # conversion); float32, when the file holds float32, for the Carrington kernel, whose gather is sparse in the
        # small image (several detector pixels per Carrington pixel) and therefore bound by L1 wavefronts, not FP64
        storage = "auto" if self.coordinate_frame == "final_carrington" else "f64"
        eng = _engine.LagSearchEngine(order=self.order, strict=self.strict_arithmetic, small_storage=storage,
                                      arithmetic=getattr(self, "arithmetic", None))
        self.engine = eng
        eng.set_small(self.data_small)
        if eng.small_count() == 0:     # `np.isnan(data_small).all()` (alignment.py:656), counted on the device
            raise ValueError("minimum or maximum value have set all small FOV to nan")
        n_r = len(self.lag_solar_r)
        cube = np.zeros(shape5 + (n_r,), dtype=np.float64)
        if self.coordinate_frame == "final_helioprojective":
            w_small = TanWcs.from_header(self.hdr_small)
            w_large = TanWcs.from_header(self.hdr_large)
            eng.prepare_hpc(self.data_large, w_large, w_small)
            self.hdr_large = self.hdr_small.copy()   # alignment.py:1000
            table, dead = eng.hpc_lag_table(self.hdr_small, refs, d1, d2, d3, d4, d5, self.cdelt_semantics)
            if self.lag_search == "coarse_to_fine":
                corr, nvalid = self._coarse_to_fine(eng, table, shape5, w_large, dead)
            elif getattr(self, "local_block", None) is not None:
                corr, nvalid, corr_b, nvalid_b = eng.search(table, block=self.local_block)
                self.lags_evaluated = int(table.shape[0])
                self._keep_local_blocks(eng.ref.shape, self.local_block, corr_b, nvalid_b, dead, shape5, n_r)
            else:
                corr, nvalid = eng.search(table, return_nvalid=True)
                self.lags_evaluated = int(table.shape[0])
            corr = np.where(dead, 0.0, corr)
            for kk in range(n_r):
                cube[..., kk] = corr.reshape(shape5)
            self.nvalid = nvalid.reshape(shape5)
        elif self.coordinate_frame == "initial_carrington":
            if fov_limits is not None or remove_fov_limits is not None:
                raise ValueError("fov_limits / remove_fov_limits need HPLN-TAN headers (utils/Util.py:283-286)")
            if self.lag_search != "dense":
                raise ValueError("lag_search='coarse_to_fine' is implemented for the helioprojective frame only")
            w_small = CarWcs.from_header(self.hdr_small)
            w_large = CarWcs.from_header(self.hdr_large)
            eng.prepare_car(self.data_large, w_large, w_small)
            self.hdr_large = self.hdr_small.copy()   # alignment.py:1000
            table, dead = _engine.car_lag_table(self.hdr_small, refs, d1, d2, d3, d4, d5, self.cdelt_semantics)
            corr, nvalid = eng.search(table, return_nvalid=True)
            self.lags_evaluated = int(table.shape[0])
            corr = np.where(dead, 0.0, corr)
            for kk in range(n_r):
                cube[..., kk] = corr.reshape(shape5)
            self.nvalid = nvalid.reshape(shape5)
        elif self.coordinate_frame == "final_carrington":
            if n_r != 1:
                raise ValueError("lag_solar_r must hold exactly one value (the reference breaks on more, "
                                 "alignment.py:646-660)")
            if getattr(self, "method_carrington_reprojection", "fa") == "sunpy":
                corr, nvalid, dead, blocks = self._surface_search(eng, refs, d1, d2, d3, d4, d5,
                                                                  float(self.lag_solar_r[0]), carrington_block)
            else:
                corr, nvalid, dead, blocks = self._carrington_search(eng, refs, d1, d2, d3, d4, d5,
                                                                     float(self.lag_solar_r[0]), carrington_block)
            if blocks is not None:
                self._keep_local_blocks(eng.ref.shape, carrington_block, *blocks, dead, shape5, n_r)
            cube[..., 0] = corr.reshape(shape5)
            self.nvalid = nvalid.reshape(shape5)
        else:
            raise NotImplementedError(self.coordinate_frame)
        self.data_large = None
        return cube

    def _keep_local_blocks(self, grid_shape, block, corr_b, nvalid_b, dead, shape5, n_r):
        """Per-block values [nby, nbx, n_lags] of a search over a (gny, gnx) grid -> `self._local_raw` (cube shape, lags
        in `dead` 0.0 in every block as in the cube), wrapped into `self.local` with the results."""
        nb = corr_b.shape[:2]
        if dead is not None and dead.any():
            corr_b = np.where(dead, 0.0, corr_b)
        cube_b = corr_b.reshape(nb + shape5 + (1,))
        if n_r > 1:
            cube_b = np.repeat(cube_b, n_r, axis=-1)
        bounds = _engine.region_bounds(grid_shape[0], grid_shape[1], block)
        self._local_raw = (cube_b, nvalid_b.reshape(nb + shape5), bounds)

    def _coarse_to_fine(self, eng, table, shape5, w_large, dead=None):
        """Sub-lattice pass over the CRVAL1 x CRVAL2 plane, then dense windows around the running maximum (SURVEY.md
        section 8f-3). Returns (corr, nvalid) over the full flat lag list, NaN / 0 where nothing was evaluated. The
        window follows the GLOBAL maximum over all CDELT / CROTA slices; lags the reference cannot evaluate (`dead`:
        they read 0.0 in the final cube) never steer it; when no coarse lag yields a coefficient (no overlap, no valid
        pixel) the search stops there and the cube is NaN where nothing could be computed, like the dense search's."""
        n1, n2 = shape5[0], shape5[1]
        rest = int(np.prod(shape5[2:]))
        stride = self.coarse_stride
        if stride is None:
            step = min(abs(float(np.diff(np.asarray(lag, dtype=np.float64)).mean())) if len(lag) > 1 else np.inf
                       for lag in (self.lag_crval1, self.lag_crval2))
            pix = abs(w_large.cdelt1) / TanWcs.from_header(self.hdr_small).unit_scale1     # large pixel, header units
            stride = int(max(2, np.floor(pix / step))) if np.isfinite(step) and step > 0 else 2
        stride = int(max(1, stride))
        corr = np.full(table.shape[0], np.nan)
        nvalid = np.zeros(table.shape[0], dtype=np.int64)
        done = np.zeros((n1, n2), dtype=bool)

        def evaluate(mask2d):
            todo = mask2d & ~done
            if not todo.any():
                return
            idx = np.nonzero(np.repeat(todo.ravel(), rest))[0]      # C order: (crval1, crval2) slowest
            c, nv = eng.search(table[idx], return_nvalid=True)
            corr[idx], nvalid[idx] = c, nv
            done[todo] = True

        coarse = np.zeros((n1, n2), dtype=bool)
        i1 = np.unique(np.r_[np.arange(0, n1, stride), n1 - 1])
        i2 = np.unique(np.r_[np.arange(0, n2, stride), n2 - 1])
        coarse[np.ix_(i1, i2)] = True
        evaluate(coarse)
        half = stride + 2
        for _ in range(8):
            score = corr if dead is None else np.where(dead, np.nan, corr)
            if np.isnan(score).all():
                break
            best = np.unravel_index(np.nanargmax(score), (n1, n2, rest))[:2]
            lo1, hi1 = max(0, best[0] - half), min(n1, best[0] + half + 1)
            lo2, hi2 = max(0, best[1] - half), min(n2, best[1] + half + 1)
            win = np.zeros((n1, n2), dtype=bool)
            win[lo1:hi1, lo2:hi2] = True
            if not (win & ~done).any():
                break
            evaluate(win)
        self.lags_evaluated = int(done.sum()) * rest
        return corr, nvalid

    @staticmethod
    def _surface_frame(hdr):
        """Observer (Stonyhurst longitude / latitude [rad], distance [m]) and observation time [s] of a header's
        helioprojective frame, as sunpy's `wcs_utils` reads them: HGLN_OBS / HGLT_OBS / DSUN_OBS, DATE-AVG else DATE-OBS."""
        from .._compat import timeutil
        for k in ("HGLN_OBS", "HGLT_OBS", "DSUN_OBS"):
            if k not in hdr:
                raise ValueError(f"method_carrington_reprojection='sunpy' needs {k} in both headers")
        date = hdr["DATE-AVG"] if "DATE-AVG" in hdr else hdr["DATE-OBS"]
        return (float(np.radians(hdr["HGLN_OBS"])), float(np.radians(hdr["HGLT_OBS"])), float(hdr["DSUN_OBS"]),
                timeutil.to_seconds(date))

    def _surface_frames(self, d_solar_r):
        """`_ext.CoregSurfaceFrames` of the pair: the small image's observer as target, the large image's as source."""
        from .. import _ext
        g_lon, g_lat, g_d, g_t = self._surface_frame(self.hdr_small)
        i_lon, i_lat, i_d, i_t = self._surface_frame(self.hdr_large)
        return _ext.CoregSurfaceFrames(g_lon, g_lat, g_d, i_lon, i_lat, i_d, (i_t - g_t) / 86400.0,
                                       d_solar_r * _engine.R_SUN_M)

    def _surface_search(self, eng, refs, d1, d2, d3, d4, d5, d_solar_r, block=None):
        """`_carrington_transform_sunpy` (`alignment.py:939-985`) on the device. Once: the large image reprojected onto
        the small image's grid through sunpy's helioprojective -> helioprojective change of observer for points on the
        solar surface (radius d_solar_r R_sun), differentially rotated over the time between the two observations
        (`propagate_with_solar_surface`), bilinear (`reproject_interp`); then `hdr_large = hdr_small` (`:955`). Per
        lag: `Map(data_small, hdr_shifted).reproject_to(WCS(hdr_small))` -- same observer and time on both sides, so
        the change of frame is the identity and the call is the helioprojective search's geometry with bilinear
        interpolation and reproject's edge rule, no float32 store. sunpy / reproject are absent from the image: the
        algorithm is restated from its published form (oracle/surface_reproject.py), parity unpinned.
        Returns (corr, nvalid, dead, blocks): blocks = the per-block (corr, nvalid) [nby, nbx, n_lags] of the small
        image's grid with `block`, else None."""
        w_small = TanWcs.from_header(self.hdr_small)
        w_large = TanWcs.from_header(self.hdr_large)
        eng.prepare_surface(self.data_large, w_large, w_small, self._surface_frames(d_solar_r))
        self.hdr_large = self.hdr_small.copy()
        table, dead = eng.surface_lag_table(self.hdr_small, refs, d1, d2, d3, d4, d5, self.cdelt_semantics)
        if block is None:
            corr, nvalid = eng.search(table, return_nvalid=True)
            blocks = None
        else:
            corr, nvalid, corr_b, nvalid_b = eng.search(table, block=block)
            blocks = (corr_b, nvalid_b)
        self.lags_evaluated = int(table.shape[0])
        return np.where(dead, 0.0, corr), nvalid, dead, blocks

    def _carrington_search(self, eng, refs, d1, d2, d3, d4, d5, d_solar_r, block=None):
        """Per CROTA-lag value one pair of detector planes; CRVAL lags are pure offsets on them
        (`alignment.py:889-901`, `utils/rectify.py:377-423`). Returns (corr, nvalid, dead, blocks): blocks = the
        per-block (corr, nvalid) [nby, nbx, n_lags] of the Carrington grid with `block` (every CROTA group's lags at
        their place in the lag list; lags in `dead` are not evaluated and read 0.0 / 0), else None."""
        for hdr in (self.hdr_small, self.hdr_large):
            warn_fa_units(hdr)
        eng.prepare_carrington_large(self.data_large, self.hdr_large, d_solar_r, self.lonlims, self.latlims,
                                     self.shape)
        n = d1.size
        corr = np.zeros(n, dtype=np.float64)
        nvalid = np.zeros(n, dtype=np.int64)
        blocks = None
        if block is not None:
            nb = _engine._ext.region_grid(eng.ref.shape[0], eng.ref.shape[1], *block)
            blocks = (np.zeros(nb + (n,), dtype=np.float64), np.zeros(nb + (n,), dtype=np.int64))
        dead = carrington_dead_lags(d3, d4, self.cdelt_semantics)
        for sel, planes, table, lag_ij in self._carrington_tables(eng, refs, d1, d2, d5, dead, d_solar_r):
            if block is None:
                c, nv = eng.search(table, planes=planes, return_nvalid=True, lag_ij=lag_ij)
            else:
                c, nv, blocks[0][..., sel], blocks[1][..., sel] = eng.search(table, planes=planes, lag_ij=lag_ij,
                                                                             block=block)
            corr[sel] = c
            nvalid[sel] = nv
        return corr, nvalid, dead, blocks

    def _carrington_tables(self, eng, refs, d1, d2, d5, dead, d_solar_r):
        """Per CROTA-lag value (generated one at a time: each holds a pair of planes the size of the grid):
        (flat indices of its lags, detector planes (tx, ty) of the rotated header on the Carrington grid, [n, 2] (x0, y0)
        offset table, CRVAL grid indices for `offset_patch_order`). Lags in `dead` are left out."""
        roll_ref = self.hdr_small["CROTA"] if "CROTA" in self.hdr_small else self.hdr_small["CROTA2"]
        shape5 = (len(self.lag_crval1), len(self.lag_crval2), len(self.lag_cdelt1), len(self.lag_cdelt2),
                  len(self.lag_crota))
        for dc in np.unique(d5):
            sel = np.nonzero((d5 == dc) & ~dead)[0]
            if sel.size == 0:
                continue
            hdr = self.hdr_small.copy()
            roll = roll_ref
            if dc != 0.0:
                roll = refs.crota_ref + dc
                hdr["CROTA" if "CROTA" in hdr else "CROTA2"] = float(roll)
            planes = eng.carrington_planes(hdr, d_solar_r, self.lonlims, self.latlims, self.shape)
            x0, y0 = eng.carrington_offset(hdr, refs.crval1_ref + d1[sel], refs.crval2_ref + d2[sel], roll)
            table = np.stack([x0, y0], axis=1).astype(np.float64)
            # CRVAL grid indices of the selected lags (flat C order: crval1 slowest ... crota fastest): the kernel
            # takes them in detector-plane patches; lags that differ only in a CDELT index never share a patch
            i1, i2, i3, i4, _ = np.unravel_index(sel, shape5)
            yield sel, planes, table, (i1, i2, i3 * shape5[3] + i4)


def warn_fa_units(hdr):
    if str(hdr["CUNIT1"]).strip() != "arcsec":
        warnings.warn("the 'fa' Carrington transform assumes arcsec headers (utils/rectify.py:362-363)")


def carrington_dead_lags(d_cdelt1, d_cdelt2, cdelt_semantics):
    """Lags of the 'fa' Carrington search the reference cannot evaluate (a CDELT2 lag: they read 0.0 in the cube);
    CDELT lags under any other semantics are not implemented in this frame."""
    if cdelt_semantics == "reference":
        return np.asarray(d_cdelt2) != 0.0
    if np.any(np.asarray(d_cdelt1) != 0.0) or np.any(np.asarray(d_cdelt2) != 0.0):
        raise NotImplementedError("CDELT lags in the Carrington frame need cdelt_semantics='reference'")
    return np.zeros(np.asarray(d_cdelt1).size, dtype=bool)
