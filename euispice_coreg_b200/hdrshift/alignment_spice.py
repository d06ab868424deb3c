"""`AlignmentSpice` -- the reference's `hdrshift/alignment_spice.py:13-120, 182-323` on top of the device engine.

Host preparation (slit-edge rows -> NaN, spectral sum of the chosen wavelength interval, 2-D header from the
4-axis WCS) is numpy; the search itself is `Alignment._find_best_header_parameters`. Like the reference
(SURVEY App. B9) the 2-D header comes out in degrees, `_check_ant_create_pcij_matrix` is not called, and
`reprojection_order`, value thresholds and `force_crota_0` are not forwarded.
"""
from __future__ import annotations

import numpy as np

from .._compat import units
from .._compat.wcs import SpiceWcs
from ..utils import Util
from .alignment import Alignment, _open_fits


def _value_in(q, unit):
    """Plain number (already in `unit`) or astropy-like quantity -> float in `unit`."""
    if hasattr(q, "to"):
        return float(q.to(unit).value)
    return float(q)


class AlignmentSpice(Alignment):

    def __init__(self, large_fov_known_pointing: str, small_fov_to_correct: str, lag_crval1=None, lag_crval2=None,
                 lag_cdelt1=None, lag_cdelt2=None, lag_crota=None, lag_solar_r=None, large_fov_window=-1,
                 small_fov_window=-1, parallelism: bool = False, counts_cpu_max: int = 40,
                 display_progress_bar: bool = False, path_save_figure=None, wavelength_interval_to_sum="all",
                 sub_fov_window="all", local_block=None):
        """Same parameters as `hdrshift/alignment_spice.py:14-49`. `wavelength_interval_to_sum` is "all" or
        [wave_min, wave_max] in the header's dispersion unit (or astropy quantities); `sub_fov_window` is "all" or
        [lon_min, lon_max, lat_min, lat_max] in arcsec (or quantities). `local_block` (rows, cols) or an int, multiples
        of 64 pixels: per-block cubes as in `Alignment`; (rows >= raster height, 64) gives one cube per band of 64 slit
        positions, i.e. per stretch of the scan's time."""
        super().__init__(large_fov_known_pointing=large_fov_known_pointing, small_fov_to_correct=small_fov_to_correct,
                         lag_crval1=lag_crval1, lag_crval2=lag_crval2, lag_cdelt1=lag_cdelt1, lag_cdelt2=lag_cdelt2,
                         lag_crota=lag_crota, display_progress_bar=display_progress_bar, lag_solar_r=lag_solar_r,
                         parallelism=parallelism, counts_cpu_max=counts_cpu_max, large_fov_window=large_fov_window,
                         small_fov_window=small_fov_window, path_save_figure=path_save_figure,
                         local_block=local_block)
        self.sub_fov_window = sub_fov_window
        self.coordinate_frame = None
        self.extend_pixel_size = None
        self.cut_from_center = None
        self.wavelength_interval_to_sum = wavelength_interval_to_sum

    def align_using_helioprojective(self, method='correlation', extend_pixel_size=False, cut_from_center=None,
                                    return_type="AlignmentResults", coefficient_l3: int = None):
        """`hdrshift/alignment_spice.py:66-120`."""
        self.lonlims = None
        self.latlims = None
        self.shape = None
        self.reference_date = None
        self.method = method
        self.coordinate_frame = "final_helioprojective"
        self.extend_pixel_size = extend_pixel_size
        self.cut_from_center = cut_from_center
        self.ang2pipi = True
        self._extract_imager_data_header()
        self.lon_ctype = "HPLN-TAN"
        self.lat_ctype = "HPLT-TAN"
        level = None
        if "L2" in self.small_fov_to_correct:
            level = 2
        elif "L3" in self.small_fov_to_correct:
            level = 3
        self._extract_spice_data_header(level=level, coeff=coefficient_l3)
        results = self._find_best_header_parameters()
        return self._wrap_results(results, return_type)

    def align_using_carrington(self, *args, **kwargs):
        raise NotImplementedError("AlignmentSpice.align_using_carrington calls a method that does not exist in the "
                                  "reference (alignment_spice.py:146); it is outside the device path")

    # ------------------------------------------------------------------------------------------------
    def _extract_imager_data_header(self):
        """`alignment_spice.py:182-187`: the large image is read as is (no PCi_j check)."""
        with _open_fits(self.large_fov_known_pointing) as hdul_large:
            self.data_large = np.array(hdul_large[self.large_fov_window].data.copy(), dtype=np.float64)
            self.hdr_large = hdul_large[self.large_fov_window].header.copy()

    def _extract_spice_data_header(self, level: int, coeff: int = None):
        """`alignment_spice.py:189-221`."""
        with _open_fits(self.small_fov_to_correct) as hdul_small:
            hdu = hdul_small[self.small_fov_window]
            dt = hdu.header.copy()["PC4_1"]
            if level == 2:
                self._prepare_spice_from_l2(hdu)
            elif level == 3:
                # the reference's own level-3 branch cannot run: `_prepare_spice_from_l3` indexes the [y, x, parameter]
                # data as `data[coeff, ...]` and leaves hdr_small without NAXIS1 / NAXIS2, which the search then needs
                # (`alignment_spice.py:341-356`, `utils/Util.py:287`); `pxlshift.AlignmentSpicePixel` handles L3 files
                raise NotImplementedError("level 3 (fitted) SPICE files: the reference's AlignmentSpice branch for "
                                          "them does not run either; use pxlshift.AlignmentSpicePixel")
            else:
                raise ValueError("level must be 2 or 3")
            for k in ("SOLAR_B0", "RSUN_REF", "DSUN_OBS", "CROTA"):
                self.hdr_small[k] = hdu.header[k]
            if self.extend_pixel_size:
                self._correct_solar_rotation(dt)

    def _correct_solar_rotation(self, dt):
        """`alignment_spice.py:223-248`: the raster steps against solar rotation, so structures are sampled with an
        effective CDELT1 = CDELT1 - dt * (helioprojective rotation rate) * cos(heliocentric longitude). Host-only
        header arithmetic, kept as the reference has it (EIT 171 rates for the 174 band; the phi range test of
        `:241` can never fire)."""
        b0 = np.deg2rad(self.hdr_small["SOLAR_B0"])
        band = self.hdr_large["WAVELNTH"]
        omega_car = np.deg2rad(360 / 25.38 / 86400)
        if band == 174:
            band = 171
        omega = omega_car + Util.diff_rot(b0, f"EIT {band}")
        rsun, dsun = self.hdr_small["RSUN_REF"], self.hdr_small["DSUN_OBS"]
        phi_rot = 1.004 * omega * rsun / (dsun - 1.004 * rsun)
        phi_rot = np.rad2deg(phi_rot) * 3600
        alpha = float(units.convert(self.hdr_small["CRVAL1"], self.hdr_small["CUNIT1"], "rad"))
        phi = np.arcsin(((dsun - 1.004 * rsun) / (1.004 * rsun)) * np.sin(alpha))
        dtx_old = float(units.convert(self.hdr_small["CDELT1"], self.hdr_small["CUNIT1"], "arcsec"))
        dtx_new = dtx_old - dt * phi_rot * np.cos(phi)
        self.hdr_small["CDELT1"] = float(units.convert(dtx_new, "arcsec", self.hdr_small["CUNIT1"]))

    def _prepare_spice_from_l2(self, hdu):
        """`alignment_spice.py:250-323`: 4-D L2 cube -> 2-D image + 2-D header."""
        header_spice = hdu.header
        ymin, ymax = Util.AlignSpiceUtil.vertical_edges_limits(header_spice)
        sw = SpiceWcs(header_spice)
        self.hdr_small = sw.xy_header().copy()
        shape4 = tuple(hdu.shape) if getattr(hdu, "shape", None) is not None else np.asarray(hdu.data).shape
        if isinstance(self.wavelength_interval_to_sum, str) and self.wavelength_interval_to_sum == "all":
            sel = np.ones(shape4[1], dtype=bool)
        elif type(self.wavelength_interval_to_sum).__name__ == "list":
            unit = str(header_spice.get("CUNIT%d" % sw.iwave, "nm")).strip()
            wave = sw.wavelength(np.arange(shape4[1]))
            lo = _value_in(self.wavelength_interval_to_sum[0], unit)
            hi = _value_in(self.wavelength_interval_to_sum[1], unit)
            sel = np.logical_and(wave >= lo, wave <= hi)
        else:
            raise ValueError("wavelength_interval_to_sum must be a [wave_min * u.angstrom, wave_max * u.angstrom] "
                             "or 'all' str ")
        raw = hdu.raw_big_endian() if hasattr(hdu, "raw_big_endian") else None
        if raw is not None and raw.ndim == 4 and raw.shape[0] == 1 and raw.dtype.itemsize == 4:
            # The float32 payload goes up as the file stores it; the device adds the selected planes in float64 in
            # ascending order, skipping NaN samples -- the bits of the host reduction below (numpy reduces the leading
            # axis of a C-ordered array plane by plane), without two float64 copies of the cube on the host
            # (25 MB -> 51 MB twice for a 40-plane raster: 45 ms of a 48 ms search).
            from .. import _ext
            self.data_small = _ext.spice_wave_sum(raw[0], sel, ymin, ymax).cpu().numpy()
        else:
            data_small = np.array(hdu.data.copy(), dtype=np.float64)
            data_small[:, :, :ymin, :] = np.nan
            data_small[:, :, ymax:, :] = np.nan
            self.data_small = np.nansum(data_small[0, sel, :, :], axis=0)
            self.data_small[:ymin, :] = np.nan
            self.data_small[ymax:, :] = np.nan
        if self.cut_from_center is not None:
            xlen = self.cut_from_center
            xmid = self.data_small.shape[1] // 2
            self.data_small[:, :(xmid - xlen // 2 - 1)] = np.nan
            self.data_small[:, (xmid + xlen // 2):] = np.nan
        if isinstance(self.sub_fov_window, str) and self.sub_fov_window == "all":
            pass
        elif type(self.sub_fov_window).__name__ == "list":
            w = sw.celestial()
            x, y = np.meshgrid(np.arange(shape4[3]), np.arange(shape4[2]))
            lon, lat = w.pixel_to_world(x, y)     # degrees, wcslib's longitude range
            lims = [_value_in(v, "arcsec") * units.factor("arcsec", "deg") for v in self.sub_fov_window]
            sel = (lon >= lims[0]) & (lon <= lims[1]) & (lat >= lims[2]) & (lat <= lims[3])
            self.data_small[~sel] = np.nan
        else:
            raise ValueError("sub_fov_window must be a [lon_min * u.arcsec, lon_max * u.arcsec,"
                             " lat_min * u.arcsec, lat_max * u.arcsec] or 'all' str ")
        self.hdr_small["NAXIS1"] = self.data_small.shape[1]
        self.hdr_small["NAXIS2"] = self.data_small.shape[0]
