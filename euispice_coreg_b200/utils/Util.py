"""Host-side mirror of the reference's `utils/Util.py` for the pointing-search path.

Same class / function names, argument meaning and error behaviour as the reference
(`utils/Util.py:76-215, 283-312, 430-455`); the per-pixel work (pixel->world grids, spline
resampling) runs on the device through the C ABI (`_ext`). Angles that the reference returns as
`astropy.units.Quantity` come back as plain float64 ndarrays in DEGREES (astropy is optional here).
"""
from __future__ import annotations

import warnings

import numpy as np

from .. import _ext
from .._compat import fits_lite, units
from .._compat.wcs import TanWcs


def _fits():
    """astropy.io.fits when it is installed, otherwise the bundled minimal reader/writer."""
    try:  # pragma: no cover - astropy is absent from the build image
        from astropy.io import fits
        return fits
    except Exception:
        return fits_lite


def _is_float32_rice(hdu):
    """A fits_lite RICE_1 tile-compressed float32 image: its tiles decode to the `<f4` pixels a corrected copy holds."""
    if not isinstance(hdu, fits_lite.CompImageHDU):
        return False
    th = hdu.table_header
    return str(th.get("ZCMPTYPE", "")).strip().upper() in ("RICE_1", "RICE_ONE") and int(th["ZBITPIX"]) == -32


class AlignCommonUtil:

    @staticmethod
    def ang2pipi(ang, unit="deg"):
        """put angle between ]-180, +180] deg (`utils/Util.py:76-80`). `ang` is a plain array in `unit`
        (or any object with `.value`/`.unit`)."""
        if hasattr(ang, "unit") and hasattr(ang, "value"):
            return units.ang2pipi(ang.value, ang.unit)
        return units.ang2pipi(ang, unit)

    @staticmethod
    def interpol2d(image, x, y, fill, order, dst=None):
        """`scipy.ndimage.map_coordinates(image, [y, x], order, mode='constant', cval=fill,
        prefilter=False)` evaluated on the GPU (`utils/Util.py:82-104`). Like the reference, the result is
        written into `dst` (its dtype decides the output precision) or returned with `image.dtype`."""
        import torch
        image = np.asarray(image)
        if image.dtype not in (np.float32, np.float64):
            image = image.astype(np.float64)
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        out_dtype = np.dtype(image.dtype if dst is None else dst.dtype)
        dev_dtype = torch.float32 if out_dtype == np.float32 else torch.float64
        d_img = torch.from_numpy(np.ascontiguousarray(image)).cuda()
        d_x = torch.from_numpy(x).cuda()
        d_y = torch.from_numpy(y).cuda()
        res = _ext.map_coordinates(d_img, d_y, d_x, order, fill, dev_dtype).cpu().numpy()
        if dst is None:
            return res.astype(out_dtype, copy=False)
        dst[...] = res.astype(out_dtype, copy=False).reshape(dst.shape)
        return None

    # ------------------------------------------------------------------ header correction / FITS writing
    @staticmethod
    def _check_and_create_pcij_crota_hdr(hdr):
        """`utils/Util.py:217-245`."""
        if "PC1_1" not in hdr:
            warnings.warn("PCi_j matrix not found in header of the FITS file to align. Adding it to the header.")
            if "CROTA" in hdr:
                crot = hdr["CROTA"]
            elif "CROTA2" in hdr:
                crot = hdr["CROTA2"]
            else:
                hdr["CROTA"] = 0.0
                crot = 0.0
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

    @staticmethod
    def correct_pointing_header(header, lag_cdelt1, lag_cdelt2, lag_crota, lag_crval1, lag_crval2):
        """Apply a (sub-lag) shift to CRVAL/CDELT/CROTA/PCi_j in place (`utils/Util.py:163-215`).
        Shifts are in arcsec (degrees for `lag_crota`)."""
        AlignCommonUtil._check_and_create_pcij_crota_hdr(header)
        if header["PC1_1"] > 1.0:
            warnings.warn(f'header["PC1_1"]={header["PC1_1"]}, set it to 1.0')
            header["PC1_1"] = 1.0
            header["PC2_2"] = 1.0
            header["PC1_2"] = 0.0
            header["PC2_1"] = 0.0
            header["CROTA"] = 0.0
        change_pcij = False
        if lag_crval1 is not None:
            header["CRVAL1"] = header["CRVAL1"] + float(units.convert(lag_crval1, "arcsec", header["CUNIT1"]))
        if lag_crval2 is not None:
            header["CRVAL2"] = header["CRVAL2"] + float(units.convert(lag_crval2, "arcsec", header["CUNIT2"]))
        key_rota = None
        if "CROTA" in header:
            key_rota = "CROTA"
            crota = header[key_rota]
        elif "CROTA2" in header:
            key_rota = "CROTA2"
            crota = header[key_rota]
        else:
            crota = float(np.rad2deg(np.arccos(header["PC1_1"])))
            s = -np.sign(header["PC1_2"]) + (header["PC1_2"] == 0.0)
            crota = crota * s
        if lag_crota is not None:
            crota += lag_crota
            if key_rota is not None:
                header[key_rota] = float(crota)
            change_pcij = True
        if lag_cdelt1 is not None:
            header["CDELT1"] = header["CDELT1"] + float(units.convert(lag_cdelt1, "arcsec", header["CUNIT1"]))
            change_pcij = True
        if lag_cdelt2 is not None:
            header["CDELT2"] = header["CDELT2"] + float(units.convert(lag_cdelt2, "arcsec", header["CUNIT2"]))
            change_pcij = True
        if change_pcij:
            theta = float(units.convert(crota, "deg", "rad"))
            lam = header["CDELT2"] / header["CDELT1"]
            header["PC1_1"] = float(np.cos(theta))
            header["PC2_2"] = float(np.cos(theta))
            header["PC1_2"] = float(-lam * np.sin(theta))
            header["PC2_1"] = float((1 / lam) * np.sin(theta))

    @staticmethod
    def write_corrected_fits(path_to_l2_input: str, window_list_to_apply_shift, path_to_l3_output: str, corr,
                             lag_crval1=None, lag_crval2=None, lag_crota=None, lag_cdelt1=None, lag_cdelt2=None,
                             shift_arcsec=None):
        """Copy the input FITS, correcting the headers of the selected windows (`utils/Util.py:106-159`).

        The reference writes a selected window's pixels as `np.array(data, dtype="<f4")`. Without astropy, a selected
        RICE_1 tile-compressed window with ZBITPIX = -32 decodes to exactly those float32 values, so it is written as
        a tile-compressed image: the corrected header folded into the table header, the table and the heap byte for
        byte as read (`fits_lite.CompImageHDU.with_header`). Nothing is decoded, quantised or encoded, and no GPU is
        needed. astropy would re-quantise the pixels when it re-compresses such a window; that output is not restated
        here, because neither astropy nor cfitsio is a dependency it could be pinned against. Any other selected
        compressed window is decoded (on the GPU) and written as a float32 IMAGE extension holding the `<f4` cast.
        A compressed HDU that is not selected is, as before, decoded and written as a plain image."""
        fits = _fits()
        if shift_arcsec is None:
            max_index = np.unravel_index(np.nanargmax(corr), corr.shape)
            shift_arcsec = [lag_crval1[max_index[0]], lag_crval2[max_index[1]], lag_cdelt1[max_index[2]],
                            lag_cdelt2[max_index[3]], lag_crota[max_index[4]]]
        n_corrected = 0
        with fits.open(path_to_l2_input) as hdul:
            hdul_out = fits.HDUList()
            for ii in range(len(hdul)):
                hdu = hdul[ii]
                extname = hdu.header["EXTNAME"] if "EXTNAME" in hdu.header else "nothing98695"
                if (extname in window_list_to_apply_shift) or (ii in window_list_to_apply_shift) or \
                        ((ii - len(hdul)) in window_list_to_apply_shift):
                    header = hdu.header.copy()
                    AlignCommonUtil.correct_pointing_header(
                        header, lag_crval1=shift_arcsec[0], lag_crval2=shift_arcsec[1], lag_cdelt1=shift_arcsec[2],
                        lag_cdelt2=shift_arcsec[3], lag_crota=shift_arcsec[4])
                    if _is_float32_rice(hdu):
                        # never touches `.data`: decoding would release the compressed tiles
                        hdu_out = hdu.with_header(header)
                    else:
                        data = np.array(hdu.data.copy(), dtype="<f4")
                        # HDU kind preserved (Primary / Image / CompImage when astropy provides it)
                        cls = fits_lite.ImageHDU if isinstance(hdu, fits_lite.CompImageHDU) else type(hdu)
                        hdu_out = cls(data=data, header=header)
                        if hasattr(hdu_out, "verify"):
                            hdu_out.verify("silentfix")
                    n_corrected += 1
                else:
                    hdu_out = hdu
                hdul_out.append(hdu_out)
            hdul_out.writeto(path_to_l3_output, overwrite=True)
        if n_corrected == 0:
            raise ValueError("has not corrected any window.")


class AlignEUIUtil:

    @staticmethod
    def extract_EUI_coordinates(hdr, dsun=True, lon_ctype="HPLN-TAN", lat_ctype="HPLT-TAN", as_device=False):
        """Longitude / latitude [deg, wrapped to (-180, 180]] of every pixel of `hdr`'s image
        (`utils/Util.py:283-312`), computed on the GPU (K3). With `as_device=True` the two float64 CUDA
        tensors are returned instead of numpy arrays."""
        if lon_ctype != "HPLN-TAN" or lat_ctype != "HPLT-TAN":
            raise NotImplementedError("only the HPLN-TAN / HPLT-TAN pair is on the device path")
        w = TanWcs.from_header(hdr)
        lng, lat = _ext.tan_pix2world(w, w.naxis1, w.naxis2, wrap_pipi=True)
        if not as_device:
            lng, lat = lng.cpu().numpy(), lat.cpu().numpy()
        if dsun:
            return lng, lat, hdr["DSUN_OBS"]
        return lng, lat


def diff_rot(lat, wvl="default"):
    """`AlignEUIUtil.diff_rot` (`utils/Util.py:314-345`): omega_diff(lat) - omega_Carrington [rad / s]; lat in
    radians; A + B sin^2 + C sin^4 in deg / day from Hortin (2003) per EIT band."""
    p = {"EIT 171": (14.56, -2.65, 0.96), "EIT 195": (14.50, -2.14, 0.66), "EIT 284": (14.60, -0.71, -1.18),
         "EIT 304": (14.51, -3.12, 0.34)}
    p["default"] = p["EIT 195"]
    a, b, c = p[wvl]
    a_car = 360 / 25.38
    corr = a - a_car + b * np.sin(lat) ** 2 + c * np.sin(lat) ** 4
    return np.deg2rad(corr / 86400)


class PlotFits:
    """Only the grid helper the pointing search uses (`utils/Util.py:874-904`); plotting lives in `plot/`."""

    @staticmethod
    def build_regular_grid(longitude, latitude, lonlims=None, latlims=None):
        """Regular lon / lat grid [deg] spanning the image's footprint at its own sampling. `longitude`, `latitude`:
        degrees, already wrapped to (-180, 180] (what `extract_EUI_coordinates` returns); limits in degrees.
        Returns (longitude_grid, latitude_grid, dlon, dlat), all in degrees."""
        x = np.abs(longitude[0, 1] - longitude[0, 0])
        y = np.abs(latitude[0, 1] - latitude[0, 0])
        dlon = np.sqrt(x ** 2 + y ** 2)
        x = np.abs(longitude[1, 0] - longitude[0, 0])
        y = np.abs(latitude[1, 0] - latitude[0, 0])
        dlat = np.sqrt(x ** 2 + y ** 2)
        longitude1d = np.arange(np.min(longitude), np.max(longitude), dlon)
        latitude1d = np.arange(np.min(latitude), np.max(latitude), dlat)
        if (lonlims is not None) or (latlims is not None):
            longitude1d = longitude1d[(longitude1d > lonlims[0]) & (longitude1d < lonlims[1])]
            latitude1d = latitude1d[(latitude1d > latlims[0]) & (latitude1d < latlims[1])]
        longitude_grid, latitude_grid = np.meshgrid(longitude1d, latitude1d)
        return longitude_grid, latitude_grid, dlon, dlat


AlignEUIUtil.diff_rot = staticmethod(diff_rot)


class AlignSpiceUtil:

    @staticmethod
    def slit_pxl(header):
        """First and last pixel of the SPICE slit (`utils/Util.py:430-448`)."""
        ybin = header["NBIN2"]
        h_detector = 1024 / ybin
        if header["DETECTOR"] == "SW":
            h_slit = 600 / ybin
        elif header["DETECTOR"] == "LW":
            h_slit = 626 / ybin
        else:
            raise ValueError(f"unknown detector: {header['DETECTOR']}")
        slit_beg = (h_detector - h_slit) / 2
        slit_end = h_detector - slit_beg
        slit_beg = slit_beg - header["PXBEG2"] / ybin + 1
        slit_end = slit_end - header["PXBEG2"] / ybin + 1
        return int(np.ceil(slit_beg)), int(np.floor(slit_end))

    @staticmethod
    def vertical_edges_limits(header):
        """`utils/Util.py:450-455`."""
        iymin, iymax = AlignSpiceUtil.slit_pxl(header)
        iymin += int(20 / header["NBIN2"])
        iymax -= int(20 / header["NBIN2"])
        return iymin, iymax
