"""Minimal stand-ins for the astropy pieces the reference's hot path leans on.

The reference imports astropy for FITS I/O, units and WCS (`hdrshift/alignment.py:6-20`,
`utils/Util.py:3-17`). astropy is not installed in this image and cannot be fetched, so the
host layer ships small, dependency-free equivalents:

* `fits_lite`  -- read/write image HDUs, plain or RICE tile-compressed, + headers (replaces `astropy.io.fits`)
* `units`      -- arcsec/arcmin/deg/rad conversions (replaces `astropy.units` on this path)
* `wcs`        -- header -> TAN constants and host pixel<->world (replaces `astropy.wcs.WCS`)
* `timeutil`   -- ISO-8601 FITS dates -> seconds/days (replaces `astropy.time.Time` differences)
"""
