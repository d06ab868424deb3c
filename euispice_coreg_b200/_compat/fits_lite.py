"""Dependency-free FITS reader/writer for image HDUs, plain or RICE tile-compressed.

Stands in for the `astropy.io.fits` calls of the reference's pointing-search path
(`hdrshift/alignment.py:299-316`, `utils/Util.py:106-159`, `synras/map_builder.py:106-131,192-203`).
Scope: primary + IMAGE extension HDUs, BITPIX in {8, 16, 32, 64, -32, -64}, BSCALE/BZERO,
string/logical/int/float cards, CONTINUE-less headers. Tile-compressed images (`ZIMAGE` binary tables with
`ZCMPTYPE = 'RICE_1'`, the form real Solar Orbiter L2 files come in; `utils/Util.py:144-145`) are read as
`CompImageHDU`: the header is folded back to an image header on the host, the pixels are decoded ON THE GPU
(`coreg_rice_decode`, one thread per tile) the first time `.data` is touched, so only the compressed heap crosses
PCIe. Writing is uncompressed, except for a `CompImageHDU.with_header` copy: it is written as a tile-compressed image
whose table and heap are the ones read, with the new image header folded back into the table header (no decoding,
no encoding, no GPU).

If astropy is importable the caller may still hand astropy headers to the package: everything
downstream only needs the mapping protocol (`in`, `[]`, `.copy()`, `.keys()`).
"""
from __future__ import annotations

import os
from collections import OrderedDict

import numpy as np

BLOCK = 2880
CARD = 80

_BITPIX_DTYPE = {8: ">u1", 16: ">i2", 32: ">i4", 64: ">i8", -32: ">f4", -64: ">f8"}
_DTYPE_BITPIX = {"u1": 8, "i2": 16, "i4": 32, "i8": 64, "f4": -32, "f8": -64}


class Header:
    """Ordered FITS header with the subset of the `astropy.io.fits.Header` mapping API the
    reference uses: `hdr[k]`, `hdr[k] = v`, `k in hdr`, `hdr.copy()`, `hdr.keys()`, `hdr.get`."""

    def __init__(self, cards=None):
        self._cards: "OrderedDict[str, tuple]" = OrderedDict()
        self._commentary: list[tuple[str, str]] = []
        if cards is not None:
            if isinstance(cards, Header):
                self._cards = OrderedDict(cards._cards)
                self._commentary = list(cards._commentary)
            else:
                items = cards.items() if hasattr(cards, "items") else cards
                for k, v in items:
                    self[k] = v

    # -- mapping protocol -------------------------------------------------
    @staticmethod
    def _norm(key):
        return str(key).strip().upper()

    def __contains__(self, key):
        return self._norm(key) in self._cards

    def __getitem__(self, key):
        k = self._norm(key)
        if k not in self._cards:
            raise KeyError(f"Keyword {key!r} not found.")
        return self._cards[k][0]

    def __setitem__(self, key, value):
        k = self._norm(key)
        comment = ""
        if isinstance(value, tuple) and len(value) == 2 and isinstance(value[1], str):
            value, comment = value
        elif k in self._cards:
            comment = self._cards[k][1]
        if isinstance(value, np.generic):
            value = value.item()
        self._cards[k] = (value, comment)

    def __delitem__(self, key):
        del self._cards[self._norm(key)]

    def __iter__(self):
        return iter(self._cards)

    def __len__(self):
        return len(self._cards)

    def keys(self):
        return self._cards.keys()

    def items(self):
        return [(k, v[0]) for k, v in self._cards.items()]

    def values(self):
        return [v[0] for v in self._cards.values()]

    def get(self, key, default=None):
        k = self._norm(key)
        return self._cards[k][0] if k in self._cards else default

    def comment(self, key):
        return self._cards[self._norm(key)][1]

    def copy(self):
        return Header(self)

    def update(self, other):
        for k, v in (other.items() if hasattr(other, "items") else other):
            self[k] = v

    def __eq__(self, other):
        if not isinstance(other, Header):
            return NotImplemented
        return self.items() == other.items()

    def __repr__(self):
        return "\n".join(_format_card(k, v, c).rstrip() for k, (v, c) in self._cards.items())


# --------------------------------------------------------------------------
# card parsing / formatting
# --------------------------------------------------------------------------
def _parse_value(field: str):
    """Parse the value field (columns 11-80) of a card -> (value, comment)."""
    s = field.strip()
    if not s:
        return None, ""
    if s[0] == "'":
        # quoted string; '' is an escaped quote
        i = 1
        out = []
        while i < len(s):
            if s[i] == "'":
                if i + 1 < len(s) and s[i + 1] == "'":
                    out.append("'")
                    i += 2
                    continue
                break
            out.append(s[i])
            i += 1
        val = "".join(out).rstrip()
        rest = s[i + 1:]
        comment = rest.split("/", 1)[1].strip() if "/" in rest else ""
        return val, comment
    if "/" in s:
        vs, comment = s.split("/", 1)
        vs, comment = vs.strip(), comment.strip()
    else:
        vs, comment = s, ""
    if vs == "T":
        return True, comment
    if vs == "F":
        return False, comment
    if not vs:
        return None, comment
    try:
        return int(vs), comment
    except ValueError:
        pass
    try:
        return float(vs.replace("D", "E").replace("d", "e")), comment
    except ValueError:
        return vs, comment


def _format_float(v: float) -> str:
    if v != v:
        return "'NaN'"
    s = repr(float(v)).upper()
    if "INF" in s:
        return "'%s'" % s
    if "E" in s:
        mant, exp = s.split("E")
        if "." not in mant:
            mant += ".0"
        s = f"{mant}E{int(exp):+03d}"
    elif "." not in s:
        s += ".0"
    return s


def _format_card(key: str, value, comment: str = "") -> str:
    if key in ("COMMENT", "HISTORY", ""):
        return f"{key:<8}{str(value)}"[:CARD].ljust(CARD)
    if isinstance(value, bool):
        vs = f"{'T' if value else 'F':>20}"
    elif isinstance(value, (int, np.integer)):
        vs = f"{int(value):>20d}"
    elif isinstance(value, (float, np.floating)):
        vs = f"{_format_float(float(value)):>20}"
    elif value is None:
        vs = " " * 20
    else:
        txt = str(value).replace("'", "''")
        vs = f"'{txt:<8}'"
        vs = f"{vs:<20}"
    if len(key) > 8:
        card = f"HIERARCH {key} = {vs.strip()}"
    else:
        card = f"{key:<8}= {vs}"
    if comment:
        card += f" / {comment}"
    return card[:CARD].ljust(CARD)


def _parse_header_block(raw: bytes):
    hdr = Header()
    for i in range(0, len(raw), CARD):
        card = raw[i:i + CARD].decode("ascii", errors="replace")
        key = card[:8].strip()
        if key == "END":
            return hdr, True
        if key in ("COMMENT", "HISTORY", ""):
            hdr._commentary.append((key, card[8:].rstrip()))
            continue
        if key == "HIERARCH" and "=" in card:
            k, rest = card[8:].split("=", 1)
            v, c = _parse_value(rest)
            hdr._cards[k.strip().upper()] = (v, c)
            continue
        if card[8:10] != "= ":
            continue
        v, c = _parse_value(card[10:])
        hdr._cards[key] = (v, c)
    return hdr, False


# --------------------------------------------------------------------------
# HDUs
# --------------------------------------------------------------------------
class ImageHDU:
    """Image HDU. Read from a file the pixel data stay in the (memory-mapped) file until `.data` is first touched:
    `raw_big_endian()` hands the payload over as it is stored (for a device-side byte swap), `read_window()` converts
    only a sub-window -- what the pointing search needs of a large image whose field the small image covers by a few
    hundred pixels."""
    is_primary = False

    def __init__(self, data=None, header=None, name=None):
        self.header = Header(header) if header is not None else Header()
        self._data = None if data is None else np.asarray(data)
        self._raw = None          # (big-endian ndarray view of the stored payload, bscale, bzero) until converted
        if name is not None:
            self.header["EXTNAME"] = name

    @classmethod
    def _from_file(cls, raw, header, bscale, bzero):
        h = cls(None, header)
        blank = header.get("BLANK", None) if raw.dtype.kind in "iu" else None
        h._raw = (raw, bscale, bzero) if blank is None else (raw, bscale, bzero, int(blank))
        return h

    @staticmethod
    def _convert(arr, bscale, bzero, blank=None):
        """Stored (big-endian) values -> what `astropy.io.fits` returns as `.data`."""
        dt = arr.dtype
        scaled = float(bscale) != 1.0 or float(bzero) != 0.0
        if scaled and dt.kind == "i" and float(bscale) == 1.0 and float(bzero) == float(2 ** (8 * dt.itemsize - 1)):
            return (arr.astype(np.int64) + int(bzero)).astype(f"u{dt.itemsize}")   # unsigned-integer convention
        if scaled:
            # same promotion rule as astropy: <=16-bit ints -> float32, everything else float64
            out_dt = np.float32 if (dt.kind in "iu" and dt.itemsize <= 2) or dt.itemsize == 4 and dt.kind == "f" \
                else np.float64
            out = arr.astype(out_dt) * out_dt(bscale) + out_dt(bzero)
            if blank is not None:         # astropy: BLANK pixels of an integer image that is scaled to float are NaN
                out[arr == blank] = np.nan
            return out
        return arr.astype(dt.newbyteorder("="))

    @property
    def data(self):
        if self._data is None and self._raw is not None:
            self._data = self._convert(*self._raw)
            self._raw = None
        return self._data

    @data.setter
    def data(self, value):
        self._data = None if value is None else np.asarray(value)
        self._raw = None

    @property
    def shape(self):
        if self._raw is not None:
            return self._raw[0].shape
        return None if self._data is None else self._data.shape

    def raw_big_endian(self):
        """The stored payload as a big-endian float array (no copy, read-only) when `.data` would hold exactly these
        values (BITPIX -32 / -64, no BSCALE / BZERO); None otherwise or once `.data` has been materialised."""
        if self._raw is None:
            return None
        raw, bscale, bzero = self._raw[:3]
        if raw.dtype.kind != "f" or float(bscale) != 1.0 or float(bzero) != 0.0:
            return None
        return raw

    def read_window(self, y0, y1, x0, x1):
        """`.data[y0:y1, x0:x1]` (2-D images) without converting the rest of the image."""
        if self._raw is not None and self._raw[0].ndim == 2:
            return self._convert(self._raw[0][y0:y1, x0:x1], *self._raw[1:])
        return np.array(self.data[y0:y1, x0:x1])

    @property
    def name(self):
        return self.header.get("EXTNAME", "PRIMARY" if self.is_primary else "")

    def copy(self):
        return type(self)(None if self.data is None else self.data.copy(), self.header.copy())


class PrimaryHDU(ImageHDU):
    is_primary = True


_TFORM_BYTES = {"L": 1, "X": 1, "B": 1, "I": 2, "J": 4, "K": 8, "A": 1, "E": 4, "D": 8, "C": 8, "M": 16, "P": 8, "Q": 16}
_Z_DROP = ("ZIMAGE", "ZCMPTYPE", "ZQUANTIZ", "ZDITHER0", "ZBLANK", "ZSCALE", "ZZERO", "TFIELDS", "THEAP", "ZMASKCMP",
           "ZSIMPLE", "ZEXTEND", "ZBLOCKED", "ZHECKSUM", "ZDATASUM", "CHECKSUM", "DATASUM")
_TABLE_CARDS = {"XTENSION", "BITPIX", "NAXIS", "NAXIS1", "NAXIS2", "PCOUNT", "GCOUNT", "ZNAXIS", "ZBITPIX", "ZPCOUNT",
                "ZGCOUNT", "ZTENSION", *_Z_DROP}
_TABLE_INDEXED = ("ZNAXIS", "ZTILE", "ZNAME", "ZVAL", "TTYPE", "TFORM", "TUNIT", "TDIM", "TSCAL", "TZERO", "TNULL", "TDISP")
# cover the header bytes, which a new image header changes; DATASUM / ZDATASUM cover the table and the pixels
_STALE_CHECKSUMS = ("CHECKSUM", "ZHECKSUM")


def _is_table_card(key):
    """A card of the binary table itself (structure, columns, compression, checksums), not of the image it holds."""
    return key in _TABLE_CARDS or any(key.startswith(p) and key[len(p):].isdigit() for p in _TABLE_INDEXED)


def _tform(tform):
    """'1PB(3241)' -> (repeat, code, element code of a variable-length array or None)."""
    t = str(tform).strip()
    i = 0
    while i < len(t) and t[i].isdigit():
        i += 1
    rep = int(t[:i]) if i else 1
    code = t[i].upper()
    sub = t[i + 1].upper() if code in "PQ" and len(t) > i + 1 else None
    return rep, code, sub


class CompImageHDU:
    """A tile-compressed image extension. `header` is the image's own header; `data` decodes on first access.

    `writeto` decodes an HDU as read and writes it as a plain IMAGE extension; it writes a `with_header` copy
    tile-compressed."""
    is_primary = False

    def __init__(self, table_header, body):
        self._thdr = table_header
        self._body = body
        self._data = None
        self.header = self._image_header(table_header)
        self.write_compressed = False

    @property
    def name(self):
        return self.header.get("EXTNAME", "")

    @property
    def table_header(self):
        """The binary table's header as read: structure, columns, `Z*` compression cards and the image's cards."""
        return self._thdr

    def with_header(self, header):
        """The same tiles under the image header `header` (typically a modified `.header.copy()`), to be written by
        `writeto` as a tile-compressed image: the table and its heap byte for byte as read, the header folded back
        into the table header (`_table_header`). Neither this HDU nor the copy decodes anything, so no GPU is needed."""
        if self._body is None:
            raise OSError("compressed payload already released")
        out = CompImageHDU(self._thdr, self._body)
        out.header = header
        out.write_compressed = True
        return out

    @staticmethod
    def _image_header(th):
        h = Header()
        naxis = int(th["ZNAXIS"])
        h["XTENSION"] = "IMAGE"
        h["BITPIX"] = int(th["ZBITPIX"])
        h["NAXIS"] = naxis
        for i in range(1, naxis + 1):
            h[f"NAXIS{i}"] = int(th[f"ZNAXIS{i}"])
        h["PCOUNT"] = int(th.get("ZPCOUNT", 0))
        h["GCOUNT"] = int(th.get("ZGCOUNT", 1))
        for k, (v, c) in th._cards.items():
            if not _is_table_card(k):
                h._cards[k] = (v, c)
        h._commentary = list(th._commentary)
        return h

    @staticmethod
    def _table_header(th, image_header):
        """Inverse of `_image_header`: the table header `th` with its image cards replaced by those of `image_header`.
        The table's own cards (`_is_table_card`) stay as read, in place, except the header checksums CHECKSUM and
        ZHECKSUM, which are dropped. An image card keeps its place in `th`, takes `image_header`'s value, or goes
        if `image_header` lacks it; cards new in `image_header` follow the table's cards. Structural image cards
        (BITPIX, NAXISn, BSCALE, ...) are left out, as `writeto` leaves them out of a plain image's header."""
        img = OrderedDict((k, vc) for k, vc in image_header._cards.items()
                          if not (_is_structural(k) or _is_table_card(k)))
        out = Header()
        for k, vc in th._cards.items():
            if _is_table_card(k):
                if k not in _STALE_CHECKSUMS:
                    out._cards[k] = vc
            elif k in img:
                out._cards[k] = img.pop(k)
        out._cards.update(img)
        out._commentary = list(image_header._commentary)
        return out

    @property
    def data(self):
        if self._data is None:
            self._data = self._decode(as_device=False)
            self._body = None
        return self._data

    @data.setter
    def data(self, value):
        self._data = None if value is None else np.asarray(value)
        self._body = None

    def device_data(self, out_dtype=None):
        """The decoded image as a CUDA tensor, without a round trip through the host (float images only)."""
        return self._decode(as_device=True, out_dtype=out_dtype)

    def copy(self):
        return ImageHDU(None if self.data is None else self.data.copy(), self.header.copy())

    def _decode(self, as_device, out_dtype=None):
        th, body = self._thdr, self._body
        if body is None:
            raise OSError("compressed payload already released")
        cmp = str(th.get("ZCMPTYPE", "")).strip().upper()
        if cmp not in ("RICE_1", "RICE_ONE"):
            raise NotImplementedError(f"ZCMPTYPE={cmp!r}: only RICE_1 tiles are decoded here (install astropy for others)")
        if int(th["ZNAXIS"]) != 2:
            raise NotImplementedError("only 2-D tile-compressed images are supported")
        nx, ny = int(th["ZNAXIS1"]), int(th["ZNAXIS2"])
        tw, tht = int(th.get("ZTILE1", nx)), int(th.get("ZTILE2", 1))
        row_bytes, n_rows = int(th["NAXIS1"]), int(th["NAXIS2"])
        params = {str(th[f"ZNAME{i}"]).strip().upper(): th[f"ZVAL{i}"] for i in range(1, 10) if f"ZNAME{i}" in th}
        blocksize, bytepix = int(params.get("BLOCKSIZE", 32)), int(params.get("BYTEPIX", 4))
        cols, off = {}, 0
        for i in range(1, int(th["TFIELDS"]) + 1):
            rep, code, sub = _tform(th[f"TFORM{i}"])
            width = _TFORM_BYTES[code] * (1 if code in "PQ" else rep)
            cols[str(th.get(f"TTYPE{i}", f"COL{i}")).strip().upper()] = (off, code, sub, rep)
            off += width
        if off != row_bytes or "COMPRESSED_DATA" not in cols:
            raise OSError("malformed tile-compressed table")
        table = np.frombuffer(body, dtype=np.uint8, count=row_bytes * n_rows).reshape(n_rows, row_bytes)
        theap = int(th.get("THEAP", row_bytes * n_rows))
        heap = memoryview(body)[theap:theap + int(th.get("PCOUNT", 0))]

        def column(name, dtype):
            o, code, _, rep = cols[name]
            w = np.dtype(dtype).itemsize
            return np.ascontiguousarray(table[:, o:o + w]).view(dtype).ravel()

        o, code, sub, _ = cols["COMPRESSED_DATA"]
        dsc = np.ascontiguousarray(table[:, o:o + (8 if code == "P" else 16)]).view(">i4" if code == "P" else ">i8")
        counts, offsets = dsc[:, 0].astype(np.int64), dsc[:, 1].astype(np.int64)
        zbitpix = int(th["ZBITPIX"])
        is_float = zbitpix < 0
        # tiles cfitsio could not quantise / compress carry an empty COMPRESSED_DATA descriptor and their pixels in
        # GZIP_COMPRESSED_DATA (gzip of the big-endian values) or UNCOMPRESSED_DATA: decoded here on the host and
        # patched into the device image below (the RICE kernel sees an empty stream for them)
        fallback = {}
        if np.any(counts <= 0):
            import zlib
            pix_dt = np.dtype({-32: ">f4", -64: ">f8", 8: "u1", 16: ">i2", 32: ">i4"}[zbitpix])
            tiles_x = (nx + tw - 1) // tw

            def var_column(name):
                o2, code2, sub2, _ = cols[name]
                d2 = np.ascontiguousarray(table[:, o2:o2 + (8 if code2 == "P" else 16)]).view(
                    ">i4" if code2 == "P" else ">i8")
                return d2[:, 0].astype(np.int64), d2[:, 1].astype(np.int64), sub2

            alt = {k: var_column(k) for k in ("GZIP_COMPRESSED_DATA", "UNCOMPRESSED_DATA") if k in cols}
            for row in np.nonzero(counts <= 0)[0]:
                x0, y0 = (row % tiles_x) * tw, (row // tiles_x) * tht
                w_, h_ = min(tw, nx - x0), min(tht, ny - y0)
                vals = None
                if "GZIP_COMPRESSED_DATA" in alt and alt["GZIP_COMPRESSED_DATA"][0][row] > 0:
                    c, o2, _ = alt["GZIP_COMPRESSED_DATA"]
                    raw = zlib.decompress(bytes(heap[o2[row]:o2[row] + c[row]]), 15 + 32)
                    vals = np.frombuffer(raw, dtype=pix_dt, count=w_ * h_)
                elif "UNCOMPRESSED_DATA" in alt and alt["UNCOMPRESSED_DATA"][0][row] > 0:
                    c, o2, sub2 = alt["UNCOMPRESSED_DATA"]
                    el = np.dtype({"E": ">f4", "D": ">f8", "J": ">i4", "I": ">i2", "B": "u1"}[sub2])
                    vals = np.frombuffer(bytes(heap[o2[row]:o2[row] + c[row] * el.itemsize]), dtype=el, count=w_ * h_)
                if vals is None:
                    raise OSError(f"tile {row}: no COMPRESSED_DATA, GZIP_COMPRESSED_DATA or UNCOMPRESSED_DATA payload")
                fallback[(int(y0), int(x0))] = vals.reshape(h_, w_)
            counts = np.maximum(counts, 0)
            offsets = np.where(counts > 0, offsets, 0)

        def patch(dev):
            for (y0, x0), tile in fallback.items():
                t = torch.from_numpy(np.ascontiguousarray(tile.astype(tile.dtype.newbyteorder("="))))
                dev[y0:y0 + tile.shape[0], x0:x0 + tile.shape[1]] = t.to(dev.device).to(dev.dtype)
            return dev

        from .. import _ext   # device decode: the CUDA library is required (no host fallback)
        torch = _ext._torch()
        if not torch.cuda.is_available():
            raise OSError("tile-compressed FITS images are decoded on the GPU: no CUDA device (or install astropy)")
        if is_float:
            method = {"NO_DITHER": 0, "NONE": 0, "SUBTRACTIVE_DITHER_1": 1, "SUBTRACTIVE_DITHER_2": 2}.get(
                str(th.get("ZQUANTIZ", "NO_DITHER")).strip().upper())
            if method is None:
                raise NotImplementedError(f"ZQUANTIZ={th.get('ZQUANTIZ')!r}")
            zscale = column("ZSCALE", ">f8").astype(np.float64) if "ZSCALE" in cols else np.full(n_rows, float(th["ZSCALE"]))
            zzero = column("ZZERO", ">f8").astype(np.float64) if "ZZERO" in cols else np.full(n_rows, float(th["ZZERO"]))
            blank = int(th["ZBLANK"]) if "ZBLANK" in th else None
            if "ZBLANK" in cols:
                zb = column("ZBLANK", ">i4")
                if zb.size and np.all(zb == zb[0]):
                    blank = int(zb[0])
                else:
                    raise NotImplementedError("per-tile ZBLANK values")
            odt = out_dtype or (torch.float32 if zbitpix == -32 else torch.float64)
            dev = patch(_ext.rice_decode(heap, offsets, counts, tw, tht, nx, ny, blocksize, bytepix, zscale, zzero,
                                         method, int(th.get("ZDITHER0", 1)), blank, odt))
            return dev if as_device else dev.cpu().numpy()
        dev = patch(_ext.rice_decode(heap, offsets, counts, tw, tht, nx, ny, blocksize, bytepix))
        if as_device:
            return dev
        arr = dev.cpu().numpy().astype({8: np.uint8, 16: np.int16, 32: np.int32}[zbitpix])
        bscale, bzero = float(th.get("BSCALE", 1)), float(th.get("BZERO", 0))
        if bscale != 1.0 or bzero != 0.0:
            if bscale == 1.0 and bzero == float(2 ** (zbitpix - 1)) and zbitpix > 8:
                arr = (arr.astype(np.int64) + int(bzero)).astype(f"u{zbitpix // 8}")
            else:
                odt = np.float32 if zbitpix <= 16 else np.float64
                arr = arr.astype(odt) * odt(bscale) + odt(bzero)
        return arr


class HDUList(list):
    def __getitem__(self, key):
        if isinstance(key, str):
            k = key.strip().upper()
            for h in self:
                if str(h.name).strip().upper() == k:
                    return h
            raise KeyError(f"Extension {key!r} not found.")
        return list.__getitem__(self, key)

    def close(self):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def writeto(self, path, overwrite=False):
        writeto(path, self, overwrite=overwrite)


def _data_nbytes(hdr: Header) -> int:
    naxis = int(hdr.get("NAXIS", 0))
    if naxis == 0:
        return 0
    n = 1
    for i in range(1, naxis + 1):
        n *= int(hdr[f"NAXIS{i}"])
    n *= abs(int(hdr["BITPIX"])) // 8
    n *= int(hdr.get("GCOUNT", 1))
    n += int(hdr.get("PCOUNT", 0))
    return n


def open(path, mode="readonly", **_):  # noqa: A001 - mirrors astropy.io.fits.open
    """Open a FITS file: headers are parsed, image payloads stay in the memory-mapped file until used. Returns an
    `HDUList`."""
    import mmap
    with builtins_open(os.fspath(path), "rb") as f:
        try:
            buf = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
        except (ValueError, OSError):       # empty file, or a file system without mmap
            buf = f.read()
    hdus = HDUList()
    pos = 0
    first = True
    while pos < len(buf):
        raw = b""
        done = False
        hdr = Header()
        while not done:
            if pos >= len(buf):
                if first:
                    raise OSError(f"{path}: truncated FITS header")
                return hdus
            blk = buf[pos:pos + BLOCK]
            pos += BLOCK
            part, done = _parse_header_block(blk)
            hdr._cards.update(part._cards)
            hdr._commentary.extend(part._commentary)
        if first and "SIMPLE" not in hdr:
            raise OSError(f"{path}: not a FITS file (no SIMPLE card)")
        nbytes = _data_nbytes(hdr)
        data = None
        xt = str(hdr.get("XTENSION", "IMAGE")).strip().upper()
        if nbytes and (first or xt == "IMAGE"):
            naxis = int(hdr["NAXIS"])
            shape = tuple(int(hdr[f"NAXIS{i}"]) for i in range(naxis, 0, -1))
            dt = np.dtype(_BITPIX_DTYPE[int(hdr["BITPIX"])])
            arr = np.frombuffer(buf, dtype=dt, count=int(np.prod(shape)), offset=pos).reshape(shape)
            data = (arr, hdr.get("BSCALE", 1), hdr.get("BZERO", 0))
        elif nbytes and xt == "BINTABLE" and hdr.get("ZIMAGE", False):
            hdus.append(CompImageHDU(hdr, bytes(buf[pos:pos + nbytes])))
            pos += ((nbytes + BLOCK - 1) // BLOCK) * BLOCK
            first = False
            continue
        pos += ((nbytes + BLOCK - 1) // BLOCK) * BLOCK
        cls = PrimaryHDU if first else ImageHDU
        hdus.append(cls(None, hdr) if data is None else cls._from_file(data[0], hdr, data[1], data[2]))
        first = False
    return hdus


import builtins  # noqa: E402

builtins_open = builtins.open


def _structural_cards(hdu, primary: bool):
    data = hdu.data
    cards = []
    if primary:
        cards.append(("SIMPLE", True, "conforms to FITS standard"))
    else:
        cards.append(("XTENSION", "IMAGE", "Image extension"))
    if data is None:
        cards += [("BITPIX", 8, ""), ("NAXIS", 0, "")]
    else:
        key = data.dtype.newbyteorder("=").str[1:]
        if key not in _DTYPE_BITPIX:
            raise TypeError(f"unsupported FITS dtype {data.dtype}")
        cards += [("BITPIX", _DTYPE_BITPIX[key], "array data type"), ("NAXIS", data.ndim, "")]
        for i, n in enumerate(reversed(data.shape), 1):
            cards.append((f"NAXIS{i}", int(n), ""))
    if primary:
        cards.append(("EXTEND", True, ""))
    else:
        cards += [("PCOUNT", 0, ""), ("GCOUNT", 1, "")]
    return cards


_STRUCTURAL = {"SIMPLE", "XTENSION", "BITPIX", "NAXIS", "EXTEND", "PCOUNT", "GCOUNT", "BSCALE", "BZERO"}


def _is_structural(key):
    """A card `writeto` derives from the data of an image HDU rather than copying it from the header."""
    return key in _STRUCTURAL or (key.startswith("NAXIS") and key[5:].isdigit())


def _header_bytes(cards, commentary):
    raw = "".join([*cards, *(f"{k:<8}{txt}"[:CARD].ljust(CARD) for k, txt in commentary), "END".ljust(CARD)])
    raw = raw.encode("ascii", errors="replace")
    return raw + b" " * ((-len(raw)) % BLOCK)


def writeto(path, hdus, overwrite=False):
    """Write an `HDUList` (or a single HDU) as a FITS file: image HDUs uncompressed, `CompImageHDU`s as read decoded
    to plain IMAGE extensions, `CompImageHDU.with_header` copies as tile-compressed images."""
    path = os.fspath(path)
    if os.path.exists(path) and not overwrite:
        raise OSError(f"File {path!r} already exists.")
    if isinstance(hdus, ImageHDU):
        hdus = [hdus]
    out = bytearray()
    for idx, hdu in enumerate(hdus):
        primary = idx == 0
        if isinstance(hdu, CompImageHDU) and hdu.write_compressed:
            if primary:
                raise ValueError("a tile-compressed image cannot be the primary HDU")
            if hdu._body is None:
                raise OSError("compressed payload already released")
            th = CompImageHDU._table_header(hdu.table_header, hdu.header)
            out += _header_bytes([_format_card(k, v, c) for k, (v, c) in th._cards.items()], th._commentary)
            out += hdu._body + b"\0" * ((-len(hdu._body)) % BLOCK)
            continue
        cards = [_format_card(k, v, c) for k, v, c in _structural_cards(hdu, primary)]
        for k, (v, c) in hdu.header._cards.items():
            if _is_structural(k):
                continue
            cards.append(_format_card(k, v, c))
        out += _header_bytes(cards, hdu.header._commentary)
        if hdu.data is not None:
            d = np.ascontiguousarray(hdu.data)
            d = d.astype(d.dtype.newbyteorder(">"))
            b = d.tobytes()
            out += b + b"\0" * ((-len(b)) % BLOCK)
    tmp = path + ".tmp~"
    with builtins_open(tmp, "wb") as f:
        f.write(out)
    os.replace(tmp, path)


def getheader(path, ext=0):
    return open(path)[ext].header


def getdata(path, ext=0):
    return open(path)[ext].data
