"""Corrected L3 files of RICE tile-compressed float32 L2 windows are written tile-compressed, without a GPU: the table
and heap as read, the corrected header folded back into the table header (`AlignCommonUtil.write_corrected_fits`,
`fits_lite.CompImageHDU.with_header`)."""
import numpy as np
import pytest

SHIFT = [1.5, -2.25, 0.01, -0.02, 0.3]          # CRVAL1, CRVAL2 [arcsec], CDELT1, CDELT2 [arcsec], CROTA [deg]
BLANK = -2147483647
SUMS = [("CHECKSUM", "9aBa9ZAZ9aAa9YAZ"), ("DATASUM", "3211467342"), ("ZHECKSUM", "Ia5VJZ4TIa4TIZ4T"),
        ("ZDATASUM", "1183928431")]
STRUCTURAL = {"XTENSION", "BITPIX", "NAXIS", "NAXIS1", "NAXIS2", "PCOUNT", "GCOUNT"}

# (ZQUANTIZ method, ZBLANK, tile (width, height) or None for row tiles, pointing cards, window selector)
CASES = [
    (1, None, None, "CROTA", 1),
    (2, BLANK, (16, 5), "PC", -1),
    (0, BLANK, None, "PC", "EUI_WIN"),
    (1, BLANK, (13, 4), "CROTA2", "EUI_WIN"),
    (2, None, (37, 3), "none", 1),                 # no CROTA / PCi_j: the correction adds them
]


def _image(seed, nan):
    rng = np.random.default_rng(seed)
    img = (800 + 120 * rng.standard_normal((23, 37))).astype(np.float32)
    img[4, 9] = 0.0
    if nan:
        img[2, 3] = img[17, 36] = np.nan
    return img


def _cards(rot, extname="EUI_WIN"):
    cards = [("CTYPE1", "HPLN-TAN"), ("CTYPE2", "HPLT-TAN"), ("CUNIT1", "arcsec"), ("CUNIT2", "arcsec"),
             ("CRPIX1", 18.5), ("CRPIX2", 12.0), ("CDELT1", 0.492), ("CDELT2", 0.5), ("CRVAL1", -310.25),
             ("CRVAL2", 122.5), ("DATE-AVG", "2022-03-17T09:50:45.000")]
    if rot == "CROTA":
        cards.append(("CROTA", 2.5))
    elif rot == "CROTA2":
        cards.append(("CROTA2", -1.25))
    elif rot == "PC":
        cards += [("PC1_1", 0.9990482215818578), ("PC1_2", -0.04274115646396571), ("PC2_1", 0.04448431396958154),
                  ("PC2_2", 0.9990482215818578)]
    return cards + [("EXTNAME", extname), ("BUNIT", "DN/s")] + SUMS


def _write_input(path, case, seed=0):
    from oracle import rice
    method, blank, tile, rot, _ = case
    rice.write_compressed_image(path, _image(seed, blank is not None), extra_cards=_cards(rot), tile=tile,
                                quantize_scale=0.125, zdither0=seed + 11, method=method, blank=blank)


def _plain_copy(src, dst):
    """The same file with its compressed window replaced by a plain float32 image under the same image header."""
    from euispice_coreg_b200._compat import fits_lite
    h = fits_lite.open(src)
    img = np.zeros((h[1].header["NAXIS2"], h[1].header["NAXIS1"]), np.float32)
    fits_lite.writeto(dst, [h[0], fits_lite.ImageHDU(img, h[1].header)], overwrite=True)


def _oracle_decode(hdu):
    """Every tile of a compressed HDU decoded by oracle/rice.py (pure Python)."""
    from oracle import rice
    th, body = hdu.table_header, hdu._body
    nx, ny, tw, tht = th["ZNAXIS1"], th["ZNAXIS2"], th["ZTILE1"], th["ZTILE2"]
    rowb, nrows = th["NAXIS1"], th["NAXIS2"]
    table = np.frombuffer(body, np.uint8, rowb * nrows).reshape(nrows, rowb)
    dsc = np.ascontiguousarray(table[:, :8]).view(">i4")
    heap = body[rowb * nrows:]
    method = {"NO_DITHER": 0, "SUBTRACTIVE_DITHER_1": 1, "SUBTRACTIVE_DITHER_2": 2}[th["ZQUANTIZ"]]
    out = np.zeros((ny, nx), np.float32)
    n = 0
    for y0 in range(0, ny, tht):
        for x0 in range(0, nx, tw):
            w, h = min(tw, nx - x0), min(tht, ny - y0)
            q = rice.rice_decode(heap[dsc[n, 1]:dsc[n, 1] + dsc[n, 0]], w * h, th["ZVAL1"], th["ZVAL2"])
            zs, zz = np.ascontiguousarray(table[n, 8:24]).view(">f8")
            out[y0:y0 + h, x0:x0 + w] = rice.unquantize_tile(q, float(zs), float(zz), n + 1, th["ZDITHER0"],
                                                             method=method, blank=th.get("ZBLANK")).reshape(h, w)
            n += 1
    return out


def _card_list(header):
    """(key, value, comment) of every card; the comment of the cards `writeto` derives from the data is its own."""
    return [(k, header[k], "" if k in STRUCTURAL else header.comment(k)) for k in header.keys()]


@pytest.fixture
def no_decode(monkeypatch):
    from euispice_coreg_b200._compat import fits_lite

    def _decode(self, *a, **k):
        raise AssertionError("compressed tiles were decoded")
    monkeypatch.setattr(fits_lite.CompImageHDU, "_decode", _decode)


@pytest.mark.parametrize("case", CASES)
def test_selected_window_is_written_with_its_tiles(tmp_path, no_decode, case):
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.utils.Util import AlignCommonUtil
    src, out = str(tmp_path / "l2.fits"), str(tmp_path / "l3.fits")
    _write_input(src, case)
    AlignCommonUtil.write_corrected_fits(src, [case[-1]], out, corr=None, shift_arcsec=SHIFT)
    hin, hout = fits_lite.open(src), fits_lite.open(out)
    assert len(hout) == 2 and isinstance(hout[1], fits_lite.CompImageHDU)
    assert hout[1]._body == hin[1]._body                              # table and heap, byte for byte
    assert np.array_equal(_oracle_decode(hout[1]), _oracle_decode(hin[1]), equal_nan=True)
    assert hout[0].header == hin[0].header

    # the image header is, card for card, the one the plain path writes for the same cards and the same shift
    plain, plain_out = str(tmp_path / "plain.fits"), str(tmp_path / "plain_l3.fits")
    _plain_copy(src, plain)
    AlignCommonUtil.write_corrected_fits(plain, [case[-1]], plain_out, corr=None, shift_arcsec=SHIFT)
    want = fits_lite.open(plain_out)[1].header
    assert _card_list(hout[1].header) == _card_list(want)
    assert hout[1].header._commentary == want._commentary
    assert hout[1].header["CRVAL1"] == hin[1].header["CRVAL1"] + SHIFT[0]
    assert hout[1].header["PC1_1"] != hin[1].header.get("PC1_1")

    # the table's own cards as read, in their order, less the header checksums
    tin, tout = hin[1].table_header, hout[1].table_header
    own = [k for k in tin.keys() if fits_lite._is_table_card(k) and k not in ("CHECKSUM", "ZHECKSUM")]
    assert [k for k in tout.keys() if fits_lite._is_table_card(k)] == own
    assert all(tout[k] == tin[k] and tout.comment(k) == tin.comment(k) for k in own)
    assert "CHECKSUM" not in tout and "ZHECKSUM" not in tout
    assert (tout["DATASUM"], tout["ZDATASUM"]) == (tin["DATASUM"], tin["ZDATASUM"])


def test_unchanged_header_folds_back_to_the_table_header(tmp_path, no_decode):
    """`_table_header` inverts `_image_header`: only the stale header checksums go."""
    from euispice_coreg_b200._compat import fits_lite
    src = str(tmp_path / "l2.fits")
    _write_input(src, CASES[1])
    hdu = fits_lite.open(src)[1]
    th = hdu.table_header
    folded = fits_lite.CompImageHDU._table_header(th, hdu.header.copy())
    assert folded.items() == [(k, v) for k, v in th.items() if k not in ("CHECKSUM", "ZHECKSUM")]
    assert fits_lite.CompImageHDU._image_header(folded) == hdu.header


def test_plain_window_of_the_same_file_is_written_as_before(tmp_path, no_decode):
    """A file holding a compressed window and a plain one, both selected: the plain extension is written byte for byte
    as from a file that holds only it, the compressed one as from a file that holds only it."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.utils.Util import AlignCommonUtil
    comp, plain, mixed = (str(tmp_path / f"{n}.fits") for n in ("comp", "plain", "mixed"))
    _write_input(comp, CASES[3], seed=5)
    h = fits_lite.Header(_cards("PC", extname="PLAIN_WIN"))
    fits_lite.writeto(plain, [fits_lite.PrimaryHDU(), fits_lite.ImageHDU(_image(6, True) * 3, h)])
    comp_b, plain_b = (open(p, "rb").read() for p in (comp, plain))
    assert plain_b[2880:2880 + 8] == b"XTENSION"                      # the primary HDU is one header block
    with open(mixed, "wb") as f:
        f.write(comp_b + plain_b[2880:])
    outs = {}
    for name, src, windows in (("comp", comp, [1]), ("plain", plain, ["PLAIN_WIN"]), ("mixed", mixed, [1, "PLAIN_WIN"])):
        outs[name] = str(tmp_path / f"{name}_l3.fits")
        AlignCommonUtil.write_corrected_fits(src, windows, outs[name], corr=None, shift_arcsec=SHIFT)
    comp_o, plain_o, mixed_o = (open(outs[n], "rb").read() for n in ("comp", "plain", "mixed"))
    assert mixed_o == comp_o + plain_o[2880:]
    hdul = fits_lite.open(outs["mixed"])
    assert [type(x).__name__ for x in hdul] == ["PrimaryHDU", "CompImageHDU", "ImageHDU"]
    assert np.array_equal(hdul["PLAIN_WIN"].data, _image(6, True) * 3, equal_nan=True)


def test_compressed_copy_cannot_be_the_primary_hdu(tmp_path, no_decode):
    from euispice_coreg_b200._compat import fits_lite
    src = str(tmp_path / "l2.fits")
    _write_input(src, CASES[0])
    hdu = fits_lite.open(src)[1]
    with pytest.raises(ValueError):
        fits_lite.writeto(str(tmp_path / "bad.fits"), [hdu.with_header(hdu.header.copy())])
