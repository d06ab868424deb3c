"""Jitter correction and `write_corrected_fits` on RICE tile-compressed float32 L2 frames: the same cubes, headers and
decoded pixels as the same runs over plain copies holding the device-decoded pixels, with every L3 file written
tile-compressed from the L2 tiles."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

JC_LAG = np.arange(-4.0, 4.1, 0.5)
JC_GRID = dict(lonlims=(249.3, 250.7), latlims=(-2.6, -1.4), shape=[120, 110])
STRUCTURAL = {"XTENSION", "BITPIX", "NAXIS", "NAXIS1", "NAXIS2", "PCOUNT", "GCOUNT"}
# row tiles with SUBTRACTIVE_DITHER_1, then 2-D tiles with SUBTRACTIVE_DITHER_2 and a ZBLANK
STORAGE = [dict(tile=None, method=1), dict(tile=(32, 12), method=2, blank=-2147483647)]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def frames(torch_cuda, tmp_path_factory):
    """Five jittered frames as compressed L2 files (primary + RICE float32 extension), and plain copies (primary +
    float32 IMAGE extension) holding the device-decoded pixels under the same image headers."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200._synth.scene import make_pair, master_scene, small_spec
    from oracle import rice
    d = tmp_path_factory.mktemp("cl3")
    true = (-12.0, 8.0)
    sky = master_scene(small_spec(96, 160, true_crval=true))
    comp, plain = [], []
    for i, jit in enumerate([(0.0, 0.0), (1.3, -0.8), (-2.1, 0.4), (0.6, 2.2), (-0.9, -1.5)]):
        spec = small_spec(96, 160, true_crval=true, jitter=jit, true_shift=jit, noise_seed=500 + i,
                          date=f"2022-03-17T09:5{i}:45.000")
        h = fits_lite.open(make_pair(str(d), spec, tag=f"j{i}", sky=sky, write_large=False)[1])[0]
        cards = [(k, h.header[k]) for k in h.header.keys() if k not in ("SIMPLE", "EXTEND") and k not in STRUCTURAL]
        cards += [("EXTNAME", "EUI_IMAGE"), ("CHECKSUM", "9aBa9ZAZ9aAa9YAZ"), ("DATASUM", "3211467342")]
        pc, pp = str(d / f"c{i}.fits"), str(d / f"p{i}.fits")
        rice.write_compressed_image(pc, h.data.astype(np.float32), extra_cards=cards, quantize_scale=1.0 / 64,
                                    zdither0=i + 1, **STORAGE[i % 2])
        c = fits_lite.open(pc)
        fits_lite.writeto(pp, [c[0], fits_lite.ImageHDU(c[1].device_data().cpu().numpy(), c[1].header)])
        comp.append(pc)
        plain.append(pp)
    return comp, plain


def _card_list(header):
    return [(k, header[k], "" if k in STRUCTURAL else header.comment(k)) for k in header.keys()]


def _assert_l3_pair(torch, l3_comp, l3_plain, l2_comp):
    """The compressed L3 file: L2's tiles, the plain L3's headers, and pixels decoding to the L2's, bit for bit."""
    from euispice_coreg_b200._compat import fits_lite
    c, p, l2 = fits_lite.open(l3_comp), fits_lite.open(l3_plain), fits_lite.open(l2_comp)
    assert len(c) == len(p) == 2 and isinstance(c[1], fits_lite.CompImageHDU)
    assert c[1]._body == l2[1]._body
    assert _card_list(c[0].header) == _card_list(p[0].header)
    assert _card_list(c[1].header) == _card_list(p[1].header)
    got, want = c[1].device_data(), l2[1].device_data()
    assert got.dtype == want.dtype == torch.float32
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    assert np.array_equal(got.cpu().numpy().view(np.int32), p[1].data.view(np.int32))


@pytest.mark.parametrize("method", ["carrington", "helioprojective"])
def test_jitter_correction_of_compressed_frames(torch_cuda, frames, tmp_path, method):
    """Sublists [0, 1, 2] and [2, 3, 4]: the second reads its reference back from the compressed L3 file of frame 2."""
    from euispice_coreg_b200.jitter_correction.jitter_correction import jitter_correction_imagers
    kw = dict(JC_GRID, method_carrington_reprojection="fa") if method == "carrington" else {}
    runs = {}
    for name, paths in zip(("comp", "plain"), frames):
        out = tmp_path / name
        out.mkdir()
        runs[name] = (out, jitter_correction_imagers(paths, str(out), lag_crval1=JC_LAG, lag_crval2=JC_LAG,
                                                      sublist_length=2, overlap=1, alignement_method=method, **kw))
    (out_c, res_c), (out_p, res_p) = runs["comp"], runs["plain"]
    assert len(res_c) == len(res_p) == 4
    for a, b in zip(res_c, res_p):
        assert np.array_equal(a.corr, b.corr, equal_nan=True)
        assert a.max_index == b.max_index and a.shift_arcsec == b.shift_arcsec
    assert any(float(r.shift_arcsec[0]) != 0.0 for r in res_c)          # the L3 headers do move
    comp, plain = frames
    name = os.path.basename
    assert (out_c / name(comp[0])).read_bytes() == open(comp[0], "rb").read()     # the reference, copied verbatim
    for k in range(1, 5):
        _assert_l3_pair(torch_cuda, str(out_c / name(comp[k])), str(out_p / name(plain[k])), comp[k])


def test_alignment_writes_a_compressed_l3_file(torch_cuda, frames, tmp_path):
    from euispice_coreg_b200.hdrshift import Alignment
    lags = dict(lag_crval1=JC_LAG, lag_crval2=JC_LAG, lag_cdelt1=[0], lag_cdelt2=[0], lag_crota=[0])
    comp, plain = frames
    outs = []
    for paths, tag in ((comp, "c"), (plain, "p")):
        r = Alignment(paths[0], paths[3], parallelism=True, **lags).align_using_helioprojective()
        outs.append(str(tmp_path / f"{tag}_l3.fits"))
        r.write_corrected_fits([-1], path_to_l3_output=outs[-1])
    _assert_l3_pair(torch_cuda, outs[0], outs[1], comp[3])


def test_compressed_int16_window_is_written_as_a_plain_float32_image(torch_cuda, tmp_path):
    """Not a float32 image, so the tiles cannot stand for the `<f4` pixels: decoded and written as a float32 IMAGE."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.utils.Util import AlignCommonUtil
    from oracle import rice
    rng = np.random.default_rng(4)
    img = (1000 + np.cumsum(rng.integers(-40, 41, (30, 70)), axis=1)).astype(np.int16)
    cards = [("CUNIT1", "arcsec"), ("CUNIT2", "arcsec"), ("CDELT1", 0.492), ("CDELT2", 0.492), ("CRVAL1", 15.0),
             ("CRVAL2", -7.5), ("CROTA", 1.5), ("BSCALE", 0.5), ("BZERO", 20.0), ("EXTNAME", "INT_WIN")]
    src, out = str(tmp_path / "l2.fits"), str(tmp_path / "l3.fits")
    rice.write_compressed_image(src, img, extra_cards=cards, tile=(16, 8), bytepix=2)
    shift = [2.0, -1.0, 0.0, 0.0, 0.25]
    AlignCommonUtil.write_corrected_fits(src, ["INT_WIN"], out, corr=None, shift_arcsec=shift)
    l2, l3 = fits_lite.open(src), fits_lite.open(out)
    assert type(l3[1]) is fits_lite.ImageHDU and l3[1].header["BITPIX"] == -32
    assert "BSCALE" not in l3[1].header and "BZERO" not in l3[1].header
    want = np.array(l2[1].data, dtype="<f4")
    assert np.array_equal(want, img.astype(np.float32) * 0.5 + 20.0)
    assert l3[1].data.dtype == np.float32 and np.array_equal(l3[1].data, want)
    assert l3[1].header["CRVAL1"] == 17.0 and l3[1].header["CROTA"] == 1.75
