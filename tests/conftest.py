import os
import sys
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def toy_pair(tmp_path_factory):
    """96^2 small vs 160^2 large synthetic pair, true correction (24, 6) arcsec."""
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    d = tmp_path_factory.mktemp("toy")
    p_large, p_small, spec = make_pair(str(d), small_spec(96, 160, true_crval=(-12.0, 8.0)), tag="toy")
    return p_large, p_small, spec


@pytest.fixture(scope="session")
def toy_rect_pair(tmp_path_factory):
    """Ragged sizes (not multiples of the 64x32 tile): 150x70 small image written by hand."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    d = tmp_path_factory.mktemp("rect")
    p_large, p_small, spec = make_pair(str(d), small_spec(160, 200, true_crval=(-12.0, 8.0)), tag="rect")
    hd = fits_lite.open(p_small)[0]
    data = np.ascontiguousarray(hd.data[10:80, 5:155])
    h = hd.header.copy()
    h["NAXIS1"], h["NAXIS2"] = 150, 70
    h["CRPIX1"] = h["CRPIX1"] - 5
    h["CRPIX2"] = h["CRPIX2"] - 10
    fits_lite.writeto(p_small, [fits_lite.PrimaryHDU(data, h)], overwrite=True)
    return p_large, p_small, spec


@pytest.fixture(scope="session")
def config1_pair(tmp_path_factory):
    """BASELINE configs[0] pair (2048^2 small vs 3072^2 large, the scene bench.py times), written once per session."""
    from euispice_coreg_b200._synth.scene import make_config1
    p_large, p_small, _ = make_config1(str(tmp_path_factory.mktemp("config1")))
    return p_large, p_small


def load_pair(p_large, p_small):
    from euispice_coreg_b200._compat import fits_lite
    L, S = fits_lite.open(p_large)[0], fits_lite.open(p_small)[0]
    return L.data, dict(L.header.items()), S.data, dict(S.header.items())


@pytest.fixture(autouse=True)
def _quiet():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        yield
