"""`SequenceAlignment.align_using_carrington` rejects what it cannot search on the host, before any device work: these
run without a GPU, and no engine is ever created."""
import numpy as np
import pytest

LAGS = dict(lag_crval1=np.arange(20, 29, 2.0), lag_crval2=np.arange(2, 11, 2.0), lag_cdelt1=[0], lag_cdelt2=[0],
            lag_crota=[0.0])
GRID = dict(lonlims=(244.0, 256.0), latlims=(-8.0, 4.0), shape=(150, 130))


class _NoEngine:
    def __init__(self, *a, **k):
        raise AssertionError("a search engine was created")


@pytest.fixture
def no_engine(monkeypatch):
    from euispice_coreg_b200.hdrshift import engine
    monkeypatch.setattr(engine, "LagSearchEngine", _NoEngine)


def _seq(pair, **kw):
    from euispice_coreg_b200.hdrshift import SequenceAlignment
    return SequenceAlignment(pair[0], [pair[1], pair[1]], **dict(LAGS, **kw))


def test_size_deg_grid_is_rejected(no_engine, toy_pair):
    with pytest.raises(ValueError, match="size_deg_carrington"):
        _seq(toy_pair).align_using_carrington(size_deg_carrington=(4.0, 4.0))
    with pytest.raises(ValueError, match="no in between"):
        _seq(toy_pair).align_using_carrington(lonlims=GRID["lonlims"], latlims=GRID["latlims"])


@pytest.mark.parametrize("method", ["fa", "sunpy"])
def test_several_solar_radii_are_rejected(no_engine, toy_pair, method):
    with pytest.raises(ValueError, match="lag_solar_r"):
        _seq(toy_pair, lag_solar_r=[1.0, 1.004]).align_using_carrington(method_carrington_reprojection=method, **GRID)


def test_unknown_reprojection_method_is_rejected(no_engine, toy_pair):
    with pytest.raises(ValueError, match="method_carrington_reprojection"):
        _seq(toy_pair).align_using_carrington(method_carrington_reprojection="exact", **GRID)


def test_reference_date_is_required_without_date_avg(no_engine, toy_pair, tmp_path):
    from euispice_coreg_b200._compat import fits_lite
    hd = fits_lite.open(toy_pair[0])[0]
    h = hd.header.copy()
    del h["DATE-AVG"]
    p_large = str(tmp_path / "large_no_date_avg.fits")
    fits_lite.writeto(p_large, [fits_lite.PrimaryHDU(np.array(hd.data), h)], overwrite=True)
    with pytest.raises(ValueError, match="DATE-AVG"):
        _seq((p_large, toy_pair[1])).align_using_carrington(**GRID)
    # with an explicit date the checks pass and the search would start: the first device step is the engine
    with pytest.raises(AssertionError, match="engine was created"):
        _seq((p_large, toy_pair[1])).align_using_carrington(reference_date="2022-03-17T09:50:45.000", **GRID)


def test_cdelt_lags_need_the_reference_semantics(no_engine, toy_pair):
    with pytest.raises(NotImplementedError, match="cdelt_semantics"):
        _seq(toy_pair, lag_cdelt1=[0.0, 0.1], cdelt_semantics="intended").align_using_carrington(**GRID)


def test_sunpy_needs_the_observer_keywords_of_the_reference(no_engine, toy_pair):
    with pytest.raises(ValueError, match="HGLN_OBS"):
        _seq(toy_pair).align_using_carrington(method_carrington_reprojection="sunpy")
