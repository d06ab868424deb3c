"""Carrington-frame frame sequences: every cube of `SequenceAlignment.align_using_carrington` is bit-identical to the
single-pair `Alignment` cube, for both reprojection methods; batched jitter correction writes byte-identical files."""
import os
import shutil

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# two CROTA values (two plane pairs per frame), a value threshold, and a grid much larger than the frames' FOV
LAGS = dict(lag_crval1=np.arange(18, 31, 2.0), lag_crval2=np.arange(0, 13, 2.0), lag_cdelt1=[0], lag_cdelt2=[0],
            lag_crota=[0.0, 0.5], small_fov_value_min=80.0)
GRID = dict(lonlims=(244.0, 256.0), latlims=(-8.0, 4.0), shape=(150, 130))
JITTERS = [(0.0, 0.0), (1.3, -0.8), (-2.1, 0.4)]
# "sunpy": the frames' observer, and the reference's: a second spacecraft 0.3 deg away, closer, half an hour later
OBS_SMALL = (10.0, -3.0, None, None)
OBS_LARGE = (10.3, -2.9, 5.5e10, "2022-03-17T10:20:45.000")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _with_observer(path, obs, out):
    from euispice_coreg_b200._compat import fits_lite
    lon, lat, dsun, date = obs
    hd = fits_lite.open(path)[0]
    h = hd.header.copy()
    h["HGLN_OBS"], h["HGLT_OBS"] = float(lon), float(lat)
    if dsun is not None:
        h["DSUN_OBS"] = float(dsun)
    if date is not None:
        h["DATE-AVG"] = date
    fits_lite.writeto(out, [fits_lite.PrimaryHDU(np.array(hd.data), h)], overwrite=True)
    return out


@pytest.fixture(scope="module")
def frames(tmp_path_factory):
    """{"fa" / "sunpy": (reference path, [frame paths])}: jittered renderings of one sky."""
    from euispice_coreg_b200._synth.scene import make_pair, master_scene, small_spec
    d = tmp_path_factory.mktemp("seqcar")
    sky = master_scene(small_spec(96, 160, true_crval=(-12.0, 8.0)))
    p_large, paths = None, []
    for i, jit in enumerate(JITTERS):
        spec = small_spec(96, 160, true_crval=(-12.0, 8.0), jitter=jit, noise_seed=400 + i,
                          date=f"2022-03-17T09:5{i}:45.000")
        pl, ps, _ = make_pair(str(d), spec, tag=f"c{i}", sky=sky, write_large=(i == 0))
        p_large = p_large or pl
        paths.append(ps)
    obs_large = _with_observer(p_large, OBS_LARGE, str(d / "obs_large.fits"))
    obs_paths = [_with_observer(p, OBS_SMALL, str(d / f"obs_small_{i}.fits")) for i, p in enumerate(paths)]
    return {"fa": (p_large, paths), "sunpy": (obs_large, obs_paths)}


_SINGLE = {}


def _single(p_large, p, method):
    """The single-pair result the sequence must reproduce (cached: it does not depend on the sequence)."""
    from euispice_coreg_b200.hdrshift import Alignment
    key = (p_large, p, method)
    if key not in _SINGLE:
        a = Alignment(p_large, p, parallelism=True, **LAGS)
        _SINGLE[key] = a.align_using_carrington(method="correlation", method_carrington_reprojection=method, **GRID)
    return _SINGLE[key]


@pytest.mark.parametrize("n_frames", [1, 2, 3])
@pytest.mark.parametrize("method", ["fa", "sunpy"])
def test_sequence_equals_per_pair_alignment(torch_cuda, frames, method, n_frames):
    from euispice_coreg_b200.hdrshift import SequenceAlignment
    p_large, paths = frames[method]
    seq = SequenceAlignment(p_large, paths[:n_frames], **LAGS)
    res = seq.align_using_carrington(method_carrington_reprojection=method, **GRID)
    assert len(res) == n_frames and seq.frames_per_s > 0
    for p, r in zip(paths, res):
        one = _single(p_large, p, method)
        assert r.corr.shape == one.corr.shape == (7, 7, 1, 1, 2, 1)
        assert np.array_equal(r.corr, one.corr, equal_nan=True)
        assert r.max_index == one.max_index and r.shift_arcsec == one.shift_arcsec
        assert r.image_to_align_path == p
    if n_frames == 3:
        # the jittered frames peak at different sub-lag shifts
        assert len({r.shift_arcsec[:2] for r in res}) == 3


@pytest.mark.parametrize("method", ["fa", "sunpy"])
def test_frame_result_does_not_depend_on_its_pipeline_slot(torch_cuda, frames, method):
    from euispice_coreg_b200.hdrshift import SequenceAlignment
    p_large, paths = frames[method]
    ab = SequenceAlignment(p_large, [paths[1], paths[2]], **LAGS).align_using_carrington(
        method_carrington_reprojection=method, return_type="corr", **GRID)
    ba = SequenceAlignment(p_large, [paths[2], paths[1]], **LAGS).align_using_carrington(
        method_carrington_reprojection=method, return_type="corr", **GRID)
    assert np.array_equal(ab[0], ba[1], equal_nan=True) and np.array_equal(ab[1], ba[0], equal_nan=True)
    assert not np.array_equal(ab[0], ab[1], equal_nan=True)


# ------------------------------------------------------------------------------------------------ jitter correction
JC_LAG = np.arange(-4.0, 4.1, 0.5)
JC_GRID = dict(lonlims=(249.3, 250.7), latlims=(-2.6, -1.4), shape=[120, 110])


@pytest.fixture(scope="module")
def jitter_frames(tmp_path_factory):
    """Five frames whose headers all claim the same pointing while the true pointing jitters."""
    from euispice_coreg_b200._synth.scene import make_pair, master_scene, small_spec
    d = str(tmp_path_factory.mktemp("jc"))
    true = (-12.0, 8.0)
    sky = master_scene(small_spec(96, 160, true_crval=true))
    paths = []
    for i, jit in enumerate([(0.0, 0.0), (1.3, -0.8), (-2.1, 0.4), (0.6, 2.2), (-0.9, -1.5)]):
        spec = small_spec(96, 160, true_crval=true, jitter=jit, true_shift=jit, noise_seed=500 + i,
                          date=f"2022-03-17T09:5{i}:45.000")
        paths.append(make_pair(d, spec, tag=f"j{i}", sky=sky, write_large=False)[1])
    return paths


def _chain_by_hand(paths, out, method):
    """What `jitter_correction_imagers(sublist_length=2, overlap=1)` does, one `Alignment` per frame."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.hdrshift import Alignment
    dates = [fits_lite.open(p)[0].header["DATE-AVG"] for p in paths]
    idx = list(range(len(paths)))
    shutil.copyfile(paths[0], os.path.join(out, os.path.basename(paths[0])))
    results = []
    for sub in (idx[n:n + 3] for n in range(0, len(idx), 2)):
        ref = os.path.join(out, os.path.basename(paths[sub[0]]))
        for i in sub[1:]:
            a = Alignment(ref, paths[i], lag_crval1=JC_LAG, lag_crval2=JC_LAG, lag_cdelt1=np.arange(0, 1, 1),
                          lag_cdelt2=np.arange(0, 1, 1), lag_crota=np.arange(0, 1, 1), parallelism=True)
            if method == "carrington":
                r = a.align_using_carrington(method="correlation", reference_date=dates[sub[0]], **JC_GRID)
            else:
                r = a.align_using_helioprojective(method="correlation")
            r.write_corrected_fits(window_list_to_apply_shift=[-1],
                                   path_to_l3_output=os.path.join(out, os.path.basename(paths[i])))
            results.append(r)
    return results


@pytest.mark.parametrize("method", ["carrington", "helioprojective"])
def test_batched_jitter_correction_writes_the_per_frame_files(torch_cuda, jitter_frames, tmp_path, method):
    from euispice_coreg_b200.jitter_correction.jitter_correction import jitter_correction_imagers
    out_batched, out_hand = tmp_path / "batched", tmp_path / "hand"
    out_batched.mkdir()
    out_hand.mkdir()
    kw = JC_GRID if method == "carrington" else {}
    res = jitter_correction_imagers(jitter_frames, str(out_batched), lag_crval1=JC_LAG, lag_crval2=JC_LAG,
                                    sublist_length=2, overlap=1, alignement_method=method, **kw)
    want = _chain_by_hand(jitter_frames, str(out_hand), method)
    assert len(res) == len(want) == 4
    for r, w in zip(res, want):
        assert r.max_index == w.max_index and r.shift_arcsec == w.shift_arcsec
        assert np.array_equal(r.corr, w.corr, equal_nan=True)
    names = sorted(os.listdir(out_hand))
    assert names == sorted(os.listdir(out_batched)) and len(names) == 5
    for name in names:
        assert (out_batched / name).read_bytes() == (out_hand / name).read_bytes(), name
