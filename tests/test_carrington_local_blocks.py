"""Per-block correlation cubes of the Carrington searches (`align_using_carrington(..., local_block=...)`): argument
checks, the block-cube oracle of both reprojection methods, the C entries' validation and the all-gather of per-frame
block values. No GPU needed."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import load_pair

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAGS = dict(lag_crval1=[22.0, 24.0], lag_crval2=[6.0, 8.0], lag_cdelt1=[0.0], lag_cdelt2=[0.0, 0.5],
            lag_crota=[0.0, 0.5])
GRID = dict(lonlims=(248.0, 252.0), latlims=(-4.0, 0.0), shape=(120, 100))
BAD_BLOCKS = (0, -64, 100, 32, (64, 96), (0, 64), (64.0, 64), (64,), (64, 64, 64), "64", True)


def carrington_block_cube(search, block, counts=False):
    """Oracle of the per-block cubes of the Carrington searches, on the unchanged CPU restatements: the masked Pearson r
    (`oracle.pearson`) of each block's pixels of the one-time projection of the large image and of the per-lag
    reprojected small image. `search`: `oracle.carrington.CarringtonSearch` ("fa": its Carrington grid) or
    `oracle.surface_reproject.SurfaceSearch` ("sunpy": the small image's grid; the per-lag image is the body of its
    `step`). block = (rows, cols) or an int: blocks from pixel (0, 0), the last block row and column taking whatever
    remains. Returns [nby, nbx, n_crval1, n_crval2, n_cdelt1, n_cdelt2, n_crota, 1]; lags that kill the reference's
    worker read 0.0 in every block, as in `search.cube()`. counts=True: also the valid pixel pairs per block and lag
    [nby, nbx, n_crval1, ..., n_crota] (0 for those lags)."""
    from oracle import surface_reproject as sr
    from oracle.hpc import LagKillsWorker, shift_header
    from oracle.pearson import masked_pearson
    rows, cols = (block, block) if np.isscalar(block) else block
    if isinstance(search, sr.SurfaceSearch):
        ref = search.ref

        def sample(*lag):
            hdr = dict(search.hdr_small)
            shift_header(hdr, search.refs, *lag, cdelt_mode=search.cdelt_mode)
            return sr.reproject_to(search.data_small, hdr, search.hdr_small, search.rsun)
    else:
        ref, sample = search.data_large, search.reprojected
    gny, gnx = ref.shape
    ys = [(y, min(y + rows, gny)) for y in range(0, gny, rows)]
    xs = [(x, min(x + cols, gnx)) for x in range(0, gnx, cols)]
    r = search.refs
    lag_axes = (r.lag_crval1, r.lag_crval2, r.lag_cdelt1, r.lag_cdelt2, r.lag_crota)
    shape5 = tuple(len(v) for v in lag_axes)
    out = np.zeros((len(ys), len(xs)) + shape5 + (1,), dtype=np.float64)
    nvalid = np.zeros((len(ys), len(xs)) + shape5, dtype=np.int64)
    for idx in np.ndindex(*shape5):
        try:
            img = sample(*(v[i] for v, i in zip(lag_axes, idx)))
        except LagKillsWorker:
            continue
        for i, (y0, y1) in enumerate(ys):
            for j, (x0, x1) in enumerate(xs):
                a, b = ref[y0:y1, x0:x1], img[y0:y1, x0:x1]
                out[(i, j) + idx + (0,)] = masked_pearson(a, b)
                nvalid[(i, j) + idx] = np.count_nonzero(np.isfinite(a) & np.isfinite(b))
    return (out, nvalid) if counts else out


def with_observers(pair, out_dir, small=(10.0, -3.0, None, None), large=(10.3, -2.9, 5.5e10, None), tag="obs"):
    """Copies of a pair whose headers carry the observer keywords of the "sunpy" path: (HGLN_OBS, HGLT_OBS, DSUN_OBS or
    None, DATE-AVG or None) per image."""
    from euispice_coreg_b200._compat import fits_lite
    out = []
    for path, (lon, lat, dsun, date), name in ((pair[0], large, "large"), (pair[1], small, "small")):
        hd = fits_lite.open(path)[0]
        h = hd.header.copy()
        h["HGLN_OBS"], h["HGLT_OBS"] = float(lon), float(lat)
        if dsun is not None:
            h["DSUN_OBS"] = float(dsun)
        if date is not None:
            h["DATE-AVG"] = date
        p = os.path.join(str(out_dir), f"{tag}_{name}.fits")
        fits_lite.writeto(p, [fits_lite.PrimaryHDU(np.array(hd.data), h)], overwrite=True)
        out.append(p)
    return out[0], out[1]


# ------------------------------------------------------------------------------------------------ arguments
@pytest.mark.parametrize("method", ["fa", "sunpy"])
def test_call_level_block_is_checked_before_any_file_is_opened(method):
    """The paths do not exist: a check that ran after opening them would raise FileNotFoundError instead."""
    from euispice_coreg_b200.hdrshift import Alignment, SequenceAlignment
    for bad in BAD_BLOCKS:
        a = Alignment("missing_large.fits", "missing_small.fits", **LAGS)
        with pytest.raises(ValueError, match="local_block"):
            a.align_using_carrington(method_carrington_reprojection=method, local_block=bad, **GRID)
        assert a.local_block is None and a.hdr_small is None
        seq = SequenceAlignment("missing_large.fits", ["missing_small.fits"], **LAGS)
        with pytest.raises(ValueError, match="local_block"):
            seq.align_using_carrington(method_carrington_reprojection=method, local_block=bad, **GRID)
    # a good block gets as far as the files
    with pytest.raises(FileNotFoundError):
        Alignment("missing_large.fits", "missing_small.fits", **LAGS).align_using_carrington(
            method_carrington_reprojection=method, local_block=(128, 64), **GRID)


def test_constructor_level_refusal_fires_first():
    from euispice_coreg_b200.hdrshift import Alignment
    a = Alignment("missing_large.fits", "missing_small.fits", local_block=64, **LAGS)
    for blk in (None, 64, 100):
        with pytest.raises(ValueError, match="local_block is implemented for align_using_helioprojective only, not "
                                             "align_using_carrington"):
            a.align_using_carrington(local_block=blk, **GRID)
    assert a.local_block == (64, 64)


def test_sequence_refuses_corr_return_type_with_blocks():
    from euispice_coreg_b200.hdrshift import SequenceAlignment
    seq = SequenceAlignment("missing_large.fits", ["missing_small.fits"], **LAGS)
    for method in ("fa", "sunpy"):
        with pytest.raises(ValueError, match="return_type"):
            seq.align_using_carrington(method_carrington_reprojection=method, return_type="corr", local_block=64,
                                       **GRID)


def test_carrington_block_does_not_reach_the_helioprojective_search(toy_pair, monkeypatch):
    """The call-level blocks are not stored in `local_block`: a later helioprojective search of the same object (here
    stopped at its first device step) sees none."""
    from euispice_coreg_b200.hdrshift import Alignment, engine

    class Stop(Exception):
        pass

    class NoEngine:
        def __init__(self, *a, **k):
            raise Stop

    a = Alignment(toy_pair[0], toy_pair[1], **LAGS)
    monkeypatch.setattr(engine, "LagSearchEngine", NoEngine)
    with pytest.raises(Stop):
        a.align_using_carrington(local_block=64, **GRID)
    assert a.local_block is None
    with pytest.raises(Stop):
        a.align_using_helioprojective()
    assert a.local_block is None and a.local is None


# ------------------------------------------------------------------------------------------------ oracle
def test_fa_oracle_block_cube_of_one_block_is_the_global_cube(toy_pair):
    from oracle.carrington import CarringtonSearch
    s = CarringtonSearch(*load_pair(*toy_pair[:2]), **LAGS, **GRID)
    glob = s.cube()
    assert s.data_large.shape == (100, 120)           # rows: latitude samples, columns: longitude samples
    one = carrington_block_cube(s, 4096)
    assert one.shape == (1, 1) + glob.shape
    assert np.array_equal(one[0, 0].view(np.uint64), glob.view(np.uint64))
    blocks = carrington_block_cube(s, (64, 64))
    assert blocks.shape == (2, 2) + glob.shape
    assert (blocks[:, :, :, :, :, 1] == 0.0).all()     # CDELT2 lags kill the reference's worker: 0.0 in every block
    assert not np.allclose(blocks[0, 0], blocks[1, 1], equal_nan=True)


def test_sunpy_oracle_block_cube_of_one_block_is_the_global_cube(toy_pair, tmp_path):
    from oracle.surface_reproject import SurfaceSearch
    pl, ps = with_observers(toy_pair, tmp_path)
    s = SurfaceSearch(*load_pair(pl, ps), **LAGS)
    glob = s.cube()
    one = carrington_block_cube(s, 4096)
    assert np.array_equal(one[0, 0].view(np.uint64), glob.view(np.uint64))
    blocks = carrington_block_cube(s, 64)
    assert blocks.shape == (2, 2) + glob.shape           # the 96 x 96 small grid
    assert (blocks[:, :, :, :, :, 1] == 0.0).all()
    assert np.isfinite(blocks[:, :, :, :, :, 0]).all()


# ------------------------------------------------------------------------------------------------ C entries
def test_carrington_c_entries_refuse_bad_regions_before_any_cuda_call():
    from euispice_coreg_b200 import _ext
    lib = _ext.load()
    null, fake = None, ctypes.c_void_p(0x1000)          # never dereferenced: validation fails first
    EINVAL = -1
    big = 1 << 30

    def msg():
        return lib.coreg_last_error().decode()

    entries = {
        "coreg_offset_lag_corr_regions": lambda rg, f, gnx=256, gny=128: (fake, fake, _ext.F32, 8, 8, gnx, gny, fake,
                                                                          fake, fake, 4, 2, fake, fake, big, fake,
                                                                          null, rg, f, null),
        "coreg_hpc_lag_corr_edge_regions": lambda rg, f, gnx=256, gny=128: (fake, fake, 8, 8, gnx, gny, fake, fake, 4,
                                                                            fake, fake, big, fake, null, rg, f, null),
    }

    def regions(bh=64, bw=64, ld=4, corr=0x2000, nvalid=0x3000):
        return _ext.CoregRegions(bh, bw, ld, corr, nvalid)

    bad = [(regions(bh=0), "multiples of 64"), (regions(bw=-64), "multiples of 64"), (regions(bh=100), "multiples of 64"),
           (regions(bw=32), "multiples of 64"), (regions(bh=96), "multiples of 64"), (regions(ld=3), "ld < n_lags"),
           (regions(corr=None), "null"), (regions(nvalid=None), "null")]
    for name, args in entries.items():
        fn = getattr(lib, name)
        for rg, what in bad:
            rc = fn(*args(ctypes.byref(rg), 0))
            assert rc == EINVAL and what in msg() and msg().startswith(name), (name, what, msg())
        rc = fn(*args(None, 0))
        assert rc == EINVAL and "null" in msg(), (name, msg())
        rc = fn(*args(ctypes.byref(regions()), _ext.FLAG_MIXED))
        assert rc == EINVAL and "mixed" in msg(), (name, msg())
        rc = fn(*args(ctypes.byref(regions()), 0, 64 * 300, 64 * 300))
        assert rc == EINVAL and "65535 blocks" in msg(), (name, msg())
        rc = fn(*args(ctypes.byref(regions(ld=1 << 20)), 1 << 9))         # the whole-grid call's own checks follow
        assert rc == EINVAL and "reserved flag bits" in msg(), (name, msg())


# ------------------------------------------------------------------------------------------------ frame all-gather
_GLOO = r"""
import sys
sys.path.insert(0, {root!r})
import numpy as np
import torch.distributed as dist
from euispice_coreg_b200.hdrshift import sequence
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()


def frame_blocks(k, n_lags):
    # frames of different grids (the "sunpy" grid is each frame's own): 1 + k % 3 blocks
    nb = 1 + k % 3
    grid = (64 * nb + k, 70 + k)
    corr = np.arange(nb * n_lags, dtype=np.float64).reshape(nb, n_lags) * 0.25 + k
    corr[0, ::3] = np.nan
    nvalid = (np.arange(nb * n_lags, dtype=np.int64).reshape(nb, n_lags) + 1000 * k) * (1 << 40)
    return grid, corr, nvalid


for n_frames in (1, 2, 5):
    for n_lags in (1, 7):
        mine = {{k: frame_blocks(k, n_lags) for k in sequence.frames_of_rank(n_frames, rank, world)}}
        full = sequence.gather_frame_blocks(mine, n_frames, n_lags, "cpu")
        assert sorted(full) == list(range(n_frames)), (n_frames, sorted(full))
        for k in range(n_frames):
            grid, corr, nvalid = frame_blocks(k, n_lags)
            g, c, nv = full[k]
            assert g == grid and c.shape == corr.shape and nv.dtype == np.int64, (k, g, c.shape)
            assert np.array_equal(c, corr, equal_nan=True) and np.array_equal(nv, nvalid), (n_frames, n_lags, k)
dist.barrier()
if rank == 0:
    print("GLOO_FRAME_BLOCKS_OK")
"""


@pytest.mark.parametrize("world", [2, 3])
def test_frame_block_gather_gloo(tmp_path, world):
    """Per-frame block values all-gathered over 2 and 3 ranks, also with more ranks than frames."""
    script = tmp_path / "gloo_frame_blocks.py"
    script.write_text(_GLOO.format(root=ROOT))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={world}",
                          str(script)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "GLOO_FRAME_BLOCKS_OK" in out.stdout
