"""Per-block correlation cubes of the helioprojective search (`Alignment(..., local_block=...)`): argument checks, block
geometry, the oracle's block cubes, the all-gather of per-block values and the C entries' validation. No GPU needed."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAGS = dict(lag_crval1=np.arange(19, 30, 5.0), lag_crval2=np.arange(1, 12, 5.0), lag_cdelt1=[0.0], lag_cdelt2=[0.0, 0.5],
            lag_crota=[0.0])


@pytest.fixture(scope="module")
def rect_pair(tmp_path_factory):
    """150 x 70 small image (not a multiple of any tile side) cut from a 160^2 synthetic one."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    d = tmp_path_factory.mktemp("rect_blocks")
    p_large, p_small, spec = make_pair(str(d), small_spec(160, 200, true_crval=(-12.0, 8.0)), tag="rect")
    hd = fits_lite.open(p_small)[0]
    data = np.ascontiguousarray(hd.data[10:80, 5:155])
    h = hd.header.copy()
    h["NAXIS1"], h["NAXIS2"] = 150, 70
    h["CRPIX1"] = h["CRPIX1"] - 5
    h["CRPIX2"] = h["CRPIX2"] - 10
    fits_lite.writeto(p_small, [fits_lite.PrimaryHDU(data, h)], overwrite=True)
    return p_large, p_small


def block_cube(search, block, reuse_world=True):
    """Oracle of the per-block cubes, on top of the CPU restatement `oracle.hpc.HpcSearch`: the masked Pearson r
    (`oracle.pearson`) of each block's pixels of the one-time cut and of the per-lag resampled image.
    block = (rows, cols) or an int: blocks of the common grid from pixel (0, 0), the last block row and column taking
    whatever remains. Returns [nby, nbx, n_crval1, ..., n_crota, 1] (or [nby, nbx, n_lags] with several solar radii);
    lags that kill the reference's worker read 0.0 in every block, as in `HpcSearch.cube`."""
    from oracle.hpc import LagKillsWorker
    from oracle.pearson import masked_pearson
    rows, cols = (block, block) if np.isscalar(block) else block
    gny, gnx = search.data_large.shape
    ys = [(y, min(y + rows, gny)) for y in range(0, gny, rows)]
    xs = [(x, min(x + cols, gnx)) for x in range(0, gnx, cols)]
    l1, l2, l3, l4, l5 = search.flat_lags()
    out = np.zeros((len(ys), len(xs), l1.size), dtype=np.float64)
    for k in range(l1.size):
        try:
            interp = search.reprojected(l1[k], l2[k], l3[k], l4[k], l5[k], reuse_world)
        except LagKillsWorker:
            continue
        for i, (y0, y1) in enumerate(ys):
            for j, (x0, x1) in enumerate(xs):
                out[i, j, k] = masked_pearson(search.data_large[y0:y1, x0:x1], interp[y0:y1, x0:x1])
    if len(search.refs.lag_solar_r) == 1:
        return out.reshape((len(ys), len(xs)) + search.shape[:5] + (1,))
    return out


def _oracle(p_large, p_small, **lags):
    from euispice_coreg_b200._compat import fits_lite
    from oracle.hpc import HpcSearch
    L, S = fits_lite.open(p_large)[0], fits_lite.open(p_small)[0]
    return HpcSearch(L.data, dict(L.header.items()), S.data, dict(S.header.items()), **lags)


def test_local_block_argument_checks():
    from euispice_coreg_b200.hdrshift import Alignment, AlignmentSpice
    from euispice_coreg_b200.hdrshift.engine import local_block_shape
    assert local_block_shape(256) == (256, 256) and local_block_shape((128, 64)) == (128, 64)
    assert local_block_shape(np.int64(64)) == (64, 64)
    for bad in (0, -64, 100, 32, (64, 96), (0, 64), (64, -64), (64.0, 64), (64,), (64, 64, 64), "64", True):
        with pytest.raises(ValueError):
            Alignment("a.fits", "b.fits", local_block=bad, **LAGS)
        with pytest.raises(ValueError):
            AlignmentSpice("a.fits", "b.fits", local_block=bad, **LAGS)
    assert Alignment("a.fits", "b.fits", **LAGS).local_block is None
    assert AlignmentSpice("a.fits", "b.fits", local_block=(128, 64), **LAGS).local_block == (128, 64)
    # combinations the per-block cubes do not support
    with pytest.raises(ValueError, match="coarse_to_fine|dense"):
        Alignment("a.fits", "b.fits", local_block=64, lag_search="coarse_to_fine", **LAGS)
    with pytest.raises(ValueError, match="FP64"):
        Alignment("a.fits", "b.fits", local_block=64, arithmetic="mixed", **LAGS)
    a = Alignment("a.fits", "b.fits", local_block=64, **LAGS)
    with pytest.raises(ValueError, match="align_using_carrington"):
        a.align_using_carrington(lonlims=[0, 1], latlims=[0, 1], shape=[64, 64], reference_date="2022-03-17T00:00:00")
    with pytest.raises(ValueError, match="align_using_initial_carrington"):
        a.align_using_initial_carrington()


def test_local_block_refuses_mixed_arithmetic_from_the_environment(rect_pair, monkeypatch):
    """COREG_ARITHMETIC=mixed is refused before any device work (the search stops after reading the pair)."""
    from euispice_coreg_b200.hdrshift import Alignment
    monkeypatch.setenv("COREG_ARITHMETIC", "mixed")
    a = Alignment(*rect_pair, local_block=64, **LAGS)
    with pytest.raises(ValueError, match="COREG_ARITHMETIC"):
        a.align_using_helioprojective()
    assert a.engine is None and a.local is None


def test_block_bounds_of_a_ragged_grid():
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200.hdrshift.engine import region_bounds
    b = region_bounds(70, 150, (64, 64))
    assert b.shape == (2, 3, 4) and b.dtype == np.int64
    rows, cols = [(0, 64), (64, 70)], [(0, 64), (64, 128), (128, 150)]
    for i, (y0, y1) in enumerate(rows):
        for j, (x0, x1) in enumerate(cols):
            assert tuple(b[i, j]) == (y0, y1, x0, x1)
    assert tuple(region_bounds(70, 150, (128, 64))[0, 2]) == (0, 70, 128, 150)
    assert region_bounds(70, 150, (4096, 4096)).tolist() == [[[0, 70, 0, 150]]]
    assert region_bounds(2048, 2048, (256, 256)).shape == (8, 8, 4)
    assert region_bounds(2048, 2048, (128, 128)).shape == (16, 16, 4)
    assert _ext.region_grid(832, 192, 896, 64) == (1, 3)     # SPICE raster: three bands of 64 slit positions
    # the blocks tile the grid exactly once
    cover = np.zeros((70, 150), dtype=int)
    for y0, y1, x0, x1 in b.reshape(-1, 4):
        cover[y0:y1, x0:x1] += 1
    assert (cover == 1).all()


def test_oracle_block_cube_of_one_block_is_the_global_cube(rect_pair):
    s = _oracle(*rect_pair, **LAGS)
    glob = s.cube()
    one = block_cube(s, 4096)
    assert one.shape == (1, 1) + glob.shape
    assert np.array_equal(one[0, 0], glob, equal_nan=True)
    blocks = block_cube(s, (64, 64))
    assert blocks.shape == (2, 3) + glob.shape
    assert (blocks[..., 1, 0, :] == 0.0).all()           # CDELT2 lags kill the reference's worker: 0.0 in every block
    assert np.isfinite(blocks[..., 0, 0, :]).all()
    assert not np.allclose(blocks[0, 0], blocks[1, 2])    # the blocks see different parts of the field


_GLOO = r"""
import sys
sys.path.insert(0, {root!r})
import torch, torch.distributed as dist
from euispice_coreg_b200.hdrshift import engine
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
for n in (25, 7, 2, 1):
    for n_blocks in (1, 3, 6):
        chunk, bounds = engine.shard_bounds(n, world)
        lo, hi = bounds[rank]
        # what LagSearchEngine.search gathers: per lag, the block values (r and nvalid) next to each other
        local = torch.full((chunk, 2, n_blocks), float("nan"), dtype=torch.float64)
        lags = torch.arange(lo, hi, dtype=torch.float64)[:, None]
        blocks = torch.arange(n_blocks, dtype=torch.float64)[None, :]
        local[:hi - lo, 0] = lags * 0.5 + blocks * 100.0
        local[:hi - lo, 1] = lags * 3.0 + blocks
        full = engine.gather_slices(local, n, chunk)
        lags = torch.arange(n, dtype=torch.float64)[:, None]
        assert full.shape == (n, 2, n_blocks), (n, full.shape)
        assert torch.equal(full[:, 0], lags * 0.5 + blocks * 100.0), (n, n_blocks, full)
        assert torch.equal(full[:, 1], lags * 3.0 + blocks), (n, n_blocks, full)
        # a short local slice is padded to the chunk like a 1-D one
        short = engine.gather_slices(local[:max(0, hi - lo)], n, chunk)
        assert torch.equal(short, full), (n, n_blocks)
dist.barrier()
if rank == 0:
    print("GLOO_BLOCKS_OK")
"""


@pytest.mark.parametrize("world", [2, 3])
def test_block_cube_gather_gloo(tmp_path, world):
    """Per-block values of every lag all-gathered over 2 and 3 ranks, also with more ranks than lags."""
    script = tmp_path / "gloo_blocks.py"
    script.write_text(_GLOO.format(root=ROOT))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={world}",
                          str(script)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "GLOO_BLOCKS_OK" in out.stdout


def test_c_entries_refuse_bad_regions_before_any_cuda_call():
    from euispice_coreg_b200 import _ext
    lib = _ext.load()
    null, fake = None, ctypes.c_void_p(0x1000)          # never dereferenced: validation fails first
    EINVAL = -1
    assert ctypes.sizeof(_ext.CoregRegions) == 32

    def msg():
        return lib.coreg_last_error().decode()

    good_wcs = ctypes.byref(_ext.CoregTanWcs(1, 1, 1.0, 1.0, 1, 0, 0, 1, 0, 0, 180))
    big = 1 << 30
    entries = {
        "coreg_hpc_lag_corr_wcs_regions": lambda rg, f, gnx=256, gny=128: (fake, fake, 8, 8, gnx, gny, good_wcs, fake,
                                                                           4, 2, fake, fake, big, fake, null, rg, f,
                                                                           null),
        "coreg_hpc_lag_corr_regions": lambda rg, f, gnx=256, gny=128: (fake, fake, _ext.F64, 8, 8, gnx, gny, fake, fake,
                                                                       4, 2, fake, fake, big, fake, null, rg, f, null),
    }

    def regions(bh=64, bw=64, ld=4, corr=0x2000, nvalid=0x3000):
        return _ext.CoregRegions(bh, bw, ld, corr, nvalid)

    bad = [(regions(bh=0), "multiples of 64"), (regions(bw=-64), "multiples of 64"), (regions(bh=100), "multiples of 64"),
           (regions(bw=32), "multiples of 64"), (regions(ld=3), "ld < n_lags"), (regions(corr=None), "null"),
           (regions(nvalid=None), "null")]
    for name, args in entries.items():
        fn = getattr(lib, name)
        for rg, what in bad:
            rc = fn(*args(ctypes.byref(rg), 0))
            assert rc == EINVAL and what in msg() and msg().startswith(name), (name, what, msg())
        rc = fn(*args(None, 0))
        assert rc == EINVAL and "null" in msg(), (name, msg())
        rc = fn(*args(ctypes.byref(regions()), _ext.FLAG_MIXED))
        assert rc == EINVAL and "mixed" in msg(), (name, msg())
        rc = fn(*args(ctypes.byref(regions(ld=1 << 20)), 1 << 9))         # the whole-grid call's own checks follow
        assert rc == EINVAL and "reserved flag bits" in msg(), (name, msg())
        rc = fn(*args(ctypes.byref(regions()), 0, 64 * 300, 64 * 300))
        assert rc == EINVAL and "65535 blocks" in msg(), (name, msg())
