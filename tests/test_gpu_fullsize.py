"""Full-size parity (`-m gpu`): the CUDA path through the public API against oracle cubes computed ONCE on CPU and
committed under tests/golden/ by `tests/golden/make_fullsize_golden.py` (the oracle needs 1.5 - 4 s per lag per core):

* BASELINE.json configs[0]: every one of the 3600 helioprojective lags, both arithmetic modes;
* configs[1]: ~290 of the 14 400 Carrington-grid lags (a 15 x 15 sub-lattice, 64 random lags, the peak, two corners);
* configs[3]: 290 of the 1 024 000 lags of the 5-D grid (arg-max neighbourhood + random), both arithmetic modes.

Bar (north_star): |r_gpu - r_oracle| <= 1e-6 for every stored lag, identical arg-max. One documented exception: the
helioprojective lag (0, 0, 0, 0, 0), where the candidate header IS the grid's header, the map is the identity to
~1e-11 pixel, and which border rows pass map_coordinates' closed bound [0, n-1] is rounding noise of the pixel -> world
-> pixel chain (DESIGN.md section 4, README): there only border pixels may differ.
"""
import hashlib
import os

import numpy as np
import pytest

from conftest import load_pair

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
R_TOL = 1e-6
OBSERVED = {"fp64": 1e-10, "mixed": 2e-8}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from euispice_coreg_b200 import _ext
    _ext.load()
    return torch


@pytest.fixture(scope="module")
def config1(config1_pair):
    pl, ps = config1_pair
    dl, _, ds, _ = load_pair(pl, ps)
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(dl).tobytes())
    h.update(np.ascontiguousarray(ds).tobytes())
    return pl, ps, h.hexdigest()


def _golden(name, sha):
    z = np.load(os.path.join(GOLD, name))
    assert str(z["payload_sha256"]) == sha, "the synthetic config-1 scene differs from the one the golden was made from"
    return z


@pytest.mark.parametrize("arithmetic", ["fp64", "mixed"])
def test_config1_every_lag_vs_oracle_cube(torch_cuda, config1, arithmetic):
    import bench
    from euispice_coreg_b200.hdrshift import Alignment
    pl, ps, sha = config1
    z = _golden("config1_full_cube.npz", sha)
    assert z["index"].size == 3600 and np.array_equal(z["index"], np.arange(3600))
    a = Alignment(pl, ps, parallelism=True, arithmetic=arithmetic, **bench.LAGS)
    cube = a.align_using_helioprojective(return_type="corr")
    assert cube.shape == (60, 60, 1, 1, 1, 1) == tuple(z["shape"])
    assert (a.engine.small32 is not None) == (arithmetic == "mixed")
    assert a.engine.flagged_lags == 0          # the guard of the mixed kernel has nothing to object to here
    gpu, ref = cube.ravel(), z["r"]
    err = np.abs(gpu - ref)
    zero = 30 * 60 + 30                       # lag (0, 0): the documented knife edge
    assert bench.LAGS["lag_crval1"][30] == 0.0
    others = np.delete(err, zero)
    assert others.max() <= R_TOL, (others.max(), int(np.argmax(err)))
    assert others.max() < OBSERVED[arithmetic], others.max()
    assert err[zero] < 1e-3 and 2048 * 2048 - a.nvalid.ravel()[zero] <= 2 * (2048 + 2048)
    assert int(np.nanargmax(gpu)) == int(np.nanargmax(ref)) == 54 * 60 + 36      # (24, 6) arcsec


def test_config2_carrington_sample_vs_oracle(torch_cuda, config1):
    from euispice_coreg_b200.hdrshift import Alignment
    pl, ps, sha = config1
    z = _golden("config2_sample.npz", sha)
    lags = {k: z[k] for k in ("lag_crval1", "lag_crval2", "lag_cdelt1", "lag_cdelt2", "lag_crota")}
    a = Alignment(pl, ps, parallelism=True, **lags)
    cube = a.align_using_carrington(method="correlation", return_type="corr", lonlims=(200.0, 300.0),
                                    latlims=(-20.0, 20.0), shape=(2048, 2048))
    assert cube.shape == tuple(z["shape"]) == (120, 120, 1, 1, 1, 1)
    idx, ref = z["index"], z["r"]
    assert idx.size >= 256
    gpu = cube.ravel()[idx]
    assert np.array_equal(np.isnan(gpu), np.isnan(ref))
    err = np.nanmax(np.abs(gpu - ref))
    assert err <= R_TOL and err < 1e-9, err
    # the oracle's best sampled lag is the cube's arg-max: (24, 6) arcsec
    assert int(np.nanargmax(cube)) == int(idx[np.nanargmax(ref)]) == 84 * 120 + 66


@pytest.mark.parametrize("arithmetic", ["fp64", "mixed"])
def test_config4_5d_grid_sample_vs_oracle(torch_cuda, config1, arithmetic):
    """configs[3] at BASELINE size: 20 x 20 x 16 x 16 x 10 = 1 024 000 lags (intended CDELT semantics). The all-FP64
    run goes through the public API over the whole grid (254 launches); the mixed run evaluates the stored sample
    through the same engine (the full grid once is enough GPU time for a test)."""
    from euispice_coreg_b200.hdrshift import Alignment, engine
    pl, ps, sha = config1
    z = _golden("config4_sample.npz", sha)
    lags = {k: z[k] for k in ("lag_crval1", "lag_crval2", "lag_cdelt1", "lag_cdelt2", "lag_crota")}
    idx, ref = z["index"], z["r"]
    assert idx.size >= 256 and tuple(z["shape"]) == (20, 20, 16, 16, 10, 1)
    if arithmetic == "fp64":
        a = Alignment(pl, ps, parallelism=True, cdelt_semantics="intended", arithmetic="fp64", **lags)
        cube = a.align_using_helioprojective(return_type="corr")
        assert cube.shape == (20, 20, 16, 16, 10, 1)
        gpu = cube.ravel()[idx]
        assert np.unravel_index(int(np.nanargmax(cube)), cube.shape)[:5] == (10, 10, 8, 8, 5)   # (24", 6", 0, 0, 0)
    else:
        small = {k: (v[:2] if k.startswith("lag_crval") else v[:1]) for k, v in lags.items()}
        a = Alignment(pl, ps, parallelism=True, cdelt_semantics="intended", arithmetic="mixed", **small)
        a.align_using_helioprojective(return_type="corr")          # prepares the engine (images, cut, pivots)
        d = engine.flat_lag_grid(*(lags[k] for k in ("lag_crval1", "lag_crval2", "lag_cdelt1", "lag_cdelt2",
                                                     "lag_crota")))
        table, dead = a.engine.hpc_lag_table(a.hdr_small, a, *(v[idx] for v in d), "intended")
        assert not dead.any() and a.engine.small32 is not None
        gpu = a.engine.search(table)
        assert a.engine.flagged_lags == 0
    assert np.array_equal(np.isnan(gpu), np.isnan(ref))
    err = np.nanmax(np.abs(gpu - ref))
    assert err <= R_TOL and err < OBSERVED[arithmetic], err
    assert int(idx[np.nanargmax(gpu)]) == int(idx[np.nanargmax(ref)])
