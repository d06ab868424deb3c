"""Per-block shift maps on the device (`LocalAlignmentResults.shift_arcsec`, `coreg_gauss2d_fit`): the batched fit
against scipy's `curve_fit` on seeded Gaussian peaks, the shift maps of real block cubes against `results(i, j)` for
every producer of `.local`, helioprojective frame sequences with blocks, and the kernel's register budget."""
import importlib
import os
import re
import subprocess
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
AR = importlib.import_module("euispice_coreg_b200.hdrshift.AlignmentResults")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", torch.cuda.current_device())


def random_peaks(n=400, seed=1):
    """Gaussian-plus-noise peaks on a 60 x 60 lag grid: centres 30 +- 3, sigmas 1-6, amplitude 0.5, offset 0.4, noise
    sigma 0-0.02, all from one seeded generator. About one in sixteen puts scipy's amplitude on its bound."""
    rng = np.random.default_rng(seed)
    X, Y = np.meshgrid(np.arange(60.0), np.arange(60.0), indexing="ij")
    cubes = np.empty((n, 60, 60))
    for k in range(n):
        cx, cy = rng.uniform(27, 33, 2)
        sx, sy = rng.uniform(1, 6, 2)
        noise = rng.uniform(0, 0.02)
        cubes[k] = 0.4 + 0.5 * np.exp(-((X - cx) ** 2 / (2 * sx ** 2) + (Y - cy) ** 2 / (2 * sy ** 2))) \
            + rng.normal(0, noise, X.shape)
    return cubes.reshape(n, 60, 60, 1, 1, 1, 1)


def _device_fit(prob, rows, dev):
    import torch
    from euispice_coreg_b200 import _ext
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a[rows])).to(dev)  # noqa: E731
    out = _ext.gauss2d_fit(up(prob.points), up(prob.npts), up(prob.p0), up(prob.bounds))
    return [t.cpu().numpy() for t in out]


def test_random_peaks_match_scipy(cuda):
    from scipy.optimize import curve_fit
    cubes = random_peaks()
    mi = np.array([np.unravel_index(np.argmax(c), c.shape) for c in cubes])
    prob = AR.gaussian_fit_problems(cubes, mi)
    assert (prob.decision == AR.FIT).all()
    rows = np.arange(len(cubes))
    popt, cost, iters, status = _device_fit(prob, rows, cuda)
    assert (status == AR.FIT).all(), np.flatnonzero(status)
    at_bound = 0
    for k in rows:
        npts = prob.npts[k]
        x, y, z = prob.points[k, :npts].T
        ps, _ = curve_fit(AR.twoD_Gaussian, (x, y), z, p0=prob.p0[k], bounds=(prob.bounds[k, :6], prob.bounds[k, 6:]))
        c_scipy = float(((AR.twoD_Gaussian((x, y), *ps) - z) ** 2).sum())
        c_dev = float(((AR.twoD_Gaussian((x, y), *popt[k]) - z) ** 2).sum())
        assert abs(popt[k, 1] - ps[1]) <= 1e-3 and abs(popt[k, 2] - ps[2]) <= 1e-3, (k, popt[k], ps)
        assert cost[k] <= c_scipy * (1 + 1e-9) and c_dev <= c_scipy * (1 + 1e-9), (k, cost[k], c_scipy)
        assert np.all(popt[k] >= prob.bounds[k, :6]) and np.all(popt[k] <= prob.bounds[k, 6:])
        assert popt[k, 3] > 0 and popt[k, 4] > 0
        at_bound += ps[0] > 10 - 1e-3
    assert at_bound > 0          # the set exercises the active set
    assert iters.max() < 200
    # a problem's bits do not depend on the batch it is in
    sub = rows[::7][::-1]
    popt2, cost2, iters2, status2 = _device_fit(prob, sub, cuda)
    assert np.array_equal(popt2.view(np.uint64), popt[sub].view(np.uint64))
    assert np.array_equal(cost2.view(np.uint64), cost[sub].view(np.uint64)) and np.array_equal(iters2, iters[sub])


# ------------------------------------------------------------------------------------------------ real block cubes
LAGS = dict(lag_crval1=np.arange(16, 33, 2.0), lag_crval2=np.arange(-2, 15, 2.0), lag_cdelt1=[0], lag_cdelt2=[0],
            lag_crota=[0.0, 0.5])
GRID = dict(lonlims=(249.2, 250.8), latlims=(-2.9, -1.3), shape=(256, 256))   # inside the small FOV


@pytest.fixture(scope="module")
def scene(cuda, tmp_path_factory):
    """A 256^2 small image against a 400^2 reference, and three jittered frames of one sky."""
    from euispice_coreg_b200._synth.scene import make_pair, master_scene, small_spec
    d = str(tmp_path_factory.mktemp("shift_maps"))
    p_large, p_small, _ = make_pair(d, small_spec(256, 400, true_crval=(-12.0, 8.0)), tag="pair")
    sky = master_scene(small_spec(256, 400, true_crval=(-12.0, 8.0)))
    frames, ref = [], None
    for i, jit in enumerate([(0.0, 0.0), (1.3, -0.8), (-2.1, 0.4)]):
        spec = small_spec(256, 400, true_crval=(-12.0, 8.0), jitter=jit, noise_seed=500 + i,
                          date=f"2022-03-17T09:5{i}:45.000")
        pl, ps, _ = make_pair(d, spec, tag=f"f{i}", sky=sky, write_large=(i == 0))
        ref = ref or pl
        frames.append(ps)
    return {"pair": (p_large, p_small), "frames": (ref, frames)}


def _check_against_results(loc):
    """Every block of `loc`: the shift map agrees with `results(i, j)`. Returns the status counts."""
    nby, nbx = loc.fit_status.shape
    steps = [np.diff(loc._results_kwargs[k]).mean() for k in ("lag_crval1", "lag_crval2")]
    counts = np.bincount(loc.fit_status.ravel(), minlength=4)
    assert counts[AR.NOT_CONVERGED] == 0
    for i in range(nby):
        for j in range(nbx):
            st = loc.fit_status[i, j]
            if st == AR.NO_MAXIMUM:
                assert (loc.max_index[i, j] == -1).all() and np.isnan(loc.shift_arcsec[i, j]).all()
                continue
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                r = loc.results(i, j)
            fell_back = any("Gaussian fitting failed" in str(m.message) or "Cannot compute shift" in str(m.message)
                            for m in w)
            host = np.array(r.shift_arcsec, dtype=np.float64)
            assert fell_back == (st == AR.ARGMAX_FALLBACK), (i, j)
            if fell_back:
                assert np.array_equal(loc.shift_arcsec[i, j], host)
                assert np.array_equal(loc.shift_pixels[i, j], np.array(r.shift_pixels, dtype=np.float64))
            else:
                for a in (0, 1):
                    assert abs(loc.shift_arcsec[i, j, a] - host[a]) <= 1e-3 * abs(steps[a]), (i, j, a)
                assert np.array_equal(loc.shift_arcsec[i, j, 2:], host[2:])
                assert np.array_equal(loc.shift_pixels[i, j, 2:], np.array(r.shift_pixels[2:], dtype=np.float64))
    return counts


def test_helioprojective_pair_shift_map(scene):
    from euispice_coreg_b200.hdrshift import Alignment
    res = Alignment(*scene["pair"], parallelism=True, local_block=64, **LAGS).align_using_helioprojective()
    assert res.local.fit_status.shape == (4, 4)
    counts = _check_against_results(res.local)
    assert counts[AR.FIT] >= 8


def test_carrington_fa_pair_shift_map(scene):
    from euispice_coreg_b200.hdrshift import Alignment
    res = Alignment(*scene["pair"], parallelism=True, **LAGS).align_using_carrington(local_block=64, **GRID)
    assert res.local.fit_status.shape == (4, 4)
    _check_against_results(res.local)


@pytest.mark.parametrize("frame", ["helioprojective", "carrington"])
def test_sequence_shift_maps(scene, frame):
    from euispice_coreg_b200.hdrshift import SequenceAlignment
    ref, frames = scene["frames"]
    seq = SequenceAlignment(ref, frames, **LAGS)
    if frame == "helioprojective":
        out = seq.align_using_helioprojective(local_block=64)
    else:
        out = seq.align_using_carrington(local_block=64, **GRID)
    assert len(out) == 3
    for r in out:
        _check_against_results(r.local)


@pytest.mark.parametrize("block", [64, (128, 64)])
def test_helioprojective_sequence_blocks_equal_per_pair_alignment(scene, block):
    from euispice_coreg_b200.hdrshift import Alignment, SequenceAlignment
    ref, frames = scene["frames"]
    out = SequenceAlignment(ref, frames, **LAGS).align_using_helioprojective(local_block=block)
    for p, r in zip(frames, out):
        one = Alignment(ref, p, parallelism=True, local_block=block, **LAGS).align_using_helioprojective()
        assert np.array_equal(r.corr, one.corr, equal_nan=True)
        assert np.array_equal(r.local.corr.view(np.uint64), one.local.corr.view(np.uint64))
        assert np.array_equal(r.local.nvalid, one.local.nvalid)
        assert np.array_equal(r.local.bounds, one.local.bounds)
        assert np.array_equal(r.local.max_index, one.local.max_index)


def test_peak_fit_kernel_does_not_spill(tmp_path):
    nvcc = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    src = os.path.join(ROOT, "euispice_coreg_b200", "csrc", "coreg_peak_fit.cu")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-I", os.path.join(ROOT, "include"), "-c", src, "-o", str(tmp_path / "fit.o")],
                         capture_output=True, text=True, check=True)
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", out.stderr)
    assert spills and all(s == ("0", "0") for s in spills), out.stderr
