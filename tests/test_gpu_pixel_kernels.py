"""The pixel-shift kernel and the one-pass image kernels, called directly, against exact references.

Part A drives `coreg_pixel_shift_corr` (the only kernel behind `pxlshift.AlignmentPixels`) at the shapes and lag sets
where its structure shows: 64 x 32 tiles (aligned, one pixel past, one pixel short), chunks of up to 8 x 8 (dx, dy)
lags (full, partial, unsorted, duplicated), several rotations, the 160 KiB staged-window limit on both sides, blocks of
the select-free fast path and of the general path in one launch, NaN and +-Inf in either image, lags without a valid
pair and lags that touch the large image's edges. The reference is the float64 Pearson of the oracle with the
reference's float32 numerator, lag by lag.

Part B drives the one-pass kernels of coreg_wcs.cu: the statistics pass (mean, count, max |v|; the RMS of the
centred float32 twin), the float32 -> float64 widening, the 32-bit byte swap and the SPICE wavelength sum, at sizes
around the statistics grid's stride (592 blocks x 256 threads = 151 552) and with non-finite values sprinkled in.
Count and max |v| decide the all-NaN error and the float32 headroom rule of the mixed-arithmetic search, RMS and
max |v| feed its per-lag guard: they are checked bit for bit or to 1e-13 against `math.fsum`.
"""
import ctypes as C
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from euispice_coreg_b200 import _ext
    _ext.load()
    return torch


def _dev(torch_mod):
    return torch_mod.device("cuda", torch_mod.cuda.current_device())


def _assert_same_values(got, want, what=""):
    """Equal bit for bit wherever `want` is not NaN, NaN exactly where `want` is NaN (a NaN's sign and payload carry
    no value: CUDA's NaN constant has the sign bit set, numpy's does not)."""
    assert got.shape == want.shape and got.dtype == want.dtype, what
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), f"{what}: NaN pattern differs"
    u = np.uint64 if got.dtype == np.float64 else np.uint32
    bad = np.flatnonzero(got[~nan].view(u) != want[~nan].view(u))
    assert bad.size == 0, f"{what}: {bad.size} values differ, first got {got[~nan][bad[0]]!r} want {want[~nan][bad[0]]!r}"


# =====================================================================================================================
# A. coreg_pixel_shift_corr
# =====================================================================================================================
TILE_W, TILE_H, CHUNK = 64, 32, 8       # coreg_pixel_shift.cu: block tile of the small image, (dx, dy) lags per chunk
WINDOW_LIMIT = 160 * 1024               # staged window bytes above which the host falls back to one lag per block


def _host_chunk(dx, dy):
    """The host's rule in coreg_pixel_shift_corr: chunks of 8 x 8 lags unless the staged window of the widest chunk,
    (64 + span_x)(32 + span_y) doubles, exceeds 160 KiB; then one lag per block."""
    def span(lags):
        return max(max(lags[i:i + CHUNK]) - min(lags[i:i + CHUNK]) for i in range(0, len(lags), CHUNK))
    return CHUNK if (TILE_W + span(dx)) * (TILE_H + span(dy)) * 8 <= WINDOW_LIMIT else 1


def _block_paths(large, sny, snx, x0, y0, dx, dy, chunk):
    """(fast, general) block counts per rotation: a block takes the general path when the part of the large image its
    chunk can reach (the tile grown by the chunk's dx / dy spans, clipped to the image) holds a non-finite value."""
    bad = ~np.isfinite(large)
    lny, lnx = large.shape
    fast = general = 0
    for ty in range(-(-sny // TILE_H)):
        for tx in range(-(-snx // TILE_W)):
            for i0 in range(0, len(dx), chunk):
                for j0 in range(0, len(dy), chunk):
                    cx, cy = dx[i0:i0 + chunk], dy[j0:j0 + chunk]
                    gx0, gy0 = x0 + tx * TILE_W + min(cx), y0 + ty * TILE_H + min(cy)
                    gx1, gy1 = gx0 + TILE_W + max(cx) - min(cx), gy0 + TILE_H + max(cy) - min(cy)
                    if bad[max(gy0, 0):min(gy1, lny), max(gx0, 0):min(gx1, lnx)].any():
                        general += 1
                    else:
                        fast += 1
    return fast, general


def _reference(large, smalls, x0, y0, dx, dy):
    """Lag by lag (oracle/pxlshift.py, `step`): r with the float32 numerator, the number of valid pairs, and the
    reference's float64 sums Sab, Saa, Sbb."""
    from oracle import pxlshift as P
    sums = P._pearson_f32num_jit or P._pearson_f32num_py
    n_rot, sny, snx = smalls.shape
    shape = (len(dx), len(dy), n_rot)
    r, sab, saa, sbb = (np.full(shape, np.nan) for _ in range(4))
    n = np.zeros(shape, dtype=np.int64)
    for i, ddx in enumerate(dx):
        for j, ddy in enumerate(dy):
            assert y0 + ddy >= 0 and x0 + ddx >= 0
            win = large[y0 + ddy:y0 + ddy + sny, x0 + ddx:x0 + ddx + snx]
            assert win.shape == (sny, snx)
            for k in range(n_rot):
                m = ~np.isnan(win) & ~np.isnan(smalls[k])
                a, b = np.ascontiguousarray(smalls[k][m]), np.ascontiguousarray(win[m])
                r[i, j, k] = P.pearson_f32num(a, b)
                n[i, j, k] = m.sum()
                if a.size:
                    sab[i, j, k], saa[i, j, k], sbb[i, j, k] = sums(a, b)
    return r, n, sab, saa, sbb


def _pivots(torch, d_large, d_smalls):
    from euispice_coreg_b200 import _ext
    pivots = torch.zeros(2, dtype=torch.float64, device=d_large.device)
    _ext.finite_mean(d_large, pivots[0:1])      # as AlignmentPixels.find_best_parameters does
    _ext.finite_mean(d_smalls, pivots[1:2])
    return pivots


def _gpu_pixel_shift(torch, large, smalls, x0, y0, dx, dy):
    from euispice_coreg_b200 import _ext
    dev = _dev(torch)
    d_large = torch.from_numpy(np.ascontiguousarray(large)).to(dev)
    d_smalls = torch.from_numpy(np.ascontiguousarray(smalls)).to(dev)
    corr, nvalid = _ext.pixel_shift_corr(d_large, d_smalls, x0, y0, dx, dy, _pivots(torch, d_large, d_smalls),
                                         return_nvalid=True)
    return corr.cpu().numpy(), nvalid.cpu().numpy()


def _pair(seed, sny, snx, dx, dy, n_rot):
    """A large image that the lags reach exactly to its edges (x0 + min dx = 0, x0 + max dx + snx = lnx, same in y)
    and n_rot different small images, each a noisy copy of the window of one lag."""
    rng = np.random.default_rng(seed)
    x0, y0 = -min(dx), -min(dy)
    lnx, lny = x0 + max(dx) + snx, y0 + max(dy) + sny
    large = rng.standard_normal((lny, lnx)) * 3.0 + 10.0
    smalls = np.empty((n_rot, sny, snx))
    for k in range(n_rot):
        i, j = rng.integers(len(dx)), rng.integers(len(dy))
        win = large[y0 + dy[j]:y0 + dy[j] + sny, x0 + dx[i]:x0 + dx[i] + snx]
        smalls[k] = 0.6 * win + rng.standard_normal((sny, snx)) * (1.0 + 0.5 * k)
    return large, smalls, x0, y0


def _case_aligned_32x64():
    dx, dy = list(range(-4, 4)), list(range(-3, 5))
    return (*_pair(1, 32, 64, dx, dy, 1), dx, dy, CHUNK, "fast", None)


def _case_aligned_64x128():
    # 17 = 8 + 8 + 1 and 9 = 8 + 1 lags: full and partial chunks in both axes, three rotations; the only NaN of the
    # large image sits in its corner, inside the staged window of one (tile, chunk) only; one whole tile of the second
    # rotation's small image is NaN
    dx, dy = list(range(-8, 9)), list(range(-4, 5))
    large, smalls, x0, y0 = _pair(2, 64, 128, dx, dy, 3)
    large[0, 0] = np.nan
    smalls[1, 32:64, 64:128] = np.nan

    def check(r, n):
        assert n[:, :, 1].max() == 64 * 128 - 32 * 64 and n[0, 0, 0] == 64 * 128 - 1
    return large, smalls, x0, y0, dx, dy, CHUNK, "mixed", check


def _case_one_past_33x65():
    # tiles one pixel past the 64 x 32 edge in both axes; NaN rows and columns differ per rotation
    dx, dy = list(range(-4, 5)), list(range(-8, 9))
    large, smalls, x0, y0 = _pair(3, 33, 65, dx, dy, 3)
    smalls[0, 0, :] = smalls[0, :, 64] = np.nan
    smalls[1, 32, :] = smalls[1, :, 0] = np.nan
    smalls[2, 10:12, :] = np.nan
    smalls[2, :, [30, 31, 63]] = np.nan
    return large, smalls, x0, y0, dx, dy, CHUNK, "fast", None


def _case_one_short_31x63():
    # tiles one pixel short of the edge, a single dy lag; the second rotation keeps only column 10, and a NaN column of
    # the large image meets it at dx = -3: those lags have no valid pair
    dx, dy = list(range(-3, 5)), [0]
    large, smalls, x0, y0 = _pair(4, 31, 63, dx, dy, 2)
    keep = smalls[1, :, 10].copy()
    smalls[1] = np.nan
    smalls[1, :, 10] = keep
    large[:, x0 - 3 + 10] = np.nan

    def check(r, n):
        assert n[0, 0, 1] == 0 and np.isnan(r[0, 0, 1]) and (n[1:, 0, 1] == 31).all()
    return large, smalls, x0, y0, dx, dy, CHUNK, "general", check


def _case_single_pixel():
    # a 1 x 1 small image: one live pixel in a mostly dead tile, n <= 1 so every r is NaN; the second rotation is
    # NaN, and one NaN of the large image leaves one lag of the others without a pair
    dx, dy = list(range(-8, 9)), list(range(-8, 9))
    large, smalls, x0, y0 = _pair(5, 1, 1, dx, dy, 3)
    smalls[1] = np.nan
    large[3, 3] = np.nan

    def check(r, n):
        assert np.isnan(r).all() and (n[:, :, 1] == 0).all()
        assert n[dx.index(-5), dy.index(-5), 0] == 0 and n.sum() == 2 * (17 * 17 - 1)
    return large, smalls, x0, y0, dx, dy, CHUNK, "mixed", check


def _case_unsorted_duplicates():
    # unsorted lag arrays with repeated values; the second rotation is an exact affine copy of the window of one
    # lag, so |r| is 1 up to rounding there (and may exceed it: the numerator is rounded to float32)
    dx, dy = [3, -2, 3, 0, 7, -5, 1, 1, 2], [2, -1, -3, 2, 0, 4, -2, 1]
    large, smalls, x0, y0 = _pair(6, 48, 70, dx, dy, 2)
    smalls[1] = 2.5 * large[y0 - 3:y0 - 3 + 48, x0 + 7:x0 + 7 + 70] + 3.0

    def check(r, n):
        assert abs(r[dx.index(7), dy.index(-3), 1] - 1.0) < 1e-6
        assert np.array_equal(r[0], r[2]) and np.array_equal(r[:, 0], r[:, 3])   # repeated lags, same value
    return large, smalls, x0, y0, dx, dy, CHUNK, "fast", check


_DX_SPAN64 = [0, 9, 18, 27, 36, 45, 54, 64]


def _case_window_at_limit():
    # dx span 64, dy span 128: the staged window is (64 + 64) x (32 + 128) doubles = 160 KiB exactly, chunks of 8;
    # a NaN in the large image's first row is in reach of the first tile row only
    dx, dy = _DX_SPAN64, [0, 18, 37, 55, 73, 91, 110, 128]
    large, smalls, x0, y0 = _pair(7, 64, 64, dx, dy, 2)
    large[0, 5] = np.nan
    return large, smalls, x0, y0, dx, dy, CHUNK, "mixed", None


def _case_window_over_limit():
    # dy span 129: one byte row past 160 KiB, one lag per block
    dx, dy = _DX_SPAN64, [0, 18, 37, 55, 73, 91, 110, 129]
    large, smalls, x0, y0 = _pair(8, 64, 64, dx, dy, 2)
    large[0, 5] = np.nan
    return large, smalls, x0, y0, dx, dy, 1, "mixed", None


def _case_ragged_inf():
    # 150 x 201 (5 x 4 tiles, ragged): +Inf and -Inf in the large image's opposite corners (one lag reaches each),
    # +Inf in the first rotation's small image except at the lag where a NaN of the large image masks it, -Inf in the
    # second rotation's, a NaN hole in all three
    dx, dy = list(range(-4, 5)), list(range(-4, 4))
    large, smalls, x0, y0 = _pair(9, 150, 201, dx, dy, 3)
    large[0, 0], large[-1, -1] = np.inf, -np.inf
    smalls[:, 40:44, 100:108] = np.nan
    smalls[0, 5, 7] = np.inf
    smalls[1, 100, 150] = -np.inf
    large[y0 - 1 + 5, x0 + 2 + 7] = np.nan

    def check(r, n):
        i, j = dx.index(2), dy.index(-1)
        assert np.isfinite(r[i, j, 0]) and np.isnan(r[:, :, 0]).sum() == r[:, :, 0].size - 1
        assert np.isnan(r[:, :, 1]).all()
        assert np.isnan(r[0, 0, 2]) and np.isnan(r[-1, -1, 2]) and np.isfinite(r[:, :, 2]).sum() == r[:, :, 2].size - 2
    return large, smalls, x0, y0, dx, dy, CHUNK, "mixed", check


PX_CASES = {f.__name__[len("_case_"):]: f for f in (
    _case_aligned_32x64, _case_aligned_64x128, _case_one_past_33x65, _case_one_short_31x63, _case_single_pixel,
    _case_unsorted_duplicates, _case_window_at_limit, _case_window_over_limit, _case_ragged_inf)}


@pytest.mark.parametrize("name", list(PX_CASES))
def test_pixel_shift_matches_float64_reference(torch_cuda, name):
    large, smalls, x0, y0, dx, dy, chunk, paths, check = PX_CASES[name]()
    n_rot, sny, snx = smalls.shape
    # the case sits in the regime it was written for: chunk size, and which inner loop its blocks take
    assert _host_chunk(dx, dy) == chunk
    fast, general = _block_paths(large, sny, snx, x0, y0, dx, dy, chunk)
    assert {"fast": (True, False), "general": (False, True), "mixed": (True, True)}[paths] == (fast > 0, general > 0)

    r_gpu, n_gpu = _gpu_pixel_shift(torch_cuda, large, smalls, x0, y0, dx, dy)
    r_ref, n_ref, sab, saa, sbb = _reference(large, smalls, x0, y0, dx, dy)
    if check is not None:
        check(r_ref, n_ref)
    assert r_gpu.shape == r_ref.shape == (len(dx), len(dy), n_rot)
    assert np.array_equal(n_gpu, n_ref)
    assert np.array_equal(np.isnan(r_gpu), np.isnan(r_ref))
    fin = ~np.isnan(r_ref)
    # the float64 numerators of kernel and reference differ in their last bits and may round to neighbouring float32
    # values: one float32 ulp of the numerator
    err = np.abs(r_gpu[fin] - r_ref[fin])
    assert np.all(err <= 2.0 ** -23 * np.abs(r_ref[fin]) + 1e-12), float(err.max())
    # the float32 numerator is applied: with the reference's denominators, r * sqrt(Saa Sbb) is a float32 value (the
    # kernel's single-pass denominators agree with the two-pass ones far below 1e-9; an unrounded float64 numerator
    # lies ~3e-8 off the float32 grid)
    num = r_gpu[fin] * np.sqrt(saa[fin] * sbb[fin])
    off = np.abs(num - num.astype(np.float32).astype(np.float64))
    assert np.all(off <= 1e-9 * np.abs(num)), float((off / np.abs(num)).max())
    if fin.sum() >= 16:
        # ... and the data can tell: most reference numerators are off the float32 grid before rounding
        raw = sab[fin]
        assert np.mean(np.abs(raw - raw.astype(np.float32)) > 1e-9 * np.abs(raw)) > 0.5


def test_pixel_shift_lags_at_the_edges_accepted_one_past_refused(torch_cuda):
    from euispice_coreg_b200 import _ext
    dx, dy = [-2, 0, 3], [-3, 1, 2]
    large, smalls, x0, y0 = _pair(10, 33, 65, dx, dy, 1)
    # x0 + min dx = 0, x0 + max dx + snx = lnx and the same in y: accepted
    r, _ = _gpu_pixel_shift(torch_cuda, large, smalls, x0, y0, dx, dy)
    assert np.isfinite(r).all()
    for bad_dx, bad_dy in ((dx + [-3], dy), (dx + [4], dy), (dx, dy + [-4]), (dx, dy + [3])):
        with pytest.raises(_ext.CoregLibraryError, match="too large shift"):
            _gpu_pixel_shift(torch_cuda, large, smalls, x0, y0, bad_dx, bad_dy)


def test_alignment_pixels_equals_direct_kernel_call(torch_cuda, tmp_path):
    """The public path hands the kernel the resampled large image, the slice origin and the pivots of
    `_ext.finite_mean`: its cube is the direct call's, bit for bit."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.pxlshift.alignment_pixels import AlignmentPixels
    rng = np.random.default_rng(11)
    large = rng.standard_normal((120, 180)) * 5.0 + 50.0
    small = 0.8 * large[38:38 + 45, 52:52 + 70] + rng.standard_normal((45, 70))
    large[60:63, 100:140] = np.nan
    small[20, :] = np.nan
    h = {"CDELT1": 2.0, "CDELT2": 2.0, "CUNIT1": "arcsec", "CUNIT2": "arcsec"}
    paths = []
    for name, d in (("L", large), ("S", small)):
        hdr = fits_lite.Header()
        for k, v in h.items():
            hdr[k] = v
        paths.append(str(tmp_path / f"{name}.fits"))
        fits_lite.writeto(paths[-1], [fits_lite.PrimaryHDU(d, hdr)], overwrite=True)
    dx, dy = np.arange(-9, 10), np.array([5, -3, 0, 1, 1, -7, 2, 8, -1])
    a = AlignmentPixels(paths[0], 0, paths[1], 0)
    corr = a.find_best_parameters(dx, dy, np.array([0.0]))
    y0, x0 = a.slc_small_ref[0].start, a.slc_small_ref[1].start
    r, n = _gpu_pixel_shift(torch_cuda, a.data_large, a.data_small[None], x0, y0, list(dx), list(dy))
    assert np.array_equal(corr.view(np.uint64), r.view(np.uint64))
    assert np.array_equal(a.nvalid, n)
    assert np.isfinite(corr).sum() > corr.size // 2


# =====================================================================================================================
# B. one-pass image kernels (coreg_wcs.cu)
# =====================================================================================================================
STAT_STRIDE = 592 * 256   # kStatBlocks x kStatThreads: the grid stride of the statistics pass
SIZES = [1, 255, 256, 257, STAT_STRIDE - 1, STAT_STRIDE, STAT_STRIDE + 1, 2 * STAT_STRIDE + 7, 2048 * 2048]
PATTERNS = ["sprinkled", "all_nan", "all_inf", "only_last", "only_first"]
SENTINEL = -123456.75


def _values(n, dtype, pattern, seed=0):
    """Test image of n values. "sprinkled": finite values with NaN, +-Inf, -0.0, subnormals and a few large values
    scattered through; "only_last" / "only_first": NaN but for one finite value at index n - 1 (the last stride of
    the last block) / 0."""
    rng = np.random.default_rng(seed + n)
    if pattern == "all_nan":
        return np.full(n, np.nan, dtype=dtype)
    if pattern == "all_inf":
        x = np.full(n, np.inf, dtype=dtype)
        x[1::2] = -np.inf
        return x
    if pattern in ("only_last", "only_first"):
        x = np.full(n, np.nan, dtype=dtype)
        x[-1 if pattern == "only_last" else 0] = -3.25
        return x
    x = (rng.standard_normal(n) * 40.0 + 7.0).astype(dtype)
    if n >= 8:
        k = max(1, n // 200)
        tiny = np.finfo(dtype).smallest_normal / 8
        for v, cnt in ((np.nan, 2 * k), (np.inf, k), (-np.inf, k), (-0.0, k), (tiny, k), (-tiny, k),
                       (-4.0e5, 1), (3.5e5, 1)):
            x[rng.integers(0, n, cnt)] = v
    return x


def _ref_stats(x):
    """(count, mean, max |v|) over the finite values: count and max exact, the mean from the correctly rounded sum."""
    v = x[np.isfinite(x)].astype(np.float64)
    if v.size == 0:
        return 0, 0.0, 0.0
    return v.size, math.fsum(v.tolist()) / v.size, float(np.abs(v).max())


def _ref_rms(c32):
    """RMS of the finite values of a float32 array (squares of float32 values are exact in float64)."""
    c = c32[np.isfinite(c32)].astype(np.float64)
    return math.sqrt(math.fsum((c * c).tolist()) / c.size) if c.size else 0.0


def _check_stats_column(col, x, what):
    cnt, mean, mx = _ref_stats(x)
    assert col[1] == cnt, f"{what}: count {col[1]} != {cnt}"
    assert col[2] == mx, f"{what}: max|v| {col[2]!r} != {mx!r}"
    assert abs(col[0] - mean) <= 1e-13 * mx, f"{what}: mean {col[0]!r} vs fsum {mean!r}"
    assert col[3] == 0.0, f"{what}: row 3 not reset"


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", SIZES)
def test_image_stats_exact(torch_cuda, n, dtype):
    from euispice_coreg_b200 import _ext
    torch = torch_cuda
    widen = dtype == np.float32
    for pattern in PATTERNS:
        x = _values(n, dtype, pattern)
        stats = torch.full((4, 2), SENTINEL, dtype=torch.float64, device=_dev(torch))
        wide = _ext.image_stats(torch.from_numpy(x).to(stats.device), stats, 1, widen=widen)
        st = stats.cpu().numpy()
        _check_stats_column(st[:, 1], x, f"n={n} {np.dtype(dtype).name} {pattern}")
        assert (st[:, 0] == SENTINEL).all()
        if widen:
            _assert_same_values(wide.cpu().numpy(), x.astype(np.float64), f"widened copy n={n} {pattern}")


@pytest.mark.parametrize("n", SIZES)
def test_center_f32_exact(torch_cuda, n):
    from euispice_coreg_b200 import _ext
    torch = torch_cuda
    for pattern in PATTERNS:
        x = _values(n, np.float32, pattern, seed=1)
        stats = torch.full((4, 2), SENTINEL, dtype=torch.float64, device=_dev(torch))
        d = torch.from_numpy(x).to(stats.device)
        _ext.image_stats(d, stats, 1)
        before = stats.cpu().numpy()
        out = _ext.center_f32(d, stats, 1).cpu().numpy()
        st = stats.cpu().numpy()
        # the kernel's own pivot, rounded to float32, subtracted in float32
        want = x - np.float32(st[0, 1])
        _assert_same_values(out, want, f"centred n={n} {pattern}")
        rms = _ref_rms(want)
        assert abs(st[3, 1] - rms) <= 1e-13 * rms, (pattern, st[3, 1], rms)
        assert np.array_equal(st[:3], before[:3]) and (st[:, 0] == SENTINEL).all()


def test_stats_block_columns_and_rows(torch_cuda):
    """A [4][3] block: each call writes its own column only, and only the rows include/coreg_b200.h gives it
    (statistics: rows 0-3, row 3 = 0; centring: row 3)."""
    from euispice_coreg_b200 import _ext
    torch = torch_cuda
    dev = _dev(torch)
    imgs = {0: _values(STAT_STRIDE + 1, np.float64, "sprinkled", seed=2),
            1: _values(2 * STAT_STRIDE + 7, np.float32, "sprinkled", seed=3),
            2: _values(257, np.float32, "sprinkled", seed=4)}
    blk = torch.full((4, 3), SENTINEL, dtype=torch.float64, device=dev)
    expect = np.full((4, 3), SENTINEL)
    for col in (1, 0, 2):
        _ext.image_stats(torch.from_numpy(imgs[col]).to(dev), blk, col)
        got = blk.cpu().numpy()
        _check_stats_column(got[:, col], imgs[col], f"column {col}")
        others = [c for c in range(3) if c != col]
        assert np.array_equal(got[:, others], expect[:, others]), f"image_stats into column {col} wrote elsewhere"
        expect[:, col] = got[:, col]
    d1 = torch.from_numpy(imgs[1]).to(dev)
    _ext.center_f32(d1, blk, 1)
    got = blk.cpu().numpy()
    rms = _ref_rms(imgs[1] - np.float32(expect[0, 1]))
    assert abs(got[3, 1] - rms) <= 1e-13 * rms
    expect[3, 1] = got[3, 1]
    assert np.array_equal(got, expect)
    # centring reads row 0 and writes row 3 only
    blk2 = torch.full((4, 3), SENTINEL, dtype=torch.float64, device=dev)
    blk2[0, 1] = float(expect[0, 1])
    _ext.center_f32(d1, blk2, 1)
    got2 = blk2.cpu().numpy()
    want2 = np.full((4, 3), SENTINEL)
    want2[0, 1], want2[3, 1] = expect[0, 1], expect[3, 1]
    assert np.array_equal(got2, want2)


def _lib_stats(lib, img, stats, col, scratch, widen=None):
    from euispice_coreg_b200 import _ext
    _ext._check(lib.coreg_image_stats(_ext._ptr(img), _ext._dt(img), img.numel(),
                                      _ext._ptr(widen) if widen is not None else None,
                                      C.c_void_p(stats.data_ptr() + 8 * col), stats.shape[1], _ext._ptr(scratch),
                                      _ext._stream()), "coreg_image_stats")


def _lib_center(lib, img, out, stats, col, scratch):
    from euispice_coreg_b200 import _ext
    _ext._check(lib.coreg_center_f32(_ext._ptr(img), img.numel(), _ext._ptr(out),
                                     C.c_void_p(stats.data_ptr() + 8 * col), stats.shape[1], _ext._ptr(scratch),
                                     _ext._stream()), "coreg_center_f32")


def test_stats_scratch_reuse_is_deterministic(torch_cuda):
    """One scratch buffer (filled with 0xFF bytes, its counter included) serves a sequence of statistics and centring
    passes over alternating images, as coreg_hpc_search_host uses it: every result equals the one of a call on its
    own fresh scratch, and repeating the sequence repeats the bits."""
    from euispice_coreg_b200 import _ext
    torch = torch_cuda
    dev = _dev(torch)
    lib = _ext.load()
    nbytes = int(lib.coreg_image_stats_scratch_bytes())

    def garbage():
        return torch.full((nbytes,), 0xFF, dtype=torch.uint8, device=dev)

    small = torch.from_numpy(_values(2048 * 2048, np.float32, "sprinkled", seed=5)).to(dev)
    ref = torch.from_numpy(_values(STAT_STRIDE + 1, np.float32, "sprinkled", seed=6)).to(dev)
    other = torch.from_numpy(_values(257, np.float64, "sprinkled", seed=7)).to(dev)

    def sequence(scratch_for):
        blk = torch.full((4, 2), SENTINEL, dtype=torch.float64, device=dev)
        blk2 = torch.full((4, 2), SENTINEL, dtype=torch.float64, device=dev)
        wide = torch.empty(small.shape, dtype=torch.float64, device=dev)
        cen = torch.empty_like(small)
        _lib_stats(lib, small, blk, 1, scratch_for(), widen=wide)
        _lib_stats(lib, ref, blk, 0, scratch_for())
        _lib_center(lib, small, cen, blk, 1, scratch_for())
        _lib_stats(lib, other, blk2, 1, scratch_for())
        _lib_stats(lib, small, blk2, 0, scratch_for())
        _lib_center(lib, ref, torch.empty_like(ref), blk, 0, scratch_for())
        return [t.cpu().numpy() for t in (blk, blk2, wide, cen)]

    shared = garbage()
    runs = [sequence(lambda: shared) for _ in range(3)]
    fresh = sequence(garbage)
    for run in runs:
        for got, want in zip(run, fresh):
            assert got.tobytes() == want.tobytes()
    blk, blk2 = fresh[0], fresh[1]
    for col, x in ((blk[:, 1], small), (blk[:, 0], ref), (blk2[:, 1], other), (blk2[:, 0], small)):
        cnt, mean, mx = _ref_stats(x.cpu().numpy())
        assert col[1] == cnt and col[2] == mx and abs(col[0] - mean) <= 1e-13 * mx
    assert np.array_equal(blk2[:, 0], np.r_[blk[:3, 1], 0.0])


@pytest.mark.parametrize("byteorder", ["=", ">"])
def test_engine_mixed_statistics_column(torch_cuda, byteorder):
    """`LagSearchEngine.set_small` with mixed arithmetic on a float32 image (native, or big-endian as a FITS payload is
    stored): the small image's column of the statistics block is what the mixed kernel's guard and the float32
    headroom rule read."""
    from euispice_coreg_b200.hdrshift.engine import LagSearchEngine
    x = _values(300 * 517, np.float32, "sprinkled", seed=8).reshape(300, 517)
    eng = LagSearchEngine(order=2, arithmetic="mixed")
    eng.set_small(x.astype(np.dtype(np.float32).newbyteorder(byteorder)))
    st = eng.stats.cpu().numpy()[:, 1]
    cnt, mean, mx = _ref_stats(x)
    assert st[1] == cnt and st[2] == mx and abs(st[0] - mean) <= 1e-13 * mx
    centred = x - np.float32(st[0])
    rms = _ref_rms(centred)
    assert abs(st[3] - rms) <= 1e-13 * rms
    assert eng.small_count() == cnt
    _assert_same_values(eng.small.cpu().numpy(), x.astype(np.float64), "widened small image")
    _assert_same_values(eng.small32.cpu().numpy(), centred, "centred float32 twin")


@pytest.mark.parametrize("n", SIZES)
def test_widen_and_bswap_bit_exact(torch_cuda, n):
    from euispice_coreg_b200 import _ext
    torch = torch_cuda
    dev = _dev(torch)
    x = _values(n, np.float32, "sprinkled", seed=9)
    _assert_same_values(_ext.widen_f32(torch.from_numpy(x).to(dev)).cpu().numpy(), x.astype(np.float64), "widen")
    # byte swap: arbitrary 32-bit words (NaN payloads included), in place through the wrapper, out of place through
    # the C entry point
    words = np.random.default_rng(n).integers(0, 2 ** 32, n, dtype=np.uint32)
    swapped = words.byteswap()
    d_in = torch.from_numpy(words.view(np.int32)).to(dev)
    inplace = _ext.bswap32_to_float32(d_in.clone())
    assert np.array_equal(inplace.cpu().numpy().view(np.uint32), swapped)
    out = torch.empty_like(d_in)
    lib = _ext.load()
    _ext._check(lib.coreg_bswap32(_ext._ptr(d_in), n, _ext._ptr(out), _ext._stream()), "coreg_bswap32")
    assert np.array_equal(out.cpu().numpy().view(np.uint32), swapped)
    assert np.array_equal(d_in.cpu().numpy().view(np.uint32), words)


@pytest.mark.parametrize("shape", [(9, 37, 53), (3, 600, 611)])
@pytest.mark.parametrize("byteorder", ["=", ">"])
def test_spice_wave_sum_matches_nansum(torch_cuda, byteorder, shape):
    """`np.nansum(cube[sel].astype(np.float64), axis=0)` with the rows outside [ymin, ymax) NaN, bit for bit."""
    from euispice_coreg_b200 import _ext
    n_lambda, ny, nx = shape
    rng = np.random.default_rng(12)
    # magnitudes over many decades, both signs: a different order of the additions would show in the last bits
    cube = (rng.lognormal(0.0, 4.0, shape) * rng.choice([-1.0, 1.0], shape)).astype(np.float32)
    cube[rng.random(shape) < 0.1] = np.nan
    cube[:, 3, 4] = np.nan          # NaN in every plane: +0.0
    cube[:, 5, 6] = -0.0            # -0.0 in every plane: +0.0 (numpy's sum starts from +0.0)
    cube[0, 7, 8], cube[-1, 7, 8] = np.inf, -np.inf   # +Inf + -Inf: NaN
    payload = cube.astype(cube.dtype.newbyteorder(byteorder))
    sels = [np.arange(n_lambda) % 3 != 1,                          # gaps
            np.arange(n_lambda) == n_lambda // 2,                  # a single plane
            np.ones(n_lambda, dtype=bool)]                         # every plane
    for sel in sels:
        for ymin, ymax in ((0, ny), (2, ny - 5), (ny // 2, ny // 2)):
            got = _ext.spice_wave_sum(payload, sel, ymin, ymax).cpu().numpy()
            with np.errstate(invalid="ignore"):
                want = np.nansum(cube[sel].astype(np.float64), axis=0)
            want[:ymin] = np.nan
            want[ymax:] = np.nan
            _assert_same_values(got, want, f"sel={sel.astype(int)} rows [{ymin}, {ymax})")
            if ymin <= 3 and 5 < ymax:
                assert got[3, 4].view(np.uint64) == 0 and got[5, 6].view(np.uint64) == 0
            if sel.all() and ymin <= 7 < ymax:
                assert np.isnan(got[7, 8])
