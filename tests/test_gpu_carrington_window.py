"""The Carrington window kernel (`offset_window_kernel`, csrc/coreg_lag_offset.cu) through its C entry
`coreg_offset_lag_corr`, against a float64 reference, at the box, rim, chunk and super-tile edges.

Every case is built from dyadic values: lag offsets and the coordinate planes Tx = a gx + b gy + c,
Ty = d gx + e gy + f are multiples of 1/64 far below 2^12. The kernel forms sx = (x0 + 0.5) + Tx and samples at
sx - 0.5; the reference forms x0 + Tx. For such inputs both are exact and equal (checked for every (pixel, lag) pair
on the CPU), so every rim, liveness and fit decision is the same on both sides: the valid counts must match exactly,
r to 1e-9. The small images hold float32 values, so a float32 and a float64 copy must give the same bits.

With COREG_OFFSET_STATS=1 the launch reports how it served its (tile, chunk) pairs. `predict` restates the kernel's
decisions per (tile, chunk) -- super-tile liveness, window bounds with the 16-byte round-down, fit in the box -- and
the reported counts must equal it, so each case is known to have taken the path it was built for.
"""
import functools
import math
import os
import re

import numpy as np
import pytest
from scipy.ndimage import map_coordinates

from oracle.pearson import pearson

# csrc/coreg_lag_offset.cu: kOffTileW x kOffTileH tiles, kOffTilesPerBlock of them stacked per super-tile,
# kOffThreads lags per chunk, OffBox<T> (window box = TMA box), 16-byte alignment of the box origin
TILE_W, TILE_H, TILES_PER_SUPER = 32, 8, 8
SUPER_H = TILE_H * TILES_PER_SUPER
CHUNK = 256
BOX = {4: (192, 64), 8: (96, 56)}
MAX_GRID_Y = 65535                       # launch_offset_window: chunks per block = ceil(n_chunks / 65535)
BIG = 2.0 ** 30                          # small_magnitude (coreg_common.cuh): |v| < 2^30
FILL = -32762.0                          # a sample equal to this is missing (alignment.py: np.where(image == -32762))
R_TOL = 1e-9
FLAG_STRICT, FLAG_NO_FAST = 1, 4         # _ext.FLAG_STRICT, _ext.FLAG_NO_FAST (the CPU tests do not load the library)
MANY_LAGS = 65536 * CHUNK + 1            # 65537 chunks: two per block, an odd grid.y


# =====================================================================================================================
# reference and restatement (CPU)
# =====================================================================================================================
def reference(ref, small, tx, ty, lags, order=2):
    """(r, nvalid) per lag: scipy's map_coordinates at (y0 + Ty, x0 + Tx), constant mode with NaN outside, no
    prefilter; a pair counts when the reference value and the sample are finite, the sample is not -32762, and Tx, Ty,
    x0 + 0.5, y0 + 0.5 pass the kernel's |.| < 2^30 guards. r: two-pass float64 Pearson of the counted pairs."""
    s64 = np.asarray(small, dtype=np.float64)
    live = np.isfinite(ref) & (np.abs(tx) < BIG) & (np.abs(ty) < BIG)
    a, px, py = ref[live], tx[live], ty[live]
    r = np.full(len(lags), np.nan)
    n = np.zeros(len(lags), dtype=np.int64)
    for k, (x0, y0) in enumerate(np.asarray(lags, dtype=np.float64)):
        if not (abs(x0 + 0.5) < BIG and abs(y0 + 0.5) < BIG):
            continue
        v = map_coordinates(s64, [y0 + py, x0 + px], order=order, mode="constant", cval=np.nan, prefilter=False)
        ok = np.isfinite(v) & (v != FILL)
        n[k] = int(ok.sum())
        if n[k]:
            r[k] = pearson(a[ok], v[ok])
    return r, n


def tma_expected(case):
    """The kernel stages with TMA when the small image's base address and row pitch are 16-byte aligned."""
    small = case["small"]
    return int(case.get("offset", 0) == 0 and (small.shape[1] * small.itemsize) % 16 == 0)


def predict(case, itemsize=None):
    """The kernel's per-(tile, chunk) decisions (offset_super_live_kernel, offset_window_kernel): which super-tiles are
    live, and for every live tile and chunk with a live lag the window [wx0, wx1] x [wy0, wy1] (wx0 rounded down to
    16 bytes), skipped when it misses the image, staged when it fits the box, read from global memory otherwise."""
    ref, tx, ty, lags = case["ref"], case["tx"], case["ty"], np.asarray(case["lags"], dtype=np.float64)
    itemsize = itemsize or case["small"].itemsize
    sny, snx = case["small"].shape
    bw, bh = BOX[itemsize]
    align = 16 // itemsize
    gny, gnx = ref.shape
    live = np.isfinite(ref) & (np.abs(tx) < BIG) & (np.abs(ty) < BIG)
    x0h, y0h = lags[:, 0] + 0.5, lags[:, 1] + 0.5
    ok = (np.abs(x0h) < BIG) & (np.abs(y0h) < BIG)
    n_chunks = -(-len(lags) // CHUNK)
    cpb = -(-n_chunks // MAX_GRID_Y)

    def per_chunk(v, fn, fill):
        w = np.concatenate([np.where(ok, v, fill), np.full(n_chunks * CHUNK - len(v), fill)])
        return fn(w.reshape(n_chunks, CHUNK), axis=1)

    cx0, cx1 = per_chunk(x0h, np.min, np.inf), per_chunk(x0h, np.max, -np.inf)
    cy0, cy1 = per_chunk(y0h, np.min, np.inf), per_chunk(y0h, np.max, -np.inf)
    any_lag = cx0 <= cx1
    cx0, cx1, cy0, cy1 = cx0[any_lag], cx1[any_lag], cy0[any_lag], cy1[any_lag]
    out = dict(staged=0, global_=0, walks=0, width=0, height=0, live_super=[], dead_super=[],
               dead_chunks=int((~any_lag).sum()), cpb=cpb, tma=tma_expected(case))
    rx0, rx1 = (x0h[ok].min(), x0h[ok].max()) if ok.any() else (np.inf, -np.inf)
    ry0, ry1 = (y0h[ok].min(), y0h[ok].max()) if ok.any() else (np.inf, -np.inf)
    for oy in range(0, gny, SUPER_H):
        for ox in range(0, gnx, TILE_W):
            sl = np.s_[oy:oy + SUPER_H, ox:ox + TILE_W]
            m = live[sl]
            reach = False
            if m.any():
                px, py = tx[sl][m], ty[sl][m]
                reach = (px.max() + rx1 >= -0.5) and (px.min() + rx0 <= snx + 0.5) and \
                        (py.max() + ry1 >= -0.5) and (py.min() + ry0 <= sny + 0.5)
            out["live_super" if reach else "dead_super"].append((oy // SUPER_H, ox // TILE_W))
            if not reach:
                continue
            for t in range(TILES_PER_SUPER):
                st = np.s_[oy + t * TILE_H:min(oy + (t + 1) * TILE_H, gny), ox:ox + TILE_W]
                mt = live[st]
                if not mt.any():
                    continue
                bx, by = tx[st][mt], ty[st][mt]
                wx0 = np.floor(bx.min() + cx0).astype(np.int64) - 1
                wx0 -= wx0 % align
                wx1 = np.floor(bx.max() + cx1).astype(np.int64) + 1
                wy0 = np.floor(by.min() + cy0).astype(np.int64) - 1
                wy1 = np.floor(by.max() + cy1).astype(np.int64) + 1
                inside = ~((wx1 < 0) | (wx0 > snx - 1) | (wy1 < 0) | (wy0 > sny - 1))
                w, h = wx1 - wx0 + 1, wy1 - wy0 + 1
                fits = (w <= bw) & (h <= bh)
                out["staged"] += int((fits & inside).sum())
                out["global_"] += int((~fits & inside).sum())
                out["walks"] += int(inside.sum()) * int(mt.sum())
                if inside.any():
                    out["width"] = max(out["width"], int(w[inside].max()))
                    out["height"] = max(out["height"], int(h[inside].max()))
    return out


def window_kernel_used(small, order=2, flags=0):
    """coreg_offset_lag_corr takes the window kernel at order 2, without FLAG_STRICT / FLAG_NO_FAST, on images of at
    least 3 x 3 pixels; the generic kernel otherwise."""
    return order == 2 and not flags & (FLAG_STRICT | FLAG_NO_FAST) and min(small.shape) >= 3


# =====================================================================================================================
# cases
# =====================================================================================================================
def _planes(gny, gnx, a=4.375, b=0.125, c=0.0, d=-0.0625, e=1.75, f=0.0):
    gy, gx = np.mgrid[0:gny, 0:gnx].astype(np.float64)
    return a * gx + b * gy + c, d * gx + e * gy + f


def _images(seed, gny, gnx, sny, snx, dtype=np.float32):
    rng = np.random.default_rng(seed)
    ref = rng.normal(500.0, 50.0, (gny, gnx))
    ref[rng.random((gny, gnx)) < 0.02] = np.nan
    small = rng.normal(1000.0, 100.0, (sny, snx)).astype(np.float32).astype(dtype)
    return ref, small


def _patch_lags(x0, y0, n1=16, n2=16, step=0.5):
    """An n1 x n2 CRVAL-like lag grid `step` pixels apart, in the engine's patch order (NaN dummies in the gaps)."""
    from euispice_coreg_b200.hdrshift.engine import offset_patch_order
    i1, i2 = (g.ravel() for g in np.meshgrid(np.arange(n1), np.arange(n2), indexing="ij"))
    slot, n_slots = offset_patch_order(i1, i2)
    table = np.full((n_slots, 2), np.nan)
    table[slot] = np.stack([x0 + step * i1, y0 + step * i2], axis=1)
    return table


def _case(ref, small, tx, ty, lags, **claims):
    return dict(ref=ref, small=small, tx=tx, ty=ty, lags=np.ascontiguousarray(lags, dtype=np.float64), claims=claims)


def _staged(dtype):
    """Two 16 x 16 patches of lags half a pixel apart over a 70 x 100 grid (ragged super-tiles); the second patch
    pushes part of the grid off the image's left and top edges. Neighbouring grid pixels land 4.375 (float32) or 2.5
    (float64) detector pixels apart: every window fits its box."""
    a = 4.375 if dtype == np.float32 else 2.5
    ref, small = _images(1, 70, 100, 200, 480 if dtype == np.float32 else 300, dtype)
    tx, ty = _planes(70, 100, a=a, c=2.0, f=3.0)
    lags = np.concatenate([_patch_lags(10.0, 20.0), _patch_lags(-3.25, -5.5)])
    return _case(ref, small, tx, ty, lags, staged=True, global_=False, clean=True)


def _dirty(dtype):
    """The staged case with NaN, +inf, -inf and isolated -32762 pixels inside its windows (the pixels are not missing,
    the samples that touch the non-finite ones are), and a 3 x 3 plateau of -32762 centred where one (pixel, lag)
    pair samples at integer coordinates: that sample is exactly -32762 and missing on every path."""
    c = _staged(dtype)
    small, ref, tx, ty, lags = c["small"], c["ref"], c["tx"], c["ty"], c["lags"]
    sny, snx = small.shape
    rng = np.random.default_rng(2)
    for v in (np.nan, np.inf, -np.inf, FILL):
        small[rng.integers(30, 150, 6), rng.integers(30, 250, 6)] = v
    live = np.isfinite(lags[:, 0])
    X = lags[live, 0][:, None, None] + tx
    Y = lags[live, 1][:, None, None] + ty
    hit = (X == np.round(X)) & (Y == np.round(Y)) & (X > 40) & (X < snx - 40) & (Y > 40) & (Y < sny - 40)
    k, gy, gx = (int(i[0]) for i in np.nonzero(hit))
    cx, cy = int(X[k, gy, gx]), int(Y[k, gy, gx])
    small[cy - 1:cy + 2, cx - 1:cx + 2] = FILL
    ref[gy, gx] = 500.0
    c.update(small=small, ref=ref, plateau=(cy, cx))
    c["claims"] = dict(staged=True, global_=False, dirty=True)
    return c


def _box_edge(dtype, axis, extra):
    """One tile, one chunk of two lags whose spread makes the (tile, chunk) window exactly as wide (axis "x") or tall
    ("y") as the box, or one pixel more; x0 = 6 + 3/64 puts the window origin 2 pixels past a 16-byte boundary, so the
    round-down of wx0 is part of the width."""
    itemsize = np.dtype(dtype).itemsize
    target = BOX[itemsize][0 if axis == "x" else 1] + extra
    ref, small = _images(3, TILE_H, TILE_W, 120 if dtype == np.float32 else 100, 300 if dtype == np.float32 else 200,
                         dtype)
    ref[:] = np.where(np.isfinite(ref), ref, 480.0)
    tx, ty = _planes(TILE_H, TILE_W, a=4.375 if dtype == np.float32 else 2.5)
    x0, y0 = 6.0 + 3 / 64, 9.0 + 5 / 64
    for k in range(64 * 120):
        s = k / 64
        lags = [[x0, y0], [x0 + s, y0]] if axis == "x" else [[x0, y0], [x0, y0 + s]]
        c = _case(ref, small, tx, ty, lags)
        p = predict(c)
        if p["width" if axis == "x" else "height"] == target:
            break
    else:
        raise AssertionError("no lag spread gives the window size asked for")
    c["claims"] = {"width" if axis == "x" else "height": target, "staged": extra == 0, "global_": extra == 1}
    return c


def _copy(dtype, snx, offset=0):
    """Row pitch not a multiple of 16 bytes (float32 widths 150 and 97, an odd float64 width) or a base address 4 bytes
    past one (a contiguous view at storage offset 1): the window is staged by the block's own copy."""
    ref, small = _images(4, 40, 36, 90, snx, dtype)
    tx, ty = _planes(40, 36, a=2.25)
    c = _case(ref, small, tx, ty, _patch_lags(-2.5, -4.0), staged=True, global_=False, tma=0)
    c["offset"] = offset
    return c


def _tiny(kind):
    """A 3 x 3 image (the smallest the window kernel takes), a 4-pixel-wide float32 image (16-byte pitch: TMA, image
    narrower than the box) and a 2-row image (generic kernel)."""
    sny, snx = dict(t3x3=(3, 3), w4=(7, 4), h2=(2, 40))[kind]
    ref, small = _images(5, 4, 5, sny, snx)
    ref[:] = np.where(np.isfinite(ref), ref, 470.0)
    if kind == "h2":
        tx, ty = _planes(4, 5, a=4.375, b=0.125, d=0.0625, e=0.25)
        xs, ys = np.arange(-2.0, 20.0, 1.0 + 3 / 64), np.arange(-0.25, 0.3, 0.125)
    else:
        tx, ty = _planes(4, 5, a=0.375, b=0.125, d=0.0625, e=0.25)
        xs, ys = np.arange(-0.5, snx - 1.5, 0.125 + 1 / 64), np.arange(-0.25, sny - 1.5, 0.125 + 1 / 64)
    lags = np.stack([g.ravel() for g in np.meshgrid(xs, ys, indexing="ij")], axis=1)
    claims = dict(window=False) if kind == "h2" else dict(staged=True, global_=False, tma=int(kind == "w4"),
                                                           rim=True, out=True)
    return _case(ref, small, tx, ty, lags, **claims)


def _global():
    """Lags 30 pixels apart: no (tile, chunk) window fits the box, every pair reads global memory."""
    ref, small = _images(6, 40, 64, 200, 300)
    tx, ty = _planes(40, 64, c=-20.0)
    i1, i2 = np.meshgrid(np.arange(5), np.arange(5), indexing="ij")
    lags = np.stack([-40.0 + 30 * i1.ravel() + 3 / 64, -20.0 + 30 * i2.ravel() + 5 / 64], axis=1)
    return _case(ref, small, tx, ty, lags, staged=False, global_=True)


def _rim(dtype):
    """Lags that put one grid pixel exactly at x = 0, n - 1, -1/64, n - 1 + 1/64, 1/64, n - 1 - 1/64, half a pixel in,
    on either axis and at the corners: samples on, just inside and just outside every edge of the image (mirrored taps
    within one pixel of an edge), and the grid around that pixel across the rim."""
    ref, small = _images(7, 24, 32, 40, 48, dtype)
    tx, ty = _planes(24, 32, a=1.25, e=1.25)
    sny, snx = small.shape
    px, py = tx[12, 16], ty[12, 16]
    ref[12, 16] = 505.0

    def edge(n):
        return [0.0, n - 1.0, -1 / 64, n - 1 + 1 / 64, 1 / 64, n - 1 - 1 / 64, 0.5, n - 1.5, 63 / 64, n - 2 + 1 / 64]

    tgt = [(x, 20.0) for x in edge(snx)] + [(24.0, y) for y in edge(sny)]
    tgt += [(x, y) for x in (0.0, -1 / 64, snx - 1.0, snx - 1 + 1 / 64) for y in (0.0, sny - 1.0, sny - 1 + 1 / 64)]
    lags = np.array([(x - px, y - py) for x, y in tgt])
    return _case(ref, small, tx, ty, lags, rim=True, out=True)


def _grid(gnx, gny):
    """Grids of 1, 33 and 100 columns by 7, 65 and 130 rows (ragged super-tiles of 32 x 64). The leftmost super-tile
    column lies left of the image under every lag but the launch's largest x0, which puts its rightmost pixels exactly
    on x = 0; it is alive only through the lag range. Where the grid has them, one super-tile has no finite reference
    value and one has NaN coordinates (behind the limb): both dead."""
    ref, small = _images(8 + gnx + gny, gny, gnx, 260, 320)
    c0 = -64.375 if gnx == 1 else -200.0
    tx, ty = _planes(gny, gnx, b=0.0, c=c0, f=5.0)
    supers = [(oy, ox) for oy in range(0, gny, SUPER_H) for ox in range(TILE_W, gnx, TILE_W)]
    if len(supers) >= 3:
        oy, ox = supers[-1]
        ref[oy:oy + SUPER_H, ox:ox + TILE_W] = np.nan
        oy, ox = supers[-2]
        tx[oy:oy + SUPER_H, ox:ox + TILE_W] = np.nan
        ty[oy:oy + SUPER_H, ox:ox + TILE_W] = np.nan
    extreme = -(tx[:, :TILE_W].max())          # the largest x0: the first column's rightmost pixels sample x = 0
    lags = np.concatenate([_patch_lags(40.0, 10.0), [[extreme, 12.0]]])
    claims = dict(alive_by_extreme_lag=True, rim=True)
    if len(supers) >= 3:
        claims["dead_super"] = True
    return _case(ref, small, tx, ty, lags, **claims)


def _chunks(n, zero_pivots=False):
    """n lags in one launch, live ones interleaved with NaN, +-inf and 2^31 offsets (dead: nothing evaluated, r NaN,
    count 0); with n = 600 the whole second chunk is dead."""
    ref, small = _images(9, 40, 64, 120, 320)
    tx, ty = _planes(40, 64, c=-10.0, f=-6.0)
    i = np.arange(n)
    lags = np.stack([3 / 64 + 0.25 * (i % 16), 5 / 64 + 0.25 * (i // 16 % 16)], axis=1)
    lags[i % 7 == 3, 0] = np.nan
    lags[i % 11 == 5, 0] = np.inf
    lags[i % 13 == 6, 1] = -np.inf
    lags[i % 17 == 8] = 2.0 ** 31
    dead = (i >= CHUNK) & (i < 2 * CHUNK) if n == 600 else np.zeros(n, bool)
    lags[dead] = np.where((i[dead] % 3 == 0)[:, None], np.nan, np.where((i[dead] % 3 == 1)[:, None], -np.inf, 2.0 ** 31))
    claims = dict(staged=True, global_=False)
    if n == 600:
        claims["dead_chunk"] = True
    c = _case(ref, small, tx, ty, lags, **claims)
    c["zero_pivots"] = zero_pivots
    return c


def _many_lag_distinct():
    """The 97 distinct offsets the 65536 * 256 + 1 lag launch cycles through (one of them NaN)."""
    k = np.arange(97)
    lags = np.stack([-2.0 + (k * 37 % 97) * (5 / 16) + 1 / 64, -1.0 + (k * 53 % 97) * (3 / 8) + 3 / 64], axis=1)
    lags[41] = np.nan
    return lags


def _many_lags():
    ref, small = _images(10, 3, 5, 40, 60)
    ref[:] = np.where(np.isfinite(ref), ref, 490.0)
    tx, ty = _planes(3, 5, a=4.375, e=1.75)
    c = _case(ref, small, tx, ty, _many_lag_distinct(), staged=True, global_=False)
    c["cycle_to"] = MANY_LAGS
    return c


CASES = {
    "staged_f32": lambda: _staged(np.float32),
    "staged_f64": lambda: _staged(np.float64),
    "dirty_f32": lambda: _dirty(np.float32),
    "dirty_f64": lambda: _dirty(np.float64),
    **{f"box_f{dt.__name__[-2:]}_{ax}_{'over' if e else 'fit'}": (lambda dt=dt, ax=ax, e=e: _box_edge(dt, ax, e))
       for dt in (np.float32, np.float64) for ax in ("x", "y") for e in (0, 1)},
    "copy_f32_w150": lambda: _copy(np.float32, 150),
    "copy_f32_w97": lambda: _copy(np.float32, 97),
    "copy_f64_w101": lambda: _copy(np.float64, 101),
    "copy_f32_base4": lambda: _copy(np.float32, 128, offset=1),
    "tiny_3x3": lambda: _tiny("t3x3"),
    "tiny_w4": lambda: _tiny("w4"),
    "tiny_h2": lambda: _tiny("h2"),
    "global": _global,
    "rim_f32": lambda: _rim(np.float32),
    "rim_f64": lambda: _rim(np.float64),
    **{f"grid_{gx}x{gy}": (lambda gx=gx, gy=gy: _grid(gx, gy)) for gx in (1, 33, 100) for gy in (7, 65, 130)},
    **{f"chunks_{n}": (lambda n=n: _chunks(n)) for n in (1, 255, 256, 257, 600)},
    "chunks_257_zero_pivots": lambda: _chunks(257, zero_pivots=True),
    "many_lags": _many_lags,
}
WINDOW_CASES = [k for k in CASES if k not in ("tiny_h2", "many_lags")]


@functools.lru_cache(maxsize=None)
def case(name):
    return CASES[name]()


@functools.lru_cache(maxsize=None)
def expected(name, order=2):
    c = case(name)
    return reference(c["ref"], c["small"], c["tx"], c["ty"], c["lags"], order)


def full_lags(c):
    """The lag table a case launches (the many-lag case cycles its distinct offsets)."""
    n = c.get("cycle_to")
    return c["lags"] if n is None else np.resize(c["lags"], (n, 2))


# =====================================================================================================================
# CPU: the cases are exact and take the paths they are built for
# =====================================================================================================================
@pytest.mark.parametrize("name", list(CASES))
def test_case_inputs_are_exact(name):
    """Dyadic lags and planes, and ((x0 + 0.5) + Tx) - 0.5 == x0 + Tx for every live (pixel, lag) pair: the kernel's
    coordinates equal the reference's bit for bit. Small-image values are float32 values. No lag has 1 or 2 pairs
    (where one-pass moments leave a residue that two-pass ones do not)."""
    c = case(name)
    lags, tx, ty = c["lags"], c["tx"], c["ty"]
    ok = (np.abs(lags[:, 0] + 0.5) < BIG) & (np.abs(lags[:, 1] + 0.5) < BIG)
    live = np.isfinite(c["ref"]) & (np.abs(tx) < BIG) & (np.abs(ty) < BIG)
    for v in (lags[ok], tx[live], ty[live]):
        assert np.array_equal(v * 64, np.round(v * 64)) and np.abs(v).max() < 2 ** 12
    for p, q in ((lags[ok, 0], tx[live]), (lags[ok, 1], ty[live])):
        assert np.array_equal(((p[:, None] + 0.5) + q[None, :]) - 0.5, p[:, None] + q[None, :])
    small = c["small"]
    assert np.array_equal(small.astype(np.float32).astype(small.dtype), small, equal_nan=True)
    _, n = expected(name)
    assert not np.any((n > 0) & (n < 3)), name
    assert n.max() > 0


@pytest.mark.parametrize("name", list(CASES))
def test_case_designs_take_the_paths_they_claim(name):
    c = case(name)
    claims = c["claims"]
    if claims.get("window") is False:
        assert not window_kernel_used(c["small"])
        return
    assert window_kernel_used(c["small"])
    c_full = dict(c, lags=full_lags(c))
    p = predict(c_full)
    for key in ("staged", "global_"):
        if key in claims:
            assert (p[key] > 0) == claims[key], (name, key, p[key])
    for key in ("width", "height", "tma"):
        if key in claims:
            assert p[key] == claims[key], (name, key, p[key])
    if claims.get("dead_super"):
        assert len(p["dead_super"]) >= 2, p["dead_super"]
    if claims.get("dead_chunk"):
        assert p["dead_chunks"] >= 1
    if claims.get("alive_by_extreme_lag"):
        assert (0, 0) in p["live_super"]
        without = predict(dict(c, lags=c["lags"][:-1]))
        assert (0, 0) in without["dead_super"]
        # under the extreme lag the first column's rightmost pixels sample x = 0 exactly
        assert (c["lags"][-1, 0] + c["tx"][:, :TILE_W]).max() == 0.0
    if claims.get("rim") or claims.get("out"):
        ok = (np.abs(c["lags"][:, 0] + 0.5) < BIG) & (np.abs(c["lags"][:, 1] + 0.5) < BIG)
        live = np.isfinite(c["ref"]) & (np.abs(c["tx"]) < BIG) & (np.abs(c["ty"]) < BIG)
        X = c["lags"][ok, 0][:, None] + c["tx"][live][None, :]
        Y = c["lags"][ok, 1][:, None] + c["ty"][live][None, :]
        sny, snx = c["small"].shape
        inside = (X >= 0) & (X <= snx - 1) & (Y >= 0) & (Y <= sny - 1)
        # the exact sampler takes the samples whose nine taps are not all inside the image
        assert not claims.get("rim") or np.any(inside & ((X < 0.5) | (X >= snx - 1.5) | (Y < 0.5) | (Y >= sny - 1.5)))
        assert not claims.get("out") or np.any(~inside)
        if name.startswith("rim_"):
            for on_edge in (X == 0, X == snx - 1, Y == 0, Y == sny - 1, (X == 0) & (Y == 0),
                            (X == snx - 1) & (Y == sny - 1)):
                assert np.any(on_edge & inside)
            assert np.any((X == -1 / 64) & (Y >= 0)) and np.any((X == snx - 1 + 1 / 64) & (Y >= 0))
    if name.startswith("box_"):
        # the window origin was rounded down to the 16-byte boundary
        x0h = c["lags"][:, 0].min() + 0.5
        assert (np.floor(c["tx"].min() + x0h) - 1) % (16 // c["small"].itemsize) != 0
    if claims.get("dirty"):
        cy, cx = c["plateau"]
        assert np.all(c["small"][cy - 1:cy + 2, cx - 1:cx + 2] == FILL)
        v = map_coordinates(c["small"].astype(np.float64), [[float(cy)], [float(cx)]], order=2, mode="constant",
                            cval=np.nan, prefilter=False)
        assert v[0] == FILL
    if name == "many_lags":
        n_chunks = -(-MANY_LAGS // CHUNK)
        assert p["cpb"] == 2 and -(-n_chunks // 2) % 2 == 1        # two chunks per block, an odd grid.y
        assert p["staged"] == n_chunks


def test_float32_and_float64_cases_decide_differently():
    """The same staged scene fits the float32 box and overflows the float64 one: the bit-for-bit comparison of the two
    instantiations crosses paths, not just types."""
    c = case("staged_f32")
    assert predict(c)["global_"] == 0
    p64 = predict(c, itemsize=8)
    assert p64["global_"] > 0


# =====================================================================================================================
# GPU
# =====================================================================================================================
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from euispice_coreg_b200 import _ext
    _ext.load()
    return torch


STATS_RE = re.compile(r"\[coreg offset kernel\] tma=(\d+) lags=(\d+) \(tile, chunk\) pairs: (\d+) staged, (\d+) global; "
                      r"(\d+) live pixel-walks .*?outside the image (\d+), exact-path (\d+); lane-tiles on a dirty "
                      r"window (\d+); largest window asked for (\d+) x (\d+)")
STATS_KEYS = ("tma", "lags", "staged", "global_", "walks", "out", "exact", "dirty", "width", "height")


def run(torch, c, lags=None, small=None, order=2, flags=0, capfd=None, no_tma=False):
    """One `coreg_offset_lag_corr` call. Returns (corr, nvalid, stats); stats (COREG_OFFSET_STATS=1) when `capfd` is
    given: None if the launch printed none (generic kernel)."""
    from euispice_coreg_b200 import _ext
    dev = torch.device("cuda", torch.cuda.current_device())
    lags = c["lags"] if lags is None else lags
    small = c["small"] if small is None else small
    gny, gnx = c["ref"].shape
    n = len(lags)
    ref_d, tx_d, ty_d = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (c["ref"], c["tx"], c["ty"]))
    off = c.get("offset", 0)
    buf = torch.empty(small.size + off, dtype=torch.float32 if small.itemsize == 4 else torch.float64, device=dev)
    small_d = buf[off:].view(small.shape)      # off = 1: a contiguous view whose base is not 16-byte aligned
    small_d.copy_(torch.from_numpy(np.ascontiguousarray(small)))
    assert (small_d.data_ptr() % 16 != 0) == (off != 0)
    if c.get("zero_pivots"):
        piv = [0.0, 0.0]
    else:
        # correctly rounded means: the same pivots for a float32 image and its float64 copy (numpy's pairwise sums
        # group a float32 array differently)
        piv = [math.fsum(v) / v.size for v in (c["ref"][np.isfinite(c["ref"])],
                                               small[np.isfinite(small)].astype(np.float64))]
    pivots = torch.tensor(piv, dtype=torch.float64, device=dev)
    nbytes = _ext.lag_corr_workspace_bytes(gnx, gny, n, offset_window=window_kernel_used(small, order, flags))
    work = torch.full((nbytes,), 255, dtype=torch.uint8, device=dev)    # partials never written read as NaN
    lags_d = torch.from_numpy(np.ascontiguousarray(lags, dtype=np.float64)).to(dev)
    corr = torch.full((n,), 7.0, dtype=torch.float64, device=dev)
    nvalid = torch.full((n,), -1, dtype=torch.int64, device=dev)
    env = {"COREG_OFFSET_STATS": "1" if capfd is not None else None, "COREG_NO_TMA": "1" if no_tma else None}
    saved = {k: os.environ.get(k) for k in env}
    if capfd is not None:
        capfd.readouterr()
    try:
        for k, v in env.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        _ext.offset_lag_corr(ref_d, small_d, tx_d, ty_d, lags_d, order, pivots, work, corr, nvalid, flags)
        torch.cuda.synchronize()
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    stats = None
    if capfd is not None:
        found = STATS_RE.findall(capfd.readouterr().err)
        assert len(found) <= 1
        stats = dict(zip(STATS_KEYS, map(int, found[0]))) if found else None
    return corr.cpu().numpy(), nvalid.cpu().numpy(), stats


def assert_matches(corr, nvalid, want, what):
    r_ref, n_ref = want
    bad = np.flatnonzero(nvalid != n_ref)
    assert bad.size == 0, f"{what}: nvalid differs at {bad.size} lags, lag {bad[0]}: {nvalid[bad[0]]} != {n_ref[bad[0]]}"
    assert np.array_equal(np.isnan(corr), np.isnan(r_ref)), f"{what}: NaN pattern differs"
    fin = ~np.isnan(r_ref)
    err = float(np.max(np.abs(corr[fin] - r_ref[fin]))) if fin.any() else 0.0
    assert err <= R_TOL, f"{what}: max |dr| = {err:.3e}"


def assert_same_bits(a, b, what):
    """(corr, nvalid) pairs equal bit for bit (NaN in the same places)."""
    ra, rb = np.asarray(a[0]), np.asarray(b[0])
    assert np.array_equal(np.isnan(ra), np.isnan(rb)), f"{what}: NaN pattern differs"
    fin = ~np.isnan(ra)
    assert np.array_equal(ra[fin].view(np.int64), rb[fin].view(np.int64)), f"{what}: r differs"
    assert np.array_equal(a[1], b[1]), f"{what}: nvalid differs"


@pytest.mark.gpu
@pytest.mark.parametrize("name", WINDOW_CASES)
def test_window_kernel_matches_reference(torch_cuda, capfd, name):
    c = case(name)
    corr, nvalid, st = run(torch_cuda, c, capfd=capfd)
    assert_matches(corr, nvalid, expected(name), name)
    p = predict(c)
    assert st is not None, "the window kernel printed no statistics"
    for key in ("tma", "staged", "global_", "walks", "width", "height"):
        assert st[key] == p[key], (name, key, st[key], p[key])
    claims = c["claims"]
    if claims.get("dirty"):
        assert st["dirty"] > 0
    if claims.get("clean"):
        assert st["dirty"] == 0
    # samples the window walk sends to the exact sampler (image rim) or drops as outside the image; the global walk
    # does not count them
    if claims.get("rim"):
        assert st["exact"] > 0, st
    if claims.get("out"):
        assert st["out"] > 0, st


@pytest.mark.gpu
def test_generic_kernel_for_two_row_images(torch_cuda, capfd):
    c = case("tiny_h2")
    corr, nvalid, st = run(torch_cuda, c, capfd=capfd)
    assert st is None
    assert_matches(corr, nvalid, expected("tiny_h2"), "tiny_h2")


@pytest.mark.gpu
def test_two_chunks_per_block(torch_cuda, capfd):
    """65536 * 256 + 1 lags: more chunks than grid.y may hold, so each block walks two chunks and the last block one.
    97 distinct offsets cycle through the list: every copy of an offset gives the reference's r and count, with the
    same bits wherever it sits in its chunk."""
    torch = torch_cuda
    c = case("many_lags")
    lags = full_lags(c)
    corr, nvalid, st = run(torch, c, lags=lags, capfd=capfd)
    p = predict(dict(c, lags=lags))
    for key in ("staged", "global_", "walks", "width", "height"):
        assert st[key] == p[key], (key, st[key], p[key])
    k = len(c["lags"])
    assert_matches(corr[:k], nvalid[:k], expected("many_lags"), "many_lags")
    idx = np.arange(len(lags)) % k
    assert np.array_equal(nvalid, nvalid[:k][idx])
    assert np.array_equal(np.isnan(corr), np.isnan(corr[:k][idx]))
    fin = ~np.isnan(corr)
    assert np.array_equal(corr[fin].view(np.int64), corr[:k][idx][fin].view(np.int64))


GENERIC = [(0, 0), (1, 0), (3, 0), (2, FLAG_STRICT), (2, FLAG_NO_FAST)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rim_f32", "dirty_f32", "chunks_257"])
@pytest.mark.parametrize("order,flags", GENERIC, ids=["order0", "order1", "order3", "strict", "no_fast"])
def test_generic_kernel_matches_reference(torch_cuda, name, order, flags):
    c = case(name)
    corr, nvalid, _ = run(torch_cuda, c, order=order, flags=flags)
    assert_matches(corr, nvalid, expected(name, order), f"{name} order {order} flags {flags}")
    if order == 2:
        _, nv_window, _ = run(torch_cuda, c)
        assert np.array_equal(nvalid, nv_window)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dirty_f32", "rim_f32", "grid_100x130"])
def test_lag_bits_do_not_depend_on_the_launch(torch_cuda, name):
    """A lag's (r, nvalid) are the same bits alone, in patch order, shuffled, in separate calls split at non-multiples
    of 256, and with NaN dummies between the lags."""
    torch = torch_cuda
    c = case(name)
    lags = c["lags"]
    base = run(torch, c)
    live = np.flatnonzero(np.isfinite(lags[:, 0]))
    rng = np.random.default_rng(11)
    for k in rng.choice(live, size=min(12, live.size), replace=False):
        one = run(torch, c, lags=lags[k:k + 1])
        assert_same_bits((one[0], one[1]), (base[0][k:k + 1], base[1][k:k + 1]), f"lag {k} alone")
    perm = rng.permutation(len(lags))
    sh = run(torch, c, lags=lags[perm])
    assert_same_bits((sh[0], sh[1]), (base[0][perm], base[1][perm]), "shuffled")
    cuts = [0, 100, 357, len(lags)] if len(lags) > 357 else [0, len(lags) // 3, len(lags)]
    parts = [run(torch, c, lags=lags[perm][a:b]) for a, b in zip(cuts[:-1], cuts[1:]) if b > a]
    split = (np.concatenate([q[0] for q in parts]), np.concatenate([q[1] for q in parts]))
    assert_same_bits(split, (base[0][perm], base[1][perm]), "split calls")
    padded = np.full((2 * len(lags), 2), np.nan)
    padded[1::2] = lags
    pad = run(torch, c, lags=padded)
    assert_same_bits((pad[0][1::2], pad[1][1::2]), (base[0], base[1]), "NaN dummies between")
    assert np.all(pad[1][0::2] == 0) and np.all(np.isnan(pad[0][0::2]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["staged_f32", "dirty_f32", "rim_f32", "box_f32_x_fit", "copy_f32_w97"])
def test_float32_and_float64_small_images_give_the_same_bits(torch_cuda, capfd, name):
    c = case(name)
    a = run(torch_cuda, c, capfd=capfd)
    b = run(torch_cuda, c, small=c["small"].astype(np.float64), capfd=capfd)
    assert_same_bits(a, b, name)
    assert a[2]["global_"] == predict(c)["global_"] and b[2]["global_"] == predict(c, itemsize=8)["global_"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["staged_f32", "dirty_f32", "dirty_f64", "rim_f32", "grid_100x130"])
def test_tma_and_cooperative_copy_give_the_same_bits(torch_cuda, capfd, name):
    c = case(name)
    a = run(torch_cuda, c, capfd=capfd)
    b = run(torch_cuda, c, capfd=capfd, no_tma=True)
    assert a[2]["tma"] == 1 and b[2]["tma"] == 0
    assert a[2]["staged"] == b[2]["staged"] > 0
    assert_same_bits(a, b, name)
