"""Cost of the per-block shift maps (`LocalAlignmentResults.shift_arcsec`) against the host loop over `results(i, j)`.

Three numbers, with the card's name and power limit read in the same run:
- device: 16 384 fits (256 frames x 8 x 8 blocks) of seeded Gaussian peaks on a 60 x 60 lag grid, one `coreg_gauss2d_fit`
  launch, timed with CUDA events after a warm-up (best and median of --reps launches);
- sequence: a `SequenceAlignment.align_using_helioprojective(local_block=64)` run over 256 frames of 512^2 pixels (8 x 8
  blocks, 60 x 60 CRVAL lags), then the wall time of `.shift_arcsec` on every frame's `.local` (one launch per frame,
  host gathering and D2H included);
- host: the loop over `results(i, j).shift_arcsec` for the first 512 of those blocks, and its time per fit.
Prints one JSON line and writes it to --out when given.

    python tools/shift_map_bench.py --out /tmp/shift_map_bench.json
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import tempfile
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

LAGS = dict(lag_crval1=np.arange(-6.0, 54.0, 1.0), lag_crval2=np.arange(-24.0, 36.0, 1.0))


def random_peaks(n, seed=1):
    rng = np.random.default_rng(seed)
    X, Y = np.meshgrid(np.arange(60.0), np.arange(60.0), indexing="ij")
    cubes = np.empty((n, 60, 60))
    for k in range(n):
        cx, cy = rng.uniform(27, 33, 2)
        sx, sy = rng.uniform(1, 6, 2)
        cubes[k] = 0.4 + 0.5 * np.exp(-((X - cx) ** 2 / (2 * sx ** 2) + (Y - cy) ** 2 / (2 * sy ** 2))) \
            + rng.normal(0, rng.uniform(0, 0.02), X.shape)
    return cubes.reshape(n, 60, 60, 1, 1, 1, 1)


def device_fits(n, reps):
    import torch
    from euispice_coreg_b200 import _ext
    AR = importlib.import_module("euispice_coreg_b200.hdrshift.AlignmentResults")
    cubes = random_peaks(n)
    mi = np.array([np.unravel_index(np.argmax(c), c.shape) for c in cubes])
    prob = AR.gaussian_fit_problems(cubes, mi)
    dev = torch.device("cuda", 0)
    args = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (prob.points, prob.npts, prob.p0, prob.bounds)]
    for _ in range(3):
        _ext.gauss2d_fit(*args)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _, _, iters, status = _ext.gauss2d_fit(*args)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    status, iters = status.cpu().numpy(), iters.cpu().numpy()
    return {"problems": n, "best_ms": min(ms), "median_ms": float(np.median(ms)),
            "converged": int((status == _ext.FIT_CONVERGED).sum()), "iterations_max": int(iters.max()),
            "iterations_mean": float(iters.mean())}


def sequence_run(n_frames, host_blocks):
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200._synth.scene import make_pair, small_spec
    from euispice_coreg_b200.hdrshift import SequenceAlignment
    d = tempfile.mkdtemp(prefix="shift_map_bench_")
    p_large, p_small, _ = make_pair(d, small_spec(512, 800, true_crval=(-12.0, 8.0)), tag="seq")
    h = fits_lite.open(p_small)[0]
    rng = np.random.default_rng(7)
    frames = []
    for k in range(n_frames):      # the same image under jittered pointing keywords
        hdr = h.header.copy()
        hdr["CRVAL1"] = float(hdr["CRVAL1"]) + rng.uniform(-3, 3)
        hdr["CRVAL2"] = float(hdr["CRVAL2"]) + rng.uniform(-3, 3)
        p = os.path.join(d, f"frame_{k:03d}.fits")
        fits_lite.writeto(p, [fits_lite.PrimaryHDU(np.array(h.data), hdr)], overwrite=True)
        frames.append(p)
    seq = SequenceAlignment(p_large, frames, **LAGS)
    t0 = time.perf_counter()
    out = seq.align_using_helioprojective(local_block=64)
    t_search = time.perf_counter() - t0
    assert out[0].local.corr.shape[:2] == (8, 8)
    t0 = time.perf_counter()
    maps = [r.local.shift_arcsec for r in out]
    t_maps = time.perf_counter() - t0
    status = np.stack([r.local.fit_status for r in out])
    blocks = [(f, i, j) for f in range(len(out)) for i in range(8) for j in range(8)][:host_blocks]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        host = [out[f].local.results(i, j).shift_arcsec for f, i, j in blocks]
        t_host = time.perf_counter() - t0
    dev = np.array([maps[f][i, j] for f, i, j in blocks])
    fitted = np.array([status[f, i, j] == 0 for f, i, j in blocks])
    diff = np.abs(dev[fitted, :2] - np.array(host, dtype=np.float64)[fitted, :2])
    return {"frames": n_frames, "blocks": int(status.size), "search_s": t_search, "shift_arcsec_all_frames_s": t_maps,
            "status_counts": np.bincount(status.ravel(), minlength=4).tolist(), "host_blocks": len(blocks),
            "host_loop_s": t_host, "host_ms_per_fit": 1e3 * t_host / len(blocks),
            "max_crval_diff_vs_host_arcsec": float(diff.max()) if diff.size else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--problems", type=int, default=256 * 64)
    ap.add_argument("--host-blocks", type=int, default=512)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("shift_map_bench needs a CUDA device")
    from local_blocks_bench import card
    res = {"card": card(), "device_fits": device_fits(a.problems, a.reps),
           "sequence": sequence_run(a.frames, a.host_blocks)}
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
