"""Carrington-frame frame sequences on one GPU: single-pair `Alignment.align_using_carrington` in a loop against
`SequenceAlignment.align_using_carrington`, for both reprojection methods, and the wall time per frame of
`jitter_correction_imagers` (batched) against the same chain built from per-frame `Alignment` calls.

Inputs: the configs[4] frames (`bench.ensure_sequence`: HRIEUV-like 2048^2 renderings with pointing jitter) against the
configs[1] FSI-like 3072^2 reference, on the configs[1] Carrington grid (`bench.CARRINGTON_GRID`), with the configs[1]
lags (`bench.CARRINGTON_LAGS`, 120 x 120 at 1") and a jitter-correction-sized grid (100 x 100 at 0.1"). Every timed
section ends in a device synchronise; both paths are warmed up, run in the same process and alternated. Every cube of
both paths goes into a SHA-256 digest per path: the digests must be equal. Prints one JSON line (and writes it to
--out when given). The "sunpy" inputs are copies of the files with Stonyhurst observer keywords, written to a temporary
directory."""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402

JITTER_LAGS = dict(lag_crval1=np.arange(-5, 5, 0.1), lag_crval2=np.arange(-5, 5, 0.1), lag_cdelt1=np.array([0.0]),
                   lag_cdelt2=np.array([0.0]), lag_crota=np.array([0.0]))
LAG_GRIDS = {"configs1_120x120_1arcsec": bench.CARRINGTON_LAGS, "jitter_100x100_0.1arcsec": JITTER_LAGS}


def gpu_identity(torch):
    out = {"torch_device_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=60)
        out["nvidia_smi"] = q.stdout.strip() or q.stderr.strip()
    except Exception as exc:       # the query is informative only; the numbers stand with the device name
        out["nvidia_smi"] = f"unavailable: {exc}"
    return out


def with_observer(path, obs, out):
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


def digest(cubes):
    h = hashlib.sha256()
    for c in cubes:
        h.update(np.ascontiguousarray(c, dtype=np.float64).tobytes())
    return h.hexdigest()


def compare_paths(torch, pl, frames, lags, method, rounds):
    """Frames/s of a loop of single-pair searches and of one sequence call over the same frames, alternated."""
    from euispice_coreg_b200.hdrshift import Alignment, SequenceAlignment
    grid = bench.CARRINGTON_GRID

    def single():
        return [Alignment(pl, p, parallelism=True, **lags).align_using_carrington(
            method="correlation", method_carrington_reprojection=method, return_type="corr", **grid) for p in frames]

    def sequence():
        seq = sequence.last = SequenceAlignment(pl, frames, **lags)
        return seq.align_using_carrington(method_carrington_reprojection=method, return_type="corr", **grid)

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cubes = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, cubes

    Alignment(pl, frames[0], parallelism=True, **lags).align_using_carrington(      # warm-up of every shape
        method_carrington_reprojection=method, return_type="corr", **grid)
    SequenceAlignment(pl, frames[:2], **lags).align_using_carrington(
        method_carrington_reprojection=method, return_type="corr", **grid)
    walls = {"single_pair_loop": [], "sequence": []}
    digests = {}
    for r in range(rounds):
        order = [("single_pair_loop", single), ("sequence", sequence)]
        for name, fn in (order if r % 2 == 0 else order[::-1]):
            dt, cubes = timed(fn)
            walls[name].append(dt)
            digests.setdefault(name, digest(cubes))
    n = len(frames)
    res = {name: {"frames_per_s_best": n / min(w), "frames_per_s_each_round": [n / x for x in w],
                  "wall_s_each_round": w} for name, w in walls.items()}
    res["sequence"]["frames_per_s_inner_loop_last_round"] = sequence.last.frames_per_s
    res["speedup_best"] = min(walls["single_pair_loop"]) / min(walls["sequence"])
    res["digests"] = digests
    res["digests_equal"] = digests["single_pair_loop"] == digests["sequence"]
    return res


def jitter_correction(torch, frame_files, tmp, lags, rounds):
    """Wall per frame of `jitter_correction_imagers` (sublist_length 10, Carrington "fa" on the configs[1] grid) and of
    the same chain as per-frame `Alignment` calls + `write_corrected_fits`; output files compared byte for byte."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.hdrshift import Alignment
    from euispice_coreg_b200.jitter_correction.jitter_correction import jitter_correction_imagers
    grid = bench.CARRINGTON_GRID
    sub = 10
    n = len(frame_files)

    def batched(out):
        jitter_correction_imagers(frame_files, out, sublist_length=sub, overlap=1, alignement_method="carrington",
                                  **lags, **grid)

    def per_frame(out):
        dates = [fits_lite.open(p)[0].header["DATE-AVG"] for p in frame_files]
        idx = list(range(n))
        shutil.copyfile(frame_files[0], os.path.join(out, os.path.basename(frame_files[0])))
        for s in (idx[k:k + sub + 1] for k in range(0, n, sub)):
            ref = os.path.join(out, os.path.basename(frame_files[s[0]]))
            for i in s[1:]:
                r = Alignment(ref, frame_files[i], parallelism=True, **lags).align_using_carrington(
                    method="correlation", reference_date=dates[s[0]], **grid)
                r.write_corrected_fits(window_list_to_apply_shift=[-1],
                                       path_to_l3_output=os.path.join(out, os.path.basename(frame_files[i])))

    walls = {"batched": [], "per_frame_alignment": []}
    outs = {}
    for r in range(rounds + 1):                  # round 0: warm-up
        order = [("batched", batched), ("per_frame_alignment", per_frame)]
        for name, fn in (order if r % 2 == 0 else order[::-1]):
            out = os.path.join(tmp, f"jc_{name}_{r}")
            os.makedirs(out)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(out)
            torch.cuda.synchronize()
            if r:
                walls[name].append(time.perf_counter() - t0)
            outs[name] = out
    searched = n - 1                            # every frame after the first is searched once
    names = sorted(os.listdir(outs["batched"]))
    same = names == sorted(os.listdir(outs["per_frame_alignment"])) and all(
        open(os.path.join(outs["batched"], f), "rb").read() == open(os.path.join(outs["per_frame_alignment"], f),
                                                                    "rb").read() for f in names)
    return {"frames": n, "frames_searched": searched, "sublist_length": sub,
            **{f"{k}_wall_per_frame_s_best": min(w) / searched for k, w in walls.items()},
            **{f"{k}_wall_s_each_round": w for k, w in walls.items()},
            "files_byte_identical": bool(same), "files": len(names)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--frames", type=int, default=8, help="frames per sequence (distinct jittered files)")
    ap.add_argument("--sunpy-frames", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--jitter-frames", type=int, default=11, help="files of the jitter-correction run")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    pl, _ = bench.ensure_config1()
    frames = bench.ensure_sequence(args.frames)
    res = {"gpu": gpu_identity(torch), "grid": {k: list(v) if isinstance(v, tuple) else v
                                                for k, v in bench.CARRINGTON_GRID.items()}}
    with tempfile.TemporaryDirectory(prefix="carr_seq_bench_") as tmp:
        for lag_name, lags in LAG_GRIDS.items():
            res[f"fa_{lag_name}"] = compare_paths(torch, pl, frames, lags, "fa", args.rounds)
        # "sunpy": the reference seen by a second spacecraft 0.3 deg away, closer to the Sun, half an hour later
        obs_large = with_observer(pl, (10.3, -2.9, 5.5e10, "2022-03-17T10:20:45.000"),
                                  os.path.join(tmp, "obs_large.fits"))
        obs_frames = [with_observer(p, (10.0, -3.0, None, None), os.path.join(tmp, f"obs_{i}.fits"))
                      for i, p in enumerate(frames[:args.sunpy_frames])]
        for lag_name, lags in LAG_GRIDS.items():
            res[f"sunpy_{lag_name}"] = compare_paths(torch, obs_large, obs_frames, lags, "sunpy", args.rounds)
        # jitter correction: distinct file names (the output of a frame is named after its input)
        jc_dir = os.path.join(tmp, "jc_in")
        os.makedirs(jc_dir)
        jc_files = []
        for i in range(args.jitter_frames):
            p = os.path.join(jc_dir, f"hrieuv_{i:03d}.fits")
            shutil.copyfile(frames[i % len(frames)], p)
            jc_files.append(p)
        res["jitter_correction_fa_jitter_100x100_0.1arcsec"] = jitter_correction(torch, jc_files, tmp, JITTER_LAGS,
                                                                                 args.rounds)
    res["all_digests_equal"] = all(v["digests_equal"] for k, v in res.items() if isinstance(v, dict)
                                   and "digests_equal" in v)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
