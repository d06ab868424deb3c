"""Cost of the per-block correlation cubes of the Carrington "fa" search (`align_using_carrington(local_block=...)`).

Workload: the BASELINE configs[1] pair and grid (the config-1 2048^2 HRIEUV-like vs 3072^2 FSI-like pair on the 2048^2
Carrington grid lon 200-300 deg, lat +-20 deg, 120 x 120 = 14 400 CRVAL lags at 1", as bench.py runs it). Arms: no
blocks, 256-pixel blocks (8 x 8) and 128-pixel blocks (16 x 16), alternated in every round after a warm-up of each.
Per arm:
  * device search: the resident engine of one `align_using_carrington` call, the padded patch-ordered lag table on the
    device, CUDA events around `evaluate` (window kernel + whole-grid fold + the per-block fold), --reps searches per
    sample;
  * whole call: wall time of `align_using_carrington(return_type="corr", local_block=...)` ending in a device
    synchronise (file reads, projection of the large image, planes, search, D2H and the host-side reshaping);
  * the SHA-256 of the global cube, which must be the same in all three arms.
The card's name and power limit are read in the same run. Prints one JSON line and writes it to --out when given.

    python tools/carrington_local_blocks_bench.py --rounds 3 --out /tmp/carrington_local_blocks_bench.json
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import tempfile
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench  # noqa: E402
from tools.local_blocks_bench import card  # noqa: E402

ARMS = {"none": None, "256": 256, "128": 128}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._synth.scene import make_config1
    from euispice_coreg_b200.hdrshift import Alignment
    from euispice_coreg_b200.hdrshift import engine as E
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the B200 path only")
    torch.cuda.set_device(0)
    warnings.simplefilter("ignore")
    tmp = tempfile.mkdtemp(prefix="carrington_local_blocks_bench_")
    p_large, p_small, _ = make_config1(tmp)
    grid, lags = bench.CARRINGTON_GRID, bench.CARRINGTON_LAGS

    def call(block):
        a = Alignment(p_large, p_small, parallelism=True, **lags)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cube = a.align_using_carrington(return_type="corr", local_block=block, **grid)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        digest = hashlib.sha256(np.ascontiguousarray(cube).tobytes()).hexdigest()
        return wall * 1e3, digest, None if a.local is None else list(a.local.corr.shape[:2]), a

    # the device search: the engine one call left resident, its one CROTA group's table in the kernel's lag order
    a0 = call(None)[3]
    eng = a0.engine
    d1, d2, _, _, _ = E.flat_lag_grid(a0.lag_crval1, a0.lag_crval2, a0.lag_cdelt1, a0.lag_cdelt2, a0.lag_crota)
    planes = eng.carrington_planes(a0.hdr_small, float(a0.lag_solar_r[0]), a0.lonlims, a0.latlims, a0.shape)
    roll = a0.hdr_small["CROTA"] if "CROTA" in a0.hdr_small else a0.hdr_small["CROTA2"]
    x0, y0 = eng.carrington_offset(a0.hdr_small, a0.crval1_ref + d1, a0.crval2_ref + d2, roll)
    i1, i2 = np.unravel_index(np.arange(d1.size), (len(a0.lag_crval1), len(a0.lag_crval2)))
    slot, n_slots = E.offset_patch_order(i1, i2)
    padded = np.full((n_slots, 2), np.nan)
    padded[slot] = np.stack([x0, y0], axis=1)
    tab = eng._upload(padded)
    out = torch.empty(n_slots, dtype=torch.float64, device=eng.device)
    nv = torch.empty(n_slots, dtype=torch.int64, device=eng.device)
    gny, gnx = eng.ref.shape
    regions = {}
    for name, block in ARMS.items():
        if block is not None:
            nb = int(np.prod(_ext.region_grid(gny, gnx, block, block)))
            regions[name] = (block, block, torch.empty((nb, n_slots), dtype=torch.float64, device=eng.device),
                             torch.empty((nb, n_slots), dtype=torch.int64, device=eng.device))

    def device_search(name, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            eng.evaluate(tab, out, nv, planes, regions=regions.get(name))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    for name, block in ARMS.items():
        for _ in range(args.warmup):
            call(block)
            device_search(name, 2)
    walls = {name: [] for name in ARMS}
    devs = {name: [] for name in ARMS}
    digests = {name: set() for name in ARMS}
    shapes = {}
    for _ in range(args.rounds):
        for name, block in ARMS.items():
            wall, digest, shape, _ = call(block)
            walls[name].append(wall)
            digests[name].add(digest)
            shapes[name] = shape
            devs[name].append(device_search(name, args.reps))
    res = {"workload": "configs[1]: config-1 pair on the Carrington grid 2048x2048 (lon 200-300 deg, lat +-20 deg), "
                       "120x120 CRVAL lags @1arcsec, align_using_carrington(return_type='corr')",
           "card": card(), "rounds": args.rounds, "reps": args.reps, "lags": int(d1.size), "padded_lags": int(n_slots),
           "arms": {}}
    dev0, wall0 = min(devs["none"]), min(walls["none"])
    for name in ARMS:
        nb = 0 if shapes[name] is None else int(np.prod(shapes[name]))
        res["arms"][name] = {"blocks": shapes[name], "block_output_mb": nb * int(d1.size) * 16 / 1e6,
                             "device_search_ms_best": min(devs[name]),
                             "device_search_ms_median": float(np.median(devs[name])),
                             "device_overhead_vs_none_ms": min(devs[name]) - dev0,
                             "wall_ms_best": min(walls[name]), "wall_ms_median": float(np.median(walls[name])),
                             "wall_overhead_vs_none_ms": min(walls[name]) - wall0,
                             "cube_sha256": sorted(digests[name])}
    res["global_digests_equal"] = len(set().union(*digests.values())) == 1
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not res["global_digests_equal"]:
        raise SystemExit("global cube digests differ between arms")


if __name__ == "__main__":
    main()
