"""Cost of the per-block correlation cubes (`Alignment(..., local_block=...)`) on the config-1 pair.

Times the helioprojective search of BASELINE configs[0] (2048^2 HRIEUV-like vs 3072^2 FSI-like, the 60 x 60 = 3600-lag
CRVAL grid bench.py uses) with no blocks, 256-pixel blocks (8 x 8) and 128-pixel blocks (16 x 16), alternating the three
in every round after a warm-up of each. Per arm: the best and median wall time of `align_using_helioprojective`
(return_type="corr": file reads, uploads, one-time cut, search, D2H), the summed device time of the lag-kernel launches
(`coreg_profile_begin` / `end`: the fused kernel only, not the finalizes), and the digest of the global cube, which must
be the same in all three arms. The card's name and power limit are read in the same run. Prints one JSON line and writes
it to --out when given.

    python tools/local_blocks_bench.py --rounds 5 --out /tmp/local_blocks_bench.json
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LAGS = dict(lag_crval1=np.arange(-30, 30, 1.0), lag_crval2=np.arange(-30, 30, 1.0), lag_cdelt1=np.array([0.0]),
            lag_cdelt2=np.array([0.0]), lag_crota=np.array([0.0]))
ARMS = {"none": None, "256": 256, "128": 128}


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["max_sm_mhz"] = float(q[0]), float(q[1])
    except Exception as exc:      # the timing stands without it; say so
        out["power_limit_w"] = f"unavailable: {exc}"
    return out


def _refs(a):
    """The reference header values `Alignment._find_best_header_parameters` hands to the lag tables."""
    from euispice_coreg_b200.hdrshift.alignment import _Refs
    r = _Refs()
    r.crval1_ref, r.crval2_ref, r.crota_ref = a.crval1_ref, a.crval2_ref, a.crota_ref
    r.cdelt1_ref, r.cdelt2_ref = a.cdelt1_ref, a.cdelt2_ref
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._synth.scene import make_config1
    from euispice_coreg_b200.hdrshift import Alignment
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the B200 path only")
    torch.cuda.set_device(0)
    tmp = tempfile.mkdtemp(prefix="local_blocks_bench_")
    p_large, p_small, _ = make_config1(tmp)

    def run(block):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            a = Alignment(p_large, p_small, parallelism=True, local_block=block, **LAGS)
            torch.cuda.synchronize()
            _ext.profile_begin()
            t0 = time.perf_counter()
            cube = a.align_using_helioprojective(return_type="corr")
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            dev_ms, launches = _ext.profile_end()
        digest = hashlib.sha256(np.ascontiguousarray(cube).tobytes()).hexdigest()
        shape = None if a.local is None else list(a.local.corr.shape[:2])
        return wall * 1e3, dev_ms, launches, digest, shape

    # the device search alone: one engine prepared once, CUDA events around `evaluate` (lag kernel + finalize + the
    # per-block finalize), 10 searches per sample
    a0 = Alignment(p_large, p_small, parallelism=True, **LAGS)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a0.align_using_helioprojective(return_type="corr")
    eng = a0.engine
    from euispice_coreg_b200.hdrshift import engine as E
    from euispice_coreg_b200._compat.wcs import TanWcs
    d = E.flat_lag_grid(*(LAGS[k] for k in ("lag_crval1", "lag_crval2", "lag_cdelt1", "lag_cdelt2", "lag_crota")))
    w = TanWcs.from_header(a0.hdr_small)
    table, _ = E.tan_wcs_table(a0.hdr_small, _refs(a0), *d)
    eng.pure_shift_hint = True
    tab = eng._upload(table)
    n = table.shape[0]
    out = torch.empty(n, dtype=torch.float64, device=eng.device)
    nv = torch.empty(n, dtype=torch.int64, device=eng.device)
    regions = {}
    for name, block in ARMS.items():
        if block is not None:
            nby, nbx = _ext.region_grid(w.naxis2, w.naxis1, block, block)
            regions[name] = (block, block, torch.empty((nby * nbx, n), dtype=torch.float64, device=eng.device),
                             torch.empty((nby * nbx, n), dtype=torch.int64, device=eng.device))

    def device_search(name, reps=10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            eng.evaluate(tab, out, nv, regions=regions.get(name))
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    for name, block in ARMS.items():
        for _ in range(args.warmup):
            run(block)
            device_search(name, 2)
    samples = {name: [] for name in ARMS}
    dev_samples = {name: [] for name in ARMS}
    for _ in range(args.rounds):
        for name, block in ARMS.items():
            samples[name].append(run(block))
            dev_samples[name].append(device_search(name))
    res = {"workload": "config-1 pair, 3600 CRVAL lags, align_using_helioprojective(return_type='corr')",
           "card": card(), "rounds": args.rounds, "arms": {}}
    base = min(s[0] for s in samples["none"])
    dev_base = min(dev_samples["none"])
    for name, s in samples.items():
        wall = [x[0] for x in s]
        dev = [x[1] for x in s]
        res["arms"][name] = {"blocks": s[0][4], "wall_ms_best": min(wall), "wall_ms_median": float(np.median(wall)),
                             "lag_kernel_ms_best": min(dev), "lag_kernel_launches": s[0][2],
                             "device_search_ms_best": min(dev_samples[name]),
                             "device_search_ms_median": float(np.median(dev_samples[name])),
                             "wall_overhead_vs_none_pct": 100.0 * (min(wall) / base - 1.0),
                             "device_overhead_vs_none_pct": 100.0 * (min(dev_samples[name]) / dev_base - 1.0),
                             "cube_sha256": sorted({x[3] for x in s})}
    digests = {d for a in res["arms"].values() for d in a["cube_sha256"]}
    res["global_digests_equal"] = len(digests) == 1
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
