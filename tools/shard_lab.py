"""Per-shard cost of the config-1 search: K1 time of each of the G contiguous lag slices on one GPU (GPU box).
    python tools/shard_lab.py --shards 8
Tells a load imbalance between ranks (slices differ) from a per-launch overhead (all slices above total / G)."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import bench
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._compat.wcs import TanWcs
    from euispice_coreg_b200.hdrshift import engine as E
    from euispice_coreg_b200.hdrshift.alignment import Alignment
    ap = argparse.ArgumentParser()
    ap.add_argument("--shards", type=int, default=8)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--interleave", action="store_true", help="round-robin slices instead of contiguous ones")
    args = ap.parse_args()
    pl, ps = bench.ensure_config1()
    a = Alignment(pl, ps, parallelism=True, **bench.LAGS)
    a.method, a.coordinate_frame = "correlation", "final_helioprojective"
    a._load_pair()
    a._set_initial_header_values(True)
    w_small, w_large = TanWcs.from_header(a.hdr_small), TanWcs.from_header(a.hdr_large)
    d = E.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
    eng = E.LagSearchEngine(order=2)
    eng.set_small(a.data_small)
    eng.prepare_hpc(a.data_large, w_large, w_small)
    table, _ = eng.hpc_lag_table(a.hdr_small, a, *d)
    n = table.shape[0]
    chunk, bounds = E.shard_bounds(n, args.shards)
    out = []
    for r in range(-1, args.shards):
        if r < 0:
            sel = np.arange(n)
        elif args.interleave:
            sel = np.arange(r, n, args.shards)
        else:
            sel = np.arange(*bounds[r])
        tab = eng._upload(table[sel])
        res = torch.empty(len(sel), dtype=torch.float64, device=eng.device)
        eng.evaluate(tab, res)
        torch.cuda.synchronize()
        _ext.profile_begin()
        for _ in range(args.steps):
            eng.evaluate(tab, res)
        ms, k = _ext.profile_end()
        out.append({"shard": r, "lags": int(len(sel)), "k1_ms": ms / args.steps, "us_per_lag": 1e3 * ms / args.steps / len(sel)})
        print(json.dumps(out[-1]), flush=True)
    print(json.dumps({"interleave": args.interleave,
                      "max_shard_ms": max(o["k1_ms"] for o in out[1:]), "mean_shard_ms": float(np.mean([o["k1_ms"] for o in out[1:]])),
                      "whole_over_G_ms": out[0]["k1_ms"] / args.shards}))


if __name__ == "__main__":
    main()
