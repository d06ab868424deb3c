"""A/B of the FP64 and the mixed-arithmetic rolling kernel on config 1 and on a rotated / rescaled lag set (GPU box).
    python tools/mixed_lab.py [--out gpurun_out/mixed_lab.json]
"""
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
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default="gpurun_out/mixed_lab.json")
    ap.add_argument("--combos", default="fp64:0,mixed:0,mixed:1",
                    help="arithmetic:variant pairs; variant 0 = flavour from the lag grid, 1 = pure-shift flavour")
    ap.add_argument("--lagsets", default="config1,rotated")
    args = ap.parse_args()
    pl, ps = bench.ensure_config1()
    lagsets = {
        "config1": dict(bench.LAGS),
        "rotated": dict(lag_crval1=np.arange(20, 28, 1.0), lag_crval2=np.arange(2, 10, 1.0),
                        lag_cdelt1=np.array([-0.002, 0.0, 0.002]), lag_cdelt2=np.array([0.0]),
                        lag_crota=np.array([-0.5, -0.1, 0.0, 0.1, 0.5])),
    }
    results = []
    for name, lags in lagsets.items():
        if name not in args.lagsets.split(","):
            continue
        kw = {} if name == "config1" else {"cdelt_semantics": "intended"}
        a = Alignment(pl, ps, parallelism=True, **lags, **kw)
        a.method, a.coordinate_frame = "correlation", "final_helioprojective"
        a._load_pair()
        a._set_initial_header_values(True)
        w_small, w_large = TanWcs.from_header(a.hdr_small), TanWcs.from_header(a.hdr_large)
        d = E.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
        base = None
        for combo in args.combos.split(","):
            arith, v = combo.split(":")
            eng = E.LagSearchEngine(order=2, variant=int(v), arithmetic=arith)
            eng.set_small(a.data_small)
            eng.prepare_hpc(a.data_large, w_large, w_small)
            table, _ = eng.hpc_lag_table(a.hdr_small, a, *d, kw.get("cdelt_semantics", "reference"))
            tab = eng._upload(table)
            out = torch.empty(table.shape[0], dtype=torch.float64, device=eng.device)
            nv = torch.empty(table.shape[0], dtype=torch.int64, device=eng.device)
            eng.evaluate(tab, out, nv)
            torch.cuda.synchronize()
            _ext.profile_begin()
            for _ in range(args.steps):
                eng.evaluate(tab, out, nv)
            ms, n = _ext.profile_end()
            c, nvh = out.cpu().numpy(), nv.cpu().numpy()
            if base is None:
                base, base_nv = c, nvh
            rec = {"lags": name, "n_lags": int(table.shape[0]), "arithmetic": arith, "variant": int(v),
                   "small32": eng.small32 is not None, "k1_ms_per_search": ms / args.steps,
                   "max_abs_diff_vs_fp64": float(np.nanmax(np.abs(c - base))),
                   "rms_diff_vs_fp64": float(np.sqrt(np.nanmean((c - base) ** 2))),
                   "nvalid_equal": bool(np.array_equal(nvh, base_nv)),
                   "argmax": int(np.nanargmax(c)), "argmax_equal": bool(np.nanargmax(c) == np.nanargmax(base))}
            print(json.dumps(rec), flush=True)
            results.append(rec)
            del eng, tab, out
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    json.dump(results, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
