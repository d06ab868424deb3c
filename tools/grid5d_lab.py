"""Where the time of BASELINE configs[3] (1 024 000-lag 5-D grid) goes: host table, upload, device time per lag for
rotated / rescaled lags and for pure CRVAL lags of the same count (GPU box).    python tools/grid5d_lab.py [--lags 31744]"""
import argparse
import json
import os
import sys
import time

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
    ap.add_argument("--lags", type=int, default=31744)
    args = ap.parse_args()
    pl, ps = bench.ensure_config1()
    a = Alignment(pl, ps, parallelism=True, cdelt_semantics="intended", **bench.GRID5D_LAGS)
    a.method, a.coordinate_frame = "correlation", "final_helioprojective"
    a._load_pair()
    a._set_initial_header_values(True)
    w_small, w_large = TanWcs.from_header(a.hdr_small), TanWcs.from_header(a.hdr_large)
    t0 = time.perf_counter()
    d = E.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
    eng = E.LagSearchEngine(order=2)
    eng.set_small(a.data_small)
    eng.prepare_hpc(a.data_large, w_large, w_small)
    t1 = time.perf_counter()
    table, dead = eng.hpc_lag_table(a.hdr_small, a, *d, "intended")
    t2 = time.perf_counter()
    print(json.dumps({"lags": int(table.shape[0]), "prep_s": t1 - t0, "host_table_s": t2 - t1,
                      "table_MB": table.nbytes / 1e6}), flush=True)
    n = min(args.lags, table.shape[0])
    # a representative block: lags spread over the whole grid
    sel = np.linspace(0, table.shape[0] - 1, n).astype(np.int64)
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    tab = eng._upload(table[sel])
    torch.cuda.synchronize()
    t4 = time.perf_counter()
    out = torch.empty(n, dtype=torch.float64, device=eng.device)
    eng.evaluate(tab, out)
    torch.cuda.synchronize()
    _ext.profile_begin()
    t5 = time.perf_counter()
    eng.evaluate(tab, out)
    torch.cuda.synchronize()
    t6 = time.perf_counter()
    ms, k = _ext.profile_end()
    print(json.dumps({"lags": n, "upload_s": t4 - t3, "evaluate_wall_s": t6 - t5, "lag_kernel_ms": ms, "launches": k,
                      "us_per_lag_kernel": 1e3 * ms / n, "us_per_lag_wall": 1e6 * (t6 - t5) / n}), flush=True)
    # pure CRVAL lags of the same count, for comparison
    pure = table[sel].copy()
    pure[:, 4:8] = table[0, 4:8] * 0 + np.array([np.cos(np.deg2rad(3.0)), -np.sin(np.deg2rad(3.0)),
                                               np.sin(np.deg2rad(3.0)), np.cos(np.deg2rad(3.0))])
    pure[:, 2:4] = table[0, 2:4] * 0 + a.hdr_small["CDELT1"] / 3600.0
    eng.flags |= _ext.FLAG_PURE_SHIFT
    tab = eng._upload(pure)
    out = torch.empty(n, dtype=torch.float64, device=eng.device)
    eng.evaluate(tab, out)
    torch.cuda.synchronize()
    _ext.profile_begin()
    eng.evaluate(tab, out)
    ms, k = _ext.profile_end()
    print(json.dumps({"pure_crval_lags_same_count": n, "lag_kernel_ms": ms, "us_per_lag_kernel": 1e3 * ms / n}))


if __name__ == "__main__":
    main()
