#!/usr/bin/env python
"""bench.py -- lag-evaluations/s of the helioprojective pointing search on BASELINE.json configs[0]
(HRIEUV-like 2048^2 vs FSI-174-like 3072^2, 60x60 CRVAL lags at 1 arcsec, synthetic FITS).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole 3600-lag grid (homographies + fused lag kernel + finalize, plus
the all-gather of the cube when N > 1; the lag list is sharded over the N ranks => strong scaling). The headline is
the ALL-FP64 kernel -- the reference's arithmetic (`dtype: "f64"`); the opt-in mixed-arithmetic kernel is reported
under `mixed`. `value` is device-timed with inputs resident in HBM; `e2e` is the same search through the host-facing
engine call with HOST buffers (H2D of both images and the lag table, statistics, the one-time resampling, the
search, D2H of the cube). `cube_sha256` is the digest of the gathered cube: equal for every N.
Beside the headline, in the same JSON line (`configs`): BASELINE configs[1] (Carrington grid, 14 400 lags sharded
over the ranks), configs[3] (1 024 000-lag 5-D grid sharded over the ranks) and configs[4] (256 frames sharded
over the ranks), each checked against committed oracle values where they exist.
`--impl reference` times the reference's CPU path: the reference itself cannot be installed in this image
(astropy / sunpy / poetry-core absent, no network), so the reference-structured oracle port runs with one process
per host core on a bounded sample of the same lag grid.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOAD = "config1: HRIEUV-like 2048x2048 vs FSI174-like 3072x3072, helioprojective, 60x60 CRVAL lags @1arcsec"
LAGS = dict(lag_crval1=np.arange(-30, 30, 1.0), lag_crval2=np.arange(-30, 30, 1.0), lag_cdelt1=np.array([0.0]),
            lag_cdelt2=np.array([0.0]), lag_crota=np.array([0.0]))
CARRINGTON_LAGS = dict(lag_crval1=np.arange(-60, 60, 1.0), lag_crval2=np.arange(-60, 60, 1.0),
                       lag_cdelt1=np.array([0.0]), lag_cdelt2=np.array([0.0]), lag_crota=np.array([0.0]))
CARRINGTON_GRID = dict(lonlims=(200.0, 300.0), latlims=(-20.0, 20.0), shape=(2048, 2048))
GRID5D_LAGS = dict(lag_crval1=np.arange(14, 34, 1.0), lag_crval2=np.arange(-4, 16, 1.0),
                   lag_cdelt1=(np.arange(16) - 8) * 0.001, lag_cdelt2=(np.arange(16) - 8) * 0.001,
                   lag_crota=(np.arange(10) - 5) * 0.1)
SEQUENCE_FRAMES, SEQUENCE_DISTINCT = 256, 16

# ---- roofline constants (DESIGN.md section 5 derives them) ----------------------------------------------------------
# Unit of work: one pixel-sample (one common-grid pixel under one lag). The binding resource is the FP64 pipe / the
# warp scheduler's dispatch port, not HBM and not the tensor cores (gather + reduction, no dense contraction).
# FLOOR = FP64 instructions per pixel-sample that the FORMULATION needs, counted by hand (not what the binary executes):
#   helioprojective rolling kernel, P rows per thread: 4 (two quadratic coordinates; 3 on a grid of pure CRVAL shifts,
#   where x is a line in the row index: `kLinXTol`, csrc/coreg_lag_roll.cu) + 5 (P + 2) / P (coefficients of the
#   new tap row) + 6 (three Horner forms in x) + 7 (coefficients + Horner form in y) + 4 (pivot, three moments)
#   + 28 / P (per thread and lag: first-pixel coordinates, floors, reciprocal, quadratic coefficients)
#   Carrington kernel, per evaluated (pixel, lag) pair: 8 (coordinates, floors, fractions) + 12 (weights) + 12 (taps)
#   + 4 (pivot, moments)
SURVEY_FP64_PER_SAMPLE_HPC = 69.0        # SURVEY.md 8(d): the reference's formulation (pixel -> world -> pixel per lag)
SURVEY_FP64_PER_SAMPLE_CARRINGTON = 54.0
BYTES_PER_SAMPLE = 8.0                   # un-amortised: one f32 sample of each image per pixel-sample


def hpc_floor(rows_per_thread, linear_x=False):
    p = float(rows_per_thread)
    return (3.0 if linear_x else 4.0) + 5.0 * (p + 2.0) / p + 6.0 + 7.0 + 4.0 + 28.0 / p


CARRINGTON_FLOOR = 36.0


def csrc_digest():
    """SHA-256 over the CUDA sources and the C header: ties ncu-derived constants to the code they were measured on."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "euispice_coreg_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(d, f), "rb").read())
    h.update(open(os.path.join(ROOT, "include", "coreg_b200.h"), "rb").read())
    return h.hexdigest()


def measured_constants():
    """profiles/kernel_constants.json: per kernel the ncu-measured executed FP64 instructions per pixel-sample and DRAM
    bytes per launch, with the source digest they belong to. Returned only when the digest matches the tree."""
    try:
        c = json.load(open(os.path.join(ROOT, "profiles", "kernel_constants.json")))
    except Exception:
        return {}, "profiles/kernel_constants.json missing"
    if c.get("csrc_sha256") != csrc_digest():
        return {}, "ncu constants withheld: profiles/kernel_constants.json was captured on other kernel sources"
    return c.get("kernels", {}), None


def synth_dir():
    """Cache of the seeded synthetic inputs (outside the source tree, which may be read-only). Per user: in a shared
    temporary directory another user's copy is not writable."""
    d = os.environ.get("COREG_BENCH_DATA") or os.path.join(tempfile.gettempdir(), f"coreg_bench_data_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return d


def ensure_config1(rank=0, barrier=None):
    from euispice_coreg_b200._synth.scene import make_config1
    d = synth_dir()
    pl, ps = os.path.join(d, "config1_large.fits"), os.path.join(d, "config1_small.fits")
    if rank == 0 and not (os.path.exists(pl) and os.path.exists(ps)):
        make_config1(d)
    if barrier is not None:
        barrier()
    return pl, ps


def ensure_sequence(n_distinct, rank=0, barrier=None):
    """configs[4]: the config-1 scene re-rendered with per-frame pointing jitter N(0, 1.5 arcsec), seeds 1000 + i."""
    from euispice_coreg_b200._synth.scene import PairSpec, make_pair, master_scene
    d = os.path.join(synth_dir(), "sequence")
    os.makedirs(d, exist_ok=True)
    paths = [os.path.join(d, f"frame{i:03d}_small.fits") for i in range(n_distinct)]
    if rank == 0 and not all(os.path.exists(p) for p in paths):
        sky = master_scene(PairSpec())
        rng = np.random.default_rng(1000)
        for i in range(n_distinct):
            jit = tuple(float(v) for v in rng.normal(0.0, 1.5, 2))
            make_pair(d, PairSpec(jitter=jit, noise_seed=1000 + i), tag=f"frame{i:03d}", sky=sky, write_large=False)
    if barrier is not None:
        barrier()
    return paths


def load_pair(pl, ps):
    from euispice_coreg_b200._compat import fits_lite
    L, S = fits_lite.open(pl)[0], fits_lite.open(ps)[0]
    return L.data, L.header, S.data, S.header


def run_config(n_gpus):
    """`config` of the JSON line: identical for the GPU arm and the reference arm."""
    return {"workload": WORKLOAD, "lags": 3600, "grid": [2048, 2048], "spline_order": 2,
            "arithmetic": "fp64 (spline, float32 store and Pearson moments as the reference evaluates them)",
            "parallelism": f"lag grid sharded over {n_gpus} rank(s) (GPU arm) / over the host cores (reference arm)",
            "l2": "flushed: a 256 MiB device buffer is rewritten before every timed step, inside the timed region "
                  "(GPU arm)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------
# CPU arm (reference-structured oracle port)
# ---------------------------------------------------------------------------------------------------------
_CPU_SEARCH = None


def cpu_search():
    """The CPU arm's one-time preparation (FITS read, PCi_j checks, the one-time cut of the large image), done once
    per process -- like the reference does it once per `align_using_helioprojective` call, outside the lag loop."""
    global _CPU_SEARCH
    if _CPU_SEARCH is None:
        from oracle.hpc import HpcSearch
        pl, ps = ensure_config1()
        dl, hl, ds, hs = load_pair(pl, ps)
        _CPU_SEARCH = HpcSearch(dl, dict(hl.items()), ds, dict(hs.items()), **LAGS)
    return _CPU_SEARCH


def cpu_sample(n_lags_per_core=1, cores=None):
    """Evaluate a bounded sample of the config-1 lag grid the way the reference does (per lag: pixel->world and
    world->pixel of the full grid, scipy map_coordinates, NaN compaction, two-pass Pearson) with one forked
    process per host core. Returns (lag_evals_per_s, seconds, n_lags, cores)."""
    from oracle.hpc import cube_multiprocess
    cores = cores or len(os.sched_getaffinity(0))
    search = cpu_search()
    n_total = 3600
    n = cores * n_lags_per_core
    sel = np.linspace(0, n_total - 1, n).astype(int)   # spread over the grid: in- and out-of-overlap lags alike
    t0 = time.perf_counter()
    cube_multiprocess(search, cores, sel)
    dt = time.perf_counter() - t0
    return n / dt, dt, n, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    per_core = 1
    secs = []
    cores = len(os.sched_getaffinity(0))
    cpu_search()
    for i in range(args.warmup + args.steps):
        v, dt, n, cores = cpu_sample(per_core, cores)
        if i >= args.warmup:
            secs.append(dt)
    total_lags = cores * per_core * args.steps
    value = total_lags / sum(secs)
    sample = (f"{cores * per_core} of 3600 lags per step (1 per core, spread over the grid), {args.steps} steps, "
              f"{sum(secs):.1f} s; rate extrapolated to the grid; one-time cut of the large image outside the timed "
              "region; NumPy port of the reference's per-lag body (numpy WCS in place of wcslib), "
              "multiprocessing over host cores")
    line = {"impl": "reference", "metric": "lag_evals_per_s", "value": value, "unit": "lag-evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sum(secs) / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": run_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "lag-evals/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "lag-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "reference not installable here (astropy, sunpy, poetry-core absent); oracle port of "
                    "hdrshift/alignment.py:509-549 with multiprocessing over host cores"}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------
# GPU arm: helpers
# ---------------------------------------------------------------------------------------------------------
class Ctx:
    """torch / dist handles + the collectives the measurements need."""

    def __init__(self, torch, dist, rank, world, device):
        self.torch, self.dist, self.rank, self.world, self.device = torch, dist, rank, world, device

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, v):
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.device)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v):
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.device)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def timed_device(ctx, step, steps, warmup):
    """W warm-up steps, then K steps between CUDA events, bracketed by barrier + synchronize; max over ranks [ms]."""
    torch = ctx.torch
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1))


def golden(name):
    try:
        return np.load(os.path.join(ROOT, "tests", "golden", name))
    except Exception:
        return None


def carrington_secondary(pl, ps, steps, world, barrier, torch, dist, variant=0, align_wall=True, fp64_peak=None,
                         shard=None):
    """BASELINE.json configs[1] (same image pair on a user Carrington grid 2048^2, 120 x 120 CRVAL lags), measured
    beside the headline: device-timed search with everything resident (lags sharded like the headline) and the wall
    time of the public call. Returns a dict for the JSON line."""
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200.hdrshift import engine as E
    from euispice_coreg_b200.hdrshift.alignment import Alignment
    a = Alignment(pl, ps, parallelism=True, **CARRINGTON_LAGS)
    a.method, a.coordinate_frame, a.method_carrington_reprojection = "correlation", "final_carrington", "fa"
    a._load_pair()
    a._set_initial_header_values(True)
    a.lonlims, a.latlims, a.shape = (CARRINGTON_GRID[k] for k in ("lonlims", "latlims", "shape"))
    d1, d2, _, _, _ = E.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
    eng = E.LagSearchEngine(order=2, small_storage="auto", variant=variant)   # float32 storage, as Alignment does here
    eng.set_small(a.data_small)
    r_sun = float(a.lag_solar_r[0])
    eng.prepare_carrington_large(a.data_large, a.hdr_large, r_sun, a.lonlims, a.latlims, a.shape)
    planes = eng.carrington_planes(a.hdr_small, r_sun, a.lonlims, a.latlims, a.shape)
    roll = a.hdr_small["CROTA"] if "CROTA" in a.hdr_small else a.hdr_small["CROTA2"]
    x0, y0 = eng.carrington_offset(a.hdr_small, a.crval1_ref + d1, a.crval2_ref + d2, roll)
    table = np.stack([x0, y0], axis=1).astype(np.float64)
    n = table.shape[0]
    rank = dist.get_rank() if world > 1 else 0
    chunk, bounds = E.shard_bounds(n, world)
    lo, hi = bounds[rank]
    if shard is not None:      # tools/carr_lab.py: the slice rank r of w ranks would get, on one GPU (no collective)
        chunk, bounds = E.shard_bounds(n, shard[1])
        lo, hi = bounds[shard[0]]
    # the kernel takes its lags in detector-plane patches (engine.offset_patch_order), padded with dummy lags
    i1, i2 = np.unravel_index(np.arange(lo, hi), (len(a.lag_crval1), len(a.lag_crval2)))
    slot, n_slots = E.offset_patch_order(i1, i2)
    padded = np.full((n_slots, 2), np.nan)
    padded[slot] = table[lo:hi]
    tab_dev = eng._upload(padded)
    slot_dev = torch.from_numpy(slot).to(eng.device)
    out_p = torch.empty(n_slots, dtype=torch.float64, device=eng.device)
    nv_p = torch.zeros(n_slots, dtype=torch.int64, device=eng.device)
    out = torch.full((chunk,), float("nan"), dtype=torch.float64, device=eng.device)
    full = torch.empty(chunk * world, dtype=torch.float64, device=eng.device)

    def step():
        eng.evaluate(tab_dev, out_p, nv_p, planes)
        out[:hi - lo] = out_p.index_select(0, slot_dev)
        if world > 1:
            dist.all_gather_into_tensor(full, out)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    barrier()
    _ext.profile_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    k_ms, k_n = _ext.profile_end()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=eng.device)
    eff = nv_p.index_select(0, slot_dev).sum().to(torch.float64).reshape(1)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(eff, op=dist.ReduceOp.SUM)
    ms = float(t.item()) / steps
    if shard is not None:
        return {"shard": list(shard), "lags": hi - lo, "ms_per_search": ms, "kernel_ms": k_ms / max(1, steps),
                "kernel_launches_per_search": k_n // max(1, steps), "effective_pixel_samples": float(eff.item())}
    cube = (full[:n] if world > 1 else out[:n]).cpu().numpy()
    res = {"workload": "configs[1]: same pair on a Carrington grid 2048x2048 (lon 200-300 deg, lat +-20 deg), 120x120 "
                       "CRVAL lags @1arcsec, lags sharded over the ranks", "lags": n, "ms_per_search": ms,
           "lag_evals_per_s": n / (ms * 1e-3),
           "effective_pixel_samples_per_s": float(eff.item()) / (ms * 1e-3),
           "effective_fraction_of_grid": float(eff.item()) / (n * 2048.0 * 2048.0),
           "kernel_ms_this_rank": k_ms / max(1, steps), "kernel_launches_per_search": k_n // max(1, steps),
           "cube_sha256": hashlib.sha256(np.ascontiguousarray(cube).tobytes()).hexdigest()}
    if fp64_peak:
        eff_rate = float(eff.item()) / (ms * 1e-3)
        res["roofline"] = {"bound": "fp64", "unit": "T FP64-instr/s", "peak": world * fp64_peak / 1e12,
                           "achieved": CARRINGTON_FLOOR * eff_rate / 1e12,
                           "frac": CARRINGTON_FLOOR * eff_rate / (world * fp64_peak),
                           "algorithmic": f"{CARRINGTON_FLOOR:.0f} FP64 instr per evaluated (pixel, lag) pair (hand count "
                                          "of this kernel's formulation, DESIGN.md 5) x effective pixel-samples/s",
                           "frac_survey_count": SURVEY_FP64_PER_SAMPLE_CARRINGTON * eff_rate / (world * fp64_peak)}
        kc = measured_constants()[0].get("offset_window_kernel", {})
        if kc:
            res["roofline"]["executed_fp64_per_evaluated_pair"] = kc.get("fp64_instr_per_pixel_sample")
            res["roofline"]["traffic"] = kc.get("dram_bytes_per_launch") if world == 1 else None
    z = golden("config2_sample.npz")
    if z is not None:
        res["oracle_check"] = {"lags": int(z["index"].size),
                               "max_abs_err": float(np.nanmax(np.abs(cube[z["index"]] - z["r"]))),
                               "source": "tests/golden/config2_sample.npz (oracle/carrington.py on the same synthetic pair)"}
    am = np.unravel_index(int(np.nanargmax(cube)), (len(a.lag_crval1), len(a.lag_crval2)))
    res["argmax_lag_arcsec"] = [float(CARRINGTON_LAGS["lag_crval1"][am[0]]), float(CARRINGTON_LAGS["lag_crval2"][am[1]])]
    barrier()
    if align_wall:
        t0 = time.perf_counter()
        Alignment(pl, ps, parallelism=True, **CARRINGTON_LAGS).align_using_carrington(method="correlation",
                                                                                    **CARRINGTON_GRID)
        torch.cuda.synchronize()
        res["align_wall_s"] = time.perf_counter() - t0
    return res


def grid5d_secondary(ctx, pl, ps):
    """BASELINE configs[3]: 20 x 20 x 16 x 16 x 10 = 1 024 000 lags (intended CDELT semantics) through the public API,
    the flat lag list sharded over the ranks, one all-gather; checked on the committed oracle sample."""
    from euispice_coreg_b200.hdrshift import Alignment
    torch = ctx.torch
    n = int(np.prod([len(v) for v in GRID5D_LAGS.values()]))
    ctx.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    a = Alignment(pl, ps, parallelism=True, cdelt_semantics="intended", **GRID5D_LAGS)
    cube = a.align_using_helioprojective(return_type="corr")
    torch.cuda.synchronize()
    wall = ctx.max_over_ranks(time.perf_counter() - t0)
    res = {"workload": "configs[3]: 5-D lag grid 20x20x16x16x10 (CRVAL1 x CRVAL2 x CDELT1 x CDELT2 x CROTA, steps 1 arcsec / "
                       "0.001 arcsec / 0.1 deg, intended CDELT semantics), all-FP64, lags sharded over the ranks",
           "lags": n, "wall_s_public_api": wall, "lag_evals_per_s": n / wall,
           "pixel_samples_per_s": n * 2048.0 * 2048.0 / wall,
           "argmax_index": [int(v) for v in np.unravel_index(int(np.nanargmax(cube)), cube.shape)[:5]],
           "cube_sha256": hashlib.sha256(np.ascontiguousarray(cube).tobytes()).hexdigest()}
    z = golden("config4_sample.npz")
    if z is not None:
        res["oracle_check"] = {"lags": int(z["index"].size),
                               "max_abs_err": float(np.nanmax(np.abs(cube.ravel()[z["index"]] - z["r"]))),
                               "source": "tests/golden/config4_sample.npz (oracle/hpc.py, cdelt_mode='intended')"}
    return res


SPICE_LAGS = dict(lag_crval1=np.arange(-43, -2, 1.0), lag_crval2=np.arange(16, 57, 1.0), lag_cdelt1=np.array([0.0]),
                  lag_cdelt2=np.array([0.0]), lag_crota=np.array([0.0]))


def ensure_spice(rank=0, barrier=None):
    """configs[2]: synthetic SPICE L2 raster (192 x 832 x 40) + 12 FSI-304-like frames of 3072^2 (`_synth/spice.py`)."""
    from euispice_coreg_b200._synth.spice import SpiceSpec, make_spice_case
    d = os.path.join(synth_dir(), "spice")
    os.makedirs(d, exist_ok=True)
    spec = SpiceSpec(cadence_s=250.0)      # 12 frames over the 2880 s of the scan: every column within 130 s of a frame
    p_spice = os.path.join(d, "solo_L2_spice-n-ras_config3.fits")
    imagers = [os.path.join(d, f"config3_fsi304_{k:02d}.fits") for k in range(spec.n_frames)]
    if rank == 0 and not all(os.path.exists(p) for p in [p_spice] + imagers):
        make_spice_case(d, spec, tag="config3")
    if barrier is not None:
        barrier()
    return p_spice, imagers, spec, d


def spice_secondary(ctx, rank):
    """BASELINE configs[2]: the synthetic raster of a SPICE scan built from the FSI 304 sequence at the exposure times of
    its columns (`SPICEComposedMapBuilder`, `synras/map_builder.py:57-131`), then `AlignmentSpice` of the SPICE L2 cube
    against it in the helioprojective frame (41 x 41 CRVAL lags, sharded over the ranks). Every rank builds the raster
    (it is the search's reference image, replicated like every image); checked against oracle/synras.py + oracle/hpc.py."""
    from euispice_coreg_b200._compat import fits_lite
    from euispice_coreg_b200.hdrshift import AlignmentSpice
    from euispice_coreg_b200.synras import SPICEComposedMapBuilder
    torch = ctx.torch
    p_spice, imagers, spec, d = ensure_spice(rank, ctx.barrier)
    name = f"synras_rank{rank}.fits"
    walls = {}
    for rep in range(2):          # the first pass pays the page cache of 450 MB of imager files
        ctx.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        synras = SPICEComposedMapBuilder(p_spice, imagers, threshold_time=150.0).process(
            folder_path_output=d, basename_output=name, print_filename=False, return_synras_name=True)
        torch.cuda.synchronize()
        walls["synras"] = ctx.max_over_ranks(time.perf_counter() - t0)
        ctx.barrier()
        t0 = time.perf_counter()
        a = AlignmentSpice(synras, p_spice, parallelism=True, small_fov_window=0, large_fov_window=-1, **SPICE_LAGS)
        cube = a.align_using_helioprojective(return_type="corr")
        torch.cuda.synchronize()
        walls["search"] = ctx.max_over_ranks(time.perf_counter() - t0)
    n = int(cube.size)
    am = np.unravel_index(int(np.nanargmax(cube)), cube.shape)
    res = {"workload": f"configs[2]: SPICE-like L2 raster {spec.n_x}x{spec.n_y}x{spec.n_lambda} vs the synthetic raster built "
                       f"from {spec.n_frames} FSI-304-like frames of {spec.large_n}^2, helioprojective, 41x41 CRVAL lags "
                       "@1arcsec, lags sharded over the ranks",
           "lags": n, "synras_build_wall_s": walls["synras"], "search_wall_s_public_api": walls["search"],
           "lag_evals_per_s": n / walls["search"],
           "pixel_samples_per_s": n * float(spec.n_x * spec.n_y) / walls["search"],
           "argmax_lag_arcsec": [float(SPICE_LAGS["lag_crval1"][am[0]]), float(SPICE_LAGS["lag_crval2"][am[1]])],
           "true_shift_arcsec": [float(v) for v in spec.true_shift],
           "cube_sha256": hashlib.sha256(np.ascontiguousarray(cube).tobytes()).hexdigest()}
    # Oracle check. A synthetic raster carries the SPICE header by construction, so the one-time cut maps pixel (i, j) onto
    # (i, j) +- 1e-11 and whole border rows sit exactly on map_coordinates' closed [0, n-1] bound: whether they count
    # is decided by the last bit of the WCS round trip, in the reference as much as here (README, "documented
    # exception"; tests/test_gpu_spice.py). The strict check therefore runs on a copy of the raster whose CRPIX is moved
    # by a fraction of a pixel; the unmodified case is reported beside it.
    hd = fits_lite.open(synras)[0]
    h_off = hd.header.copy()
    h_off["CRPIX1"] = h_off["CRPIX1"] + 0.37
    h_off["CRPIX2"] = h_off["CRPIX2"] - 0.41
    synras_off = os.path.join(d, f"synras_off_rank{rank}.fits")
    fits_lite.writeto(synras_off, [fits_lite.PrimaryHDU(np.array(hd.data), h_off)], overwrite=True)
    ctx.barrier()
    cube_off = AlignmentSpice(synras_off, p_spice, parallelism=True, small_fov_window=0, large_fov_window=-1,
                              **SPICE_LAGS).align_using_helioprojective(return_type="corr")
    if rank == 0:
        try:
            from oracle.hpc import HpcSearch
            from oracle.synras import spice_l2_image
            sp = fits_lite.open(p_spice)[0]
            img, hdr = spice_l2_image(np.asarray(sp.data), dict(sp.header.items()))
            rng = np.random.default_rng(2)
            flat = np.unique(np.concatenate([[am[0] * 41 + am[1], 0, n - 1], rng.integers(0, n, 13)]))
            for key, path, got_cube in (("oracle_check", synras_off, cube_off), ("oracle_check_unmodified", synras, cube)):
                hdl = fits_lite.open(path)[0]
                srch = HpcSearch(np.asarray(hdl.data), dict(hdl.header.items()), img, hdr, **SPICE_LAGS)
                l1, l2, l3, l4, l5 = srch.flat_lags()
                ref = np.array([srch.step(l1[i], l2[i], l3[i], l4[i], l5[i]) for i in flat])
                got = got_cube.ravel()[flat]
                ok = np.isfinite(ref) & np.isfinite(got)
                res[key] = {"lags": int(flat.size), "max_abs_err": float(np.max(np.abs(ref[ok] - got[ok]))),
                            "nan_pattern_equal": bool(np.array_equal(np.isfinite(ref), np.isfinite(got))),
                            "source": "oracle/hpc.py on the device-built synthetic raster (itself checked against "
                                      "oracle/synras.py in tests/test_gpu_spice.py)"
                                      + ("; CRPIX moved by (0.37, -0.41) pixel" if key == "oracle_check" else
                                         "; border rows on the closed bound: the documented knife edge")}
        except Exception as exc:      # the check must never cost the measurement
            res["oracle_check"] = {"error": repr(exc)}
    return res


def sequence_secondary(ctx, pl, rank, n_frames, n_distinct):
    """BASELINE configs[4]: `n_frames` frame searches (60 x 60 lags each) against one resident reference image, FRAMES
    sharded over the ranks, one all-gather of the cubes. The frame files are `n_distinct` jittered renderings of the
    scene, each used n_frames / n_distinct times (every use is a full read + upload + cut + search; nothing is cached
    between frames)."""
    from euispice_coreg_b200.hdrshift import SequenceAlignment
    torch = ctx.torch
    paths = ensure_sequence(n_distinct, rank, ctx.barrier)
    frames = [paths[k % n_distinct] for k in range(n_frames)]
    SequenceAlignment(pl, frames[:2 * ctx.world], **LAGS).align_using_helioprojective(return_type="corr")   # warm-up
    ctx.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    seq = SequenceAlignment(pl, frames, **LAGS)
    cubes = seq.align_using_helioprojective(return_type="corr")
    torch.cuda.synchronize()
    wall = ctx.max_over_ranks(time.perf_counter() - t0)
    peaks = [np.unravel_index(int(np.nanargmax(c)), c.shape)[:2] for c in cubes[:n_distinct]]
    same = all(np.array_equal(cubes[k], cubes[k % n_distinct], equal_nan=True) for k in range(n_frames))
    h = hashlib.sha256()
    for c in cubes:
        h.update(np.ascontiguousarray(c).tobytes())
    return {"workload": f"configs[4]: {n_frames} frame searches (60x60 lags each) vs one resident FSI-like image, frames "
                        f"sharded over the ranks; {n_distinct} distinct jittered frame files used {n_frames // n_distinct}x",
            "frames": n_frames, "wall_s_public_api": wall, "frames_per_s": n_frames / wall,
            "lag_evals_per_s": n_frames * 3600 / wall, "pixel_samples_per_s": n_frames * 3600 * 2048.0 * 2048.0 / wall,
            "repeated_frames_bit_identical": bool(same),
            "argmax_lags_arcsec_first_frames": [[float(LAGS["lag_crval1"][i]), float(LAGS["lag_crval2"][j])]
                                                for i, j in peaks[:4]],
            "cubes_sha256": h.hexdigest()}


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from euispice_coreg_b200 import _ext
    from euispice_coreg_b200._compat.wcs import TanWcs
    from euispice_coreg_b200.hdrshift import engine as E
    from euispice_coreg_b200.hdrshift.alignment import Alignment

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    _ext.load()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local),
                                timeout=datetime.timedelta(seconds=600))
    ctx = Ctx(torch, dist, rank, world, torch.device("cuda", local))
    barrier = ctx.barrier
    warmup = max(args.warmup, 3)

    pl, ps = ensure_config1(rank, barrier)
    # host-side preparation exactly as Alignment does it (header checks, lag units, PC matrix)
    a = Alignment(pl, ps, parallelism=True, **LAGS)
    a.method, a.coordinate_frame = "correlation", "final_helioprojective"
    a._load_pair()
    a._set_threshold_minmax_to_nan()
    a._set_initial_header_values(True)
    w_small, w_large = TanWcs.from_header(a.hdr_small), TanWcs.from_header(a.hdr_large)
    d = E.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)
    gny, gnx = a.data_small.shape
    n_pix = gnx * gny
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=ctx.device)

    def make_engine(arith):
        e = E.LagSearchEngine(order=2, strict=args.strict, variant=args.variant, small_storage=args.small_storage,
                              no_fast=args.no_fast, arithmetic=arith)
        e.set_small(a.data_small)
        e.prepare_hpc(a.data_large, w_large, w_small)
        return e

    def device_arm(arith):
        """Device-timed search with everything resident: ms per step over all ranks, kernel ms of this rank, launches,
        the gathered cube, the engine, the lags the mixed kernel's guard sent back to FP64."""
        eng = make_engine(arith)
        table, _ = eng.hpc_lag_table(a.hdr_small, a, *d)
        n_lags = table.shape[0]
        chunk, bounds = E.shard_bounds(n_lags, world)
        lo, hi = bounds[rank]
        tab_dev = eng._upload(table[lo:hi])
        local_out = torch.full((chunk,), float("nan"), dtype=torch.float64, device=eng.device)
        full = torch.empty(chunk * world, dtype=torch.float64, device=eng.device)

        def step():
            # L2 hygiene: a 256 MiB buffer (> the 126 MB L2) is rewritten before every step, inside the timed region
            l2_flush.zero_()
            eng.evaluate(tab_dev, local_out[:hi - lo])
            if world > 1:
                dist.all_gather_into_tensor(full, local_out)

        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        barrier()
        _ext.profile_begin()
        ms_total = timed_device(ctx, step, args.steps, 0)
        k_ms, k_n = _ext.profile_end()
        flagged = eng.resolve_flags(tab_dev, local_out[:hi - lo])   # mixed only
        if world > 1:
            dist.all_gather_into_tensor(full, local_out)
        last = (full[:n_lags] if world > 1 else local_out[:n_lags]).cpu().numpy()   # the last timed step's cube
        # evaluated (pixel, lag) pairs of this rank's slice: what the roofline counts (one more pass, untimed)
        nv = torch.zeros(max(hi - lo, 1), dtype=torch.int64, device=eng.device)
        if hi > lo:
            eng.evaluate(tab_dev, local_out[:hi - lo], nv[:hi - lo])
            eng.resolve_flags(tab_dev, local_out[:hi - lo], nv[:hi - lo])
        if world > 1:
            dist.all_gather_into_tensor(full, local_out)
        cube = (full[:n_lags] if world > 1 else local_out[:n_lags]).cpu().numpy()
        return dict(ms=ms_total / args.steps, k_ms=k_ms / max(1, k_n), k_n=k_n, cube=cube, last=last, eng=eng,
                    table=table, lo=lo, hi=hi, n_lags=n_lags, flagged=int(ctx.sum_over_ranks(flagged)),
                    evaluated=float(nv[:hi - lo].sum().item()) if hi > lo else 0.0,
                    fast=table.shape[1] == _ext.TAN_WCS_DOUBLES)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    main = device_arm(args.arithmetic or "fp64")
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives: r per lag, flat in the lag order of the cube (lag_crval1 major)
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "corr.npy"), main["last"].astype(np.float64))
    eng, table, n_lags, lo, hi = main["eng"], main["table"], main["n_lags"], main["lo"], main["hi"]
    value = n_lags / (main["ms"] * 1e-3)
    mixed = None
    if not args.no_mixed and (args.arithmetic or "fp64") == "fp64" and main["fast"]:
        m = device_arm("mixed")
        mixed = {"what": "opt-in mixed arithmetic (Alignment(arithmetic='mixed')): FP64 projection, FP32 spline on the "
                         "pivot-centred float32 payload, float32 store reproduced, per-lag guard + FP64 re-evaluation",
                 "dtype": "f64+f32", "value": n_lags / (m["ms"] * 1e-3), "unit": "lag-evals/s", "ms_per_step": m["ms"],
                 "kernel_ms": m["k_ms"], "lags_flagged_by_guard": m["flagged"],
                 "max_abs_diff_vs_fp64_cube": float(np.nanmax(np.abs(m["cube"] - main["cube"]))),
                 "same_argmax": bool(int(np.nanargmax(m["cube"])) == int(np.nanargmax(main["cube"])))}
        del m

    # ---- end to end: host buffers -> cube on the host, every step -------------------------------------------
    # host inputs: the images as the FITS files hold them (float32), in pinned memory
    h_large = torch.from_numpy(np.ascontiguousarray(a.data_large)).pin_memory().numpy()
    h_small = torch.from_numpy(np.ascontiguousarray(a.data_small)).pin_memory().numpy()
    e2e_steps = args.steps

    def e2e_step():
        e = E.LagSearchEngine(order=2, strict=args.strict, variant=args.variant, small_storage=args.small_storage,
                              no_fast=args.no_fast, arithmetic=args.arithmetic or "fp64")
        e.set_small(h_small, pinned=True)
        e.prepare_hpc(h_large, w_large, w_small)
        e.pure_shift_hint = eng.pure_shift_hint     # what hpc_lag_table derived from the lag grid
        return e.search(table)

    e2e_step()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        cube_e2e = e2e_step()
    torch.cuda.synchronize()
    barrier()
    e2e_s = ctx.max_over_ranks(time.perf_counter() - t0)
    h2d = h_large.nbytes + h_small.nbytes + table[lo:hi].nbytes
    d2h = n_lags * 8

    # full public API once on every rank (FITS read + host prep + sharded search + all-gather + Gaussian fit):
    # the "align() wall time" metric. It contains a collective, so all ranks take part.
    # Called three times: the first call of a process pays one-time costs (page cache of the FITS files, allocator
    # growth); `align_wall_s` is the best of the three (what a caller aligning a sequence sees per pair), the first call
    # is reported beside it.
    align_walls = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        res = Alignment(pl, ps, parallelism=True, arithmetic=args.arithmetic, **LAGS).align_using_helioprojective()
        torch.cuda.synchronize()
        align_walls.append(ctx.max_over_ranks(time.perf_counter() - t0))
    align_wall = min(align_walls)
    fp64_peak = _ext.fp64_peak(40000)          # FP64 FMA lane-instructions / s, measured now on this GPU
    configs = {}
    if not args.no_secondary:
        for name, fn in (("configs1_carrington",
                          lambda: carrington_secondary(pl, ps, args.steps, world, barrier, torch, dist,
                                                       args.carrington_variant, fp64_peak=fp64_peak)),
                         ("configs2_spice", lambda: spice_secondary(ctx, rank)),
                         ("configs3_grid5d", lambda: grid5d_secondary(ctx, pl, ps)),
                         ("configs4_sequence", lambda: sequence_secondary(ctx, pl, rank, args.frames, SEQUENCE_DISTINCT))):
            try:
                configs[name] = fn()
            except Exception as exc:   # never lose the headline line over a secondary measurement
                if world > 1:
                    raise              # (a rank that skips a collective would hang the others)
                configs[name] = {"error": repr(exc)}
    widened = None
    if world == 1 and not args.no_secondary:
        # the SURVEY 8f-4 paths, timed for the record (single GPU only: not part of `value`)
        try:
            from tools import car_bench, pxl_bench, surface_bench
            widened = {"initial_carrington": car_bench.run(2048, 1024, 60), "pixel_shift": pxl_bench.run(),
                       "sunpy_reprojection": surface_bench.run(3)}
        except Exception as exc:
            widened = {"error": repr(exc)}
    if rank == 0:
        am = tuple(int(v) for v in res.max_index[:2])
        best = (float(LAGS["lag_crval1"][am[0]]), float(LAGS["lag_crval2"][am[1]]))
        assert np.array_equal(np.nan_to_num(cube_e2e), np.nan_to_num(res.corr.ravel())), "e2e cube != public API cube"
        assert np.array_equal(np.nan_to_num(cube_e2e), np.nan_to_num(main["cube"])), "e2e cube != device-timed cube"
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        consts, withheld = measured_constants()
        fast = main["fast"]
        arith = eng.arithmetic if fast else "generic"
        rows = 12 if args.variant == 3 else (14 if args.variant == 2 else 16)
        kname = ("lag_corr_roll_kernel<MIXED>" if arith == "mixed" else "lag_corr_roll_kernel") if fast \
            else "lag_corr_kernel<TanCoord>"
        kc = consts.get(kname, {})
        launches_per_step = max(1, main["k_n"] // args.steps)
        samples_per_launch = n_pix * (hi - lo) / launches_per_step
        floor = hpc_floor(rows, linear_x=bool(eng.pure_shift_hint)) if fast else SURVEY_FP64_PER_SAMPLE_HPC
        # the floor is per EVALUATED pixel-sample: a few per cent of the nominal ones lie outside the small image under
        # their lag and cost nothing
        evaluated_per_launch = main["evaluated"] / launches_per_step
        ach = floor * evaluated_per_launch / (main["k_ms"] * 1e-3)
        executed = kc.get("fp64_instr_per_pixel_sample")
        traffic = kc.get("dram_bytes_per_launch")
        roof = {"bound": "fp64", "achieved": ach / 1e12, "peak": fp64_peak / 1e12, "unit": "T FP64-instr/s",
                "frac": ach / fp64_peak,
                "traffic": (traffic * (hi - lo) / 3600.0) if (traffic and n_lags == 3600) else None,
                "traffic_unit": "B per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum of one 3600-lag launch, "
                                "scaled by this rank's share of the lags)",
                "kernel": kname, "kernel_ms": main["k_ms"], "rows_per_thread": rows,
                "algorithmic": (f"{floor:.2f} FP64 instr/pixel-sample (hand-derived floor of the homography + rolling-"
                                f"window formulation at {rows} rows per thread, DESIGN.md 5) x "
                                f"{evaluated_per_launch:.3e} evaluated pixel-samples/launch "
                                f"({evaluated_per_launch / samples_per_launch:.3f} of the nominal "
                                f"{samples_per_launch:.3e})") if fast else
                               f"{floor:.0f} FP64 instr/pixel-sample (SURVEY 8d)",
                "executed_fp64_per_nominal_pixel_sample": executed,
                "executed_over_floor": (executed * samples_per_launch / evaluated_per_launch / floor) if executed else None,
                "constants": withheld or "profiles/kernel_constants.json (ncu, same kernel sources)",
                "peak_source": "coreg_fp64_peak DFMA microbenchmark, this run (148 SMs x 64 lanes x clock: nominal 18.6)",
                "note": "FP64 issue is the binding unit (no dense contraction: no tensor cores; DRAM < 1 % of peak). A "
                        "DFMA holds the warp scheduler's dispatch port for 2 cycles and every other instruction for 1 "
                        "(profiles/r1_fp64_issue_model.md), so with this kernel's instruction mix the reachable "
                        "fraction of the DFMA peak is about 0.8"}
        if arith == "mixed":
            roof["note"] = ("mixed arithmetic moves the spline off the FP64 pipe: this fraction counts only the FP64 "
                            "instructions the formulation still needs; the binding unit is the dispatch port")
        line = {
            "metric": "lag_evals_per_s", "value": value, "unit": "lag-evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": main["ms"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64+f32" if arith == "mixed" else "f64",
            "data": "synthetic",
            "config": run_config(world),
            "run": {"arithmetic": arith, "variant": args.variant, "rows_per_thread": rows,
                    "kernel": "generic" if (args.no_fast or args.strict) else "rolling (homography)",
                    "small_storage": str(eng.small.dtype).replace("torch.", ""),
                    "workspace_MB": eng._work.numel() * 8 / 1e6},
            "pixel_samples_per_s": value * n_pix,
            "cube_sha256": hashlib.sha256(np.ascontiguousarray(main["cube"]).tobytes()).hexdigest(),
            "e2e": {"value": n_lags * e2e_steps / e2e_s, "unit": "lag-evals/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_s / e2e_steps,
                    "what": f"LagSearchEngine from pinned host arrays ({h_large.dtype} large, {h_small.dtype} small, as "
                            "the FITS files hold them): H2D images + lag table, statistics + widening, one-time "
                            "resampling, search, all-gather, D2H cube"},
            "align_wall_s": align_wall, "align_wall_first_call_s": align_walls[0], "argmax_lag_arcsec": best,
            "mixed": mixed,
            "configs": configs,
            "widened": widened,
            # own kernels inside the timed region: per lag-kernel launch the homography table (fast path), the fused
            # lag kernel and the finalize kernel (the L2 flush memset and the NCCL all-gather are not ours)
            "gpu_launches": int(main["k_n"] * (3 if fast else 2)),
            "clocks": clocks,
            "roofline": roof,
            "roofline_survey": {"bound": "fp64", "achieved": SURVEY_FP64_PER_SAMPLE_HPC * samples_per_launch
                                / (main["k_ms"] * 1e-3) / 1e12, "peak": fp64_peak / 1e12, "unit": "T FP64-instr/s",
                                "frac": SURVEY_FP64_PER_SAMPLE_HPC * samples_per_launch / (main["k_ms"] * 1e-3) / fp64_peak,
                                "algorithmic": "69 FP64 instr/pixel-sample: SURVEY 8d's count for the reference's "
                                               "pixel->world->pixel formulation; > 1 means this formulation needs fewer "
                                               "instructions than that one's minimum"},
            "roofline_hbm": {"bound": "hbm", "achieved": BYTES_PER_SAMPLE * samples_per_launch / (main["k_ms"] * 1e-3) / 1e9,
                             "peak": hbm_peak, "unit": "GB/s",
                             "frac": BYTES_PER_SAMPLE * samples_per_launch / (main["k_ms"] * 1e-3) / 1e9 / hbm_peak,
                             "traffic": None, "peak_source": hbm_src,
                             "algorithmic": f"{BYTES_PER_SAMPLE:.0f} B/pixel-sample (un-amortised: what a kernel without "
                                            "lag batching would move)"},
        }
        if world == 1 and not args.no_cpu_baseline:
            v, dt, n, cores = cpu_sample(1)
            line["cpu_baseline"] = {"value": v, "unit": "lag-evals/s", "cores": cores, "kind": "port",
                                    "sample": f"{n} of 3600 lags (1 per core, spread over the grid), {dt:.1f} s; "
                                              "NumPy port of the reference's per-lag body (numpy WCS in place of "
                                              "wcslib) with multiprocessing: a stated baseline, not the target"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every timed loop (headline, e2e, configs[1])")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the headline cube of the last step to DIR/corr.npy (float64)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--strict", action="store_true", help="scipy operation order in the spline (no FMA)")
    ap.add_argument("--variant", type=int, default=0, help="kernel tuning variant (rows per thread / occupancy)")
    ap.add_argument("--arithmetic", default=None, choices=["fp64", "mixed"],
                    help="headline kernel: everything in FP64 (default, the reference's arithmetic) or the opt-in mixed "
                         "arithmetic (then dtype = f64+f32)")
    ap.add_argument("--no-fast", action="store_true", help="force the generic fused kernel")
    ap.add_argument("--small-storage", default="f64", choices=["auto", "f64"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mixed", action="store_true", help="skip the secondary measurement of the mixed kernel")
    ap.add_argument("--no-secondary", "--no-carrington", dest="no_secondary", action="store_true",
                    help="skip BASELINE configs[1], [3], [4] and the widened paths")
    ap.add_argument("--frames", type=int, default=SEQUENCE_FRAMES, help="frame searches of configs[4]")
    ap.add_argument("--carrington-variant", type=int, default=0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU arm's cube; the reference arm times a sample of lags")
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
