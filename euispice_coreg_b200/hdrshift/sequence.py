"""`SequenceAlignment` -- many small-FOV frames of one sequence against ONE large-FOV reference image.

BASELINE.json configs[4] (a batch of HRIEUV frames aligned to one FSI 174 image); the batch pattern is the one of
the reference's `jitter_correction.jitter_correction_imagers` (`jitter_correction/jitter_correction.py:14-174`):
one `Alignment` per frame with the same lag grid, results written per frame. The reference re-opens, re-uploads
(shared memory) and re-prepares everything for every frame. Here the large image is uploaded once and stays
resident in HBM; per frame only the small image (17 MB as float32), its candidate-header table and the one-time
cut of the large image onto the frame's grid are new. Kernel launches are asynchronous, so the host reads and
decodes frame k+1 while the device searches frame k, and the cube of frame k is fetched after frame k+1 has been
enqueued. With `torch.distributed` initialised the FRAMES are sharded over the ranks (each GPU: resident
reference, its own frames, the full lag grid -- SURVEY.md section 8e) and one all-gather assembles the cubes.

Per frame the result is exactly what `Alignment(large, frame, ...).align_using_helioprojective()` returns.

`align_using_carrington` is the same pipeline in the Carrington frame, the reference's default for jitter correction.
"fa": the large image is projected onto the Carrington grid once and stays resident; per frame only the small image,
the detector planes of each CROTA lag and the offset table are new. "sunpy": the large image is uploaded and
edge-padded once; per frame its solar-surface cut onto the frame's grid is new. Per frame the result is exactly what
`Alignment(large, frame, ...).align_using_carrington(...)` returns.
"""
from __future__ import annotations

import warnings

import numpy as np

from .._compat.wcs import TanWcs
from . import engine as _engine
from .alignment import Alignment, _Refs, carrington_dead_lags, warn_fa_units


_SIDE = {}


def _side_stream(device):
    """One upload / preparation stream per device for the life of the process (the caching allocator keeps a pool per
    stream: a fresh stream per call would re-allocate every per-frame buffer)."""
    torch = _engine._torch()
    key = str(device)
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=device)
    return _SIDE[key]


def frames_of_rank(n_frames, rank, world):
    """Round-robin frame sharding: rank r searches frames r, r + world, ..."""
    return list(range(rank, n_frames, world))


def gather_frame_cubes(cubes, n_frames, n_lags, device):
    """{frame index: flat cube} of this rank's frames -> the same for ALL frames, on every rank: one all-gather of a
    [frames per rank, n_lags] block (NCCL: `all_gather_into_tensor`; gloo, for the CPU tests of this logic: list
    `all_gather`). A rank without frames (more ranks than frames) contributes an all-NaN block of the same shape."""
    torch = _engine._torch()
    dist, rank, world = _engine._dist_info()
    if dist is None or world == 1 or n_frames == 0:
        return cubes
    per = (n_frames + world - 1) // world
    width = max(n_lags, 1)
    local = torch.full((per, width), float("nan"), dtype=torch.float64, device=device)
    for j, k in enumerate(frames_of_rank(n_frames, rank, world)):
        local[j, :n_lags] = torch.from_numpy(np.ascontiguousarray(cubes[k], dtype=np.float64).ravel()).to(device)
    if local.is_cuda:
        full = torch.empty((world * per, width), dtype=torch.float64, device=device)
        dist.all_gather_into_tensor(full, local)
    else:
        parts = [torch.empty((per, width), dtype=torch.float64) for _ in range(world)]
        dist.all_gather(parts, local)
        full = torch.cat(parts)
    full = full.cpu().numpy().reshape(world, per, -1)
    return {r + world * j: full[r, j, :n_lags] for r in range(world) for j in range(per) if r + world * j < n_frames}


def _lag_grid(a):
    return _engine.flat_lag_grid(a.lag_crval1, a.lag_crval2, a.lag_cdelt1, a.lag_cdelt2, a.lag_crota)


def _shape5(a):
    return len(a.lag_crval1), len(a.lag_crval2), len(a.lag_cdelt1), len(a.lag_cdelt2), len(a.lag_crota)


def _refs(a):
    refs = _Refs()
    refs.crval1_ref, refs.crval2_ref, refs.crota_ref = a.crval1_ref, a.crval2_ref, a.crota_ref
    refs.cdelt1_ref, refs.cdelt2_ref = a.cdelt1_ref, a.cdelt2_ref
    return refs


class _Frame:
    """One frame in flight: its host-side `Alignment`, the mask of lags that read 0.0, the device result [n_lags], the
    call that enqueues its search on the current stream and, optionally, the call that completes the result on the
    side stream before it is fetched."""
    __slots__ = ("a", "dead", "out", "search", "resolve")

    def __init__(self, a, dead, out, search, resolve=None):
        self.a, self.dead, self.out, self.search, self.resolve = a, dead, out, search, resolve


class SequenceAlignment:

    def __init__(self, large_fov_known_pointing: str, list_small_fov_to_correct, lag_crval1, lag_crval2,
                 lag_cdelt1=None, lag_cdelt2=None, lag_crota=None, small_fov_value_min=None,
                 small_fov_value_max=None, large_fov_window=-1, small_fov_window=-1, reprojection_order=2,
                 force_crota_0=False, unit_lag="arcsec", cdelt_semantics="reference", strict_arithmetic=False,
                 arithmetic=None, lag_solar_r=None):
        self.large_fov_known_pointing = large_fov_known_pointing
        self.list_small = list(list_small_fov_to_correct)
        self.kw = dict(lag_crval1=lag_crval1, lag_crval2=lag_crval2, lag_cdelt1=lag_cdelt1, lag_cdelt2=lag_cdelt2,
                       lag_crota=lag_crota, small_fov_value_min=small_fov_value_min,
                       small_fov_value_max=small_fov_value_max, large_fov_window=large_fov_window,
                       small_fov_window=small_fov_window, reprojection_order=reprojection_order,
                       force_crota_0=force_crota_0, unit_lag=unit_lag, cdelt_semantics=cdelt_semantics,
                       strict_arithmetic=strict_arithmetic, parallelism=True, arithmetic=arithmetic,
                       lag_solar_r=lag_solar_r)
        self.engine = None
        self.frames_per_s = None

    def _host_prepare(self, path_small, coordinate_frame="final_helioprojective"):
        """Everything `Alignment` does on the host before the device search, for one frame."""
        a = Alignment(self.large_fov_known_pointing, path_small, **self.kw)
        a.method, a.coordinate_frame = "correlation", coordinate_frame
        a.lon_ctype, a.lat_ctype, a.ang2pipi = "HPLN-TAN", "HPLT-TAN", True
        f_small = a._open_small()
        a.hdr_small = f_small[a.small_fov_window].header.copy()
        a._check_ant_create_pcij_matrix(a.hdr_small)
        h_small = f_small[a.small_fov_window]
        masking = a.small_fov_value_min is not None or a.small_fov_value_max is not None
        raw = h_small.raw_big_endian() if (not masking and hasattr(h_small, "raw_big_endian")) else None
        if raw is not None and raw.dtype == np.dtype(">f4") and raw.ndim == 2:
            a.data_small = raw      # as stored: swapped on the device; the all-NaN check happens there too (`finish`)
        else:
            a.data_small = a._float_image(h_small.data)
            a._set_removed_values_to_nan_in_datasmall(fov_limits=None, remove_fov_limits=None)
            if np.isnan(a.data_small).all():
                raise ValueError("minimum or maximum value have set all small FOV to nan")
        a._set_initial_header_values(True)
        if a.unit_lag != a.hdr_small["CUNIT1"] or a.unit_lag != a.hdr_small["CUNIT2"]:
            raise ValueError("lag.unit and cUNIT are not the same")
        return a

    def _open_reference(self):
        """Header (PCi_j checked) and image of the reference, read once for the whole sequence."""
        a0 = Alignment(self.large_fov_known_pointing, self.list_small[0] if self.list_small else "", **self.kw)
        f_large = a0._open_large()
        hdr_large = f_large[a0.large_fov_window].header.copy()
        a0._check_ant_create_pcij_matrix(hdr_large)
        return hdr_large, a0._float_image(f_large[a0.large_fov_window].data)

    def _engines(self, small_storage="f64"):
        """Two engines = two sets of per-frame device buffers (small image, per-frame planes or cut of the reference,
        lag tables, workspace) sharing the one resident reference: frame k+1 is uploaded and prepared on a side stream
        while frame k is being searched on the main stream."""
        return [_engine.LagSearchEngine(order=self.kw["reprojection_order"], strict=self.kw["strict_arithmetic"],
                                        arithmetic=self.kw["arithmetic"], small_storage=small_storage)
                for _ in range(2)]

    def align_using_helioprojective(self, return_type="AlignmentResults"):
        """-> list (one entry per frame, input order) of `AlignmentResults` or, with return_type="corr", of cubes
        float64 [n_crval1, n_crval2, n_cdelt1, n_cdelt2, n_crota, 1]."""
        torch = _engine._torch()
        engs = self._engines()
        # the reference image: read, checked and uploaded once
        hdr_large, data_large = self._open_reference()
        engs[0].set_large(data_large, TanWcs.from_header(hdr_large))
        engs[1].d_large, engs[1].wcs_large = engs[0].d_large, engs[0].wcs_large

        def prepare(path, e):
            a = self._host_prepare(path)
            e.set_small(a.data_small, pinned=True)
            e.cut_large(TanWcs.from_header(a.hdr_small))
            table, dead = e.hpc_lag_table(a.hdr_small, _refs(a), *_lag_grid(a), a.cdelt_semantics)
            tab_dev = e._upload(table, pinned=True)
            out = torch.empty(table.shape[0], dtype=torch.float64, device=e.device)
            # mixed arithmetic (opt-in): lags that tripped the kernel's guard are redone in FP64 on the side stream
            return _Frame(a, dead, out, lambda: e.evaluate(tab_dev, out), lambda: e.resolve_flags(tab_dev, out))

        return self._run(engs, prepare, return_type, "final_helioprojective")

    def _check_carrington(self, lonlims, latlims, shape, reference_date, method_carrington_reprojection,
                          size_deg_carrington):
        """Host-side checks of `align_using_carrington`, before any device work: what `Alignment` rejects, plus
        size_deg_carrington. Returns (reference header, reference image, reference date, d_solar_r)."""
        if method_carrington_reprojection not in ("fa", "sunpy"):
            raise ValueError("method_carrington_reprojection must be either 'fa' or 'sunpy")
        lag_solar_r = self.kw["lag_solar_r"]
        lag_solar_r = np.array([1.004]) if lag_solar_r is None else lag_solar_r
        if len(lag_solar_r) != 1:
            raise ValueError("lag_solar_r must hold exactly one value (the reference breaks on more, "
                             "alignment.py:646-660)")
        d_cdelt1, d_cdelt2 = (np.asarray([0.0] if self.kw[k] is None else self.kw[k], dtype=np.float64)
                              for k in ("lag_cdelt1", "lag_cdelt2"))
        if method_carrington_reprojection == "fa":
            if lonlims is None and latlims is None and size_deg_carrington is not None:
                raise ValueError("size_deg_carrington centres the grid on each frame's own CRLN_OBS / CRLT_OBS, so "
                                 "the reference would be projected onto a different grid for every frame: give an "
                                 "explicit lonlims / latlims / shape grid to SequenceAlignment")
            if lonlims is None or latlims is None or shape is None:
                raise ValueError("either set lonlims as None, or not. no in between.")
            carrington_dead_lags(d_cdelt1, d_cdelt2, self.kw["cdelt_semantics"])
        elif self.kw["cdelt_semantics"] not in ("reference", "intended"):
            raise ValueError("cdelt_semantics must be 'reference' or 'intended'")
        hdr_large, data_large = self._open_reference()
        if method_carrington_reprojection == "fa":
            if reference_date is None:
                if "DATE-AVG" not in hdr_large:
                    raise ValueError("Either provide a reference date manualy or the reference file header must have "
                                     "a DATE-AVG keyword.")
                reference_date = hdr_large["DATE-AVG"]
            if shape[0] * shape[1] > 25000000:
                warnings.warn(f"shape parameter is shape={shape}, which is very large."
                              "Computational time might significantly increase")
            warn_fa_units(hdr_large)
        else:
            Alignment._surface_frame(hdr_large)       # the observer keywords of the reference
            reference_date = None
        return hdr_large, data_large, reference_date, float(lag_solar_r[0])

    def align_using_carrington(self, lonlims=None, latlims=None, shape=None, reference_date=None,
                               method_carrington_reprojection="fa", return_type="AlignmentResults",
                               size_deg_carrington=None):
        """Carrington-frame search of every frame against the reference: the cube of each frame is the one of
        `Alignment(reference, frame, ...).align_using_carrington(...)` with the same arguments. -> list (one entry per
        frame, input order) of `AlignmentResults` or, with return_type="corr", of cubes float64
        [n_crval1, n_crval2, n_cdelt1, n_cdelt2, n_crota, 1].

        "fa": the reference is projected onto the Carrington grid once and stays resident; per frame, the detector
        planes of each distinct CROTA lag and the offset-window search. Only an explicit lonlims / latlims / shape grid
        is accepted (size_deg_carrington would centre a different grid on every frame). "sunpy": the reference is
        uploaded and edge-padded once; per frame, its solar-surface cut onto the frame's grid and the bilinear search
        (grid arguments are not read, as in `Alignment`)."""
        torch = _engine._torch()
        hdr_large, data_large, reference_date, d_solar_r = self._check_carrington(
            lonlims, latlims, shape, reference_date, method_carrington_reprojection, size_deg_carrington)
        engs = self._engines(small_storage="auto")

        if method_carrington_reprojection == "sunpy":
            engs[0].set_surface_large(data_large, TanWcs.from_header(hdr_large))
            engs[1].d_large_pad, engs[1].wcs_large = engs[0].d_large_pad, engs[0].wcs_large

            def prepare(path, e):
                a = self._host_prepare(path, "final_carrington")
                a.method_carrington_reprojection, a.hdr_large = "sunpy", hdr_large
                e.set_small(a.data_small, pinned=True)
                e.cut_surface(TanWcs.from_header(a.hdr_small), a._surface_frames(d_solar_r))
                table, dead = e.surface_lag_table(a.hdr_small, _refs(a), *_lag_grid(a), a.cdelt_semantics)
                tab_dev = e._upload(table, pinned=True)
                out = torch.empty(table.shape[0], dtype=torch.float64, device=e.device)
                return _Frame(a, dead, out, lambda: e.evaluate(tab_dev, out))
        else:
            engs[0].prepare_carrington_large(data_large, hdr_large, d_solar_r, lonlims, latlims, shape)
            engs[1].adopt_reference(engs[0])

            def prepare(path, e):
                a = self._host_prepare(path, "final_carrington")
                a.method_carrington_reprojection, a.hdr_large = "fa", hdr_large
                a.lonlims, a.latlims, a.shape, a.reference_date = lonlims, latlims, shape, reference_date
                warn_fa_units(a.hdr_small)
                d1, d2, d3, d4, d5 = _lag_grid(a)
                e.set_small(a.data_small, pinned=True)
                dead = carrington_dead_lags(d3, d4, a.cdelt_semantics)
                groups = [(e._upload(sel, pinned=True), planes, table, lag_ij)
                          for sel, planes, table, lag_ij in a._carrington_tables(e, _refs(a), d1, d2, d5, dead,
                                                                                 d_solar_r)]
                out = torch.zeros(d1.size, dtype=torch.float64, device=e.device)

                def search():
                    for sel_dev, planes, table, lag_ij in groups:
                        corr, _ = e.evaluate_patch_ordered(table, lag_ij, planes, pinned=True)
                        out.index_copy_(0, sel_dev, corr)
                return _Frame(a, dead, out, search)

        return self._run(engs, prepare, return_type, "final_carrington")

    def _run(self, engs, prepare, return_type, coordinate_frame):
        """The frame loop of every search frame. `prepare(path, engine)` runs with the side stream current once that
        engine's previous search has finished: host reading and preparation of the frame (overlapping the device
        search of the previous frame), its uploads and its one-time device steps; it returns a `_Frame`, whose search
        is then enqueued on the main stream. The cube of frame k is fetched after frame k+1 has been enqueued. With
        torch.distributed up, this rank searches its own frames (`frames_of_rank`) and the cubes are all-gathered:
        every rank returns all frames."""
        import time
        torch = _engine._torch()
        dist, rank, world = _engine._dist_info()
        n_frames = len(self.list_small)
        mine = frames_of_rank(n_frames, rank, world)
        eng = engs[0]
        self.engine = eng
        lag_solar_r = self.kw["lag_solar_r"]
        n_r = 1 if lag_solar_r is None else len(lag_solar_r)
        # the cube shape depends on the lag arrays only: every rank needs it for the all-gather, also one that gets no
        # frame (more ranks than frames)
        shape5 = None
        if n_frames and not mine:
            shape5 = _shape5(self._host_prepare(self.list_small[0], coordinate_frame))
        pending = None                                      # (frame index, _Frame, event after its search, engine)
        cubes = {}
        aligns = {}

        def finish(item):
            # fetch on the side stream, ordered after THIS frame's search only: the main stream may already be busy
            # with the next frame, and a copy enqueued there would make the host wait for that one too
            k, fr, evt, e = item
            with torch.cuda.device(fr.out.device), torch.cuda.stream(side):
                side.wait_event(evt)
                # (this engine's buffers are not touched again before the side stream reaches its next frame)
                if fr.resolve is not None:
                    fr.resolve()
                host = fr.out.cpu()
                if e.small_count() == 0:     # (this engine's statistics still describe frame k: see above)
                    raise ValueError("minimum or maximum value have set all small FOV to nan")
            cubes[k] = np.where(fr.dead, 0.0, host.numpy())
            aligns[k] = fr.a

        with torch.cuda.device(eng.device):
            main = torch.cuda.current_stream()
            side = _side_stream(eng.device)
            searched = [None, None]                         # per engine: event after its last search on `main`
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for n, k in enumerate(mine):
            e = engs[n & 1]
            with torch.cuda.device(e.device), torch.cuda.stream(side):
                if searched[n & 1] is not None:
                    side.wait_event(searched[n & 1])         # this engine's buffers are free again
                fr = prepare(self.list_small[k], e)
                ready = side.record_event()
            shape5 = _shape5(fr.a)
            with torch.cuda.device(e.device):
                main.wait_event(ready)
                fr.search()                                 # asynchronous: returns once the kernels are enqueued
                searched[n & 1] = main.record_event()
            fr.a.data_small = None
            if pending is not None:
                finish(pending)
            pending = (k, fr, searched[n & 1], e)
        if pending is not None:
            finish(pending)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        self.frames_per_s = len(mine) / dt if dt > 0 and mine else None
        # assemble: every rank ends with all cubes (one all-gather of [frames per rank, n_lags])
        n_lags = int(np.prod(shape5)) if shape5 is not None else 0
        cubes = gather_frame_cubes(cubes, n_frames, n_lags, eng.device)
        out = []
        for k in range(n_frames):
            cube = cubes[k].reshape(shape5 + (1,))
            if n_r > 1:         # (helioprojective frame: `Alignment` repeats the cube along the solar-radius axis)
                cube = np.repeat(cube, n_r, axis=5)
            if return_type == "corr":
                out.append(cube)
                continue
            a = aligns.get(k)
            if a is None:                                   # frame searched by another rank: host prep only
                a = self._host_prepare(self.list_small[k], coordinate_frame)
                a.data_small = None
            out.append(a._wrap_results(cube, "AlignmentResults"))
        return out
