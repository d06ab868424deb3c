"""Device engine under `Alignment._find_best_header_parameters` (the seam of SURVEY.md section 8b).

The reference fans the flattened lag list out over `multiprocessing.Process` workers that share the
two images through POSIX shared memory (`hdrshift/alignment.py:634-756`). Here the images are uploaded
once and stay resident in HBM, the lag list becomes a table of per-lag constants, and one fused kernel
launch (per <= `max_lags_per_launch` lags) evaluates the whole table. With `torch.distributed`
initialised (one process per GPU), every rank holds both images, evaluates a contiguous slice of the
C-ordered lag list -- the same decomposition as `np.array_split` at `alignment.py:677-687` -- and one
all-gather assembles the cube.
"""
from __future__ import annotations

import math
import os

import numpy as np

from .. import _ext
from .._compat import units
from .._compat.wcs import CarWcs, TanWcs

R2D = 180.0 / math.pi
D2R = math.pi / 180.0
R_SUN_M = 695700000.0  # astropy.constants.R_sun.value (IAU 2015 nominal), utils/rectify.py:405


def _torch():
    import torch
    return torch


def flat_lag_grid(lag_crval1, lag_crval2, lag_cdelt1, lag_cdelt2, lag_crota):
    """C-order flattening of the 5-D lag meshgrid, crval1 slowest (`alignment.py:667-674`)."""
    g = np.meshgrid(np.asarray(lag_crval1, dtype=np.float64), np.asarray(lag_crval2, dtype=np.float64),
                    np.asarray(lag_cdelt1, dtype=np.float64), np.asarray(lag_cdelt2, dtype=np.float64),
                    np.asarray(lag_crota, dtype=np.float64), indexing="ij")
    return [a.ravel() for a in g]


def shard_bounds(n_lags: int, world: int):
    """Contiguous equal slices of the padded lag list: rank r owns [r*c, (r+1)*c) with c = ceil(n/world)."""
    c = (n_lags + world - 1) // world if world > 0 else n_lags
    return c, [(min(r * c, n_lags), min((r + 1) * c, n_lags)) for r in range(world)]


def shifted_pc(hdr, crota_ref, d_cdelt1, d_cdelt2, d_crota, cdelt1, cdelt2, wcs_cls=TanWcs):
    """PCi_j of the shifted header, vectorised over lags (`_shift_header`, `alignment.py:401-468`).
    Lags that touch none of CDELT/CROTA keep the header's own PC."""
    change = (d_cdelt1 != 0.0) | (d_cdelt2 != 0.0) | (d_crota != 0.0)
    crot = np.where(d_crota != 0.0, crota_ref + d_crota, crota_ref)
    rho = np.deg2rad(crot)
    lam = cdelt2 / cdelt1
    own = wcs_cls.from_header(hdr)   # PCi_j as wcslib would read them (identity when absent)
    pc11 = np.where(change, np.cos(rho), own.pc11)
    pc22 = np.where(change, np.cos(rho), own.pc22)
    pc12 = np.where(change, -lam * np.sin(rho), own.pc12)
    pc21 = np.where(change, (1 / lam) * np.sin(rho), own.pc21)
    return pc11, pc12, pc21, pc22


def _shifted_header_constants(hdr_small, refs, d_crval1, d_crval2, d_cdelt1, d_cdelt2, d_crota, cdelt_semantics,
                              wcs_cls=TanWcs):
    """Per-lag constants of `_shift_header` (`alignment.py:401-468`) in degrees, vectorised over lags."""
    w0 = wcs_cls.from_header(hdr_small)
    s1, s2 = w0.unit_scale1, w0.unit_scale2
    n = d_crval1.size
    crval1 = (refs.crval1_ref + d_crval1) * s1
    crval2 = (refs.crval2_ref + d_crval2) * s2
    cdelt1_h = np.full(n, float(hdr_small["CDELT1"]))
    cdelt2_h = np.full(n, float(hdr_small["CDELT2"]))
    dead = np.zeros(n, dtype=bool)
    if cdelt_semantics == "intended":
        cdelt1_h = np.where(d_cdelt1 != 0.0, refs.cdelt1_ref + d_cdelt1, cdelt1_h)
        cdelt2_h = np.where(d_cdelt2 != 0.0, refs.cdelt2_ref + d_cdelt2, cdelt2_h)
    elif cdelt_semantics == "reference":
        dead = d_cdelt2 != 0.0
    else:
        raise ValueError("cdelt_semantics must be 'reference' or 'intended'")
    pc = shifted_pc(hdr_small, refs.crota_ref, d_cdelt1, d_cdelt2, d_crota, cdelt1_h, cdelt2_h, wcs_cls)
    return w0, crval1, crval2, cdelt1_h * s1, cdelt2_h * s2, pc, dead


def tan_lag_table(hdr_small, refs, d_crval1, d_crval2, d_cdelt1, d_cdelt2, d_crota, alpha_ref_deg,
                  cdelt_semantics="reference"):
    """[n_lags, 10] float64 rows of `CoregLagTan` + a mask of lags the reference cannot evaluate.

    `refs` carries crval1_ref, crval2_ref, crota_ref, cdelt1_ref, cdelt2_ref (header units).
    cdelt_semantics="reference": a CDELT1 lag only triggers the PC rebuild, a non-zero CDELT2 lag kills the
    reference's worker (cube entry stays 0.0) -> reported in the returned `dead` mask (SURVEY App. B1).
    cdelt_semantics="intended": CDELTi = ref + lag, then PC rebuild with the new CDELT2/CDELT1.
    """
    w0, crval1, crval2, cd1, cd2, (pc11, pc12, pc21, pc22), dead = _shifted_header_constants(
        hdr_small, refs, d_crval1, d_crval2, d_cdelt1, d_cdelt2, d_crota, cdelt_semantics)
    n = d_crval1.size
    # forward matrix [deg/pixel] and its inverse, times 180/pi (the kernel's plane coordinates are radians)
    f11, f12 = cd1 * pc11, cd1 * pc12
    f21, f22 = cd2 * pc21, cd2 * pc22
    det = f11 * f22 - f12 * f21
    i11, i12, i21, i22 = f22 / det, -f12 / det, -f21 / det, f11 / det
    # native-longitude rotation by LONPOLE folded in: (xp, yp) = (-cp xi + sp eta, -sp xi - cp eta)
    sp, cp = math.sin(w0.lonpole * D2R), math.cos(w0.lonpole * D2R)
    if w0.lonpole == 180.0:
        sp, cp = 0.0, -1.0
    m11 = (i11 * -cp + i12 * -sp) * R2D
    m12 = (i11 * sp + i12 * -cp) * R2D
    m21 = (i21 * -cp + i22 * -sp) * R2D
    m22 = (i21 * sp + i22 * -cp) * R2D
    tab = np.empty((n, _ext.LAG_TAN_DOUBLES), dtype=np.float64)
    da = (crval1 - alpha_ref_deg) * D2R
    tab[:, 0] = np.sin(da)
    tab[:, 1] = np.cos(da)
    tab[:, 2] = np.sin(crval2 * D2R)
    tab[:, 3] = np.cos(crval2 * D2R)
    tab[:, 4], tab[:, 5], tab[:, 6], tab[:, 7] = m11, m12, m21, m22
    tab[:, 8] = w0.crpix1 - 1.0
    tab[:, 9] = w0.crpix2 - 1.0
    return tab, dead


def tan_wcs_table(hdr_small, refs, d_crval1, d_crval2, d_cdelt1, d_cdelt2, d_crota, cdelt_semantics="reference"):
    """[n_lags, 11] float64 rows of `CoregTanWcs`: the candidate headers themselves (output of `_shift_header`,
    `alignment.py:401-468`, as wcslib would hold them, degrees). Input of the homography kernel
    (`coreg_hpc_lag_corr_wcs`), which derives its per-lag 3x3 matrix on the device."""
    w0, crval1, crval2, cd1, cd2, (pc11, pc12, pc21, pc22), dead = _shifted_header_constants(
        hdr_small, refs, d_crval1, d_crval2, d_cdelt1, d_cdelt2, d_crota, cdelt_semantics)
    n = d_crval1.size
    tab = np.empty((n, _ext.TAN_WCS_DOUBLES), dtype=np.float64)
    tab[:, 0], tab[:, 1] = w0.crpix1, w0.crpix2
    tab[:, 2], tab[:, 3] = cd1, cd2
    tab[:, 4], tab[:, 5], tab[:, 6], tab[:, 7] = pc11, pc12, pc21, pc22
    tab[:, 8], tab[:, 9] = crval1, crval2
    tab[:, 10] = w0.lonpole
    return tab, dead


def car_lag_table(hdr_small, refs, d_crval1, d_crval2, d_cdelt1, d_cdelt2, d_crota, cdelt_semantics="reference"):
    """[n_lags, 16] float64 rows of `CoregLagCar` for candidate headers of a Carrington map (CRLN-CAR / CRLT-CAR):
    `_shift_header` (`alignment.py:401-468`) followed by what `WCS(hdr_shifted)` derives in wcslib's celset -- the
    native pole of every candidate, as a sphere rotation. The returned mask also flags candidates wcslib rejects
    (an explicit LONPOLE that admits no native pole once CRVAL2 changes sign): the reference's worker dies on them."""
    w0, crval1, crval2, cd1, cd2, (pc11, pc12, pc21, pc22), dead = _shifted_header_constants(
        hdr_small, refs, d_crval1, d_crval2, d_cdelt1, d_cdelt2, d_crota, cdelt_semantics, wcs_cls=CarWcs)
    tab, bad = CarWcs.lag_rows(crval1, crval2, cd1, cd2, pc11, pc12, pc21, pc22, w0.crpix1, w0.crpix2, w0.lonpole,
                               w0.latpole)
    return tab, dead | bad


OFFSET_CHUNK = 256   # lags per block of the Carrington-frame kernel (one per thread, csrc/coreg_lag_offset.cu)


def offset_patch_order(i1, i2, group=None, patch=(16, 16), sub=(16, 2)):
    """Order in which the Carrington-frame kernel wants a CRVAL lag list: its blocks take 256 consecutive lags (one per
    thread) and stage the part of the small image those lags can touch, so consecutive lags must be neighbours in
    the detector plane. Lags are grouped into patches of 16 x 16 grid indices (i1 = CRVAL1 index, i2 = CRVAL2 index),
    inside a patch into sub-patches of 16 x 2 (one warp each: the lane layout with the fewest shared-memory bank
    conflicts, csrc/coreg_lag_offset.cu:OffBox); every patch is padded to 256 slots so that a block
    never straddles two patches. `group`: optional integer key of lags that must not share a patch (e.g. the CDELT
    index). Returns (slot_of_lag [n], n_slots): lag k goes to row slot_of_lag[k] of a [n_slots, 2] table whose
    other rows are NaN (dummy lags: evaluate nothing)."""
    i1 = np.asarray(i1, dtype=np.int64)
    i2 = np.asarray(i2, dtype=np.int64)
    g = np.zeros_like(i1) if group is None else np.asarray(group, dtype=np.int64)
    if i1.size:      # patches start at the list's own first indices: a rank's slice of the grid gets no ragged leading patch
        i1, i2 = i1 - i1.min(), i2 - i2.min()
    p1, p2 = i1 // patch[0], i2 // patch[1]
    q1, q2 = i1 % patch[0], i2 % patch[1]
    s1, s2 = q1 // sub[0], q2 // sub[1]
    # position inside the patch: sub-patch major, then row-major inside the sub-patch (CRVAL1 index fastest)
    inner = ((s2 * (patch[0] // sub[0]) + s1) * (sub[0] * sub[1]) + (q2 % sub[1]) * sub[0] + (q1 % sub[0]))
    _, pid = np.unique(np.stack([g, p1, p2], axis=1), axis=0, return_inverse=True)
    slot = pid.ravel() * (patch[0] * patch[1]) + inner
    n_slots = int((pid.max() + 1) * patch[0] * patch[1]) if i1.size else 0
    if i1.size and np.unique(slot).size != slot.size:   # repeated (i1, i2) pairs inside one group: no structure to use
        return np.arange(i1.size, dtype=np.int64), int(i1.size)
    return slot, n_slots


def _dist_info():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist, dist.get_rank(), dist.get_world_size()
    except Exception:
        pass
    return None, 0, 1


def gather_slices(local, n_total, chunk):
    """All-gather equal `chunk`-sized slices (last ones padded) into one [n_total] tensor.
    NCCL: a single `all_gather_into_tensor` (in place: every rank's slice is already at its offset).
    gloo (CPU tests of the host logic): list-based `all_gather`."""
    torch = _torch()
    dist, rank, world = _dist_info()
    if dist is None or world == 1:
        return local[:n_total]
    full = torch.empty(chunk * world, dtype=local.dtype, device=local.device)
    send = local
    if send.numel() != chunk:
        pad = torch.full((chunk,), float("nan"), dtype=local.dtype, device=local.device)
        pad[:send.numel()] = send
        send = pad
    if local.is_cuda:
        dist.all_gather_into_tensor(full, send.contiguous())
    else:
        parts = [torch.empty(chunk, dtype=local.dtype) for _ in range(world)]
        dist.all_gather(parts, send.contiguous())
        full = torch.cat(parts)
    return full[:n_total]


class LagSearchEngine:
    """Resident images + workspaces for one (large, small) pair on the current CUDA device."""

    max_workspace_bytes = 4 << 30   # 8128 lags of a 2048^2 grid per launch (525 KB of warp records per lag)

    # the reference evaluates every sample in FP64 (scipy accumulates in double, utils/Util.py:98-102) and only then
    # stores it as float32 (alignment.py:1024): FP64 is the default, "mixed" an explicit opt-in
    default_arithmetic = "fp64"

    def __init__(self, order=2, strict=False, device=None, variant=0, small_storage="f64", no_fast=False,
                 arithmetic=None):
        """arithmetic: "fp64" (default: everything in FP64, the reference's arithmetic) or "mixed" (opt-in: FP64
        projection, FP32 spline on the pivot-centred float32 payload of the small image; applies to the homography
        kernel when every small-image pixel is a float32 value; lags whose error model exceeds 1e-7 in r are
        re-evaluated in FP64, see `resolve_flags`). None: the COREG_ARITHMETIC environment variable, else
        `default_arithmetic`."""
        torch = _torch()
        arithmetic = arithmetic or os.environ.get("COREG_ARITHMETIC") or self.default_arithmetic
        if arithmetic not in ("fp64", "mixed"):
            raise ValueError('arithmetic must be "fp64" or "mixed"')
        self.arithmetic = arithmetic
        self.small32 = None      # float32 payload of the small image, centred on its float32 pivot (mixed arithmetic)
        self.lag_flags = None    # int32 [n]: lags of the last mixed `evaluate` that tripped the kernel's guard
        self.flagged_lags = 0    # how many lags `resolve_flags` re-evaluated in FP64 (diagnostic)
        self.pure_shift_hint = False   # set by `hpc_lag_table`: the lag grid holds CRVAL shifts only
        _ext.load()  # fail loudly when the CUDA library is missing
        if not torch.cuda.is_available():
            raise _ext.CoregLibraryError("no CUDA device: the pointing search has no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.order = int(order)
        self.strict = bool(strict)
        self.variant, self.no_fast = int(variant), bool(no_fast)
        self.flags = _ext.make_flags(strict, variant, no_fast=no_fast)
        self.small_storage = small_storage
        # statistics block [4, 2]: rows = mean (the pivot), count, max |v|, RMS about the pivot; columns = ref, small
        self.stats = torch.zeros((_ext.STATS_ROWS, 2), dtype=torch.float64, device=self.device)
        self.pivots = self.stats[0]
        self.ref = None        # large image on the common grid
        self.frame = None      # "hpc" | "car" | "carrington", set by the prepare_* call
        self.small = None
        self.planes = None     # TAN: [3, gny, gnx]; Carrington: (tx, ty)
        self._work = None
        self.d_large = None
        self.wcs_large = None
        self.last_launches = 0

    # ---- uploads -----------------------------------------------------------------------------
    def _upload(self, arr, pinned=False):
        torch = _torch()
        arr = np.asarray(arr)
        if arr.dtype == np.dtype(">f4"):
            # a FITS BITPIX -32 payload as stored (possibly a read-only view of the memory-mapped file): the bytes go
            # up as they are and are swapped on the device
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")      # "non-writable array": it is only read
                t = torch.from_numpy(np.ascontiguousarray(arr).view("<i4"))
            if pinned:
                t = t.pin_memory()
            with torch.cuda.device(self.device):
                return _ext.bswap32_to_float32(t.to(self.device, non_blocking=pinned))
        t = torch.from_numpy(np.ascontiguousarray(arr))
        if pinned:
            t = t.pin_memory()
        return t.to(self.device, non_blocking=pinned)

    @staticmethod
    def _native_float(arr):
        """float32 / float64 arrays go up as they are (float32 -> float64 is exact, so FITS BITPIX -32 payloads need
        no widening on the host), big-endian float32 as stored; anything else is converted to float64 like the
        reference does."""
        arr = np.asarray(arr)
        if arr.dtype == np.dtype(">f4"):
            return arr
        if arr.dtype not in (np.float32, np.float64) or not arr.dtype.isnative:
            arr = arr.astype(np.float64)
        return arr

    def set_small(self, data_small, pinned=False):
        """Small image (NaN for masked pixels), float32 or float64 on the host. small_storage="f64" (default): kept
        as float64 on the device (a float32 input is uploaded as float32 and widened there); "auto": kept as float32
        when the input is float32 -- half the gather traffic, same values, but 9 f32->f64 conversions per sample on the
        quarter-rate conversion pipe and no homography kernel: measured slower on B200 (profiles/r1_k1_tuning.md)."""
        torch = _torch()
        small = self._upload(self._native_float(data_small), pinned=pinned)
        self.small32 = None
        self._mixed_pair = None
        mixed = self.arithmetic == "mixed" and self.small_storage == "f64" and not self.strict and self.order == 2
        with torch.cuda.device(self.device):
            if small.dtype == torch.float32 and self.small_storage == "f64":
                s32 = small
                small = _ext.image_stats(s32, self.stats, 1, widen=True)    # pivot + float64 copy in one pass
                if mixed:
                    self.small32 = _ext.center_f32(s32, self.stats, 1)
            else:
                _ext.image_stats(small, self.stats, 1)
                if mixed and small.dtype == torch.float64:
                    # a float64 input whose pixels are all float32 values (an integer FITS payload, a float32 image
                    # the caller widened): the mixed kernel sees exactly the same image
                    s32 = small.to(torch.float32)
                    if bool(((s32.to(torch.float64) == small) | torch.isnan(small)).all()):
                        self.small32 = _ext.center_f32(s32.contiguous(), self.stats, 1)
        self.small = small

    def small_count(self):
        """Number of finite pixels of the small image (from its statistics pass; one 8-byte D2H)."""
        return int(self.stats[1, 1].item())

    # float32 moments need headroom on both sides: the mixed kernel squares pivot-centred pixel values and sums 16 of
    # them in float32, so images whose magnitudes sit near the ends of the float32 range (|v| beyond 1e12, or nothing
    # above 1e-9: flux units far from DN/s or W/m2/sr/nm) are searched by the all-FP64 kernel from the start. (The
    # per-lag guard of the finalize kernel would catch them too -- underflowing squares make the sampled variance
    # vanish -- at the price of running the search twice.)
    MIXED_ABS_RANGE = (1e-9, 1e12)

    def _mixed_applies(self):
        """Mixed arithmetic for the current (small, ref) pair: requested, a centred float32 twin of the small image
        exists, and both images leave the float32 sums enough range. Decided once per pair (one 64-byte D2H + sync)."""
        if self.arithmetic != "mixed" or self.small32 is None or self.ref is None:
            return False
        # (the pair is identified by the tensor objects themselves: a new image may land on a recycled address)
        if getattr(self, "_mixed_pair", None) is None or self._mixed_pair[0] is not self.small32 \
                or self._mixed_pair[1] is not self.ref:
            self._mixed_pair = (self.small32, self.ref)
            lo, hi = self.MIXED_ABS_RANGE
            mags = self.stats[2].tolist()
            self._mixed_ok = all(lo < m < hi for m in mags)
        return self._mixed_ok

    # ---- helioprojective ------------------------------------------------------------------------
    def set_large(self, data_large, wcs_large: TanWcs, origin=(0, 0)):
        """Upload the large image once; it stays resident for any number of `cut_large` calls (frame sequences).
        origin = (x0, y0): `data_large` is the window [y0:, x0:] of the image `wcs_large` describes."""
        torch = _torch()
        with torch.cuda.device(self.device):
            self.d_large = self._upload(self._native_float(data_large))
        self.wcs_large = wcs_large
        self.large_origin = (int(origin[0]), int(origin[1]))

    @staticmethod
    def large_window(wcs_large: TanWcs, wcs_small: TanWcs, shape_large, margin=4):
        """(x0, x1, y0, y1): the part of the large image the one-time cut onto the small grid can touch. Both maps are
        gnomonic, so large-image coordinates are a PROJECTIVE function of small-grid coordinates: along a straight edge
        of the grid each is a linear-fractional function of one variable, hence monotonic, and a projective map has no
        interior extrema -- the extremes over the grid are those of its four CORNERS (mapped on the host: 4 points
        instead of the 4 (nx + ny) edge pixels, 1 ms of numpy per pair on the GPU box's host). The denominator of the map
        is linear over the grid, so corners in front of the large image's tangent plane (finite coordinates) put the
        whole grid there. `margin` covers the spline support. None when the window cannot be bounded."""
        nx, ny = int(wcs_small.naxis1), int(wcs_small.naxis2)
        ny_l, nx_l = int(shape_large[0]), int(shape_large[1])
        ex = np.array([0.0, nx - 1.0, 0.0, nx - 1.0])
        ey = np.array([0.0, 0.0, ny - 1.0, ny - 1.0])
        lon, lat = wcs_small.pixel_to_world(ex, ey)
        xl, yl = wcs_large.world_to_pixel(lon, lat)
        if not (np.all(np.isfinite(xl)) and np.all(np.isfinite(yl))):
            return None
        x0 = max(0, int(np.floor(xl.min())) - margin)
        x1 = min(nx_l, int(np.ceil(xl.max())) + margin + 1)
        y0 = max(0, int(np.floor(yl.min())) - margin)
        y1 = min(ny_l, int(np.ceil(yl.max())) + margin + 1)
        if x1 - x0 < 4 or y1 - y0 < 4:      # no overlap worth cropping to: keep the whole image
            return None
        return x0, x1, y0, y1

    def cut_large(self, wcs_small: TanWcs):
        """One-time part of a helioprojective search: world grid of the unshifted small grid (K3), the resident
        large image resampled onto it as float32 (K2, `_create_submap_of_large_data`, `alignment.py:987-1016`) and
        the ref pivot. The common grid of the search is this unshifted small grid (`alignment.py:649-651, 1000`)."""
        torch = _torch()
        with torch.cuda.device(self.device):
            # world grid -> large-image coordinates (computed as in the full image; the integer origin of the uploaded
            # window comes off exactly, so every tap and every weight is the one the full image would give) -> spline
            # sample -> float32, in one kernel: the bits of tan_pix2world -> tan_world2pix -> map_coordinates
            # (tests/test_gpu_parity.py), without the coordinate planes
            self.ref = _ext.hpc_cut(wcs_small, self.wcs_large, self.d_large, getattr(self, "large_origin", (0, 0)),
                                    self.order)
            self.planes = None          # trig planes of the generic kernel: built on first use (`_hpc_planes`)
            self.grid_wcs = wcs_small
            self.alpha_ref_deg = wcs_small.crval1
            self.delta_ref_deg = wcs_small.crval2
            _ext.image_stats(self.ref, self.stats, 0)
        self.frame = "hpc"

    def prepare_hpc(self, data_large, wcs_large: TanWcs, wcs_small: TanWcs):
        """`set_large` + `cut_large` for a single pair; the large image is released afterwards. Only the window of
        the large image the small grid can reach is converted (when `data_large` is a lazily read FITS HDU:
        `fits_lite.ImageHDU.read_window`) and uploaded: a few hundred pixels across for an HRIEUV field inside a full-disc FSI image."""
        shape = data_large.shape
        win = self.large_window(wcs_large, wcs_small, shape) if len(shape) == 2 else None
        if win is None:
            full = data_large.data if hasattr(data_large, "read_window") else data_large
            self.set_large(full, wcs_large)
        else:
            x0, x1, y0, y1 = win
            part = data_large.read_window(y0, y1, x0, x1) if hasattr(data_large, "read_window") \
                else data_large[y0:y1, x0:x1]
            self.set_large(part, wcs_large, origin=(x0, y0))
        self.cut_large(wcs_small)
        self.d_large = None
        self.large_origin = (0, 0)

    # ---- solar-surface reprojection (method_carrington_reprojection="sunpy") ------------------------------------
    def prepare_surface(self, data_large, wcs_large: TanWcs, wcs_small: TanWcs, frames):
        """One-time part of the "sunpy" Carrington search (`alignment.py:939-985`, first branch): the large image on the
        grid of the small one through the solar-surface change of observer (`coreg_surface_cut`), float64; the
        edge-padded small image and the grid's trig planes for the bilinear per-lag search. `frames`:
        `_ext.CoregSurfaceFrames`. Restated third-party algorithm, parity unpinned (oracle/surface_reproject.py)."""
        self.set_surface_large(data_large, wcs_large)
        self.cut_surface(wcs_small, frames)
        self.d_large_pad = None

    def set_surface_large(self, data_large, wcs_large: TanWcs):
        """Upload the large image once and edge-pad it once; it stays resident for any number of `cut_surface` calls
        (frame sequences)."""
        torch = _torch()
        with torch.cuda.device(self.device):
            d_large = self._upload(self._native_float(data_large))
            self.d_large_pad = _ext.pad_edge(d_large)
            del d_large
        self.wcs_large = wcs_large

    def cut_surface(self, wcs_small: TanWcs, frames):
        """Per-pair part of the "sunpy" search, after `set_small`: the resident padded large image cut onto the small
        grid, the grid's trig planes and the edge-padded small image."""
        torch = _torch()
        with torch.cuda.device(self.device):
            self.ref = _ext.surface_cut(wcs_small, self.wcs_large, self.d_large_pad, frames)
            lng, lat = _ext.tan_pix2world(wcs_small, wcs_small.naxis1, wcs_small.naxis2, True, self.device)
            self.planes = _ext.tan_trig_planes(lng, lat, wcs_small.crval1)
            del lng, lat
            self.small_pad = _ext.pad_edge(self.small)
            self.grid_wcs = wcs_small
            self.alpha_ref_deg = wcs_small.crval1
            self.delta_ref_deg = wcs_small.crval2
            _ext.image_stats(self.ref, self.stats, 0)
        self.frame = "surface"

    def surface_lag_table(self, hdr_small, refs, d1, d2, d3, d4, d5, cdelt_semantics="reference"):
        """`CoregLagTanEdge` rows: the candidate headers as `CoregLagTan` + the bounds of reproject's edge rule."""
        self.pure_shift_hint = False
        tab, dead = tan_lag_table(hdr_small, refs, d1, d2, d3, d4, d5, self.alpha_ref_deg, cdelt_semantics)
        out = np.empty((tab.shape[0], _ext.LAG_TAN_EDGE_DOUBLES), dtype=np.float64)
        out[:, :_ext.LAG_TAN_DOUBLES] = tab
        out[:, _ext.LAG_TAN_DOUBLES] = self.small.shape[1] - 0.5
        out[:, _ext.LAG_TAN_DOUBLES + 1] = self.small.shape[0] - 0.5
        return out, dead

    # ---- Carrington maps as inputs (CRLN-CAR / CRLT-CAR) -----------------------------------------------------
    def prepare_car(self, data_large, wcs_large: CarWcs, wcs_small: CarWcs):
        """One-time part of `align_using_initial_carrington` (`alignment.py:344-399, 987-1016`): Carrington
        coordinates of the unshifted small grid, the large map resampled onto it as float32, the grid's unit-vector
        planes and the ref pivot."""
        torch = _torch()
        with torch.cuda.device(self.device):
            d_large = self._upload(self._native_float(data_large))
            lng, lat = _ext.car_pix2world(wcs_small.lag_row(), wcs_small.naxis1, wcs_small.naxis2, self.device)
            x, y = _ext.car_world2pix(wcs_large.lag_row(), lng, lat)
            self.ref = _ext.map_coordinates(d_large, y, x, self.order, float("nan"), torch.float32)
            self.planes = _ext.tan_trig_planes(lng, lat, 0.0)
            del x, y, lng, lat, d_large
            self.grid_wcs = wcs_small
            _ext.image_stats(self.ref, self.stats, 0)
        self.frame = "car"
        # launch shape of the generic kernel: the default 4 pixels x 4 CTAs / SM (64 registers, the atan2 temporaries
        # spill to L1-resident local memory) measured faster than 8 x 2 with 128 registers: 101.9 vs 115.7 ms on
        # 2048 x 1024 maps, 3600 lags (profiles/r1_widened_kernels.md)
        self.flags = _ext.make_flags(self.strict, int(os.environ.get("COREG_CAR_VARIANT", "0")), no_fast=self.no_fast)

    def _hpc_planes(self):
        """Lag-independent trig planes of the generic helioprojective kernel (101 MB at 2048^2), built lazily:
        the homography kernel does not need them."""
        if self.planes is None:
            torch = _torch()
            w = self.grid_wcs
            with torch.cuda.device(self.device):
                lng, lat = _ext.tan_pix2world(w, w.naxis1, w.naxis2, True, self.device)
                self.planes = _ext.tan_trig_planes(lng, lat, w.crval1)
        return self.planes

    def hpc_fast_eligible(self):
        """The homography kernel covers spline order 2 with FMA arithmetic on images of at least 3x3 pixels."""
        torch = _torch()
        return (self.order == 2 and not self.strict and not self.no_fast and self.small is not None
                and self.small.dtype == torch.float64 and min(self.small.shape) >= 3)

    def hpc_lag_table(self, hdr_small, refs, d1, d2, d3, d4, d5, cdelt_semantics="reference"):
        """Host lag table for `search` in the helioprojective frame + the mask of lags the reference cannot
        evaluate: candidate-header rows for the homography kernel when it applies, `CoregLagTan` rows otherwise."""
        # True when every lag is a pure CRVAL shift (no column segment of the rolling kernel changes a floor out of
        # step; rotated / rescaled lags send such segments through the kernel's adaptive segment): selects the kernel
        # flavour in `evaluate`. Set from the WHOLE lag grid: every shard must launch the same flavour for the cube to
        # be bit-identical for any GPU count.
        self.pure_shift_hint = not (np.any(np.asarray(d3)) or np.any(np.asarray(d4)) or np.any(np.asarray(d5)))
        if self.hpc_fast_eligible():
            return tan_wcs_table(hdr_small, refs, d1, d2, d3, d4, d5, cdelt_semantics)
        return tan_lag_table(hdr_small, refs, d1, d2, d3, d4, d5, self.alpha_ref_deg, cdelt_semantics)

    # ---- Carrington --------------------------------------------------------------------------------
    @staticmethod
    def carrington_vectors(lonlims, latlims, shape, crln_obs):
        """The float32 half of `Rectifier.__call__` + `SphericalTransform.forward` on the separable grid
        (`utils/rectify.py:345-349, 876-877`), evaluated with NumPy exactly as the reference does."""
        lon = np.linspace(lonlims[0], lonlims[1], shape[0], dtype=np.float32)
        lat = np.linspace(latlims[0], latlims[1], shape[1], dtype=np.float32)
        lon_r = np.radians(lon) - np.radians(crln_obs)      # float32 - float64 scalar -> float64
        lat_r = np.radians(lat)                             # float32
        return (np.sin(lon_r), np.cos(lon_r),
                np.sin(lat_r).astype(np.float64), np.cos(lat_r).astype(np.float64))

    @staticmethod
    def carrington_struct(hdr, d_solar_r):
        """`CoregCarrington` of one header: the constants of `CarringtonTransform.__init__` (`utils/rectify.py:377-415`)."""
        roll_deg = hdr["CROTA"] if "CROTA" in hdr else hdr["CROTA2"]
        return _ext.CoregCarrington(float(np.radians(hdr["CRLN_OBS"])), float(np.radians(hdr["CRLT_OBS"])),
                                    float(np.radians(roll_deg)), float(hdr["DSUN_OBS"] / (d_solar_r * R_SUN_M)),
                                    float(hdr["CDELT1"]), float(hdr["CDELT2"]))

    def carrington_planes(self, hdr, d_solar_r, lonlims, latlims, shape):
        """(tx, ty) detector-plane planes of one header on the Carrington grid (K5 coordinates)."""
        c = self.carrington_struct(hdr, d_solar_r)
        vec = self.carrington_vectors(lonlims, latlims, shape, hdr["CRLN_OBS"])
        sinlon, coslon, sinlat, coslat = (self._upload(v) for v in vec)
        return _ext.carrington_planes(c, sinlon, coslon, sinlat, coslat)

    @staticmethod
    def carrington_offset(hdr, crval1, crval2, roll_deg):
        """x0, y0 of `CarringtonTransform.__init__` (`utils/rectify.py:394-404`), vectorised over lags."""
        cos = np.cos(np.radians(roll_deg))
        sin = np.sin(np.radians(roll_deg))
        dx = cos * crval1 + sin * crval2
        dy = -sin * crval1 + cos * crval2
        return (hdr["CRPIX1"] - 1) - dx / hdr["CDELT1"], (hdr["CRPIX2"] - 1) - dy / hdr["CDELT2"]

    def prepare_carrington_large(self, data_large, hdr_large, d_solar_r, lonlims, latlims, shape):
        """Large image -> Carrington grid, float64, -32762 fill -> NaN (`alignment.py:646-648, 889-901`)."""
        torch = _torch()
        with torch.cuda.device(self.device):
            tx, ty = self.carrington_planes(hdr_large, d_solar_r, lonlims, latlims, shape)
            roll = hdr_large["CROTA"] if "CROTA" in hdr_large else hdr_large["CROTA2"]
            x0, y0 = self.carrington_offset(hdr_large, hdr_large["CRVAL1"], hdr_large["CRVAL2"], roll)
            d_large = self._upload(self._native_float(data_large))
            nx = float(x0) + tx
            ny = float(y0) + ty
            ref = _ext.map_coordinates(d_large, ny, nx, self.order, -32762.0, torch.float64)
            ref = torch.where(ref == -32762.0, torch.full_like(ref, float("nan")), ref)
            self.ref = ref.contiguous()
            _ext.image_stats(self.ref, self.stats, 0)
        self.frame = "carrington"

    # ---- evaluation ------------------------------------------------------------------------------------
    def _offset_window(self):
        """The Carrington-frame window kernel applies (order 2, FMA arithmetic): its workspace is a quarter of the
        general one."""
        return self.frame == "carrington" and self.order == 2 and not self.strict and not self.no_fast \
            and self.small is not None and min(self.small.shape) >= 3

    def _workspace(self, gnx, gny, n_lags):
        torch = _torch()
        need = _ext.lag_corr_workspace_bytes(gnx, gny, n_lags, self._offset_window())
        if self._work is None or self._work.numel() * 8 < need:
            self._work = None
            self._work = torch.empty((need + 7) // 8, dtype=torch.float64, device=self.device)
        return self._work

    def lags_per_launch(self, gnx, gny):
        """Largest multiple of 256 lags whose workspace fits `max_workspace_bytes` (the size is affine in the lags;
        256 = `OFFSET_CHUNK`: a launch boundary must not cut a patch of the Carrington-frame lag order)."""
        ow = self._offset_window()
        fixed = _ext.lag_corr_workspace_bytes(gnx, gny, 1, ow)
        per_lag = max(1, (_ext.lag_corr_workspace_bytes(gnx, gny, 1025, ow) - fixed) // 1024)
        return max(OFFSET_CHUNK, ((self.max_workspace_bytes - fixed) // per_lag) // OFFSET_CHUNK * OFFSET_CHUNK)

    def evaluate(self, table_dev, out_dev, nvalid_dev=None, planes=None, allow_mixed=True):
        """Run the fused kernel over a device lag table [n, k]; results into out_dev[n]. Helioprojective frame:
        k = 11 (`CoregTanWcs` rows, `tan_wcs_table`) selects the homography kernel, k = 10 (`CoregLagTan` rows,
        `tan_lag_table`) the generic one. Asynchronous. With mixed arithmetic `self.lag_flags` receives the per-lag
        guard verdicts: follow with `resolve_flags` (which synchronises) before trusting `out_dev`."""
        torch = _torch()
        n = table_dev.shape[0]
        gny, gnx = self.ref.shape
        step = self.lags_per_launch(gnx, gny)
        self.last_launches = 0
        mixed = (allow_mixed and self.frame == "hpc" and table_dev.shape[1] == _ext.TAN_WCS_DOUBLES
                 and self._mixed_applies())
        with torch.cuda.device(self.device):
            self.lag_flags = torch.zeros(n, dtype=torch.int32, device=self.device) if mixed else None
            work = self._workspace(gnx, gny, min(n, step))
            for lo in range(0, n, step):
                hi = min(n, lo + step)
                nv = None if nvalid_dev is None else nvalid_dev[lo:hi]
                if self.frame == "hpc" and table_dev.shape[1] == _ext.TAN_WCS_DOUBLES:
                    flags = self.flags
                    if self.variant == 0 and self.pure_shift_hint:
                        # a grid of pure CRVAL shifts: the kernel flavour without the adaptive segment (1 - 3 % faster
                        # on the regular path, csrc/coreg_lag_roll.cu); decided on the WHOLE lag grid, never on a shard
                        flags = _ext.make_flags(self.strict, 1, no_fast=self.no_fast)
                    _ext.hpc_lag_corr_wcs(self.ref, self.small, self.grid_wcs, table_dev[lo:hi], self.order,
                                          self.stats if mixed else self.pivots, work, out_dev[lo:hi], nv, flags,
                                          small32c=self.small32 if mixed else None,
                                          flagged=self.lag_flags[lo:hi] if mixed else None)
                elif self.frame == "surface":
                    _ext.hpc_lag_corr_edge(self.ref, self.small_pad, self.planes, table_dev[lo:hi], self.pivots, work,
                                           out_dev[lo:hi], nv, self.flags)
                elif self.frame == "car":
                    _ext.car_lag_corr(self.ref, self.small, self.planes, table_dev[lo:hi], self.order,
                                      self.pivots, work, out_dev[lo:hi], nv, self.flags)
                elif self.frame == "hpc":
                    _ext.hpc_lag_corr(self.ref, self.small, self._hpc_planes(), table_dev[lo:hi], self.order,
                                      self.pivots, work, out_dev[lo:hi], nv, self.flags)
                else:
                    tx, ty = planes
                    _ext.offset_lag_corr(self.ref, self.small, tx, ty, table_dev[lo:hi], self.order, self.pivots,
                                         work, out_dev[lo:hi], nv, self.flags)
                self.last_launches += 2  # lag kernel + finalize
        return out_dev

    def resolve_flags(self, table_dev, out_dev, nvalid_dev=None):
        """After a mixed-arithmetic `evaluate`: re-evaluate, with the all-FP64 kernel, every lag whose error model
        (FP32 rounding of the centred spline against the variance of the sampled image, `mixed_guard_trips` in
        csrc/coreg_lag_roll.cu) exceeded 1e-7 in r. The decision is per lag, so the cube does not depend on how the
        lag list was sharded. Synchronises on the flag count. Returns the number of lags re-evaluated."""
        torch = _torch()
        if self.lag_flags is None:
            return 0
        with torch.cuda.device(self.device):
            idx = torch.nonzero(self.lag_flags, as_tuple=False).flatten()   # (synchronises)
            self.lag_flags = None
            k = int(idx.numel())
            if k:
                sub = table_dev.index_select(0, idx).contiguous()
                out = torch.empty(k, dtype=torch.float64, device=self.device)
                nv = torch.empty(k, dtype=torch.int64, device=self.device) if nvalid_dev is not None else None
                self.evaluate(sub, out, nv, allow_mixed=False)
                out_dev.index_copy_(0, idx, out)
                if nvalid_dev is not None:
                    nvalid_dev.index_copy_(0, idx, nv)
            self.flagged_lags = k
        return k

    def evaluate_patch_ordered(self, table, lag_ij, planes, return_nvalid=False, pinned=False):
        """Carrington frame, on this device alone: host offset table [n, 2] -> device corr [n] (and nvalid [n] or
        None), in the order of `table`. The lags are handed to the kernel in `offset_patch_order` of their grid indices
        lag_ij = (i1, i2[, group]) and scattered back. Asynchronous; pinned=True stages the uploads in page-locked
        memory so that the host does not wait for the stream."""
        torch = _torch()
        slot, n_slots = offset_patch_order(*lag_ij)
        padded = np.full((n_slots, table.shape[1]), np.nan, dtype=np.float64)
        padded[slot] = table
        with torch.cuda.device(self.device):
            tab_dev = self._upload(padded, pinned=pinned)
            idx = self._upload(slot, pinned=pinned)
            out = torch.empty(n_slots, dtype=torch.float64, device=self.device)
            nv = torch.empty(n_slots, dtype=torch.int64, device=self.device) if return_nvalid else None
            self.evaluate(tab_dev, out, nv, planes)
            return out.index_select(0, idx), (nv.index_select(0, idx) if return_nvalid else None)

    def adopt_reference(self, other):
        """Search against `other`'s resident reference on the common grid (Carrington frame: one projection shared by
        the engines of a frame sequence): the same tensor and its statistics column."""
        torch = _torch()
        with torch.cuda.device(self.device):
            self.ref = other.ref
            self.stats[:, 0].copy_(other.stats[:, 0])
        self.frame = other.frame

    def search(self, table, planes=None, return_nvalid=False, lag_ij=None):
        """Host lag table [n_lags, k] -> numpy corr[n_lags]; shards over ranks when torch.distributed is up.
        lag_ij = (i1, i2[, group]): CRVAL1 / CRVAL2 grid indices of every lag (Carrington frame): each rank's slice is
        handed to the kernel in `offset_patch_order`."""
        torch = _torch()
        n = table.shape[0]
        dist, rank, world = _dist_info()
        chunk, bounds = shard_bounds(n, world)
        lo, hi = bounds[rank]
        with torch.cuda.device(self.device):
            local = torch.full((chunk,), float("nan"), dtype=torch.float64, device=self.device)
            nvalid = torch.zeros(chunk, dtype=torch.int64, device=self.device) if return_nvalid else None
            if hi > lo and lag_ij is not None and self.frame == "carrington":
                out, nv = self.evaluate_patch_ordered(table[lo:hi], [np.asarray(v)[lo:hi] for v in lag_ij], planes,
                                                      return_nvalid=return_nvalid)
                local[:hi - lo] = out
                if return_nvalid:
                    nvalid[:hi - lo] = nv
            elif hi > lo:
                tab_dev = self._upload(table[lo:hi])
                nv = None if nvalid is None else nvalid[:hi - lo]
                self.evaluate(tab_dev, local[:hi - lo], nv, planes)
                self.resolve_flags(tab_dev, local[:hi - lo], nv)
            full = gather_slices(local, n, chunk)
            corr = full.cpu().numpy()
            if return_nvalid:
                nv_full = gather_slices(nvalid.to(torch.float64), n, chunk).cpu().numpy().astype(np.int64)
                return corr, nv_full
        return corr


def lag_unit_to_header_unit(values, unit_lag, unit_hdr, wrap):
    """`ang2pipi(Quantity(values, unit_lag)).to(unit_hdr).value` (`alignment.py:819-837`)."""
    v = np.asarray(values, dtype=np.float64)
    if wrap:
        v = units.ang2pipi(v, unit_lag)
    return units.convert(v, unit_lag, unit_hdr)
