"""ctypes binding of `csrc/libcoreg_b200.so` (the C ABI declared in include/coreg_b200.h).

PyTorch supplies device memory and the CUDA stream; every compute step goes through the C entry
points below -- there is no CPU fallback and no alternative backend. If the shared library has not
been built (`python -c "import __graft_entry__ as g; g.build()"`), importing this module still works
(so host-only utilities and CPU tests can run) but the first compute call raises `CoregLibraryError`.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcoreg_b200.so")

F32, F64, I32 = 0, 1, 2
FLAG_STRICT = 1
FLAG_NO_FAST = 4
FLAG_MIXED = 8      # coreg_hpc_search_host: opt in to the mixed-arithmetic kernel (float32 small payload, guarded)
FLAG_PURE_SHIFT = 0x100   # every lag is a pure CRVAL shift: the rolling kernel without the adaptive segment


def make_flags(strict=False, no_fast=False, pure_shift=False):
    """flags word of the lag kernels: bit 0 strict scipy op order, bit 2 force the generic kernel,
    bit 8 the rolling kernel's flavour for lag grids of pure CRVAL shifts (other kernels ignore it)."""
    return (FLAG_STRICT if strict else 0) | (FLAG_NO_FAST if no_fast else 0) | (FLAG_PURE_SHIFT if pure_shift else 0)


class CoregLibraryError(RuntimeError):
    pass


class CoregTanWcs(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("crpix1", "crpix2", "cdelt1", "cdelt2", "pc11", "pc12", "pc21", "pc22",
                                          "crval1", "crval2", "lonpole")]


class CoregCarrington(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("lon0", "lat0", "roll", "dist", "cdelt1", "cdelt2")]


class CoregSurfaceFrames(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("grid_lon", "grid_lat", "grid_dsun", "image_lon", "image_lat", "image_dsun",
                                          "dt_days", "rsun")]


class CoregRegions(C.Structure):
    _fields_ = [("block_h", C.c_int), ("block_w", C.c_int), ("ld", C.c_int64), ("corr_dev", C.c_void_p),
                ("nvalid_dev", C.c_void_p)]


REGION_ALIGN = 64   # block sides of the per-block outputs: multiples of the lag kernels' 64-pixel tile sides


LAG_TAN_DOUBLES = 10    # sizeof(CoregLagTan) / 8
LAG_TAN_EDGE_DOUBLES = 12   # sizeof(CoregLagTanEdge) / 8
TAN_WCS_DOUBLES = 11    # sizeof(CoregTanWcs) / 8
LAG_OFFSET_DOUBLES = 2  # sizeof(CoregLagOffset) / 8
LAG_CAR_DOUBLES = 16    # sizeof(CoregLagCar) / 8

_P = C.c_void_p
_SIGNATURES = {
    "coreg_last_error": (C.c_char_p, []),
    "coreg_version": (C.c_int, []),
    "coreg_device_sm_count": (C.c_int, []),
    "coreg_tan_pix2world": (C.c_int, [C.POINTER(CoregTanWcs), C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "coreg_tan_world2pix": (C.c_int, [C.POINTER(CoregTanWcs), _P, _P, C.c_int64, _P, _P, _P]),
    "coreg_map_coordinates": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int64, C.c_int, C.c_double,
                                        _P, C.c_int, _P]),
    "coreg_hpc_cut": (C.c_int, [C.POINTER(CoregTanWcs), C.c_int, C.c_int, C.POINTER(CoregTanWcs), _P, C.c_int, C.c_int,
                                C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "coreg_pad_edge": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "coreg_surface_cut": (C.c_int, [C.POINTER(CoregTanWcs), C.c_int, C.c_int, C.POINTER(CoregTanWcs), _P, C.c_int,
                                    C.c_int, C.POINTER(CoregSurfaceFrames), _P, _P]),
    "coreg_hpc_lag_corr_edge": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int64, _P, _P,
                                          C.c_size_t, _P, _P, C.c_int, _P]),
    "coreg_hpc_lag_corr_edge_regions": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int64, _P,
                                                  _P, C.c_size_t, _P, _P, C.POINTER(CoregRegions), C.c_int, _P]),
    "coreg_surface_search_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(CoregTanWcs), _P, C.c_int, C.c_int,
                                            C.c_int, C.POINTER(CoregTanWcs), C.POINTER(CoregSurfaceFrames), _P,
                                            C.c_int64, C.c_int, _P, _P]),
    "coreg_tan_trig_planes": (C.c_int, [_P, _P, C.c_int64, C.c_double, _P, _P]),
    "coreg_widen_f32": (C.c_int, [_P, C.c_int64, _P, _P]),
    "coreg_rice_decode": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P,
                                    C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int, _P]),
    "coreg_bswap32": (C.c_int, [_P, C.c_int64, _P, _P]),
    "coreg_image_stats_scratch_bytes": (C.c_size_t, []),
    "coreg_image_stats": (C.c_int, [_P, C.c_int, C.c_int64, _P, _P, C.c_int, _P, _P]),
    "coreg_center_f32": (C.c_int, [_P, C.c_int64, _P, _P, C.c_int, _P, _P]),
    "coreg_lag_corr_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int64]),
    "coreg_offset_window_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int64]),
    "coreg_hpc_lag_corr": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int64,
                                     C.c_int, _P, _P, C.c_size_t, _P, _P, C.c_int, _P]),
    "coreg_hpc_lag_corr_wcs": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(CoregTanWcs),
                                         _P, C.c_int64, C.c_int, _P, _P, C.c_size_t, _P, _P, C.c_int, _P]),
    "coreg_hpc_lag_corr_regions": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int64,
                                             C.c_int, _P, _P, C.c_size_t, _P, _P, C.POINTER(CoregRegions), C.c_int,
                                             _P]),
    "coreg_hpc_lag_corr_wcs_regions": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(CoregTanWcs),
                                                 _P, C.c_int64, C.c_int, _P, _P, C.c_size_t, _P, _P,
                                                 C.POINTER(CoregRegions), C.c_int, _P]),
    "coreg_hpc_lag_corr_wcs_mixed": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.POINTER(CoregTanWcs), _P, C.c_int64, C.c_int, _P, _P, C.c_size_t, _P,
                                               _P, _P, C.c_int, _P]),
    "coreg_tan_homography_emax": (C.c_int, [C.POINTER(CoregTanWcs), C.c_int, C.c_int, _P, C.c_int64, _P, _P, _P]),
    "coreg_carrington_planes": (C.c_int, [C.POINTER(CoregCarrington), _P, _P, C.c_int, _P, _P, C.c_int, _P, _P, _P]),
    "coreg_offset_lag_corr": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int64,
                                        C.c_int, _P, _P, C.c_size_t, _P, _P, C.c_int, _P]),
    "coreg_offset_lag_corr_regions": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P,
                                                C.c_int64, C.c_int, _P, _P, C.c_size_t, _P, _P,
                                                C.POINTER(CoregRegions), C.c_int, _P]),
    "coreg_car_pix2world": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P]),
    "coreg_car_world2pix": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P]),
    "coreg_car_lag_corr": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int64,
                                     C.c_int, _P, _P, C.c_size_t, _P, _P, C.c_int, _P]),
    "coreg_pixel_shift_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "coreg_pixel_shift_corr": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int), C.c_int, _P, _P, C.c_size_t,
                                         _P, _P, _P]),
    "coreg_spice_wave_sum": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P, _P]),
    "coreg_synras_build": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(CoregTanWcs),
                                     C.POINTER(C.c_int), _P, _P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "coreg_synras_build_windows": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(CoregTanWcs),
                                             C.POINTER(C.c_int), C.POINTER(C.c_int), _P, _P, C.c_int, C.c_int, C.c_int,
                                             _P, _P]),
    "coreg_hpc_search_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(CoregTanWcs), _P, C.c_int, C.c_int,
                                        C.c_int, C.POINTER(CoregTanWcs), _P, C.c_int64, C.c_int, C.c_int, _P, _P]),
    "coreg_hpc_search_host_multi": (C.c_int, [C.POINTER(C.c_int), C.c_int, _P, C.c_int, C.c_int, C.c_int,
                                              C.POINTER(CoregTanWcs), _P, C.c_int, C.c_int, C.c_int,
                                              C.POINTER(CoregTanWcs), _P, C.c_int64, C.c_int, C.c_int, _P, _P]),
    "coreg_carrington_search_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(CoregCarrington), C.c_double,
                                               C.c_double, _P, C.c_int, C.c_int, C.c_int, C.POINTER(CoregCarrington),
                                               _P, _P, _P, _P, C.c_int, _P, _P, C.c_int, _P, C.c_int64, C.c_int,
                                               C.c_int, _P, _P]),
    "coreg_synras_build_host": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(CoregTanWcs),
                                          C.POINTER(C.c_int), _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    "coreg_gauss2d_fit": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P, _P, _P]),
    "coreg_fp64_peak": (C.c_int, [C.POINTER(C.c_double), C.c_int, _P]),
    "coreg_profile_begin": (C.c_int, []),
    "coreg_profile_end": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int)]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load(path: str | None = None):
    """dlopen the C-ABI library and set the prototypes. Raises if it is missing (no fallback)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("COREG_LIB_PATH") or LIB_PATH   # COREG_LIB_PATH: A/B runs of tuning builds
    if not os.path.exists(p):
        raise CoregLibraryError(
            f"{p} not found: the CUDA library is not built. Run `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a). There is no CPU fallback for the pointing search.")
    lib = C.CDLL(p)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def _check(rc, what):
    if rc != 0:
        msg = load().coreg_last_error()
        raise CoregLibraryError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")


def tan_struct(w) -> CoregTanWcs:
    """`_compat.wcs.TanWcs` -> C struct."""
    return CoregTanWcs(w.crpix1, w.crpix2, w.cdelt1, w.cdelt2, w.pc11, w.pc12, w.pc21, w.pc22,
                       w.crval1, w.crval2, w.lonpole)


# ------------------------------------------------------------------------------------------------
# torch plumbing
# ------------------------------------------------------------------------------------------------
def _torch():
    import torch
    return torch


def _stream():
    torch = _torch()
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr())


def _dt(t):
    torch = _torch()
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    raise TypeError(f"unsupported dtype {t.dtype}")


def _require_cuda(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise CoregLibraryError("device tensor expected (the pointing search has no CPU path)")
        if not t.is_contiguous():
            raise ValueError("contiguous tensor expected")


def tan_pix2world(wcs, nx, ny, wrap_pipi=True, device=None):
    """K3 -> (lng, lat) float64 device tensors [ny, nx], degrees."""
    torch = _torch()
    lib = load()
    dev = device or torch.device("cuda", torch.cuda.current_device())
    lng = torch.empty((ny, nx), dtype=torch.float64, device=dev)
    lat = torch.empty((ny, nx), dtype=torch.float64, device=dev)
    s = tan_struct(wcs)
    with torch.cuda.device(dev):
        _check(lib.coreg_tan_pix2world(C.byref(s), nx, ny, int(bool(wrap_pipi)), _ptr(lng), _ptr(lat), _stream()),
               "coreg_tan_pix2world")
    return lng, lat


def tan_world2pix(wcs, lng, lat):
    torch = _torch()
    lib = load()
    _require_cuda(lng, lat)
    x = torch.empty_like(lng)
    y = torch.empty_like(lat)
    s = tan_struct(wcs)
    with torch.cuda.device(lng.device):
        _check(lib.coreg_tan_world2pix(C.byref(s), _ptr(lng), _ptr(lat), lng.numel(), _ptr(x), _ptr(y), _stream()),
               "coreg_tan_world2pix")
    return x, y


def map_coordinates(img, y, x, order, cval, out_dtype):
    """Device `map_coordinates(img, [y, x], order, mode='constant', cval, prefilter=False)`."""
    torch = _torch()
    lib = load()
    _require_cuda(img, y, x)
    out = torch.empty(x.shape, dtype=out_dtype, device=img.device)
    with torch.cuda.device(img.device):
        _check(lib.coreg_map_coordinates(_ptr(img), _dt(img), img.shape[0], img.shape[1], _ptr(y), _ptr(x),
                                         x.numel(), int(order), float(cval), _ptr(out), _dt(out), _stream()),
               "coreg_map_coordinates")
    return out


def hpc_cut(wcs_small, wcs_large, large, origin, order):
    """The one-time cut, fused (`coreg_hpc_cut`): the large image (or its window starting at origin = (x0, y0)) on the
    unshifted small grid, float32 [naxis2, naxis1]."""
    torch = _torch()
    lib = load()
    _require_cuda(large)
    nx, ny = int(wcs_small.naxis1), int(wcs_small.naxis2)
    out = torch.empty((ny, nx), dtype=torch.float32, device=large.device)
    ss, sl = tan_struct(wcs_small), tan_struct(wcs_large)
    with torch.cuda.device(large.device):
        _check(lib.coreg_hpc_cut(C.byref(ss), nx, ny, C.byref(sl), _ptr(large), _dt(large), large.shape[0],
                                 large.shape[1], int(origin[0]), int(origin[1]), int(order), _ptr(out), _stream()),
               "coreg_hpc_cut")
    return out


def tan_trig_planes(lng, lat, alpha_ref_deg):
    torch = _torch()
    lib = load()
    _require_cuda(lng, lat)
    planes = torch.empty((3,) + tuple(lng.shape), dtype=torch.float64, device=lng.device)
    with torch.cuda.device(lng.device):
        _check(lib.coreg_tan_trig_planes(_ptr(lng), _ptr(lat), lng.numel(), float(alpha_ref_deg), _ptr(planes),
                                         _stream()), "coreg_tan_trig_planes")
    return planes


_RAND = {}


def fits_rand_values():
    """cfitsio's dither sequence (`fits_init_randoms`): Park-Miller a = 16807, m = 2^31 - 1, seed 1, 10000 numbers
    stored as float32."""
    a, m, seed = 16807.0, 2147483647.0, 1.0
    out = np.empty(10000, dtype=np.float32)
    for i in range(10000):
        temp = a * seed
        seed = temp - m * int(temp / m)
        out[i] = np.float32(seed / m)
    return out


def rice_decode(heap, offsets, counts, tile_w, tile_h, nx, ny, blocksize, bytepix, zscale=None, zzero=None, method=-1,
                zdither0=1, blank=None, out_dtype=None, device=None):
    """Decode a RICE_1 tile-compressed image on the device. `heap`: bytes-like (the table heap); `offsets`, `counts`:
    per tile. Returns a device tensor [ny, nx] (int32 for integer images, float32 / float64 for quantised ones)."""
    torch = _torch()
    lib = load()
    dev = device or torch.device("cuda", torch.cuda.current_device())
    n_tiles = len(offsets)
    h = torch.frombuffer(bytearray(heap) if len(heap) else bytearray(1), dtype=torch.uint8).to(dev)
    o = torch.as_tensor(np.asarray(offsets, dtype=np.int64)).to(dev)
    c = torch.as_tensor(np.asarray(counts, dtype=np.int32)).to(dev)
    quant = method >= 0
    if quant:
        zs = torch.as_tensor(np.asarray(zscale, dtype=np.float64)).to(dev)
        zz = torch.as_tensor(np.asarray(zzero, dtype=np.float64)).to(dev)
        key = str(dev)
        if key not in _RAND:
            _RAND[key] = torch.from_numpy(fits_rand_values()).to(dev)
        rnd = _RAND[key]
        odt = out_dtype or torch.float32
        code = F32 if odt == torch.float32 else F64
    else:
        zs = zz = rnd = None
        odt, code = torch.int32, I32
    out = torch.empty((ny, nx), dtype=odt, device=dev)
    with torch.cuda.device(dev):
        _check(lib.coreg_rice_decode(_ptr(h), _ptr(o), _ptr(c), n_tiles, int(tile_w), int(tile_h), int(nx), int(ny),
                                     int(blocksize), int(bytepix), _ptr(zs) if quant else None,
                                     _ptr(zz) if quant else None, int(method), int(zdither0),
                                     int(blank is not None), int(blank or 0), _ptr(rnd) if quant else None, _ptr(out),
                                     code, _stream()), "coreg_rice_decode")
    return out


def widen_f32(img):
    """float32 device image -> float64 (exact), on the device."""
    torch = _torch()
    lib = load()
    _require_cuda(img)
    if img.dtype != torch.float32:
        raise TypeError("float32 tensor expected")
    out = torch.empty(img.shape, dtype=torch.float64, device=img.device)
    with torch.cuda.device(img.device):
        _check(lib.coreg_widen_f32(_ptr(img), img.numel(), _ptr(out), _stream()), "coreg_widen_f32")
    return out


def bswap32_to_float32(words):
    """Device int32 tensor holding big-endian float32 words (a FITS BITPIX -32 payload as stored) -> the float32 image,
    swapped in place on the device."""
    torch = _torch()
    lib = load()
    _require_cuda(words)
    if words.dtype != torch.int32:
        raise TypeError("int32 tensor of raw big-endian words expected")
    with torch.cuda.device(words.device):
        _check(lib.coreg_bswap32(_ptr(words), words.numel(), _ptr(words), _stream()), "coreg_bswap32")
    return words.view(torch.float32)


STATS_ROWS = 4   # rows of a statistics block: mean (the pivot), count, max |v|, RMS about the pivot


def _stats_scratch(device):
    torch = _torch()
    n = int(load().coreg_image_stats_scratch_bytes())
    return torch.empty((n + 7) // 8, dtype=torch.float64, device=device)


def image_stats(img, stats, column=0, widen=False):
    """One deterministic multi-block pass over `img`: stats[0, column] = mean of the finite values (the pivot),
    stats[1, column] = their count, stats[2, column] = max |v|. `stats`: device float64 [4, k]. widen=True (float32
    image) also returns the float64 copy written by the same pass."""
    torch = _torch()
    lib = load()
    _require_cuda(img, stats)
    if stats.dtype != torch.float64 or stats.dim() != 2 or stats.shape[0] != STATS_ROWS:
        raise TypeError("stats must be a float64 [4, k] device tensor")
    wide = torch.empty(img.shape, dtype=torch.float64, device=img.device) if widen else None
    with torch.cuda.device(img.device):
        scratch = _stats_scratch(img.device)
        _check(lib.coreg_image_stats(_ptr(img), _dt(img), img.numel(), _ptr(wide) if widen else None,
                                     C.c_void_p(stats.data_ptr() + 8 * int(column)), int(stats.shape[1]),
                                     _ptr(scratch), _stream()), "coreg_image_stats")
    return wide


def center_f32(img32, stats, column=1):
    """Float32 twin of a float32 image centred on the float32-rounded pivot stats[0, column]; stats[3, column] = RMS of
    the centred finite values (input of the mixed kernel's guard)."""
    torch = _torch()
    lib = load()
    _require_cuda(img32, stats)
    if img32.dtype != torch.float32:
        raise TypeError("float32 tensor expected")
    out = torch.empty_like(img32)
    with torch.cuda.device(img32.device):
        scratch = _stats_scratch(img32.device)
        _check(lib.coreg_center_f32(_ptr(img32), img32.numel(), _ptr(out),
                                    C.c_void_p(stats.data_ptr() + 8 * int(column)), int(stats.shape[1]),
                                    _ptr(scratch), _stream()), "coreg_center_f32")
    return out


def finite_mean(img, out):
    """mean of finite values of `img` -> out[0] (device double, e.g. a view into a pivots tensor)."""
    torch = _torch()
    _require_cuda(img, out)
    st = torch.empty((STATS_ROWS, 1), dtype=torch.float64, device=img.device)
    image_stats(img, st)
    with torch.cuda.device(img.device):
        out[0:1].copy_(st[0])


def lag_corr_workspace_bytes(gnx, gny, n_lags, offset_window=False):
    """Scratch bytes of one lag-kernel launch; offset_window=True: the Carrington-frame window kernel only."""
    lib = load()
    fn = lib.coreg_offset_window_workspace_bytes if offset_window else lib.coreg_lag_corr_workspace_bytes
    return int(fn(int(gnx), int(gny), int(n_lags)))


def region_grid(gny, gnx, block_h, block_w):
    """(nby, nbx): blocks of block_h x block_w pixels over a gny x gnx grid from pixel (0, 0), the last block row and
    column clipped to the grid (`CoregRegions`)."""
    return -(-int(gny) // int(block_h)), -(-int(gnx) // int(block_w))


def _regions_struct(regions, gny, gnx, n_lags):
    """regions = (block_h, block_w, corr [n_blocks, >= n_lags] float64, nvalid [n_blocks, >= n_lags] int64) ->
    `CoregRegions`. The outputs may be column slices [:, lo:hi] of wider device arrays: ld is their row stride."""
    torch = _torch()
    bh, bw, corr, nvalid = regions
    if not (corr.is_cuda and nvalid.is_cuda):
        raise CoregLibraryError("device tensors expected for the per-block outputs")
    if corr.dtype != torch.float64 or nvalid.dtype != torch.int64:
        raise TypeError("per-block outputs: float64 corr and int64 nvalid")
    if corr.dim() != 2 or corr.shape != nvalid.shape or corr.stride() != nvalid.stride() or \
            (corr.shape[1] > 1 and corr.stride(1) != 1) or corr.shape[1] < n_lags:
        raise ValueError("per-block outputs: two [n_blocks, >= n_lags] arrays with unit column stride and equal strides")
    if bh > 0 and bw > 0 and corr.shape[0] != int(np.prod(region_grid(gny, gnx, bh, bw))):
        raise ValueError("per-block outputs: one row per block of the grid")
    return CoregRegions(int(bh), int(bw), corr.stride(0), corr.data_ptr(), nvalid.data_ptr())


def hpc_lag_corr(ref, small, planes, lags, order, pivots, work, corr_out, nvalid_out=None, flags=0, regions=None):
    """K1. `lags`: device float64 [n_lags, 10] (CoregLagTan rows). Writes corr_out[n_lags]. `regions` =
    (block_h, block_w, corr_blocks, nvalid_blocks): also the per-block outputs (`coreg_hpc_lag_corr_regions`)."""
    torch = _torch()
    lib = load()
    _require_cuda(ref, small, planes, lags, pivots, work, corr_out)
    if ref.dtype != torch.float32:
        raise TypeError("ref must be float32 (the reference keeps the cut large image in float32)")
    n_lags = lags.shape[0]
    gny, gnx = ref.shape
    args = (_ptr(ref), _ptr(small), _dt(small), small.shape[1], small.shape[0], gnx, gny, _ptr(planes), _ptr(lags),
            n_lags, int(order), _ptr(pivots), _ptr(work), work.numel() * work.element_size(), _ptr(corr_out),
            _ptr(nvalid_out) if nvalid_out is not None else None)
    with torch.cuda.device(ref.device):
        if regions is not None:
            rg = _regions_struct(regions, gny, gnx, n_lags)
            _check(lib.coreg_hpc_lag_corr_regions(*args, C.byref(rg), int(flags), _stream()),
                   "coreg_hpc_lag_corr_regions")
            return
        _check(lib.coreg_hpc_lag_corr(*args, int(flags), _stream()), "coreg_hpc_lag_corr")


def pad_edge(img):
    """One replicated pixel around a device image, float64 (`coreg_pad_edge`: reproject's `pad_edge_pixels`)."""
    torch = _torch()
    lib = load()
    _require_cuda(img)
    ny, nx = img.shape
    out = torch.empty((ny + 2, nx + 2), dtype=torch.float64, device=img.device)
    with torch.cuda.device(img.device):
        _check(lib.coreg_pad_edge(_ptr(img), _dt(img), ny, nx, _ptr(out), _stream()), "coreg_pad_edge")
    return out


def surface_cut(wcs_small, wcs_large, large_pad, frames):
    """The large image on the small grid through the solar-surface change of observer (`coreg_surface_cut`): float64
    [naxis2, naxis1]. `large_pad`: `pad_edge` of the large image; `frames`: `CoregSurfaceFrames`."""
    torch = _torch()
    lib = load()
    _require_cuda(large_pad)
    if large_pad.dtype != torch.float64:
        raise TypeError("large_pad must be the float64 output of pad_edge")
    nx, ny = int(wcs_small.naxis1), int(wcs_small.naxis2)
    out = torch.empty((ny, nx), dtype=torch.float64, device=large_pad.device)
    ss, sl = tan_struct(wcs_small), tan_struct(wcs_large)
    with torch.cuda.device(large_pad.device):
        _check(lib.coreg_surface_cut(C.byref(ss), nx, ny, C.byref(sl), _ptr(large_pad), large_pad.shape[0] - 2,
                                     large_pad.shape[1] - 2, C.byref(frames), _ptr(out), _stream()),
               "coreg_surface_cut")
    return out


def hpc_lag_corr_edge(ref, small_pad, planes, lags, pivots, work, corr_out, nvalid_out=None, flags=0, regions=None):
    """Bilinear helioprojective search with reproject's edge rule (`coreg_hpc_lag_corr_edge`). `small_pad`: `pad_edge` of
    the small image; `lags`: device float64 [n_lags, 12] (CoregLagTanEdge rows); `ref`: float64. `regions` =
    (block_h, block_w, corr_blocks, nvalid_blocks): also the per-block outputs (`coreg_hpc_lag_corr_edge_regions`)."""
    torch = _torch()
    lib = load()
    _require_cuda(ref, small_pad, planes, lags, pivots, work, corr_out)
    if ref.dtype != torch.float64 or small_pad.dtype != torch.float64:
        raise TypeError("ref and small_pad must be float64")
    if lags.shape[1] != LAG_TAN_EDGE_DOUBLES:
        raise TypeError("lags must be CoregLagTanEdge rows [n_lags, 12]")
    gny, gnx = ref.shape
    args = (_ptr(ref), _ptr(small_pad), small_pad.shape[1] - 2, small_pad.shape[0] - 2, gnx, gny, _ptr(planes),
            _ptr(lags), lags.shape[0], _ptr(pivots), _ptr(work), work.numel() * work.element_size(), _ptr(corr_out),
            _ptr(nvalid_out) if nvalid_out is not None else None)
    with torch.cuda.device(ref.device):
        if regions is not None:
            rg = _regions_struct(regions, gny, gnx, lags.shape[0])
            _check(lib.coreg_hpc_lag_corr_edge_regions(*args, C.byref(rg), int(flags), _stream()),
                   "coreg_hpc_lag_corr_edge_regions")
            return
        _check(lib.coreg_hpc_lag_corr_edge(*args, int(flags), _stream()), "coreg_hpc_lag_corr_edge")


def hpc_lag_corr_wcs(ref, small, grid_wcs, lag_wcs, order, pivots, work, corr_out, nvalid_out=None, flags=0,
                     small32c=None, flagged=None, regions=None):
    """K1, homography form. `lag_wcs`: device float64 [n_lags, 11] (CoregTanWcs rows of the shifted headers);
    `grid_wcs`: `_compat.wcs.TanWcs` of the common grid. `small32c` (the float32 payload `small` was widened from,
    centred on its float32 pivot: `center_f32`) selects the mixed-arithmetic kernel -- FP64 projection, FP32 spline --;
    `pivots` must then be the [4, 2] statistics block and `flagged` a zeroed int32 device counter that receives the
    number of lags tripping the kernel's error-model guard. `regions` = (block_h, block_w, corr_blocks, nvalid_blocks):
    also the per-block outputs (`coreg_hpc_lag_corr_wcs_regions`; not with mixed arithmetic)."""
    torch = _torch()
    lib = load()
    _require_cuda(ref, small, lag_wcs, pivots, work, corr_out)
    if ref.dtype != torch.float32:
        raise TypeError("ref must be float32 (the reference keeps the cut large image in float32)")
    if small.dtype != torch.float64:
        raise TypeError("the homography kernel reads a float64 small image")
    gny, gnx = ref.shape
    g = tan_struct(grid_wcs)
    if regions is not None:
        if small32c is not None:
            raise ValueError("no per-block outputs in mixed arithmetic (its guard is calibrated on whole-grid moments)")
        rg = _regions_struct(regions, gny, gnx, lag_wcs.shape[0])
        with torch.cuda.device(ref.device):
            _check(lib.coreg_hpc_lag_corr_wcs_regions(
                _ptr(ref), _ptr(small), small.shape[1], small.shape[0], gnx, gny, C.byref(g), _ptr(lag_wcs),
                lag_wcs.shape[0], int(order), _ptr(pivots), _ptr(work), work.numel() * work.element_size(),
                _ptr(corr_out), _ptr(nvalid_out) if nvalid_out is not None else None, C.byref(rg), int(flags),
                _stream()), "coreg_hpc_lag_corr_wcs_regions")
        return
    if small32c is not None:
        _require_cuda(small32c, flagged)
        if small32c.dtype != torch.float32 or small32c.shape != small.shape:
            raise TypeError("small32c must be the contiguous centred float32 twin of small")
        if pivots.shape != (STATS_ROWS, 2) or flagged.dtype != torch.int32:
            raise TypeError("mixed arithmetic needs the [4, 2] statistics block and an int32 flag counter")
        with torch.cuda.device(ref.device):
            _check(lib.coreg_hpc_lag_corr_wcs_mixed(
                _ptr(ref), _ptr(small), _ptr(small32c), small.shape[1], small.shape[0], gnx, gny, C.byref(g),
                _ptr(lag_wcs), lag_wcs.shape[0], int(order), _ptr(pivots), _ptr(work),
                work.numel() * work.element_size(), _ptr(corr_out),
                _ptr(nvalid_out) if nvalid_out is not None else None, _ptr(flagged), int(flags), _stream()),
                "coreg_hpc_lag_corr_wcs_mixed")
        return
    with torch.cuda.device(ref.device):
        _check(lib.coreg_hpc_lag_corr_wcs(_ptr(ref), _ptr(small), small.shape[1], small.shape[0], gnx, gny,
                                          C.byref(g), _ptr(lag_wcs), lag_wcs.shape[0], int(order), _ptr(pivots),
                                          _ptr(work), work.numel() * work.element_size(), _ptr(corr_out),
                                          _ptr(nvalid_out) if nvalid_out is not None else None, int(flags),
                                          _stream()), "coreg_hpc_lag_corr_wcs")


def homography_emax(grid_wcs, lag_wcs, gnx, gny):
    """max |1 - D| of each candidate header's homography over the common grid (device float64 [n_lags])."""
    torch = _torch()
    lib = load()
    _require_cuda(lag_wcs)
    n = lag_wcs.shape[0]
    scratch = torch.empty(12 * max(n, 1), dtype=torch.float64, device=lag_wcs.device)
    out = torch.empty(n, dtype=torch.float64, device=lag_wcs.device)
    g = tan_struct(grid_wcs)
    with torch.cuda.device(lag_wcs.device):
        _check(lib.coreg_tan_homography_emax(C.byref(g), int(gnx), int(gny), _ptr(lag_wcs), n, _ptr(scratch), _ptr(out),
                                             _stream()), "coreg_tan_homography_emax")
    return out


def carrington_planes(c: CoregCarrington, sinlon, coslon, sinlat, coslat):
    torch = _torch()
    lib = load()
    _require_cuda(sinlon, coslon, sinlat, coslat)
    n_lon, n_lat = sinlon.numel(), sinlat.numel()
    tx = torch.empty((n_lat, n_lon), dtype=torch.float64, device=sinlon.device)
    ty = torch.empty_like(tx)
    with torch.cuda.device(tx.device):
        _check(lib.coreg_carrington_planes(C.byref(c), _ptr(sinlon), _ptr(coslon), n_lon, _ptr(sinlat), _ptr(coslat),
                                           n_lat, _ptr(tx), _ptr(ty), _stream()), "coreg_carrington_planes")
    return tx, ty


def offset_lag_corr(ref, small, tx, ty, lags, order, pivots, work, corr_out, nvalid_out=None, flags=0, regions=None):
    """K4. `lags`: device float64 [n_lags, 2] (CoregLagOffset rows). `regions` = (block_h, block_w, corr_blocks,
    nvalid_blocks): also the per-block outputs over the Carrington grid (`coreg_offset_lag_corr_regions`)."""
    torch = _torch()
    lib = load()
    _require_cuda(ref, small, tx, ty, lags, pivots, work, corr_out)
    if ref.dtype != torch.float64:
        raise TypeError("ref must be float64 (the reference keeps the Carrington-projected image in float64)")
    gny, gnx = ref.shape
    args = (_ptr(ref), _ptr(small), _dt(small), small.shape[1], small.shape[0], gnx, gny, _ptr(tx), _ptr(ty),
            _ptr(lags), lags.shape[0], int(order), _ptr(pivots), _ptr(work), work.numel() * work.element_size(),
            _ptr(corr_out), _ptr(nvalid_out) if nvalid_out is not None else None)
    with torch.cuda.device(ref.device):
        if regions is not None:
            rg = _regions_struct(regions, gny, gnx, lags.shape[0])
            _check(lib.coreg_offset_lag_corr_regions(*args, C.byref(rg), int(flags), _stream()),
                   "coreg_offset_lag_corr_regions")
            return
        _check(lib.coreg_offset_lag_corr(*args, int(flags), _stream()), "coreg_offset_lag_corr")


def _car_row(row):
    row = np.ascontiguousarray(row, dtype=np.float64)
    if row.shape != (LAG_CAR_DOUBLES,):
        raise ValueError("one CoregLagCar row (16 float64) expected")
    return row


def car_pix2world(car_row, nx, ny, device=None):
    """(lng, lat) float64 device tensors [ny, nx], degrees, of a plate-carree image; `car_row`: one `CoregLagCar`
    row (`_compat.wcs.CarWcs.lag_rows`)."""
    torch = _torch()
    lib = load()
    dev = device or torch.device("cuda", torch.cuda.current_device())
    lng = torch.empty((ny, nx), dtype=torch.float64, device=dev)
    lat = torch.empty((ny, nx), dtype=torch.float64, device=dev)
    row = _car_row(car_row)
    with torch.cuda.device(dev):
        _check(lib.coreg_car_pix2world(row.ctypes.data_as(_P), int(nx), int(ny), _ptr(lng), _ptr(lat), _stream()),
               "coreg_car_pix2world")
    return lng, lat


def car_world2pix(car_row, lng, lat):
    torch = _torch()
    lib = load()
    _require_cuda(lng, lat)
    x = torch.empty_like(lng)
    y = torch.empty_like(lat)
    row = _car_row(car_row)
    with torch.cuda.device(lng.device):
        _check(lib.coreg_car_world2pix(row.ctypes.data_as(_P), _ptr(lng), _ptr(lat), lng.numel(), _ptr(x), _ptr(y),
                                       _stream()), "coreg_car_world2pix")
    return x, y


def car_lag_corr(ref, small, planes, lags, order, pivots, work, corr_out, nvalid_out=None, flags=0):
    """Lag search on plate-carree images. `planes`: unit-vector planes of the common grid (`tan_trig_planes(lng, lat,
    0.0)`); `lags`: device float64 [n_lags, 16] (`CoregLagCar` rows)."""
    torch = _torch()
    lib = load()
    _require_cuda(ref, small, planes, lags, pivots, work, corr_out)
    if ref.dtype != torch.float32:
        raise TypeError("ref must be float32 (the reference keeps the cut large image in float32)")
    gny, gnx = ref.shape
    with torch.cuda.device(ref.device):
        _check(lib.coreg_car_lag_corr(_ptr(ref), _ptr(small), _dt(small), small.shape[1], small.shape[0], gnx, gny,
                                      _ptr(planes), _ptr(lags), lags.shape[0], int(order), _ptr(pivots), _ptr(work),
                                      work.numel() * work.element_size(), _ptr(corr_out),
                                      _ptr(nvalid_out) if nvalid_out is not None else None,
                                      int(flags), _stream()), "coreg_car_lag_corr")


def pixel_shift_corr(large, smalls, x0, y0, lag_dx, lag_dy, pivots, return_nvalid=False):
    """Pixel-shift lag search. large: device float64 [lny, lnx]; smalls: device float64 [n_rot, sny, snx]; lag_dx /
    lag_dy: integer sequences. Returns device corr [n_dx, n_dy, n_rot] (and nvalid)."""
    torch = _torch()
    lib = load()
    _require_cuda(large, smalls, pivots)
    if large.dtype != torch.float64 or smalls.dtype != torch.float64:
        raise TypeError("float64 images expected (the reference reads both as float64)")
    n_rot, sny, snx = smalls.shape
    lny, lnx = large.shape
    n_dx, n_dy = len(lag_dx), len(lag_dy)
    dx = (C.c_int * n_dx)(*[int(v) for v in lag_dx])
    dy = (C.c_int * n_dy)(*[int(v) for v in lag_dy])
    need = int(lib.coreg_pixel_shift_workspace_bytes(snx, sny, n_dx, n_dy, n_rot))
    work = torch.empty((need + 7) // 8, dtype=torch.float64, device=large.device)
    corr = torch.empty((n_dx, n_dy, n_rot), dtype=torch.float64, device=large.device)
    nvalid = torch.empty((n_dx, n_dy, n_rot), dtype=torch.int64, device=large.device) if return_nvalid else None
    with torch.cuda.device(large.device):
        _check(lib.coreg_pixel_shift_corr(_ptr(large), lnx, lny, _ptr(smalls), n_rot, snx, sny, int(x0), int(y0),
                                          dx, n_dx, dy, n_dy, _ptr(pivots), _ptr(work), work.numel() * 8, _ptr(corr),
                                          _ptr(nvalid) if nvalid is not None else None, _stream()),
               "coreg_pixel_shift_corr")
        torch.cuda.current_stream().synchronize()   # `dx` / `dy` are host temporaries, `work` is freed on return
    return (corr, nvalid) if return_nvalid else corr


def spice_wave_sum(raw, sel, ymin, ymax, device=None):
    """`coreg_spice_wave_sum`: raw = the [n_lambda, ny, nx] float32 planes of a SPICE L2 cube as a numpy array, big-endian
    (the FITS payload as stored) or native; sel = boolean [n_lambda]. Returns the float64 [ny, nx] image on the device."""
    torch = _torch()
    lib = load()
    raw = np.asarray(raw)
    if raw.ndim != 3 or raw.dtype.itemsize != 4 or raw.dtype.kind != "f":
        raise TypeError("raw must be a [n_lambda, ny, nx] float32 array")
    big = 0 if raw.dtype.isnative else 1
    n_lambda, ny, nx = raw.shape
    dev = device or torch.device("cuda", torch.cuda.current_device())
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")      # "non-writable array": it is only read
        words = torch.from_numpy(np.ascontiguousarray(raw).view("<i4" if big else "=i4"))
    d_cube = words.to(dev)
    out = torch.empty((ny, nx), dtype=torch.float64, device=dev)
    mask = np.ascontiguousarray(np.asarray(sel, dtype=np.uint8))
    if mask.shape != (n_lambda,):
        raise ValueError("sel must hold one flag per wavelength plane")
    with torch.cuda.device(dev):
        _check(lib.coreg_spice_wave_sum(_ptr(d_cube), big, n_lambda, ny, nx, mask.ctypes.data_as(_P), int(ymin),
                                        int(ymax), _ptr(out), _stream()), "coreg_spice_wave_sum")
    return out


def synras_build(frames, wcs_list, frame_of_col, lng, lat, order, origins=None):
    """K6. frames: device [n_frames, fny, fnx]; lng/lat: device [n_rows, n_cols] degrees. origins: [(x0, y0)] per frame
    when `frames` holds windows [y0:, x0:] of the images the WCS describe (`coreg_synras_build_windows`)."""
    torch = _torch()
    lib = load()
    _require_cuda(frames, lng, lat)
    n_frames, fny, fnx = frames.shape
    n_rows, n_cols = lng.shape
    arr = (CoregTanWcs * n_frames)(*[tan_struct(w) for w in wcs_list])
    cols = (C.c_int * n_cols)(*[int(v) for v in frame_of_col])
    out = torch.empty((n_rows, n_cols), dtype=torch.float64, device=frames.device)
    org = None
    if origins is not None:
        flat = [int(v) for xy in origins for v in xy]
        if len(flat) != 2 * n_frames:
            raise ValueError("origins must hold one (x0, y0) per frame")
        org = (C.c_int * (2 * n_frames))(*flat)
    with torch.cuda.device(frames.device):
        _check(lib.coreg_synras_build_windows(_ptr(frames), _dt(frames), n_frames, fnx, fny, arr, org, cols, _ptr(lng),
                                              _ptr(lat), n_rows, n_cols, int(order), _ptr(out), _stream()),
               "coreg_synras_build")
        torch.cuda.current_stream().synchronize()  # `arr` / `cols` are host temporaries
    return out


def _np_dt(a):
    if a.dtype == np.float32:
        return F32
    if a.dtype == np.float64:
        return F64
    raise TypeError(f"unsupported dtype {a.dtype}")


def hpc_search_host(large, wcs_large, small, wcs_small, lag_wcs, order=2, flags=0):
    """Whole helioprojective search from HOST numpy buffers (the C caller's entry point). `large` / `small`:
    float32 or float64 arrays; `lag_wcs`: [n_lags, 11] float64 `CoregTanWcs` rows (`engine.tan_wcs_table`)."""
    lib = load()
    large = np.ascontiguousarray(large, dtype=None if large.dtype in (np.float32, np.float64) else np.float64)
    small = np.ascontiguousarray(small, dtype=None if small.dtype in (np.float32, np.float64) else np.float64)
    lag_wcs = np.ascontiguousarray(lag_wcs, dtype=np.float64)
    if lag_wcs.ndim != 2 or lag_wcs.shape[1] != TAN_WCS_DOUBLES:
        raise ValueError("lag_wcs must be [n_lags, 11] CoregTanWcs rows")
    n_lags = lag_wcs.shape[0]
    corr = np.empty(n_lags, dtype=np.float64)
    nvalid = np.empty(n_lags, dtype=np.int64)
    sl, ss = tan_struct(wcs_large), tan_struct(wcs_small)
    _check(lib.coreg_hpc_search_host(large.ctypes.data_as(_P), _np_dt(large), large.shape[1], large.shape[0],
                                     C.byref(sl), small.ctypes.data_as(_P), _np_dt(small), small.shape[1],
                                     small.shape[0], C.byref(ss), lag_wcs.ctypes.data_as(_P), n_lags, int(order),
                                     int(flags), corr.ctypes.data_as(_P), nvalid.ctypes.data_as(_P)),
           "coreg_hpc_search_host")
    return corr, nvalid


def surface_search_host(large, wcs_large, small, wcs_small, frames, lag_wcs, flags=0):
    """Whole "sunpy" Carrington search from HOST numpy buffers (`coreg_surface_search_host`). `frames`:
    `CoregSurfaceFrames`; `lag_wcs`: [n_lags, 11] float64 `CoregTanWcs` rows (`engine.tan_wcs_table`)."""
    lib = load()
    large = np.ascontiguousarray(large, dtype=None if large.dtype in (np.float32, np.float64) else np.float64)
    small = np.ascontiguousarray(small, dtype=None if small.dtype in (np.float32, np.float64) else np.float64)
    lag_wcs = np.ascontiguousarray(lag_wcs, dtype=np.float64)
    if lag_wcs.ndim != 2 or lag_wcs.shape[1] != TAN_WCS_DOUBLES:
        raise ValueError("lag_wcs must be [n_lags, 11] CoregTanWcs rows")
    n_lags = lag_wcs.shape[0]
    corr = np.empty(n_lags, dtype=np.float64)
    nvalid = np.empty(n_lags, dtype=np.int64)
    sl, ss = tan_struct(wcs_large), tan_struct(wcs_small)
    _check(lib.coreg_surface_search_host(large.ctypes.data_as(_P), _np_dt(large), large.shape[1], large.shape[0],
                                         C.byref(sl), small.ctypes.data_as(_P), _np_dt(small), small.shape[1],
                                         small.shape[0], C.byref(ss), C.byref(frames), lag_wcs.ctypes.data_as(_P),
                                         n_lags, int(flags), corr.ctypes.data_as(_P), nvalid.ctypes.data_as(_P)),
           "coreg_surface_search_host")
    return corr, nvalid


def hpc_search_host_multi(devices, large, wcs_large, small, wcs_small, lag_wcs, order=2, flags=0):
    """`hpc_search_host` with the lag list split over the CUDA devices `devices` of this process (one host thread per
    device, slices gathered in the host buffers)."""
    lib = load()
    large = np.ascontiguousarray(large, dtype=None if large.dtype in (np.float32, np.float64) else np.float64)
    small = np.ascontiguousarray(small, dtype=None if small.dtype in (np.float32, np.float64) else np.float64)
    lag_wcs = np.ascontiguousarray(lag_wcs, dtype=np.float64)
    if lag_wcs.ndim != 2 or lag_wcs.shape[1] != TAN_WCS_DOUBLES:
        raise ValueError("lag_wcs must be [n_lags, 11] CoregTanWcs rows")
    n_lags = lag_wcs.shape[0]
    corr = np.empty(n_lags, dtype=np.float64)
    nvalid = np.empty(n_lags, dtype=np.int64)
    sl, ss = tan_struct(wcs_large), tan_struct(wcs_small)
    dev = (C.c_int * len(devices))(*[int(d) for d in devices])
    _check(lib.coreg_hpc_search_host_multi(dev, len(devices), large.ctypes.data_as(_P), _np_dt(large), large.shape[1],
                                           large.shape[0], C.byref(sl), small.ctypes.data_as(_P), _np_dt(small),
                                           small.shape[1], small.shape[0], C.byref(ss), lag_wcs.ctypes.data_as(_P),
                                           n_lags, int(order), int(flags), corr.ctypes.data_as(_P),
                                           nvalid.ctypes.data_as(_P)), "coreg_hpc_search_host_multi")
    return corr, nvalid


def carrington_search_host(large, c_large, xy0_large, small, c_small, vec_large, vec_small, lags, order=2, flags=0):
    """Whole Carrington-frame search from HOST numpy buffers. c_*: `CoregCarrington`; xy0_large: the large header's
    detector offset; vec_* = (sinlon, coslon, sinlat, coslat) of `LagSearchEngine.carrington_vectors` for each header
    (the latitude vectors are the grid's and must agree); lags: [n_lags, 2] (x0, y0) rows."""
    lib = load()
    large = np.ascontiguousarray(large, dtype=None if large.dtype in (np.float32, np.float64) else np.float64)
    small = np.ascontiguousarray(small, dtype=None if small.dtype in (np.float32, np.float64) else np.float64)
    lags = np.ascontiguousarray(lags, dtype=np.float64)
    v = [np.ascontiguousarray(a, dtype=np.float64) for a in (vec_large[0], vec_large[1], vec_small[0], vec_small[1],
                                                            vec_small[2], vec_small[3])]
    n_lon, n_lat, n_lags = v[0].size, v[4].size, lags.shape[0]
    corr = np.empty(n_lags, dtype=np.float64)
    nvalid = np.empty(n_lags, dtype=np.int64)
    _check(lib.coreg_carrington_search_host(large.ctypes.data_as(_P), _np_dt(large), large.shape[1], large.shape[0],
                                            C.byref(c_large), float(xy0_large[0]), float(xy0_large[1]),
                                            small.ctypes.data_as(_P), _np_dt(small), small.shape[1], small.shape[0],
                                            C.byref(c_small), v[0].ctypes.data_as(_P), v[1].ctypes.data_as(_P),
                                            v[2].ctypes.data_as(_P), v[3].ctypes.data_as(_P), n_lon,
                                            v[4].ctypes.data_as(_P), v[5].ctypes.data_as(_P), n_lat,
                                            lags.ctypes.data_as(_P), n_lags, int(order), int(flags),
                                            corr.ctypes.data_as(_P), nvalid.ctypes.data_as(_P)),
           "coreg_carrington_search_host")
    return corr, nvalid


def synras_build_host(frames, wcs_list, frame_of_col, lng, lat, order):
    """Synthetic raster from HOST numpy buffers: frames [n_frames, fny, fnx] float32 / float64, lng / lat [n_rows,
    n_cols] degrees -> float64 [n_rows, n_cols]."""
    lib = load()
    frames = np.ascontiguousarray(frames, dtype=None if frames.dtype in (np.float32, np.float64) else np.float64)
    lng = np.ascontiguousarray(lng, dtype=np.float64)
    lat = np.ascontiguousarray(lat, dtype=np.float64)
    n_frames, fny, fnx = frames.shape
    n_rows, n_cols = lng.shape
    arr = (CoregTanWcs * n_frames)(*[tan_struct(w) for w in wcs_list])
    cols = (C.c_int * n_cols)(*[int(c) for c in frame_of_col])
    out = np.empty((n_rows, n_cols), dtype=np.float64)
    _check(lib.coreg_synras_build_host(frames.ctypes.data_as(_P), _np_dt(frames), n_frames, fnx, fny, arr, cols,
                                       lng.ctypes.data_as(_P), lat.ctypes.data_as(_P), n_rows, n_cols, int(order),
                                       out.ctypes.data_as(_P)), "coreg_synras_build_host")
    return out


FIT_MAX_POINTS = 26     # COREG_FIT_MAX_POINTS: points of one Gaussian peak fit
FIT_CONVERGED, FIT_NOT_CONVERGED = 0, 3


def gauss2d_fit(points, n_points, p0, bounds):
    """Batched bounded 2-D Gaussian fits (`coreg_gauss2d_fit`). points: device float64 [n, 26, 3] (x, y, value);
    n_points: int32 [n]; p0: float64 [n, 6]; bounds: float64 [n, 12] (lo then hi). Returns device (popt [n, 6],
    cost [n], iterations [n] int32, status [n] int32: FIT_CONVERGED or FIT_NOT_CONVERGED). Asynchronous."""
    torch = _torch()
    lib = load()
    _require_cuda(points, n_points, p0, bounds)
    n = points.shape[0]
    if points.dtype != torch.float64 or p0.dtype != torch.float64 or bounds.dtype != torch.float64 or \
            n_points.dtype != torch.int32:
        raise TypeError("gauss2d_fit: float64 points / p0 / bounds and int32 n_points")
    if points.shape != (n, FIT_MAX_POINTS, 3) or n_points.shape != (n,) or p0.shape != (n, 6) or bounds.shape != (n, 12):
        raise ValueError("gauss2d_fit: points [n, 26, 3], n_points [n], p0 [n, 6], bounds [n, 12]")
    popt = torch.empty((n, 6), dtype=torch.float64, device=points.device)
    cost = torch.empty(n, dtype=torch.float64, device=points.device)
    iters = torch.empty(n, dtype=torch.int32, device=points.device)
    status = torch.empty(n, dtype=torch.int32, device=points.device)
    with torch.cuda.device(points.device):
        _check(lib.coreg_gauss2d_fit(_ptr(points), _ptr(n_points), _ptr(p0), _ptr(bounds), n, _ptr(popt), _ptr(cost),
                                     _ptr(iters), _ptr(status), _stream()), "coreg_gauss2d_fit")
    return popt, cost, iters, status


def fp64_peak(iters=20000):
    lib = load()
    v = C.c_double(0.0)
    _check(lib.coreg_fp64_peak(C.byref(v), int(iters), None), "coreg_fp64_peak")
    return v.value


def profile_begin():
    _check(load().coreg_profile_begin(), "coreg_profile_begin")


def profile_end():
    """-> (summed device ms of the fused lag kernel launches since profile_begin, their count)."""
    ms, n = C.c_double(0.0), C.c_int(0)
    _check(load().coreg_profile_end(C.byref(ms), C.byref(n)), "coreg_profile_end")
    return ms.value, n.value
