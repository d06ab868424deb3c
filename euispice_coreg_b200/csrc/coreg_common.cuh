// coreg_common.cuh -- shared by every translation unit of libcoreg_b200.so: error reporting, the scipy-exact
// spline sampler, TAN device constants, the tile / workspace geometry of the fused lag kernels, coordinate
// functors and warp butterflies. Kernels live in the .cu files; everything here is inline / template code.
#pragma once
#include <cuda_runtime.h>
#include <math.h>

#include <algorithm>
#include <type_traits>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/coreg_b200.h"

namespace coreg {
// one error string and one set of profiling events per host thread, shared by all translation units (coreg_core.cu)
extern thread_local char g_err[512];
struct ProfPair { cudaEvent_t a, b; };
extern thread_local bool g_prof_on;
extern thread_local ProfPair g_prof[4096];
extern thread_local int g_prof_n;

inline int fail(int code, const char* fmt, const char* a = "", const char* b = "") {
  snprintf(g_err, sizeof(g_err), fmt, a, b);
  return code;
}
inline int cuda_fail(cudaError_t e, const char* where) {
  return fail(COREG_ECUDA, "%s: %s", where, cudaGetErrorString(e));
}
// flags bits 9..11 are reserved: a lag-correlation entry point refuses them before any CUDA call
inline int check_lag_flags(int flags, const char* entry) {
  return (flags & 0xE00) ? fail(COREG_EINVAL, "%s: reserved flag bits (9..11) set", entry) : COREG_OK;
}
#define CK(call)                                         \
  do {                                                   \
    cudaError_t _e = (call);                             \
    if (_e != cudaSuccess) return cuda_fail(_e, #call);  \
  } while (0)
#define CK_LAUNCH(name)                                       \
  do {                                                        \
    cudaError_t _e = cudaGetLastError();                      \
    if (_e != cudaSuccess) return cuda_fail(_e, name);        \
  } while (0)

constexpr double kD2R = 0.017453292519943295769236907684886;
constexpr double kR2D = 57.295779513082320876798154814105;
constexpr double kMagic = 6755399441055744.0;  // 1.5 * 2^52

// ---------------------------------------------------------------------------------------------------------
// arithmetic helpers: `STRICT` keeps scipy's separate multiply / add (no FMA contraction)
// ---------------------------------------------------------------------------------------------------------
template <bool STRICT>
__device__ __forceinline__ double mul_(double a, double b) {
  return STRICT ? __dmul_rn(a, b) : a * b;
}
template <bool STRICT>
__device__ __forceinline__ double add_(double a, double b) {
  return STRICT ? __dadd_rn(a, b) : a + b;
}
template <bool STRICT>
__device__ __forceinline__ double sub_(double a, double b) {
  return STRICT ? __dsub_rn(a, b) : a - b;
}

// floor(s) for |s| < 2^31 on the FP64 pipe only (no F2F/F2I): add 1.5*2^52 rounding toward -inf, the integer
// lands in the low mantissa word. Exact, i.e. identical to floor().
__device__ __forceinline__ double floor_magic(double s, int& i) {
  const double m = __dadd_rd(s, kMagic);
  i = __double2loint(m);
  return __dsub_rn(m, kMagic);
}

// Spline start index and weights of scipy's map_coordinates without prefilter (ni_splines.c), orders 0..3.
template <int ORDER, bool STRICT>
__device__ __forceinline__ void spline_weights(double t, int& start, double (&w)[ORDER + 1]) {
  int i0;
  if (ORDER == 0) {
    floor_magic(__dadd_rn(t, 0.5), i0);
    start = i0;
    w[0] = 1.0;
  } else if (ORDER == 1) {
    const double fl = floor_magic(t, i0);
    const double d = __dsub_rn(t, fl);
    start = i0;
    w[0] = __dsub_rn(1.0, d);
    w[ORDER >= 1 ? 1 : 0] = __dsub_rn(1.0, w[0]);
  } else if (ORDER == 2) {
    const double fl = floor_magic(__dadd_rn(t, 0.5), i0);
    const double d = __dsub_rn(t, fl);
    start = i0 - 1;
    const double u = __dsub_rn(0.5, d);
    if (STRICT) {
      w[ORDER >= 2 ? 1 : 0] = __dsub_rn(0.75, __dmul_rn(d, d));
      w[0] = __dmul_rn(__dmul_rn(0.5, u), u);
    } else {
      w[ORDER >= 2 ? 1 : 0] = fma(-d, d, 0.75);
      w[0] = (0.5 * u) * u;
    }
    w[ORDER >= 2 ? 2 : 0] = __dsub_rn(__dsub_rn(1.0, w[0]), w[ORDER >= 2 ? 1 : 0]);
  } else {
    const double fl = floor_magic(t, i0);
    const double d = __dsub_rn(t, fl);
    start = i0 - 1;
    const double z = __dsub_rn(1.0, d);
    const double w1 = __ddiv_rn(__dadd_rn(__dmul_rn(__dmul_rn(__dmul_rn(d, d), __dsub_rn(d, 2.0)), 3.0), 4.0), 6.0);
    const double w2 = __ddiv_rn(__dadd_rn(__dmul_rn(__dmul_rn(__dmul_rn(z, z), __dsub_rn(z, 2.0)), 3.0), 4.0), 6.0);
    const double w0 = __ddiv_rn(__dmul_rn(__dmul_rn(z, z), z), 6.0);
    w[0] = w0;
    w[ORDER >= 3 ? 1 : 0] = w1;
    w[ORDER >= 3 ? 2 : 0] = w2;
    w[ORDER >= 3 ? 3 : 0] = __dsub_rn(__dsub_rn(__dsub_rn(1.0, w0), w1), w2);
  }
}

__device__ __forceinline__ int mirror_index(int i, int n) {
  // scipy 'constant' mode keeps the full spline support near an edge by reflecting about the edge pixel centre
  if (n == 1) return 0;
  if (i < 0) i = -i;
  if (i > n - 1) i = 2 * (n - 1) - i;
  return min(max(i, 0), n - 1);
}

template <typename T>
__device__ __forceinline__ double ldval(const T* p) {
  return (double)__ldg(p);
}

// One sample of map_coordinates(img, (y, x), order=ORDER, mode='constant', prefilter=False).
// Returns false when the point is outside [0, n-1] on either axis (NaN coordinates included) -> caller uses cval.
template <int ORDER, bool STRICT, typename T>
__device__ __forceinline__ bool spline_sample(const T* __restrict__ img, int ny, int nx, double y, double x,
                                              double& out) {
  const bool inside = (y >= 0.0) && (y <= (double)(ny - 1)) && (x >= 0.0) && (x <= (double)(nx - 1));
  if (!inside) return false;
  int sy, sx;
  double wy[ORDER + 1], wx[ORDER + 1];
  spline_weights<ORDER, STRICT>(y, sy, wy);
  spline_weights<ORDER, STRICT>(x, sx, wx);
  double t = 0.0;
  const bool interior = (sy >= 0) && (sy + ORDER <= ny - 1) && (sx >= 0) && (sx + ORDER <= nx - 1);
  if (interior) {
    const T* p = img + (sy * nx + sx);  // callers guarantee ny*nx < 2^31
    if (STRICT) {
#pragma unroll
      for (int a = 0; a <= ORDER; ++a) {
#pragma unroll
        for (int b = 0; b <= ORDER; ++b) {
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(ldval(p + b), wy[a]), wx[b]));
        }
        p += nx;
      }
    } else {
#pragma unroll
      for (int a = 0; a <= ORDER; ++a) {
        double row = ldval(p) * wx[0];
#pragma unroll
        for (int b = 1; b <= ORDER; ++b) row = fma(ldval(p + b), wx[b], row);
        t = fma(row, wy[a], t);
        p += nx;
      }
    }
  } else {
    int iy[ORDER + 1], ix[ORDER + 1];
#pragma unroll
    for (int a = 0; a <= ORDER; ++a) {
      iy[a] = mirror_index(sy + a, ny);
      ix[a] = mirror_index(sx + a, nx);
    }
#pragma unroll
    for (int a = 0; a <= ORDER; ++a) {
#pragma unroll
      for (int b = 0; b <= ORDER; ++b) {
        const double v = ldval(img + (iy[a] * nx + ix[b]));
        if (STRICT)
          t = __dadd_rn(t, __dmul_rn(__dmul_rn(v, wy[a]), wx[b]));
        else
          t = fma(v * wy[a], wx[b], t);
      }
    }
  }
  out = t;
  return true;
}

// ---------------------------------------------------------------------------------------------------------
// TAN (gnomonic) device math
// ---------------------------------------------------------------------------------------------------------
struct TanDev {
  double crpix1, crpix2;
  double f11, f12, f21, f22;  // cdelt_i * pc_ij * D2R : pixel offset -> projection plane [rad]
  double i11, i12, i21, i22;  // inverse, projection plane [rad] -> pixel offset
  double a0_deg, s0, c0;      // CRVAL1 [deg], sin/cos CRVAL2
  double lonpole_rad;
  double a0_rad;
};

inline int make_tan(const CoregTanWcs* w, TanDev* t) {
  if (!w) return fail(COREG_EINVAL, "null CoregTanWcs");
  const double f11 = w->cdelt1 * w->pc11, f12 = w->cdelt1 * w->pc12;
  const double f21 = w->cdelt2 * w->pc21, f22 = w->cdelt2 * w->pc22;
  const double det = f11 * f22 - f12 * f21;
  if (!(det != 0.0) || det != det) return fail(COREG_EINVAL, "singular CDELT*PC matrix");
  t->crpix1 = w->crpix1;
  t->crpix2 = w->crpix2;
  t->f11 = f11 * kD2R;
  t->f12 = f12 * kD2R;
  t->f21 = f21 * kD2R;
  t->f22 = f22 * kD2R;
  t->i11 = (f22 / det) * kR2D;
  t->i12 = (-f12 / det) * kR2D;
  t->i21 = (-f21 / det) * kR2D;
  t->i22 = (f11 / det) * kR2D;
  t->a0_deg = w->crval1;
  t->a0_rad = w->crval1 * kD2R;
  t->s0 = sin(w->crval2 * kD2R);
  t->c0 = cos(w->crval2 * kD2R);
  t->lonpole_rad = w->lonpole * kD2R;
  return COREG_OK;
}

// ---------------------------------------------------------------------------------------------------------
// plate-carree (-CAR) device math: a sphere rotation followed by (phi, theta) -> pixel, see CoregLagCar
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void car_map_unit(const CoregLagCar& L, double cx, double cy, double cz, double& x,
                                             double& y) {
  const double vx = fma(L.r[0], cx, fma(L.r[1], cy, L.r[2] * cz));
  const double vy = fma(L.r[3], cx, fma(L.r[4], cy, L.r[5] * cz));
  const double vz = fma(L.r[6], cx, fma(L.r[7], cy, L.r[8] * cz));
  const double phi = atan2(vy, vx) * kR2D;
  const double theta = atan2(vz, sqrt(fma(vx, vx, vy * vy))) * kR2D;
  x = fma(L.m11, phi, fma(L.m12, theta, L.x0));
  y = fma(L.m21, phi, fma(L.m22, theta, L.y0));
}

// ---------------------------------------------------------------------------------------------------------
// fused lag search
// ---------------------------------------------------------------------------------------------------------
constexpr int kTileW = 64;
constexpr int kThreads = 256;
constexpr int kRowsPerPass = kThreads / kTileW;  // 4 grid rows per pass of the block
constexpr int kWarps = kThreads / 32;
constexpr int kLagSub = 64;   // lags staged in shared memory at a time
constexpr int kMom = 8;       // n, Sa, Sb, Saa, Sbb, Sab, pad, pad  (64 B per (tile, lag) partial)
constexpr int kMinTileH = 16; // tile height of the generic kernel (4 pixels per thread): sizes its partials

// rows per thread the rolling kernel's record rows are laid out for (tiles of 48 grid rows, more record rows than the
// kernel's 16-row tiles write): sizes the workspace only
constexpr int kRollWorkspaceRows = 12;
struct RollWLayout {
  size_t rows, rec, corr, cst, mask, total;   // byte offsets into the workspace
};
inline RollWLayout rollw_layout(int gnx, int gny, int64_t n_lags) {
  RollWLayout L;
  const size_t tiles = (size_t)((gnx + kTileW - 1) / kTileW) *
                       ((gny + 4 * kRollWorkspaceRows - 1) / (4 * kRollWorkspaceRows));
  L.rows = tiles * (kThreads / 32);
  L.rec = 0;
  L.corr = L.rec + L.rows * (size_t)n_lags * 3 * sizeof(double);
  L.cst = L.corr + L.rows * (size_t)n_lags * 3 * sizeof(double);
  L.mask = L.cst + L.rows * 3 * sizeof(double);
  L.total = L.mask + ((tiles * (size_t)n_lags * sizeof(unsigned) + 15) / 16) * 16;
  return L;
}
// ---- per-block outputs of the lag search (CoregRegions) ----
// Block sides are multiples of 64 grid pixels, so every block edge is a tile edge of both lag kernels (64 x 64 rolling,
// 64 x 16 generic) and a block's moments are the sum of whole tiles' records. Refused before any CUDA call: a bad
// block side, ld < n_lags, more blocks than one launch can index, and COREG_FLAG_MIXED (the mixed kernel's per-lag
// guard is calibrated on whole-grid moments).
constexpr int kRegionAlign = 64;
inline int check_regions(const CoregRegions* rg, int gnx, int gny, int64_t n_lags, int flags, const char* entry) {
  if (!rg || !rg->corr_dev || !rg->nvalid_dev) return fail(COREG_EINVAL, "%s: null CoregRegions pointer", entry);
  if (rg->block_h <= 0 || rg->block_w <= 0 || rg->block_h % kRegionAlign || rg->block_w % kRegionAlign)
    return fail(COREG_EINVAL, "%s: block sides must be positive multiples of 64 pixels", entry);
  if (rg->ld < n_lags) return fail(COREG_EINVAL, "%s: CoregRegions.ld < n_lags", entry);
  if (flags & COREG_FLAG_MIXED) return fail(COREG_EINVAL, "%s: no per-block outputs in mixed arithmetic", entry);
  if (gnx > 0 && gny > 0 &&
      (int64_t)((gny + rg->block_h - 1) / rg->block_h) * ((gnx + rg->block_w - 1) / rg->block_w) > 65535)
    return fail(COREG_EINVAL, "%s: more than 65535 blocks", entry);
  return COREG_OK;
}

// Pearson r of a fold of moments (NaN without a valid pixel): the arithmetic of the whole-grid finalize kernels
__device__ __forceinline__ double pearson_from_moments(double n, double sa, double sb, double saa, double sbb,
                                                       double sab) {
  double r = CUDART_NAN;
  if (n > 0.0) {
    const double cov = sab - sa * sb / n;
    const double va = saa - sa * sa / n;
    const double vb = sbb - sb * sb / n;
    r = cov / sqrt(va * vb);
  }
  return r;
}

// tiles [ty0, ty1) x [tx0, tx1) of block `blk` (row-major over nbx blocks per row; bt_h x bt_w tiles per block, the
// last block row / column clipped to the grid)
struct RegionTiles {
  int ty0, tx0, ntx, n_tiles;
};
__device__ __forceinline__ RegionTiles region_tiles(int blk, int nbx, int bt_h, int bt_w, int tiles_x, int tiles_y) {
  RegionTiles R;
  const int by = blk / nbx, bx = blk - by * nbx;
  R.ty0 = by * bt_h;
  R.tx0 = bx * bt_w;
  R.ntx = min(tiles_x, R.tx0 + bt_w) - R.tx0;
  R.n_tiles = (min(tiles_y, R.ty0 + bt_h) - R.ty0) * R.ntx;
  return R;
}

inline size_t partials_bytes(int gnx, int gny, int64_t n_lags) {
  const size_t tiles = (size_t)((gnx + kTileW - 1) / kTileW) * ((gny + kMinTileH - 1) / kMinTileH);
  // a multiple of 16: the per-lag homographies (16-byte aligned records) follow the partials in the workspace
  return (std::max(tiles * (size_t)n_lags * kMom * sizeof(double), rollw_layout(gnx, gny, n_lags).total) + 15) / 16 * 16;
}

struct TanCoord {
  typedef CoregLagTan Lag;
  struct Planes {
    const double* p;  // [3][n]
    int64_t n;
  };
  struct Pix {
    double p0, p1, p2;
  };
  __device__ static __forceinline__ Pix load(const Planes& pl, int64_t idx) {
    Pix q;
    q.p0 = __ldg(pl.p + idx);
    q.p1 = __ldg(pl.p + pl.n + idx);
    q.p2 = __ldg(pl.p + 2 * pl.n + idx);
    return q;
  }
  __device__ static __forceinline__ Pix dead() {
    Pix q;
    q.p0 = q.p1 = q.p2 = CUDART_NAN;
    return q;
  }
  // world -> pixel of the lag's header; NaN when behind the tangent hemisphere
  __device__ static __forceinline__ void map(const Pix& q, const Lag& L, double& x, double& y) {
    const double qs = fma(q.p1, L.cos_da, -(q.p2 * L.sin_da));  // cos(lat) sin(dA)
    const double pc = fma(q.p2, L.cos_da, q.p1 * L.sin_da);     // cos(lat) cos(dA)
    const double den = fma(pc, L.cos_d0, q.p0 * L.sin_d0);
    const double en = fma(-pc, L.sin_d0, q.p0 * L.cos_d0);
    const double inv = 1.0 / den;
    const double xi = qs * inv, eta = en * inv;
    x = fma(L.m11, xi, fma(L.m12, eta, L.x0));
    y = fma(L.m21, xi, fma(L.m22, eta, L.y0));
    if (!(den > 0.0)) x = CUDART_NAN;
  }
};

// TanCoord with reproject's edge rule, for an image that carries one replicated pixel of padding: coordinates within
// half a pixel of the (unpadded) array edge are kept and moved into the padded frame, anything else is "outside".
struct TanEdgeCoord {
  typedef CoregLagTanEdge Lag;
  typedef TanCoord::Planes Planes;
  typedef TanCoord::Pix Pix;
  __device__ static __forceinline__ Pix load(const Planes& pl, int64_t idx) { return TanCoord::load(pl, idx); }
  __device__ static __forceinline__ Pix dead() { return TanCoord::dead(); }
  __device__ static __forceinline__ void map(const Pix& q, const Lag& L, double& x, double& y) {
    TanCoord::map(q, L.t, x, y);
    const bool in = (x >= -0.5) && (x <= L.xhi) && (y >= -0.5) && (y <= L.yhi);
    x = in ? x + 1.0 : CUDART_NAN;
    y = y + 1.0;
  }
};

struct OffsetCoord {
  typedef CoregLagOffset Lag;
  struct Planes {
    const double* tx;
    const double* ty;
  };
  struct Pix {
    double tx, ty;
  };
  __device__ static __forceinline__ Pix load(const Planes& pl, int64_t idx) {
    Pix q;
    q.tx = __ldg(pl.tx + idx);
    q.ty = __ldg(pl.ty + idx);
    return q;
  }
  __device__ static __forceinline__ Pix dead() {
    Pix q;
    q.tx = q.ty = CUDART_NAN;
    return q;
  }
  __device__ static __forceinline__ void map(const Pix& q, const Lag& L, double& x, double& y) {
    x = __dadd_rn(L.x0, q.tx);
    y = __dadd_rn(L.y0, q.ty);
  }
};

// plate-carree candidate headers: planes = (sin lat, cos lat sin lng, cos lat cos lng) of the common grid's pixels
// (coreg_tan_trig_planes with alpha_ref = 0), per lag one sphere rotation + two atan2
struct CarCoord {
  typedef CoregLagCar Lag;
  typedef TanCoord::Planes Planes;
  typedef TanCoord::Pix Pix;
  __device__ static __forceinline__ Pix load(const Planes& pl, int64_t idx) { return TanCoord::load(pl, idx); }
  __device__ static __forceinline__ Pix dead() { return TanCoord::dead(); }
  __device__ static __forceinline__ void map(const Pix& q, const Lag& L, double& x, double& y) {
    car_map_unit(L, q.p2, q.p1, q.p0, x, y);
  }
};

// butterfly that leaves, in every lane, the warp total of value index (lane >> 2) & 7 : 9 shuffles instead of 40
__device__ __forceinline__ double warp_transpose_reduce8(double (&v)[8], int lane) {
  double w4[4], w2[2], w1;
  {
    const bool up = lane & 16;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const double send = up ? v[i] : v[i + 4];
      const double keep = up ? v[i + 4] : v[i];
      w4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
  }
  {
    const bool up = lane & 8;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const double send = up ? w4[i] : w4[i + 2];
      const double keep = up ? w4[i + 2] : w4[i];
      w2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
  }
  {
    const bool up = lane & 4;
    const double send = up ? w2[0] : w2[1];
    const double keep = up ? w2[1] : w2[0];
    w1 = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  w1 += __shfl_xor_sync(0xffffffffu, w1, 2);
  w1 += __shfl_xor_sync(0xffffffffu, w1, 1);
  return w1;  // value index = 4*bit4 + 2*bit3 + bit2 = (lane >> 2) & 7
}


// |v| < 2^30 (false for NaN / Inf): the range in which the magic-number floor of the fast kernels is exact
__device__ __forceinline__ bool small_magnitude(double v) {
  return (unsigned)(__double2hiint(v) & 0x7FFFFFFF) < 0x41D00000u;
}

// butterfly for 4 values: every lane ends with the warp total of value index (lane >> 3) & 3 (6 shuffles)
__device__ __forceinline__ double warp_transpose_reduce4(double (&v)[4], int lane) {
  double w2[2], w1;
  {
    const bool up = lane & 16;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const double send = up ? v[i] : v[i + 2];
      const double keep = up ? v[i + 2] : v[i];
      w2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
  }
  {
    const bool up = lane & 8;
    const double send = up ? w2[0] : w2[1];
    const double keep = up ? w2[1] : w2[0];
    w1 = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  w1 += __shfl_xor_sync(0xffffffffu, w1, 4);
  w1 += __shfl_xor_sync(0xffffffffu, w1, 2);
  w1 += __shfl_xor_sync(0xffffffffu, w1, 1);
  return w1;  // value index = 2*bit4 + bit3
}

// grid for a (rows per tile, resident blocks per SM) choice: blockIdx.x = tile, blockIdx.y = slice of the lag list,
// enough slices for a few waves of resident blocks; returns false when the lag list does not fit one launch
inline bool lag_grid(int tile_h, int minb, int gnx, int gny, int64_t n_lags, int sms, dim3* grid, int* lags_per_block,
                     int* tiles_out, int lag_sub, bool amortise_block_setup = false) {
  const int tiles = ((gnx + kTileW - 1) / kTileW) * ((gny + tile_h - 1) / tile_h);
  *tiles_out = tiles;
  // many more blocks than resident slots: border tiles take the per-pixel path and run longer, so a fine
  // granularity keeps the last wave short
  constexpr int waves = 128;
  const int want_blocks = sms * minb * waves;
  int splits = (want_blocks + tiles - 1) / tiles;
  const int max_splits = (int)((n_lags + lag_sub - 1) / lag_sub);
  splits = std::max(1, std::min(splits, max_splits));
  // ... but not so fine that a block's own set-up (its pixels of the reference image, their moments: worth about
  // two lags) stops being amortised. Tail ~ 1 / waves and set-up ~ splits / n_lags balance at
  // splits ~ sqrt(1.3 * resident blocks * n_lags / tiles): the 128-wave value for a 3600-lag search of a 2048^2 grid,
  // fewer slices for short lag lists (one rank's share of a sharded search). Measured on 450-lag slices of config 1
  // (tools/shard_lab.py): 29 slices of 16 lags 4.06 ms, 19 of 24 3.95, 12 of 40 3.86, 4 of 120 4.07.
  if (amortise_block_setup) {
    const double s = sqrt(1.315 * (double)(sms * minb) * (double)n_lags / (double)tiles);
    splits = std::max(1, std::min(splits, (int)lround(s)));
  }
  int lpb = (int)((n_lags + splits - 1) / splits);
  lpb = ((lpb + lag_sub - 1) / lag_sub) * lag_sub;
  splits = (int)((n_lags + lpb - 1) / lpb);
  if (splits > 65535) return false;
  *grid = dim3(tiles, splits);
  *lags_per_block = lpb;
  return true;
}

inline int grid_for(int64_t n, int threads = 256) {
  return (int)std::max<int64_t>(1, std::min<int64_t>((n + threads - 1) / threads, 148 * 8));
}

// per-lag 3x3 homography of the helioprojective rolling kernel (coreg_lag_roll.cu); sizes the workspace tail
struct HomLag {
  double hx0, hx1, hx2, hy0, hy1, hy2, he0, he1, he2, x0h, y0h;  // he = (0,0,1) - (denominator row)
  // |emax| = max |e| over the common grid (e is linear in (i, j): attained at a corner), +inf if not finite. The SIGN
  // bit marks a lag under which a column segment drifts off the one-row-per-row lattice (|hx1| or |hy1 - 1| above
  // 2^-12 pixel per row: rotated / rescaled candidates), so that the kernel tests it with one integer compare.
  double emax;
};


// ---- launchers defined in one translation unit and used from another ----
// fixed-order fold of [tile][lag][kMom] partials -> Pearson r (coreg_lag_generic.cu)
int launch_finalize_tiles(const double* work, int tiles, int64_t n_lags, double* corr, int64_t* nvalid, cudaStream_t s);// Carrington-frame lag kernel + its finalize (coreg_lag_offset.cu); small_dtype COREG_F32 / COREG_F64
int launch_offset_fast(int gnx, int gny, int64_t n_lags, cudaStream_t s, const double* ref, const void* small,
                       int small_dtype, int snx, int sny, const double* tx, const double* ty,
                       const CoregLagOffset* lags, const double* pivots, void* work, double* corr, int64_t* nvalid);
// per-block fold of the partials launch_offset_fast left in `work` (coreg_lag_offset.cu)
int launch_offset_regions(int gnx, int gny, int64_t n_lags, const void* work, const CoregRegions* rg, cudaStream_t s);
size_t offset_workspace_bytes(int gnx, int gny, int64_t n_lags);
}  // namespace coreg
