// coreg_lag_offset.cu -- Carrington-frame lag kernel (K4): order-2 spline, FMA arithmetic, FP64 throughout.
//
// Replaces `Alignment._step` with function_to_apply = `_carrington_transform_fa` for a list of CRVAL lags
// (hdrshift/alignment.py:509-542, 889-901; utils/rectify.py:340-374, 865-888). For such lags the detector coordinate
// of a Carrington-grid pixel is  x = x0(lag) + Tx[pixel],  y = y0(lag) + Ty[pixel]  (SURVEY App. A.3): a translated
// gather. Neighbouring grid pixels land several detector pixels apart (4.4 x 1.7 at BASELINE configs[1]), so a warp
// that walks a grid row scatters its nine taps per sample over 4 - 5 cache lines each: the first version of this
// kernel kept the L1 data pipe 94 % busy and the FP64 pipe 29 % (profiles/r1_ncu_carrington_v0.txt).
//
// This version turns the warp around: LANES ARE LAGS. A block owns a super-tile of the grid (eight stacked tiles of
// 32 x 8 pixels) and a chunk of 256 consecutive lags (one per thread; the caller orders the lag list so that
// consecutive lags are neighbours in the detector plane -- 16 x 16 patches, 16 x 2 per warp). For each tile
//   * the live pixels (finite reference value, in front of the limb) are compacted into a shared-memory table
//     (Tx, Ty, ref - pivot): every lane reads the same entry, a broadcast;
//   * the part of the small image that ANY (pixel, lag) pair of the tile and chunk can touch -- the tile's detector
//     footprint grown by the chunk's offset spread plus the spline support -- is staged in shared memory by ONE TMA
//     tile load (cp.async.bulk.tensor.2d, completion on an mbarrier; the box starts on a 16-byte boundary of the image
//     row; out-of-image parts arrive as zeros and are never read). A window that does not fit the box (coarse grids, unordered lags) falls back to global loads; an image
//     whose row pitch is not a multiple of 16 bytes is staged by a cooperative copy instead of TMA;
//   * every lane walks the pixel table for its own lag: coordinates, floors by magic-number add, one unsigned
//     compare per axis for "all nine taps inside image and window", weights, nine LDS.32 -- the 32 lanes of a warp
//     now touch a 16 x 8 pixel neighbourhood of the window instead of a 140-pixel row --, moments. Samples on the
//     image border take the exact out-of-line sampler on global memory, as before.
// The six moments of a (super-tile, lag) pair therefore accumulate in the registers of one thread, in a fixed order:
// no warp shuffles, no shared-memory accumulators, one 64-byte partial per (live super-tile, lag). Super-tiles that
// cannot reach the small image under any lag of the launch (87 % of the grid at configs[1]) get no partial at all:
// a pre-pass marks them and a single-block scan assigns partial slots in ascending order, so the finalize kernel
// adds the partials of a lag in the same order whatever the launch contained (bit-identical cubes for any sharding).
#include <cuda.h>

#include "coreg_common.cuh"

namespace coreg {

constexpr int kOffThreads = 256;          // = lags per chunk (one lag per thread)
constexpr int kOffMinBlocks = 3;          // resident blocks per SM (__launch_bounds__)
constexpr int kOffUnroll = 2;             // pixels of the walk in flight per lane (timed with tools/carr_lab.py)
constexpr int kOffWarps = kOffThreads / 32;
constexpr int kOffTileW = 32, kOffTileH = 8, kOffTilePx = kOffTileW * kOffTileH;   // one pixel per thread
constexpr int kOffTilesPerBlock = 8;      // stacked vertically: super-tile = 32 x 64 grid pixels
constexpr int kOffSuperH = kOffTileH * kOffTilesPerBlock;

template <typename T>
struct OffBox {   // shared-memory window = TMA box. With a warp's 32 lags laid out 16 x 2 (two detector pixels apart
                  // along x at BASELINE configs[1]) a row pitch of 0 (mod 32) words gives the unavoidable 2-way bank
                  // conflict of a stride-2 access and no more (tools/ubench/bank_model.py: 18 wavefronts for the nine
                  // taps against 30 with 8 x 4 lags per warp and a pitch of 8 mod 32, measured 33)
  static constexpr int W = sizeof(T) == 4 ? 192 : 96;
  static constexpr int H = sizeof(T) == 4 ? 64 : 56;
  static constexpr int kBytes = W * H * (int)sizeof(T);
};

struct OffPx {   // one live pixel of the current tile (32 B: one LDS.128 + one LDS.64, broadcast)
  double tx, ty, ac, pad;
};

struct OffWork {   // byte offsets into the workspace (all 16-byte aligned)
  size_t partials, slots, nslots, range, total;
  int n_super;
};
inline OffWork offw_layout(int gnx, int gny, int64_t n_lags) {
  OffWork L;
  L.n_super = ((gnx + kOffTileW - 1) / kOffTileW) * ((gny + kOffSuperH - 1) / kOffSuperH);
  L.partials = 0;
  L.slots = (size_t)L.n_super * (size_t)n_lags * kMom * sizeof(double);
  L.nslots = L.slots + (((size_t)L.n_super * sizeof(int) + 15) / 16) * 16;
  L.range = L.nslots + 16;
  L.total = L.range + 4 * sizeof(double);
  return L;
}
size_t offset_workspace_bytes(int gnx, int gny, int64_t n_lags) { return offw_layout(gnx, gny, n_lags).total; }

// ---- pre-pass ---------------------------------------------------------------------------------------------------
// range of the lag offsets (+0.5) of the whole launch; NaN / absurd offsets never evaluate anything and are ignored
__global__ void __launch_bounds__(256) offset_lag_range_kernel(const CoregLagOffset* __restrict__ lags, int n_lags,
                                                               double* __restrict__ range) {
  __shared__ double s[4][256];
  double x0 = CUDART_INF, x1 = -CUDART_INF, y0 = CUDART_INF, y1 = -CUDART_INF;
  for (int i = threadIdx.x; i < n_lags; i += 256) {
    const double x = lags[i].x0 + 0.5, y = lags[i].y0 + 0.5;
    if (small_magnitude(x) && small_magnitude(y)) {
      x0 = fmin(x0, x); x1 = fmax(x1, x);
      y0 = fmin(y0, y); y1 = fmax(y1, y);
    }
  }
  s[0][threadIdx.x] = x0; s[1][threadIdx.x] = x1; s[2][threadIdx.x] = y0; s[3][threadIdx.x] = y1;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      s[0][threadIdx.x] = fmin(s[0][threadIdx.x], s[0][threadIdx.x + o]);
      s[1][threadIdx.x] = fmax(s[1][threadIdx.x], s[1][threadIdx.x + o]);
      s[2][threadIdx.x] = fmin(s[2][threadIdx.x], s[2][threadIdx.x + o]);
      s[3][threadIdx.x] = fmax(s[3][threadIdx.x], s[3][threadIdx.x + o]);
    }
    __syncthreads();
  }
  if (threadIdx.x < 4) range[threadIdx.x] = s[threadIdx.x][0];
}

// live[s] = 1 when super-tile s has a live pixel whose 3 x 3 support can touch the image under some lag of the launch
__global__ void __launch_bounds__(256) offset_super_live_kernel(const double* __restrict__ ref,
                                                                const double* __restrict__ tx,
                                                                const double* __restrict__ ty, int gnx, int gny,
                                                                int snx, int sny, const double* __restrict__ range,
                                                                int* __restrict__ live) {
  __shared__ double s[4][256];
  const int sx_tiles = (gnx + kOffTileW - 1) / kOffTileW;
  const int ox = (blockIdx.x % sx_tiles) * kOffTileW, oy = (blockIdx.x / sx_tiles) * kOffSuperH;
  double x0 = CUDART_INF, x1 = -CUDART_INF, y0 = CUDART_INF, y1 = -CUDART_INF;
  for (int i = threadIdx.x; i < kOffTileW * kOffSuperH; i += 256) {
    const int gx = ox + (i & (kOffTileW - 1)), gy = oy + i / kOffTileW;
    if (gx < gnx && gy < gny) {
      const int64_t idx = (int64_t)gy * gnx + gx;
      const double a = ref[idx], px = tx[idx], py = ty[idx];
      if (isfinite(a) && small_magnitude(px) && small_magnitude(py)) {
        x0 = fmin(x0, px); x1 = fmax(x1, px);
        y0 = fmin(y0, py); y1 = fmax(y1, py);
      }
    }
  }
  s[0][threadIdx.x] = x0; s[1][threadIdx.x] = x1; s[2][threadIdx.x] = y0; s[3][threadIdx.x] = y1;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      s[0][threadIdx.x] = fmin(s[0][threadIdx.x], s[0][threadIdx.x + o]);
      s[1][threadIdx.x] = fmax(s[1][threadIdx.x], s[1][threadIdx.x + o]);
      s[2][threadIdx.x] = fmin(s[2][threadIdx.x], s[2][threadIdx.x + o]);
      s[3][threadIdx.x] = fmax(s[3][threadIdx.x], s[3][threadIdx.x + o]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    // sample valid <=> 0 <= x <= n - 1 <=> 0.5 <= x + 0.5 <= n - 0.5; one pixel of slack for rounding. An empty box
    // (no live pixel: +inf / -inf) or an empty lag range fails the test.
    const bool reach = (s[1][0] + range[1] >= -0.5) && (s[0][0] + range[0] <= (double)snx + 0.5) &&
                       (s[3][0] + range[3] >= -0.5) && (s[2][0] + range[2] <= (double)sny + 0.5);
    live[blockIdx.x] = reach ? 1 : 0;
  }
}

// in place: live flags -> partial slot (ascending over live super-tiles) or -1; *n_slots = number of live super-tiles
__global__ void __launch_bounds__(1024) offset_slot_scan_kernel(int* __restrict__ slot, int n, int* __restrict__ n_slots) {
  __shared__ int s[1024];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = (i < n) ? slot[i] : 0;
    s[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
      const int add = ((int)threadIdx.x >= o) ? s[threadIdx.x - o] : 0;
      __syncthreads();
      s[threadIdx.x] += add;
      __syncthreads();
    }
    if (i < n) slot[i] = v ? carry + s[threadIdx.x] - 1 : -1;
    __syncthreads();
    if (threadIdx.x == 1023) carry += s[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_slots = carry;
}

// ---- TMA / mbarrier primitives (PTX: cp.async.bulk.tensor + mbarrier; SASS: UTMALDG, SYNCS) ----------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  unsigned done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, unsigned long long* bar, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<unsigned long long>(map)), "r"(smem_u32(bar)), "r"(x), "r"(y)
      : "memory");
}

// fixed-order block reduction through shared memory (8 warps): every thread ends with the same values
// four minima and two sums in one go (two barriers): v[0..3] -> block minima, v[4..5] -> block sums (fixed order)
__device__ __forceinline__ void block_min4_sum2(double (&v)[6], double* s_red, int lane, int warp) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = fmin(v[i], __shfl_xor_sync(0xffffffffu, v[i], o));
    v[4] += __shfl_xor_sync(0xffffffffu, v[4], o);
    v[5] += __shfl_xor_sync(0xffffffffu, v[5], o);
  }
  __syncthreads();
  if (lane < 6) {
    double mine = v[0];
#pragma unroll
    for (int i = 1; i < 6; ++i)
      if (lane == i) mine = v[i];
    s_red[warp * 6 + lane] = mine;
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double r = s_red[i];
#pragma unroll
    for (int w = 1; w < kOffWarps; ++w) r = (i < 4) ? fmin(r, s_red[w * 6 + i]) : r + s_red[w * 6 + i];
    v[i] = r;
  }
}

// explicit shared-memory loads on 32-bit shared addresses with immediate offsets: the window base is formed once per
// tile (through a generic pointer the compiler re-derived it -- S2UR SR_CgaCtaId, UMOV, ULEA -- for every sample)
template <int OFF>
__device__ __forceinline__ double lds_tap(unsigned a, float) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(a), "n"(OFF));
  return (double)v;
}
template <int OFF>
__device__ __forceinline__ double lds_tap(unsigned a, double) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1+%2];" : "=d"(v) : "r"(a), "n"(OFF));
  return v;
}
__device__ __forceinline__ void lds_px(unsigned a, double& tx, double& ty, double& ac) {
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(tx), "=d"(ty) : "r"(a));
  asm volatile("ld.shared.f64 %0, [%1+16];" : "=d"(ac) : "r"(a));
}

// One lag's walk over the live pixels of a tile, nine taps from the staged window (shared address `win` already
// offset to the tap of the first allowed floor index; row pitch = the box width). CHECK: the window holds a
// non-finite value or the -32762 fill somewhere, so every sample is tested; a clean window needs no test.
template <typename T, bool CHECK>
__device__ __forceinline__ void offset_walk_window(unsigned win, int lo_x, int lo_y, unsigned span_x, unsigned span_y,
                                                   const T* __restrict__ small, int snx, int sny, unsigned px,
                                                   int n_live, double x0h, double y0h, double pivot_b, double& sb,
                                                   double& sbb, double& sab, int& n_miss, double& sa_miss,
                                                   double& saa_miss, int& n_out, int& n_exact) {
  constexpr int ROW = OffBox<T>::W * (int)sizeof(T), E = (int)sizeof(T);
#pragma unroll kOffUnroll
  for (int k = 0; k < n_live; ++k, px += (unsigned)sizeof(OffPx)) {
    double ptx, pty, ac;
    lds_px(px, ptx, pty, ac);
    const double sx = x0h + ptx, sy = y0h + pty;   // coordinates + 0.5
    const double mx = __dadd_rd(sx, kMagic), my = __dadd_rd(sy, kMagic);
    const unsigned rx = (unsigned)(__double2loint(mx) - lo_x), ry = (unsigned)(__double2loint(my) - lo_y);
    double v;
    bool ok;
    // all nine taps inside the image and the window (which covers every coordinate this tile reaches under this
    // chunk's lags, so the magic-number floor is in range)
    if ((rx <= span_x) && (ry <= span_y)) {
      const double vx = sx - (mx - kMagic), vy = sy - (my - kMagic);   // = d + 0.5 in [0, 1)
      const double wx2 = (0.5 * vx) * vx;
      const double wx0 = (wx2 + 0.5) - vx;
      const double wx1 = fma(-2.0, wx2, vx + 0.5);
      const double wy2 = (0.5 * vy) * vy;
      const double wy0 = (wy2 + 0.5) - vy;
      const double wy1 = fma(-2.0, wy2, vy + 0.5);
      const unsigned a = win + ry * (unsigned)ROW + rx * (unsigned)E;
      const double r0 = fma(lds_tap<2 * E>(a, T()), wx2, fma(lds_tap<E>(a, T()), wx1, lds_tap<0>(a, T()) * wx0));
      const double r1 =
          fma(lds_tap<ROW + 2 * E>(a, T()), wx2, fma(lds_tap<ROW + E>(a, T()), wx1, lds_tap<ROW>(a, T()) * wx0));
      const double r2 = fma(lds_tap<2 * ROW + 2 * E>(a, T()), wx2,
                            fma(lds_tap<2 * ROW + E>(a, T()), wx1, lds_tap<2 * ROW>(a, T()) * wx0));
      v = fma(r2, wy2, fma(r1, wy1, r0 * wy0));
      ok = true;
      if (CHECK) ok = (((unsigned)__double2hiint(v) & 0x7FF00000u) != 0x7FF00000u) && (v != -32762.0);
    } else if ((sx < 0.5) || (sx > (double)snx - 0.5) || (sy < 0.5) || (sy > (double)sny - 0.5)) {
      // outside the image: exactly the closed-bound test 0 <= x <= n - 1 of the sampler on x = sx - 0.5 (the
      // subtraction is exact), without the call -- the common case on tiles at the rim of the small image's footprint
      ok = false;
      v = 0.0;
      ++n_out;
    } else {
      ++n_exact;
      ok = spline_sample<2, false, T>(small, sny, snx, sy - 0.5, sx - 0.5, v);
      // finite and not the -32762 fill (`np.where(image == -32762, nan, image)`, alignment.py:900-901)
      ok = ok && (((unsigned)__double2hiint(v) & 0x7FF00000u) != 0x7FF00000u) && (v != -32762.0);
    }
    if (ok) {
      const double bc = v - pivot_b;
      sb += bc;
      sbb = fma(bc, bc, sbb);
      sab = fma(ac, bc, sab);
    } else {
      ++n_miss;
      sa_miss += ac;
      saa_miss = fma(ac, ac, saa_miss);
    }
  }
}

// The same walk straight from the image in global memory: (tile, chunk) pairs whose window does not fit the box.
template <typename T>
__device__ __forceinline__ void offset_walk_global(const T* __restrict__ small, int snx, int sny,
                                                   const OffPx* __restrict__ s_px, int n_live, double x0h, double y0h,
                                                   double pivot_b, double& sb, double& sbb, double& sab, int& n_miss,
                                                   double& sa_miss, double& saa_miss) {
  const unsigned span_x = (unsigned)(snx - 3), span_y = (unsigned)(sny - 3);   // floor index in [1, n - 2]
  for (int k = 0; k < n_live; ++k) {
    const double ac = s_px[k].ac;
    const double sx = x0h + s_px[k].tx, sy = y0h + s_px[k].ty;
    const double mx = __dadd_rd(sx, kMagic), my = __dadd_rd(sy, kMagic);
    const unsigned rx = (unsigned)(__double2loint(mx) - 1), ry = (unsigned)(__double2loint(my) - 1);
    double v;
    bool ok;
    if ((rx <= span_x) && (ry <= span_y) && small_magnitude(sx) && small_magnitude(sy)) {
      const double vx = sx - (mx - kMagic), vy = sy - (my - kMagic);
      const double wx2 = (0.5 * vx) * vx;
      const double wx0 = (wx2 + 0.5) - vx;
      const double wx1 = fma(-2.0, wx2, vx + 0.5);
      const double wy2 = (0.5 * vy) * vy;
      const double wy0 = (wy2 + 0.5) - vy;
      const double wy1 = fma(-2.0, wy2, vy + 0.5);
      const T* r0p = small + ((size_t)ry * snx + rx);
      const T* r1p = r0p + snx;
      const T* r2p = r1p + snx;
      const double r0 = fma(ldval(r0p + 2), wx2, fma(ldval(r0p + 1), wx1, ldval(r0p) * wx0));
      const double r1 = fma(ldval(r1p + 2), wx2, fma(ldval(r1p + 1), wx1, ldval(r1p) * wx0));
      const double r2 = fma(ldval(r2p + 2), wx2, fma(ldval(r2p + 1), wx1, ldval(r2p) * wx0));
      v = fma(r2, wy2, fma(r1, wy1, r0 * wy0));
      ok = true;
    } else {
      ok = spline_sample<2, false, T>(small, sny, snx, sy - 0.5, sx - 0.5, v);
    }
    ok = ok && (((unsigned)__double2hiint(v) & 0x7FF00000u) != 0x7FF00000u) && (v != -32762.0);
    if (ok) {
      const double bc = v - pivot_b;
      sb += bc;
      sbb = fma(bc, bc, sbb);
      sab = fma(ac, bc, sab);
    } else {
      ++n_miss;
      sa_miss += ac;
      saa_miss = fma(ac, ac, saa_miss);
    }
  }
}

// does a window element force the per-sample test? (non-finite, or the reference's -32762 fill value)
__device__ __forceinline__ bool dirty_bits(unsigned u) {   // float32
  return ((u & 0x7F800000u) == 0x7F800000u) || (u == 0xC6FFF400u);
}
__device__ __forceinline__ bool dirty_value(float v) { return dirty_bits(__float_as_uint(v)); }
__device__ __forceinline__ bool dirty_value(double v) {
  return (((unsigned)__double2hiint(v) & 0x7FF00000u) == 0x7FF00000u) || (v == -32762.0);
}

template <typename T>
__global__ void __launch_bounds__(kOffThreads, kOffMinBlocks)
offset_window_kernel(const __grid_constant__ CUtensorMap tmap, int use_tma, const double* __restrict__ ref,
                     const T* __restrict__ small, int snx, int sny, int gnx, int gny, const double* __restrict__ tx,
                     const double* __restrict__ ty, const CoregLagOffset* __restrict__ lags, int n_lags,
                     int chunks_per_block, const double* __restrict__ pivots, const int* __restrict__ slot_of_super,
                     double* __restrict__ work, unsigned long long* __restrict__ stats) {
  constexpr int BW = OffBox<T>::W, BH = OffBox<T>::H;
  extern __shared__ __align__(128) unsigned char off_smem[];
  T* s_win = reinterpret_cast<T*>(off_smem);
  OffPx* s_px = reinterpret_cast<OffPx*>(off_smem + OffBox<T>::kBytes);
  double* s_red = reinterpret_cast<double*>(s_px + kOffTilePx);
  int* s_cnt = reinterpret_cast<int*>(s_red + 6 * kOffWarps);
  unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(s_cnt + 2 * kOffWarps);

  const int slot = slot_of_super[blockIdx.x];
  if (slot < 0) return;   // cannot reach the small image under any lag of this launch: no partial
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int sx_tiles = (gnx + kOffTileW - 1) / kOffTileW;
  const int ox = (blockIdx.x % sx_tiles) * kOffTileW, oy = (blockIdx.x / sx_tiles) * kOffSuperH;
  const double pivot_a = pivots[0], pivot_b = pivots[1];
  unsigned phase = 0;
  if (tid == 0) mbar_init(s_bar, 1);
  __syncthreads();

  const int n_chunks = (n_lags + kOffThreads - 1) / kOffThreads;
  const int c_end = min(n_chunks, ((int)blockIdx.y + 1) * chunks_per_block);
  for (int chunk = blockIdx.y * chunks_per_block; chunk < c_end; ++chunk) {
    const int lag = chunk * kOffThreads + tid;
    double x0h = CUDART_NAN, y0h = CUDART_NAN;
    if (lag < n_lags) {
      x0h = lags[lag].x0 + 0.5;
      y0h = lags[lag].y0 + 0.5;
    }
    const bool lag_ok = small_magnitude(x0h) && small_magnitude(y0h);   // false for NaN (dummy / dead lags)
    // spread of the chunk's offsets
    double lr[6] = {lag_ok ? x0h : CUDART_INF, lag_ok ? -x0h : CUDART_INF, lag_ok ? y0h : CUDART_INF,
                    lag_ok ? -y0h : CUDART_INF, 0.0, 0.0};
    block_min4_sum2(lr, s_red, lane, warp);
    const double lx0 = lr[0], lx1 = -lr[1], ly0 = lr[2], ly1 = -lr[3];
    const bool any_lag = lx0 <= lx1;

    double sb = 0.0, sbb = 0.0, sab = 0.0, sa_v = 0.0, saa_v = 0.0;
    int n_v = 0;
    for (int t = 0; t < kOffTilesPerBlock && any_lag; ++t) {
      // ---- live pixels of the tile -> shared table, in pixel order; their detector-plane box and reference moments
      double bx0 = CUDART_INF, bx1n = CUDART_INF, by0 = CUDART_INF, by1n = CUDART_INF, sa_t = 0.0, saa_t = 0.0;
      int base = 0;
      __syncthreads();   // previous tile's walk is over: table and window may be rewritten
#pragma unroll
      for (int pass = 0; pass < kOffTilePx / kOffThreads; ++pass) {
        const int i = pass * kOffThreads + tid;
        const int gx = ox + (i & (kOffTileW - 1)), gy = oy + t * kOffTileH + i / kOffTileW;
        double a = CUDART_NAN, px = CUDART_NAN, py = CUDART_NAN;
        if (gx < gnx && gy < gny) {
          const int64_t idx = (int64_t)gy * gnx + gx;
          a = ref[idx];
          px = __ldg(tx + idx);
          py = __ldg(ty + idx);
        }
        const bool live = isfinite(a) && small_magnitude(px) && small_magnitude(py);
        const unsigned bal = __ballot_sync(0xffffffffu, live);
        if (lane == 0) s_cnt[pass * kOffWarps + warp] = __popc(bal);
        __syncthreads();
        int before = base;
        for (int w = 0; w < warp; ++w) before += s_cnt[pass * kOffWarps + w];
        int total = 0;
        for (int w = 0; w < kOffWarps; ++w) total += s_cnt[pass * kOffWarps + w];
        if (live) {
          const double ac = a - pivot_a;
          OffPx e;
          e.tx = px; e.ty = py; e.ac = ac; e.pad = 0.0;
          s_px[before + __popc(bal & ((1u << lane) - 1u))] = e;
          bx0 = fmin(bx0, px); bx1n = fmin(bx1n, -px);
          by0 = fmin(by0, py); by1n = fmin(by1n, -py);
          sa_t += ac;
          saa_t = fma(ac, ac, saa_t);
        }
        base += total;
      }
      const int n_live = base;
      if (n_live == 0) continue;   // block-uniform
      double tr[6] = {bx0, bx1n, by0, by1n, sa_t, saa_t};
      block_min4_sum2(tr, s_red, lane, warp);
      bx0 = tr[0];
      const double bx1 = -tr[1];
      by0 = tr[2];
      const double by1 = -tr[3];
      sa_t = tr[4];
      saa_t = tr[5];
      // ---- window: every tap any (pixel, lag) pair of this tile and chunk can touch
      const double fx0 = floor(bx0 + lx0), fx1 = floor(bx1 + lx1), fy0 = floor(by0 + ly0), fy1 = floor(by1 + ly1);
      // (box and offsets passed small_magnitude: |.| < 2^31, the casts are exact)
      // TMA wants the box to start on a 16-byte boundary of the image row (a misaligned inner coordinate is an illegal
      // instruction: tools/ubench/tma_probe.cu): the window origin is rounded down to a multiple of 4 (2) pixels
      constexpr int kAlign = 16 / (int)sizeof(T);
      int wx0 = (int)fx0 - 1;
      wx0 -= ((wx0 % kAlign) + kAlign) % kAlign;
      const int wx1 = (int)fx1 + 1, wy0 = (int)fy0 - 1, wy1 = (int)fy1 + 1;
      if (wx1 < 0 || wx0 > snx - 1 || wy1 < 0 || wy0 > sny - 1) continue;   // nothing of it inside the image
      const bool fits = (wx1 - wx0 + 1 <= BW) && (wy1 - wy0 + 1 <= BH);
      if (stats != nullptr && tid == 0) {   // COREG_OFFSET_STATS=1: how the (tile, chunk) pairs were served
        atomicAdd(stats + (fits ? 0 : 1), 1ull);
        atomicAdd(stats + 2, (unsigned long long)n_live);
        atomicMax(stats + 3, (unsigned long long)(wx1 - wx0 + 1));
        atomicMax(stats + 4, (unsigned long long)(wy1 - wy0 + 1));
      }
      int lo_x = 1, lo_y = 1, hi_x = snx - 2, hi_y = sny - 2, base_off = 0, dirty = 0;
      if (fits) {
        lo_x = max(1, wx0 + 1);
        lo_y = max(1, wy0 + 1);
        hi_x = min(snx - 2, wx0 + BW - 2);
        hi_y = min(sny - 2, wy0 + BH - 2);
        base_off = (lo_y - 1 - wy0) * BW + (lo_x - 1 - wx0);
        if (use_tma) {
          if (tid == 0) {
            mbar_expect_tx(s_bar, (unsigned)OffBox<T>::kBytes);
            tma_load_2d(s_win, &tmap, s_bar, wx0, wy0);
          }
          mbar_wait(s_bar, phase);
          phase ^= 1u;
          // the whole box was just rewritten: look at it once, so that the walk can skip the per-sample test
          const uint4* w4 = reinterpret_cast<const uint4*>(s_win);
          for (int i = tid; i < OffBox<T>::kBytes / 16; i += kOffThreads) {
            const uint4 q = w4[i];
            if (sizeof(T) == 4)
              dirty |= dirty_bits(q.x) || dirty_bits(q.y) || dirty_bits(q.z) || dirty_bits(q.w);
            else
              dirty |= dirty_value(__hiloint2double((int)q.y, (int)q.x)) ||
                       dirty_value(__hiloint2double((int)q.w, (int)q.z));
          }
        } else {
          const int w = wx1 - wx0 + 1, h = wy1 - wy0 + 1;
          for (int i = tid; i < w * h; i += kOffThreads) {
            const int yy = i / w, xx = i - yy * w;
            const int gx = wx0 + xx, gy = wy0 + yy;
            T val = (T)0;
            if (gx >= 0 && gx < snx && gy >= 0 && gy < sny) val = __ldg(small + ((size_t)gy * snx + gx));
            dirty |= dirty_value(val);
            s_win[yy * BW + xx] = val;
          }
        }
      }
      unsigned span_x = 0, span_y = 0;
      if (hi_x >= lo_x && hi_y >= lo_y) {
        span_x = (unsigned)(hi_x - lo_x);
        span_y = (unsigned)(hi_y - lo_y);
      } else {
        lo_x = lo_y = 0x40000000;   // no pixel can take the fast path
      }
      dirty = __syncthreads_or(dirty);   // also: table complete, cooperative copy (if any) complete
      if (lag_ok) {
        int n_miss = 0, n_out = 0, n_exact = 0;
        double sa_miss = 0.0, saa_miss = 0.0, tsb = 0.0, tsbb = 0.0, tsab = 0.0;
        if (fits) {
          const unsigned win = smem_u32(s_win) + (unsigned)base_off * (unsigned)sizeof(T);
          if (dirty)
            offset_walk_window<T, true>(win, lo_x, lo_y, span_x, span_y, small, snx, sny, smem_u32(s_px), n_live, x0h,
                                        y0h, pivot_b, tsb, tsbb, tsab, n_miss, sa_miss, saa_miss, n_out, n_exact);
          else
            offset_walk_window<T, false>(win, lo_x, lo_y, span_x, span_y, small, snx, sny, smem_u32(s_px), n_live, x0h,
                                         y0h, pivot_b, tsb, tsbb, tsab, n_miss, sa_miss, saa_miss, n_out, n_exact);
        } else {
          offset_walk_global<T>(small, snx, sny, s_px, n_live, x0h, y0h, pivot_b, tsb, tsbb, tsab, n_miss, sa_miss,
                                saa_miss);
        }
        if (stats != nullptr) {
          atomicAdd(stats + 5, (unsigned long long)n_out);
          atomicAdd(stats + 6, (unsigned long long)n_exact);
          atomicAdd(stats + 7, (unsigned long long)(dirty ? 1 : 0));
        }
        // per tile, so that a tile this lag cannot reach adds exactly nothing -- whether the block skipped it for
        // the whole chunk or walked it for the sake of other lags (sharding-invariant partials)
        if (n_miss < n_live) {
          n_v += n_live - n_miss;
          sa_v += (n_miss == 0) ? sa_t : sa_t - sa_miss;
          saa_v += (n_miss == 0) ? saa_t : saa_t - saa_miss;
          sb += tsb;
          sbb += tsbb;
          sab += tsab;
        }
      }
    }
    if (lag < n_lags) {
      double* out = work + ((size_t)slot * n_lags + lag) * kMom;
      double4* o4 = reinterpret_cast<double4*>(out);
      o4[0] = make_double4((double)n_v, sa_v, sb, saa_v);
      o4[1] = make_double4(sbb, sab, 0.0, 0.0);
    }
  }
}

// fold the partials of the live super-tiles in slot order (= ascending super-tile index), moments -> Pearson r.
// One block = 32 consecutive lags x 8 moments: a slot's 2 KB of partials for those lags is one coalesced read.
__global__ void __launch_bounds__(256)
offset_finalize_kernel(const double* __restrict__ work, const int* __restrict__ n_slots_ptr, int n_lags,
                       double* __restrict__ corr, int64_t* __restrict__ nvalid) {
  __shared__ double s[32][kMom + 1];
  const int l0 = blockIdx.x * 32, t = threadIdx.x, lag = l0 + t / kMom, q = t % kMom;
  const int n_slots = *n_slots_ptr;
  double acc = 0.0;
  if (lag < n_lags) {
    const double* p = work + (size_t)lag * kMom + q;
    for (int sl = 0; sl < n_slots; ++sl) acc += p[(size_t)sl * n_lags * kMom];
  }
  s[t / kMom][q] = acc;
  __syncthreads();
  if (t < 32 && l0 + t < n_lags) {
    const double n = s[t][0], sa = s[t][1], sb = s[t][2], saa = s[t][3], sbb = s[t][4], sab = s[t][5];
    double r = CUDART_NAN;
    if (n > 0.0) {
      const double cov = sab - sa * sb / n;
      const double va = saa - sa * sa / n;
      const double vb = sbb - sb * sb / n;
      r = cov / sqrt(va * vb);
    }
    corr[l0 + t] = r;
    if (nvalid) nvalid[l0 + t] = (int64_t)n;
  }
}

// Per-block form of offset_finalize_kernel (CoregRegions): blockIdx.y = block of the grid. The block's super-tiles are
// walked in ascending index and their partials added serially from 0.0; slot order is ascending super-tile order, so
// one block covering the grid adds the same partials in the same order as the whole-grid fold. A super-tile without a
// slot in this launch contributes nothing, as in the whole-grid fold.
__global__ void __launch_bounds__(256)
offset_finalize_regions_kernel(const double* __restrict__ work, const int* __restrict__ slot_of_super, int n_lags,
                               int sx_tiles, int sy_tiles, int bt_h, int bt_w, int nbx, double* __restrict__ corr,
                               int64_t* __restrict__ nvalid, int64_t ld) {
  __shared__ double s[32][kMom + 1];
  const RegionTiles R = region_tiles(blockIdx.y, nbx, bt_h, bt_w, sx_tiles, sy_tiles);
  const int l0 = blockIdx.x * 32, t = threadIdx.x, lag = l0 + t / kMom, q = t % kMom;
  double acc = 0.0;
  if (lag < n_lags) {
    const double* p = work + (size_t)lag * kMom + q;
    for (int k = 0; k < R.n_tiles; ++k) {
      const int sl = slot_of_super[(R.ty0 + k / R.ntx) * sx_tiles + R.tx0 + k % R.ntx];
      if (sl >= 0) acc += p[(size_t)sl * n_lags * kMom];
    }
  }
  s[t / kMom][q] = acc;
  __syncthreads();
  if (t < 32 && l0 + t < n_lags) {
    const size_t o = (size_t)blockIdx.y * ld + l0 + t;
    corr[o] = pearson_from_moments(s[t][0], s[t][1], s[t][2], s[t][3], s[t][4], s[t][5]);
    nvalid[o] = (int64_t)s[t][0];
  }
}

// the per-block fold of the partials a launch_offset_fast call left in `work` (super-tiles of 32 x 64 grid pixels)
int launch_offset_regions(int gnx, int gny, int64_t n_lags, const void* work, const CoregRegions* rg, cudaStream_t s) {
  static_assert(kRegionAlign % kOffSuperH == 0 && kRegionAlign % kOffTileW == 0, "blocks hold whole super-tiles");
  const OffWork L = offw_layout(gnx, gny, n_lags);
  const char* base = static_cast<const char*>(work);
  const int sx_tiles = (gnx + kOffTileW - 1) / kOffTileW, sy_tiles = (gny + kOffSuperH - 1) / kOffSuperH;
  const int nbx = (gnx + rg->block_w - 1) / rg->block_w, nby = (gny + rg->block_h - 1) / rg->block_h;
  offset_finalize_regions_kernel<<<dim3((unsigned)((n_lags + 31) / 32), (unsigned)(nbx * nby)), 256, 0, s>>>(
      reinterpret_cast<const double*>(base + L.partials), reinterpret_cast<const int*>(base + L.slots), (int)n_lags,
      sx_tiles, sy_tiles, rg->block_h / kOffSuperH, rg->block_w / kOffTileW, nbx, rg->corr_dev, rg->nvalid_dev,
      rg->ld);
  CK_LAUNCH("offset_finalize_regions_kernel");
  return COREG_OK;
}

// ---- host side --------------------------------------------------------------------------------------------------
typedef CUresult (*TensorMapEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                           const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                           CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                           CUtensorMapFloatOOBfill);

static TensorMapEncodeTiledFn tensor_map_encoder() {
  static TensorMapEncodeTiledFn fn = []() -> TensorMapEncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<TensorMapEncodeTiledFn>(p);
  }();
  return fn;
}

// TMA descriptor of the small image with the window as its box; false when the image cannot be described (row pitch
// or base address not 16-byte aligned, driver without the entry point): the kernel then stages the window itself.
template <typename T>
static bool make_window_map(const T* small, int snx, int sny, CUtensorMap* map) {
  memset(map, 0, sizeof(*map));
  if (getenv("COREG_NO_TMA")) return false;
  TensorMapEncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return false;
  if ((reinterpret_cast<uintptr_t>(small) & 15u) || (((size_t)snx * sizeof(T)) & 15u)) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)snx, (cuuint64_t)sny};
  const cuuint64_t strides[1] = {(cuuint64_t)snx * sizeof(T)};
  const cuuint32_t box[2] = {(cuuint32_t)OffBox<T>::W, (cuuint32_t)OffBox<T>::H};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult rc = enc(map, sizeof(T) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2,
                          const_cast<T*>(small), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return rc == CUDA_SUCCESS;
}

template <typename T>
static int launch_offset_window(int gnx, int gny, int64_t n_lags, cudaStream_t s, const double* ref, const T* small,
                                int snx, int sny, const double* tx, const double* ty, const CoregLagOffset* lags,
                                const double* pivots, void* work, double* corr, int64_t* nvalid) {
  const OffWork L = offw_layout(gnx, gny, n_lags);
  char* base = static_cast<char*>(work);
  double* partials = reinterpret_cast<double*>(base + L.partials);
  int* slots = reinterpret_cast<int*>(base + L.slots);
  int* n_slots = reinterpret_cast<int*>(base + L.nslots);
  double* range = reinterpret_cast<double*>(base + L.range);
  offset_lag_range_kernel<<<1, 256, 0, s>>>(lags, (int)n_lags, range);
  offset_super_live_kernel<<<L.n_super, 256, 0, s>>>(ref, tx, ty, gnx, gny, snx, sny, range, slots);
  offset_slot_scan_kernel<<<1, 1024, 0, s>>>(slots, L.n_super, n_slots);
  CK_LAUNCH("offset pre-pass");
  CUtensorMap map;
  const int use_tma = make_window_map(small, snx, sny, &map) ? 1 : 0;
  const int n_chunks = (int)((n_lags + kOffThreads - 1) / kOffThreads);
  const int cpb = (n_chunks + 65534) / 65535;
  const dim3 grid(L.n_super, (n_chunks + cpb - 1) / cpb);
  const size_t smem = (size_t)OffBox<T>::kBytes + kOffTilePx * sizeof(OffPx) + 6 * kOffWarps * sizeof(double) +
                      2 * kOffWarps * sizeof(int) + 16;
  auto kern = offset_window_kernel<T>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const bool prof = g_prof_on && g_prof_n < 4096;
  if (prof) {
    CK(cudaEventCreate(&g_prof[g_prof_n].a));
    CK(cudaEventCreate(&g_prof[g_prof_n].b));
    CK(cudaEventRecord(g_prof[g_prof_n].a, s));
  }
  unsigned long long* stats = nullptr;
  if (getenv("COREG_OFFSET_STATS")) {
    CK(cudaMallocAsync(&stats, 8 * sizeof(unsigned long long), s));
    CK(cudaMemsetAsync(stats, 0, 8 * sizeof(unsigned long long), s));
  }
  kern<<<grid, kOffThreads, smem, s>>>(map, use_tma, ref, small, snx, sny, gnx, gny, tx, ty, lags, (int)n_lags, cpb,
                                       pivots, slots, partials, stats);
  CK_LAUNCH("offset_window_kernel");
  if (stats) {   // diagnostic only (synchronises)
    unsigned long long h[8];
    CK(cudaMemcpyAsync(h, stats, sizeof(h), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaFreeAsync(stats, s));
    fprintf(stderr, "[coreg offset kernel] tma=%d lags=%lld (tile, chunk) pairs: %llu staged, %llu global; %llu live "
            "pixel-walks (x 256 lanes); samples outside the image %llu, exact-path %llu; lane-tiles on a dirty window "
            "%llu; largest window asked for %llu x %llu (box %d x %d)\n", use_tma, (long long)n_lags, h[0], h[1], h[2],
            h[5], h[6], h[7], h[3], h[4], OffBox<T>::W, OffBox<T>::H);
  }
  if (prof) {
    CK(cudaEventRecord(g_prof[g_prof_n].b, s));
    ++g_prof_n;
  }
  offset_finalize_kernel<<<(unsigned)((n_lags + 31) / 32), 256, 0, s>>>(partials, n_slots, (int)n_lags, corr, nvalid);
  CK_LAUNCH("offset_finalize_kernel");
  return COREG_OK;
}

int launch_offset_fast(int gnx, int gny, int64_t n_lags, cudaStream_t s, const double* ref, const void* small,
                       int small_dtype, int snx, int sny, const double* tx, const double* ty,
                       const CoregLagOffset* lags, const double* pivots, void* work, double* corr, int64_t* nvalid) {
  if (small_dtype == COREG_F32)
    return launch_offset_window<float>(gnx, gny, n_lags, s, ref, (const float*)small, snx, sny, tx, ty, lags, pivots,
                                       work, corr, nvalid);
  return launch_offset_window<double>(gnx, gny, n_lags, s, ref, (const double*)small, snx, sny, tx, ty, lags, pivots,
                                      work, corr, nvalid);
}

}  // namespace coreg
