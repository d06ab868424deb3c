// coreg_lag_generic.cu -- generic fused lag kernel (orders 0-3, strict scipy arithmetic, any coordinate functor) and the tile-partial finalize.
#include "coreg_common.cuh"

namespace coreg {
// One block = one tile of the common grid (64 x 4*PPT pixels, PPT pixels per thread, their lag-independent
// constants in registers) x one slice of the lag list. work layout: [tile][lag][kMom] doubles.
// Moments: the sums over the reference image (Sa, Saa) are taken once over the pixels whose reference value is
// finite and corrected, per lag, by the (rare) pixels whose small-image sample is missing; Sb, Sbb, Sab and the
// count are accumulated per lag.
template <class Coord, int ORDER, bool STRICT, typename SmallT, typename RefT, bool ROUND32, int PPT, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
lag_corr_kernel(const RefT* __restrict__ ref, const SmallT* __restrict__ small, int snx, int sny, int gnx, int gny,
                typename Coord::Planes planes, const typename Coord::Lag* __restrict__ lags, int n_lags,
                int lags_per_block, const double* __restrict__ pivots, double* __restrict__ work) {
  typedef typename Coord::Lag Lag;
  typedef typename Coord::Pix Pix;
  constexpr int TILE_H = kRowsPerPass * PPT;
  __shared__ Lag s_lag[kLagSub];
  __shared__ double s_part[kWarps][kLagSub][kMom];

  const int tiles_x = (gnx + kTileW - 1) / kTileW;
  const int tile = blockIdx.x;
  const int tile_x = tile % tiles_x, tile_y = tile / tiles_x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = tid & (kTileW - 1), ty0 = tid / kTileW;
  const int gx = tile_x * kTileW + tx;
  const double pivot_a = pivots[0], pivot_b = pivots[1];

  Pix pix[PPT];
  double a_c[PPT];       // ref - pivot (0 where the reference pixel is missing)
  unsigned a_ok = 0;     // bit k: reference pixel k is finite
  double sa_all = 0.0, saa_all = 0.0;
#pragma unroll
  for (int k = 0; k < PPT; ++k) {
    const int gy = tile_y * TILE_H + ty0 + k * kRowsPerPass;
    a_c[k] = 0.0;
    pix[k] = Coord::dead();
    if (gx < gnx && gy < gny) {
      const int64_t idx = (int64_t)gy * gnx + gx;
      const double a = (double)ref[idx];
      if (isfinite(a)) {
        a_c[k] = a - pivot_a;
        a_ok |= 1u << k;
        pix[k] = Coord::load(planes, idx);
        sa_all += a_c[k];
        saa_all = fma(a_c[k], a_c[k], saa_all);
      }
    }
  }
  int n_all = __popc(a_ok);

  const int lag_begin = blockIdx.y * lags_per_block;
  const int lag_end = min(n_lags, lag_begin + lags_per_block);
  for (int l0 = lag_begin; l0 < lag_end; l0 += kLagSub) {
    const int cnt = min(kLagSub, lag_end - l0);
    __syncthreads();  // previous sub-chunk fully consumed
    {
      const double* src = reinterpret_cast<const double*>(lags + l0);
      double* dst = reinterpret_cast<double*>(s_lag);
      const int nd = cnt * (int)(sizeof(Lag) / sizeof(double));
      for (int i = tid; i < nd; i += kThreads) dst[i] = src[i];
    }
    __syncthreads();
    for (int l = 0; l < cnt; ++l) {
      const Lag L = s_lag[l];
      double sb = 0.0, sbb = 0.0, sab = 0.0, sa_miss = 0.0, saa_miss = 0.0;
      int n_miss = 0;
#pragma unroll
      for (int k = 0; k < PPT; ++k) {
        double x, y, v;
        Coord::map(pix[k], L, x, y);   // dead pixels carry NaN -> "outside"
        bool ok = spline_sample<ORDER, STRICT, SmallT>(small, sny, snx, y, x, v);
        double b;
        if (ROUND32) {
          const float bf = __double2float_rn(v);
          ok = ok && isfinite(bf);
          b = (double)bf;
        } else {
          ok = ok && isfinite(v) && (v != -32762.0);
          b = v;
        }
        if (ok) {
          const double bc = b - pivot_b;
          sb += bc;
          sbb = fma(bc, bc, sbb);
          sab = fma(a_c[k], bc, sab);
        } else if (a_ok & (1u << k)) {
          ++n_miss;
          sa_miss += a_c[k];
          saa_miss = fma(a_c[k], a_c[k], saa_miss);
        }
      }
      double m[8];
      m[0] = (double)(n_all - n_miss);
      m[1] = sa_all - sa_miss;
      m[2] = sb;
      m[3] = saa_all - saa_miss;
      m[4] = sbb;
      m[5] = sab;
      m[6] = 0.0;
      m[7] = 0.0;
      const double tot = warp_transpose_reduce8(m, lane);
      if ((lane & 3) == 0) s_part[warp][l][lane >> 2] = tot;
    }
    __syncthreads();
    // fold the warps in a fixed order and publish this tile's partials
    for (int i = tid; i < cnt * kMom; i += kThreads) {
      const int l = i / kMom, q = i % kMom;
      double s = s_part[0][l][q];
#pragma unroll
      for (int w = 1; w < kWarps; ++w) s += s_part[w][l][q];
      work[((size_t)tile * n_lags + (l0 + l)) * kMom + q] = s;
    }
  }
}

// one block per lag: sum the tile partials in a fixed order, moments -> Pearson r
__global__ void __launch_bounds__(128)
lag_corr_finalize_kernel(const double* __restrict__ work, int n_tiles, int n_lags, double* __restrict__ corr,
                         int64_t* __restrict__ nvalid) {
  __shared__ double s[128][6];
  const int lag = blockIdx.x;
  double m[6] = {0, 0, 0, 0, 0, 0};
  for (int t = threadIdx.x; t < n_tiles; t += 128) {
    const double* p = work + ((size_t)t * n_lags + lag) * kMom;
#pragma unroll
    for (int q = 0; q < 6; ++q) m[q] += p[q];
  }
#pragma unroll
  for (int q = 0; q < 6; ++q) s[threadIdx.x][q] = m[q];
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
#pragma unroll
      for (int q = 0; q < 6; ++q) s[threadIdx.x][q] += s[threadIdx.x + o][q];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double n = s[0][0], sa = s[0][1], sb = s[0][2], saa = s[0][3], sbb = s[0][4], sab = s[0][5];
    double r = CUDART_NAN;
    if (n > 0.0) {
      const double cov = sab - sa * sb / n;
      const double va = saa - sa * sa / n;
      const double vb = sbb - sb * sb / n;
      r = cov / sqrt(va * vb);
    }
    corr[lag] = r;
    if (nvalid) nvalid[lag] = (int64_t)n;
  }
}

int launch_finalize_tiles(const double* work, int tiles, int64_t n_lags, double* corr, int64_t* nvalid, cudaStream_t s) {
  lag_corr_finalize_kernel<<<(unsigned)n_lags, 128, 0, s>>>(work, tiles, (int)n_lags, corr, nvalid);
  CK_LAUNCH("lag_corr_finalize_kernel");
  return COREG_OK;
}

// Per-block form of lag_corr_finalize_kernel (CoregRegions): blockIdx.y = block of the grid. The block's tiles are taken
// in ascending order and its k-th tile goes to thread k % 128, as the whole-grid fold deals tile k: one block covering
// the grid folds the same sums in the same order.
__global__ void __launch_bounds__(128)
lag_corr_finalize_regions_kernel(const double* __restrict__ work, int n_lags, int tiles_x, int tiles_y, int bt_h,
                                 int bt_w, int nbx, double* __restrict__ corr, int64_t* __restrict__ nvalid,
                                 int64_t ld) {
  __shared__ double s[128][6];
  const RegionTiles R = region_tiles(blockIdx.y, nbx, bt_h, bt_w, tiles_x, tiles_y);
  const int lag = blockIdx.x;
  double m[6] = {0, 0, 0, 0, 0, 0};
  for (int k = threadIdx.x; k < R.n_tiles; k += 128) {
    const int t = (R.ty0 + k / R.ntx) * tiles_x + R.tx0 + k % R.ntx;
    const double* p = work + ((size_t)t * n_lags + lag) * kMom;
#pragma unroll
    for (int q = 0; q < 6; ++q) m[q] += p[q];
  }
#pragma unroll
  for (int q = 0; q < 6; ++q) s[threadIdx.x][q] = m[q];
  __syncthreads();
  for (int o = 64; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
#pragma unroll
      for (int q = 0; q < 6; ++q) s[threadIdx.x][q] += s[threadIdx.x + o][q];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const size_t o = (size_t)blockIdx.y * ld + lag;
    corr[o] = pearson_from_moments(s[0][0], s[0][1], s[0][2], s[0][3], s[0][4], s[0][5]);
    nvalid[o] = (int64_t)s[0][0];
  }
}

// the per-block fold of the tile partials a launch_lag call left in `work` (tiles of 64 x kMinTileH pixels)
int launch_finalize_tiles_regions(const double* work, int gnx, int gny, int64_t n_lags, const CoregRegions* rg,
                                  cudaStream_t s) {
  const int tiles_x = (gnx + kTileW - 1) / kTileW, tiles_y = (gny + kMinTileH - 1) / kMinTileH;
  const int nbx = (gnx + rg->block_w - 1) / rg->block_w, nby = (gny + rg->block_h - 1) / rg->block_h;
  lag_corr_finalize_regions_kernel<<<dim3((unsigned)n_lags, (unsigned)(nbx * nby)), 128, 0, s>>>(
      work, (int)n_lags, tiles_x, tiles_y, rg->block_h / kMinTileH, rg->block_w / kTileW, nbx, rg->corr_dev,
      rg->nvalid_dev, rg->ld);
  CK_LAUNCH("lag_corr_finalize_regions_kernel");
  return COREG_OK;
}

// generic kernel: 4 pixels per thread, 4 CTAs / SM. (Measured and dropped: 8 pixels per thread at 2 CTAs / SM,
// 115.7 vs 101.9 ms on 2048 x 1024 Carrington maps with 3600 lags, profiles/r1_widened_kernels.md.)
template <class Coord, int ORDER, bool STRICT, typename SmallT, typename RefT, bool ROUND32>
int launch_lag(int gnx, int gny, int64_t n_lags, int sms, cudaStream_t s, const RefT* ref, const SmallT* small, int snx,
               int sny, typename Coord::Planes planes, const typename Coord::Lag* lags, const double* pivots, double* w,
               int* tiles_out) {
  constexpr int PPT = 4, MINB = 4;
  static_assert(kRowsPerPass * PPT == kMinTileH, "the partials are sized for this tile height");
  dim3 grid;
  int lags_per_block;
  if (!lag_grid(kRowsPerPass * PPT, MINB, gnx, gny, n_lags, sms, &grid, &lags_per_block, tiles_out, kLagSub))
    return fail(COREG_EINVAL, "lag grid too large for one launch");
  lag_corr_kernel<Coord, ORDER, STRICT, SmallT, RefT, ROUND32, PPT, MINB><<<grid, kThreads, 0, s>>>(
      ref, small, snx, sny, gnx, gny, planes, lags, (int)n_lags, lags_per_block, pivots, w);
  return COREG_OK;
}

// the Carrington-frame window kernel serves the offset functor at order 2 with FMA arithmetic on images of at least
// 3 x 3 pixels; every other offset search takes the generic kernel (which the per-block fold must follow)
inline bool offset_window_applies(int order, int flags, int snx, int sny) {
  return order == 2 && !(flags & COREG_FLAG_STRICT) && snx >= 3 && sny >= 3 && !(flags & COREG_FLAG_NO_FAST);
}

template <class Coord, typename SmallT, typename RefT, bool ROUND32>
int launch_lag_corr(const RefT* ref, const SmallT* small, int snx, int sny, int gnx, int gny,
                    typename Coord::Planes planes, const typename Coord::Lag* lags, int64_t n_lags, int order,
                    const double* pivots, void* work, size_t work_bytes, double* corr, int64_t* nvalid, int flags,
                    cudaStream_t s) {
  if (n_lags <= 0) return COREG_OK;
  if (n_lags > (int64_t)1 << 30) return fail(COREG_EINVAL, "too many lags in one call (max 2^30)");
  if (gnx <= 0 || gny <= 0 || snx <= 0 || sny <= 0) return fail(COREG_EINVAL, "empty image");
  if ((int64_t)snx * sny >= ((int64_t)1 << 31)) return fail(COREG_EINVAL, "small image too large (>= 2^31 pixels)");
  int sms = coreg_device_sm_count();
  if (sms <= 0) sms = 148;
  const bool strict = (flags & COREG_FLAG_STRICT) != 0;
  double* w = static_cast<double*>(work);
  // window kernel for the offset (Carrington) functor: order 2, FMA arithmetic, image of at least 3x3
  const bool fast_ok = std::is_same<Coord, OffsetCoord>::value && offset_window_applies(order, flags, snx, sny);
  if (work_bytes < (fast_ok ? offset_workspace_bytes(gnx, gny, n_lags) : coreg_lag_corr_workspace_bytes(gnx, gny, n_lags)))
    return fail(COREG_ENOMEM, "workspace too small");
  if constexpr (std::is_same<Coord, OffsetCoord>::value) {
    if (fast_ok)
      return launch_offset_fast(gnx, gny, n_lags, s, ref, small, sizeof(SmallT) == 4 ? COREG_F32 : COREG_F64, snx, sny,
                                planes.tx, planes.ty, lags, pivots, work, corr, nvalid);
  }
  const bool prof = g_prof_on && g_prof_n < 4096;
  if (prof) {
    CK(cudaEventCreate(&g_prof[g_prof_n].a));
    CK(cudaEventCreate(&g_prof[g_prof_n].b));
    CK(cudaEventRecord(g_prof[g_prof_n].a, s));
  }
  int tiles = 0, rc = COREG_OK;
#define LAUNCH(ORD, STR)                                                                                         \
  rc = launch_lag<Coord, ORD, STR, SmallT, RefT, ROUND32>(gnx, gny, n_lags, sms, s, ref, small, snx, sny, planes, \
                                                          lags, pivots, w, &tiles)
  switch (order) {
    case 0: LAUNCH(0, true); break;
    case 1: LAUNCH(1, true); break;
    case 2: if (strict) LAUNCH(2, true); else LAUNCH(2, false); break;
    case 3: LAUNCH(3, true); break;
    default: return fail(COREG_EINVAL, "spline order must be 0..3");
  }
#undef LAUNCH
  if (rc) return rc;
  CK_LAUNCH("lag_corr_kernel");
  if (prof) {
    CK(cudaEventRecord(g_prof[g_prof_n].b, s));
    ++g_prof_n;
  }
  lag_corr_finalize_kernel<<<(unsigned)n_lags, 128, 0, s>>>(w, tiles, (int)n_lags, corr, nvalid);
  CK_LAUNCH("lag_corr_finalize_kernel");
  return COREG_OK;
}
}  // namespace coreg

using namespace coreg;

extern "C" {

size_t coreg_offset_window_workspace_bytes(int gnx, int gny, int64_t n_lags) {
  if (gnx <= 0 || gny <= 0 || n_lags <= 0) return 0;
  return offset_workspace_bytes(gnx, gny, n_lags);
}

size_t coreg_lag_corr_workspace_bytes(int gnx, int gny, int64_t n_lags) {
  if (gnx <= 0 || gny <= 0 || n_lags <= 0) return 0;
  return std::max(partials_bytes(gnx, gny, n_lags), offset_workspace_bytes(gnx, gny, n_lags)) +
         (size_t)n_lags * sizeof(HomLag);
}

int coreg_hpc_lag_corr(const float* ref, const void* small, int small_dtype, int snx, int sny, int gnx, int gny,
                       const double* planes, const CoregLagTan* lags, int64_t n_lags, int order,
                       const double* pivots, void* work, size_t work_bytes, double* corr, int64_t* nvalid, int flags,
                       void* stream) {
  if (!ref || !small || !planes || !lags || !pivots || !work || !corr)
    return fail(COREG_EINVAL, "coreg_hpc_lag_corr: null pointer");
  if (int rc = check_lag_flags(flags, "coreg_hpc_lag_corr")) return rc;
  TanCoord::Planes pl{planes, (int64_t)gnx * gny};
  cudaStream_t s = (cudaStream_t)stream;
  if (small_dtype == COREG_F64)
    return launch_lag_corr<TanCoord, double, float, true>(ref, (const double*)small, snx, sny, gnx, gny, pl, lags,
                                                          n_lags, order, pivots, work, work_bytes, corr, nvalid,
                                                          flags, s);
  if (small_dtype == COREG_F32)
    return launch_lag_corr<TanCoord, float, float, true>(ref, (const float*)small, snx, sny, gnx, gny, pl, lags,
                                                         n_lags, order, pivots, work, work_bytes, corr, nvalid, flags,
                                                         s);
  return fail(COREG_EINVAL, "small_dtype must be COREG_F32 or COREG_F64");
}

int coreg_hpc_lag_corr_regions(const float* ref, const void* small, int small_dtype, int snx, int sny, int gnx, int gny,
                               const double* planes, const CoregLagTan* lags, int64_t n_lags, int order,
                               const double* pivots, void* work, size_t work_bytes, double* corr, int64_t* nvalid,
                               const CoregRegions* regions, int flags, void* stream) {
  if (int rc = check_regions(regions, gnx, gny, n_lags, flags, "coreg_hpc_lag_corr_regions")) return rc;
  int rc = coreg_hpc_lag_corr(ref, small, small_dtype, snx, sny, gnx, gny, planes, lags, n_lags, order, pivots, work,
                              work_bytes, corr, nvalid, flags, stream);
  if (rc || n_lags <= 0) return rc;
  return launch_finalize_tiles_regions(static_cast<const double*>(work), gnx, gny, n_lags, regions,
                                       (cudaStream_t)stream);
}

int coreg_hpc_lag_corr_edge(const double* ref, const double* small_pad, int snx, int sny, int gnx, int gny,
                            const double* planes, const CoregLagTanEdge* lags, int64_t n_lags, const double* pivots,
                            void* work, size_t work_bytes, double* corr, int64_t* nvalid, int flags, void* stream) {
  if (!ref || !small_pad || !planes || !lags || !pivots || !work || !corr)
    return fail(COREG_EINVAL, "coreg_hpc_lag_corr_edge: null pointer");
  if (int rc = check_lag_flags(flags, "coreg_hpc_lag_corr_edge")) return rc;
  if (n_lags <= 0) return COREG_OK;
  if (n_lags > (int64_t)1 << 30) return fail(COREG_EINVAL, "too many lags in one call (max 2^30)");
  if (gnx <= 0 || gny <= 0 || snx <= 0 || sny <= 0) return fail(COREG_EINVAL, "empty image");
  const int pnx = snx + 2, pny = sny + 2;   // the padded image the kernel reads
  if ((int64_t)pnx * pny >= ((int64_t)1 << 31)) return fail(COREG_EINVAL, "small image too large (>= 2^31 pixels)");
  if (work_bytes < coreg_lag_corr_workspace_bytes(gnx, gny, n_lags)) return fail(COREG_ENOMEM, "workspace too small");
  int sms = coreg_device_sm_count();
  if (sms <= 0) sms = 148;
  cudaStream_t s = (cudaStream_t)stream;
  TanCoord::Planes pl{planes, (int64_t)gnx * gny};
  int tiles = 0;
  const bool prof = g_prof_on && g_prof_n < 4096;
  if (prof) {
    CK(cudaEventCreate(&g_prof[g_prof_n].a));
    CK(cudaEventCreate(&g_prof[g_prof_n].b));
    CK(cudaEventRecord(g_prof[g_prof_n].a, s));
  }
  // bilinear, scipy's operation order (what reproject calls), float64 reference, no float32 store
  int rc = launch_lag<TanEdgeCoord, 1, true, double, double, false>(gnx, gny, n_lags, sms, s, ref, small_pad, pnx, pny,
                                                                    pl, lags, pivots, static_cast<double*>(work), &tiles);
  if (rc) return rc;
  CK_LAUNCH("lag_corr_kernel<TanEdgeCoord>");
  if (prof) {
    CK(cudaEventRecord(g_prof[g_prof_n].b, s));
    ++g_prof_n;
  }
  return launch_finalize_tiles(static_cast<double*>(work), tiles, n_lags, corr, nvalid, s);
}

int coreg_hpc_lag_corr_edge_regions(const double* ref, const double* small_pad, int snx, int sny, int gnx, int gny,
                                    const double* planes, const CoregLagTanEdge* lags, int64_t n_lags,
                                    const double* pivots, void* work, size_t work_bytes, double* corr, int64_t* nvalid,
                                    const CoregRegions* regions, int flags, void* stream) {
  if (int rc = check_regions(regions, gnx, gny, n_lags, flags, "coreg_hpc_lag_corr_edge_regions")) return rc;
  int rc = coreg_hpc_lag_corr_edge(ref, small_pad, snx, sny, gnx, gny, planes, lags, n_lags, pivots, work, work_bytes,
                                   corr, nvalid, flags, stream);
  if (rc || n_lags <= 0) return rc;
  return launch_finalize_tiles_regions(static_cast<const double*>(work), gnx, gny, n_lags, regions,
                                       (cudaStream_t)stream);
}

int coreg_offset_lag_corr(const double* ref, const void* small, int small_dtype, int snx, int sny, int gnx, int gny,
                          const double* tx, const double* ty, const CoregLagOffset* lags, int64_t n_lags, int order,
                          const double* pivots, void* work, size_t work_bytes, double* corr, int64_t* nvalid,
                          int flags, void* stream) {
  if (!ref || !small || !tx || !ty || !lags || !pivots || !work || !corr)
    return fail(COREG_EINVAL, "coreg_offset_lag_corr: null pointer");
  if (int rc = check_lag_flags(flags, "coreg_offset_lag_corr")) return rc;
  OffsetCoord::Planes pl{tx, ty};
  cudaStream_t s = (cudaStream_t)stream;
  if (small_dtype == COREG_F64)
    return launch_lag_corr<OffsetCoord, double, double, false>(ref, (const double*)small, snx, sny, gnx, gny, pl,
                                                               lags, n_lags, order, pivots, work, work_bytes, corr,
                                                               nvalid, flags, s);
  if (small_dtype == COREG_F32)
    return launch_lag_corr<OffsetCoord, float, double, false>(ref, (const float*)small, snx, sny, gnx, gny, pl, lags,
                                                              n_lags, order, pivots, work, work_bytes, corr, nvalid,
                                                              flags, s);
  return fail(COREG_EINVAL, "small_dtype must be COREG_F32 or COREG_F64");
}

int coreg_offset_lag_corr_regions(const double* ref, const void* small, int small_dtype, int snx, int sny, int gnx,
                                  int gny, const double* tx, const double* ty, const CoregLagOffset* lags,
                                  int64_t n_lags, int order, const double* pivots, void* work, size_t work_bytes,
                                  double* corr, int64_t* nvalid, const CoregRegions* regions, int flags, void* stream) {
  if (int rc = check_regions(regions, gnx, gny, n_lags, flags, "coreg_offset_lag_corr_regions")) return rc;
  int rc = coreg_offset_lag_corr(ref, small, small_dtype, snx, sny, gnx, gny, tx, ty, lags, n_lags, order, pivots,
                                 work, work_bytes, corr, nvalid, flags, stream);
  if (rc || n_lags <= 0) return rc;
  // fold the records of the kernel that ran: the window kernel's slotted super-tile partials or the generic tiles
  if (offset_window_applies(order, flags, snx, sny))
    return launch_offset_regions(gnx, gny, n_lags, work, regions, (cudaStream_t)stream);
  return launch_finalize_tiles_regions(static_cast<const double*>(work), gnx, gny, n_lags, regions,
                                       (cudaStream_t)stream);
}

int coreg_car_lag_corr(const float* ref, const void* small, int small_dtype, int snx, int sny, int gnx, int gny,
                       const double* planes, const CoregLagCar* lags, int64_t n_lags, int order, const double* pivots,
                       void* work, size_t work_bytes, double* corr, int64_t* nvalid, int flags, void* stream) {
  if (!ref || !small || !planes || !lags || !pivots || !work || !corr)
    return fail(COREG_EINVAL, "coreg_car_lag_corr: null pointer");
  if (int rc = check_lag_flags(flags, "coreg_car_lag_corr")) return rc;
  CarCoord::Planes pl{planes, (int64_t)gnx * gny};
  cudaStream_t s = (cudaStream_t)stream;
  if (small_dtype == COREG_F64)
    return launch_lag_corr<CarCoord, double, float, true>(ref, (const double*)small, snx, sny, gnx, gny, pl, lags,
                                                          n_lags, order, pivots, work, work_bytes, corr, nvalid,
                                                          flags, s);
  if (small_dtype == COREG_F32)
    return launch_lag_corr<CarCoord, float, float, true>(ref, (const float*)small, snx, sny, gnx, gny, pl, lags,
                                                         n_lags, order, pivots, work, work_bytes, corr, nvalid, flags,
                                                         s);
  return fail(COREG_EINVAL, "small_dtype must be COREG_F32 or COREG_F64");
}

}  // extern "C"
