/*
 * coreg_b200.h -- C ABI of the B200-native lag-grid pointing search.
 *
 * Drop-in boundary for the hot path of adolliou/euispice_coreg v0.4.0 (pure Python; it has no FFI of
 * its own, so each entry point below names the Python function it replaces, file:line relative to the
 * reference checkout). Plain C types only: no torch / numpy / C++ types cross this boundary.
 *
 * Conventions
 *  - "dev" pointers are CUDA device pointers owned by the caller; "host" pointers are ordinary memory.
 *  - `stream` is a `cudaStream_t` passed as `void*` (NULL = default stream). Device entry points are
 *    stream-ordered: they enqueue work and return; they never synchronise, allocate or free.
 *  - Images are row-major [ny][nx] (FITS NAXIS2 x NAXIS1); pixel coordinates are 0-based (astropy origin 0).
 *  - Angles in `CoregTanWcs` are DEGREES (what wcslib holds after wcsset rescales CUNIT).
 *  - Return value: 0 on success, negative `COREG_E*` on error; `coreg_last_error()` gives the message of the
 *    last failure on the calling thread.
 */
#ifndef COREG_B200_H
#define COREG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COREG_OK 0
#define COREG_EINVAL (-1)  /* bad argument */
#define COREG_ECUDA (-2)   /* CUDA runtime error */
#define COREG_ENOMEM (-3)  /* workspace too small / allocation failed */

#define COREG_F32 0
#define COREG_F64 1
#define COREG_I32 2

/* flags of the lag-correlation kernels.
 * Default arithmetic: FP64 with fused multiply-add in the spline weights / tap sums (|dr| ~ 1e-15 vs strict).
 * COREG_FLAG_STRICT: scipy's exact operation order (separate multiply / add), bit-faithful per sample.
 * Bits 9..11 are reserved: every lag-correlation entry point returns COREG_EINVAL when one is set. */
#define COREG_FLAG_STRICT 1
/* COREG_FLAG_NO_FAST (value 4; 2 is reserved): force the generic kernel (testing / comparison). */
#define COREG_FLAG_NO_FAST 4
/* COREG_FLAG_MIXED: coreg_hpc_search_host only -- opt in to the mixed-arithmetic kernel (coreg_hpc_lag_corr_wcs_mixed) when
 * the small image is COREG_F32 and the fast form applies; the entry checks the kernel's per-lag guard and repeats the
 * search in FP64 when any lag trips it. Default (flag clear): all FP64, the reference's arithmetic. */
#define COREG_FLAG_MIXED 8
/* COREG_FLAG_PURE_SHIFT: every lag is a pure CRVAL shift; selects the rolling kernel (coreg_hpc_lag_corr_wcs,
 * coreg_hpc_lag_corr_wcs_mixed) without the adaptive segment; other kernels ignore it. Set it from the WHOLE lag grid:
 * both flavours are correct for any lag but round an irregular column segment differently, so every part of a sharded
 * grid must use the same one. */
#define COREG_FLAG_PURE_SHIFT 0x100

/* Constants of a 2-axis gnomonic (TAN) WCS. Replaces `astropy.wcs.WCS(hdr)`:
 * hdrshift/alignment.py:1041, utils/Util.py:284, synras/map_builder.py:119. */
typedef struct CoregTanWcs {
  double crpix1, crpix2; /* 1-based FITS reference pixel */
  double cdelt1, cdelt2; /* deg / pixel */
  double pc11, pc12, pc21, pc22;
  double crval1, crval2; /* deg */
  double lonpole;        /* deg (180 for TAN unless CRVAL2 >= 90) */
} CoregTanWcs;

/* One candidate ("lag") header in the helioprojective search, reduced on the host to the constants of its
 * world->pixel map. Replaces the per-lag `_shift_header` + `WCS(hdr_shifted)`:
 * hdrshift/alignment.py:401-468, 1041.  With (lng, lat) the world coordinate of a common-grid pixel and
 * A = lng - alpha_ref (alpha_ref = longitude the trig planes were built with):
 *   dA = A - (CRVAL1_lag - alpha_ref);  D = sin(lat) sin_d0 + cos(lat) cos_d0 cos(dA)
 *   xi = cos(lat) sin(dA) / D;  eta = (sin(lat) cos_d0 - cos(lat) sin_d0 cos(dA)) / D      [radians]
 *   x = m11 xi + m12 eta + x0;  y = m21 xi + m22 eta + y0                                  [0-based pixel]
 */
typedef struct CoregLagTan {
  double sin_da, cos_da;     /* sin / cos of (CRVAL1_lag - alpha_ref) */
  double sin_d0, cos_d0;     /* sin / cos of CRVAL2_lag */
  double m11, m12, m21, m22; /* (diag(CDELT) PC)^-1 * 180/pi */
  double x0, y0;             /* CRPIX - 1 */
} CoregLagTan;

/* One candidate header in the Carrington search whose only lag-dependent part is a detector-plane offset:
 *   x = x0 + Tx[pixel], y = y0 + Ty[pixel].  Replaces rectify.CarringtonTransform(hdr_shifted) per lag:
 * utils/rectify.py:377-404, hdrshift/alignment.py:889-901. */
typedef struct CoregLagOffset {
  double x0, y0;
} CoregLagOffset;

/* One plate-carree (-CAR) header reduced on the host to the constants of its world<->pixel maps: the common grid,
 * the large image, or one candidate ("lag") header of a search on images that already are Carrington maps
 * (CTYPE CRLN-CAR / CRLT-CAR). Replaces `_shift_header` + `WCS(hdr_shifted)` + wcslib's celset / sphs2x / cars2x:
 * hdrshift/alignment.py:344-399, 401-468, 1038-1069.  With c the unit vector of a world point
 * (cos lat cos lng, cos lat sin lng, sin lat):
 *   v = R c;  phi = atan2(v.y, v.x), theta = atan2(v.z, hypot(v.x, v.y))     [deg, native longitude / latitude]
 *   x = m11 phi + m12 theta + x0;  y = m21 phi + m22 theta + y0              [0-based pixel]
 * R = Rz(phi_p) . A(delta_p) . Rz(-alpha_p) from the header's Euler angles (celset). */
typedef struct CoregLagCar {
  double r[9];               /* row-major rotation, celestial -> native */
  double m11, m12, m21, m22; /* (diag(CDELT) PC)^-1, deg -> pixel */
  double x0, y0;             /* CRPIX - 1 */
  double lng_ref;            /* celestial longitude of the native pole [deg]: its sign picks the longitude range of
                                coreg_car_pix2world ([0, 360) when >= 0, (-360, 0] otherwise), as wcslib's sphx2s does */
} CoregLagCar;

/* Per-image constants of the Carrington ("fa") transform. Replaces rectify.CarringtonTransform.__init__ /
 * SphericalTransform.__init__: utils/rectify.py:314-338, 377-423. Angles in RADIANS (already converted on the
 * host exactly as the reference does with np.radians), cdelt in arcsec/pixel. */
typedef struct CoregCarrington {
  double lon0, lat0, roll; /* radians(CRLN_OBS), radians(CRLT_OBS), radians(CROTA) */
  double dist;             /* DSUN_OBS / (solar_r * R_sun) */
  double cdelt1, cdelt2;   /* header units per pixel (arcsec assumed by the reference) */
} CoregCarrington;

const char* coreg_last_error(void);
int coreg_version(void);
/* number of SMs of the current device (grid sizing); negative on error */
int coreg_device_sm_count(void);

/* ---- K3: pixel -> world for every pixel of an nx x ny TAN image ------------------------------------------
 * Replaces AlignEUIUtil.extract_EUI_coordinates (utils/Util.py:283-312) incl. ang2pipi (utils/Util.py:76-80).
 * lng_dev/lat_dev: [ny*nx] float64 degrees. wrap_pipi != 0 applies -((-a+180)%360-180). */
int coreg_tan_pix2world(const CoregTanWcs* wcs_host, int nx, int ny, int wrap_pipi, double* lng_dev,
                        double* lat_dev, void* stream);

/* ---- world -> pixel for n points through one TAN WCS -------------------------------------------------------
 * Replaces WCS(hdr).world_to_pixel(lon, lat): hdrshift/alignment.py:1065, synras/map_builder.py:127.
 * Points behind the tangent hemisphere give NaN. */
int coreg_tan_world2pix(const CoregTanWcs* wcs_host, const double* lng_dev, const double* lat_dev, int64_t n,
                        double* x_dev, double* y_dev, void* stream);

/* ---- spline resampling at given coordinates -----------------------------------------------------------------
 * Replaces AlignCommonUtil.interpol2d / rectify.interpol2d, i.e.
 * scipy.ndimage.map_coordinates(img, [y, x], order, mode='constant', cval, prefilter=False):
 * utils/Util.py:82-104, utils/rectify.py:22-56. order in 0..3. Same operation order as scipy (no FMA). */
int coreg_map_coordinates(const void* img_dev, int img_dtype, int img_ny, int img_nx, const double* y_dev,
                          const double* x_dev, int64_t n, int order, double cval, void* out_dev, int out_dtype,
                          void* stream);

/* ---- the one-time cut of a helioprojective search, fused ------------------------------------------------------
 * Replaces Alignment._create_submap_of_large_data (hdrshift/alignment.py:987-1016): extract_EUI_coordinates +
 * ang2pipi of the unshifted small grid (utils/Util.py:283-312, 76-80), WCS(hdr_large).world_to_pixel
 * (alignment.py:1065), interpol2d (utils/Util.py:82-104, cval NaN) and the float32 store (alignment.py:1024) in one
 * kernel: the same arithmetic as coreg_tan_pix2world -> coreg_tan_world2pix -> coreg_map_coordinates, the same bits,
 * no coordinate planes in memory. `large_dev` may be a window [origin_y:, origin_x:] of the image wcs_large describes.
 *   ref_dev  [ny*nx] float32: the large image on the small grid (the search's reference) */
int coreg_hpc_cut(const CoregTanWcs* wcs_small_host, int nx, int ny, const CoregTanWcs* wcs_large_host,
                  const void* large_dev, int large_dtype, int large_ny, int large_nx, int origin_x, int origin_y,
                  int order, float* ref_dev, void* stream);

/* ---- solar-surface reprojection (method_carrington_reprojection="sunpy") ------------------------------------------
 * Replaces Alignment._carrington_transform_sunpy (hdrshift/alignment.py:939-985), i.e. sunpy's
 * `Map.reproject_to(wcs)` under `propagate_with_solar_surface()` = reproject.reproject_interp (bilinear) through a
 * helioprojective -> helioprojective change of observer for points ON the solar surface, rotated differentially
 * (Howard et al., synodic) over the time between the two frames. Third-party algorithm, absent from the image:
 * restated from its published form, PARITY UNPINNED (oracle/surface_reproject.py, DESIGN.md section 4).
 *
 * coreg_pad_edge: reproject's `pad_edge_pixels`: out_dev [(ny+2)*(nx+2)] float64 = img with one replicated pixel around.
 * coreg_surface_cut: the one-time call -- the large image on the grid of the small one:
 *   for every pixel of the small grid: (Tx, Ty) through wcs_small, onto the sphere of radius rsun seen from `grid`
 *   (off-disc -> NaN), Stonyhurst longitude advanced by the differential rotation over dt_days, seen from `image`
 *   (points that observer cannot see -> NaN: reproject's round-trip check), pixel through wcs_large, bilinear sample
 *   of large_pad_dev (the edge-padded large image, coordinates within half a pixel of the array edge), float64.
 * coreg_hpc_lag_corr_edge: the per-lag call -- both frames come from the small image's header, so the change of
 *   observer is the identity and what is left is the helioprojective search's geometry with bilinear interpolation and
 *   reproject's edge rule: coreg_hpc_lag_corr with order 1 on the edge-padded small image, float64 reference, no
 *   float32 store; a lag row carries the bounds of the edge rule (xhi = snx - 0.5, yhi = sny - 0.5, unpadded). */
typedef struct CoregSurfaceFrames {
  double grid_lon, grid_lat, grid_dsun;    /* observer of the output grid: Stonyhurst lon / lat [rad], distance [m] */
  double image_lon, image_lat, image_dsun; /* observer of the input image */
  double dt_days;                          /* time of the input image - time of the output grid */
  double rsun;                             /* [m] */
} CoregSurfaceFrames;
typedef struct CoregLagTanEdge {
  CoregLagTan t;
  double xhi, yhi;
} CoregLagTanEdge;
int coreg_pad_edge(const void* img_dev, int dtype, int ny, int nx, double* out_dev, void* stream);
int coreg_surface_cut(const CoregTanWcs* wcs_small_host, int nx, int ny, const CoregTanWcs* wcs_large_host,
                      const double* large_pad_dev, int large_ny, int large_nx, const CoregSurfaceFrames* frames_host,
                      double* ref_dev, void* stream);
int coreg_hpc_lag_corr_edge(const double* ref_dev, const double* small_pad_dev, int snx, int sny, int gnx, int gny,
                            const double* planes_dev, const CoregLagTanEdge* lags_dev, int64_t n_lags,
                            const double* pivots_dev, void* work_dev, size_t work_bytes, double* corr_dev,
                            int64_t* nvalid_dev, int flags, void* stream);

/* ---- lag-independent per-pixel trig planes for the helioprojective search -----------------------------------
 * planes_dev: [3][n] float64 = sin(lat), cos(lat) sin(lng - alpha_ref), cos(lat) cos(lng - alpha_ref).
 * Hoists the lag-independent half of world_to_pixel out of the per-lag loop (hdrshift/alignment.py:1061-1065). */
int coreg_tan_trig_planes(const double* lng_dev, const double* lat_dev, int64_t n, double alpha_ref_deg,
                          double* planes_dev, void* stream);

/* ---- FITS tiled-image (RICE_1) decoder ---------------------------------------------------------------------------
 * Replaces what `astropy.io.fits` does inside `fits.open(path)[window].data` for a tile-compressed image HDU (the
 * form real Solar Orbiter L2 files come in): hdrshift/alignment.py:299-316, utils/Util.py:144-145. One thread per
 * tile; only the compressed heap crosses PCIe.
 *   heap_dev     the binary table's heap (device bytes)        offsets_dev / counts_dev  [n_tiles] start and length of
 *   each tile's COMPRESSED_DATA in the heap (table-row order = tiles in row-major order)
 *   tile_w/h     ZTILE1 / ZTILE2; nx, ny = ZNAXIS1 / ZNAXIS2; blocksize, bytepix = the ZVALn of BLOCKSIZE / BYTEPIX
 *   method       -1: integer image (out = the decoded integers, COREG_I32); 0 NO_DITHER, 1 SUBTRACTIVE_DITHER_1,
 *                2 SUBTRACTIVE_DITHER_2: floating-point image, out = (q - r + 0.5) * ZSCALE + ZZERO (COREG_F32 / F64)
 *   zscale_dev, zzero_dev [n_tiles]; zdither0 = ZDITHER0; blank = ZBLANK (-> NaN) when has_blank
 *   rand_dev     cfitsio's 10000-number dither sequence as float32 (fits_init_randoms) */
int coreg_rice_decode(const unsigned char* heap_dev, const long long* offsets_dev, const int* counts_dev, int n_tiles,
                      int tile_w, int tile_h, int nx, int ny, int blocksize, int bytepix, const double* zscale_dev,
                      const double* zzero_dev, int method, int zdither0, int has_blank, int blank,
                      const float* rand_dev, void* out_dev, int out_dtype, void* stream);

/* float32 image -> float64 on the device (exact). FITS BITPIX -32 payloads go up as float32 (half the H2D bytes of the
 * reference's host-side np.array(..., dtype=float64), hdrshift/alignment.py:299-316) and are widened once here: the lag
 * kernels read the small image fastest as float64 (no per-tap conversion). */
int coreg_widen_f32(const float* in_dev, int64_t n, double* out_dev, void* stream);

/* Big-endian 32-bit words -> native byte order on the device (in place when out_dev == in_dev). A FITS image is stored
 * big-endian; the reference lets astropy swap it on the host inside `hdul[w].data` (hdrshift/alignment.py:299-316).
 * Here the BITPIX -32 payload of the small image goes up as stored and is swapped where the bandwidth is. */
int coreg_bswap32(const void* in_dev, int64_t n_words, void* out_dev, void* stream);

/* ---- image statistics (pivots of the single-pass Pearson moments) ------------------------------------------------
 * One deterministic multi-block pass over an image: stats_dev[0] = mean of the finite values (the pivot: the Pearson
 * coefficient is invariant under it, it only keeps the single-pass moments well conditioned), stats_dev[stride] = their
 * count, stats_dev[2 stride] = max |v| over them, stats_dev[3 stride] = 0. With a COREG_F32 image and widen_dev != NULL
 * the same pass also writes the float64 copy (what coreg_widen_f32 does): the reference's
 * `np.array(hdul[w].data.copy(), dtype=np.float64)`, hdrshift/alignment.py:299-316, fused with the pivot.
 * The search kernels take `pivots_dev` = two such means side by side (ref, small): a [4][2] block filled with stride 2.
 * scratch_dev: coreg_image_stats_scratch_bytes() bytes, private to the call's stream while it runs. */
size_t coreg_image_stats_scratch_bytes(void);
int coreg_image_stats(const void* img_dev, int dtype, int64_t n, double* widen_dev, double* stats_dev, int stats_stride,
                      void* scratch_dev, void* stream);
/* Float32 twin of a float32 image CENTRED on the float32-rounded pivot, for the mixed-arithmetic kernel:
 * out_dev[i] = img_dev[i] - (float)stats_dev[0] (exact wherever pivot/2 <= v <= 2 pivot), and stats_dev[3 stride] =
 * RMS of the centred finite values. stats_dev[0] must hold the pivot (coreg_image_stats on the same stream before). */
int coreg_center_f32(const float* img_dev, int64_t n, float* out_dev, double* stats_dev, int stats_stride,
                     void* scratch_dev, void* stream);

/* ---- K1: fused helioprojective lag search ---------------------------------------------------------------------
 * For every lag: shift header -> world->pixel of every common-grid pixel -> order-k spline sample of the small
 * image -> round to float32 -> mask non-finite pairs -> Pearson r against `ref`.
 * Replaces Alignment._step + _interpolate_on_large_data_grid + interpol2d + c_correlate for a list of lags:
 * hdrshift/alignment.py:509-542, 1018-1029; utils/Util.py:82-104; hdrshift/c_correlate.py:39-72.
 *   ref_dev     [gny*gnx] float32  large image already on the common grid (output of the one-time resampling)
 *   small_dev   [sny*snx] small image, dtype small_dtype
 *   planes_dev  [3][gny*gnx] from coreg_tan_trig_planes
 *   lags_dev    [n_lags] CoregLagTan (device)
 *   pivots_dev  [2] device doubles: pivot of ref, pivot of small
 *   work_dev    scratch of at least coreg_lag_corr_workspace_bytes(gnx, gny, n_lags) bytes
 *   corr_dev    [n_lags] float64 out; nvalid_dev [n_lags] int64 out (may be NULL)
 */
size_t coreg_lag_corr_workspace_bytes(int gnx, int gny, int64_t n_lags);
int coreg_hpc_lag_corr(const float* ref_dev, const void* small_dev, int small_dtype, int snx, int sny, int gnx,
                       int gny, const double* planes_dev, const CoregLagTan* lags_dev, int64_t n_lags, int order,
                       const double* pivots_dev, void* work_dev, size_t work_bytes, double* corr_dev,
                       int64_t* nvalid_dev, int flags, void* stream);

/* ---- K1 (fast form): fused helioprojective lag search from headers --------------------------------------------------
 * Same computation and outputs as coreg_hpc_lag_corr for spline order 2 with FMA arithmetic and a float64 small image,
 * but each lag is given as the candidate header itself (CoregTanWcs = the output of _shift_header,
 * hdrshift/alignment.py:401-468) and the common grid as its own CoregTanWcs: two gnomonic projections of one sphere
 * are related by a plane homography, so the per-pixel map is three FMAs and a reciprocal on integer pixel indices --
 * no world-coordinate planes. The reciprocal is a 2- or 5-term series or a true division, chosen per lag on the
 * device from the exact range of the denominator over the grid (no caller guarantee needed). Threads walk grid
 * columns and share spline tap rows between consecutive pixels (column-rolling kernel, DESIGN.md section 5).
 *   grid_wcs_host  the common grid (the UNSHIFTED small header)          lag_wcs_dev  [n_lags] device array
 * Returns COREG_EINVAL for other orders / COREG_FLAG_STRICT (use coreg_hpc_lag_corr then). */
int coreg_hpc_lag_corr_wcs(const float* ref_dev, const double* small_dev, int snx, int sny, int gnx, int gny,
                           const CoregTanWcs* grid_wcs_host, const CoregTanWcs* lag_wcs_dev, int64_t n_lags,
                           int order, const double* pivots_dev, void* work_dev, size_t work_bytes, double* corr_dev,
                           int64_t* nvalid_dev, int flags, void* stream);

/* ---- K1 with per-block outputs: local correlation cubes from the same pass --------------------------------------------
 * The common grid is cut into blocks of block_h x block_w pixels starting at pixel (0, 0); the last block row and column
 * take whatever remains: nby = ceil(gny / block_h), nbx = ceil(gnx / block_w), block (i, j) is row b = i * nbx + j of
 * the outputs. Block sides are positive multiples of 64, so every block edge is a tile edge of both lag kernels and a
 * block's moments are sums of the tile records the whole-grid fold reads.
 *   corr_dev    [n_blocks][ld] float64 out: Pearson r of the block's pixels per lag (NaN where the block has no valid
 *               pixel pair under that lag)
 *   nvalid_dev  [n_blocks][ld] int64 out: the block's valid pixel pairs per lag; they sum to the whole-grid nvalid
 *   ld          elements between consecutive blocks' rows, >= n_lags (a launch over a slice [lo, hi) of a longer lag
 *               list writes columns lo .. hi - 1 when given corr_dev + lo, nvalid_dev + lo) */
typedef struct CoregRegions {
  int block_h, block_w;
  int64_t ld;
  double* corr_dev;
  int64_t* nvalid_dev;
} CoregRegions;

/* coreg_hpc_lag_corr_wcs / coreg_hpc_lag_corr + a CoregRegions: the whole-grid outputs exactly as the call without it,
 * then the per-block outputs, folded from the same tile records after the whole-grid finalize. A block's records are
 * taken in ascending order and dealt to the accumulator groups as the whole-grid fold deals them, so one block covering
 * the grid reproduces corr_dev / nvalid_dev bit for bit, and each lag's values depend only on its own records (not on
 * how a lag list is split into launches or ranks). Returns COREG_EINVAL before any CUDA call when `regions` or one of
 * its pointers is NULL, a block side is not a positive multiple of 64, ld < n_lags, the grid holds more than 65535
 * blocks, or flags has COREG_FLAG_MIXED (the mixed kernel's per-lag guard is calibrated on whole-grid moments). */
int coreg_hpc_lag_corr_wcs_regions(const float* ref_dev, const double* small_dev, int snx, int sny, int gnx, int gny,
                                   const CoregTanWcs* grid_wcs_host, const CoregTanWcs* lag_wcs_dev, int64_t n_lags,
                                   int order, const double* pivots_dev, void* work_dev, size_t work_bytes,
                                   double* corr_dev, int64_t* nvalid_dev, const CoregRegions* regions, int flags,
                                   void* stream);
int coreg_hpc_lag_corr_regions(const float* ref_dev, const void* small_dev, int small_dtype, int snx, int sny, int gnx,
                               int gny, const double* planes_dev, const CoregLagTan* lags_dev, int64_t n_lags, int order,
                               const double* pivots_dev, void* work_dev, size_t work_bytes, double* corr_dev,
                               int64_t* nvalid_dev, const CoregRegions* regions, int flags, void* stream);

/* ---- K1 (fast form, mixed arithmetic; opt-in) ------------------------------------------------------------------------
 * coreg_hpc_lag_corr_wcs with the projection in FP64 and the spline + per-segment moments in FP32, for a small image
 * whose pixels are float32 values (a BITPIX -32 FITS payload: what `Fits.open(...)[w].data` holds before the
 * reference widens it, hdrshift/alignment.py:299-316).
 *   small32c_dev  the payload centred on the float32-rounded pivot (coreg_center_f32); small_dev its float64 widening
 *                 (segments that touch the image border, a missing pixel or an irregular column are evaluated by the
 *                 exact per-pixel rules in FP64)
 *   stats_dev     the [4][2] statistics block (column 0 = ref, column 1 = small) of coreg_image_stats + coreg_center_f32;
 *                 its first row is the pivots
 *   flagged_dev   [n_lags] int32 out: 1 for every lag whose error model (FP32 rounding of the centred spline
 *                 against the sampled image's own variance, see coreg_lag_roll.cu:mixed_guard_trips) exceeds 1e-7 in
 *                 r, else 0. The caller re-evaluates the flagged lags with coreg_hpc_lag_corr_wcs (all FP64); the
 *                 decision is per lag, so a cube does not depend on how its lags were sharded. The reference computes every sample in FP64 and then stores it
 *                 as float32 (alignment.py:1024); this kernel reproduces that float32 store on the uncentred value,
 *                 so its samples equal the reference's except within a few float32 ulps OF THE DEVIATION FROM THE
 *                 PIVOT of a rounding boundary: |dr| <= 1e-7 by the model, ~1e-10 observed, independent of the image's
 *                 mean level. Without COREG_FLAG_PURE_SHIFT the kernel carries the adaptive segment for rotated /
 *                 rescaled lags; with it the adaptive segment is left out and x is taken as a line in the row index
 *                 where its quadratic term stays below 1e-11 pixel. */
int coreg_hpc_lag_corr_wcs_mixed(const float* ref_dev, const double* small_dev, const float* small32c_dev, int snx,
                                 int sny, int gnx, int gny, const CoregTanWcs* grid_wcs_host,
                                 const CoregTanWcs* lag_wcs_dev, int64_t n_lags, int order, const double* stats_dev,
                                 void* work_dev, size_t work_bytes, double* corr_dev, int64_t* nvalid_dev,
                                 int* flagged_dev, int flags, void* stream);

/* Diagnostic: max |e| = max |1 - D| of each candidate header's homography over the gnx x gny common grid (what selects
 * the reciprocal form per lag inside coreg_hpc_lag_corr_wcs). scratch_dev: at least 96 * n_lags bytes.
 * emax_dev: [n_lags] float64 out. */
int coreg_tan_homography_emax(const CoregTanWcs* grid_wcs_host, int gnx, int gny, const CoregTanWcs* lag_wcs_dev,
                              int64_t n_lags, void* scratch_dev, double* emax_dev, void* stream);

/* ---- K5 (coordinates): Carrington grid -> detector pixel of one header --------------------------------------------
 * Replaces CarringtonTransform / SphericalTransform.forward on the Rectifier grid
 * (utils/rectify.py:304-311, 340-363, 876-877). The Rectifier grid is separable (lon along x, lat along y) and the
 * reference evaluates its float32 half (np.linspace(dtype=float32), np.radians, sin/cos of the float32 latitude)
 * with NumPy; the host does exactly that on the two 1-D vectors and hands over, widened to float64:
 *   sinlon/coslon [n_lon] = sin/cos(float64(radians_f32(lon)) - radians(CRLN_OBS))
 *   sinlat/coslat [n_lat] = float64(sin_f32(radians_f32(lat))), float64(cos_f32(radians_f32(lat)))
 * The device does the per-pixel float64 part in NumPy's operation order (no FMA). Output planes [n_lat*n_lon]:
 * tx = degrees(atan(x2/z2))*3600/cdelt1, ty likewise (NaN where the point is behind the limb, zz < 0); the full
 * detector coordinate is x0 + tx with x0 = (CRPIX1-1) - dx/CDELT1 added per lag. */
int coreg_carrington_planes(const CoregCarrington* c_host, const double* sinlon_dev, const double* coslon_dev,
                            int n_lon, const double* sinlat_dev, const double* coslat_dev, int n_lat,
                            double* tx_dev, double* ty_dev, void* stream);

/* ---- K4: fused Carrington lag search (offset lags) ------------------------------------------------------------------
 * Replaces Alignment._step with function_to_apply=_carrington_transform_fa for lags that share `roll`:
 * hdrshift/alignment.py:509-542, 889-901; utils/rectify.py:865-888. ref is float64 here (the reference keeps the
 * Carrington-projected large image in float64), samples are NOT rounded to float32, and a sample equal to -32762
 * is treated as missing, like `np.where(image == -32762, nan, image)`. */
/* Workspace: coreg_lag_corr_workspace_bytes always suffices; order 2 without COREG_FLAG_STRICT / COREG_FLAG_NO_FAST (the
 * window kernel: one 64-byte partial per 32 x 64-pixel super-tile and lag) needs only
 * coreg_offset_window_workspace_bytes, about a quarter of it -- more lags per launch for the same memory. That kernel
 * serves 256 consecutive lags per block from one staged window of the small image: hand the lags over so that
 * consecutive ones are neighbours in the detector plane (e.g. 16 x 16 patches of the CRVAL grid, padded with NaN
 * dummies; `engine.offset_patch_order`), or it falls back to global loads. */
size_t coreg_offset_window_workspace_bytes(int gnx, int gny, int64_t n_lags);
int coreg_offset_lag_corr(const double* ref_dev, const void* small_dev, int small_dtype, int snx, int sny, int gnx,
                          int gny, const double* tx_dev, const double* ty_dev, const CoregLagOffset* lags_dev,
                          int64_t n_lags, int order, const double* pivots_dev, void* work_dev, size_t work_bytes,
                          double* corr_dev, int64_t* nvalid_dev, int flags, void* stream);

/* ---- Carrington-frame searches with per-block outputs (CoregRegions, as for K1 above) ----------------------------------
 * coreg_offset_lag_corr_regions: coreg_offset_lag_corr + a CoregRegions over the Carrington grid (rows = latitude
 *   samples, columns = longitude samples). The whole-grid outputs are exactly those of the call without it; then the
 *   per-block fold of the records of the kernel that ran: the window kernel's partials (one per live 32 x 64-pixel
 *   super-tile and lag, a block's super-tiles added in ascending order from 0.0, as the whole-grid fold adds its slots),
 *   or, for orders 0, 1, 3, COREG_FLAG_STRICT, COREG_FLAG_NO_FAST and images smaller than 3 x 3, the generic kernel's
 *   tile partials. A super-tile that no lag of a launch can bring onto the small image holds no partial and adds
 *   nothing, so a lag's block values do not depend on the launch it was part of.
 * coreg_hpc_lag_corr_edge_regions: coreg_hpc_lag_corr_edge + a CoregRegions over the small image's grid (the "sunpy"
 *   search), folded from the generic kernel's tile partials.
 * Both: one block covering the grid reproduces corr_dev / nvalid_dev bit for bit; COREG_EINVAL before any CUDA call on
 * the conditions of coreg_hpc_lag_corr_regions. */
int coreg_offset_lag_corr_regions(const double* ref_dev, const void* small_dev, int small_dtype, int snx, int sny,
                                  int gnx, int gny, const double* tx_dev, const double* ty_dev,
                                  const CoregLagOffset* lags_dev, int64_t n_lags, int order, const double* pivots_dev,
                                  void* work_dev, size_t work_bytes, double* corr_dev, int64_t* nvalid_dev,
                                  const CoregRegions* regions, int flags, void* stream);
int coreg_hpc_lag_corr_edge_regions(const double* ref_dev, const double* small_pad_dev, int snx, int sny, int gnx,
                                    int gny, const double* planes_dev, const CoregLagTanEdge* lags_dev, int64_t n_lags,
                                    const double* pivots_dev, void* work_dev, size_t work_bytes, double* corr_dev,
                                    int64_t* nvalid_dev, const CoregRegions* regions, int flags, void* stream);

/* ---- plate-carree (-CAR) images: the frame of Alignment.align_using_initial_carrington ------------------------------
 * hdrshift/alignment.py:344-399: both images already are Carrington maps; the search is the helioprojective one with
 * the CAR projection in place of TAN and no longitude wrapping (utils/Util.py:295-305).
 * coreg_car_pix2world: lng / lat [deg] of every pixel of an nx x ny image (extract_EUI_coordinates, utils/Util.py:283-
 *   305, for lon_ctype = "CRLN-CAR").  coreg_car_world2pix: WCS(hdr).world_to_pixel (hdrshift/alignment.py:1065).
 * coreg_car_lag_corr: same computation, outputs and workspace as coreg_hpc_lag_corr with planes_dev = the unit-vector
 *   planes of the common grid (coreg_tan_trig_planes with alpha_ref = 0) and one CoregLagCar per candidate header. */
int coreg_car_pix2world(const CoregLagCar* map_host, int nx, int ny, double* lng_dev, double* lat_dev, void* stream);
int coreg_car_world2pix(const CoregLagCar* map_host, const double* lng_dev, const double* lat_dev, int64_t n,
                        double* x_dev, double* y_dev, void* stream);
int coreg_car_lag_corr(const float* ref_dev, const void* small_dev, int small_dtype, int snx, int sny, int gnx,
                       int gny, const double* planes_dev, const CoregLagCar* lags_dev, int64_t n_lags, int order,
                       const double* pivots_dev, void* work_dev, size_t work_bytes, double* corr_dev,
                       int64_t* nvalid_dev, int flags, void* stream);

/* ---- pixel-shift lag search --------------------------------------------------------------------------------------
 * Replaces the lag loops of pxlshift.AlignmentPixels.find_best_parameters / _iteration_along_dy / _step and the numba
 * c_correlate they call: pxlshift/alignment_pixels.py:35-84, pxlshift/c_correlate.py:41-62. For every rotation k,
 * every dx[i] and every dy[j]: Pearson r of smalls[k] against large[y0 + dy : y0 + dy + sny, x0 + dx : x0 + dx + snx]
 * over the pixels where neither is NaN; the centred cross sum is rounded to float32 before the division, as the
 * reference stores it. (x0, y0) = the centred slice of `_initialise_slice_corresponding_to_small` (:145-148).
 *   large_dev   [lny*lnx] float64: the large image already at the small image's pixel size (coreg_map_coordinates)
 *   smalls_dev  [n_rot][sny*snx] float64: the small image rotated by each rotation lag (coreg_map_coordinates)
 *   lag_dx_host / lag_dy_host   integer displacements (host); a displacement that leaves the large image returns
 *                               COREG_EINVAL "too large shift : outside FSI" (`_check_boundaries`, :150-156)
 *   pivots_dev  [2]: pivot of large, pivot of smalls (coreg_finite_mean)
 *   corr_dev    [n_dx][n_dy][n_rot] float64 out; nvalid_dev same shape int64 (may be NULL) */
size_t coreg_pixel_shift_workspace_bytes(int snx, int sny, int n_dx, int n_dy, int n_rot);
int coreg_pixel_shift_corr(const double* large_dev, int lnx, int lny, const double* smalls_dev, int n_rot, int snx,
                           int sny, int x0, int y0, const int* lag_dx_host, int n_dx, const int* lag_dy_host, int n_dy,
                           const double* pivots_dev, void* work_dev, size_t work_bytes, double* corr_dev,
                           int64_t* nvalid_dev, void* stream);

/* ---- SPICE L2 cube -> 2-D image ---------------------------------------------------------------------------------
 * Replaces the host arithmetic of AlignmentSpice._prepare_spice_from_l2 (hdrshift/alignment_spice.py:250-276):
 * `np.array(hdu.data, float64)`, NaN above / below the slit, `np.nansum(data[0, sel], axis=0)`, NaN rows again.
 *   cube_dev  [n_lambda][ny][nx] float32 as the FITS file stores it (big_endian = 1) or native (0)
 *   sel_host  [n_lambda] 1 = plane inside the wavelength interval;  rows outside [ymin, ymax) -> NaN
 *   out_dev   [ny*nx] float64: planes added in ascending order in float64, NaN samples skipped (a pixel without a
 *             finite sample gives 0.0): the bits of numpy's reduction over the leading axis. Synchronises the stream. */
int coreg_spice_wave_sum(const void* cube_dev, int big_endian, int n_lambda, int ny, int nx,
                         const unsigned char* sel_host, int ymin, int ymax, double* out_dev, void* stream);

/* ---- K6: synthetic raster ----------------------------------------------------------------------------------------
 * Replaces the column loop of SPICEComposedMapBuilder._create_map_from_hdu (synras/map_builder.py:95-131):
 * output pixel (row j, column i) = order-k sample of imager frame frame_of_col[i] at the pixel position of the sky
 * point (lng[j,i], lat[j,i]) under that frame's TAN WCS; NaN outside. frames_dev: [n_frames][fny][fnx] float32/64,
 * wcs_host: [n_frames]; frame_of_col_host: [n_cols] (negative = column left NaN). out_dev float64 [n_rows*n_cols];
 * with float32 frames every sample is rounded to float32 first, as interpol2d(dst=None) returns the image dtype. */
int coreg_synras_build(const void* frames_dev, int frame_dtype, int n_frames, int fnx, int fny,
                       const CoregTanWcs* wcs_host, const int* frame_of_col_host, const double* lng_dev,
                       const double* lat_dev, int n_rows, int n_cols, int order, double* out_dev, void* stream);
/* The same with every frame given as a WINDOW of the image its WCS describes: frames_dev[f] = image_f[y0_f : y0_f + fny,
 * x0_f : x0_f + fnx], origin_xy_host = {x0_0, y0_0, x0_1, y0_1, ...} (NULL = whole frames). Coordinates are computed in
 * the full image and the integer origin is subtracted exactly, so the raster has the bits of coreg_synras_build on the
 * whole frames as long as every sampled position has its spline support inside the window: the host uploads a few
 * hundred pixels of each full-disc frame instead of 38 MB (SPICEComposedMapBuilder: 0.33 -> 0.03 s per raster). */
int coreg_synras_build_windows(const void* frames_dev, int frame_dtype, int n_frames, int fnx, int fny,
                               const CoregTanWcs* wcs_host, const int* origin_xy_host, const int* frame_of_col_host,
                               const double* lng_dev, const double* lat_dev, int n_rows, int n_cols, int order,
                               double* out_dev, void* stream);

/* ---- whole helioprojective search from HOST buffers (allocates, copies, runs, copies back, frees) ---------------
 * The call a non-Python host would make: replaces Alignment._find_best_header_parameters for the
 * helioprojective frame (hdrshift/alignment.py:613-797) given images and header constants.
 *   large_host [lny*lnx], small_host [sny*snx] (NaN = masked): COREG_F32 or COREG_F64 as given by *_dtype (float32
 *   FITS payloads need no widening on the host; the small image is widened once on the device).
 *   lag_wcs_host [n_lags] CoregTanWcs = the candidate headers (output of _shift_header, alignment.py:401-468).
 *   Order 2 without COREG_FLAG_STRICT / COREG_FLAG_NO_FAST runs the homography kernel (coreg_hpc_lag_corr_wcs),
 *   anything else the generic kernel (coreg_hpc_lag_corr).
 *   corr_host [n_lags] out, nvalid_host [n_lags] out (may be NULL). */
int coreg_hpc_search_host(const void* large_host, int large_dtype, int lnx, int lny, const CoregTanWcs* wcs_large,
                          const void* small_host, int small_dtype, int snx, int sny, const CoregTanWcs* wcs_small,
                          const CoregTanWcs* lag_wcs_host, int64_t n_lags, int order, int flags, double* corr_host,
                          int64_t* nvalid_host);

/* ---- the same search over several GPUs of one process ---------------------------------------------------------------
 * The reference spreads `np.array_split` chunks of the flat lag list over `multiprocessing.Process` workers
 * (hdrshift/alignment.py:667-744); here the chunks go to `n_devices` GPUs: one host thread per device, every device
 * holds both images and evaluates a contiguous slice of the lag list (ceil(n_lags / n_devices) lags each), the slices
 * land in corr_host / nvalid_host directly -- the gather is the host buffer. The cube is bit-identical to
 * coreg_hpc_search_host's for any device list (a device may be named more than once). Other arguments as there.
 * (Under torch.distributed the Python engine does the same with one process per GPU and one NCCL all-gather.) */
int coreg_hpc_search_host_multi(const int* devices_host, int n_devices, const void* large_host, int large_dtype, int lnx,
                                int lny, const CoregTanWcs* wcs_large, const void* small_host, int small_dtype, int snx,
                                int sny, const CoregTanWcs* wcs_small, const CoregTanWcs* lag_wcs_host, int64_t n_lags,
                                int order, int flags, double* corr_host, int64_t* nvalid_host);

/* ---- whole Carrington-frame search from HOST buffers -------------------------------------------------------------------
 * Replaces Alignment._find_best_header_parameters as driven by align_using_carrington(method_carrington_reprojection=
 * "fa") for CRVAL lags (hdrshift/alignment.py:144-261 -- the seam is the call at :237 --, 613-797, 889-901;
 * utils/rectify.py:377-423, 865-888): the large image is projected once onto the Carrington grid (float64, order-k
 * spline, fill -32762 -> NaN), then every lag's projection of the small image is correlated with it.
 *   c_large / c_small       per-image constants (CoregCarrington); x0_large, y0_large: the large header's detector
 *                           offset (`CarringtonTransform.__init__`, utils/rectify.py:394-404)
 *   sinlon_* / coslon_*     [n_lon] per image, sinlat / coslat [n_lat]: the float32 half of the Rectifier grid evaluated
 *                           by the host exactly as documented at coreg_carrington_planes
 *   lags_host               [n_lags] CoregLagOffset: x0, y0 of the small header under each CRVAL lag (same formula)
 *   order 2 without COREG_FLAG_STRICT / COREG_FLAG_NO_FAST runs the window kernel (the entry orders the lags into
 *   detector-plane patches itself), anything else the generic kernel. corr_host / nvalid_host: [n_lags] in the
 *   caller's lag order. */
int coreg_carrington_search_host(const void* large_host, int large_dtype, int lnx, int lny,
                                 const CoregCarrington* c_large, double x0_large, double y0_large,
                                 const void* small_host, int small_dtype, int snx, int sny,
                                 const CoregCarrington* c_small, const double* sinlon_large_host,
                                 const double* coslon_large_host, const double* sinlon_small_host,
                                 const double* coslon_small_host, int n_lon, const double* sinlat_host,
                                 const double* coslat_host, int n_lat, const CoregLagOffset* lags_host, int64_t n_lags,
                                 int order, int flags, double* corr_host, int64_t* nvalid_host);

/* ---- whole "sunpy" Carrington search from host buffers ---------------------------------------------------------------
 * _find_best_header_parameters as driven by align_using_carrington(method_carrington_reprojection="sunpy"): the call at
 * hdrshift/alignment.py:237 with function_to_apply = _carrington_transform_sunpy (:939-985). coreg_pad_edge +
 * coreg_surface_cut once, then coreg_hpc_lag_corr_edge over the candidate headers (CoregTanWcs rows = the output of
 * _shift_header, as for coreg_hpc_search_host). Restated third-party algorithm, parity unpinned (see coreg_surface_cut).
 *   frames_host  observers of the small image (= the output grid) and of the large image, time difference, rsun
 *   corr_host    [n_lags] float64 out; nvalid_host [n_lags] int64 out (may be NULL) */
int coreg_surface_search_host(const void* large_host, int large_dtype, int lnx, int lny,
                              const CoregTanWcs* wcs_large_host, const void* small_host, int small_dtype, int snx,
                              int sny, const CoregTanWcs* wcs_small_host, const CoregSurfaceFrames* frames_host,
                              const CoregTanWcs* lag_wcs_host, int64_t n_lags, int flags, double* corr_host,
                              int64_t* nvalid_host);

/* ---- synthetic raster from HOST buffers ----------------------------------------------------------------------------------
 * coreg_synras_build with the frame stack, the slit's sky coordinates and the raster in host memory: what
 * SPICEComposedMapBuilder.process -> _create_map_from_hdu computes between reading the imager files and writing the
 * composed FITS (synras/map_builder.py:57-79, 95-131). Arguments as coreg_synras_build. */
int coreg_synras_build_host(const void* frames_host, int frame_dtype, int n_frames, int fnx, int fny,
                            const CoregTanWcs* wcs_host, const int* frame_of_col_host, const double* lng_host,
                            const double* lat_host, int n_rows, int n_cols, int order, double* out_host);

/* ---- batched bounded 2-D Gaussian peak fits ---------------------------------------------------------------------------
 * The sub-lag fit of AlignmentResults._compute_shift (scipy curve_fit of twoD_Gaussian, bounded, on the points around a
 * cube's maximum) for n_problems cubes at once: least squares of
 *   f(x, y) = p5 + p0 exp(-((x - p1)^2 / (2 p3^2) + (y - p2)^2 / (2 p4^2)))
 * within lo <= p <= hi, by a bounded Levenberg-Marquardt with an active set, FP64, one warp per problem; sigma (p3, p4)
 * stays strictly above its lower bound. Deterministic: a problem's result does not depend on the batch it is in.
 *   points_dev     [n_problems][COREG_FIT_MAX_POINTS][3] float64: (x, y, value) of each point, the first n_points used
 *   n_points_dev   [n_problems] int32, 1 .. COREG_FIT_MAX_POINTS (other counts give COREG_FIT_NOT_CONVERGED)
 *   p0_dev         [n_problems][6] start, inside the bounds; bounds_dev [n_problems][12]: lo[6] then hi[6]
 *   popt_dev       [n_problems][6] out; cost_dev [n_problems] out: sum of squared residuals at popt
 *   iterations_dev [n_problems] int32 out; status_dev [n_problems] int32 out: COREG_FIT_CONVERGED or
 *                  COREG_FIT_NOT_CONVERGED (iteration cap reached, or a non-finite cost at the start)
 * Asynchronous on `stream`. COREG_EINVAL before any CUDA call for a null pointer or n_problems < 0. */
#define COREG_FIT_MAX_POINTS 26
#define COREG_FIT_CONVERGED 0
#define COREG_FIT_NOT_CONVERGED 3
int coreg_gauss2d_fit(const double* points_dev, const int* n_points_dev, const double* p0_dev, const double* bounds_dev,
                      int64_t n_problems, double* popt_dev, double* cost_dev, int* iterations_dev, int* status_dev,
                      void* stream);

/* Measurement hooks (bench.py): between begin and end every fused lag-kernel launch made by the calling thread is
 * bracketed by a CUDA event pair on its own stream; end() synchronises on them and returns the summed device time
 * of those launches [ms] and their count. No effect on results. */
int coreg_profile_begin(void);
int coreg_profile_end(double* lag_kernel_ms_total, int* launches);

/* FP64 issue-rate microbenchmark (dependent DFMA chains, all SMs): returns achieved FP64 FMA instructions/s in
 * *fma_per_s (lane-instructions, i.e. multiply by 2 for FLOP/s). Used by bench.py as the roofline denominator. */
int coreg_fp64_peak(double* fma_per_s, int iters, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* COREG_B200_H */
