// coreg_lag_roll.cu -- helioprojective frame: per-lag homographies and the column-rolling fused lag kernel (all-FP64 and mixed arithmetic).
#include "coreg_common.cuh"

namespace coreg {
// ---------------------------------------------------------------------------------------------------------
// Fast variant of the fused lag kernel: order-2 spline, FMA arithmetic.
//
// Helioprojective frame = homography. The common grid and every candidate header are gnomonic (TAN) projections
// of the same sphere from its centre, so pixel (i, j) of the common grid maps to the candidate's pixel through a
// plane projective transformation, exactly:
//      (nx, ny, D) = H (i, j, 1)^T ,   x = x0 + nx / D ,   y = y0 + ny / D ,
// H = [plane'->pixel'] . E(lag)^T Rz(alpha0 - alpha') E(grid) . [pixel->plane]   (3x3, one per lag, built by
// tan_homography_kernel from the two CoregTanWcs). No per-pixel trig, no world-coordinate planes; per sample the
// map costs 3 FMA + the reciprocal. D = cos(angle to the lag's reference point) * sqrt(1 + r^2) is within 2^-7 of 1
// for fields smaller than ~6 deg, where 1/D is the product form of the geometric series (1+e)(1+e^2)(1+e^4),
// e = 1 - D, exact to 2^-56 (COREG_FLAG_SMALL_ANGLE, guaranteed by the caller); otherwise a true division is used.
//
// Both functors deliver coordinates already offset by +0.5, so floor(x + 0.5) is one magic-number add, and
// "strictly interior" (all 9 taps inside the image: no closed-bound test, no mirroring) is one unsigned integer
// compare per axis on the floor index. Groups of pixels take the branch-free path together; anything else (image
// borders, missing reference pixels) falls back to the exact generic sampler with the same coordinates.
// ---------------------------------------------------------------------------------------------------------
struct HomGrid {  // pixel (i, j, 1) -> native direction (-Y, X, 1), and the grid's Euler matrix
  double c[3][3];
  double e[3][3];
  double a0_rad;
  double xmax, ymax;  // gnx - 1, gny - 1
};

// E(delta0, lonpole): native unit vector -> celestial frame whose x axis points at longitude alpha0
__host__ __device__ inline void euler_matrix(double sin_d, double cos_d, double sin_lp, double cos_lp, double (&e)[3][3]) {
  e[0][0] = -sin_d * cos_lp; e[0][1] = -sin_d * sin_lp; e[0][2] = cos_d;
  e[1][0] = sin_lp;          e[1][1] = -cos_lp;         e[1][2] = 0.0;
  e[2][0] = cos_d * cos_lp;  e[2][1] = cos_d * sin_lp;  e[2][2] = sin_d;
}

int make_hom_grid(const CoregTanWcs* w, int gnx, int gny, HomGrid* g) {
  TanDev t;
  int rc = make_tan(w, &t);
  if (rc) return rc;
  const double cx = t.f11 * (1.0 - t.crpix1) + t.f12 * (1.0 - t.crpix2);
  const double cy = t.f21 * (1.0 - t.crpix1) + t.f22 * (1.0 - t.crpix2);
  // d_native = (-Y, X, 1) with X = f11 i + f12 j + cx, Y = f21 i + f22 j + cy
  g->c[0][0] = -t.f21; g->c[0][1] = -t.f22; g->c[0][2] = -cy;
  g->c[1][0] = t.f11;  g->c[1][1] = t.f12;  g->c[1][2] = cx;
  g->c[2][0] = 0.0;    g->c[2][1] = 0.0;    g->c[2][2] = 1.0;
  euler_matrix(t.s0, t.c0, sin(t.lonpole_rad), cos(t.lonpole_rad), g->e);
  g->a0_rad = t.a0_rad;
  g->xmax = (double)(gnx - 1);
  g->ymax = (double)(gny - 1);
  return COREG_OK;
}

// reciprocal of the projective denominator D = 1 - e, chosen per lag (block-uniform) from the lag's emax:
//   |e| <= 2^-18 : 1 + e + e^2                    (2 ops, truncation e^3 <= 2^-54)
//   |e| <= 2^-7  : (1 + e)(1 + e^2)(1 + e^4)      (5 ops, truncation e^8 <= 2^-56)
//   otherwise    : true division; D <= 0 (behind the tangent hemisphere) -> NaN
constexpr double kTinyE = 3.814697265625e-06;  // 2^-18
constexpr double kSmallE = 0.0078125;          // 2^-7
// drift per row (|hx1|, |hy1 - 1|) above which a lag's segments may change a floor out of step: 2^-12 pixel, i.e. 2^-8
// pixel over a 16-row segment -- below it that practically never happens
constexpr double kRiskDriftPerRow = 0.000244140625;
// bound on hx1 he1 (P - 1)^2 [pixel] under which the rolling segment takes x as a line in the row index (1.000008 covers
// the factor 1 + 2e of the exact coefficient)
constexpr double kLinXTol = 0.99e-11;

__global__ void tan_homography_kernel(HomGrid g, const CoregTanWcs* __restrict__ lag_wcs, int n,
                                      HomLag* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  const CoregTanWcs w = lag_wcs[idx];
  double sd, cd, sl, cl, sa, ca;
  sincos(w.crval2 * kD2R, &sd, &cd);
  sincos(w.lonpole * kD2R, &sl, &cl);
  sincos(g.a0_rad - w.crval1 * kD2R, &sa, &ca);  // Rz(alpha0 - alpha')
  double e2[3][3];
  euler_matrix(sd, cd, sl, cl, e2);
  // m = Rz * E(grid) * C   (celestial direction in the lag's alpha frame, as a function of (i, j, 1))
  double ec[3][3], m[3][3], r[3][3];
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) ec[a][b] = g.e[a][0] * g.c[0][b] + g.e[a][1] * g.c[1][b] + g.e[a][2] * g.c[2][b];
#pragma unroll
  for (int b = 0; b < 3; ++b) {
    m[0][b] = ca * ec[0][b] - sa * ec[1][b];
    m[1][b] = sa * ec[0][b] + ca * ec[1][b];
    m[2][b] = ec[2][b];
  }
  // r = E(lag)^T m : native direction of the lag's projection
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) r[a][b] = e2[0][a] * m[0][b] + e2[1][a] * m[1][b] + e2[2][a] * m[2][b];
  // plane' = (r1 / r2, -r0 / r2) [rad]; pixel' = inv(cdelt pc) plane' + crpix - 1
  const double f11 = w.cdelt1 * w.pc11 * kD2R, f12 = w.cdelt1 * w.pc12 * kD2R;
  const double f21 = w.cdelt2 * w.pc21 * kD2R, f22 = w.cdelt2 * w.pc22 * kD2R;
  const double det = f11 * f22 - f12 * f21;
  const double i11 = f22 / det, i12 = -f12 / det, i21 = -f21 / det, i22 = f11 / det;
  HomLag h;
  h.hx0 = i11 * r[1][0] - i12 * r[0][0]; h.hx1 = i11 * r[1][1] - i12 * r[0][1]; h.hx2 = i11 * r[1][2] - i12 * r[0][2];
  h.hy0 = i21 * r[1][0] - i22 * r[0][0]; h.hy1 = i21 * r[1][1] - i22 * r[0][1]; h.hy2 = i21 * r[1][2] - i22 * r[0][2];
  h.he0 = -r[2][0]; h.he1 = -r[2][1]; h.he2 = 1.0 - r[2][2];
  h.x0h = (w.crpix1 - 1.0) + 0.5;
  h.y0h = (w.crpix2 - 1.0) + 0.5;
  // e = he0 i + he1 j + he2 is linear over the grid: its extreme values sit at the four corners
  const double e00 = h.he2, e10 = fma(h.he0, g.xmax, h.he2), e01 = fma(h.he1, g.ymax, h.he2),
               e11 = fma(h.he0, g.xmax, fma(h.he1, g.ymax, h.he2));
  double em = fmax(fmax(fabs(e00), fabs(e10)), fmax(fabs(e01), fabs(e11)));
  if (!(em == em) || !isfinite(h.hx0 + h.hx1 + h.hx2 + h.hy0 + h.hy1 + h.hy2)) em = CUDART_INF;
  const bool drifts = !(fmax(fabs(h.hx1), fabs(h.hy1 - 1.0)) <= kRiskDriftPerRow);
  h.emax = drifts ? -em : em;
  out[idx] = h;
}


__device__ __forceinline__ double recip_1me_tiny(double e) { return fma(e, e, 1.0 + e); }
__device__ __forceinline__ double recip_1me_small(double e) {
  const double e2 = e * e;
  double inv = 1.0 + e;
  inv = fma(e2, inv, inv);
  const double e4 = e2 * e2;
  return fma(e4, inv, inv);
}
__device__ __forceinline__ double recip_1me_div(double e) {
  const double den = 1.0 - e;
  return (den > 0.0) ? 1.0 / den : CUDART_NAN;
}

__global__ void abs_inplace_kernel(double* __restrict__ v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = fabs(v[i]);
}

// exact order-2 sample at (sx - 0.5, sy - 0.5) with float32 rounding / masking, kept out of line: only image
// borders, irregular columns and missing reference pixels come here
template <bool ROUND32>
__device__ __noinline__ bool sample_exact_half(const double* __restrict__ small, int sny, int snx, double sy,
                                               double sx, double* out) {
  double v;
  bool ok = spline_sample<2, false, double>(small, sny, snx, sy - 0.5, sx - 0.5, v);
  if (ROUND32) {
    const float bf = __double2float_rn(v);
    ok = ok && isfinite(bf);
    v = (double)bf;
  } else {
    ok = ok && isfinite(v) && (v != -32762.0);
  }
  *out = v;
  return ok;
}

// ---------------------------------------------------------------------------------------------------------
// Column-rolling form of the fused helioprojective lag kernel (order-2 spline, FMA arithmetic, float64 small image).
//
// A thread owns P CONSECUTIVE rows of one common-grid column. Under a candidate header the homography moves that
// column segment almost rigidly: x is constant to a small fraction of a pixel and y advances by one pixel per row,
// so floor(x + 0.5) is shared by the P pixels and floor(y + 0.5) increases by exactly one per row ("regular"
// column). The 3x3 tap windows of consecutive pixels then overlap in two of their three rows: the thread keeps a
// rolling window of three tap rows in registers and loads 3 new taps per pixel instead of 9 (3 (P + 2) / P per pixel
// overall) -- the L1 data pipe, not FP64 issue, bounded the per-pixel kernel. The fractional parts come from the
// shared floors (x - floor_x0, y - (floor_y0 + p)); whether they really lie in [0, 1) is checked per pixel with one
// integer compare on the high word, and a pixel that fails (a floor changed inside the segment: rotated lags, or a
// coordinate within 1e-7 of a half-integer) is re-evaluated by the exact out-of-line sampler, as is every pixel of
// a thread whose window touches the image border or whose reference pixels are not all finite. Results therefore
// equal the per-pixel kernel's up to the rounding of the reciprocal series.
// ---------------------------------------------------------------------------------------------------------
// The P pixels of a regular window, fully unrolled and free of branches, selects and predicates so that the
// independent dependency chains of consecutive pixels interleave (the FP64 pipe has an 8-cycle dependent-issue
// latency). MODE selects the reciprocal series (0: 1 + e + e^2, 1: three-factor product). Validity is tracked for the
// segment as a whole with two integer maxima: `vmax` over the high words of the fractional parts (all in [0, 1) <=>
// vmax < 0x3FF00000) and `bmax` over the magnitude bits of the float32 samples (all finite <=> bmax < 0x7F800000);
// the caller discards the sums and re-evaluates the segment pixel by pixel when either test fails.
// QUAD (MODE 0 only, |he1| < 2.2e-8): numerator x reciprocal as a quadratic in the row index p, coefficients formed
// once per lag -- two FMAs per coordinate instead of seven instructions for both (the form the mixed kernel uses;
// what it neglects, p^2 he1^2 of the reciprocal, is below 1e-9 pixel: tests/test_mixed_fraction_bits.py).
// LINX (with QUAD): x as a LINE in the row index -- its quadratic coefficient is hx1 he1 (1 + 2e), and a lag of pure
// CRVAL shifts has hx1 ~ 1e-7 and he1 ~ 1e-9 (x depends on the row only through the curvature of the projection), so
// over a 16-row segment the term stays below 1e-11 pixel (`kLinXTol`, tested per lag: block-uniform): one FMA less per
// pixel, 36.4 -> 35.2 ms on config 1.
template <int MODE, bool ROUND32, int P, bool QUAD = false, bool LINX = false>
__device__ __forceinline__ void roll_segment(const double* __restrict__ small, unsigned tap, unsigned row_elems,
                                             double be, double bnx, double bny, double he1, double hx1, double hy1,
                                             double inv0, double xoff, double yoff, double pivot_b,
                                             const double (&a_c)[P], double& sb, double& sbb, double& sab,
                                             unsigned& vmax, unsigned& bmax) {
  // A tap row (a, b, c) enters the result only through  a w0 + b w1 + c w2  with the order-2 B-spline weights
  // w0 = (1 - v)^2 / 2, w1 = 1/2 + v - v^2, w2 = v^2 / 2 of v = d + 0.5, i.e. through the quadratic
  //   A + v (B + v C),   A = (a + b) / 2,  B = b - a,  C = (a + c) / 2 - b.
  // A row serves three consecutive pixels of the column (each with its own v), so its coefficients are formed once
  // (5 operations per row) and every pixel evaluates three Horner forms in x (6 FMAs) and, the same way, one in y
  // (5 + 2): 13 + 5 (P + 2) / P operations per pixel instead of 12 for the weights plus 12 for the taps.
  // (Forming the coefficients once per image into three planes was measured slower: three times the L1 footprint.)
  auto row = [&](unsigned t, double& ca, double& cb, double& cc) {
    const double ta = __ldg(small + t), tb = __ldg(small + t + 1), tc = __ldg(small + t + 2);
    ca = 0.5 * (ta + tb);
    cb = tb - ta;
    cc = fma(0.5, ta + tc, -tb);
  };
  double r0a, r0b, r0c, r1a, r1b, r1c, r2a, r2b, r2c;
  row(tap, r0a, r0b, r0c);
  row(tap += row_elems, r1a, r1b, r1c);
  row(tap += row_elems, r2a, r2b, r2c);
  double qx0 = 0, qx1 = 0, qx2 = 0, qy0 = 0, qy1 = 0, qy2 = 0;
  if (QUAD) {
    const double dinv = fma(be + be, he1, he1);   // d(1 + e + e^2) / dp at the first pixel
    qx0 = fma(bnx, inv0, xoff);
    qy0 = fma(bny, inv0, yoff);
    qx1 = fma(hx1, inv0, bnx * dinv);
    qy1 = fma(hy1, inv0, bny * dinv) - 1.0;       // the shared floor of y advances by one per row
    qx2 = hx1 * dinv;
    qy2 = hy1 * dinv;
  }
#pragma unroll
  for (int p = 0; p < P; ++p) {
    // next row first: it is consumed one pixel later
    double r3a = 0.0, r3b = 0.0, r3c = 0.0;
    if (p + 1 < P) row(tap += row_elems, r3a, r3b, r3c);
    // fractional parts (+0.5) relative to the shared floors: v = d + 0.5 in [0, 1) on a regular column
    double vx, vy;
    if (QUAD) {
      if (LINX)
        vx = (p == 0) ? qx0 : fma(qx1, (double)p, qx0);
      else
        vx = (p == 0) ? qx0 : fma(fma(qx2, (double)p, qx1), (double)p, qx0);
      vy = (p == 0) ? qy0 : fma(fma(qy2, (double)p, qy1), (double)p, qy0);
    } else {
      const double e = (p == 0) ? be : fma(he1, (double)p, be);
      const double inv = (p == 0) ? inv0 : ((MODE == 0) ? recip_1me_tiny(e) : recip_1me_small(e));
      const double nx = (p == 0) ? bnx : fma(hx1, (double)p, bnx);
      const double ny = (p == 0) ? bny : fma(hy1, (double)p, bny);
      vx = fma(nx, inv, xoff);
      vy = fma(ny, inv, yoff - (double)p);
    }
    vmax = max(vmax, max((unsigned)__double2hiint(vx), (unsigned)__double2hiint(vy)));
    const double q0 = fma(fma(r0c, vx, r0b), vx, r0a);
    const double q1 = fma(fma(r1c, vx, r1b), vx, r1a);
    const double q2 = fma(fma(r2c, vx, r2b), vx, r2a);
    const double t = fma(fma(fma(0.5, q0 + q2, -q1), vy, q1 - q0), vy, 0.5 * (q0 + q1));
    double b;
    if (ROUND32) {
      // a non-finite float32 sample makes Sbb non-finite: the caller tests that once per segment
      b = (double)__double2float_rn(t);
    } else {
      // finite and not the -32762 fill: fold both into the same flag (the fill marks the sample as missing)
      const unsigned hi = (unsigned)__double2hiint(t) & 0x7FFFFFFFu;
      bmax = max(bmax, (t == -32762.0) ? 0x7F800000u : ((hi >= 0x7FF00000u) ? 0x7F800000u : 0u));
      b = t;
    }
    const double bc = b - pivot_b;
    sb += bc;
    sbb = fma(bc, bc, sbb);
    sab = fma(a_c[p], bc, sab);
    r0a = r1a; r0b = r1b; r0c = r1c;
    r1a = r2a; r1b = r2b; r1c = r2c;
    r2a = r3a; r2b = r3b; r2c = r3c;
  }
}

// The same segment in MIXED arithmetic: coordinates in FP64 (4 - 7 instructions per pixel), the spline and the segment's
// moments in FP32. The reference evaluates the spline in FP64 and then STORES the sample as float32
// (`alignment.py:1024`); what the Pearson sums see is round32(S). Here the FP32 spline runs on the small image
// CENTRED on the float32-rounded pivot p (c = v - p, exact by Sterbenz's lemma wherever p/2 <= v <= 2p and otherwise
// rounded to one float32 ulp of the DEVIATION), so its rounding errors scale with the local deviation from the
// pivot, not with the pixel value: t = spline(c) = S - p to ~4 ulp32(|c|). The reference's float32 store is then
// reproduced on the uncentred value: b = round32(t + p), bc = b - p -- two FADDs; b differs from the reference's
// sample only where S sits within ~4 ulp32(|c|) of a float32 rounding boundary of S (a fraction ~ulp32(|c|) /
// ulp32(S) of the samples, by one ulp32(S)). An image with mean 3e4 and sigma 1 therefore behaves like one with
// mean 0: the error model is data-independent and checked per lag by the finalize kernel (`mixed_guard`).
// A DFMA occupies the dispatch port for two cycles and an FFMA for one (profiles/r1_fp64_issue_model.md), so moving
// the spline / moment instructions off the FP64 pipe is what shortens the issue-bound loop.
// The fractional parts leave the FP64 domain without a conversion instruction: the coordinate FMA adds
// kFracMagic = 1.5 * 2^29, whose ulp is 2^-23, so the low word of the result is round((x - floor_x0) * 2^23): bits
// 23.. must be zero for x (p for y: the row index inside the segment), the low 23 bits are the float32 mantissa of
// 1 + frac. `vbad` collects the bits that must be zero; the caller re-evaluates the segment pixel by pixel when
// vbad >= 2^23 (a floor changed inside the segment, or a fraction rounded up to 1).
constexpr double kFracMagic = 805306368.0;   // 1.5 * 2^29

template <int MODE, int P, bool LINX = false>
__device__ __forceinline__ void roll_segment_mixed(const float* __restrict__ small32c, unsigned tap,
                                                   unsigned row_elems, double be, double bnx, double bny, double he1,
                                                   double hx1, double hy1, double inv0, double xoffm, double yoffm,
                                                   float pivot_b, const float (&a_c)[P], float& sb, float& sbb,
                                                   float& sab, unsigned& vbad) {
  // (Measured and dropped, profiles/r1_mixed_kernel.md: a per-image plane of these coefficients, one 16-byte load
  // per row and no arithmetic, is slower -- four times the L1 footprint; a 64-bit row pointer, walked or formed as
  // base + k * stride, compiles to four IADD3 per row where the 32-bit index + IMAD.WIDE form below costs two.)
  auto row = [&](unsigned t, float& ca, float& cb, float& cc) {
    const float ta = __ldg(small32c + t), tb = __ldg(small32c + t + 1), tc = __ldg(small32c + t + 2);
    ca = 0.5f * (ta + tb);
    cb = tb - ta;
    cc = fmaf(0.5f, ta + tc, -tb);
  };
  float r0a, r0b, r0c, r1a, r1b, r1c, r2a, r2b, r2c;
  row(tap, r0a, r0b, r0c);
  row(tap += row_elems, r1a, r1b, r1c);
  row(tap += row_elems, r2a, r2b, r2c);
  double qx0 = 0, qx1 = 0, qx2 = 0, qy0 = 0, qy1 = 0, qy2 = 0;
  if (MODE == 0) {
    const double dinv = fma(be + be, he1, he1);   // d(1 + e + e^2) / dp at the first pixel
    qx0 = fma(bnx, inv0, xoffm);
    qy0 = fma(bny, inv0, yoffm);
    qx1 = fma(hx1, inv0, bnx * dinv);
    qy1 = fma(hy1, inv0, bny * dinv);
    qx2 = hx1 * dinv;
    qy2 = hy1 * dinv;
  }
#pragma unroll
  for (int p = 0; p < P; ++p) {
    float r3a = 0.f, r3b = 0.f, r3c = 0.f;
    if (p + 1 < P) row(tap += row_elems, r3a, r3b, r3c);
    double cx, cy;   // coordinate - shared floor + kFracMagic
    if (MODE == 0) {
      // |e| <= 2^-18 over the whole grid and |he1| < 2.2e-8 (the caller's test): along the segment 1 / (1 - e) is
      // linear in p to p^2 he1^2 < 1.3e-13, so numerator x reciprocal is a quadratic in p whose coefficients are
      // formed once per lag: two FMAs per coordinate instead of seven instructions for both
      if (LINX)   // x as a line in p where its quadratic term is below kLinXTol (see roll_segment)
        cx = (p == 0) ? qx0 : fma(qx1, (double)p, qx0);
      else
        cx = (p == 0) ? qx0 : fma(fma(qx2, (double)p, qx1), (double)p, qx0);
      cy = (p == 0) ? qy0 : fma(fma(qy2, (double)p, qy1), (double)p, qy0);
    } else {
      const double e = (p == 0) ? be : fma(he1, (double)p, be);
      const double inv = (p == 0) ? inv0 : recip_1me_small(e);
      const double nx = (p == 0) ? bnx : fma(hx1, (double)p, bnx);
      const double ny = (p == 0) ? bny : fma(hy1, (double)p, bny);
      cx = fma(nx, inv, xoffm);
      cy = fma(ny, inv, yoffm);
    }
    const unsigned ux = (unsigned)__double2loint(cx);
    const unsigned uy = (unsigned)__double2loint(cy) ^ ((unsigned)p << 23);
    vbad |= ux | uy;
    const float vx = __uint_as_float(ux | 0x3F800000u) - 1.0f;
    const float vy = __uint_as_float(uy | 0x3F800000u) - 1.0f;
    const float q0 = fmaf(fmaf(r0c, vx, r0b), vx, r0a);
    const float q1 = fmaf(fmaf(r1c, vx, r1b), vx, r1a);
    const float q2 = fmaf(fmaf(r2c, vx, r2b), vx, r2a);
    // t = sample - pivot (the taps are centred); the reference's float32 store happens on the uncentred value
    const float t = fmaf(fmaf(fmaf(0.5f, q0 + q2, -q1), vy, q1 - q0), vy, 0.5f * (q0 + q1));
    const float bc = __fadd_rn(__fadd_rn(t, pivot_b), -pivot_b);
    sb += bc;
    sbb = fmaf(bc, bc, sbb);
    sab = fmaf(a_c[p], bc, sab);
    r0a = r1a; r0b = r1b; r0c = r1c;
    r1a = r2a; r1b = r2b; r1c = r2c;
    r2a = r3a; r2b = r3b; r2c = r3c;
  }
}

// The rolling segment for IRREGULAR columns: every pixel takes its own floors (the per-pixel rule), the three tap rows
// still roll. Under a rotated or rescaled candidate header x drifts by P |hx1| pixels along a segment and y by
// P |hy1 - 1| beyond one pixel per row, so in that fraction of the segments a floor moves "out of step" once -- and
// because neighbouring columns share the fractional parts to within the same drift, the segments of a warp do so
// together: on the 5-D grid of BASELINE configs[3] 16 % of the warps had more than ten such lanes and walked their
// segments pixel by pixel (9 taps each, five times the cost of a regular segment), 26 % a few
// (tools/irregular_segments.py). Here the window (r0, r1, r2) belongs to the tap index `wtap`; a pixel whose own tap
// index is the expected one (one row further) just rolls, any other reloads the three rows -- once or twice per
// segment. 10 FP64 instructions per pixel for coordinates (quadratics in the row index where the lag allows, else the
// series: 13), floors and fractions instead of 4, everything else as in
// `roll_segment`. Requires every pixel's 3 x 3 window strictly inside the image with one spare row / column (the
// caller checks the two end pixels with that margin; the coordinates are monotonic along the segment).
template <int MODE, bool ROUND32, int P, typename AT>
__device__ __forceinline__ bool roll_segment_adaptive(const double* __restrict__ small, unsigned row_elems, double be,
                                                      double bnx, double bny, double he1, double hx1, double hy1,
                                                      double x0h, double y0h, double pivot_b, const AT (&a_c)[P],
                                                      double& sb, double& sbb, double& sab) {
  // Four pixels per trip of a ROLLED loop: the four row-register sets (three window rows + the prefetched one) return to
  // their roles after four shifts, and the body stays ~6 KB. (Fully unrolled, this routine made the kernel's working
  // set of code exceed the 32 KB instruction cache: 15 % of the stall samples were "no instruction".)
  static_assert(P % 4 == 0, "four row-register sets");
  auto row = [&](unsigned t, double (&c)[3]) {
    const double ta = __ldg(small + t), tb = __ldg(small + t + 1), tc = __ldg(small + t + 2);
    c[0] = 0.5 * (ta + tb);
    c[1] = tb - ta;
    c[2] = fma(0.5, ta + tc, -tb);
  };
  double W[4][3];
#pragma unroll
  for (int k = 0; k < 4; ++k) W[k][0] = W[k][1] = W[k][2] = 0.0;
  unsigned wtap = 0xFFFFFFFFu, bmax = 0;   // no window yet: tap indices stay below 2^31
  double dp = 0.0;
  sb = sbb = sab = 0.0;
  // MODE 0 (|e| <= 2^-18 over the grid and |he1| < 2.2e-8, the caller's test): the coordinates as quadratics in the row
  // index, the form of `roll_segment` -- two FMAs each instead of seven instructions for both
  double qx0 = 0, qx1 = 0, qx2 = 0, qy0 = 0, qy1 = 0, qy2 = 0;
  if (MODE == 0) {
    const double inv0 = recip_1me_tiny(be);
    const double dinv = fma(be + be, he1, he1);
    qx0 = fma(bnx, inv0, x0h);
    qy0 = fma(bny, inv0, y0h);
    qx1 = fma(hx1, inv0, bnx * dinv);
    qy1 = fma(hy1, inv0, bny * dinv);
    qx2 = hx1 * dinv;
    qy2 = hy1 * dinv;
  }
#pragma unroll 1
  for (int p0 = 0; p0 < P; p0 += 4) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      double sx, sy;
      if (MODE == 0) {
        sx = fma(fma(qx2, dp, qx1), dp, qx0);
        sy = fma(fma(qy2, dp, qy1), dp, qy0);
      } else {
        const double e = fma(he1, dp, be);
        const double inv = recip_1me_small(e);
        sx = fma(fma(hx1, dp, bnx), inv, x0h);
        sy = fma(fma(hy1, dp, bny), inv, y0h);
      }
      const double mx = __dadd_rd(sx, kMagic), my = __dadd_rd(sy, kMagic);
      const unsigned tap = (unsigned)(__double2loint(my) - 1) * row_elems + (unsigned)(__double2loint(mx) - 1);
      const double vx = sx - (mx - kMagic), vy = sy - (my - kMagic);
      if (tap != wtap) {   // a floor moved other than by one row (and the first pixel)
        row(tap, W[k & 3]);
        row(tap + row_elems, W[(k + 1) & 3]);
        row(tap + 2u * row_elems, W[(k + 2) & 3]);
        wtap = tap;
      }
      // the row the next pixel most likely needs (inside the image: one spare row)
      row(wtap + 3u * row_elems, W[(k + 3) & 3]);
      const double(&r0)[3] = W[k & 3];
      const double(&r1)[3] = W[(k + 1) & 3];
      const double(&r2)[3] = W[(k + 2) & 3];
      const double q0 = fma(fma(r0[2], vx, r0[1]), vx, r0[0]);
      const double q1 = fma(fma(r1[2], vx, r1[1]), vx, r1[0]);
      const double q2 = fma(fma(r2[2], vx, r2[1]), vx, r2[0]);
      const double t = fma(fma(fma(0.5, q0 + q2, -q1), vy, q1 - q0), vy, 0.5 * (q0 + q1));
      double b;
      if (ROUND32) {
        b = (double)__double2float_rn(t);
      } else {
        const unsigned hi = (unsigned)__double2hiint(t) & 0x7FFFFFFFu;
        bmax = max(bmax, (t == -32762.0) ? 0x7F800000u : ((hi >= 0x7FF00000u) ? 0x7F800000u : 0u));
        b = t;
      }
      AT acs = a_c[k];
#pragma unroll
      for (int g = 1; g < P / 4; ++g)
        if (p0 == 4 * g) acs = a_c[4 * g + k];
      const double bc = b - pivot_b;
      sb += bc;
      sbb = fma(bc, bc, sbb);
      sab = fma((double)acs, bc, sab);
      wtap += row_elems;
      dp += 1.0;
    }
  }
  // every sample finite (as in the regular segment: a non-finite sample makes Sbb non-finite)
  return (bmax < 0x7F800000u) && (((unsigned)__double2hiint(sbb) & 0x7FF00000u) != 0x7FF00000u);
}

constexpr int kAdaptMin = 1;   // irregular lanes from which the whole warp takes the adaptive segment (measured 1 / 3 / 6: 15.0 / 15.7 / 16.6 us per lag)

// One pixel by the per-pixel rules: own floors, 9 taps when they are all inside the image, otherwise the exact
// out-of-line sampler. (sx, sy) are the coordinates + 0.5. Returns false when the sample is missing.
template <bool ROUND32>
__device__ __forceinline__ bool sample_pixel_half(const double* __restrict__ small, int sny, int snx,
                                                  unsigned row_elems, double sx, double sy, double* out) {
  const double mx = __dadd_rd(sx, kMagic), my = __dadd_rd(sy, kMagic);
  const int ix = __double2loint(mx), iy = __double2loint(my);
  const bool interior = small_magnitude(sx) && small_magnitude(sy) && ((unsigned)(ix - 1) < (unsigned)(snx - 2)) &&
                        ((unsigned)(iy - 1) < (unsigned)(sny - 2));
  if (!interior) return sample_exact_half<ROUND32>(small, sny, snx, sy, sx, out);
  const double vx = sx - (mx - kMagic), vy = sy - (my - kMagic);
  const double wx2 = (0.5 * vx) * vx;
  const double wx0 = (wx2 + 0.5) - vx;
  const double wx1 = fma(-2.0, wx2, vx + 0.5);
  const double wy2 = (0.5 * vy) * vy;
  const double wy0 = (wy2 + 0.5) - vy;
  const double wy1 = fma(-2.0, wy2, vy + 0.5);
  const double* r0p = small + ((unsigned)(iy - 1) * row_elems + (unsigned)(ix - 1));
  const double* r1p = r0p + row_elems;
  const double* r2p = r1p + row_elems;
  const double q0 = fma(__ldg(r0p + 2), wx2, fma(__ldg(r0p + 1), wx1, __ldg(r0p) * wx0));
  const double q1 = fma(__ldg(r1p + 2), wx2, fma(__ldg(r1p + 1), wx1, __ldg(r1p) * wx0));
  const double q2 = fma(__ldg(r2p + 2), wx2, fma(__ldg(r2p + 1), wx1, __ldg(r2p) * wx0));
  const double t = fma(q2, wy2, fma(q1, wy1, q0 * wy0));
  if (ROUND32) {
    const float bf = __double2float_rn(t);
    *out = (double)bf;
    return isfinite(bf);
  }
  *out = t;
  return isfinite(t) && (t != -32762.0);
}

// One lag for one thread's column segment: first-pixel coordinates, shared floors, window test, the regular rolling
// segment or -- image borders, irregular columns (rotated lags), missing pixels, division-mode lags -- the segment
// pixel by pixel. Out: the thread's Sb, Sbb, Sab over its valid samples and the mask of pixels that have a finite
// reference value but no valid sample.
template <bool ROUND32, int P, bool MIXED, bool ADAPT, typename AT>
__device__ __forceinline__ void roll_lag(const HomLag& C, const double* __restrict__ small,
                                         const float* __restrict__ small32, int snx, int sny, unsigned row_elems,
                                         double di, double dj0, const AT (&a_c)[P], unsigned a_ok, bool all_ref,
                                         double pivot_b, double& sb, double& sbb, double& sab, unsigned& miss,
                                         bool& slow) {
  const double hx1 = C.hx1, hy1 = C.hy1, he1 = C.he1, x0h = C.x0h, y0h = C.y0h;
  const int mode = (fabs(C.emax) <= kTinyE) ? 0 : ((fabs(C.emax) <= kSmallE) ? 1 : 2);  // block-uniform
  // numerators and e = 1 - D of the segment's first pixel (row gy0); pixel p adds p times the row slopes
  const double bnx = fma(hx1, dj0, fma(C.hx0, di, C.hx2));
  const double bny = fma(hy1, dj0, fma(C.hy0, di, C.hy2));
  const double be = fma(he1, dj0, fma(C.he0, di, C.he2));
  const double inv0 = (mode == 0) ? recip_1me_tiny(be) : ((mode == 1) ? recip_1me_small(be) : recip_1me_div(be));
  const double sx0 = fma(bnx, inv0, x0h), sy0 = fma(bny, inv0, y0h);  // coordinates + 0.5
  // floors shared by the segment
  const double mx0 = __dadd_rd(sx0, kMagic), my0 = __dadd_rd(sy0, kMagic);
  const int ix0 = __double2loint(mx0), iy0 = __double2loint(my0);
  const double xoff = x0h - (mx0 - kMagic), yoff = y0h - (my0 - kMagic);
  sb = sbb = sab = 0.0;
  // the quadratic term of x along the segment, hx1 he1 (1 + 2e) p^2 with |e| <= 2^-18, negligible? (block-uniform.)
  // Only in the flavour for lag grids of pure CRVAL shifts (!ADAPT), where every lag qualifies: in the flavour with the
  // adaptive segment one more instantiation of the unrolled segment pushes the hot code past the instruction cache
  // (5-D grid 14.1 -> 15.8 us per lag, measured), and its rotated / rescaled lags would not take it anyway.
  const bool lin_x = !ADAPT && fabs(hx1 * he1) * (double)((P - 1) * (P - 1)) < kLinXTol;
  // whole window inside the image: columns ix0-1 .. ix0+1, rows iy0-1 .. iy0+P; |coordinate| < 2^30 keeps the
  // magic-number floor meaningful (NaN fails the compare as well); division-mode lags go pixel by pixel
  bool fast = all_ref && (mode != 2) && small_magnitude(sx0) && small_magnitude(sy0) &&
              ((unsigned)(ix0 - 1) < (unsigned)(snx - 2)) && (iy0 >= 1) && (iy0 + P <= sny - 1);
  miss = 0;  // bit p: pixel p has a finite reference value but no valid sample
  slow = false;
  if (ADAPT && (P % 4 == 0) && mode != 2 && __double2hiint(C.emax) < 0) {   // block-uniform: the lag rotates / rescales
    // rotated / rescaled lag: do the floors of the last pixel follow from the first one's? If not for a few lanes of
    // the warp, all of it takes the adaptive segment (no lane waits for another's pixel-by-pixel walk)
    const double eL = fma(he1, (double)(P - 1), be);
    const double invL = (mode == 0) ? recip_1me_tiny(eL) : recip_1me_small(eL);
    const double sxL = fma(fma(hx1, (double)(P - 1), bnx), invL, x0h);
    const double syL = fma(fma(hy1, (double)(P - 1), bny), invL, y0h);
    const int ixL = __double2loint(__dadd_rd(sxL, kMagic)), iyL = __double2loint(__dadd_rd(syL, kMagic));
    const unsigned wx = (snx > 4) ? (unsigned)(snx - 4) : 0u, wy = (sny > 4) ? (unsigned)(sny - 4) : 0u;
    const bool inside2 = small_magnitude(sx0) && small_magnitude(sy0) && small_magnitude(sxL) && small_magnitude(syL) &&
                         ((unsigned)(ix0 - 2) < wx) && ((unsigned)(ixL - 2) < wx) && ((unsigned)(iy0 - 2) < wy) &&
                         ((unsigned)(iyL - 2) < wy);
    const bool irregular = (ixL != ix0) || (iyL != iy0 + P - 1);
    const unsigned b_ok = __ballot_sync(0xffffffffu, all_ref && inside2);
    const unsigned b_irr = __ballot_sync(0xffffffffu, irregular);
    if (b_ok == 0xffffffffu && __popc(b_irr) >= kAdaptMin) {
      bool ok = false;
      if constexpr (ADAPT && P % 4 == 0)
        ok = (mode == 0 && fabs(he1) < 2.2e-8)
                 ? roll_segment_adaptive<0, ROUND32, P, AT>(small, row_elems, be, bnx, bny, he1, hx1, hy1, x0h,
                                                                    y0h, pivot_b, a_c, sb, sbb, sab)
                         : roll_segment_adaptive<1, ROUND32, P, AT>(small, row_elems, be, bnx, bny, he1, hx1, hy1, x0h,
                                                                    y0h, pivot_b, a_c, sb, sbb, sab);
      slow = !ok;   // a non-finite sample: pixel by pixel
      if (!ok) sb = sbb = sab = 0.0;
      return;
    }
  }
  if constexpr (MIXED) {
    // the low word of coordinate + kFracMagic holds the offset from the shared floor only while that offset stays
    // below 2^9 pixels: true for any sane lag, guaranteed here by bounding the per-row slopes (block-uniform test)
    fast = fast && (fabs(hx1) < 8.0) && (fabs(hy1) < 8.0);
    if (fast) {
      const unsigned tap = (unsigned)(iy0 - 1) * row_elems + (unsigned)(ix0 - 1);
      // xoff + kFracMagic rounds to 2^-23 pixel; the residual (exact) goes into the numerator, whose factor inv is
      // 1 + O(2^-7): what is lost is below 1e-9 pixel, the same for every pixel of the lag
      const double xoffm = xoff + kFracMagic, yoffm = yoff + kFracMagic;
      const double bnx2 = bnx + (xoff - (xoffm - kFracMagic)), bny2 = bny + (yoff - (yoffm - kFracMagic));
      float fsb = 0.f, fsbb = 0.f, fsab = 0.f;
      unsigned vbad = 0;
      // the quadratic form of the coordinates drops p^2 he1^2 of the reciprocal: below 1e-9 pixel for |he1| < 2.2e-8
      // (P <= 16 rows, numerators below 8192 pixels) -- any 2048-row grid in this mode has |he1| < 4e-9; a small grid
      // with a steep denominator takes the per-pixel series instead (block-uniform choice)
      if (!ADAPT && mode == 0 && fabs(he1) < 2.2e-8 && lin_x) {
        if constexpr (!ADAPT)
          roll_segment_mixed<0, P, true>(small32, tap, row_elems, be, bnx2, bny2, he1, hx1, hy1, inv0, xoffm, yoffm,
                                         (float)pivot_b, a_c, fsb, fsbb, fsab, vbad);
      } else if (mode == 0 && fabs(he1) < 2.2e-8)
        roll_segment_mixed<0, P>(small32, tap, row_elems, be, bnx2, bny2, he1, hx1, hy1, inv0, xoffm, yoffm,
                                 (float)pivot_b, a_c, fsb, fsbb, fsab, vbad);
      else
        roll_segment_mixed<1, P>(small32, tap, row_elems, be, bnx2, bny2, he1, hx1, hy1, inv0, xoffm, yoffm,
                                 (float)pivot_b, a_c, fsb, fsbb, fsab, vbad);
      // every offset inside its cell, every sample finite (a non-finite sample makes Sbb non-finite; so does a
      // finite sample beyond 1.8e19, which then just takes the exact path)
      fast = (vbad < 0x00800000u) && ((__float_as_uint(fsbb) & 0x7F800000u) != 0x7F800000u);
      sb = (double)fsb;
      sbb = (double)fsbb;
      sab = (double)fsab;
    }
  } else if (fast) {
    const unsigned tap = (unsigned)(iy0 - 1) * row_elems + (unsigned)(ix0 - 1);
    unsigned vmax = 0, bmax = 0;
    if (!ADAPT && mode == 0 && fabs(he1) < 2.2e-8 && lin_x) {
      if constexpr (!ADAPT)
        roll_segment<0, ROUND32, P, true, true>(small, tap, row_elems, be, bnx, bny, he1, hx1, hy1, inv0, xoff, yoff,
                                                pivot_b, a_c, sb, sbb, sab, vmax, bmax);
    } else if (mode == 0 && fabs(he1) < 2.2e-8)
      roll_segment<0, ROUND32, P, true>(small, tap, row_elems, be, bnx, bny, he1, hx1, hy1, inv0, xoff, yoff,
                                        pivot_b, a_c, sb, sbb, sab, vmax, bmax);
    else if (mode == 0)
      roll_segment<0, ROUND32, P>(small, tap, row_elems, be, bnx, bny, he1, hx1, hy1, inv0, xoff, yoff, pivot_b,
                                  a_c, sb, sbb, sab, vmax, bmax);
    else
      roll_segment<1, ROUND32, P>(small, tap, row_elems, be, bnx, bny, he1, hx1, hy1, inv0, xoff, yoff, pivot_b,
                                  a_c, sb, sbb, sab, vmax, bmax);
    // all fractional parts in [0, 1), every sample finite (|bc| < 2^129 keeps bc^2 finite, so Sbb is finite
    // exactly when all samples are)
    fast = (vmax < 0x3FF00000u) && (bmax < 0x7F800000u) &&
           (((unsigned)__double2hiint(sbb) & 0x7FF00000u) != 0x7FF00000u);
  }
  if (!fast && a_ok && mode != 2) {
    // A segment that lies outside the small image as a whole has no sample at all. Along the segment each
    // coordinate is numerator / (1 - e) with both linear in p and 1 - e > 0, hence monotonic: it stays between its
    // values at the first and the last pixel. (1e-6 pixel covers the rounding of the reciprocal series; NaN
    // coordinates fail every compare and go pixel by pixel.)
    const double eL = fma(he1, (double)(P - 1), be);
    const double invL = (mode == 0) ? recip_1me_tiny(eL) : recip_1me_small(eL);
    const double sxL = fma(fma(hx1, (double)(P - 1), bnx), invL, x0h);
    const double syL = fma(fma(hy1, (double)(P - 1), bny), invL, y0h);
    const double lo = 0.5 - 1e-6, hix = (double)snx - 0.5 + 1e-6, hiy = (double)sny - 0.5 + 1e-6;
    if ((fmax(sx0, sxL) < lo) || (fmin(sx0, sxL) > hix) || (fmax(sy0, syL) < lo) || (fmin(sy0, syL) > hiy)) {
      sb = sbb = sab = 0.0;
      miss = a_ok;
      return;
    }
  }
  // image borders, irregular columns (rotated lags), missing pixels, division-mode lags: the segment still has to be
  // evaluated pixel by pixel -- by the warp together (`roll_pixels_warp`) or, when most lanes need it, by each thread
  // for itself (`roll_pixels_serial`)
  slow = !fast && a_ok;
  if (!fast) sb = sbb = sab = 0.0;
}

// One pixel of a segment by the per-pixel rules. (gx, gy0): grid column and first row of the segment; p: row inside it.
template <bool ROUND32>
__device__ __forceinline__ bool roll_one_pixel(const HomLag& C, int mode, const double* __restrict__ small, int snx,
                                               int sny, unsigned row_elems, double di, double dj0, int p, double* b) {
  const double bnx = fma(C.hx1, dj0, fma(C.hx0, di, C.hx2));
  const double bny = fma(C.hy1, dj0, fma(C.hy0, di, C.hy2));
  const double be = fma(C.he1, dj0, fma(C.he0, di, C.he2));
  const double e = fma(C.he1, (double)p, be);
  const double inv = (mode == 0) ? recip_1me_tiny(e) : ((mode == 1) ? recip_1me_small(e) : recip_1me_div(e));
  const double sx = fma(fma(C.hx1, (double)p, bnx), inv, C.x0h);
  const double sy = fma(fma(C.hy1, (double)p, bny), inv, C.y0h);
  return sample_pixel_half<ROUND32>(small, sny, snx, row_elems, sx, sy, b);
}

// The segment pixel by pixel, every thread for itself (all lanes busy: division-mode lags, tiles on the image border).
template <bool ROUND32, int P, typename AT>
__device__ __forceinline__ void roll_pixels_serial(const HomLag& C, int mode, const double* __restrict__ small,
                                                   int snx, int sny, unsigned row_elems, double di, double dj0,
                                                   const AT (&a_c)[P], unsigned a_ok, double pivot_b, double& sb,
                                                   double& sbb, double& sab, unsigned& miss) {
  sb = sbb = sab = 0.0;
  miss = 0;
#pragma unroll 1
  for (int p = 0; p < P; ++p) {
    if (!(a_ok & (1u << p))) continue;
    AT acs = a_c[0];
#pragma unroll
    for (int q = 1; q < P; ++q)
      if (q == p) acs = a_c[q];
    const double ac = (double)acs;
    double b;
    if (roll_one_pixel<ROUND32>(C, mode, small, snx, sny, row_elems, di, dj0, p, &b)) {
      const double bc = b - pivot_b;
      sb += bc;
      sbb = fma(bc, bc, sbb);
      sab = fma(ac, bc, sab);
    } else {
      miss |= 1u << p;
    }
  }
}

// The same for the FEW lanes of a warp whose segment needs it (rotated / rescaled lags: a floor changes inside ~10 - 25 %
// of the segments; tiles on the rim of the image), without making the other lanes wait for a 12- or 16-pixel serial
// loop: two segments at a time, one per half-warp, one pixel per lane; the sums come back to the owner by a butterfly
// (fixed order). A helper lane derives the owner's column and rows from the owner's lane number and re-reads the
// reference pixel (an L1 hit). (Measured against a variant that deals the pixels of all needy segments out densely
// over the 32 lanes through shared-memory slots: that one is slower for the all-FP64 kernel, 37.6 vs 36.4 ms on
// config 1, profiles/r2_k1_tuning.md.)
constexpr int kSlowOwners = 10;     // more needy lanes than this: every thread for itself

template <typename RefT, bool ROUND32, int P, bool MIXED>
__device__ __forceinline__ void roll_pixels_warp(unsigned need, const HomLag& C, int mode, const RefT* __restrict__ ref,
                                                 const double* __restrict__ small, int snx, int sny, int gnx, int gny,
                                                 unsigned row_elems, int gx_base, int gy_base, int lane,
                                                 double pivot_a, double pivot_b, double& sb, double& sbb, double& sab,
                                                 unsigned& miss) {
  static_assert(P <= 16, "one segment per half-warp");
  const int half = lane >> 4, p = lane & 15;
  while (need) {   // warp-uniform
    const int o0 = __ffs(need) - 1;
    need &= need - 1;
    const int o1 = need ? __ffs(need) - 1 : -1;
    if (o1 >= 0) need &= need - 1;
    const int owner = half ? o1 : o0;
    double psb = 0.0, psbb = 0.0, psab = 0.0;
    bool pmiss = false;
    if (owner >= 0 && p < P) {
      const int gx = gx_base + owner, gy = gy_base + p;   // a warp covers 32 consecutive columns of one row group
      if (gx < gnx && gy < gny) {
        const double a = (double)ref[(int64_t)gy * gnx + gx];
        if (isfinite(a)) {
          const double ac = MIXED ? (double)(float)(a - pivot_a) : a - pivot_a;
          double b;
          if (roll_one_pixel<ROUND32>(C, mode, small, snx, sny, row_elems, (double)gx, (double)gy_base, p, &b)) {
            const double bc = b - pivot_b;
            psb = bc;
            psbb = bc * bc;
            psab = ac * bc;
          } else {
            pmiss = true;
          }
        }
      }
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      psb += __shfl_xor_sync(0xffffffffu, psb, o);
      psbb += __shfl_xor_sync(0xffffffffu, psbb, o);
      psab += __shfl_xor_sync(0xffffffffu, psab, o);
    }
    const unsigned bal = __ballot_sync(0xffffffffu, pmiss);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const double r0 = __shfl_sync(0xffffffffu, psb, 16 * k), r1 = __shfl_sync(0xffffffffu, psbb, 16 * k),
                   r2 = __shfl_sync(0xffffffffu, psab, 16 * k);
      if (lane == (k ? o1 : o0)) {
        sb = r0;
        sbb = r1;
        sab = r2;
        miss = (bal >> (16 * k)) & 0xFFFFu;
      }
    }
  }
}

constexpr int kRollChunk = 8;  // lags whose per-lane sums wait in a warp's shared-memory slice for one fold

// ---------------------------------------------------------------------------------------------------------
// The rolling kernel proper. Warps are independent: no block barrier inside the lag walk. Every warp keeps its own
// shared-memory slice (its lanes' Sb, Sbb, Sab for kRollChunk lags, and its own copy of the chunk's 3x3 matrices),
// folds it with __syncwarp only, and writes one 24-byte record per (warp, lag) straight to the workspace; the
// finalize kernel sums 8 records per tile instead of one. Corrections for missing samples (rare) go to a second
// array that is only read where a bit of the per-(tile, lag) mask is set, so it needs no initialisation; the
// mask itself (4 B per tile and lag) is cleared by the launcher.
// ---------------------------------------------------------------------------------------------------------
constexpr int kAccPad = 33;   // lane stride of the per-warp accumulators (bank-conflict-free transposed reads)

struct RollWShared {
  double acc[kWarps][kRollChunk][3][kAccPad];
  HomLag lag[kWarps][kRollChunk];
};

template <typename RefT, bool ROUND32, int P, int MINB, bool MIXED, bool ADAPT>
__global__ void __launch_bounds__(kThreads, MINB)
lag_corr_roll_kernel(const RefT* __restrict__ ref, const double* __restrict__ small,
                      const float* __restrict__ small32, int snx, int sny, int gnx,
                      int gny, const HomLag* __restrict__ lags, int n_lags, int lags_per_block,
                      const double* __restrict__ pivots, double* __restrict__ wrec, double* __restrict__ wcorr,
                      double* __restrict__ wconst, unsigned* __restrict__ wmask) {
  constexpr int TILE_H = kRowsPerPass * P;
  extern __shared__ __align__(16) unsigned char roll_smem[];
  RollWShared& S = *reinterpret_cast<RollWShared*>(roll_smem);

  const int tiles_x = (gnx + kTileW - 1) / kTileW;
  const int tiles_y = (gny + TILE_H - 1) / TILE_H;
  // Tiles on the rim of the grid run longest (segments that straddle the image border go pixel by pixel), so they are
  // launched first: block indices 0 .. n_rim - 1 walk the rim, the rest the interior. Records are indexed by the tile,
  // not by the block, so the order changes nothing but the tail of the launch.
  int tile_x, tile_y;
  {
    const int b = blockIdx.x;
    const int n_rim = (tiles_x <= 2 || tiles_y <= 2) ? tiles_x * tiles_y : 2 * tiles_x + 2 * (tiles_y - 2);
    if (b >= n_rim) {
      const int i = b - n_rim;
      tile_x = 1 + i % (tiles_x - 2);
      tile_y = 1 + i / (tiles_x - 2);
    } else if (tiles_x <= 2 || tiles_y <= 2) {
      tile_x = b % tiles_x;
      tile_y = b / tiles_x;
    } else if (b < 2 * tiles_x) {
      tile_x = b % tiles_x;
      tile_y = (b < tiles_x) ? 0 : tiles_y - 1;
    } else {
      const int i = b - 2 * tiles_x;
      tile_x = (i & 1) ? tiles_x - 1 : 0;
      tile_y = 1 + (i >> 1);
    }
  }
  const int tile = tile_y * tiles_x + tile_x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = tid & (kTileW - 1), rg = tid / kTileW;
  const int gx = tile_x * kTileW + tx;
  const int gy0 = tile_y * TILE_H + rg * P;
  // MIXED: float32-representable pivots, so that the float32 segment sums and the FP64 fallback subtract the same
  // numbers and a - pivot_a is (nearly always) exact in float32. r does not depend on the pivots.
  const double pivot_a = MIXED ? (double)(float)pivots[0] : pivots[0];
  const double pivot_b = MIXED ? (double)(float)pivots[1] : pivots[1];
  const unsigned row_elems = (unsigned)snx;
  const double di = (double)gx, dj0 = (double)gy0;
  const size_t wid = (size_t)tile * kWarps + warp;   // this warp's record row

  using AT = typename std::conditional<MIXED, float, double>::type;
  AT a_c[P];
  unsigned a_ok = 0;
  double sa_all = 0.0, saa_all = 0.0;
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const int gy = gy0 + p;
    a_c[p] = (AT)0;
    if (gx < gnx && gy < gny) {
      const double a = (double)ref[(int64_t)gy * gnx + gx];
      if (isfinite(a)) {
        a_c[p] = (AT)(a - pivot_a);
        a_ok |= 1u << p;
        // MIXED: every sum sees the float32 value of a - pivot_a, i.e. one consistent reference image
        const double ac = (double)a_c[p];
        sa_all += ac;
        saa_all = fma(ac, ac, saa_all);
      }
    }
  }
  const bool all_ref = a_ok == ((P >= 32) ? 0xFFFFFFFFu : ((1u << (P & 31)) - 1u));
  if (blockIdx.y == 0) {
    // lag-independent reference moments of this warp's pixels (n, Sa, Saa): one record per warp, written once
    double wsa = sa_all, wsaa = saa_all;
    int wn = __popc(a_ok);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      wsa += __shfl_xor_sync(0xffffffffu, wsa, o);
      wsaa += __shfl_xor_sync(0xffffffffu, wsaa, o);
      wn += __shfl_xor_sync(0xffffffffu, wn, o);
    }
    if (lane == 0) {
      wconst[wid * 3 + 0] = (double)wn;
      wconst[wid * 3 + 1] = wsa;
      wconst[wid * 3 + 2] = wsaa;
    }
  }

  const int lag_begin = blockIdx.y * lags_per_block;
  const int lag_end = min(n_lags, lag_begin + lags_per_block);
  for (int l0 = lag_begin; l0 < lag_end; l0 += kRollChunk) {
    const int cnt = min(kRollChunk, lag_end - l0);
    __syncwarp();   // previous chunk folded
    {
      const double* src = reinterpret_cast<const double*>(lags + l0);
      double* dst = reinterpret_cast<double*>(&S.lag[warp][0]);
      const int nd = cnt * (int)(sizeof(HomLag) / sizeof(double));
      for (int i = lane; i < nd; i += 32) dst[i] = __ldg(src + i);
    }
    __syncwarp();
    for (int l = 0; l < cnt; ++l) {
      double sb, sbb, sab;
      unsigned miss;
      bool slow;
      const HomLag& C = S.lag[warp][l];
      roll_lag<ROUND32, P, MIXED, ADAPT, AT>(C, small, small32, snx, sny, row_elems, di, dj0, a_c, a_ok, all_ref, pivot_b, sb,
                                      sbb, sab, miss, slow);
      const unsigned need = __ballot_sync(0xffffffffu, slow);
      if (need) {
        const int mode = (fabs(C.emax) <= kTinyE) ? 0 : ((fabs(C.emax) <= kSmallE) ? 1 : 2);
        if (__popc(need) > kSlowOwners) {      // most lanes: every thread walks its own segment, nobody waits
          if (slow)
            roll_pixels_serial<ROUND32, P, AT>(C, mode, small, snx, sny, row_elems, di, dj0, a_c, a_ok, pivot_b, sb, sbb,
                                               sab, miss);
        } else {
          roll_pixels_warp<RefT, ROUND32, P, MIXED>(need, C, mode, ref, small, snx, sny, gnx, gny, row_elems, gx - lane,
                                                    gy0, lane, pivot_a, pivot_b, sb, sbb, sab, miss);
        }
      }
      S.acc[warp][l][0][lane] = sb;
      S.acc[warp][l][1][lane] = sbb;
      S.acc[warp][l][2][lane] = sab;
      if (__any_sync(0xffffffffu, miss != 0)) {
        double m[4] = {(double)__popc(miss), 0.0, 0.0, 0.0};
#pragma unroll
        for (int p = 0; p < P; ++p)
          if (miss & (1u << p)) {
            const double ac = (double)a_c[p];
            m[1] += ac;
            m[2] = fma(ac, ac, m[2]);
          }
        const double tot = warp_transpose_reduce4(m, lane);  // lanes 0, 8, 16: n, Sa, Saa of the missing pixels
        if ((lane & 7) == 0 && lane < 24) wcorr[(wid * n_lags + (l0 + l)) * 3 + (lane >> 3)] = tot;
        if (lane == 0) atomicOr(wmask + ((size_t)tile * n_lags + (l0 + l)), 1u << warp);
      }
    }
    __syncwarp();
    if (lane < cnt * 3) {
      const int l = lane / 3, v = lane - 3 * l;
      const double* src = &S.acc[warp][l][v][0];
      double t = src[0];
#pragma unroll
      for (int k = 1; k < 32; ++k) t += src[k];
      wrec[(wid * n_lags + (l0 + l)) * 3 + v] = t;
    }
  }
}

// Finalize: one block per chunk of kRollChunk consecutive lags. A record row holds the chunk's (Sb, Sbb, Sab) as 24
// contiguous doubles, so 24 adjacent threads read one row's 192 bytes together (the first version read 24 bytes per
// 86 KB stride: 0.41 ms per 3600-lag search, now bounded by the records' HBM read). Ten row groups walk the rows in
// a fixed order, are folded in a fixed order, and the moments become Pearson r. The lag-independent reference moments
// (n, Sa, Saa per row) and their rare per-lag corrections ride in a second accumulator of the same threads.
// `guard` (mixed arithmetic only) points at the image statistics: per lag, the error model of the FP32 spline is
// compared with the sampled image's own variance and flagged[lag] = 1 marks the lags that cannot be trusted to 1e-7
// (the caller re-evaluates those with the all-FP64 kernel).
constexpr int kFinGroups = 10, kFinElems = kRollChunk * 3;
constexpr int kRollRows = 16;   // rows per thread of the launched rolling kernel: tiles of 64 x 64 grid pixels

__device__ __forceinline__ bool mixed_guard_trips(const double* __restrict__ guard, double n, double vb) {
  // guard = [4][2] statistics block: row 2 = max |v|, row 3 = RMS of (v - pivot); column 1 = the small image.
  //   s_t   RMS error of the centred FP32 spline sample. Measured (numpy emulation of this arithmetic on smooth and
  //         noisy scenes, profiles/r2_mixed_error_model.md): 0.8 - 0.9 x 2^-24 x rms; taken as 2 x 2^-24 x rms
  //   ulpS  float32 spacing of the uncentred sample (what the reference's float32 store rounds to) at max |v|
  //   a sample within s_t of a rounding boundary of S (probability ~ s_t / ulpS) lands one ulpS away from the
  //   reference's: s_eff^2 = s_t^2 + s_t * ulpS (measured 1.06e-5 sigma against 1.08e-5 predicted for mean 3e4, sigma 1).
  //   Independent errors of that size move r by ~ s_eff / (sigma_b sqrt(n)) (random part, taken at 4 sigma) +
  //   (s_eff / sigma_b)^2 (the variance they add to Sbb). Bar: 1e-7, ten times under the contract.
  const double rms = guard[3 * 2 + 1], mx = guard[2 * 2 + 1];
  const double st = 2.0 * 5.9604644775390625e-08 * rms;
  int ex = 0;
  frexp(mx, &ex);                                   // mx = m * 2^ex, 0.5 <= m < 1: ulp32(mx) = 2^(ex - 24)
  const double ulps = (mx > 0.0) ? ldexp(1.0, ex - 24) : 0.0;
  const double q = (st * st + st * ulps) * n / vb;   // (s_eff / sigma_b)^2 with vb = n sigma_b^2
  return !(4.0 * sqrt(q / n) + q <= 1e-7);
}

__global__ void __launch_bounds__(256)
lag_corr_finalize_w_kernel(const double* __restrict__ wrec, const double* __restrict__ wcorr,
                           const double* __restrict__ wconst, const unsigned* __restrict__ wmask, int n_rows,
                           int n_lags, double* __restrict__ corr, int64_t* __restrict__ nvalid,
                           const double* __restrict__ guard, int* __restrict__ flagged) {
  __shared__ double s_var[kFinGroups][kFinElems], s_cst[kFinGroups][kFinElems];
  __shared__ double s_tot[2][kFinElems];
  const int l0 = blockIdx.x * kRollChunk;
  const int t = threadIdx.x, e = t % kFinElems, g = t / kFinElems;
  const int lag = l0 + e / 3, v = e % 3;
  if (g < kFinGroups) {
    double av = 0.0, ac = 0.0;
    if (lag < n_lags) {
      for (int r = g; r < n_rows; r += kFinGroups) {
        const size_t o = ((size_t)r * n_lags + lag) * 3 + v;
        av += wrec[o];
        ac += wconst[(size_t)r * 3 + v];
        if ((wmask[(size_t)(r / kWarps) * n_lags + lag] >> (r % kWarps)) & 1u) ac -= wcorr[o];
      }
    }
    s_var[g][e] = av;
    s_cst[g][e] = ac;
  }
  __syncthreads();
  if (t < kFinElems) {
    double av = s_var[0][t], ac = s_cst[0][t];
#pragma unroll
    for (int k = 1; k < kFinGroups; ++k) {
      av += s_var[k][t];
      ac += s_cst[k][t];
    }
    s_tot[0][t] = av;
    s_tot[1][t] = ac;
  }
  __syncthreads();
  if (t < kRollChunk && l0 + t < n_lags) {
    const double sb = s_tot[0][3 * t], sbb = s_tot[0][3 * t + 1], sab = s_tot[0][3 * t + 2];
    const double n = s_tot[1][3 * t], sa = s_tot[1][3 * t + 1], saa = s_tot[1][3 * t + 2];
    double r = CUDART_NAN;
    if (n > 0.0) {
      const double cov = sab - sa * sb / n;
      const double va = saa - sa * sa / n;
      const double vb = sbb - sb * sb / n;
      r = cov / sqrt(va * vb);
      if (guard != nullptr) flagged[l0 + t] = mixed_guard_trips(guard, n, vb) ? 1 : 0;
    } else if (guard != nullptr) {
      flagged[l0 + t] = 0;
    }
    corr[l0 + t] = r;
    if (nvalid) nvalid[l0 + t] = (int64_t)n;
  }
}

// Per-block form of lag_corr_finalize_w_kernel (CoregRegions): blockIdx.y = block of the grid. The block's record rows
// are taken in ascending order (tile rows, tiles, warps) and its k-th row goes to row group k % kFinGroups, as the
// whole-grid fold deals row k: one block covering the grid folds the same sums in the same order.
__global__ void __launch_bounds__(256)
lag_corr_finalize_w_regions_kernel(const double* __restrict__ wrec, const double* __restrict__ wcorr,
                                   const double* __restrict__ wconst, const unsigned* __restrict__ wmask, int n_lags,
                                   int tiles_x, int tiles_y, int bt_h, int bt_w, int nbx, double* __restrict__ corr,
                                   int64_t* __restrict__ nvalid, int64_t ld) {
  __shared__ double s_var[kFinGroups][kFinElems], s_cst[kFinGroups][kFinElems];
  __shared__ double s_tot[2][kFinElems];
  const RegionTiles R = region_tiles(blockIdx.y, nbx, bt_h, bt_w, tiles_x, tiles_y);
  const int n_rows = R.n_tiles * kWarps;
  const int l0 = blockIdx.x * kRollChunk;
  const int t = threadIdx.x, e = t % kFinElems, g = t / kFinElems;
  const int lag = l0 + e / 3, v = e % 3;
  if (g < kFinGroups) {
    double av = 0.0, ac = 0.0;
    if (lag < n_lags) {
      for (int k = g; k < n_rows; k += kFinGroups) {
        const int tl = k / kWarps;
        const int tile = (R.ty0 + tl / R.ntx) * tiles_x + R.tx0 + tl % R.ntx;
        const size_t r = (size_t)tile * kWarps + k % kWarps;
        const size_t o = (r * n_lags + lag) * 3 + v;
        av += wrec[o];
        ac += wconst[r * 3 + v];
        if ((wmask[(size_t)tile * n_lags + lag] >> (k % kWarps)) & 1u) ac -= wcorr[o];
      }
    }
    s_var[g][e] = av;
    s_cst[g][e] = ac;
  }
  __syncthreads();
  if (t < kFinElems) {
    double av = s_var[0][t], ac = s_cst[0][t];
#pragma unroll
    for (int k = 1; k < kFinGroups; ++k) {
      av += s_var[k][t];
      ac += s_cst[k][t];
    }
    s_tot[0][t] = av;
    s_tot[1][t] = ac;
  }
  __syncthreads();
  if (t < kRollChunk && l0 + t < n_lags) {
    const double n = s_tot[1][3 * t];
    const size_t o = (size_t)blockIdx.y * ld + l0 + t;
    corr[o] = pearson_from_moments(n, s_tot[1][3 * t + 1], s_tot[0][3 * t], s_tot[1][3 * t + 2], s_tot[0][3 * t + 1],
                                   s_tot[0][3 * t + 2]);
    nvalid[o] = (int64_t)n;
  }
}

// the per-block fold of the records a launch_lag_rollw call left in `work` (its tiles: kRollRows rows per thread)
int launch_finalize_w_regions(int gnx, int gny, int64_t n_lags, void* work, const CoregRegions* rg, cudaStream_t s) {
  constexpr int TILE_H = kRowsPerPass * kRollRows;
  const RollWLayout L = rollw_layout(gnx, gny, n_lags);
  char* base = static_cast<char*>(work);
  const int tiles_x = (gnx + kTileW - 1) / kTileW, tiles_y = (gny + TILE_H - 1) / TILE_H;
  const int nbx = (gnx + rg->block_w - 1) / rg->block_w, nby = (gny + rg->block_h - 1) / rg->block_h;
  const dim3 grid((unsigned)((n_lags + kRollChunk - 1) / kRollChunk), (unsigned)(nbx * nby));
  lag_corr_finalize_w_regions_kernel<<<grid, 256, 0, s>>>(
      reinterpret_cast<const double*>(base + L.rec), reinterpret_cast<const double*>(base + L.corr),
      reinterpret_cast<const double*>(base + L.cst), reinterpret_cast<const unsigned*>(base + L.mask), (int)n_lags,
      tiles_x, tiles_y, rg->block_h / TILE_H, rg->block_w / kTileW, nbx, rg->corr_dev, rg->nvalid_dev, rg->ld);
  CK_LAUNCH("lag_corr_finalize_w_regions_kernel");
  return COREG_OK;
}

// rolling kernel + its finalize: 16 rows per thread, 2 CTAs / SM. `adapt` selects the flavour with the adaptive segment
// for rotated / rescaled lags; without it (COREG_FLAG_PURE_SHIFT) the kernel serves lag grids of pure CRVAL shifts,
// where no segment drifts. The adaptive code is never executed there, but its presence in the kernel costs the regular
// path 1 % (all-FP64) to 3 % (mixed) through register allocation and code placement -- so the caller that knows its
// WHOLE lag grid holds shifts only asks for this flavour (the choice must not depend on how the grid is sharded: both
// flavours are correct for any lag, but they round an irregular segment differently). small32 != nullptr selects the
// mixed-arithmetic kernel (FP64 coordinates, FP32 spline on the float32 copy of the small image).
// (Measured and dropped: 12 and 14 rows per thread -- 40.1 and 39.4 against 37.8 ms on config 1,
// profiles/r2_k1_tuning.md; with the adaptive segment 16 rows win for rotated / rescaled lags too, 14.0 vs 14.4 us per
// lag on the 5-D grid against 12 rows; 3 CTAs per SM at 80 registers -- spills; 24 and 32 rows per thread -- spills and
// partial tiles; a precomputed row-coefficient plane: tools/mixed_lab.py, profiles/r1_mixed_kernel.md.)
template <typename RefT, bool ROUND32>
int launch_lag_rollw(bool adapt, int gnx, int gny, int64_t n_lags, int sms, cudaStream_t s, const RefT* ref,
                     const double* small, const float* small32, int snx, int sny,
                     const HomLag* ft, const double* pivots, void* work, double* corr, int64_t* nvalid, bool prof,
                     int* flagged) {
  constexpr int P = kRollRows, MINB = 2;
  const bool mixed = small32 != nullptr;
  const RollWLayout L = rollw_layout(gnx, gny, n_lags);
  char* base = static_cast<char*>(work);
  double* wrec = reinterpret_cast<double*>(base + L.rec);
  double* wcorr = reinterpret_cast<double*>(base + L.corr);
  double* wconst = reinterpret_cast<double*>(base + L.cst);
  unsigned* wmask = reinterpret_cast<unsigned*>(base + L.mask);
  dim3 grid;
  int lpb, tiles;
  if (!lag_grid(kRowsPerPass * P, MINB, gnx, gny, n_lags, sms, &grid, &lpb, &tiles, kRollChunk, true))
    return fail(COREG_EINVAL, "lag grid too large for one launch");
  CK(cudaMemsetAsync(wmask, 0, (size_t)tiles * (size_t)n_lags * sizeof(unsigned), s));
  if (prof) CK(cudaEventRecord(g_prof[g_prof_n].a, s));
  auto kern = mixed ? (adapt ? lag_corr_roll_kernel<RefT, ROUND32, P, MINB, true, true>
                             : lag_corr_roll_kernel<RefT, ROUND32, P, MINB, true, false>)
                    : (adapt ? lag_corr_roll_kernel<RefT, ROUND32, P, MINB, false, true>
                             : lag_corr_roll_kernel<RefT, ROUND32, P, MINB, false, false>);
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RollWShared));
  kern<<<grid, kThreads, sizeof(RollWShared), s>>>(ref, small, small32, snx, sny, gnx, gny, ft, (int)n_lags, lpb, pivots,
                                                   wrec, wcorr, wconst, wmask);
  CK_LAUNCH("lag_corr_roll_kernel");
  if (prof) {
    CK(cudaEventRecord(g_prof[g_prof_n].b, s));
    ++g_prof_n;
  }
  // record rows actually written: 8 warps per 16-row tile (<= L.rows)
  // mixed arithmetic: `pivots` is the head of the [4][2] statistics block (coreg_image_stats / coreg_center_f32)
  lag_corr_finalize_w_kernel<<<(unsigned)((n_lags + kRollChunk - 1) / kRollChunk), 256, 0, s>>>(
      wrec, wcorr, wconst, wmask, tiles * kWarps, (int)n_lags, corr, nvalid, (mixed && flagged) ? pivots : nullptr, flagged);
  CK_LAUNCH("lag_corr_finalize_w_kernel");
  return COREG_OK;
}

int hpc_lag_corr_wcs_impl(const float* ref, const double* small, const float* small32, int snx, int sny, int gnx,
                          int gny,
                          const CoregTanWcs* grid_wcs, const CoregTanWcs* lag_wcs, int64_t n_lags,
                          const double* pivots, void* work, double* corr, int64_t* nvalid, int flags, cudaStream_t s,
                          int* flagged = nullptr) {
  HomGrid g;
  int rc = make_hom_grid(grid_wcs, gnx, gny, &g);
  if (rc) return rc;
  int sms = coreg_device_sm_count();
  if (sms <= 0) sms = 148;
  HomLag* ft = reinterpret_cast<HomLag*>(static_cast<char*>(work) + partials_bytes(gnx, gny, n_lags));
  tan_homography_kernel<<<((int)n_lags + 127) / 128, 128, 0, s>>>(g, lag_wcs, (int)n_lags, ft);
  CK_LAUNCH("tan_homography_kernel");
  const bool prof = g_prof_on && g_prof_n < 4096;
  if (prof) {
    CK(cudaEventCreate(&g_prof[g_prof_n].a));
    CK(cudaEventCreate(&g_prof[g_prof_n].b));
  }
  return launch_lag_rollw<float, true>(!(flags & COREG_FLAG_PURE_SHIFT), gnx, gny, n_lags, sms, s, ref, small, small32,
                                       snx, sny, ft, pivots, work, corr, nvalid, prof, flagged);
}
}  // namespace coreg

using namespace coreg;

extern "C" {

int coreg_hpc_lag_corr_wcs(const float* ref, const double* small, int snx, int sny, int gnx, int gny,
                           const CoregTanWcs* grid_wcs, const CoregTanWcs* lag_wcs, int64_t n_lags, int order,
                           const double* pivots, void* work, size_t work_bytes, double* corr, int64_t* nvalid,
                           int flags, void* stream) {
  if (!ref || !small || !grid_wcs || !lag_wcs || !pivots || !work || !corr)
    return fail(COREG_EINVAL, "coreg_hpc_lag_corr_wcs: null pointer");
  if (int rc = check_lag_flags(flags, "coreg_hpc_lag_corr_wcs")) return rc;
  if (n_lags <= 0) return COREG_OK;
  if (order != 2 || (flags & COREG_FLAG_STRICT))
    return fail(COREG_EINVAL, "coreg_hpc_lag_corr_wcs: only order 2 with FMA arithmetic; use coreg_hpc_lag_corr");
  if (gnx <= 0 || gny <= 0 || snx < 3 || sny < 3) return fail(COREG_EINVAL, "image too small for the fast kernel");
  if ((int64_t)snx * sny >= ((int64_t)1 << 31)) return fail(COREG_EINVAL, "small image too large (>= 2^31 pixels)");
  if (n_lags > (int64_t)1 << 30) return fail(COREG_EINVAL, "too many lags in one call (max 2^30)");
  if (work_bytes < coreg_lag_corr_workspace_bytes(gnx, gny, n_lags)) return fail(COREG_ENOMEM, "workspace too small");
  return hpc_lag_corr_wcs_impl(ref, small, nullptr, snx, sny, gnx, gny, grid_wcs, lag_wcs, n_lags, pivots, work, corr,
                               nvalid, flags, (cudaStream_t)stream);
}

int coreg_hpc_lag_corr_wcs_regions(const float* ref, const double* small, int snx, int sny, int gnx, int gny,
                                   const CoregTanWcs* grid_wcs, const CoregTanWcs* lag_wcs, int64_t n_lags, int order,
                                   const double* pivots, void* work, size_t work_bytes, double* corr, int64_t* nvalid,
                                   const CoregRegions* regions, int flags, void* stream) {
  if (int rc = check_regions(regions, gnx, gny, n_lags, flags, "coreg_hpc_lag_corr_wcs_regions")) return rc;
  int rc = coreg_hpc_lag_corr_wcs(ref, small, snx, sny, gnx, gny, grid_wcs, lag_wcs, n_lags, order, pivots, work,
                                  work_bytes, corr, nvalid, flags, stream);
  if (rc || n_lags <= 0) return rc;
  return launch_finalize_w_regions(gnx, gny, n_lags, work, regions, (cudaStream_t)stream);
}

int coreg_hpc_lag_corr_wcs_mixed(const float* ref, const double* small, const float* small32c, int snx, int sny,
                                 int gnx, int gny, const CoregTanWcs* grid_wcs, const CoregTanWcs* lag_wcs,
                                 int64_t n_lags, int order, const double* stats, void* work, size_t work_bytes,
                                 double* corr, int64_t* nvalid, int* flagged, int flags, void* stream) {
  if (!ref || !small || !small32c || !grid_wcs || !lag_wcs || !stats || !work || !corr || !flagged)
    return fail(COREG_EINVAL, "coreg_hpc_lag_corr_wcs_mixed: null pointer");
  if (int rc = check_lag_flags(flags, "coreg_hpc_lag_corr_wcs_mixed")) return rc;
  if (n_lags <= 0) return COREG_OK;
  if (order != 2 || (flags & COREG_FLAG_STRICT))
    return fail(COREG_EINVAL, "coreg_hpc_lag_corr_wcs_mixed: only order 2 with FMA arithmetic; use coreg_hpc_lag_corr");
  if (gnx <= 0 || gny <= 0 || snx < 3 || sny < 3) return fail(COREG_EINVAL, "image too small for the fast kernel");
  if ((int64_t)snx * sny >= ((int64_t)1 << 31)) return fail(COREG_EINVAL, "small image too large (>= 2^31 pixels)");
  if (n_lags > (int64_t)1 << 30) return fail(COREG_EINVAL, "too many lags in one call (max 2^30)");
  if (work_bytes < coreg_lag_corr_workspace_bytes(gnx, gny, n_lags)) return fail(COREG_ENOMEM, "workspace too small");
  return hpc_lag_corr_wcs_impl(ref, small, small32c, snx, sny, gnx, gny, grid_wcs, lag_wcs, n_lags, stats, work, corr,
                               nvalid, flags, (cudaStream_t)stream, flagged);
}

int coreg_tan_homography_emax(const CoregTanWcs* grid_wcs, int gnx, int gny, const CoregTanWcs* lag_wcs, int64_t n_lags,
                              void* scratch, double* emax, void* stream) {
  if (!grid_wcs || !lag_wcs || !scratch || !emax) return fail(COREG_EINVAL, "coreg_tan_homography_emax: null pointer");
  if (n_lags <= 0) return COREG_OK;
  HomGrid g;
  int rc = make_hom_grid(grid_wcs, gnx, gny, &g);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  HomLag* ft = static_cast<HomLag*>(scratch);
  tan_homography_kernel<<<((int)n_lags + 127) / 128, 128, 0, s>>>(g, lag_wcs, (int)n_lags, ft);
  CK_LAUNCH("tan_homography_kernel");
  CK(cudaMemcpy2DAsync(emax, sizeof(double), &ft[0].emax, sizeof(HomLag), sizeof(double), (size_t)n_lags,
                       cudaMemcpyDeviceToDevice, s));
  abs_inplace_kernel<<<((int)n_lags + 255) / 256, 256, 0, s>>>(emax, (int)n_lags);   // the sign bit is a flag
  CK_LAUNCH("abs_inplace_kernel");
  return COREG_OK;
}

}  // extern "C"
