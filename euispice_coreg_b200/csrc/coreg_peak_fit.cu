// coreg_peak_fit.cu -- batched bounded 2-D Gaussian peak fits: the sub-lag fit of `AlignmentResults._compute_shift`
// (scipy `curve_fit` of `twoD_Gaussian` on the <= 26 points around a cube's maximum) for many cubes at once, e.g. every
// block of a per-block search or every block of every frame of a sequence.
//
// One warp per problem, one lane per point. Each iteration every lane evaluates the model, its residual and its
// analytic Jacobian row at the trial parameters; the cost, J^T r and the 21 distinct entries of J^T J are summed with
// xor butterflies, so every lane holds the same bits (a + b == b + a) and solves the same 6x6 system: no divergence,
// no shared memory, and results that do not depend on the launch.
//
// Solver: Levenberg-Marquardt with Marquardt's diagonal scaling and Nielsen's damping update, FP64 throughout. Bounds
// are constraints, handled by an active set: a parameter on a bound whose gradient points outward is held there; a
// free parameter whose step would leave the box is put on that bound and held, and the step of the remaining free
// parameters is solved again (at most six passes). The sigmas are the exception: their lower bound is 0, where the
// model is undefined, so a step that reaches it is rejected like a step that raises the cost, and sigma stays > 0.
// Convergence: an accepted step that changes every parameter by <= 1e-10 relative, or the cost by <= 1e-15 relative,
// or no descent step left at damping 1e16. A problem still running after kFitMaxIter iterations is "not converged".
#include "coreg_common.cuh"

namespace coreg {

constexpr int kFitPoints = COREG_FIT_MAX_POINTS;
constexpr int kFitMaxIter = 200;      // 16 384 seeded random peaks: at most 140 iterations, mean 23
constexpr int kFitWarps = 8;          // problems per 256-thread block

__host__ __device__ constexpr int tri(int i, int j) { return i * (i + 1) / 2 + j; }   // packed lower triangle, i >= j

__device__ __forceinline__ double fit_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// cost, J^T r [6] and J^T J [21] of parameters p over this lane's point (lanes without a point add zeros)
__device__ __forceinline__ void fit_normal_equations(const double (&p)[6], bool live, double x, double y, double z,
                                                     double& cost, double (&g)[6], double (&h)[21]) {
  double r = 0.0, j[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  if (live) {
    const double dx = x - p[1], dy = y - p[2];
    const double sx2 = p[3] * p[3], sy2 = p[4] * p[4];
    const double e = exp(-((dx * dx) / (2.0 * sx2) + (dy * dy) / (2.0 * sy2)));
    const double ae = p[0] * e;
    r = p[5] + ae - z;
    j[0] = e;
    j[1] = ae * dx / sx2;
    j[2] = ae * dy / sy2;
    j[3] = ae * dx * dx / (sx2 * p[3]);
    j[4] = ae * dy * dy / (sy2 * p[4]);
    j[5] = 1.0;
  }
  cost = fit_warp_sum(r * r);
#pragma unroll
  for (int a = 0; a < 6; ++a) g[a] = fit_warp_sum(j[a] * r);
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int b = 0; b <= a; ++b) h[tri(a, b)] = fit_warp_sum(j[a] * j[b]);
}

// Solves m d = rhs for a symmetric packed 6x6 m by Cholesky; false when m is not positive definite
__device__ __forceinline__ bool fit_cholesky_solve(double (&m)[21], double (&d)[6]) {
  bool pd = true;
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    double s = m[tri(c, c)];
#pragma unroll
    for (int k = 0; k < c; ++k) s -= m[tri(c, k)] * m[tri(c, k)];
    pd = pd && s > 0.0;
    const double l = sqrt(pd ? s : 1.0);
    m[tri(c, c)] = l;
    d[c] /= l;   // forward substitution, column by column
#pragma unroll
    for (int i = c + 1; i < 6; ++i) {
      double t = m[tri(i, c)];
#pragma unroll
      for (int k = 0; k < c; ++k) t -= m[tri(i, k)] * m[tri(c, k)];
      m[tri(i, c)] = t / l;
      d[i] -= m[tri(i, c)] * d[c];
    }
  }
#pragma unroll
  for (int i = 5; i >= 0; --i) {
#pragma unroll
    for (int k = i + 1; k < 6; ++k) d[i] -= m[tri(k, i)] * d[k];
    d[i] /= m[tri(i, i)];
  }
  return pd;
}

__global__ void __launch_bounds__(32 * kFitWarps) gauss2d_fit_kernel(
    const double* __restrict__ points, const int* __restrict__ n_points, const double* __restrict__ p0,
    const double* __restrict__ bounds, int64_t n_problems, double* __restrict__ popt, double* __restrict__ cost_out,
    int* __restrict__ iterations, int* __restrict__ status) {
  const int64_t q = (int64_t)blockIdx.x * kFitWarps + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (q >= n_problems) return;     // whole warps leave together
  const int np = n_points[q];
  const bool live = lane < kFitPoints && lane < np;
  double x = 0.0, y = 0.0, z = 0.0;
  if (live) {
    const double* pt = points + (q * kFitPoints + lane) * 3;
    x = pt[0];
    y = pt[1];
    z = pt[2];
  }
  double p[6], lo[6], hi[6];
#pragma unroll
  for (int a = 0; a < 6; ++a) {
    p[a] = p0[q * 6 + a];
    lo[a] = bounds[q * 12 + a];
    hi[a] = bounds[q * 12 + 6 + a];
  }
  double cost, g[6], h[21];
  fit_normal_equations(p, live, x, y, z, cost, g, h);
  int st = COREG_FIT_NOT_CONVERGED, it = 0;
  double lam = 1e-3, nu = 2.0;
  if (np >= 1 && np <= kFitPoints && isfinite(cost)) {
    for (it = 1; it <= kFitMaxIter; ++it) {
      // active set: on a bound, pushed outward by the gradient (descent direction is -g)
      unsigned held = 0;
#pragma unroll
      for (int a = 0; a < 6; ++a)
        if ((p[a] <= lo[a] && g[a] > 0.0) || (p[a] >= hi[a] && g[a] < 0.0)) held |= 1u << a;
      double dfix[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, d[6];
      bool solved = false;
      for (int pass = 0; pass < 6; ++pass) {
        // free rows: (H + lam diag H)_FF d_F = -g_F - (H + lam diag H)_FB d_B; held rows: identity, d = dfix
        double m[21];
#pragma unroll
        for (int a = 0; a < 6; ++a) {
          const bool fa = !(held >> a & 1u);
          double rhs = -g[a];
#pragma unroll
          for (int b = 0; b < 6; ++b)
            if (b != a && (held >> b & 1u)) rhs -= h[a > b ? tri(a, b) : tri(b, a)] * dfix[b];
          d[a] = fa ? rhs : dfix[a];
#pragma unroll
          for (int b = 0; b < a; ++b) m[tri(a, b)] = (fa && !(held >> b & 1u)) ? h[tri(a, b)] : 0.0;
          m[tri(a, a)] = fa ? h[tri(a, a)] + lam * fmax(h[tri(a, a)], 1e-30) : 1.0;
        }
        if (!fit_cholesky_solve(m, d)) break;
        unsigned out = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a) {
          if (held >> a & 1u) continue;
          const double t = p[a] + d[a];
          if (t > hi[a]) {
            out |= 1u << a;
            dfix[a] = hi[a] - p[a];
          } else if (t < lo[a] && a != 3 && a != 4) {
            out |= 1u << a;
            dfix[a] = lo[a] - p[a];
          }
        }
        if (!out) {
          solved = true;
          break;
        }
        held |= out;
      }
      double pt[6];
      bool ok = solved;
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        // a parameter put on a bound in this step lands on it exactly
        pt[a] = (held >> a & 1u) ? (dfix[a] == 0.0 ? p[a] : (p[a] + dfix[a] > p[a] ? hi[a] : lo[a])) : p[a] + d[a];
        if (held >> a & 1u) d[a] = pt[a] - p[a];
      }
      ok = ok && pt[3] > lo[3] && pt[4] > lo[4];
      double ct = 0.0, gt[6], ht[21];
      if (ok) {
        fit_normal_equations(pt, live, x, y, z, ct, gt, ht);
        ok = isfinite(ct) && ct < cost;
      }
      if (ok) {
        // predicted reduction of the linear model: -(2 g.d + d.H.d)
        double gd = 0.0, dhd = 0.0;
#pragma unroll
        for (int a = 0; a < 6; ++a) {
          gd += g[a] * d[a];
          double hd = 0.0;
#pragma unroll
          for (int b = 0; b < 6; ++b) hd += h[a >= b ? tri(a, b) : tri(b, a)] * d[b];
          dhd += d[a] * hd;
        }
        const double pred = -(2.0 * gd + dhd);
        const double rho = pred > 0.0 ? (cost - ct) / pred : 0.0;
        bool small = (cost - ct) <= 1e-15 * ct;
        bool tiny = true;
#pragma unroll
        for (int a = 0; a < 6; ++a) tiny = tiny && fabs(pt[a] - p[a]) <= 1e-10 * (fabs(p[a]) + 1e-10);
#pragma unroll
        for (int a = 0; a < 6; ++a) {
          p[a] = pt[a];
          g[a] = gt[a];
        }
#pragma unroll
        for (int a = 0; a < 21; ++a) h[a] = ht[a];
        cost = ct;
        const double s = 2.0 * rho - 1.0;
        lam *= fmax(1.0 / 3.0, 1.0 - s * s * s);
        nu = 2.0;
        if (small || tiny) {
          st = COREG_FIT_CONVERGED;
          break;
        }
      } else {
        lam *= nu;
        nu *= 2.0;
        if (lam > 1e16) {   // no step at any damping lowers the cost: a minimum to working precision
          st = COREG_FIT_CONVERGED;
          break;
        }
      }
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int a = 0; a < 6; ++a) popt[q * 6 + a] = p[a];
    cost_out[q] = cost;
    iterations[q] = it > kFitMaxIter ? kFitMaxIter : it;
    status[q] = st;
  }
}

}  // namespace coreg

using namespace coreg;

extern "C" {

int coreg_gauss2d_fit(const double* points_dev, const int* n_points_dev, const double* p0_dev, const double* bounds_dev,
                      int64_t n_problems, double* popt_dev, double* cost_dev, int* iterations_dev, int* status_dev,
                      void* stream) {
  if (n_problems < 0) return fail(COREG_EINVAL, "coreg_gauss2d_fit: n_problems < 0");
  if (!points_dev || !n_points_dev || !p0_dev || !bounds_dev || !popt_dev || !cost_dev || !iterations_dev || !status_dev)
    return fail(COREG_EINVAL, "coreg_gauss2d_fit: null pointer");
  if ((n_problems + kFitWarps - 1) / kFitWarps > 0x7fffffff)
    return fail(COREG_EINVAL, "coreg_gauss2d_fit: too many problems for one launch");
  if (n_problems == 0) return COREG_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned blocks = (unsigned)((n_problems + kFitWarps - 1) / kFitWarps);
  gauss2d_fit_kernel<<<blocks, 32 * kFitWarps, 0, s>>>(points_dev, n_points_dev, p0_dev, bounds_dev, n_problems,
                                                       popt_dev, cost_dev, iterations_dev, status_dev);
  CK_LAUNCH("gauss2d_fit_kernel");
  return COREG_OK;
}

}  // extern "C"
