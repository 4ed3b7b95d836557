// mcgpu_cellbound.cuh -- rigorous bounds of the reference-mode acceptance ratio over a cell of x-space (d = 2).
//
// A remote candidate x' is accepted when u < R(x') with, exactly as remote_exact (mh_kernels.cuh) computes it,
//     R(x) = max(FPEPS, max_s Q_s(x)) / (FPEPS + sum_s Q_s(x)),   Q_s(x) = exp(a_s(x)),   a_s(x) = sum_i h_si (x_i - mu_si)^2,
// h = -1/(2 sigma^2) as the kernels stage it.  R depends on x and on the pool only, and the pool is fixed for a
// window, so the table kernel bounds R once per window on every cell of a grid and a candidate whose cell bounds
// settle u skips the pool loop (DESIGN.md section 3.1).
//
// cell_bounds2 gives R_lo <= R(x) <= R_hi for every x of the box |x_i - c_i| <= w_i.  With a reference slot r
// (the largest a_s at the centre) and d_s = a_s - a_r, which is separable with a 1-D quadratic per axis,
//     R = max_s e^{d_s} / (sum_s e^{d_s} + FPEPS e^{-a_r})     whenever Q_r >= FPEPS,
// so the exact ranges [dlo_s, dhi_s] of d_s and [alo, ahi] of a_r over the box give
//     R_lo = max_s e^{dlo_s} / (sum_s e^{dhi_s} + FPEPS e^{-alo}),   R_hi = max_s e^{dhi_s} / (sum_s e^{dlo_s} + FPEPS e^{-ahi}).
// Per axis, with y = x - c in [-w, w]:  d(y) = f0 + b y + k y^2 (k = h_s - h_r); its range is spanned by the two
// ends and, when the vertex -b / 2k may lie inside, the vertex value f0 - b^2 / 4k, taken with |b| raised by its
// rounding error (always a valid bound: the unconstrained extreme).  All of it runs in fp64; the widening 64 u
// sum_i (|h_si| (|y_si| + w)^2 + |h_ri| (|y_ri| + w)^2) per slot covers the roundings of this evaluation and of
// the fp64 a_s, a_r in remote_exact (<= 6 u |a| each), and the relative 1e-9 on R covers mc_exp (1.5 ulp), its
// flush to 0 below e^-708 (< 1e-290 of a sum >= 1e-10), the fp64 sum of <= 4096 terms and the division.
// A cell where Q_r may fall below 1e4 FPEPS, or with NaN / inf anywhere, is undecidable: (0, +inf).
//
// The routine is written for a group of `nl` cooperating lanes (slots s = lane, lane + nl, ...), with `red`
// combining a value over the group: the table kernel runs it on a warp, the host test (tests/cellbound_check.cc)
// on one lane.
#pragma once
#include <math.h>
#include <float.h>

#ifdef __CUDACC__
#define MCGPU_CB_HD __host__ __device__ __forceinline__
#else
#define MCGPU_CB_HD inline
#endif

namespace mcgpu {

// one lane: the group's reduction is the value itself
struct CellRedSelf {
  MCGPU_CB_HD double max(double v) const { return v; }
  MCGPU_CB_HD double sum(double v) const { return v; }
  MCGPU_CB_HD int min(int v) const { return v; }
};

// (mu, h) of slot s, parameter i, from the pool as the engine publishes it: pool[(s * 2 + i) * 2 + {0, 1}] = (mu, sigma^2),
// with h = -0.5 / sigma^2 formed as stage_pool forms it (the same IEEE division: the same double)
MCGPU_CB_HD void cell_slot(const double *pool, int s, int i, double &m, double &h)
{
  m = pool[(s * 2 + i) * 2]; h = -0.5 / pool[(s * 2 + i) * 2 + 1];
}

// the M slots of the pool; the box is centre c, half-widths w
template <class Red>
MCGPU_CB_HD void cell_bounds2(const double *pool, int M, double c0, double c1, double w0, double w1, int lane, int nl,
                              const Red &red, double &R_lo, double &R_hi)
{
  const double U = 1.1102230246251565e-16;             // 2^-53
  const double c[2] = {c0, c1}, w[2] = {w0, w1};
  R_lo = 0.0; R_hi = INFINITY;                         // undecidable until shown otherwise
  // reference slot: the largest a_s at the centre (lowest index on ties); any non-finite input spoils the cell
  double best = -INFINITY; int bad = 0;
  for (int s = lane; s < M; s += nl) {
    double a = 0.0;
    for (int i = 0; i < 2; ++i) {
      double m, h; cell_slot(pool, s, i, m, h);
      if (!(fabs(m) <= DBL_MAX) || !(h < 0.0) || !(h >= -DBL_MAX)) bad = 1;
      a += h * (c[i] - m) * (c[i] - m);
    }
    best = a > best ? a : best;
  }
  const double amax = red.max(best);
  if (red.max(bad ? 1.0 : 0.0) != 0.0 || !(amax > -INFINITY) || !(fabs(c0) <= DBL_MAX) || !(fabs(c1) <= DBL_MAX) ||
      !(w0 >= 0.0 && w0 <= DBL_MAX) || !(w1 >= 0.0 && w1 <= DBL_MAX)) return;
  int mine = M;
  for (int s = lane; s < M; s += nl) {
    double a = 0.0;
    for (int i = 0; i < 2; ++i) {
      double m, h; cell_slot(pool, s, i, m, h);
      a += h * (c[i] - m) * (c[i] - m);
    }
    if (a == amax && s < mine) mine = s;
  }
  const int r = red.min(mine);
  // range of a_r over the box: the nearest and the farthest point of each axis
  double alo = 0.0, ahi = 0.0;
  for (int i = 0; i < 2; ++i) {
    double m, h; cell_slot(pool, r, i, m, h);
    const double y = fabs(c[i] - m), far = y + w[i], near = y > w[i] ? y - w[i] : 0.0;
    alo += h * far * far; ahi += h * near * near;
  }
  alo -= 16.0 * U * fabs(alo); ahi += 16.0 * U * fabs(alo);
  if (!(alo >= -23.025850929940457)) return;           // Q_r >= 1e4 FPEPS = 1e-10 on the whole box (FPEPS = 1e-14)
  double nlo = 0.0, nhi = 0.0, slo = 0.0, shi = 0.0;
  for (int s = lane; s < M; s += nl) {
    double dlo = 0.0, dhi = 0.0, mag = 0.0;
    for (int i = 0; i < 2; ++i) {
      double ms, hs, mr, hr; cell_slot(pool, s, i, ms, hs); cell_slot(pool, r, i, mr, hr);
      const double ys = c[i] - ms, yr = c[i] - mr, wi = w[i];
      const double f0 = hs * ys * ys - hr * yr * yr;
      const double b = 2.0 * (hs * ys - hr * yr), k = hs - hr;   // k: exact sign, zero only for hs == hr
      const double e1 = f0 + b * wi + k * wi * wi, e2 = f0 - b * wi + k * wi * wi;
      double lo = e1 < e2 ? e1 : e2, hi = e1 < e2 ? e2 : e1;
      const double db = 8.0 * U * (fabs(hs * ys) + fabs(hr * yr));   // rounding error of b
      if (k != 0.0 && fabs(b) <= 2.0 * fabs(k) * wi + db) {
        const double bb = fabs(b) + db;
        const double v = f0 - bb * bb / (4.0 * k) * (1.0 + 8.0 * U);
        if (k > 0.0) lo = v < lo ? v : lo; else hi = v > hi ? v : hi;
      }
      dlo += lo; dhi += hi;
      const double ps = fabs(ys) + wi, pr = fabs(yr) + wi;
      mag += fabs(hs) * ps * ps + fabs(hr) * pr * pr;
    }
    const double err = 64.0 * U * mag;
    dlo -= err; dhi += err;
    const double elo = exp(dlo), ehi = exp(dhi);
    nlo = elo > nlo ? elo : nlo; nhi = ehi > nhi ? ehi : nhi;
    slo += elo; shi += ehi;
  }
  nlo = red.max(nlo); nhi = red.max(nhi); slo = red.sum(slo); shi = red.sum(shi);
  const double lo = nlo / (shi + 1.0e-14 * exp(-alo)) * (1.0 - 1.0e-9);
  const double hi = nhi / (slo + 1.0e-14 * exp(-ahi)) * (1.0 + 1.0e-9);
  if (lo >= 0.0 && lo <= 1.0) R_lo = lo;
  if (hi >= 0.0 && hi <= DBL_MAX) R_hi = hi < 1.0 ? hi : 1.0;
}

// x rounded to fp32 downwards / upwards (the stored table keeps the bounds outward)
MCGPU_CB_HD float cell_f32_down(double x)
{
#ifdef __CUDA_ARCH__
  return __double2float_rd(x);
#else
  float f = (float)x;
  if ((double)f > x) f = nextafterf(f, -INFINITY);
  return f;
#endif
}
MCGPU_CB_HD float cell_f32_up(double x)
{
#ifdef __CUDA_ARCH__
  return __double2float_ru(x);
#else
  float f = (float)x;
  if ((double)f < x) f = nextafterf(f, INFINITY);
  return f;
#endif
}

// The stored cell: (R_lo (1 - 1e-6), R_hi (1 + 1e-6)) rounded outward.  A candidate compares its uniform rounded to
// fp32 (relative 2^-24 < 1e-6) against them: uf < lo implies u < R, uf >= hi implies u >= R.
MCGPU_CB_HD void cell_store_bounds(double R_lo, double R_hi, float &lo, float &hi)
{
  lo = cell_f32_down(R_lo * (1.0 - 1.0e-6));
  hi = R_hi <= 1.0 ? cell_f32_up(R_hi * (1.0 + 1.0e-6)) : INFINITY;
}

}  // namespace mcgpu
