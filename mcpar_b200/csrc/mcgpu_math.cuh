// mcgpu_math.cuh -- fp64 exp / log / sincos(2 pi u) for the production step kernels.
//
// Why not CUDA's libm: its double routines carry every polynomial coefficient as an
// immediate (two UMOV per constant, ~90 issue slots per MH step) and evaluate long
// minimax polynomials.  These routines reduce the argument with small lookup tables
// held in SHARED memory (3.5 KB per CTA) so that degree-5/6 Taylor kernels suffice
// (~10 DFMA for exp and log, ~16 for the sin/cos pair), at <= 1.5 ulp.
// They serve the normal (Philox) mode only; the verification instantiations keep
// CUDA's libm so that they stay an independent check.
//
// All functions are __host__ __device__ so tests/test_math_host.cu can measure their
// accuracy on the CPU against long-double references.
#pragma once
#include <stdint.h>
#include <string.h>
#include <math.h>

#ifdef __CUDACC__
#define MCGPU_HD __host__ __device__ __forceinline__
#else
#define MCGPU_HD inline
#endif

namespace mcgpu {

struct MathTables { const double *exp_tab, *log_tab, *trig_tab; };

MCGPU_HD int mc_hi(double x) {
#ifdef __CUDA_ARCH__
  return __double2hiint(x);
#else
  uint64_t b; memcpy(&b, &x, 8); return (int)(b >> 32);
#endif
}
MCGPU_HD int mc_lo(double x) {
#ifdef __CUDA_ARCH__
  return __double2loint(x);
#else
  uint64_t b; memcpy(&b, &x, 8); return (int)(uint32_t)b;
#endif
}
MCGPU_HD double mc_make(int hi, int lo) {
#ifdef __CUDA_ARCH__
  return __hiloint2double(hi, lo);
#else
  uint64_t b = ((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo; double x; memcpy(&x, &b, 8); return x;
#endif
}

// (float)u32_mid(w) = fp32 rounding of (w + 1/2) 2^-32, without the fp64 pipe.  The top 24 bits of w and
// (low 8 bits + 1/2) are both exact in fp32, and so are their products with 2^-32, so the one rounding of
// the final sum is the rounding of (w + 1/2) 2^-32 itself, with or without FMA contraction.  Equal for all
// 2^32 words: tests/test_u32_mid.py.
MCGPU_HD float u32_mid_f32(uint32_t w) {
  const float lo = (float)(w & 0xffu) * 2.3283064365386963e-10f + 1.1641532182693481e-10f;   // (w mod 2^8 + 1/2) 2^-32
  return (float)(w & 0xffffff00u) * 2.3283064365386963e-10f + lo;
}

#define MCGPU_MAGIC 6755399441055744.0      /* 1.5 * 2^52: adding it leaves rint(x) in the low word */

// Scalar coefficients live in CONSTANT memory on the device so that DFMA takes them as
// c[bank][offset] operands; as literals each would cost two UMOV issue slots per use.
#define MCGPU_COEF_LIST                                                                         \
  MCGPU_64_OVER_LN2, -MCGPU_LN2_64_HI, -MCGPU_LN2_64_LO, MCGPU_MAGIC,       /* 0-3  exp reduce */ \
  1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0, 0.5, 1.0,                              /* 4-8  exp poly   */ \
  -1.0 / 6.0, 0.2, -0.25, 1.0 / 3.0, -0.5, -1.0,                             /* 9-14 log poly   */ \
  MCGPU_LN2_HI, MCGPU_LN2_LO,                                                /* 15-16           */ \
  64.0, -1.0 / 64.0, MCGPU_TWO_PI,                                           /* 17-19 trig red. */ \
  -1.0 / 5040.0, 1.0 / 120.0, -1.0 / 6.0,                                    /* 20-22 sin       */ \
  1.0 / 40320.0, -1.0 / 720.0, 1.0 / 24.0, -0.5,                             /* 23-26 cos       */ \
  -708.0, 709.0, -2.0, 0.0                                                   /* 27-30 misc      */
#if defined(__CUDACC__) && !defined(MCGPU_MATH_HOST_ONLY)
static __constant__ double mc_coef_dev[] = {MCGPU_COEF_LIST};
#endif
static const double mc_coef_host[] = {MCGPU_COEF_LIST};
#ifdef __CUDA_ARCH__
#define MCK(i) mc_coef_dev[i]
#else
#define MCK(i) mc_coef_host[i]
#endif

// exp(x).  x < -708 flushes to 0 (the true value is below the normal range);
// x > 709 gives +inf; NaN propagates.
MCGPU_HD double mc_exp(double x, const MathTables &T)
{
  if (((unsigned)mc_hi(x) & 0x7fffffffu) >= 0x40862000u) {   // |x| >= 708, inf or NaN: one integer test on the fast path
    if (x < MCK(27)) return 0.0;
    if (x > MCK(28)) return INFINITY;
    if (x != x) return x;
  }
  const double nd = fma(x, MCK(0), MCK(3));
  const int n = mc_lo(nd);
  const double nf = nd - MCK(3);
  double r = fma(nf, MCK(1), x);
  r = fma(nf, MCK(2), r);                             // |r| <= ln2/128
  const double t = T.exp_tab[n & 63];
  double p = fma(r, MCK(4), MCK(5));                  // Taylor, error r^6/720 < 4e-17
  p = fma(p, r, MCK(6));
  p = fma(p, r, MCK(7));
  p = fma(p, r, MCK(8));
  const double res = fma(t, p * r, t);                // 2^(j/64) * e^r
  return mc_make(mc_hi(res) + ((n >> 6) << 20), mc_lo(res));   // * 2^k, k in [-1022, 1023]
}

// exp(x) for x <= 0 without a branch: the polynomial always runs and x <= -708 (also -inf, and NaN, whose
// result the callers discard) selects 0 at the end -- one integer test and a select instead of a divergent
// special-case block in the step loop.
MCGPU_HD double mc_exp_nonpos(double x, const MathTables &T)
{
  const bool tiny = ((unsigned)mc_hi(x) & 0x7fffffffu) >= 0x40862000u;
  const double nd = fma(x, MCK(0), MCK(3));
  const int n = mc_lo(nd);
  const double nf = nd - MCK(3);
  double r = fma(nf, MCK(1), x);
  r = fma(nf, MCK(2), r);
  const double t = T.exp_tab[n & 63];
  double p = fma(r, MCK(4), MCK(5));
  p = fma(p, r, MCK(6));
  p = fma(p, r, MCK(7));
  p = fma(p, r, MCK(8));
  const double res = fma(t, p * r, t);
  const double y = mc_make(mc_hi(res) + ((n >> 6) << 20), mc_lo(res));
  return tiny ? 0.0 : y;
}

// log(x) for normal positive x.  0 and subnormals give -inf (their logs, below -708, only
// ever mark proposals that are rejected anyway), negative x gives NaN, +inf and NaN pass through.
// CHECKED = false: the caller guarantees a normal, positive, finite x (the Box-Muller argument
// (w+1) 2^-32 in (0, 1]; 1 + e^-t in [1, 2]) and the special-case test disappears.
template <bool CHECKED>
MCGPU_HD double mc_log_t(double x, const MathTables &T)
{
  const int hi = mc_hi(x);
  if (CHECKED && (hi < 0x00100000 || hi >= 0x7ff00000))   // <= 0, subnormal, inf, NaN
    return hi < 0 && x < 0.0 ? NAN : (hi >= 0x7ff00000 && hi > 0 ? x : -INFINITY);
  const int idx = (hi >> 13) & 127;
  const int big = idx >= 53;                           // m >= 1.4140625: use m/2, exponent + 1
  const int e = (hi >> 20) - 1023 + big;
  const double m = mc_make((hi & 0x000fffff) | (big ? 0x3fe00000 : 0x3ff00000), mc_lo(x));
  const double c = T.log_tab[2 * idx], l = T.log_tab[2 * idx + 1];
  const double r = fma(m, c, MCK(14));                 // |r| < 2^-8
  double p = fma(r, MCK(9), MCK(10));                  // log1p(r) = r + r^2 p(r), error r^7/7 < 2e-18
  p = fma(p, r, MCK(11));
  p = fma(p, r, MCK(12));
  p = fma(p, r, MCK(13));
  const double lg = fma(r * r, p, r);
  const double ef = (double)e;
  double res = fma(ef, MCK(15), l);                    // exact-ish: LN2_HI has 26 trailing zero bits
  res += lg;
  return fma(ef, MCK(16), res);
}
MCGPU_HD double mc_log(double x, const MathTables &T) { return mc_log_t<true>(x, T); }
MCGPU_HD double mc_log_pos(double x, const MathTables &T) { return mc_log_t<false>(x, T); }

// sqrt(L) for 0 <= L < 2^100 (the Box-Muller radius: L = -2 ln v <= 44.4).  CUDA's double sqrt is
// 27 issue slots (MUFU.RSQ64H, a Newton chain and a special-case branch); here the SFU's fp32
// reciprocal square root y0 = (1 + d) / sqrt(L), |d| <= 2^-21 (twice the documented bound), seeds two
// Newton corrections r <- r + (L - r^2) y0 / 2 of r = L y0, each with an exact fma residual: the
// relative error e of r becomes -e^2/2 - e d, i.e. 2^-21 -> 2^-41 -> 2^-62, and the last fma rounds once:
// <= 0.51 ulp in 2 DMUL + 4 DFMA.  L = 0 gives 0.  `seed_err` perturbs the host stand-in of the SFU seed
// so that the accuracy test covers the worst case.
MCGPU_HD double mc_sqrt_pos(double L, double seed_err = 0.0)
{
#ifdef __CUDA_ARCH__
  float y0f;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y0f) : "f"(fmaxf((float)L, 1.0e-30f)));
  const double y0 = (double)y0f;
#else
  const float lf = (float)L > 1.0e-30f ? (float)L : 1.0e-30f;
  const double y0 = (double)(float)((1.0 / sqrt((double)lf)) * (1.0 + seed_err));
#endif
  const double h = 0.5 * y0;
  double r = L * y0;
  r = fma(fma(-r, r, L), h, r);
  return fma(fma(-r, r, L), h, r);
}

// (sin, cos)(2 pi u) for u in [0, 1]
MCGPU_HD void mc_sincos2pi(double u, double &s, double &c, const MathTables &T)
{
  const double kd = fma(u, MCK(17), MCK(3));
  const int k = mc_lo(kd);
  const double f = fma(kd - MCK(3), MCK(18), u);               // exact, |f| <= 1/128
  const double b = f * MCK(19);                                // |b| <= pi/64
  const double sa = T.trig_tab[2 * (k & 63)], ca = T.trig_tab[2 * (k & 63) + 1];
  const double b2 = b * b;
  double ps = fma(b2, MCK(20), MCK(21));                       // sin b = b + b^3 ps, error b^9/9!
  ps = fma(ps, b2, MCK(22));
  const double sb = fma(b * b2, ps, b);
  double pc = fma(b2, MCK(23), MCK(24));                       // cos b - 1 = b^2 pc, error b^10/10!
  pc = fma(pc, b2, MCK(25));
  pc = fma(pc, b2, MCK(26));
  const double cm1 = pc * b2;
  s = fma(ca, sb, fma(sa, cm1, sa));
  c = fma(-sa, sb, fma(ca, cm1, ca));
}

}  // namespace mcgpu
