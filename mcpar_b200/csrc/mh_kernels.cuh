// mh_kernels.cuh -- the fused Metropolis-Hastings step kernels (sm_100a).
//
// Included by two translation units:
//   mh_fast.cu   (default FMA contraction)           -> namespace mcgpu::fast
//   mh_exact.cu  (-fmad=false, MCGPU_EXACT_TU)       -> namespace mcgpu::exact
// The exact unit evaluates every expression operation by operation exactly as the
// reference's C++ does (src/mcpar.cc, src/rosenbrock.cc), so states and polynomial
// log-likelihoods are bit-identical to the CPU oracle on shared streams.
//
// Kernel 1  mh_steps_kernel<LIK,D,RNG,PHASE>  production path: one thread per chain,
//           K steps per launch, state in registers; fuses proposal generation
//           (genLocal mcpar.cc:302-312 / genRemote :315-451), likelihood
//           (VLFunc, rosenbrock.cc), accept + update (:65-75,:165-175), running
//           moments (:186-209), publication to the exchange pool (:205-208) and the
//           sample store (MCout::add, mcout.cc:129-145).
// Kernel 2  mh_verify_kernel                  verification mode: one CTA per emulated
//           MPI rank, the reference's lock-step stream protocol (SURVEY.md 8c).
#pragma once
#include <stdlib.h>
#include "mcgpu_device.cuh"
#include "../../include/mcgpu.h"
#ifndef MCGPU_EXACT_TU
#define MCGPU_TABLE_QUAL static __device__ __align__(16)
#include "mcgpu_tables.h"
#else
#define MCGPU_64_OVER_LN2 0.0
#define MCGPU_LN2_64_HI 0.0
#define MCGPU_LN2_64_LO 0.0
#define MCGPU_LN2_HI 0.0
#define MCGPU_LN2_LO 0.0
#define MCGPU_TWO_PI 0.0
#endif
#include "mcgpu_math.cuh"

namespace mcgpu {
namespace MCGPU_NS {

enum { RNG_PHILOX = 0, RNG_REPLAY = 1 };

// transcendental calls of the step kernels: table-driven routines in the production
// unit, CUDA libm in the exact (verification) unit
#ifdef MCGPU_EXACT_TU
#define MC_EXP(x) exp(x)
#define MC_LOG(x) log(x)
#define MCGPU_MATH_SMEM 0
#else
#define MC_EXP(x) mc_exp((x), T)
#define MC_LOG(x) mc_log((x), T)
#define MCGPU_MATH_SMEM (MCGPU_EXP_TAB + 2 * MCGPU_LOG_TAB + 2 * MCGPU_TRIG_TAB)   /* doubles */
#endif

#ifndef MCGPU_EXACT_TU
// copy the exp / log / trig tables (3.5 KB) into shared memory, 16 bytes per access
__device__ __forceinline__ void stage_math_tables(double *smem)
{
  double2 *d = reinterpret_cast<double2 *>(smem);
  const double2 *e = reinterpret_cast<const double2 *>(MCGPU_EXP_TABLE), *l = reinterpret_cast<const double2 *>(MCGPU_LOG_TABLE),
                *t = reinterpret_cast<const double2 *>(MCGPU_TRIG_TABLE);
  for (int i = threadIdx.x; i < MCGPU_EXP_TAB / 2; i += blockDim.x) d[i] = e[i];
  for (int i = threadIdx.x; i < MCGPU_LOG_TAB; i += blockDim.x) d[MCGPU_EXP_TAB / 2 + i] = l[i];
  for (int i = threadIdx.x; i < MCGPU_TRIG_TAB; i += blockDim.x) d[MCGPU_EXP_TAB / 2 + MCGPU_LOG_TAB + i] = t[i];
}
#endif

// Box-Muller pair, MKL BOXMULLER2 convention: z0 = r sin(2 pi u2), z1 = r cos(2 pi u2)
__device__ __forceinline__ void normal_pair_t(uint32_t wa, uint32_t wb, double &z0, double &z1, const MathTables &T)
{
#ifdef MCGPU_EXACT_TU
  normal_pair(wa, wb, z0, z1);
#else
  // v = (w+1) 2^-32 in (0, 1] is normal and positive, so the unchecked log applies and ln v <= 0 (exactly 0 at
  // v = 1: table entry 0 is (1, 0)): L = -2 ln v >= 0 needs no clamp
  const double r = mc_sqrt_pos(-2.0 * mc_log_pos(u32_pos(wa), T));
  double s, c;
  mc_sincos2pi(u32_half(wb), s, c, T);
  z0 = r * s; z1 = r * c;
#endif
}

// ----------------------------------------------------------------------------
// likelihood functors (device side of the VLFunc plugin surface)
// ----------------------------------------------------------------------------
template <int LIK, int D> struct Lik;

// Rosenbrock1::operator(), rosenbrock.cc:4-21: non-overlapping pairs
template <int D> struct Lik<MCGPU_ROSENBROCK1, D> {
  static __device__ __forceinline__ double eval(const double (&x)[D], const StepParams &, const MathTables &) {
    double y = 0.0;
#pragma unroll
    for (int i = 0; i + 1 < D; i += 2) {
      const double t1 = 1 - x[i];
      const double t2 = x[i + 1] - x[i] * x[i];
      y -= t1 * t1 + 100.0 * t2 * t2;
    }
    return y;
  }
};

// Gaussian::operator(), rosenbrock.cc:44-61; lp = {mu0, mu1, 1/sig2_0, 1/sig2_1}
template <> struct Lik<MCGPU_GAUSSIAN, 2> {
  static __device__ __forceinline__ double eval(const double (&x)[2], const StepParams &p, const MathTables &T) {
    double y = 0.0;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const double arg = x[k] - p.lp[k];
      y -= 0.5 * arg * arg * p.lp[2 + k];
    }
    return y;
  }
};

// DualGaussian::operator(), rosenbrock.cc:63-78; lp = {w}.  No log-sum-exp guard,
// as in the reference: far from both modes this is log(0) = -inf.
template <> struct Lik<MCGPU_DUALGAUSSIAN, 2> {
  static __device__ __forceinline__ double eval(const double (&x)[2], const StepParams &p, const MathTables &T) {
    const double arg1 = 0.5 * (x[0] * x[0] + x[1] * x[1]);
    const double t2a = x[0] - 5.0, t2b = x[1] - 5.0;
    const double narg2 = -0.5 * (t2a * t2a + t2b * t2b);
#ifdef MCGPU_EXACT_TU
    return MC_LOG(p.lp[0] * MC_EXP(-arg1) + MC_EXP(narg2));
#else
    // the same value with one exponential instead of two:  log(w e^-a1 + e^-a2) = M + log(1 + e^-|t1 - t2|),
    // t1 = log w - a1, t2 = -a2, M = max(t1, t2)  (lp[1] = log w, set on the host).  When BOTH exponentials of
    // the two-exp form flush to zero (a1, a2 >= 708, DESIGN.md 4.6) the result is log(0) = -inf, as in the
    // reference; a single flushed term only ever changes the sum below 1e-16 relative (the other term is
    // then e^37 times larger) unless both are within reach of the flush, where the reference itself runs on
    // denormals.  The comparisons are integer tests on the high words.
    const double t1 = p.lp[1] - arg1;
    const double dt = t1 - narg2;
    const double M = __double2hiint(dt) < 0 ? narg2 : t1;
    const double r = M + mc_log_pos(1.0 + mc_exp_nonpos(-fabs(dt), T), T);   // argument in [1, 2]
    const bool dead = __double2hiint(arg1) >= 0x40862000 && (unsigned)__double2hiint(narg2) >= 0xC0862000u;
    return dead ? -INFINITY : r;
#endif
  }
};

// GaussMix (new; SURVEY.md 8a L5): log sum_k w_k exp(-1/2 sum_i (x_i-mu_ki)^2/s2_ki)
// with log-sum-exp.  lik_dev = {mu[K][d], 1/s2[K][d], log w[K]} (prepared on upload).
template <int D> struct Lik<MCGPU_GAUSSMIX, D> {
  static __device__ __forceinline__ double eval(const double (&x)[D], const StepParams &p, const MathTables &T) {
    const int K = p.lik_k;
    const double *mu = p.lik_dev, *is2 = mu + (size_t)K * D, *lw = is2 + (size_t)K * D;
    double m = -INFINITY, s = 0.0;
    for (int k = 0; k < K; ++k) {
      double q = 0.0;
#pragma unroll
      for (int i = 0; i < D; ++i) { const double xm = x[i] - mu[k * D + i]; q += xm * xm * is2[k * D + i]; }
      const double a = lw[k] - 0.5 * q;
      if (a > m) { s = s * MC_EXP(m - a) + 1.0; m = a; } else s += MC_EXP(a - m);
    }
    return m + MC_LOG(s);
  }
};

// ----------------------------------------------------------------------------
// Kernel 1: production path
// ----------------------------------------------------------------------------

// Out-of-line Philox call for d > 4: keeps the step's several blocks from being scheduled all
// at once (every Philox state live -> past 255 registers).
__device__ __noinline__ Words philox_call(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1)
{
  return philox4x32_10(c0, c1, c2, c3, k0, k1);
}
// RK: take the precomputed round keys from the launch parameters (constant-bank operands of the LOP3s)
template <int D, bool RK>
__device__ __forceinline__ Words philox_d(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const StepParams &p)
{
  if (D <= 4 && RK) return philox4x32_10_rk(c0, c1, c2, c3, p.rk);
  if (D <= 4) return philox4x32_10(c0, c1, c2, c3, p.key0, p.key1);
  return philox_call(c0, c1, c2, c3, p.key0, p.key1);
}

// proposal factor entry from shared memory.  At d > 4 the read is volatile: the d(d+1)/2
// entries are loop-invariant and would otherwise be hoisted into registers for the whole step loop.
template <int D>
__device__ __forceinline__ double factor_at(const double *sT, int idx)
{
#ifdef MCGPU_FACTOR_HOIST
  if (D <= 4) return sT[idx];
#endif
  return *reinterpret_cast<const volatile double *>(sT + idx);
}

// exp2 on the SFU (fp32): used only to BOUND quantities whose exact value is not
// needed -- decisions fall back to fp64 whenever a bound does not settle them.
__device__ __forceinline__ float ex2_approx(float x)
{
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// the exact evaluation behind every bounded accept test: rare (~1e-4 of the steps), so one out-of-line copy
__device__ __noinline__ bool accept_exact(double u, double delta, double cfac, const MathTables T)
{
  return u < MC_EXP(delta) * cfac;
}

// The accept test  u < exp(delta) * cfac  (mcpar.cc:67-69 / :167-169).  Only the
// decision is needed, so it is settled by rigorous fp32 bounds on exp(delta) and
// computed exactly (fp64 exp) only when u falls between the bounds (~1e-4 of cases).
__device__ __forceinline__ bool accept_test(double u, double delta, double cfac, const MathTables &T, int exact_tests)
{
#ifdef MCGPU_EXACT_TU
  return u < exp(delta) * cfac;
#else
  if (exact_tests) return accept_exact(u, delta, cfac, T);   // audit mode (MCGPU_EXACT_TESTS): no fp32 short cut
  const float dc = fminf(fmaxf((float)delta, -80.0f), 80.0f);
  const double e = (double)ex2_approx(dc * 1.4426950408889634f);
  const double lo = (delta >= -80.0) ? e * cfac * (1.0 - 1.0e-4) : 0.0;   // valid lower bound (clamped above 80)
  const double hi = (delta <= 80.0) ? e * cfac * (1.0 + 1.0e-4) : INFINITY;
  if (u < lo) return true;
  if (u >= hi) return false;
  return accept_exact(u, delta, cfac, T);             // also the NaN path: comparisons above are false
#endif
}

// The same for steps without a Hastings factor (local proposals, burn-in): u < exp(delta).  exp(80) > 1 > u and
// exp(-80) < 2^-33 <= u settle |delta| >= 80 outright; in between the comparison runs in fp32 -- u rounded to
// fp32 (relative 2^-24) against exp2.approx with the same 1e-4 margin -- so the FP64 pipe sees no compare at all.
__device__ __forceinline__ bool accept_test_local(double u, double delta, const MathTables &T, int exact_tests)
{
#ifdef MCGPU_EXACT_TU
  return u < exp(delta);
#else
  if (exact_tests) return accept_exact(u, delta, 1.0, T);              // audit mode
  // No clamps: ex2.approx saturates the right way -- delta >= 88.8 (also +inf) gives e = +inf > u: accept;
  // delta <= -87.4 (also -inf) gives e = 0 <= u: reject; NaN fails both comparisons and reaches the exact test,
  // where u < NaN is false.  In between e carries < 2e-5 relative error (float(delta) and the product 1.3e-5
  // at |delta| <= 88, the fp32 log2(e) 2e-6, ex2.approx 2.4e-7), inside the 1e-4 margin.
  const float df = (float)delta;
  const float e = ex2_approx(df * 1.4426950408889634f), uf = (float)u;
  if (uf < e * (1.0f - 1.0e-4f)) return true;
  if (uf >= e * (1.0f + 1.0e-4f)) return false;
  return accept_exact(u, delta, 1.0, T);
#endif
}

// One candidate of the remote rejection loop, exactly: draws (component pick, uniform, normals) from the
// candidate's Philox blocks, x' = mu_c + sigma_c z and pacpt = qimax / qisum (mcpar.cc:337-398), all in
// fp64.  Out of line: it runs for ~1e-3 of the candidates and must not bloat the hot loop.
template <int D>
__device__ __noinline__ bool remote_exact(uint32_t tlo, uint32_t thi, uint32_t step, uint32_t slot, uint32_t k0, uint32_t k1,
                                          const double2 *sPmh, const double *sPs, int M, const MathTables &T)
{
  constexpr int NP = (D + 1) / 2;
  Words blk = philox4x32_10(tlo, thi, step, slot, k0, k1);
  const int c = (int)__umulhi(blk.w0, (uint32_t)M);
  const double u = u32_mid(blk.w1);
  double xc[D];
#pragma unroll
  for (int q = 0; q < NP; ++q) {
    const int qq = q + 1;
    if ((qq & 1) == 0) blk = philox4x32_10(tlo, thi, step, slot + (uint32_t)(qq >> 1), k0, k1);
    double za, zb;
    normal_pair_t((qq & 1) ? blk.w2 : blk.w0, (qq & 1) ? blk.w3 : blk.w1, za, zb, T);
    xc[2 * q] = sPmh[c * D + 2 * q].x + sPs[c * D + 2 * q] * za;
    if (2 * q + 1 < D) xc[2 * q + 1] = sPmh[c * D + 2 * q + 1].x + sPs[c * D + 2 * q + 1] * zb;
  }
  double qmax = MCGPU_FPEPS, qsum = MCGPU_FPEPS;
  for (int s = 0; s < M; ++s) {
    double a = 0.0;
#pragma unroll
    for (int i = 0; i < D; ++i) { const double2 mh = sPmh[s * D + i]; const double xm = mh.x - xc[i]; a += xm * xm * mh.y; }
    const double gv = mc_exp(a, T);
    qsum += gv; qmax = gv > qmax ? gv : qmax;
  }
  return u < qmax / qsum;
}

// c_recip[n] = ceil(2^16 / n): (lane * c_recip[n]) >> 16 == lane / n for lane < 32, n <= 32
__constant__ unsigned c_recip[33] = {0u, 65536u, 32768u, 21846u, 16384u, 13108u, 10923u, 9363u, 8192u, 7282u, 6554u, 5958u, 5462u,
  5042u, 4682u, 4370u, 4096u, 3856u, 3641u, 3450u, 3277u, 3121u, 2979u, 2850u, 2731u, 2622u, 2521u, 2428u, 2341u, 2260u, 2185u,
  2115u, 2048u};
// c_stride_mask[n]: bits 0, n, 2n, ... below 32
__constant__ unsigned c_stride_mask[33] = {0u,
  0xffffffffu, 0x55555555u, 0x49249249u, 0x11111111u, 0x42108421u, 0x41041041u, 0x10204081u, 0x01010101u,
  0x08040201u, 0x40100401u, 0x00400801u, 0x01001001u, 0x04002001u, 0x10004001u, 0x40008001u, 0x00010001u,
  0x00020001u, 0x00040001u, 0x00080001u, 0x00100001u, 0x00200001u, 0x00400001u, 0x00800001u, 0x01000001u,
  0x02000001u, 0x04000001u, 0x08000001u, 0x10000001u, 0x20000001u, 0x40000001u, 0x80000001u, 0x00000001u};

// SFU approximations (fp32).  Documented error bounds used below, each with a margin of 3x or more:
// lg2.approx |err| <= 2^-22 absolute on [0.5, 2] (2 ulp elsewhere); sin/cos.approx |err| <= 2^-20.9 on
// [-pi, pi]; sqrt.approx and ex2.approx 2 ulp.
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rsqrt_approx(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sin_approx(float x) { float y; asm("sin.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float cos_approx(float x) { float y; asm("cos.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// fp32 image of the Box-Muller pair of normal_pair_t (same words, same convention).  Returns a bound on
// the absolute error of both normals:
//   L = -2 ln v:  |dL| <= 1.39 dlg2 + 2.4e-7 (1 + L) <= 1.6e-6, with dlg2 = 1e-6 (4x the documented bound);
//   r = sqrt L = L rsqrt(L):   |dr| <= dL / (r~ + r) + 3e-7 r, and never more than sqrt(dL) = 1.3e-3 (below
//   r = 1.3e-3 the capped 1/r makes r~ = 770 L <= r, still within 1.3e-3 of it);
//   angle 2 pi (a - 1/2), |a - 1/2| <= 1/2: argument error <= 8e-7, sin/cos error <= 2e-6 (the
//   approximation's 5.1e-7 tripled, plus the argument's);  z = r trig:  |dz| <= dr + r (2e-6 + 1.2e-7)
//   <= 1.7e-6 min(1/r~, 770) + 2.4e-6 r~.
__device__ __forceinline__ float normal_pair_f32(uint32_t wa, uint32_t wb, float &z0, float &z1, float &lg)
{
  // ((float)wa + 1) 2^-32 in one FFMA: scaling by 2^-32 is exact here, so the single rounding is that of the sum
  const float v = fmaf((float)wa, 2.3283064365386963e-10f, 2.3283064365386963e-10f);   // (0, 1]
  lg = lg2_approx(v);                                                           // = -(z0^2 + z1^2)/2 * log2(e), in [-32, 0]
  const float L = -1.3862943611198906f * lg;
  const float rs = fminf(rsqrt_approx(L), 770.0f);                              // 1/r, capped at 1/1.3e-3 (also L = 0: inf)
  const float r = L * rs;                                                       // sqrt L (2 ulp + the cap, which only bites below r = 1.3e-3)
  const float ang = 6.283185307179586f * ((float)wb * 2.3283064365386963e-10f - 0.5f);   // 2 pi u - pi in [-pi, pi]
  z0 = -r * sin_approx(ang); z1 = -r * cos_approx(ang);                         // sin(t + pi) = -sin t, cos(t + pi) = -cos t
  return fmaf(2.4e-6f, r, 1.7e-6f * rs);
}

// The fp32 pool copy sPf (stage_pool) holds the slots in pairs: sPf[(s / 2) D + i] = (g mu_si, g mu_s'i, g_si, g_s'i)
// for the even slot s and s' = s + 1 (the pool is padded to a multiple of 8 slots), so one FFMA2 evaluates a
// parameter for both slots of a pair.  Each lane of FFMA2 is the same IEEE round-to-nearest fma as fmaf, so
// every value below is bit for bit that of the slot-by-slot scalar loop.
// Returns acc_s - sum_i (g mu_si - g_si x_i)^2 for the pair (s, s + 1), s even, summed over i = 0, 1, ... in
// order; xx[i] = (x_i, x_i).
template <int D>
__device__ __forceinline__ float2 pool_pair(const float4 *sPf, int s, const float2 (&xx)[D], float2 acc)
{
#pragma unroll
  for (int i = 0; i < D; ++i) {
    const float4 f = sPf[(s >> 1) * D + i];
    const float2 y = __ffma2_rn(make_float2(-f.z, -f.w), xx[i], make_float2(f.x, f.y));   // g (mu - x)
    acc = __ffma2_rn(make_float2(-y.x, -y.y), y, acc);
  }
  return acc;
}

// (g mu_ci, g_ci) of one slot c of the paired layout above
__device__ __forceinline__ float2 pool_slot(const float4 *sPf, int D, int c, int i)
{
  const float *f = reinterpret_cast<const float *>(sPf + (c >> 1) * D + i) + (c & 1);
  return make_float2(f[0], f[2]);
}

// One candidate of the remote rejection loop (genRemote, mcpar.cc:331-409), decision only: draw the
// component c, the uniform u and the normals z from the candidate's Philox blocks, form
// x' = mu_c + sigma_c z and decide  u < max_s Q_s(x') / sum_s Q_s(x')  over the pool.  Rejected candidates
// leave no trace and the accepted one is re-materialised in fp64 by its chain afterwards, so everything
// here runs in fp32 on an fp32 copy of the pool -- sPf = (g mu, g) with g = sqrt(log2(e)/(2 sigma^2)) in slot pairs
// (pool_pair), sSf = (sigma, mu), padded to a multiple of 8 slots whose Q is 0; SFU log2/sqrt/sin/cos/exp2; chunks of
// 8 slots for ILP with one rescale per chunk -- under a rigorous bound on the relative error of
//     R = sum_s exp(a_s - max a),   a_s = -sum_i (mu_si - x'_i)^2 / (2 sigma_si^2);
// when the bound does not settle u the candidate is redone exactly in fp64 (remote_exact).
// Error bound.  mu_s - x' (formed as (g mu - g x') / g) is off by at most delta = zerr sigma_c,max (normals,
// normal_pair_f32) + 3 u24 (|mu|max + |x'|) (roundings of mu_c, sigma_c, g mu_s, g and the fmas), u24 = 2^-24.  A term with |a_s| <= A then moves by at
// most sqrt(2 A D) theta + (6 + D) u24 A, theta = delta / sigma_min.  Terms that matter have A <= 35 (the
// bound is only used when max a > -10; terms 25 below the max contribute < 1.4e-11 each, and their own
// error cannot lift them: sqrt(|a|) theta << |a| - 35).  Both a_s and the max move, so every term of R is
// right to a factor exp(+-2 (8.4 sqrt(D) theta + (6 + D) 2.1e-6)); exp2.approx and the fp32 sum add
// < 1e-6 M.  eps below covers all of it with margin.  theta >= 2e-3 (components far tighter than others or
// than their distance from the origin: e.g. the first window, where sigma ~ 1e-7) goes to the exact test.
// tests/test_gpu_audit.py checks the decisions against an all-fp64 run of the same kernels.
// The launch-uniform inputs come from the caller, once per remote step: mu_max, isig_max (s_scal), eps0 =
// (1.01e-4 + 1e-5 D) + 2e-5 M (remote_eps0), Mpad, and bounded = !p.exact_tests.
#ifdef MCGPU_CELL_COUNT
// counting build (tools/build_variant.py): table-decided candidates, rounds with a table miss, rounds
__device__ unsigned long long mcgpu_cell_count[4];
#endif
template <int D>
__device__ __forceinline__ float remote_eps0(int M) { return fmaf(2.0e-5f, (float)M, 1.01e-4f + 1.0e-5f * (float)D); }

template <int D, bool RK>
__device__ __forceinline__ bool remote_candidate(uint32_t tlo, uint32_t thi, uint32_t step, uint32_t slot, const StepParams &p,
                                                 const float4 *sPf, const float2 *sSf, const double2 *sPmh, const double *sPs,
                                                 float mu_max, float isig_max, float eps0, int Mpad, bool bounded,
                                                 const MathTables &T, unsigned int *s_fallback)
{
  constexpr int CH = 8;
  constexpr int NP = (D + 1) / 2;
  const int M = p.pool_m;
  Words blk = philox_d<D, RK>(tlo, thi, step, slot, p);
  const int c = (int)__umulhi(blk.w0, (uint32_t)M);                 // viRngUniform(0, tchains), mcpar.cc:337
  const uint32_t uw = blk.w1;                                       // vsRngUniform, mcpar.cc:401: u = u32_mid(uw)
  float xf[D], xabs = 0.0f, sgmax = 0.0f, zerr = 0.0f, ref = 0.0f;
#pragma unroll
  for (int q = 0; q < NP; ++q) {                                    // pair q = words (2+2q, 3+2q) of the candidate's stream
    const int qq = q + 1;
    if ((qq & 1) == 0) blk = philox_d<D, RK>(tlo, thi, step, slot + (uint32_t)(qq >> 1), p);
    float za, zb, lg;
    zerr = fmaxf(zerr, normal_pair_f32((qq & 1) ? blk.w2 : blk.w0, (qq & 1) ? blk.w3 : blk.w1, za, zb, lg));
    ref += lg;                                                      // a_c * log2(e) of the picked component itself
    {
      const int i = 2 * q; const float2 sm = sSf[c * D + i];
      xf[i] = fmaf(sm.x, za, sm.y);                                 // DIAGONAL storage, :348-350
      xabs = fmaxf(xabs, fabsf(xf[i])); sgmax = fmaxf(sgmax, sm.x);
    }
    if (2 * q + 1 < D) {
      const int i = 2 * q + 1; const float2 sm = sSf[c * D + i];
      xf[i] = fmaf(sm.x, zb, sm.y);
      xabs = fmaxf(xabs, fabsf(xf[i])); sgmax = fmaxf(sgmax, sm.x);
    }
  }
  float2 xx[D];
#pragma unroll
  for (int i = 0; i < D; ++i) xx[i] = make_float2(xf[i], xf[i]);
  const float dx = fmaf(1.9e-7f, mu_max + xabs, zerr * sgmax);    // bounds |x'_f32 - x'_fp64| per parameter
  const float theta = dx * isig_max;
  // the comparison itself runs in fp32 as well: u rounded to fp32 and three fp32 roundings add < 3e-7 to eps
  const float epsf = fmaf(theta, 21.3f * sqrtf((float)D), eps0);
  if constexpr (D <= 4) {
    // Exponents are taken relative to the picked component's own a_c = log2 v (>= -32 per normal pair), which
    // the Box-Muller step already has: 2^(a_s - a_c) <= 2^64 cannot overflow, so the sum needs no running
    // maximum and no rescaling -- the accumulator simply starts at -a_c.
    // Early reject: Q_s <= 1, so max_s Q_s / sum_s Q_s <= 1 / (Q_c S) with S any partial sum of 2^(a_s - a_c):
    // the candidate is rejected as soon as u S (1 - eps) >= 2^(-a_c), without the rest of the pool (at the
    // plateau max/sum ~ 1/M, so most candidates leave after the first chunks; the FPEPS offsets of
    // mcpar.cc:357-358 only lower the ratio further).
    const bool fastok = theta < 2.0e-3f && bounded;
    const float uf = u32_mid_f32(uw);                                // (float)u
    const float uf_lo = uf * (1.0f - epsf) * (1.0f - 2.0e-7f), ebound = ex2_approx(-ref) * (1.0f + 1.0e-6f);
    if constexpr (D == 2) {
      // The window's table of rigorous bounds on R (mcgpu_cellbound.cuh): each cell was dilated by 1/64 of its width,
      // which covers |x'_f32 - x'_fp64| < 1/128 of a width and the fp32 rounding of the cell index.  The fp64
      // candidate that remote_exact would evaluate lies in the dilated cell, so the stored bounds settle u as that
      // evaluation would; a candidate outside the grid or between the bounds runs the pool loop below.
      const float4 *const tab = p.cell_tab;
      if (tab != nullptr) {
        const float4 hd = __ldg(tab);                  // (origin x, origin y, 1/width x, 1/width y); NaN: no valid table
        const int gx = __float2int_rd((xf[0] - hd.x) * hd.z), gy = __float2int_rd((xf[1] - hd.y) * hd.w);
        bool hit = false, dec = false;
        if (dx * fmaxf(hd.z, hd.w) < 0.0078125f && (unsigned)gx < (unsigned)MCGPU_CELL_G && (unsigned)gy < (unsigned)MCGPU_CELL_G) {
          const float2 b = __ldg(reinterpret_cast<const float2 *>(tab + 1) + gy * MCGPU_CELL_G + gx);
          dec = uf < b.x;                              // u < R_lo
          hit = dec || uf >= b.y;                      // or u >= R_hi
        }
#ifdef MCGPU_CELL_COUNT
        const unsigned miss = __ballot_sync(0xffffffffu, !hit);
        if ((threadIdx.x & 31) == 0) {
          atomicAdd(&mcgpu_cell_count[0], (unsigned long long)(32 - __popc(miss)));
          atomicAdd(&mcgpu_cell_count[1], miss ? 1ull : 0ull);
          atomicAdd(&mcgpu_cell_count[2], 1ull);
        }
#endif
        if (hit) return dec;
      }
    }
    const float2 acc0 = make_float2(-ref, -ref);
    float mr = -INFINITY, S = 0.0f;                    // max_s and sum_s of 2^(a_s - a_c)
    for (int s0 = 0; s0 < Mpad;) {                     // (before the first chunk S = 0 and ebound >= 1: no test)
#pragma unroll
      for (int q = 0; q < CH; q += 2) {
        const float2 acc = pool_pair<D>(sPf, s0 + q, xx, acc0);
        mr = fmaxf(mr, acc.x); S += ex2_approx(acc.x);
        mr = fmaxf(mr, acc.y); S += ex2_approx(acc.y);
      }
      s0 += CH;
      if (s0 < Mpad && fastok && uf_lo * S >= ebound) return false;
    }
    if (mr + ref > -14.0f && fastok) {                 // max a > -9.7: then FPEPS/qmax < 2e-10 (mcpar.cc:357-358 offsets)
      const float E = ex2_approx(mr);                               // R = S / E
      if (uf * fmaf(S, 1.0f + epsf, 3.0e-10f * E) < E) return true;  // u < r_lo
      if (uf * (S * (1.0f - epsf)) >= E) return false;               // u >= r_hi
    }
  } else {
    const double u = u32_mid(uw), eps = (double)epsf;
    float m = -INFINITY;                               // running max of a_s * log2(e)
    float S = 0.0f;                                    // sum_s 2^(a_s - m)
    for (int s0 = 0; s0 < Mpad; s0 += CH) {
      float a[CH];
#pragma unroll
      for (int q = 0; q < CH; q += 2) {
        const float2 acc = pool_pair<D>(sPf, s0 + q, xx, make_float2(0.0f, 0.0f));
        a[q] = acc.x; a[q + 1] = acc.y;
      }
      float mc = a[0];
#pragma unroll
      for (int q = 1; q < CH; ++q) mc = fmaxf(mc, a[q]);
      float sc = 0.0f;
#pragma unroll
      for (int q = 0; q < CH; ++q) sc += ex2_approx(a[q] - mc);                   // each <= 1
      const bool gt = mc > m;
      const float e = ex2_approx(-fabsf(m - mc));                                 // 0 on the first chunk
      S = gt ? fmaf(S, e, sc) : fmaf(sc, e, S);
      m = gt ? mc : m;
    }
    if (m > -14.0f && theta < 2.0e-3f && bounded) {
      const double Sd = (double)S;
      if (u * (Sd * (1.0 + eps) + 3.0e-10) < 1.0) return true;      // u < r_lo
      if (u * (Sd * (1.0 - eps)) >= 1.0) return false;              // u >= r_hi
    }
  }
  atomicAdd(s_fallback, 1u);                            // statistics: candidates the fp32 bounds did not settle
  return remote_exact<D>(tlo, thi, step, slot, p.key0, p.key1, sPmh, sPs, M, T);   // rare: the bounds straddle u (also the NaN path)
}

#ifndef MCGPU_MINB_LOCAL
#define MCGPU_MINB_LOCAL 9    // d = 2 local-only kernels: <= 56 registers, 36 warps per SM (10 -> 48 registers costs ~5 % more
                              // instructions in rematerialised constants: 7.33e10 vs 7.56e10 chain-steps/s, profiles/r02_tuning.md)
#endif
#ifndef MCGPU_MINB
#define MCGPU_MINB 7      // d = 2: cap registers at 72 (7 CTAs of 128 per SM); +2 % over 6 in all three remote configurations (profiles/r02_tuning.md)
#endif
// PHASE selects what a launch may contain:
//   PH_BURN    burn-in steps (local proposals, no moments, no history)            mcpar.cc:56-97
//   PH_MIXED   main steps, one local/remote coin per group of <= 32 chains (a warp may hold
//              both kinds of step)                                                  mcpar.cc:113-210
//   PH_LOCAL   main steps known to be local for every chain (job-wide coin, or t < SYNCSTEP)
// With a job-wide coin (coin_group = 0: "one coin per rank per step", the rank being the whole
// job) the host knows each step's kind in advance -- the coin is a counter-based draw -- and
// launches chunks of up to 32 steps: the lean PH_LOCAL kernel (no remote code, few registers,
// full occupancy) when no step of the chunk is remote, otherwise PH_MIXED with the chunk's plan.
//   PH_MIXED_SUM  PH_MIXED with remote mode 1: the sum-mixture proposal below
// PH_REMOTE / PH_REMOTE_SUM (all steps remote) are phases of the wide kernels only (mh_wide.cuh).
enum { PH_BURN = 0, PH_MIXED = 1, PH_LOCAL = 2, PH_REMOTE = 3, PH_MIXED_SUM = 4, PH_REMOTE_SUM = 5 };

// ---- remote mode 1: sum-mixture independence proposal ----------------------------------------------
// (SURVEY.md section 7 H1: Murray's mixture proposal in place of the reference's rejection loop,
// mcpar.cc:333-443.)  x' is drawn from the uniform mixture of the pool's diagonal Gaussians -- one pick,
// one set of normals, no loop -- and the Metropolis ratio carries the exact Hastings factor
//     cfac = q(x) / q(x'),   q(y) = sum_s N(y; mu_s, diag sig2_s)    (NORMALISED components),
// so the chain leaves the target invariant whatever the widths in the pool (the reference's
// max_i Q_i / max_i Q_i correction with unnormalised Q_i does not: DESIGN.md section 4).  Cost: two
// passes over the pool, O(M d), instead of ~M candidates x O(M d).
//
// Only the accept decision is needed, so cfac is first BOUNDED in fp32: with A_s(y) = nb_s - sum_i
// (g_si mu_si - g_si y_i)^2 the log2 of component s at y (nb_s = -1/2 sum_i log2 sig2_si, g as in
// stage_pool) and ref = A_c(x') of the picked component, So = sum_s 2^(A_s(x) - ref) and Sn = sum_s
// 2^(A_s(x') - ref) give cfac = So / Sn; Sn >= 1 (its term c) and neither sum needs a running maximum.
// Error bound of one sum at point y.  y_i - mu_si is off by at most (roundings of g mu, g, y and the
// fma) 2.55 u24 (|mu|max + |y|max) / sigma =: theta' sigma-units, so A_s moves by at most
//     dA = 2 theta' sqrt(D E) + (4 + D) u24 E + 4 u24 |nb|max + D theta'^2,    E = nb_s - A_s(y).
// Terms within 2^-30 of the largest carry the sum (the others add < M 2^-30 whatever their error); for
// those E <= |nb|max - (ref + log2(S / M)) + 30 =: Erel, everything on the right known after the loop.
// ex2.approx (2^-22), the 8 partial sums + tree ((M/8 + 3) u24) and the margin make
//     eps = 0.75 dA(Erel) + 1e-5 + 1e-8 M.
// Sums that overflowed, theta' >= 1e-3 (pools with sigma ~ 1e-7: the first windows) or eps >= 0.02 send
// the step to the exact fp64 evaluation (summix_lse_exact), as does a uniform that falls between the
// bounds (~3e-4 of the steps).  Terms flushed to zero (ftz) are covered by the absolute term M 2e-38 of
// the upper bound.  tests/test_bounds_model.py replays this arithmetic in numpy with every approximation
// pushed to the edge of its bound; MCGPU_EXACT_TESTS=1 forces the fp64 route (tests/test_gpu_audit.py).
template <int D> struct PointD { double v[D]; };

template <int D>
__device__ __noinline__ double summix_lse_exact(const PointD<D> x, const double2 *sPmh, const double *sPn, int M, const MathTables &T)
{
  double m = -INFINITY, s = 0.0;
  for (int k = 0; k < M; ++k) {
    double a = sPn[k];
#pragma unroll
    for (int i = 0; i < D; ++i) { const double2 mh = sPmh[k * D + i]; const double xm = mh.x - x.v[i]; a += xm * xm * mh.y; }
    if (a > m) { s = s * mc_exp(m - a, T) + 1.0; m = a; }
    else if (a > -INFINITY) s += mc_exp(a - m, T);
  }
  return m + mc_log(s, T);                             // no finite term: -inf + log 0 = -inf
}

// The finish of the bound above, shared by every kernel family: from the two sums sn = Sn and so = So, the level ref,
// max |x'| and max |x| over the parameters and the pool scalars (max |mu|, max 1/sigma, max |nb|) to cfac in [cf_lo,
// cf_hi]; false when the bound cannot settle the step.  ru and rn are the rounding terms cu = (ru + D) u24 and cn = rn
// |nb|max + ...: 4 and 2.4e-7 for sums taken relative to ref slot by slot, more where they are not (mh_coop.cuh).
__device__ __forceinline__ bool summix_cfac_bounds(float sn, float so, float ref, float xabs_n, float xabs_o, float mumax,
                                                   float isig, float nbmax, int M, int D, float ru, float rn,
                                                   float &cf_lo, float &cf_hi)
{
  const float th_n = 1.6e-7f * (mumax + xabs_n) * isig, th_o = 1.6e-7f * (mumax + xabs_o) * isig;
  const float lvl = nbmax - ref + lg2_approx((float)M) + 30.0f;
  const float En = fmaxf(lvl - lg2_approx(sn), 30.0f), Eo = fmaxf(lvl - lg2_approx(fmaxf(so, 1.0e-37f)), 30.0f);
  const float cD = (float)D, cu = (ru + cD) * 6.0e-8f, cn = rn * nbmax + 1.0e-5f + 1.0e-8f * (float)M;
  const float eps_n = 0.75f * (2.0f * th_n * sqrtf(cD * En) + cu * En + cD * th_n * th_n) + cn;
  const float eps_o = 0.75f * (2.0f * th_o * sqrtf(cD * Eo) + cu * Eo + cD * th_o * th_o) + cn;
  cf_lo = __fdividef(so * (1.0f - eps_o), sn * (1.0f + eps_n)) * (1.0f - 1.0e-6f);
  cf_hi = __fdividef(fmaf(so, 1.0f + eps_o, 2.0e-38f * (float)M), sn * (1.0f - eps_n)) * (1.0f + 1.0e-6f);
  return sn < 1.0e30f && so < 1.0e30f && sn > 0.5f &&          // overflow / NaN: exact path
         th_n < 1.0e-3f && th_o < 1.0e-3f && eps_n < 0.02f && eps_o < 0.02f;
}

template <int D>
__device__ __forceinline__ bool summix_bounds(const double (&xo)[D], const double (&xn)[D], int c, int M,
                                              const float4 *sPf, const float *sNb, const float *s_scal,
                                              float &cf_lo, float &cf_hi)
{
  constexpr int CH = 8;
  const int Mpad = (M + CH - 1) & ~(CH - 1);
  float xof[D], xnf[D], xabs_o = 0.0f, xabs_n = 0.0f;
  float2 xxo[D], xxn[D];
#pragma unroll
  for (int i = 0; i < D; ++i) {
    xof[i] = (float)xo[i]; xnf[i] = (float)xn[i];
    xabs_o = fmaxf(xabs_o, fabsf(xof[i])); xabs_n = fmaxf(xabs_n, fabsf(xnf[i]));
    xxo[i] = make_float2(xof[i], xof[i]); xxn[i] = make_float2(xnf[i], xnf[i]);
  }
  float ref = sNb[c];                                  // A_c(x'): the level both sums are taken relative to
#pragma unroll
  for (int i = 0; i < D; ++i) { const float2 f = pool_slot(sPf, D, c, i); const float y = fmaf(-f.y, xnf[i], f.x); ref = fmaf(-y, y, ref); }
  float Sn[4] = {0.0f, 0.0f, 0.0f, 0.0f}, So[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  for (int s0 = 0; s0 < Mpad; s0 += CH) {
#pragma unroll
    for (int q = 0; q < CH; q += 2) {                  // a slot pair: both points, both slots, in packed fp32 (pool_pair)
      const float2 base = make_float2(sNb[s0 + q] - ref, sNb[s0 + q + 1] - ref);
      const float2 an = pool_pair<D>(sPf, s0 + q, xxn, base), ao = pool_pair<D>(sPf, s0 + q, xxo, base);
      Sn[q & 3] += ex2_approx(an.x); So[q & 3] += ex2_approx(ao.x);
      Sn[(q + 1) & 3] += ex2_approx(an.y); So[(q + 1) & 3] += ex2_approx(ao.y);
    }
  }
  const float sn = (Sn[0] + Sn[1]) + (Sn[2] + Sn[3]), so = (So[0] + So[1]) + (So[2] + So[3]);
  // (the overflow test once more, ahead of the arithmetic: it keeps the step loop of this kernel two instructions shorter)
  if (!(sn < 1.0e30f) || !(so < 1.0e30f) || !(sn > 0.5f)) return false;
  return summix_cfac_bounds(sn, so, ref, xabs_n, xabs_o, s_scal[0], s_scal[1], s_scal[2], M, D, 4.0f, 2.4e-7f, cf_lo, cf_hi);
}

// u < exp(delta) cfac with cfac in [cf_lo, cf_hi]:  1 accept, 0 reject, -1 the bounds straddle u.
// Relative error of the fp32 exponential: (float)delta and the product with log2(e) 1.2e-5 at |delta| <= 80,
// ex2.approx 2.4e-7.
__device__ __forceinline__ int accept_test_bounded(double u, double delta, float cf_lo, float cf_hi)
{
  const float dc = fminf(fmaxf((float)delta, -80.0f), 80.0f);
  const double e = (double)ex2_approx(dc * 1.4426950408889634f);
  const double lo = (delta >= -80.0) ? e * (double)cf_lo * (1.0 - 2.0e-5) : 0.0;
  const double hi = (delta <= 80.0) ? e * (double)cf_hi * (1.0 + 2.0e-5) : INFINITY;
  if (u < lo) return 1;
  if (u >= hi) return 0;
  return -1;                                           // also the NaN path: both comparisons are false
}

// Stage the exchange pool [M][D][2] (mu, sigma^2) into shared memory as (mu, -1/(2 sigma^2)) pairs + sigma.
// With a peer-to-peer exchange the CTA first waits until the pool has arrived from every GPU.  Out of
// line: it runs once per launch from inside the step loop, whose register allocation it must not disturb.
// Returns false when a peer-to-peer wait has timed out (now or in an earlier launch): the caller stops stepping
// instead of sampling from an incomplete pool; the host reports MCGPU_EPEER at the next synchronize.
template <int D>
__device__ __noinline__ bool stage_pool(const double *pool_cur, int pool_m, const unsigned long long *arrivals,
                                        unsigned long long wait_target, int *xflag, unsigned long long *xstat,
                                        double2 *sPmh, double *sPs, float4 *sPf, float2 *sSf, double *sPn, float *sNb,
                                        float *s_scal, int Mpad, const MathTables T)
{
  if (wait_target) wait_arrivals(arrivals, wait_target, xflag, xstat);
  if (threadIdx.x < 3) s_scal[threadIdx.x] = 0.0f;
  if (threadIdx.x == 0) s_scal[3] = (wait_target && *reinterpret_cast<volatile int *>(xflag)) ? 1.0f : 0.0f;
  __syncthreads();
  if (s_scal[3] != 0.0f) return false;
  float mumax = 0.0f, isig = 0.0f;
  for (int i = threadIdx.x; i < Mpad * D; i += blockDim.x) {
    float *pf = reinterpret_cast<float *>(sPf + (i / D >> 1) * D + i % D) + (i / D & 1);   // slot pairs (pool_pair)
    if (i < pool_m * D) {
      const double m = pool_cur[i * 2], s2 = pool_cur[i * 2 + 1];
      const double h = -0.5 / s2, sd = sqrt(s2);       // sigma = sqrt(sig^2), mcpar.cc:346
      sPmh[i] = make_double2(m, h); sPs[i] = sd;
      const double g = sqrt(-h * 1.4426950408889634);   // sqrt(log2(e) / (2 sigma^2)): a_s log2(e) = -sum_i (g mu - g x)^2
      pf[0] = (float)(g * m); pf[2] = (float)g; sSf[i] = make_float2((float)sd, (float)m);
      mumax = fmaxf(mumax, __double2float_ru(fabs(m))); isig = fmaxf(isig, __double2float_ru(1.0 / sd));
    } else {                                           // padding: (mu - x)^2 overflows / is huge, a = -inf, Q = 0
      sPmh[i] = make_double2(1.0e300, -1.0); pf[0] = 1.0e18f; pf[2] = 0.0f; sSf[i] = make_float2(0.0f, 0.0f);
    }
  }
  // normalisation of the components (remote mode 1): n_s = -1/2 sum_i log sig2_si, and nb_s = n_s log2(e) in fp32
  float nbabs = 0.0f;
  for (int k = threadIdx.x; k < Mpad; k += blockDim.x) {
    double n = 0.0;
    if (k < pool_m) {
#pragma unroll
      for (int i = 0; i < D; ++i) n -= 0.5 * MC_LOG(pool_cur[(k * D + i) * 2 + 1]);
    }
    sPn[k] = n; sNb[k] = (float)(n * 1.4426950408889634);
    nbabs = fmaxf(nbabs, __double2float_ru(fabs(n * 1.4426950408889634)));
  }
  // max over the CTA (non-negative floats order like their bit patterns; NaN/inf sort above every
  // number, which makes theta fail its test and sends every candidate to the exact path)
  atomicMax(reinterpret_cast<int *>(&s_scal[0]), __float_as_int(mumax));
  atomicMax(reinterpret_cast<int *>(&s_scal[1]), __float_as_int(isig));
  atomicMax(reinterpret_cast<int *>(&s_scal[2]), __float_as_int(nbabs));
  __syncthreads();
  return true;
}

template <int LIK, int D, int RNGK, int PHASE>
__global__ void __launch_bounds__(128, (D <= 2 ? ((PHASE == PH_BURN || PHASE == PH_LOCAL) ? MCGPU_MINB_LOCAL : MCGPU_MINB) : 1))
mh_steps_kernel(const StepParams p)
{
  constexpr bool MAIN = PHASE != PH_BURN;
  constexpr bool SUMMIX = PHASE == PH_MIXED_SUM;                                  // remote mode 1
  constexpr bool MIXED = PHASE == PH_MIXED || PHASE == PH_MIXED_SUM;
  constexpr bool CAN_REMOTE = RNGK == RNG_PHILOX && MIXED;
  extern __shared__ __align__(16) double smem[];
  __shared__ unsigned char s_rank[4][32];               // per warp: lanes of the chains still in the remote loop
  __shared__ unsigned int s_stat[3];                    // remote chain-steps of this CTA, the candidates they tried, exact-path fallbacks
  __shared__ unsigned int s_itacc[128];                 // per chain: index of the accepted candidate of the current remote step
  // smem: math tables | [D*D] factor | [nsteps] 1/pwgt table | pool: mu, -1/(2 sig^2), sigma
  double *sT = smem + MCGPU_MATH_SMEM;
  double *sW = sT + D * D;
  double2 *sPmh = reinterpret_cast<double2*>(sW + ((p.nsteps + 1) & ~1));     // (mu, -1/(2 sig^2)) pairs, 16-byte aligned
  const int Mpad = (p.pool_m + 7) & ~7;
  double *sPs = reinterpret_cast<double*>(sPmh + Mpad * D);
  float4 *sPf = reinterpret_cast<float4*>(sPs + Mpad * D);                    // fp32 copy: (g mu, g), g = sqrt(log2(e)/(2 sig^2)), slot pairs
  float2 *sSf = reinterpret_cast<float2*>(sPf + Mpad / 2 * D);                //            (sigma, mu)
  double *sPn = reinterpret_cast<double*>(sSf + Mpad * D);                    // n_s = -1/2 sum_i log sig2_si (remote mode 1)
  float *sNb = reinterpret_cast<float*>(sPn + Mpad);                          // n_s log2(e)
  __shared__ float s_scal[4];                           // pool-wide max |mu|, max 1/sigma, max |nb| (error bounds of the fp32 pool tests)
  MathTables T;
#ifndef MCGPU_EXACT_TU
  T.exp_tab = smem; T.log_tab = smem + MCGPU_EXP_TAB; T.trig_tab = T.log_tab + 2 * MCGPU_LOG_TAB;
  stage_math_tables(smem);
#else
  T.exp_tab = T.log_tab = T.trig_tab = nullptr;
#endif

  if (MAIN && exchange_failed(p.xc)) return;
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = j < p.C;
  const long long jc = live ? j : p.C - 1;           // idle lanes shadow the last chain, never store
  const unsigned long long g = (unsigned long long)(p.chain0 + jc);
  const uint32_t glo = (uint32_t)g, ghi = (uint32_t)(g >> 32);
  const int lane = threadIdx.x & 31;
  const int leader = lane & ~(p.coin_group - 1);

  for (int i = threadIdx.x; i < D * D; i += blockDim.x) sT[i] = p.factor[i];
  if (CAN_REMOTE && threadIdx.x < 3) s_stat[threadIdx.x] = 0u;
  if (MAIN)
    for (int k = threadIdx.x; k < p.nsteps; k += blockDim.x) sW[k] = 1.0 / (double)(p.t0 + k + 1);
  __syncthreads();

  double x[D], mu[D], ps[D];
#pragma unroll
  for (int i = 0; i < D; ++i) x[i] = p.x[i * p.ld + jc];
  double ly = p.ly[jc];
  if (MAIN) {
#pragma unroll
    for (int i = 0; i < D; ++i) { mu[i] = p.mu[i * p.ld + jc]; ps[i] = p.ps[i * p.ld + jc]; }
  }
  unsigned int nacc = 0, nrem = 0;
  int tmod = MAIN ? p.t0 % p.thin : 0;                // t % thin without per-step divisions
  int tring = p.hist_ring0;                           // ring row of the next kept step

  // Stage the exchange pool into shared memory before the first step (with a peer-to-peer exchange this is
  // where the CTA waits for the peers' publications).  Measured alternatives that defer the staging to the
  // window's first remote step -- a barrier inside the step loop, or the loop split in two segments -- cost
  // 3-9 % of the kernel's throughput on every GPU and bought 3 % at 8 GPUs: profiles/r01_history.md.
  if constexpr (CAN_REMOTE) {
    if (p.t0 + p.nsteps > p.first_remote_t)
      if (!stage_pool<D>(p.pool_cur, p.pool_m, p.xc.arrivals, p.xc.wait_target, p.xc.xflag, p.xc.xstat, sPmh, sPs, sPf, sSf, sPn, sNb, s_scal, Mpad, T)) return;
  }
  for (int k = 0; k < p.nsteps; ++k) {
    const uint32_t step = p.step0 + (uint32_t)k;
    const int t = p.t0 + k;
    double u_acc;
    bool remote = false;
    long long zoff = 0;
    constexpr int NP = (D + 1) / 2;                   // normal pairs per proposal
    constexpr int ABLK = (2 * NP) / 4, AW = (2 * NP) % 4;   // accept uniform: word 2*NP of the local stream
    Words wacc;
    if (RNGK == RNG_PHILOX) {
      wacc = philox_d<D, true>(glo, ghi, step, (uint32_t)ABLK, p);
      u_acc = u32_mid(word_of(wacc, AW));
      if (MIXED) {
        if (p.plan_valid) remote = (p.plan_mask >> k) & 1u;   // job-wide coin, drawn by the host (launch-uniform)
        else if (t >= p.first_remote_t) {              // one coin per group: the leader's word 2*NP+1
          const uint32_t cw = __shfl_sync(0xffffffffu, word_of(wacc, AW + 1), leader);
          remote = !(u32_half(cw) <= p.pl);            // mcpar.cc:152
        }
      }
    } else {
      // reference stream offsets for an all-local run of ONE rank hosting the C chains
      const long long s = MAIN ? (long long)p.nburn_total + t : (long long)step;
      const long long ncoin = (MAIN && t >= p.sync) ? (long long)(t - p.sync + 1) : 0;
      const long long uoff = s * p.C + ncoin + jc;
      zoff = (s * p.C + jc) * D;
      bool bad = uoff >= p.nu || zoff + D > p.nz;
      u_acc = bad ? 2.0 : p.U[uoff];
      if (MAIN && t >= p.sync) {
        const double coin = p.U[s * p.C + ncoin - 1];
        if (!(coin <= p.pl)) bad = true;               // a remote step cannot be replayed here
      }
      if (bad) *p.overrun = 1;
    }

    double xt[D];
    double cfac = 1.0;
    int cpick = 0;                                     // component the accepted remote draw came from

    if constexpr (RNGK == RNG_PHILOX) {
      // ---- proposal generation: genLocal (mcpar.cc:302-312) and genRemote (:315-451) ----
      // Remote steps first run the reference's rejection loop: it tries candidate iterations
      // it = 0,1,2,... until one is accepted.  Candidates are independent counter-based draws that
      // do not depend on the chain's state, so the warp evaluates 32 of them per round, spread over
      // the chains still looping (finished chains' lanes help the stragglers), and each chain
      // keeps the INDEX of its first accepted candidate in iteration order -- the sequential
      // loop's outcome, without lock-step divergence.  Only decisions are needed here, so the
      // candidates are evaluated in fp32 under rigorous bounds (remote_candidate).
      unsigned rm = (CAN_REMOTE && !SUMMIX) ? __ballot_sync(0xffffffffu, remote && live) : 0u;
      const unsigned rm0 = rm;                          // the chains of this warp that take a remote step
      if constexpr (CAN_REMOTE && !SUMMIX) {
        bool pending = remote && live;
        uint32_t it_next = 0;                           // this chain's next candidate; once it is done, its accepted one
        // launch-uniform inputs of remote_candidate, read once per remote step instead of once per candidate
        const float mu_max = s_scal[0], isig_max = s_scal[1], eps0 = remote_eps0<D>(p.pool_m);
        const bool bounded = !p.exact_tests;
        // A lane only ever serves a pending chain, and pending lanes are live, so the chain of lane tgt is
        // chain0 + (j - lane) + tgt: its Philox counter needs no shuffle.
        const unsigned long long gwarp = (unsigned long long)(p.chain0 + (j - lane));
        unsigned char *const rank = s_rank[threadIdx.x >> 5];
        while (rm) {
          // schedule 32 candidates over the unfinished chains
          const int n = __popc(rm);
          const int kk = (int)(((unsigned)lane * c_recip[n]) >> 16), r = lane - kk * n;   // lane / n, lane % n
          const int my_r = __popc(rm & ((1u << lane) - 1u));      // rank of this lane's chain among the unfinished
          if (pending) rank[my_r] = (unsigned char)lane;
          __syncwarp();
          const int tgt = rank[r];                      // lane owning the r-th unfinished chain
          __syncwarp();
          const uint32_t it = __shfl_sync(0xffffffffu, it_next, tgt) + (uint32_t)kk;
          const unsigned long long gt = gwarp + (unsigned)tgt;
          const bool acc = remote_candidate<D, true>((uint32_t)gt, (uint32_t)(gt >> 32), step, MCGPU_SLOT_REMOTE | (it << 6), p,
                                                     sPf, sSf, sPmh, sPs, mu_max, isig_max, eps0, Mpad, bounded, T, &s_stat[2]);
          const unsigned accmask = __ballot_sync(0xffffffffu, acc);
          if (pending) {
            // lanes my_r, my_r+n, ... served this chain, in iteration order; the lowest accepting lane (if any)
            // holds the first accepted candidate: advance past the candidates before it, or past all of them
            const unsigned cm = c_stride_mask[n] << my_r, hit = accmask & cm;
            it_next += (uint32_t)__popc(cm & ((hit & (0u - hit)) - 1u));
            pending = !hit && it_next < (1u << 24) - 64u;              // or the slot space is exhausted (never in practice)
          }
          rm = __ballot_sync(0xffffffffu, pending);
        }
        if (rm0) s_itacc[threadIdx.x] = it_next;
      }
      // Materialise the proposal in fp64, once per step and with one copy of the Philox + Box-Muller
      // code for both kinds: a local step draws its normals from the chain's local stream and
      // applies x' = x + T z; a remote step re-draws its accepted candidate (same Philox blocks)
      // and applies x' = mu_c + sigma_c z.
      // Word stream: local pair q = words (2q, 2q+1); remote pair q = words (2+2q, 3+2q) behind the
      // pick / rejection-uniform words of block 0.
      {
        const bool rem = CAN_REMOTE && remote;
        uint32_t slot = 0;
        Words blk;
        if (rem) {                                      // remote mode 1 draws candidate 0 of the remote stream, once
          slot = SUMMIX ? MCGPU_SLOT_REMOTE : (MCGPU_SLOT_REMOTE | (s_itacc[threadIdx.x] << 6));
          blk = philox_d<D, true>(glo, ghi, step, slot, p);
          cpick = (int)__umulhi(blk.w0, (uint32_t)p.pool_m);
        } else if (ABLK == 0) blk = wacc;               // d = 2: the accept block also carries pair 0
        const int woff = rem ? 1 : 0;                   // in units of pairs
        // normals are consumed as they are produced (no z[D] array: registers at d = 16):
        // local  x'_i = x_i + sum_{q<=i} T[i][q] z_q, accumulated column by column, which adds
        //        the terms of every row in the same q = 0,1,.. order as the row-wise loop
        double xz[D];
#pragma unroll
        for (int i = 0; i < D; ++i) xz[i] = rem ? sPmh[cpick * D + i].x : x[i];
#pragma unroll
        for (int q = 0; q < NP; ++q) {
          const int qq = q + woff;                      // pair position in the stream
          if ((qq & 1) == 0 && !(qq == 0 && ABLK == 0 && !rem))
            blk = philox_d<D, true>(glo, ghi, step, slot + (uint32_t)(qq >> 1), p);
          const uint32_t wa = (qq & 1) ? blk.w2 : blk.w0, wb = (qq & 1) ? blk.w3 : blk.w1;
          double za, zb;
          normal_pair_t(wa, wb, za, zb, T);
          if (!rem) {
#pragma unroll
            for (int i = 2 * q; i < D; ++i) xz[i] += factor_at<D>(sT, i * D + 2 * q) * za;
#pragma unroll
            for (int i = 2 * q + 1; i < D; ++i) xz[i] += factor_at<D>(sT, i * D + 2 * q + 1) * zb;
          } else {
            xz[2 * q] += sPs[cpick * D + 2 * q] * za;                                   // DIAGONAL storage, :348-350
            if (2 * q + 1 < D) xz[2 * q + 1] += sPs[cpick * D + 2 * q + 1] * zb;
          }
        }
#pragma unroll
        for (int i = 0; i < D; ++i) xt[i] = xz[i];
      }
      if constexpr (CAN_REMOTE && !SUMMIX) {
        if (rm0) {                // statistics: remote chain-steps and the iterations the reference's
          unsigned wi = (rm0 >> lane) & 1u ? s_itacc[threadIdx.x] + 1u : 0u;   // loop (mcpar.cc:331-409) would have run for them
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) wi += __shfl_xor_sync(0xffffffffu, wi, o);
          if (lane == 0) { atomicAdd(&s_stat[0], (unsigned)__popc(rm0)); atomicAdd(&s_stat[1], wi); }
        }
        if (remote) {
          // cfac = max_i Q_i(x_old) / max_i Q_i(x'), mcpar.cc:412-439: both maxima in fp64, one pass over the pool
          double aold = -INFINITY, anew = -INFINITY;
          for (int s = 0; s < p.pool_m; ++s) {
            double a = 0.0, b = 0.0;
#pragma unroll
            for (int i = 0; i < D; ++i) {
              const double2 mh = sPmh[s * D + i];
              const double xm = mh.x - x[i], ym = mh.x - xt[i];
              a += xm * xm * mh.y; b += ym * ym * mh.y;
            }
            aold = a > aold ? a : aold; anew = b > anew ? b : anew;
          }
          double qmax = MC_EXP(anew);
          qmax = qmax > MCGPU_FPEPS ? qmax : MCGPU_FPEPS;              // qimax starts at FPEPS, :357
          cfac = MC_EXP(aold) / qmax;
        }
      }
    } else {
      // replayed streams: genLocal with the supplied normals
      double z[D + 1];
#pragma unroll
      for (int i = 0; i < D; ++i) z[i] = (zoff + D <= p.nz) ? p.Z[zoff + i] : 0.0;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        double acc = x[i];
#pragma unroll
        for (int q = 0; q <= i; ++q) acc += sT[i * D + q] * z[q];
        xt[i] = acc;
      }
    }

    const double lyt = Lik<LIK, D>::eval(xt, p, T);
    bool a;
    if constexpr (SUMMIX) {
      if (remote) {
        // remote mode 1:  u < exp(lyt - ly + log q(x) - log q(x')), decided from fp32 bounds on q(x)/q(x')
        // whenever they settle it
        float cf_lo = 0.0f, cf_hi = 0.0f;
        int dec = -1;
        if (!p.exact_tests && summix_bounds<D>(x, xt, cpick, p.pool_m, sPf, sNb, s_scal, cf_lo, cf_hi))
          dec = accept_test_bounded(u_acc, lyt - ly, cf_lo, cf_hi);
        if (dec < 0) {
          atomicAdd(&s_stat[2], 1u);                     // statistics: remote steps the fp32 bounds did not settle
          PointD<D> po, pn;
#pragma unroll
          for (int i = 0; i < D; ++i) { po.v[i] = x[i]; pn.v[i] = xt[i]; }
          const double lcf = summix_lse_exact<D>(po, sPmh, sPn, p.pool_m, T) - summix_lse_exact<D>(pn, sPmh, sPn, p.pool_m, T);
          dec = accept_exact(u_acc, (lyt - ly) + lcf, 1.0, T) ? 1 : 0;
        }
        a = dec != 0;
        nrem += live ? 1u : 0u;
      } else
        a = accept_test_local(u_acc, lyt - ly, T, p.exact_tests);             // mcpar.cc:167-169 with cfac = 1
    } else if constexpr (!CAN_REMOTE) {
      a = accept_test_local(u_acc, lyt - ly, T, p.exact_tests);               // mcpar.cc:67-69 / :167-169 with cfac = 1
    } else {
      a = remote ? accept_test(u_acc, lyt - ly, cfac, T, p.exact_tests)       // mcpar.cc:167-169
                 : accept_test_local(u_acc, lyt - ly, T, p.exact_tests);
    }
    if (a) {
      ly = lyt;
#pragma unroll
      for (int i = 0; i < D; ++i) x[i] = xt[i];
    }
    nacc += a ? 1u : 0u;

    if (MAIN) {
      if (p.hist && live && tmod == 0) {               // MCout::add, mcout.cc:129-145 (a ring of hist_cap kept steps)
        double *row = p.hist + ((long long)tring * p.C + j) * (D + 1);
#pragma unroll
        for (int i = 0; i < D; ++i) row[i] = x[i];
        row[D] = ly;
      }
      if (++tmod == p.thin) { tmod = 0; if (++tring == p.hist_cap) tring = 0; }
      const double pwgt = (double)(t + 1), winv = sW[k];
      const bool adopt = CAN_REMOTE && remote && a;    // mcpar.cc:190-197
#pragma unroll
      for (int i = 0; i < D; ++i) {
        if (adopt) {                                   // sigma -> sigma^2 round trip of :346,:447-448
          const double sd = sPs[cpick * D + i];
          mu[i] = sPmh[cpick * D + i].x;
          ps[i] = (sd * sd) * (pwgt - 1.0);
        }
        const double delta = x[i] - mu[i];
        mu[i] += delta * winv;
        ps[i] += delta * (x[i] - mu[i]);
      }
    }
  }

  if (live) {
#pragma unroll
    for (int i = 0; i < D; ++i) p.x[i * p.ld + j] = x[i];
    p.ly[j] = ly;
    if (MAIN) {
#pragma unroll
      for (int i = 0; i < D; ++i) { p.mu[i * p.ld + j] = mu[i]; p.ps[i * p.ld + j] = ps[i]; }
      // publish to the next exchange pool (musigall slot rule, mcpar.cc:205-208)
      const long long gg = p.chain0 + j;
      if (p.xc.pool_next && gg % p.xc.pool_stride == 0 && gg / p.xc.pool_stride < p.pool_m)
        publish_slot<D>(p.xc, gg / p.xc.pool_stride, D, 0, mu, ps, 1.0 / (double)(p.t0 + p.nsteps));
    }
  }
  // acceptance counters of this window
  unsigned int wacc = live ? nacc : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) wacc += __shfl_xor_sync(0xffffffffu, wacc, o);
  const unsigned int nlive = __popc(__ballot_sync(0xffffffffu, live));
  if (lane == 0) {
    atomicAdd(p.counts, (unsigned long long)wacc);
    atomicAdd(p.counts + 1, (unsigned long long)nlive * (unsigned long long)p.nsteps);
  }
  if constexpr (SUMMIX) {                              // one candidate per remote chain-step
    unsigned int wr = nrem;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wr += __shfl_xor_sync(0xffffffffu, wr, o);
    if (lane == 0 && wr) { atomicAdd(&s_stat[0], wr); atomicAdd(&s_stat[1], wr); }
  }
  if constexpr (CAN_REMOTE) {                          // main-phase statistics: counts[2] remote chain-steps, [3] candidates
    __syncthreads();
    if (threadIdx.x == 0 && s_stat[0]) {
      atomicAdd(p.counts + 2, (unsigned long long)s_stat[0]); atomicAdd(p.counts + 3, (unsigned long long)s_stat[1]);
      if (s_stat[2]) atomicAdd(p.counts + 6, (unsigned long long)s_stat[2]);
    }
  }
}

// CTA size of the step kernels (<= 128, the kernels' launch bound); MCGPU_BLOCK env overrides for tuning
int step_block()
{
  static int b = 0;
  if (!b) { const char *e = getenv("MCGPU_BLOCK"); b = e ? atoi(e) : 128; if (b != 32 && b != 64 && b != 128) b = 128; }
  return b;
}

// smem: the math tables, the [d*d] factor, the [nsteps] 1/pwgt table and, for the phases that can take a remote
// step, the pool: (mu, h) + sigma in fp64, (g mu, g) + (sigma, mu) in fp32 = 40 bytes per slot and parameter,
// + n_s (fp64) and nb_s (fp32) per slot
size_t steps_smem_bytes(int d, int nsteps, int pool_m, bool with_pool)
{
  const size_t mpad = (size_t)((pool_m + 7) & ~7);
  return sizeof(double) * ((size_t)MCGPU_MATH_SMEM + (size_t)d * d + (size_t)((nsteps + 1) & ~1) + (with_pool ? mpad * d * 5 + mpad * 2 : 0));
}

// The launch rule of mh_steps_kernel<LIK, d, RNG, phase>, for built-in likelihoods (mh_dispatch.inl) and
// thread-per-chain plugins (mcgpu_api.cu) alike: one thread per chain in CTAs of step_block() threads.
StepLaunch steps_launch(int d, long long C, int nsteps, int pool_m, int phase)
{
  StepLaunch s;
  const int block = step_block();
  s.block = (unsigned)block;
  s.grid = (unsigned)((C + block - 1) / block);
  s.smem = steps_smem_bytes(d, nsteps, pool_m, phase != PH_BURN && phase != PH_LOCAL);
  return s;
}

// Burn-in tuning, mcpar.cc:78-96, applied at a window boundary.
// counts = {accepted, tried} of the window just finished (already summed over
// engines when sharded); cum = cumulative pair since the last rescale.
static __global__ void tune_kernel(unsigned long long *counts, unsigned long long *cum, double *factor,
                                   int dd, double armin, double armax, double dfac, double ifac)
{
  __shared__ double s_f;
  if (threadIdx.x == 0) {
    cum[0] += counts[0]; cum[1] += counts[1];
    counts[0] = 0; counts[1] = 0;
    const double arate = (double)cum[0] / (double)cum[1];
    double f = 1.0;
    if (arate < armin) { f = dfac; cum[0] = cum[1] = 0; }
    else if (arate > armax) { f = ifac; cum[0] = cum[1] = 0; }
    s_f = f;
  }
  __syncthreads();
  const double f = s_f;
  if (f != 1.0)
    for (int i = threadIdx.x; i < dd; i += blockDim.x) factor[i] *= f;
}

// initial log-likelihoods L(nchain, pvals, lylast), mcpar.cc:53, on the SoA state
template <int LIK, int D>
__global__ void init_loglik_kernel(const StepParams p)
{
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= p.C) return;
  double x[D];
#pragma unroll
  for (int i = 0; i < D; ++i) x[i] = p.x[i * p.ld + j];
  MathTables T;
#ifndef MCGPU_EXACT_TU
  T.exp_tab = MCGPU_EXP_TABLE; T.log_tab = MCGPU_LOG_TABLE; T.trig_tab = MCGPU_TRIG_TABLE;   // global-memory tables
#else
  T.exp_tab = T.log_tab = T.trig_tab = nullptr;
#endif
  p.ly[j] = Lik<LIK, D>::eval(x, p, T);
}

#ifdef MCGPU_EXACT_TU
// ----------------------------------------------------------------------------
// generic (runtime d, runtime likelihood) batched evaluation on AoS data:
// VLFunc::operator()(npset, x, y) for chain j of a batch of npset
// ----------------------------------------------------------------------------

static __device__ double loglik_aos(const LikSpec &L, const double *x, int npset, int j)
{
  const int d = L.d;
  const double *xj = x + (size_t)j * d;
  switch (L.lik) {
  case MCGPU_ROSENBROCK1: {
    double y = 0.0;
    for (int i = 0; i + 1 < d; i += 2) {
      const double t1 = 1 - xj[i];
      const double t2 = xj[i + 1] - xj[i] * xj[i];
      y -= t1 * t1 + 100.0 * t2 * t2;
    }
    return y;
  }
  case MCGPU_ROSENBROCK2: {
    // rosenbrock.cc:25-41 runs over the FLAT batch: set j's last parameter pairs with
    // set j+1's first; the last set of the batch has d-1 terms
    double y = 0.0;
    const int last = (j == npset - 1) ? d - 1 : d;
    for (int i = 0; i < last; ++i) {
      const double t1 = 1 - xj[i];
      const double t2 = xj[i + 1] - xj[i] * xj[i];
      y -= t1 * t1 - 100.0 * t2 * t2;
    }
    return y;
  }
  case MCGPU_GAUSSIAN: {
    double y = 0.0;
    for (int k = 0; k < 2; ++k) { const double arg = xj[k] - L.lp[k]; y -= 0.5 * arg * arg * L.lp[2 + k]; }
    return y;
  }
  case MCGPU_DUALGAUSSIAN: {
    const double arg1 = 0.5 * (xj[0] * xj[0] + xj[1] * xj[1]);
    const double t2a = xj[0] - 5.0, t2b = xj[1] - 5.0;
    const double arg2 = 0.5 * (t2a * t2a + t2b * t2b);
    return log(L.lp[0] * exp(-arg1) + exp(-arg2));
  }
  case MCGPU_GAUSSMIX: {
    const int K = L.k;
    const double *mu = L.dev, *is2 = mu + (size_t)K * d, *lw = is2 + (size_t)K * d;
    double m = -INFINITY;
    for (int k = 0; k < K; ++k) {
      double q = 0.0;
      for (int i = 0; i < d; ++i) { const double xm = xj[i] - mu[k * d + i]; q += xm * xm * is2[k * d + i]; }
      const double a = lw[k] - 0.5 * q;
      m = a > m ? a : m;
    }
    double s = 0.0;
    for (int k = 0; k < K; ++k) {
      double q = 0.0;
      for (int i = 0; i < d; ++i) { const double xm = xj[i] - mu[k * d + i]; q += xm * xm * is2[k * d + i]; }
      s += exp(lw[k] - 0.5 * q - m);
    }
    return m + log(s);
  }
  }
  return 0.0;
}

static __global__ void loglik_aos_kernel(LikSpec L, const double *x, double *y, int npset)
{
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < npset) y[j] = loglik_aos(L, x, npset, j);
}

// ----------------------------------------------------------------------------
// Kernel 2: verification mode -- one CTA per emulated MPI rank
// ----------------------------------------------------------------------------

static __device__ __forceinline__ int block_excl_scan(int flag, int *s_warp, int &total)
{
  const unsigned int b = __ballot_sync(0xffffffffu, flag);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  const int within = __popc(b & ((1u << lane) - 1u));
  __syncthreads();
  if (lane == 0) s_warp[w] = __popc(b);
  __syncthreads();
  int before = 0; total = 0;
  for (int i = 0; i < nw; ++i) { const int c = s_warp[i]; if (i < w) before += c; total += c; }
  return before + within;
}

static __global__ void __launch_bounds__(1024)
mh_verify_kernel(const VerifyParams p)
{
  __shared__ int s_warp[32];
  __shared__ double s_scale;
  const int r = blockIdx.x, j = threadIdx.x, d = p.d, C = p.C, N = p.N;
  const bool live = j < C;
  const int nt = C * d;
  double *pv = p.pvals + (size_t)r * nt, *pt = p.ptrial + (size_t)r * nt;
  double *lyv = p.ly + (size_t)r * C;
  double *muv = p.mu + (size_t)r * nt, *sgv = p.sig + (size_t)r * nt, *psv = p.ps + (size_t)r * nt;
  double *mtv = p.mutrial + (size_t)r * nt, *stv = p.sigtrial + (size_t)r * nt;
  double *T = p.factor + (size_t)r * d * d;
  double *ms = p.musig + (size_t)r * 2 * N * d;
  const long long *so = p.soff + (size_t)r * 6;
  const double *Zr = p.Z + so[0]; const long long nz = so[1];
  const double *Ur = p.U + so[2]; const long long nu = so[3];
  const int *Ir = p.I + so[4];    const long long ni = so[5];
  long long iz = p.cursors[r * 3], iu = p.cursors[r * 3 + 1], ii = p.cursors[r * 3 + 2];
  unsigned long long nacc = p.counts[r * 2], ntry = p.counts[r * 2 + 1];
  int irate = p.irate[r];
  const int grank = p.rank0 + r;
  bool bad = false;
#define RDZ(k) ((k) < nz ? Zr[(k)] : (bad = true, 0.0))
#define RDU(k) ((k) < nu ? Ur[(k)] : (bad = true, 0.0))
#define RDI(k) ((k) < ni ? Ir[(k)] : (bad = true, 0))

  // the in-place all-gather of mcpar.cc:127-140: other ranks' slots come from the snapshot
  if (p.phase == 1 && p.refresh) {
    for (int q = j; q < 2 * N * d; q += blockDim.x) {
      const int owner = q / (2 * nt);
      if (owner != grank) ms[q] = p.snap_cur[q];
    }
  }
  __syncthreads();

  double mut[MCGPU_MAX_D], sgt[MCGPU_MAX_D], xt[MCGPU_MAX_D];
  unsigned long long racc = 0;

  for (int k = 0; k < p.nsteps; ++k) {
    const int isamp = p.s0 + k;
    bool remote = false;
    int iters = 0;
    double cfac = 1.0;
    if (p.phase == 1 && isamp >= p.sync) {             // mcpar.cc:142-146
      const double rnd = RDU(iu); iu += 1;
      remote = !(rnd <= p.pl);
    }
    if (!remote) {                                      // genLocal, mcpar.cc:302-312
      if (live) {
        for (int i = 0; i < d; ++i) {
          double acc = pv[j * d + i];
          for (int q = 0; q <= i; ++q) acc += T[i * d + q] * RDZ(iz + (long long)j * d + q);
          xt[i] = acc;
        }
      }
      iz += (long long)C * d;
    } else {                                            // genRemote, mcpar.cc:315-451
      int rjct = live ? 1 : 0;
      double qimax = 0.0;
      int any;
      do {
        ++iters;
        const int chn = live ? RDI(ii + j) : 0; ii += C;                  // :337
        int total;
        const int before = block_excl_scan(rjct, s_warp, total);
        if (rjct) {                                                       // :339-352
          for (int i = 0; i < d; ++i) {
            const int tix = 2 * (d * chn + i);
            mut[i] = ms[tix];
            sgt[i] = sqrt(ms[tix + 1]);
            xt[i] = mut[i] + sgt[i] * RDZ(iz + (long long)before * d + i);
          }
        }
        iz += (long long)total * d;
        double pacpt = 0.0;
        if (rjct) {                                                       // :355-398
          qimax = MCGPU_FPEPS; double qisum = MCGPU_FPEPS;
          for (int qi = 0; qi < N; ++qi) {
            double arg = 0.0;
            for (int i = 0; i < d; ++i) {
              const double xm = ms[2 * (qi * d + i)] - xt[i];
              arg += xm * xm / ms[2 * (qi * d + i) + 1];
            }
            const double gv = exp(-0.5 * arg);
            qisum += gv; qimax = gv > qimax ? gv : qimax;
          }
          pacpt = qimax / qisum;
        }
        const double u = live ? RDU(iu + j) : 1.0; iu += C;               // :401
        if (rjct && u < pacpt) {                                          // :405-440
          rjct = 0;
          cfac = 0.0;
          for (int qi = 0; qi < N; ++qi) {
            double arg = 0.0;
            for (int i = 0; i < d; ++i) {
              const double xm = ms[2 * (qi * d + i)] - pv[j * d + i];
              arg += xm * xm / ms[2 * (qi * d + i) + 1];
            }
            const double gv = exp(-0.5 * arg);
            cfac = gv > cfac ? gv : cfac;
          }
          cfac /= qimax;
        }
        any = __syncthreads_or(rjct);
      } while (any);
      if (live) for (int i = 0; i < d; ++i) { sgt[i] *= sgt[i]; mtv[j * d + i] = mut[i]; stv[j * d + i] = sgt[i]; }
    }
    if (live) for (int i = 0; i < d; ++i) pt[j * d + i] = xt[i];
    __syncthreads();
    double lyt = 0.0, u = 1.0;
    if (live) lyt = loglik_aos(p.L, pt, C, j);           // L(nchain,ptrial,lytrial) :60/:160
    if (live) u = RDU(iu + j);
    iu += C;                                             // :63/:163
    bool a = false;
    if (live) {
      double pac = exp(lyt - lyv[j]);                    // :67/:167
      if (p.phase == 1) pac *= cfac;
      a = u < pac;
      if (a) { lyv[j] = lyt; for (int i = 0; i < d; ++i) pv[j * d + i] = xt[i]; }
    }
    const int na = __syncthreads_count(a);
    nacc += na; ntry += C; racc += na;

    const int tix = p.trace_base + k;
    if (p.tr_accept && tix < p.trace_cap) {
      if (live) {
        const size_t o = ((size_t)r * p.trace_cap + tix) * C + j;
        p.tr_accept[o] = a; p.tr_trial_ly[o] = lyt; p.tr_cfac[o] = cfac;
        for (int i = 0; i < d; ++i) p.tr_trial_p[o * d + i] = xt[i];
      }
      if (j == 0) { p.tr_remote[(size_t)r * p.trace_cap + tix] = remote; p.tr_iters[(size_t)r * p.trace_cap + tix] = iters; }
    }

    if (p.phase == 0) {                                  // tuning, mcpar.cc:78-96
      if (isamp > irate) {
        const double arate = (double)nacc / (double)ntry;
        double f = 1.0;
        if (arate < p.armin) { f = p.dfac; nacc = ntry = 0; }
        else if (arate > p.armax) { f = p.ifac; nacc = ntry = 0; }
        if (f != 1.0) for (int i = j; i < d * d; i += blockDim.x) T[i] *= f;
        irate += 50;
      }
      __syncthreads();
    } else {
      if (j == 0 && remote) { atomicAdd(p.rstats, 1ull); atomicAdd(p.rstats + 1, (unsigned long long)iters); }
      if (live) {
        if (p.hist) {                                    // MCout::add
          double *row = p.hist + ((size_t)isamp * p.hist_chains + (size_t)r * C + j) * (d + 1);
          for (int i = 0; i < d; ++i) row[i] = pv[j * d + i];
          row[d] = lyv[j];
        }
        const double pwgt = (double)(isamp + 1), winv = 1.0 / pwgt;       // :186-187
        const bool adopt = remote && a;
        for (int i = 0; i < d; ++i) {                                      // :188-209
          const int ix = j * d + i;
          if (adopt) { muv[ix] = mtv[ix]; sgv[ix] = stv[ix]; psv[ix] = sgv[ix] * (pwgt - 1.0); }
          const double pvi = pv[ix];
          const double delta = pvi - muv[ix];
          muv[ix] += delta * winv;
          psv[ix] += delta * (pvi - muv[ix]);
          sgv[ix] = psv[ix] * winv;
          const size_t islot = 2 * ((size_t)grank * nt + ix);
          ms[islot] = muv[ix]; ms[islot + 1] = sgv[ix];
        }
      }
      __syncthreads();
    }
  }
  (void)s_scale;
  if (p.phase == 1 && p.publish && live)
    for (int i = 0; i < d; ++i) {
      const size_t islot = 2 * ((size_t)grank * nt + (size_t)j * d + i);
      p.snap_next[islot] = ms[islot]; p.snap_next[islot + 1] = ms[islot + 1];
    }
  if (j == 0) {
    p.cursors[r * 3] = iz; p.cursors[r * 3 + 1] = iu; p.cursors[r * 3 + 2] = ii;
    p.counts[r * 2] = nacc; p.counts[r * 2 + 1] = ntry;
    p.irate[r] = irate;
    if (p.phase == 1) { atomicAdd(p.rstats + 2, racc); atomicAdd(p.rstats + 3, (unsigned long long)C * p.nsteps); }
  }
  if (bad) *p.overrun = 1;
#undef RDZ
#undef RDU
#undef RDI
}
#endif  // MCGPU_EXACT_TU

}  // namespace MCGPU_NS
}  // namespace mcgpu
