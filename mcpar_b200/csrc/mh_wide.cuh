// mh_wide.cuh -- fused MH step kernel for d >= 8: D/2 lanes per chain, two parameters per lane,
// NCH chains per lane group.
//
// At d = 16..64 a thread-per-chain kernel needs 150-255 registers (x, x', mu, psum2 are 4d
// doubles) and runs at 2 warps per scheduler.  Here a chain is spread over L = D/2 lanes
// (d = 64: one lane group per warp; d = 16: four groups per warp); each lane owns two
// consecutive parameters of NCH chains, draws their Box-Muller pairs itself, and the lanes of
// a group meet only where the algorithm couples parameters:
//   * x' = x + T z for a non-diagonal factor (z staged in shared memory, T column-major),
//   * the likelihood (lane-local pair terms + a shuffle reduction for Rosenbrock1; for GaussMix
//     two mixture components per lane over the staged x'),
//   * the remote proposal's pool test (one pool slot per lane over the staged x').
// NCH > 1 exists for register-level reuse: the GaussMix / pool parameters stream through L1
// (64 KB per evaluation at d = 64, K = 64), and at one chain per group the kernel is bound by
// L1 bandwidth; with NCH chains per group every loaded (mu, 1/s2) pair serves NCH chains.
//
// Same reference lines as mh_steps_kernel: genLocal mcpar.cc:302-312, genRemote :315-451,
// accept :165-175, moments :186-209, MCout::add mcout.cc:129-145.  Job-wide coin only
// (phases PH_BURN / PH_LOCAL / PH_REMOTE are launch-uniform).  Production (Philox) unit only.
#pragma once

namespace mcgpu {
namespace MCGPU_NS {

#ifndef MCGPU_WIDE_UNROLL
#define MCGPU_WIDE_UNROLL 4
#endif
constexpr int kWideUnroll = MCGPU_WIDE_UNROLL;   // inner-loop unroll of the streamed-parameter loops

template <int L>
__device__ __forceinline__ double group_sum(double v)
{
#pragma unroll
  for (int o = L / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int L>
__device__ __forceinline__ double group_max(double v)
{
#pragma unroll
  for (int o = L / 2; o > 0; o >>= 1) { const double w = __shfl_xor_sync(0xffffffffu, v, o); v = w > v ? w : v; }
  return v;
}
template <int L>
__device__ __forceinline__ float group_sumf(float v)
{
#pragma unroll
  for (int o = L / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int L>
__device__ __forceinline__ float group_maxf(float v)
{
#pragma unroll
  for (int o = L / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// the same for fp32 staging (remote mode 1: the pool test runs in fp32)
template <int NCH>
__device__ __forceinline__ void load_staged_f(const float *s, float (&v)[NCH])
{
  if (NCH % 4 == 0) {
#pragma unroll
    for (int c = 0; c < NCH; c += 4) { const float4 t = *reinterpret_cast<const float4 *>(s + c); v[c] = t.x; v[c + 1] = t.y; v[c + 2] = t.z; v[c + 3] = t.w; }
  } else if (NCH % 2 == 0) {
#pragma unroll
    for (int c = 0; c < NCH; c += 2) { const float2 t = *reinterpret_cast<const float2 *>(s + c); v[c] = t.x; v[c + 1] = t.y; }
  } else {
#pragma unroll
    for (int c = 0; c < NCH; ++c) v[c] = s[c];
  }
}

// the NCH staged values of one parameter (16-byte aligned when NCH is even): LDS.128 where possible
template <int NCH>
__device__ __forceinline__ void load_staged(const double *s, double (&v)[NCH])
{
  if (NCH % 2 == 0) {
#pragma unroll
    for (int c = 0; c < NCH; c += 2) { const double2 t = *reinterpret_cast<const double2 *>(s + c); v[c] = t.x; v[c + 1] = t.y; }
  } else {
#pragma unroll
    for (int c = 0; c < NCH; ++c) v[c] = s[c];
  }
}

// A wide device likelihood plugin (LIK = MCGPU_DEVICE_PLUGIN): partial(x, xs, p, part) is share `part` of the
// log-likelihood at the point x[i * xs].  Declared only: mh_plugin.cu specialises it around the user's
// UserLik::partial (include/mcgpu_plugin.cuh).
template <int LIK, int D> struct WideLik;

// log-likelihoods of the group's NCH chains; their points are staged in sx[i*NCH + c] and held
// as (x0[c], x1[c]) per lane.  Every lane of the group returns the same values.
template <int LIK, int D, int NCH>
__device__ __forceinline__ void wide_loglik(const double (&x0)[NCH], const double (&x1)[NCH], const double *sx, int r,
                                            const WideParams &p, const MathTables &T, double (&out)[NCH])
{
  constexpr int L = D / 2;
  if constexpr (LIK == MCGPU_ROSENBROCK1) {     // rosenbrock.cc:4-21: the pair (2r, 2r+1) lives in lane r
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const double t1 = 1 - x0[c];
      const double t2 = x1[c] - x0[c] * x0[c];
      out[c] = -group_sum<L>(t1 * t1 + 100.0 * t2 * t2);
    }
  } else if constexpr (LIK == MCGPU_DEVICE_PLUGIN) {   // lane r returns share r; the butterfly order fixes the sum
#pragma unroll
    for (int c = 0; c < NCH; ++c) out[c] = group_sum<L>(WideLik<LIK, D>::partial(sx + c, NCH, p, r));
  } else {
    // GaussMix: lane r evaluates components r, r+L, ... two at a time (kpad is a multiple of 2L;
    // padding components carry c = -inf).  The exponent is expanded once on the host,
    //     log w_k - 1/2 sum_i (x_i - mu_ki)^2 / s2_ki = c_k + sum_i x_i (a_ki x_i + b_ki),
    //     a = -1/(2 s2), b = mu / s2, c = log w - 1/2 sum_i mu^2 / s2,
    // so a (component, parameter, chain) costs two DFMA instead of DADD + DMUL + DFMA (the terms reach
    // ~50 per parameter against a sum of ~ -d/2: ~1e-13 absolute on the log-likelihood at d = 64).  One pointer
    // walks a component's (a, b) pairs down the parameters; the partner component sits L pairs further.
    double m[NCH], s[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) { m[c] = -INFINITY; s[c] = 0.0; }
    for (int k = r; k < p.kpad; k += 2 * L) {
      const double2 *g = p.gm2 + k;
      double q0[NCH], q1[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) { q0[c] = 0.0; q1[c] = 0.0; }
#pragma unroll kWideUnroll
      for (int i = 0; i < D; ++i) {
        const double2 a = __ldg(g), b = __ldg(g + L);
        g += p.kpad;
        double xi[NCH];
        load_staged<NCH>(sx + i * NCH, xi);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          q0[c] = fma(fma(a.x, xi[c], a.y), xi[c], q0[c]);
          q1[c] = fma(fma(b.x, xi[c], b.y), xi[c], q1[c]);
        }
      }
      const double lw0 = __ldg(p.gm_lw + k), lw1 = __ldg(p.gm_lw + k + L);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const double a0 = lw0 + q0[c], a1 = lw1 + q1[c];
        if (a0 > m[c]) { s[c] = s[c] * mc_exp(m[c] - a0, T) + 1.0; m[c] = a0; } else if (a0 > -INFINITY) s[c] += mc_exp(a0 - m[c], T);
        if (a1 > m[c]) { s[c] = s[c] * mc_exp(m[c] - a1, T) + 1.0; m[c] = a1; } else if (a1 > -INFINITY) s[c] += mc_exp(a1 - m[c], T);
      }
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const double gm = group_max<L>(m[c]);
      const double tot = group_sum<L>(s[c] * mc_exp(m[c] - gm, T));
      out[c] = gm + mc_log(tot, T);
    }
  }
}

// For the NCH points staged in sx: amax[c] = max_s log Q_s (exact fp64) and S[c] = fp32 bound
// material sum_s exp(log Q_s - amax[c]).  Lane r evaluates pool slots r, r+L, ...
// NORM: the components are normalised, log Q_s = n_s - 1/2 sum_i (mu - x)^2 / sig2 (remote mode 1).
template <int D, int NCH, bool NORM>
__device__ __forceinline__ void wide_pool_eval(const double *sx, int r, const WideParams &p, double (&amax)[NCH], float (&S)[NCH])
{
  constexpr int L = D / 2;
  constexpr float L2E = 1.4426950408889634f;
  double m[NCH]; float sl[NCH];
#pragma unroll
  for (int c = 0; c < NCH; ++c) { m[c] = -INFINITY; sl[c] = 0.0f; }
  for (int s = r; s < p.mpad; s += L) {
    double a[NCH];
    const double n0 = NORM ? __ldg(p.pnb + s) : 0.0;
#pragma unroll
    for (int c = 0; c < NCH; ++c) a[c] = n0;
    const double2 *g = p.pmh + s;
#pragma unroll 4
    for (int i = 0; i < D; ++i) {
      const double2 mh = __ldg(g);
      g += p.mpad;
      double xi[NCH];
      load_staged<NCH>(sx + i * NCH, xi);
#pragma unroll
      for (int c = 0; c < NCH; ++c) { const double xm = mh.x - xi[c]; a[c] += xm * xm * mh.y; }
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const bool gt = a[c] > m[c];
      // a = -inf (a padding slot, or a point hopelessly far away) contributes 0; without the guard the first
      // such slot of a lane (m still -inf) would make a - m NaN and poison the group's sum
      const float e = a[c] == -INFINITY ? 0.0f : ex2_approx(-fabsf((float)(a[c] - m[c])) * L2E);
      sl[c] = gt ? fmaf(sl[c], e, 1.0f) : sl[c] + e;
      m[c] = gt ? a[c] : m[c];
    }
  }
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    amax[c] = group_max<L>(m[c]);
    S[c] = group_sumf<L>(m[c] == -INFINITY ? 0.0f : sl[c] * ex2_approx((float)(m[c] - amax[c]) * L2E));   // a lane that saw no live slot adds 0
  }
}

// Remote mode 1, fast path: bounds on q(x)/q(x') for the group's NCH chains from an fp32 evaluation of both
// mixtures in ONE pass over the pool (summix_bounds of mh_kernels.cuh, spread over the group's lanes: lane r
// takes pool slots r, r+L, ...; same error analysis with D parameters per term).  sf holds the fp32 points,
// [0][D][NCH] = x', [1][D][NCH] = x.  The fp32 copy of the pool (8 bytes per slot and parameter: 131 KB at
// M = 256, d = 64) stays in L1, where the fp64 pairs (262 KB) streamed from L2 for every group.
template <int D, int NCH>
__device__ __forceinline__ void wide_summix_bounds(const float *sf, int r, const int (&cpick)[NCH], const WideParams &p,
                                                   float (&cf_lo)[NCH], float (&cf_hi)[NCH], bool (&ok)[NCH])
{
  constexpr int L = D / 2;
  const int i0 = 2 * r;
  const float *sn = sf, *so = sf + D * NCH;
  float ref[NCH], xabs_n[NCH], xabs_o[NCH];
#pragma unroll
  for (int c = 0; c < NCH; ++c) {                    // level of both sums: the picked component's exponent at x'
    const float2 f0 = __ldg(p.pf + (size_t)i0 * p.mpad + cpick[c]), f1 = __ldg(p.pf + (size_t)(i0 + 1) * p.mpad + cpick[c]);
    const float xn0 = sn[i0 * NCH + c], xn1 = sn[(i0 + 1) * NCH + c], xo0 = so[i0 * NCH + c], xo1 = so[(i0 + 1) * NCH + c];
    const float y0 = fmaf(-f0.y, xn0, f0.x), y1 = fmaf(-f1.y, xn1, f1.x);
    ref[c] = __ldg(p.pnbf + cpick[c]) - group_sumf<L>(fmaf(y0, y0, y1 * y1));
    xabs_n[c] = group_maxf<L>(fmaxf(fabsf(xn0), fabsf(xn1)));
    xabs_o[c] = group_maxf<L>(fmaxf(fabsf(xo0), fabsf(xo1)));
  }
  float Sn[NCH], So[NCH];
#pragma unroll
  for (int c = 0; c < NCH; ++c) { Sn[c] = 0.0f; So[c] = 0.0f; }
  for (int s = r; s < p.mpad; s += L) {
    const float nb = __ldg(p.pnbf + s);
    float an[NCH], ao[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) { an[c] = nb - ref[c]; ao[c] = an[c]; }
    const float2 *g = p.pf + s;
#pragma unroll 4
    for (int i = 0; i < D; ++i) {
      const float2 f = __ldg(g);
      g += p.mpad;
      float xn[NCH], xo[NCH];
      load_staged_f<NCH>(sn + i * NCH, xn);
      load_staged_f<NCH>(so + i * NCH, xo);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const float yn = fmaf(-f.y, xn[c], f.x), yo = fmaf(-f.y, xo[c], f.x);
        an[c] = fmaf(-yn, yn, an[c]); ao[c] = fmaf(-yo, yo, ao[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) { Sn[c] += ex2_approx(an[c]); So[c] += ex2_approx(ao[c]); }
  }
  const float mumax = __ldg(p.pscal), isig = __ldg(p.pscal + 1), nbmax = __ldg(p.pscal + 2);
#pragma unroll
  for (int c = 0; c < NCH; ++c)
    ok[c] = summix_cfac_bounds(group_sumf<L>(Sn[c]), group_sumf<L>(So[c]), ref[c], xabs_n[c], xabs_o[c], mumax, isig, nbmax,
                               p.pool_m, D, 4.0f, 2.4e-7f, cf_lo[c], cf_hi[c]);
}

// exact log of the normalised sum-mixture at chain c's staged point (remote mode 1, rare path)
// (the out-of-line rare paths take the few fields they need BY VALUE: a reference to the kernel's parameter struct would
// force every thread to copy all of it -- 520 bytes -- from the constant bank to its stack at kernel entry)
template <int D, int NCH>
__device__ __noinline__ double wide_pool_lse_exact(const double *sx, int c, int r, const double2 *pmh, const double *pnb, int pool_m, int mpad,
                                                   const MathTables T)
{
  constexpr int L = D / 2;
  double m = -INFINITY, sm = 0.0;
  for (int s = r; s < pool_m; s += L) {
    double a = __ldg(pnb + s);
    const double2 *g = pmh + s;
    for (int i = 0; i < D; ++i) {
      const double2 mh = __ldg(g);
      g += mpad;
      const double xm = mh.x - sx[i * NCH + c];
      a += xm * xm * mh.y;
    }
    if (a > m) { sm = sm * mc_exp(m - a, T) + 1.0; m = a; }
    else if (a > -INFINITY) sm += mc_exp(a - m, T);
  }
  const double gm = group_max<L>(m);
  const double tot = group_sum<L>(m == -INFINITY ? 0.0 : sm * mc_exp(m - gm, T));
  return gm + mc_log(tot, T);
}

// exact pacpt material for chain c of the staged points (rare path)
template <int D, int NCH>
__device__ __noinline__ double2 wide_pool_exact_sum(const double *sx, int c, int r, const double2 *pmh, int pool_m, int mpad, const MathTables T)
{
  constexpr int L = D / 2;
  double qs = 0.0, qm = 0.0;
  for (int s = r; s < pool_m; s += L) {
    double a = 0.0;
    const double2 *g = pmh + s;
    for (int i = 0; i < D; ++i) {
      const double2 mh = __ldg(g);
      g += mpad;
      const double xm = mh.x - sx[i * NCH + c];
      a += xm * xm * mh.y;
    }
    const double gv = mc_exp(a, T);
    qs += gv; qm = gv > qm ? gv : qm;
  }
  return make_double2(group_sum<L>(qs), group_max<L>(qm));      // (sum, max)
}

// chains per lane group: register-level reuse of the streamed GaussMix / pool parameters
#ifndef MCGPU_WIDE_NCH64
#define MCGPU_WIDE_NCH64 4
#endif
constexpr int wide_nch(int d) { return d >= 64 ? MCGPU_WIDE_NCH64 : (d >= 32 ? 2 : 1); }
template <int D> struct WideNch { static constexpr int value = wide_nch(D); };

// The launch rule of mh_wide_kernel<LIK, d, WideNch<d>, PHASE>, for built-in likelihoods (mh_fast.cu) and wide
// plugins (mcgpu_api.cu) alike: 128 threads, 128 / L lane groups per CTA, NCH chains per group, and in shared
// memory the math tables plus each group's staged points sx[d][NCH] and normals sz[d][NCH].
WideLaunch wide_launch(int d, long long C)
{
  const int L = d / 2, block = 128, gpb = block / L;
  WideLaunch w;
  w.nch = wide_nch(d); w.block = block;
  w.grid = (unsigned)((C + gpb * w.nch - 1) / (gpb * w.nch));
  w.smem = sizeof(double) * ((size_t)MCGPU_MATH_SMEM + (size_t)gpb * 2 * d * w.nch);
  return w;
}

#ifndef MCGPU_WIDE_MINB
#define MCGPU_WIDE_MINB 3       // d >= 32: <= 170 registers, 12 warps per SM (gpurun_out/tune_wide.log)
#endif
#ifndef MCGPU_WIDE_MINB_SMALL
#define MCGPU_WIDE_MINB_SMALL 6 // d <= 16: <= 80 registers, 24 warps per SM (+16 % local, +6 % sum-mixture over 4: profiles/r02_tuning.md)
#endif
template <int LIK, int D, int NCH, int PHASE>
__global__ void __launch_bounds__(128, (D >= 32 ? MCGPU_WIDE_MINB : MCGPU_WIDE_MINB_SMALL))
mh_wide_kernel(const WideParams p)
{
  constexpr int L = D / 2;                      // lanes per group
  constexpr bool MAIN = PHASE != PH_BURN;
  constexpr bool SUMMIX = PHASE == PH_REMOTE_SUM;                         // remote mode 1 (mh_kernels.cuh)
  constexpr bool REMOTE = PHASE == PH_REMOTE || PHASE == PH_REMOTE_SUM;
  constexpr int ABLK = (2 * L) / 4, AW = (2 * L) % 4;     // accept uniform: word 2*NP (NP = L pairs) of the local stream
  extern __shared__ __align__(16) double smem[];
  // smem: math tables | per group of the CTA: staged points sx[D][NCH] and staged normals sz[D][NCH]
  MathTables T;
  T.exp_tab = smem; T.log_tab = smem + MCGPU_EXP_TAB; T.trig_tab = T.log_tab + 2 * MCGPU_LOG_TAB;
  stage_math_tables(smem);
  if (exchange_failed(p.xc)) return;
  const int gib = threadIdx.x / L;              // group within the CTA
  double *sx = smem + MCGPU_MATH_SMEM + (size_t)gib * 2 * D * NCH;
  double *sz = sx + D * NCH;
  __syncthreads();

  const int r = threadIdx.x % L;                // lane within the group: owns parameters 2r, 2r+1
  const int i0 = 2 * r;
  const long long jb = ((long long)blockIdx.x * (blockDim.x / L) + gib) * NCH;
  long long jc[NCH]; bool live[NCH]; uint32_t glo[NCH], ghi[NCH];
  double x0[NCH], x1[NCH], ly[NCH], mu0[NCH], mu1[NCH], ps0[NCH], ps1[NCH];
  unsigned int nacc[NCH], nit = 0, nfb = 0;       // accepted steps; candidate iterations of the remote steps; exact-path fallbacks
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    live[c] = jb + c < p.C;
    jc[c] = live[c] ? jb + c : p.C - 1;          // idle slots shadow the last chain, never store
    const unsigned long long g = (unsigned long long)(p.chain0 + jc[c]);
    glo[c] = (uint32_t)g; ghi[c] = (uint32_t)(g >> 32);
    x0[c] = p.x[jc[c] * D + i0]; x1[c] = p.x[jc[c] * D + i0 + 1];
    ly[c] = p.ly[jc[c]];
    mu0[c] = mu1[c] = ps0[c] = ps1[c] = 0.0;
    if (MAIN) { mu0[c] = p.mu[jc[c] * D + i0]; mu1[c] = p.mu[jc[c] * D + i0 + 1]; ps0[c] = p.ps[jc[c] * D + i0]; ps1[c] = p.ps[jc[c] * D + i0 + 1]; }
    nacc[c] = 0;
  }
  const double tdiag0 = p.factor_rm[i0 * D + i0], tdiag1 = p.factor_rm[(i0 + 1) * D + i0 + 1];
  const bool diag = *p.diagonal != 0;
  int tmod = MAIN ? p.t0 % p.thin : 0;
  int tring = p.hist_ring0;                     // ring row of the next kept step

  for (int k = 0; k < p.nsteps; ++k) {
    const uint32_t step = p.step0 + (uint32_t)k;
    const int t = p.t0 + k;
    double u_acc[NCH], xt0[NCH], xt1[NCH], cfac[NCH];
    int cpick[NCH];
    float cf_lo[NCH], cf_hi[NCH]; bool cf_ok[NCH];  // remote mode 1: fp32 bounds on q(x)/q(x')
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const Words wacc = philox4x32_10_rk(glo[c], ghi[c], step, (uint32_t)ABLK, p.rk);
      u_acc[c] = u32_mid(word_of(wacc, AW));
      cfac[c] = 1.0; cpick[c] = 0; xt0[c] = x0[c]; xt1[c] = x1[c];
    }

    if (!REMOTE) {
      // genLocal: lane r's Box-Muller pair = words (2r, 2r+1) of the chain's local stream
      double za[NCH], zb[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const Words b = philox4x32_10_rk(glo[c], ghi[c], step, (uint32_t)(r >> 1), p.rk);
        normal_pair_t((r & 1) ? b.w2 : b.w0, (r & 1) ? b.w3 : b.w1, za[c], zb[c], T);
      }
      if (diag) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) { xt0[c] = x0[c] + tdiag0 * za[c]; xt1[c] = x1[c] + tdiag1 * zb[c]; }
      } else {
#pragma unroll
        for (int c = 0; c < NCH; ++c) { sz[i0 * NCH + c] = za[c]; sz[(i0 + 1) * NCH + c] = zb[c]; }
        __syncwarp();
        double a0[NCH], a1[NCH];                  // rows 2r and 2r+1, terms added in q = 0,1,.. order
#pragma unroll
        for (int c = 0; c < NCH; ++c) { a0[c] = x0[c]; a1[c] = x1[c]; }
        for (int q = 0; q <= i0; ++q) {
          const double t0 = __ldg(p.factor_cm + q * D + i0), t1 = __ldg(p.factor_cm + q * D + i0 + 1);
#pragma unroll
          for (int c = 0; c < NCH; ++c) { const double zq = sz[q * NCH + c]; a0[c] += t0 * zq; a1[c] += t1 * zq; }
        }
        const double tl = __ldg(p.factor_cm + (i0 + 1) * D + i0 + 1);
#pragma unroll
        for (int c = 0; c < NCH; ++c) { xt0[c] = a0[c]; xt1[c] = a1[c] + tl * zb[c]; }
        __syncwarp();
      }
    } else if (SUMMIX) {
      // remote mode 1 (sum-mixture proposal, no rejection loop): candidate 0 of the remote stream is THE
      // proposal; lane r tests pool slots r, r+L, ... against x' and against x for all NCH chains
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const Words w0 = philox4x32_10_rk(glo[c], ghi[c], step, MCGPU_SLOT_REMOTE, p.rk);
        cpick[c] = (int)__umulhi(w0.w0, (uint32_t)p.pool_m);
        const int qq = r + 1;                       // lane r's pair = words (2+2r, 3+2r)
        Words b = w0;
        if ((qq >> 1) != 0) b = philox4x32_10_rk(glo[c], ghi[c], step, MCGPU_SLOT_REMOTE + (uint32_t)(qq >> 1), p.rk);
        double za, zb;
        normal_pair_t((qq & 1) ? b.w2 : b.w0, (qq & 1) ? b.w3 : b.w1, za, zb, T);
        xt0[c] = __ldg(p.pmh + (size_t)i0 * p.mpad + cpick[c]).x + __ldg(p.psd + (size_t)i0 * p.mpad + cpick[c]) * za;
        xt1[c] = __ldg(p.pmh + (size_t)(i0 + 1) * p.mpad + cpick[c]).x + __ldg(p.psd + (size_t)(i0 + 1) * p.mpad + cpick[c]) * zb;
      }
      // both points in fp32 in the normals' staging area (unused in a remote step): [0] = x', [1] = x
      float *sf = reinterpret_cast<float *>(sz);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        sf[i0 * NCH + c] = (float)xt0[c]; sf[(i0 + 1) * NCH + c] = (float)xt1[c];
        sf[D * NCH + i0 * NCH + c] = (float)x0[c]; sf[D * NCH + (i0 + 1) * NCH + c] = (float)x1[c];
        nit += live[c] ? 1u : 0u;
      }
      __syncwarp();
      wide_summix_bounds<D, NCH>(sf, r, cpick, p, cf_lo, cf_hi, cf_ok);
      if (p.exact_tests) {                            // audit mode: every Hastings factor in fp64
#pragma unroll
        for (int c = 0; c < NCH; ++c) cf_ok[c] = false;
      }
      __syncwarp();
    } else {
      // genRemote: the group's chains run the reference's rejection loop in step: candidate
      // iteration `it` of every chain is evaluated together (lane r tests pool slots r, r+L, ...
      // against all NCH candidates), each chain keeps its first accepted candidate, and the
      // loop is warp-uniform: chains that are done keep evaluating (discarded) candidates until
      // the warp's last chain is done, so every warp-wide primitive is reached by all lanes.
      double amax_acc[NCH];
      bool done[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) { done[c] = false; amax_acc[c] = 0.0; }
      for (uint32_t it = 0;; ++it) {
        const uint32_t slot = MCGPU_SLOT_REMOTE | (it << 6);
        double c0[NCH], c1[NCH], u[NCH]; int cc[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const Words w0 = philox4x32_10_rk(glo[c], ghi[c], step, slot, p.rk);   // same block in every lane of the group
          cc[c] = (int)__umulhi(w0.w0, (uint32_t)p.pool_m);                              // viRngUniform, mcpar.cc:337
          u[c] = u32_mid(w0.w1);                                                         // vsRngUniform, mcpar.cc:401
          const int qq = r + 1;                     // lane r's pair = words (2+2r, 3+2r) of the candidate's stream
          Words b = w0;
          if ((qq >> 1) != 0) b = philox4x32_10_rk(glo[c], ghi[c], step, slot + (uint32_t)(qq >> 1), p.rk);
          double za, zb;
          normal_pair_t((qq & 1) ? b.w2 : b.w0, (qq & 1) ? b.w3 : b.w1, za, zb, T);
          c0[c] = __ldg(p.pmh + (size_t)i0 * p.mpad + cc[c]).x + __ldg(p.psd + (size_t)i0 * p.mpad + cc[c]) * za;   // DIAGONAL storage, :348-350
          c1[c] = __ldg(p.pmh + (size_t)(i0 + 1) * p.mpad + cc[c]).x + __ldg(p.psd + (size_t)(i0 + 1) * p.mpad + cc[c]) * zb;
          sx[i0 * NCH + c] = c0[c]; sx[(i0 + 1) * NCH + c] = c1[c];
        }
        __syncwarp();
        double am[NCH]; float S[NCH];
        wide_pool_eval<D, NCH, false>(sx, r, p, am, S);
        bool acc[NCH], decided[NCH], alldec = true;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          acc[c] = false; decided[c] = false;
          {
            // pacpt = qimax / qisum with the reference's FPEPS offsets (qimax = max(FPEPS, max Q), qisum = FPEPS +
            // sum Q, mcpar.cc:357-358, :397): at d >= 16 the largest Q at a candidate is e^(-d/2) ~ FPEPS, so the
            // offsets are part of the ratio.  max Q = exp(am) in fp64 (am is exact); the sum is max Q * S with S
            // right to eps (fp32: float conversion of the exponents, ex2.approx, <= M/L rescales).
            const double eps = 1.0e-4 + 2.0e-5 * (double)p.pool_m, Sd = (double)S[c];
            const double qm = mc_exp(am[c], T), num = qm > MCGPU_FPEPS ? qm : MCGPU_FPEPS;
            if (p.exact_tests) { }                      // audit mode: every rejection test in fp64 (below)
            else if (u[c] * (MCGPU_FPEPS + qm * Sd * (1.0 + eps)) < num * (1.0 - 1.0e-13)) { acc[c] = true; decided[c] = true; }
            else if (u[c] * (MCGPU_FPEPS + qm * Sd * (1.0 - eps)) >= num * (1.0 + 1.0e-13)) { decided[c] = true; }
          }
          alldec = alldec && (decided[c] || done[c]);
        }
        if (!__all_sync(0xffffffffu, alldec)) {        // rare: exact pacpt = qimax / qisum, warp-wide
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            nfb += (!decided[c] && !done[c] && live[c]) ? 1u : 0u;
            const double2 sm_ = wide_pool_exact_sum<D, NCH>(sx, c, r, p.pmh, p.pool_m, p.mpad, T);
            const double qsum = sm_.x + MCGPU_FPEPS;
            const double qmax = sm_.y > MCGPU_FPEPS ? sm_.y : MCGPU_FPEPS;
            if (!decided[c]) acc[c] = u[c] < qmax / qsum;
          }
        }
        __syncwarp();
        bool alldone = true;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          if (!done[c] && (acc[c] || it >= (1u << 24) - 2u)) { xt0[c] = c0[c]; xt1[c] = c1[c]; cpick[c] = cc[c]; amax_acc[c] = am[c]; done[c] = true; nit += live[c] ? it + 1u : 0u; }
          alldone = alldone && done[c];
        }
        if (__all_sync(0xffffffffu, alldone)) break;
      }
      // cfac = max_i Q_i(x_old) / max_i Q_i(x'), mcpar.cc:412-439
#pragma unroll
      for (int c = 0; c < NCH; ++c) { sx[i0 * NCH + c] = x0[c]; sx[(i0 + 1) * NCH + c] = x1[c]; }
      __syncwarp();
      double aold[NCH]; float dummy[NCH];
      wide_pool_eval<D, NCH, false>(sx, r, p, aold, dummy);
      __syncwarp();
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        double qmax = mc_exp(amax_acc[c], T);
        qmax = qmax > MCGPU_FPEPS ? qmax : MCGPU_FPEPS;
        cfac[c] = mc_exp(aold[c], T) / qmax;
      }
    }

    if (LIK != MCGPU_ROSENBROCK1) {
#pragma unroll
      for (int c = 0; c < NCH; ++c) { sx[i0 * NCH + c] = xt0[c]; sx[(i0 + 1) * NCH + c] = xt1[c]; }
      __syncwarp();
    }
    double lyt[NCH];
    wide_loglik<LIK, D, NCH>(xt0, xt1, sx, r, p, T, lyt);
    if (LIK != MCGPU_ROSENBROCK1) __syncwarp();

    const double pwgt = (double)(t + 1), winv = 1.0 / pwgt;
    int dec[NCH];
    if (SUMMIX) {
      // u < exp(lyt - ly) q(x)/q(x') from the fp32 bounds on the Hastings factor wherever they settle it
      bool alldec = true;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        dec[c] = cf_ok[c] ? accept_test_bounded(u_acc[c], lyt[c] - ly[c], cf_lo[c], cf_hi[c]) : -1;
        alldec = alldec && dec[c] >= 0;
      }
      if (!__all_sync(0xffffffffu, alldec)) {          // rare: exact log q(x) - log q(x'), warp-wide
        double lo_[NCH], ln_[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) nfb += (dec[c] < 0 && live[c]) ? 1u : 0u;
        __syncwarp();
#pragma unroll
        for (int c = 0; c < NCH; ++c) { sx[i0 * NCH + c] = xt0[c]; sx[(i0 + 1) * NCH + c] = xt1[c]; }
        __syncwarp();
#pragma unroll
        for (int c = 0; c < NCH; ++c) ln_[c] = wide_pool_lse_exact<D, NCH>(sx, c, r, p.pmh, p.pnb, p.pool_m, p.mpad, T);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < NCH; ++c) { sx[i0 * NCH + c] = x0[c]; sx[(i0 + 1) * NCH + c] = x1[c]; }
        __syncwarp();
#pragma unroll
        for (int c = 0; c < NCH; ++c) lo_[c] = wide_pool_lse_exact<D, NCH>(sx, c, r, p.pmh, p.pnb, p.pool_m, p.mpad, T);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < NCH; ++c) if (dec[c] < 0) dec[c] = u_acc[c] < mc_exp((lyt[c] - ly[c]) + (lo_[c] - ln_[c]), T) ? 1 : 0;
      }
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const bool a = SUMMIX ? dec[c] != 0 : accept_test(u_acc[c], lyt[c] - ly[c], MAIN ? cfac[c] : 1.0, T, p.exact_tests);   // same inputs in every lane of the group
      if (a) { ly[c] = lyt[c]; x0[c] = xt0[c]; x1[c] = xt1[c]; }
      nacc[c] += a ? 1u : 0u;
      if (MAIN) {
        if (p.hist && live[c] && tmod == 0) {          // MCout::add: one row per chain, coalesced over the lanes
          double *row = p.hist + ((long long)tring * p.C + jb + c) * (D + 1);
          row[i0] = x0[c]; row[i0 + 1] = x1[c];
          if (r == 0) row[D] = ly[c];
        }
        if (REMOTE && a) {                             // adopt the component's moments, mcpar.cc:190-197
          const double sd0 = __ldg(p.psd + (size_t)i0 * p.mpad + cpick[c]), sd1 = __ldg(p.psd + (size_t)(i0 + 1) * p.mpad + cpick[c]);
          mu0[c] = __ldg(p.pmh + (size_t)i0 * p.mpad + cpick[c]).x; mu1[c] = __ldg(p.pmh + (size_t)(i0 + 1) * p.mpad + cpick[c]).x;
          ps0[c] = (sd0 * sd0) * (pwgt - 1.0); ps1[c] = (sd1 * sd1) * (pwgt - 1.0);
        }
        double dl = x0[c] - mu0[c]; mu0[c] += dl * winv; ps0[c] += dl * (x0[c] - mu0[c]);
        dl = x1[c] - mu1[c]; mu1[c] += dl * winv; ps1[c] += dl * (x1[c] - mu1[c]);
      }
    }
    if (MAIN) { if (++tmod == p.thin) { tmod = 0; if (++tring == p.hist_cap) tring = 0; } }
  }

  unsigned int wacc = 0, nlive = 0;
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    if (live[c]) {
      const long long j = jb + c;
      p.x[j * D + i0] = x0[c]; p.x[j * D + i0 + 1] = x1[c];
      if (r == 0) p.ly[j] = ly[c];
      if (MAIN) {
        p.mu[j * D + i0] = mu0[c]; p.mu[j * D + i0 + 1] = mu1[c]; p.ps[j * D + i0] = ps0[c]; p.ps[j * D + i0 + 1] = ps1[c];
        const long long gg = p.chain0 + j;
        if (p.xc.pool_next && gg % p.xc.pool_stride == 0 && gg / p.xc.pool_stride < p.pool_m) {   // each lane its two parameters
          const double m[2] = {mu0[c], mu1[c]}, v[2] = {ps0[c], ps1[c]};
          publish_slot<2>(p.xc, gg / p.xc.pool_stride, D, i0, m, v, 1.0 / (double)(p.t0 + p.nsteps));
        }
      }
      if (r == 0) { wacc += nacc[c]; ++nlive; }
    }
  }
  // acceptance counters: one count per chain (lane 0 of each group)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { wacc += __shfl_xor_sync(0xffffffffu, wacc, o); nlive += __shfl_xor_sync(0xffffffffu, nlive, o); }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(p.counts, (unsigned long long)wacc);
    atomicAdd(p.counts + 1, (unsigned long long)nlive * (unsigned long long)p.nsteps);
  }
  if (REMOTE) {                                 // main-phase statistics: counts[2] remote chain-steps, [3] candidates
    unsigned int wi = r == 0 ? nit : 0u, wf = r == 0 ? nfb : 0u;   // every lane of a group counted the same
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { wi += __shfl_xor_sync(0xffffffffu, wi, o); wf += __shfl_xor_sync(0xffffffffu, wf, o); }
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(p.counts + 2, (unsigned long long)nlive * (unsigned long long)p.nsteps);
      atomicAdd(p.counts + 3, (unsigned long long)wi);
      if (wf) atomicAdd(p.counts + 6, (unsigned long long)wf);
    }
  }
}

// pool [M][D][2] (mu, sigma^2) -> the prepared pool w (WidePool); padding slots get Q = 0
static __global__ void pool_prep_kernel(const double *pool, int M, int mpad, int D, const WidePool w, const ExchangeParams xc)
{
  wait_pool(xc);
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < mpad) {                                   // n_s = -1/2 sum_i log sig2_si (remote mode 1); padding 0
    double n = 0.0;
    if (idx < M) for (int i = 0; i < D; ++i) n -= 0.5 * log(pool[((size_t)idx * D + i) * 2 + 1]);
    w.pnb[idx] = n; w.pnbf[idx] = (float)(n * 1.4426950408889634);
    atomicMax(reinterpret_cast<int *>(w.pscal + 2), __float_as_int(__double2float_ru(fabs(n * 1.4426950408889634))));
  }
  if (idx >= D * mpad) return;
  const int i = idx / mpad, s = idx % mpad;
  if (s < M) {
    const double m = pool[((size_t)s * D + i) * 2], s2 = pool[((size_t)s * D + i) * 2 + 1];
    const double sd = sqrt(s2), g = sqrt(0.5 * 1.4426950408889634 / s2);     // g = sqrt(log2(e) / (2 sig^2)), as stage_pool
    w.pmh[idx] = make_double2(m, -0.5 / s2); w.psd[idx] = sd;
    w.pf[idx] = make_float2((float)(g * m), (float)g);
    // pool-wide max |mu| and max 1/sigma for the fp32 error bound (non-negative floats order like their bit patterns)
    atomicMax(reinterpret_cast<int *>(w.pscal), __float_as_int(__double2float_ru(fabs(m))));
    atomicMax(reinterpret_cast<int *>(w.pscal + 1), __float_as_int(__double2float_ru(1.0 / sd)));
  } else { w.pmh[idx] = make_double2(1.0e300, -1.0); w.psd[idx] = 0.0; w.pf[idx] = make_float2(1.0e18f, 0.0f); }
}

// row-major lower factor -> column-major copy + "is diagonal" flag
static __global__ void factor_prep_kernel(const double *rm, double *cm, int D, int *diag)
{
  __shared__ int offd;
  if (threadIdx.x == 0) offd = 0;
  __syncthreads();
  for (int idx = threadIdx.x; idx < D * D; idx += blockDim.x) {
    const int i = idx / D, q = idx % D;
    const double v = q <= i ? rm[idx] : 0.0;          // strict upper triangle holds stale input (covar_setup)
    cm[q * D + i] = v;
    if (q < i && v != 0.0) offd = 1;
  }
  __syncthreads();
  if (threadIdx.x == 0) *diag = !offd;
}

}  // namespace MCGPU_NS
}  // namespace mcgpu
