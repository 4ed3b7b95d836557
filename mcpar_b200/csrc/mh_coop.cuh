// mh_coop.cuh -- warp-specialised, CTA-cooperative fused MH step kernel for the Gaussian-mixture likelihood
// at d = 64, K <= 64 components (BASELINE config 4: SURVEY.md 8d C4).
//
// The wide kernel (mh_wide.cuh) streams the mixture's 64 KB of (a, b) pairs through L1 for every group of
// four chains and the remote pool (131 KB in fp32 at M = 256) through L1/L2: at 12 warps per SM it is bound
// by the latency of those loads (FP64 pipe 19 % busy; a sum-mixture remote step at M = 256 costs ten local
// steps).  Here the data every chain needs stays put and the chains stream past it.  One persistent CTA of
// 512 threads per SM, two roles:
//   * MIXTURE WARPS (0-7) hold the whole mixture IN REGISTERS: thread t owns component k = t mod 64 and the
//     quarter h = t / 64 of the parameters (16 (a, b) pairs = 64 registers).  For a batch of NB chains each
//     thread accumulates its partial exponent sum_{i in quarter} x_i (a_ki x_i + b_ki) for every chain -- the
//     points come from shared memory as warp-wide broadcasts, eight chains' loads issued together ahead of
//     their 32 independent DFMA -- and leaves it in shared memory.  In remote mode 1 the same warps then run
//     the pool test against an fp32 copy of the pool (g mu, g) staged ONCE per CTA in shared memory: thread t
//     owns pool slot t mod SL and a slice of the parameters and accumulates the 2 NB exponents (x' and x of
//     every chain of the batch) in registers, 1 + NB/2 LDS per 4 NB FFMA.
//   * OWNER WARPS (8-15): one warp owns a chain for everything else (lane r = parameters 2r, 2r+1, the wide
//     kernel's layout): Philox + Box-Muller proposal (P1), and after the mixture warps are done the
//     log-sum-exp over the 64 exponents, the accept test, the running moments, the history row and the
//     publication to the exchange pool (P3).
// The two roles are decoupled by named barriers (bar.arrive / bar.sync) over two batch slots: while the
// mixture warps work on slot s the owners finish the previous batch of slot s^1 and propose its next one, so
// the FP64 pipe sees the mixture's DFMA stream while the latency-bound owner code runs beside it.  The role
// split also splits the register budget: 64 registers of mixture never coexist with the owners' chain state.
//     owners:   P1(slot 0) P1(slot 1) | wait DONE[s] . read partials . arrive EMPTY . P3(s) . P1(s) . arrive FULL[s] | ...
//     mixture:  wait FULL[s] . partials . wait EMPTY . store partials . arrive DONE[s] | ...
// A slot keeps its batch through all steps of the launch (step k+1 of a chain needs step k), then takes the
// CTA's next batch; batches are dealt round-robin over CTAs and slots.
//
// Same reference lines as the other step kernels: genLocal mcpar.cc:302-312, genRemote :315-451 (remote
// mode 1: the sum-mixture proposal of mh_kernels.cuh), accept :165-175, moments :186-209, MCout::add
// mcout.cc:129-145.  Draw addressing, arithmetic of the proposal, decisions by bounds and statistics are
// those of mh_wide.cuh; only the order of the floating-point sums of the likelihood and of the pool test
// differs (quarters, chunks).
#pragma once

namespace mcgpu {
namespace MCGPU_NS {

constexpr int kCoopThreads = 512, kCoopWarps = 8, kCoopKP = 64;   // 8 mixture warps + 8 owner warps
constexpr int kCoopHalf = kCoopThreads / 2;

enum { CB_FULL0 = 1, CB_FULL1 = 2, CB_DONE0 = 3, CB_DONE1 = 4, CB_EMPTY = 5, CB_MIX = 6 };   // named barriers (0 = __syncthreads)
__device__ __forceinline__ void nb_sync(int id, int cnt) { asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(cnt) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id, int cnt) { __threadfence_block(); asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(cnt) : "memory"); }

// dynamic shared memory of one CTA; SL = pool slots held side by side (power of two, 16..256; 0: no pool)
template <int D, int NCW>
__host__ __device__ constexpr size_t coop_smem_bytes(int SL, bool pool_in_smem)
{
  constexpr int NB = kCoopWarps * NCW, CP = 2 * NB;
  size_t b = sizeof(double) * ((size_t)MCGPU_MATH_SMEM + (size_t)2 * NB * D + (size_t)2 * NB * D + (size_t)2 * NB * 4 +
                               (size_t)kCoopWarps * D * NCW + (size_t)NB * 4 * kCoopKP);
  if (SL > 0) b += sizeof(float) * ((size_t)2 * D * CP + (size_t)kCoopHalf * CP + (size_t)SL) + (pool_in_smem ? sizeof(float2) * (size_t)D * SL : 0);
  return b;
}

// POOLSM: the fp32 pool is staged in shared memory (128 KB at M = 256: leaves room for one chain per owner warp only) or read
// through L1 (`__ldg`, coalesced over the slots; two chains per owner warp)
template <int D, int NCW, int PHASE, bool POOLSM = true>
__global__ void __launch_bounds__(kCoopThreads, 1)
mh_coop_kernel(const WideParams p, const int nbatch, const int SL, const int lsl)
{
  constexpr int L = D / 2, NW = kCoopWarps, NB = NW * NCW, KP = kCoopKP, DQ = D / 4, CP = 2 * NB;
  static_assert(L == 32, "one warp owns a chain: d = 64");
  static_assert(NB % 8 == 0, "the mixture warps take eight chains at a time");
  constexpr bool MAIN = PHASE != PH_BURN, REMOTE = PHASE == PH_REMOTE_SUM;
  constexpr int ABLK = (2 * L) / 4, AW = (2 * L) % 4;   // accept uniform: word 2*NP of the local stream
  extern __shared__ __align__(16) double smem[];
  MathTables T;
  T.exp_tab = smem; T.log_tab = smem + MCGPU_EXP_TAB; T.trig_tab = T.log_tab + 2 * MCGPU_LOG_TAB;
  stage_math_tables(smem);
  double *sx = smem + MCGPU_MATH_SMEM;                  // [2][NB][D]   proposals x' of the slot's batch
  double *stx = sx + 2 * NB * D;                        // [2][NB][D]   the chains' current points between P1 and P3
  double *sts = stx + 2 * NB * D;                       // [2][NB][4]   logL, accept uniform, picked component
  double *szw = sts + 2 * NB * 4;                       // [NW][D*NCW]  per-owner-warp scratch (normals of a dense factor; exact-path points)
  double *sq = szw + NW * D * NCW;                      // [NB][4][KP]  partial exponents of the batch being finished
  float *sxf = reinterpret_cast<float *>(sq + NB * 4 * KP);   // [2][D][CP]  fp32 points: column 2c = x' of chain c, 2c+1 = x
  float *part = sxf + 2 * D * CP;                       // [DC][CP][SL] partial pool exponents, DC * SL = 256; [0] ends up holding the totals
  float *snb = part + kCoopHalf * CP;                   // [SL]         n_s log2 e
  float2 *spool = reinterpret_cast<float2 *>(snb + SL); // [D][SL]      (g mu, g)
  if (exchange_failed(p.xc)) return;

  const int tid = threadIdx.x, warp = tid >> 5, r = tid & 31;
  if (REMOTE && POOLSM) {
    for (int idx = tid; idx < D * SL; idx += kCoopThreads) {
      const int i = idx >> lsl, s = idx & (SL - 1);
      spool[idx] = s < p.mpad ? __ldg(p.pf + (size_t)i * p.mpad + s) : make_float2(1.0e18f, 0.0f);   // padding: Q = 0
    }
  }
  if (REMOTE)
    for (int s = tid; s < SL; s += kCoopThreads) snb[s] = s < p.mpad ? __ldg(p.pnbf + s) : 0.0f;
  // batches of this CTA, dealt alternately to the two slots; a slot runs cnt = (its batches) * nsteps iterations
  const int nb_cta = (int)blockIdx.x < nbatch ? (nbatch - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int cnt0 = ((nb_cta + 1) >> 1) * p.nsteps, cnt1 = (nb_cta >> 1) * p.nsteps;
  const int total_i = 2 * cnt0, total_active = cnt0 + cnt1;
  __syncthreads();

  if (warp < NW) {
    // =========================== mixture warps ===========================
    const int kc = tid & (KP - 1), h = tid >> 6;        // this thread's mixture component and parameter quarter
    double A[DQ], B[DQ];                                // exponent of component k: c_k + sum_i x_i (a_ki x_i + b_ki)
#pragma unroll
    for (int j = 0; j < DQ; ++j) { const double2 ab = __ldg(p.gm2 + (size_t)(h * DQ + j) * p.kpad + kc); A[j] = ab.x; B[j] = ab.y; }
    int seq = 0;
    for (int i = 0; i < total_i; ++i) {
      const int s = i & 1, m = i >> 1;
      if (m >= (s ? cnt1 : cnt0)) continue;
      nb_sync(CB_FULL0 + s, kCoopThreads);              // the owners have staged the slot's proposals
      const double *sxs = sx + (size_t)s * NB * D + h * DQ;
#pragma unroll 1
      for (int c0 = 0; c0 < NB; c0 += 8) {
        double q[8];
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) q[cc] = 0.0;
        const double *xq = sxs + c0 * D;
#pragma unroll
        for (int j = 0; j < DQ; j += 2) {
          double2 xv[8];
#pragma unroll
          for (int cc = 0; cc < 8; ++cc) xv[cc] = *reinterpret_cast<const double2 *>(xq + cc * D + j);   // the same address in every lane: broadcast
#pragma unroll
          for (int cc = 0; cc < 8; ++cc) {
            q[cc] = fma(fma(A[j], xv[cc].x, B[j]), xv[cc].x, q[cc]);
            q[cc] = fma(fma(A[j + 1], xv[cc].y, B[j + 1]), xv[cc].y, q[cc]);
          }
        }
        if (c0 == 0 && seq > 0) nb_sync(CB_EMPTY, kCoopThreads);   // the owners have read the previous batch's partials (and pool totals)
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) sq[((c0 + cc) * 4 + h) * KP + kc] = q[cc];
      }
      if (REMOTE) {
        // pool slot sl, parameter chunk ch: -sum_{i in chunk} (g mu - g y_i)^2 for the 2 NB points of the batch
        const int sl = tid & (SL - 1), ch = tid >> lsl, dpc = (D * SL) >> 8;
        const int dc = kCoopHalf >> lsl;                // parameter chunks (1 when the pool fills the 256 threads: M > 128)
        const float nb0 = dc == 1 ? snb[sl] : 0.0f;     // one chunk: the sums start at n_s log2 e and ARE the totals
        float acc[CP];
#pragma unroll
        for (int v = 0; v < CP; ++v) acc[v] = nb0;
        const float2 *pp = POOLSM ? spool + (size_t)ch * dpc * SL + sl : p.pf + (size_t)ch * dpc * p.mpad + (sl < p.mpad ? sl : 0);
        const int pstride = POOLSM ? SL : p.mpad;
        const bool pad = !POOLSM && sl >= p.mpad;       // slots beyond the pool: Q = 0
        const float4 *xv4 = reinterpret_cast<const float4 *>(sxf + (size_t)s * D * CP + (size_t)ch * dpc * CP);
#pragma unroll 2
        for (int ii = 0; ii < dpc; ++ii) {
          float2 f = POOLSM ? pp[(size_t)ii * pstride] : __ldg(pp + (size_t)ii * pstride);
          if (pad) f = make_float2(1.0e18f, 0.0f);
#pragma unroll
          for (int v = 0; v < CP / 4; ++v) {
            const float4 t4 = xv4[ii * (CP / 4) + v];
            float y;
            y = fmaf(-f.y, t4.x, f.x); acc[4 * v] = fmaf(-y, y, acc[4 * v]);
            y = fmaf(-f.y, t4.y, f.x); acc[4 * v + 1] = fmaf(-y, y, acc[4 * v + 1]);
            y = fmaf(-f.y, t4.z, f.x); acc[4 * v + 2] = fmaf(-y, y, acc[4 * v + 2]);
            y = fmaf(-f.y, t4.w, f.x); acc[4 * v + 3] = fmaf(-y, y, acc[4 * v + 3]);
          }
        }
#pragma unroll
        for (int v = 0; v < CP; ++v) part[((size_t)ch * CP + v) * SL + sl] = acc[v];
        if (dc > 1) {
          nb_sync(CB_MIX, kCoopHalf);                   // mixture warps only
          // totals over the chunks: A_s(y) log2 e = nb_s - sum_i (..)^2, left in part[0][point][slot]
          for (int v = ch; v < CP; v += dc) {
            float e = snb[sl];
            for (int c2 = 0; c2 < dc; ++c2) e += part[((size_t)c2 * CP + v) * SL + sl];
            part[(size_t)v * SL + sl] = e;              // only this thread reads part[0][v][sl]
          }
        }
      }
      nb_arrive(CB_DONE0 + s, kCoopThreads);
      ++seq;
    }
    return;
  }

  // =========================== owner warps ===========================
  const int w = warp - NW, i0 = 2 * r;
  const double lw0 = __ldg(p.gm_lw + r), lw1 = __ldg(p.gm_lw + r + 32);   // lane r sums components r and r + 32
  const double tdiag0 = p.factor_rm[i0 * D + i0], tdiag1 = p.factor_rm[(i0 + 1) * D + i0 + 1];
  const bool diag = *p.diagonal != 0;
  double *sz = szw + (size_t)w * D * NCW;
  const int thin_j0 = MAIN ? (p.thin - p.t0 % p.thin) % p.thin : 0;   // first step of this launch whose sample is kept
  unsigned int wacc = 0, nlive = 0, nfb = 0;            // per lane 0: accepted steps, live chain-steps walked, exact-path fallbacks
  int seq = 0;
  double x0[NCW], x1[NCW], ly[NCW];                     // carried from P3 into the P1 of the slot's next step
  // per slot: (batch index within the slot, step) of the iteration being finished (P3); the proposal (P1) is one ahead
  int bi0 = 0, k0 = -1, bi1 = 0, k1s = -1;              // -1: the slot has not proposed yet

  for (int i = -2; i < total_i; ++i) {
    const int s = i & 1, m = i >> 1, cnt = s ? cnt1 : cnt0;   // (i = -2, -1: s = 0, 1 and m = -1: the slots' first proposals)
    const bool do_p3 = i >= 0 && m < cnt, do_p1 = m + 1 < cnt;
    if (!do_p3 && !do_p1) continue;
    double *sxs = sx + (size_t)s * NB * D, *stxs = stx + (size_t)s * NB * D, *stss = sts + (size_t)s * NB * 4;
    float *sxfs = sxf + (size_t)s * D * CP;
    long long jb = 0;

    if (do_p3) {
      // ---- P3: finish the likelihood, decide, update (step k of batch bi)
      const int bi = s ? bi1 : bi0, k = s ? k1s : k0;    // (= m / nsteps, m mod nsteps, without the divisions)
      const int batch = (int)blockIdx.x + (2 * bi + s) * (int)gridDim.x;
      jb = ((long long)batch * NW + w) * NCW;
      const int t = p.t0 + k;
      nb_sync(CB_DONE0 + s, kCoopThreads);              // the mixture warps have left the slot's partials
      double a0[NCW], a1[NCW];
      float sn[NCW], so[NCW], ref[NCW];
      int cpick[NCW];
#pragma unroll
      for (int c = 0; c < NCW; ++c) {
        const int cb = w * NCW + c;
        a0[c] = lw0; a1[c] = lw1;
#pragma unroll
        for (int hh = 0; hh < 4; ++hh) { a0[c] += sq[(cb * 4 + hh) * KP + r]; a1[c] += sq[(cb * 4 + hh) * KP + r + 32]; }
        sn[c] = so[c] = ref[c] = 0.0f; cpick[c] = 0;
        if (REMOTE) {
          cpick[c] = (int)stss[cb * 4 + 2];
          const float *En = part + (size_t)(2 * cb) * SL, *Eo = En + SL;
          ref[c] = En[cpick[c]];
          for (int sl = r; sl < SL; sl += 32) { sn[c] += ex2_approx(En[sl] - ref[c]); so[c] += ex2_approx(Eo[sl] - ref[c]); }
        }
      }
      if (seq < total_active - 1) nb_arrive(CB_EMPTY, kCoopThreads);   // the partials are in registers: the next batch may overwrite them
      ++seq;

      // the one chain of this warp's batch (if any) that owns a pool slot: smallest multiple of the stride at or above
      // the warp's first chain (one division per warp and batch, 32-bit when the operands fit)
      long long pub_j = -1, pub_s = 0;
      if (MAIN && p.xc.pool_next && k == p.nsteps - 1 && p.xc.pool_stride >= NCW) {
        const unsigned long long g0 = (unsigned long long)(p.chain0 + jb), st = (unsigned long long)p.xc.pool_stride;
        const unsigned long long qd = ((g0 | st) >> 32) == 0 ? (unsigned long long)(((unsigned)g0 + (unsigned)st - 1u) / (unsigned)st) : (g0 + st - 1) / st;
        const unsigned long long first = qd * st;
        if (first < g0 + NCW && qd < (unsigned long long)p.pool_m) { pub_j = (long long)(first - (unsigned long long)p.chain0); pub_s = (long long)qd; }
      }
      const double pwgt = (double)(t + 1), winv = 1.0 / pwgt;
      const bool keep = MAIN && p.hist && k >= thin_j0 && (k - thin_j0) % p.thin == 0;
      const int tring = keep ? (p.hist_ring0 + (k - thin_j0) / p.thin) % p.hist_cap : 0;
#pragma unroll
      for (int c = 0; c < NCW; ++c) {
        const int cb = w * NCW + c;
        const bool live = jb + c < p.C;
        const long long jc = live ? jb + c : p.C - 1;
        const double2 xo = *reinterpret_cast<const double2 *>(stxs + cb * D + i0), xn = *reinterpret_cast<const double2 *>(sxs + cb * D + i0);
        x0[c] = xo.x; x1[c] = xo.y;
        const double xt0 = xn.x, xt1 = xn.y;
        ly[c] = stss[cb * 4];
        const double u_acc = stss[cb * 4 + 1];
        double mu0 = 0.0, mu1 = 0.0, ps0 = 0.0, ps1 = 0.0;
        if (MAIN) {                                     // (lines prefetched into L2 by P1)
          const double2 mv = *reinterpret_cast<const double2 *>(p.mu + jc * D + i0), pv = *reinterpret_cast<const double2 *>(p.ps + jc * D + i0);
          mu0 = mv.x; mu1 = mv.y; ps0 = pv.x; ps1 = pv.y;
        }
        // log-sum-exp of the 64 exponents, taken relative to the chain's CURRENT logL: sum_k exp(a_k - ly) is the acceptance
        // ratio exp(lyt - ly) itself, of order one for any proposal worth a look, so no maximum has to be found first (one
        // butterfly reduction instead of two in the owners' latency chain).  A sum outside [1e-290, 1e290] (a chain stuck at
        // logL = -inf, a proposal 670 below or above) takes the maximum-first form.
        double se = group_sum<L>(mc_exp(a0[c] - ly[c], T) + mc_exp(a1[c] - ly[c], T));
        double lyt;
        if (se > 1.0e-290 && se < 1.0e290) lyt = ly[c] + mc_log_pos(se, T);
        else {                                          // warp-uniform (every lane holds the same sum)
          const double gm = group_max<L>(a0[c] > a1[c] ? a0[c] : a1[c]);
          se = (a0[c] > -INFINITY ? mc_exp(a0[c] - gm, T) : 0.0) + (a1[c] > -INFINITY ? mc_exp(a1[c] - gm, T) : 0.0);
          se = group_sum<L>(se);
          lyt = gm + mc_log(se, T);                     // no finite exponent: -inf + log 0 = -inf
        }
        bool a;
        if (REMOTE) {
          // u < exp(lyt - ly) q(x)/q(x') from fp32 bounds on the Hastings factor (summix_cfac_bounds of mh_kernels.cuh;
          // here the exponents are summed chunk by chunk and taken relative to the picked component afterwards:
          // D + 256/SL + 2 roundings instead of D, covered by the larger rounding terms cu = (24 + D) u24, cn = 4.8e-7 ...)
          const float snc = group_sumf<L>(sn[c]), soc = group_sumf<L>(so[c]);
          const float xabs_n = group_maxf<L>(fmaxf(fabsf((float)xt0), fabsf((float)xt1)));
          const float xabs_o = group_maxf<L>(fmaxf(fabsf((float)x0[c]), fabsf((float)x1[c])));
          float cf_lo, cf_hi;
          const bool ok = summix_cfac_bounds(snc, soc, ref[c], xabs_n, xabs_o, __ldg(p.pscal), __ldg(p.pscal + 1), __ldg(p.pscal + 2),
                                             p.pool_m, D, 24.0f, 4.8e-7f, cf_lo, cf_hi) && !p.exact_tests;   // (audit mode: always the fp64 route)
          int dec = ok ? accept_test_bounded(u_acc, lyt - ly[c], cf_lo, cf_hi) : -1;
          if (dec < 0) {                                // rare, warp-uniform: exact log q(x) - log q(x') in fp64
            nfb += live ? 1u : 0u;
            __syncwarp();
            sz[i0 * NCW + c] = xt0; sz[(i0 + 1) * NCW + c] = xt1;
            __syncwarp();
            const double ln_ = wide_pool_lse_exact<D, NCW>(sz, c, r, p.pmh, p.pnb, p.pool_m, p.mpad, T);
            __syncwarp();
            sz[i0 * NCW + c] = x0[c]; sz[(i0 + 1) * NCW + c] = x1[c];
            __syncwarp();
            const double lo_ = wide_pool_lse_exact<D, NCW>(sz, c, r, p.pmh, p.pnb, p.pool_m, p.mpad, T);
            __syncwarp();
            dec = u_acc < mc_exp((lyt - ly[c]) + (lo_ - ln_), T) ? 1 : 0;
          }
          a = dec != 0;
        } else {
          a = accept_test_local(u_acc, lyt - ly[c], T, p.exact_tests);      // mcpar.cc:67-69 / :167-169 with cfac = 1
        }
        if (a) { ly[c] = lyt; x0[c] = xt0; x1[c] = xt1; }
        if (r == 0 && live) { wacc += a ? 1u : 0u; ++nlive; }
        if (MAIN) {
          if (keep && live) {                            // MCout::add: one row per chain, coalesced over the lanes
            double *row = p.hist + ((long long)tring * p.C + jb + c) * (D + 1);
            row[i0] = x0[c]; row[i0 + 1] = x1[c];
            if (r == 0) row[D] = ly[c];
          }
          if (REMOTE && a) {                             // adopt the component's moments, mcpar.cc:190-197
            const double sd0 = __ldg(p.psd + (size_t)i0 * p.mpad + cpick[c]), sd1 = __ldg(p.psd + (size_t)(i0 + 1) * p.mpad + cpick[c]);
            mu0 = __ldg(p.pmh + (size_t)i0 * p.mpad + cpick[c]).x; mu1 = __ldg(p.pmh + (size_t)(i0 + 1) * p.mpad + cpick[c]).x;
            ps0 = (sd0 * sd0) * (pwgt - 1.0); ps1 = (sd1 * sd1) * (pwgt - 1.0);
          }
          double dl = x0[c] - mu0; mu0 += dl * winv; ps0 += dl * (x0[c] - mu0);
          dl = x1[c] - mu1; mu1 += dl * winv; ps1 += dl * (x1[c] - mu1);
          if (live) {
            *reinterpret_cast<double2 *>(p.mu + jc * D + i0) = make_double2(mu0, mu1);
            *reinterpret_cast<double2 *>(p.ps + jc * D + i0) = make_double2(ps0, ps1);
          }
        }
        if (k == p.nsteps - 1 && live) {
          // the batch leaves the slot: state out, publication to the next exchange pool
          const long long j = jb + c;
          *reinterpret_cast<double2 *>(p.x + j * D + i0) = make_double2(x0[c], x1[c]);
          if (r == 0) p.ly[j] = ly[c];
          long long sidx = pub_s;
          bool is_pub = jb + c == pub_j;
          if (MAIN && p.xc.pool_next && p.xc.pool_stride < NCW) {        // several pool chains in one warp's batch: test each
            const long long gg = p.chain0 + j;
            sidx = gg / p.xc.pool_stride; is_pub = gg - sidx * p.xc.pool_stride == 0 && sidx < p.pool_m;
          }
          if (MAIN && p.xc.pool_next && is_pub) {                        // musigall slot rule, mcpar.cc:205-208: chain s * stride is slot s
            const double m[2] = {mu0, mu1}, v[2] = {ps0, ps1};
            publish_slot<2>(p.xc, sidx, D, i0, m, v, 1.0 / (double)(p.t0 + p.nsteps));
          }
        }
      }
    }

    if (do_p1) {
      // ---- P1: propose step k1 of batch b1 (genLocal / sum-mixture genRemote) and stage x'
      int b1 = s ? bi1 : bi0, k1 = (s ? k1s : k0) + 1;   // the slot's next (batch, step)
      if (k1 == p.nsteps) { k1 = 0; ++b1; }
      if (s) { bi1 = b1; k1s = k1; } else { bi0 = b1; k0 = k1; }
      const int batch = (int)blockIdx.x + (2 * b1 + s) * (int)gridDim.x;
      jb = ((long long)batch * NW + w) * NCW;
      const uint32_t step = p.step0 + (uint32_t)k1;
      uint32_t glo[NCW], ghi[NCW];
      double u_acc[NCW], xt0[NCW], xt1[NCW];
      int cpick[NCW];
#pragma unroll
      for (int c = 0; c < NCW; ++c) {
        const long long jc = jb + c < p.C ? jb + c : p.C - 1;   // idle slots shadow the last chain, never store
        const unsigned long long g = (unsigned long long)(p.chain0 + jc);
        glo[c] = (uint32_t)g; ghi[c] = (uint32_t)(g >> 32);
        if (k1 == 0) {                                  // a new batch enters the slot
          const double2 xv = *reinterpret_cast<const double2 *>(p.x + jc * D + i0);
          x0[c] = xv.x; x1[c] = xv.y;
          ly[c] = p.ly[jc];
          if (MAIN && (r & 7) == 0) {                   // the running moments join in P3: pull their lines towards L2 now
            asm volatile("prefetch.global.L2 [%0];" :: "l"(p.mu + jc * D + 2 * r));
            asm volatile("prefetch.global.L2 [%0];" :: "l"(p.ps + jc * D + 2 * r));
          }
        }
        const Words wa = philox4x32_10_rk(glo[c], ghi[c], step, (uint32_t)ABLK, p.rk);
        u_acc[c] = u32_mid(word_of(wa, AW));
        cpick[c] = 0;
      }
      if (!REMOTE) {
        double za[NCW], zb[NCW];                        // lane r's Box-Muller pair = words (2r, 2r+1) of the chain's local stream
#pragma unroll
        for (int c = 0; c < NCW; ++c) {
          const Words b = philox4x32_10_rk(glo[c], ghi[c], step, (uint32_t)(r >> 1), p.rk);
          normal_pair_t((r & 1) ? b.w2 : b.w0, (r & 1) ? b.w3 : b.w1, za[c], zb[c], T);
        }
        if (diag) {
#pragma unroll
          for (int c = 0; c < NCW; ++c) { xt0[c] = x0[c] + tdiag0 * za[c]; xt1[c] = x1[c] + tdiag1 * zb[c]; }
        } else {                                        // x' = x + T z, rows 2r and 2r+1, terms added in q = 0,1,.. order
#pragma unroll
          for (int c = 0; c < NCW; ++c) { sz[i0 * NCW + c] = za[c]; sz[(i0 + 1) * NCW + c] = zb[c]; }
          __syncwarp();
          double a0[NCW], a1[NCW];
#pragma unroll
          for (int c = 0; c < NCW; ++c) { a0[c] = x0[c]; a1[c] = x1[c]; }
          for (int q = 0; q <= i0; ++q) {
            const double t0 = __ldg(p.factor_cm + q * D + i0), t1 = __ldg(p.factor_cm + q * D + i0 + 1);
#pragma unroll
            for (int c = 0; c < NCW; ++c) { const double zq = sz[q * NCW + c]; a0[c] += t0 * zq; a1[c] += t1 * zq; }
          }
          const double tl = __ldg(p.factor_cm + (i0 + 1) * D + i0 + 1);
#pragma unroll
          for (int c = 0; c < NCW; ++c) { xt0[c] = a0[c]; xt1[c] = a1[c] + tl * zb[c]; }
          __syncwarp();
        }
      } else {
        // remote mode 1: candidate 0 of the remote stream is THE proposal (one pick, one set of normals)
#pragma unroll
        for (int c = 0; c < NCW; ++c) {
          const Words w0 = philox4x32_10_rk(glo[c], ghi[c], step, MCGPU_SLOT_REMOTE, p.rk);
          cpick[c] = (int)__umulhi(w0.w0, (uint32_t)p.pool_m);
          const int qq = r + 1;                         // lane r's pair = words (2+2r, 3+2r)
          Words b = w0;
          if ((qq >> 1) != 0) b = philox4x32_10_rk(glo[c], ghi[c], step, MCGPU_SLOT_REMOTE + (uint32_t)(qq >> 1), p.rk);
          double za, zb;
          normal_pair_t((qq & 1) ? b.w2 : b.w0, (qq & 1) ? b.w3 : b.w1, za, zb, T);
          xt0[c] = __ldg(p.pmh + (size_t)i0 * p.mpad + cpick[c]).x + __ldg(p.psd + (size_t)i0 * p.mpad + cpick[c]) * za;
          xt1[c] = __ldg(p.pmh + (size_t)(i0 + 1) * p.mpad + cpick[c]).x + __ldg(p.psd + (size_t)(i0 + 1) * p.mpad + cpick[c]) * zb;
          const int cb = w * NCW + c;
          *reinterpret_cast<float2 *>(sxfs + i0 * CP + 2 * cb) = make_float2((float)xt0[c], (float)x0[c]);
          *reinterpret_cast<float2 *>(sxfs + (i0 + 1) * CP + 2 * cb) = make_float2((float)xt1[c], (float)x1[c]);
        }
      }
#pragma unroll
      for (int c = 0; c < NCW; ++c) {
        const int cb = w * NCW + c;
        *reinterpret_cast<double2 *>(sxs + cb * D + i0) = make_double2(xt0[c], xt1[c]);
        *reinterpret_cast<double2 *>(stxs + cb * D + i0) = make_double2(x0[c], x1[c]);
        if (r == 0) { stss[cb * 4] = ly[c]; stss[cb * 4 + 1] = u_acc[c]; stss[cb * 4 + 2] = (double)cpick[c]; }
      }
      nb_arrive(CB_FULL0 + s, kCoopThreads);
    }
  }

  // acceptance counters and main-phase statistics: one count per chain-step (lane 0 of the owner warp)
  if (r == 0 && nlive) {
    atomicAdd(p.counts, (unsigned long long)wacc);
    atomicAdd(p.counts + 1, (unsigned long long)nlive);
    if (REMOTE) {                                       // counts[2] remote chain-steps, [3] candidates (one each), [6] exact-path fallbacks
      atomicAdd(p.counts + 2, (unsigned long long)nlive);
      atomicAdd(p.counts + 3, (unsigned long long)nlive);
      if (nfb) atomicAdd(p.counts + 6, (unsigned long long)nfb);
    }
  }
}

}  // namespace MCGPU_NS
}  // namespace mcgpu
