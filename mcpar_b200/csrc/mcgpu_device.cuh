// mcgpu_device.cuh -- device-side building blocks shared by the step kernels.
//
// Replaces, on the device, what the reference gets from MKL VSL on the host
// (vsRngUniform / viRngUniform / vsRngGaussianMV; call sites src/mcpar.cc:63,146,
// 163,306,337,348,401): a counter-based Philox4x32-10 generator keyed on
// (global chain id, step, draw slot), and a replay reader for supplied streams.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define MCGPU_FPEPS 1.0e-14          // src/mcpar.cc:15
#define MCGPU_SLOT_REMOTE 0x40000000u
#define MCGPU_MAX_D_REG 16           // thread-per-chain kernels keep the state in registers up to this d
#define MCGPU_MAX_D 64
#ifndef MCGPU_CELL_G
#define MCGPU_CELL_G 64              // cells per axis of the d = 2 acceptance-ratio table (mcgpu_cellbound.cuh)
#endif

namespace mcgpu {

struct Words { uint32_t w0, w1, w2, w3; };

// Philox4x32-10 (Salmon et al., SC'11).  10 rounds of two 32x32->64 multiplies.
__device__ __forceinline__ Words philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1)
{
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;   // one IMAD.WIDE each
    const unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
    const uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
    const uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
    const uint32_t n0 = hi1 ^ c1 ^ k0;
    const uint32_t n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  Words w; w.w0 = c0; w.w1 = c1; w.w2 = c2; w.w3 = c3;
  return w;
}

// The same with the 10 round keys precomputed by the host (rk[2r] = k0 + r*W0, rk[2r+1] = k1 + r*W1): the
// kernels pass the copy in their launch parameters, so every round key is a constant-bank operand of the
// LOP3 and the per-round key additions (two issue slots each round) disappear.
__device__ __forceinline__ Words philox4x32_10_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const uint32_t (&rk)[20])
{
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
    const unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ rk[2 * r];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ rk[2 * r + 1];
    c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
  }
  Words w; w.w0 = c0; w.w1 = c1; w.w2 = c2; w.w3 = c3;
  return w;
}

// ---- draws ------------------------------------------------------------------------------
// Every draw is ONE 32-bit Philox word (the reference's MKL streams deliver float32, i.e.
// 24-bit, variates).  Words are addressed as a stream: word idx of (chain, step, base) is
// word idx%4 of the Philox block at slot base + idx/4.
//   local step   (base 0):            pair q -> words (2q, 2q+1); accept uniform -> word 2*NP;
//                                      local/remote coin (of the group leader) -> word 2*NP+1
//   remote candidate it (base REMOTE | it<<6): word 0 -> component pick, word 1 -> rejection
//                                      uniform, pair q -> words (2+2q, 3+2q)
// with NP = ceil(d/2) normal pairs.  At d = 2 a local step is one Philox call, and so is a
// remote candidate.
__device__ __forceinline__ double u32_half(uint32_t w) { return (double)w * (1.0 / 4294967296.0); }           // [0,1)
__device__ __forceinline__ double u32_mid(uint32_t w)  { return ((double)w + 0.5) * (1.0 / 4294967296.0); }   // (0,1)
__device__ __forceinline__ double u32_pos(uint32_t w)  { return ((double)w + 1.0) * (1.0 / 4294967296.0); }   // (0,1]
__device__ __forceinline__ uint32_t word_of(const Words &w, int k) { return k == 0 ? w.w0 : k == 1 ? w.w1 : k == 2 ? w.w2 : w.w3; }

// Box-Muller pair, MKL BOXMULLER2 convention: z0 = r sin(2 pi u2), z1 = r cos(2 pi u2)
__device__ __forceinline__ void normal_pair(uint32_t wa, uint32_t wb, double &z0, double &z1)
{
  const double r = sqrt(fmax(-2.0 * log(u32_pos(wa)), 0.0));
  double s, c;
  sincospi(2.0 * u32_half(wb), &s, &c);
  z0 = r * s; z1 = r * c;
}

// The exchange of the remote pool between windows: where a launch publishes its pool slots and, with a peer-to-peer
// exchange, what it waits for.  The protocol itself is wait_pool, publish_slot and exchange_failed below.
struct ExchangeParams {
  double *pool_next;               // publication target [pool_m][d][2], or null: this launch does not publish
  long long pool_stride;           // slot s is global chain s*pool_stride
  // peer-to-peer exchange (chains sharded over GPUs, one process each): publication stores go
  // straight into every peer's next pool buffer over NVLink, then bump the peer's arrival counter
  char *const *peers; int npeers; long long next_off, arr_off;
  // consumer side: wait until `arrivals` (this GPU's counter) reaches wait_target before reading the pool
  // (wait_target: all slots of the publication this launch READS; pub_wait_target: all slots of the
  // publication before the one it WRITES -- equal without pool lag)
  const unsigned long long *arrivals; unsigned long long wait_target, pub_wait_target; int *xflag;
  unsigned long long *xstat;       // {ns CTA 0 spent waiting for arrivals, launches that waited}
};

// One launch worth of arguments for the fused step kernels.
struct StepParams {
  // chain state, structure-of-arrays over the hosted chains: x[i*ld + j] etc.
  double *x, *ly, *mu, *ps;
  long long C, ld, chain0;
  const double *factor;            // [d*d] row-major lower Cholesky factor (scaled by tuning)
  unsigned long long *counts;      // {accepted, tried} of the current tuning / stats window
  // schedule
  uint32_t key0, key1;             // Philox key = seed
  uint32_t rk[20];                 // its 10 round keys (philox4x32_10_rk)
  uint32_t step0;                  // global step index of the first step of this launch
  int nsteps;                      // steps in this launch
  int t0;                          // main-phase index of the first step (main kernels)
  int nburn_total;                 // replay offsets: burn-in length of the run
  int sync, coin_group;
  int first_remote_t;              // main steps before this one are local: sync * (1 + pool_lag)  (mcpar.cc:142-146 with lag 0)
  double pl;
  uint32_t plan_mask; int plan_valid;   // PH_MIXED with a job-wide coin: bit k = step k of this launch is remote
  // remote-proposal pool: [pool_m][d][2] (mu, sigma^2), and where this launch publishes
  const double *pool_cur; int pool_m;
  ExchangeParams xc;
  int exact_tests;                 // audit mode: accept / rejection tests always in fp64 (MCGPU_EXACT_TESTS=1)
  // sample history: rows (p..., logL), kept step major, then hosted chain
  // (a ring of hist_cap kept steps; the first kept step of this launch goes to ring row hist_ring0)
  double *hist; int thin; int hist_cap, hist_ring0;
  // replay-local streams
  const double *Z, *U; long long nz, nu; int *overrun;
  // likelihood parameters
  double lp[8]; const double *lik_dev; int lik_k;
  // reference remote mode, d = 2: this window's table of acceptance-ratio bounds, or null.  cell_tab[0] = (origin x,
  // origin y, 1 / cell width x, 1 / cell width y), then MCGPU_CELL_G^2 cells (R_lo, R_hi) as float2, row y major
  const float4 *cell_tab;
};

// One launch worth of arguments for the wide (d >= 8, D/2 lanes per chain) kernels.
struct WideParams {
  // chain state, chain-major (AoS): x[chain*D + i], ly[chain], mu, ps like x
  double *x, *ly, *mu, *ps;
  long long C, chain0;
  const double *factor_cm;        // [D*D] COLUMN-major lower factor (factor_cm[q*D + i] = T[i][q])
  const double *factor_rm;        // [D*D] row-major copy (the tuned matrix lives here; diagonal read)
  const int *diagonal;            // device flag: factor has no off-diagonal entries
  unsigned long long *counts;
  uint32_t key0, key1, step0;
  uint32_t rk[20];                 // Philox round keys (philox4x32_10_rk)
  int nsteps, t0;
  // remote pool, prepared, slot fastest: pmh [D][Mpad] = (mu, -1/(2 sig^2)) pairs, psd [D][Mpad] = sigma
  const double2 *pmh; const double *psd; int pool_m, mpad;
  ExchangeParams xc;               // readers wait in pool_prep_kernel, publishers here
  double *hist; int thin; int hist_cap, hist_ring0;
  const double *pnb;               // [Mpad] n_s = -1/2 sum_i log sig2_si (remote mode 1: normalised components)
  const float2 *pf; const float *pnbf; const float *pscal;   // fp32 copy [D][Mpad] (g mu, g), [Mpad] n_s log2 e, {max |mu|, max 1/sigma, max |nb|}
  int summix;                      // remote mode 1
  int exact_tests;                 // audit mode: accept / rejection / Hastings-factor decisions always in fp64 (MCGPU_EXACT_TESTS=1)
  // likelihood: GaussMix parameters, component fastest: gm2 [D][Kpad] = (mu, 1/s2) pairs, gm_lw [Kpad] = log w
  const double2 *gm2; const double *gm_lw; int kpad;
  // device likelihood plugin: its par[] (lik_k reals) on the device
  const double *lik_dev; int lik_k;
};

// The wide kernels' prepared pool, written by pool_prep_kernel and read through the same fields of WideParams (one
// allocation: wide_pool in mcgpu_api.cu)
struct WidePool { double2 *pmh; double *psd, *pnb; float2 *pf; float *pnbf, *pscal; };

// Grid, block, dynamic shared memory and chains per lane group of a wide-kernel launch (wide_launch, mh_wide.cuh)
struct WideLaunch { unsigned grid, block; size_t smem; int nch; };
// Grid, block and dynamic shared memory of a thread-per-chain step-kernel launch (steps_launch, mh_kernels.cuh)
struct StepLaunch { unsigned grid, block; size_t smem; };

// One step of the host-callback likelihood path (mh_hostlik.cuh)
struct HostLikParams {
  double *x, *ly, *mu, *ps;            // [C][d], [C], [C][d], [C][d]
  double *ptrial, *aux; int *flags;    // [C][d]; [C] = cfac (remote mode 0) or log cfac (mode 1); [C]: bit 0 remote, bits 8.. component
  const double *lytrial;               // [C], from the host
  long long C, chain0; int d;
  const double *factor;                // [d][d] row-major lower factor (scaled by tuning)
  unsigned long long *counts;          // {accepted, tried} of the tuning window
  unsigned long long *mcounts;         // main phase: {accepted, tried, remote steps, candidates}
  uint32_t key0, key1, step; int t, main_phase, first_remote_t, coin_group; double pl;
  const double *pool; double *pool_next; int pool_m; long long pool_stride; int remote_mode;
  double *hist; int hist_row;          // ring row of this step's kept sample, or -1
};

// runtime-dispatched likelihood description (verification mode, batched evaluation)
struct LikSpec { int lik, d, k; double lp[8]; const double *dev; };

// One launch worth of arguments for the verification-mode kernel.
struct VerifyParams {
  int d, C, N, rank0, nsamp;
  LikSpec L;
  double *pvals, *ptrial, *ly, *mu, *sig, *ps, *mutrial, *sigtrial;   // [Rl][C*d] / [Rl][C]
  double *factor;                    // [Rl][d*d]
  double *musig;                     // [Rl][2*N*d]  each rank's private musigall
  const double *snap_cur; double *snap_next;      // [2*N*d] what the all-gather delivers
  const double *Z, *U; const int *I;
  const long long *soff;             // [Rl][6] = zoff,zlen,uoff,ulen,ioff,ilen
  long long *cursors;                // [Rl][3]
  unsigned long long *counts;        // [Rl][2]
  int *irate;                        // [Rl]
  int phase, s0, nsteps, sync, refresh, publish;
  double pl, armin, armax, dfac, ifac;
  double *hist;                      // [t][Rl*C][d+1]
  long long hist_chains;
  uint8_t *tr_accept; double *tr_trial_ly, *tr_trial_p, *tr_cfac; uint8_t *tr_remote; int *tr_iters;
  int trace_cap, trace_base;
  int *overrun;
  unsigned long long *rstats;        // {remote rank-steps, rejection iterations, accepted(main), tried(main)}
};

// ---- peer-to-peer exchange helpers ---------------------------------------------------------
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p)
{
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns()
{
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// the calling thread waits (bounded as below) for the arrivals
__device__ __forceinline__ void wait_arrivals_thread(const unsigned long long *arrivals, unsigned long long target, int *xflag)
{
  if (!target || ld_acquire_sys(arrivals) >= target) return;
  const unsigned long long t0 = global_ns();
  while (ld_acquire_sys(arrivals) < target) {
    if (global_ns() - t0 > 10000000000ull) { atomicExch(xflag, 1); break; }
    __nanosleep(100);
  }
}
// one thread per CTA waits (bounded: 10 s, then the engine reports MCGPU_EPEER) until all pool slots of
// the exchange have arrived in this GPU's memory; callers follow with __syncthreads().  CTA 0 -- the first
// one dispatched -- accounts the time it waited in xstat (the exchange time of mcgpu_stats / the log file).
__device__ __forceinline__ void wait_arrivals(const unsigned long long *arrivals, unsigned long long target, int *xflag,
                                              unsigned long long *xstat = nullptr)
{
  if (threadIdx.x != 0) return;
  if (!target || ld_acquire_sys(arrivals) >= target) return;
  const unsigned long long t0 = global_ns();
  wait_arrivals_thread(arrivals, target, xflag);
  if (xstat && blockIdx.x == 0) { atomicAdd(xstat, global_ns() - t0); atomicAdd(xstat + 1, 1ull); }
}
// A peer-to-peer wait timed out (in this launch or an earlier one): the kernel stops stepping instead of sampling from
// an incomplete pool, and the host reports MCGPU_EPEER at the next synchronize.
__device__ __forceinline__ bool exchange_failed(const ExchangeParams &x)
{
  return x.npeers > 0 && *reinterpret_cast<volatile int *>(x.xflag);
}
// The pool-side kernels (pool_prep_kernel, cell_table_kernel): the CTA waits until the publication it reads has arrived.
__device__ __forceinline__ void wait_pool(const ExchangeParams &x)
{
  if (x.wait_target) { wait_arrivals(x.arrivals, x.wait_target, x.xflag, x.xstat); __syncthreads(); }
}
// Publish parameters i0 .. i0+N-1 of pool slot s, (mu, ps * winv), into the next pool [pool_m][D][2].  With a
// peer-to-peer exchange they go into every GPU's next pool over NVLink, and the calling thread then bumps each
// peer's arrival counter once.  A GPU may not publish P+1 before all of P has reached it: its peers' last CTAs of
// the previous window may still read pool P-1, which P+2 will overwrite (three buffers).
template <int N>
__device__ __forceinline__ void publish_slot(const ExchangeParams &x, long long s, int D, int i0, const double (&mu)[N],
                                             const double (&ps)[N], double winv)
{
  if (x.npeers > 0) {
    wait_arrivals_thread(x.arrivals, x.pub_wait_target, x.xflag);
    for (int q = 0; q < x.npeers; ++q) {
      double *dst = reinterpret_cast<double *>(x.peers[q] + x.next_off);
#pragma unroll
      for (int i = 0; i < N; ++i) { dst[(s * D + i0) * 2 + 2 * i] = mu[i]; dst[(s * D + i0) * 2 + 2 * i + 1] = ps[i] * winv; }
    }
    __threadfence_system();                              // the stores are visible before the arrivals
    for (int q = 0; q < x.npeers; ++q)
      atomicAdd_system(reinterpret_cast<unsigned long long *>(x.peers[q] + x.arr_off), 1ull);
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) { x.pool_next[(s * D + i0) * 2 + 2 * i] = mu[i]; x.pool_next[(s * D + i0) * 2 + 2 * i + 1] = ps[i] * winv; }
  }
}

}  // namespace mcgpu
