// mh_fast.cu -- production instantiations of the fused step kernels (FMA contraction on).
#define MCGPU_NS fast
#include <stdlib.h>
#include <algorithm>
#include "mh_kernels.cuh"
#include "mh_wide.cuh"
#include "mh_coop.cuh"
#include "mcgpu_cellbound.cuh"
namespace mcgpu { namespace fast {
#include "mh_dispatch.inl"

// ---- wide (d >= 8, D/2 lanes per chain) kernels ------------------------------------------
bool wide_supported(int lik, int d)
{
  return (lik == MCGPU_ROSENBROCK1 || lik == MCGPU_GAUSSMIX) && (d == 8 || d == 16 || d == 32 || d == 64);
}

template <int LIK, int D>
static cudaError_t launch_wide_d(int phase, const WideParams &p, cudaStream_t st)
{
  constexpr int NCH = WideNch<D>::value;
  const WideLaunch g = wide_launch(D, p.C);
  switch (phase) {
    case PH_BURN:   mh_wide_kernel<LIK, D, NCH, PH_BURN><<<g.grid, g.block, g.smem, st>>>(p); break;
    case PH_LOCAL:  mh_wide_kernel<LIK, D, NCH, PH_LOCAL><<<g.grid, g.block, g.smem, st>>>(p); break;
    case PH_REMOTE: mh_wide_kernel<LIK, D, NCH, PH_REMOTE><<<g.grid, g.block, g.smem, st>>>(p); break;
    case PH_REMOTE_SUM: mh_wide_kernel<LIK, D, NCH, PH_REMOTE_SUM><<<g.grid, g.block, g.smem, st>>>(p); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

template <int LIK>
static cudaError_t launch_wide_lik(int d, int phase, const WideParams &p, cudaStream_t st)
{
  switch (d) {
    case 8:  return launch_wide_d<LIK, 8>(phase, p, st);
    case 16: return launch_wide_d<LIK, 16>(phase, p, st);
    case 32: return launch_wide_d<LIK, 32>(phase, p, st);
    case 64: return launch_wide_d<LIK, 64>(phase, p, st);
  }
  return cudaErrorInvalidValue;
}

// ---- CTA-cooperative kernel: GaussMix at d = 64, K <= 64 (mh_coop.cuh) -------------------
#ifndef MCGPU_COOP_NCW
#define MCGPU_COOP_NCW 4        // chains per owner warp and batch (1 / 2 / 4: 2.56 / 2.03 / 1.78 ms per local step of 2^20 chains)
#endif
#ifndef MCGPU_COOP_POOLSM
#define MCGPU_COOP_POOLSM 1     // remote kernels: 1 = fp32 pool staged in shared memory (one chain per owner warp), 0 = read through L1 (two): 2.23 vs 2.72 ms per step of config 4
#endif
template <int PHASE>
static cudaError_t launch_coop_phase(const WideParams &p, cudaStream_t st)
{
  constexpr bool REMOTE = PHASE == PH_REMOTE_SUM, POOLSM = MCGPU_COOP_POOLSM != 0;
  constexpr int D = 64, NCW = REMOTE ? (POOLSM ? 1 : 2) : MCGPU_COOP_NCW, NB = kCoopWarps * NCW;
  int SL = 0, lsl = 0;
  if (REMOTE) { SL = 16; lsl = 4; while (SL < p.mpad) { SL <<= 1; ++lsl; } }
  const size_t smem = coop_smem_bytes<D, NCW>(SL, POOLSM);
  int dev = 0, sms = 0;            // per launch: one process may drive engines on several devices, and the attribute is per device
  cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaError_t rc = cudaFuncSetAttribute(mh_coop_kernel<D, NCW, PHASE, POOLSM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (rc != cudaSuccess) return rc;
  const long long nbatch = (p.C + NB - 1) / NB;
  const unsigned grid = (unsigned)std::min<long long>(nbatch, (long long)sms);   // persistent: one CTA per SM
  mh_coop_kernel<D, NCW, PHASE, POOLSM><<<grid, kCoopThreads, smem, st>>>(p, (int)nbatch, SL, lsl);
  return cudaGetLastError();
}

static bool coop_applies(int lik, int d, int phase, const WideParams &p)
{
  static const bool off = getenv("MCGPU_NO_COOP") && atoi(getenv("MCGPU_NO_COOP"));
  if (off || lik != MCGPU_GAUSSMIX || d != 64 || p.kpad != kCoopKP) return false;
  if (phase == PH_BURN || phase == PH_LOCAL) return true;
  return phase == PH_REMOTE_SUM && p.mpad <= 256;      // the reference's rejection loop (PH_REMOTE) stays on the wide kernel
}

cudaError_t launch_wide(int lik, int d, int phase, const WideParams &p, cudaStream_t st)
{
  if (coop_applies(lik, d, phase, p)) {
    switch (phase) {
      case PH_BURN:       return launch_coop_phase<PH_BURN>(p, st);
      case PH_LOCAL:      return launch_coop_phase<PH_LOCAL>(p, st);
      case PH_REMOTE_SUM: return launch_coop_phase<PH_REMOTE_SUM>(p, st);
    }
  }
  if (lik == MCGPU_ROSENBROCK1) return launch_wide_lik<MCGPU_ROSENBROCK1>(d, phase, p, st);
  if (lik == MCGPU_GAUSSMIX) return launch_wide_lik<MCGPU_GAUSSMIX>(d, phase, p, st);
  return cudaErrorInvalidValue;
}

cudaError_t launch_pool_prep(const double *pool, int M, int mpad, int D, const WidePool &w, const ExchangeParams &xc, cudaStream_t st)
{
  cudaMemsetAsync(w.pscal, 0, 4 * sizeof(float), st);
  pool_prep_kernel<<<(D * mpad + 127) / 128, 128, 0, st>>>(pool, M, mpad, D, w, xc);
  return cudaGetLastError();
}

// ---- reference remote mode, d = 2: the window's table of acceptance-ratio bounds (mcgpu_cellbound.cuh) ----------
struct CellRedWarp {
  __device__ double max(double v) const { for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o)); return v; }
  __device__ double sum(double v) const { for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o); return v; }
  __device__ int min(int v) const { for (int o = 16; o > 0; o >>= 1) v = ::min(v, __shfl_xor_sync(0xffffffffu, v, o)); return v; }
};

// One warp per cell.  The grid spans, per axis, min_s (mu_s - 5 sigma_s) .. max_s (mu_s + 5 sigma_s): the fp32 Box-Muller
// normals stay below 6.66, so the few candidates beyond it fall back to the pool loop.  Every warp derives the grid
// from the pool itself (exact min / max reductions: all warps agree); a pool with a non-finite or non-positive entry
// gets a NaN header, which no candidate passes.  With a peer-to-peer exchange the CTAs first wait for the arrivals,
// as pool_prep_kernel does.
static __global__ void __launch_bounds__(128) cell_table_kernel(const double *pool, int M, float4 *tab, const ExchangeParams xc)
{
  wait_pool(xc);
  constexpr int G = MCGPU_CELL_G;
  const int lane = threadIdx.x & 31, cell = blockIdx.x * 4 + (threadIdx.x >> 5);
  const CellRedWarp red;
  double lo[2] = {INFINITY, INFINITY}, hi[2] = {-INFINITY, -INFINITY}, bad = 0.0;
  for (int s = lane; s < M; s += 32)
    for (int i = 0; i < 2; ++i) {
      const double m = pool[(s * 2 + i) * 2], sd = sqrt(pool[(s * 2 + i) * 2 + 1]);
      if (!(sd > 0.0 && fabs(m) + 5.0 * sd <= 1.0e30)) bad = 1.0;
      else { lo[i] = fmin(lo[i], m - 5.0 * sd); hi[i] = fmax(hi[i], m + 5.0 * sd); }
    }
  float o[2], inv[2];
  bool ok = red.max(bad) == 0.0;
  for (int i = 0; i < 2; ++i) {
    const double l = -red.max(-lo[i]), h = red.max(hi[i]);
    o[i] = __double2float_rd(l);
    inv[i] = __double2float_rn((double)G / (h - (double)o[i]));
    ok = ok && inv[i] > 0.0f && inv[i] < 1.0e30f;
  }
  if (!ok) { o[0] = o[1] = inv[0] = inv[1] = NAN; }
  if (blockIdx.x == 0 && threadIdx.x == 0) tab[0] = make_float4(o[0], o[1], inv[0], inv[1]);
  if (!ok || cell >= G * G) return;
  const int gx = cell % G, gy = cell / G;
  const double ix = 1.0 / (double)inv[0], iy = 1.0 / (double)inv[1];
  double rlo, rhi;
  cell_bounds2(pool, M, (double)o[0] + (gx + 0.5) * ix, (double)o[1] + (gy + 0.5) * iy,
               (0.5 + 1.0 / 64.0) * ix * (1.0 + 1.0e-12), (0.5 + 1.0 / 64.0) * iy * (1.0 + 1.0e-12), lane, 32, red, rlo, rhi);
  float flo, fhi;
  cell_store_bounds(rlo, rhi, flo, fhi);
  if (lane == 0) reinterpret_cast<float2 *>(tab + 1)[cell] = make_float2(flo, fhi);
}

size_t cell_table_bytes() { return sizeof(float4) + sizeof(float2) * MCGPU_CELL_G * MCGPU_CELL_G; }

cudaError_t launch_cell_table(const double *pool, int M, float4 *tab, const ExchangeParams &xc, cudaStream_t st)
{
  cell_table_kernel<<<MCGPU_CELL_G * MCGPU_CELL_G / 4, 128, 0, st>>>(pool, M, tab, xc);
  return cudaGetLastError();
}

const void *module_kernel() { return reinterpret_cast<const void *>(cell_table_kernel); }

cudaError_t launch_factor_prep(const double *rm, double *cm, int D, int *diag, cudaStream_t st)
{
  factor_prep_kernel<<<1, 256, 0, st>>>(rm, cm, D, diag);
  return cudaGetLastError();
}
}}
#ifdef MCGPU_CELL_COUNT
// counting build: read and clear the table's counters (tools/cell_hits.py)
extern "C" int mcgpu_cell_counts(unsigned long long out[4])
{
  if (cudaMemcpyFromSymbol(out, mcgpu::fast::mcgpu_cell_count, 4 * sizeof(unsigned long long)) != cudaSuccess) return 1;
  const unsigned long long z[4] = {0, 0, 0, 0};
  return cudaMemcpyToSymbol(mcgpu::fast::mcgpu_cell_count, z, sizeof z) != cudaSuccess;
}
#endif
