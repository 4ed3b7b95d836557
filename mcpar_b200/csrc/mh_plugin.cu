// mh_plugin.cu -- a device likelihood plugin: the production step kernels instantiated with a user functor, the
// thread-per-chain kernels (mh_kernels.cuh) or, when the header defines MCGPU_PLUGIN_WIDE, the wide ones (mh_wide.cuh).
//
// Never part of libmcgpu.so.  mcpar_b200/plugin.py compiles this unit once per user header into a cubin
// (`-include <header>` or -DMCGPU_PLUGIN_HEADER="<header>", -DMCGPU_KERNEL_STAMP=...), with the flags of
// mh_fast.cu; mcgpu_set_likelihood_plugin loads the cubin and launches its kernels by name
// (plugin_kernel_name in mcgpu_api.cu).  The author contract is include/mcgpu_plugin.cuh.
#define MCGPU_NS fast
#include <stdlib.h>
#ifdef MCGPU_PLUGIN_HEADER
#include MCGPU_PLUGIN_HEADER
#endif
#include "mh_kernels.cuh"

#ifndef MCGPU_PLUGIN_NPARAM
#error "the plugin header must define MCGPU_PLUGIN_NPARAM"
#endif
#ifndef MCGPU_KERNEL_STAMP
#error "build plugins with mcpar_b200/plugin.py: it passes -DMCGPU_KERNEL_STAMP"
#endif

#ifdef MCGPU_PLUGIN_WIDE
// ---- wide plugin: mh_wide_kernel, d/2 lanes per chain, UserLik::partial per lane ----------------------------------
#include "mh_wide.cuh"
static_assert(MCGPU_PLUGIN_NPARAM == 8 || MCGPU_PLUGIN_NPARAM == 16 || MCGPU_PLUGIN_NPARAM == 32 || MCGPU_PLUGIN_NPARAM == 64,
              "MCGPU_PLUGIN_NPARAM of a wide plugin (MCGPU_PLUGIN_WIDE) must be 8, 16, 32 or 64");

namespace mcgpu { namespace fast {

constexpr int PD = MCGPU_PLUGIN_NPARAM, PL = PD / 2, PNCH = WideNch<PD>::value;

template <> struct WideLik<MCGPU_DEVICE_PLUGIN, PD> {
  static __device__ __forceinline__ double partial(const double *x, int xs, const WideParams &p, int part) {
    return UserLik::partial(x, xs, p.lik_dev, p.lik_k, part, PL);
  }
};

template __global__ void mh_wide_kernel<MCGPU_DEVICE_PLUGIN, PD, PNCH, PH_BURN>(const WideParams);
template __global__ void mh_wide_kernel<MCGPU_DEVICE_PLUGIN, PD, PNCH, PH_LOCAL>(const WideParams);
template __global__ void mh_wide_kernel<MCGPU_DEVICE_PLUGIN, PD, PNCH, PH_REMOTE>(const WideParams);
template __global__ void mh_wide_kernel<MCGPU_DEVICE_PLUGIN, PD, PNCH, PH_REMOTE_SUM>(const WideParams);

}}  // namespace mcgpu::fast

// VLFunc::operator()(npset, x, y) for the plugin: x is npset*nparam chain-major (AoS), y is npset.  One lane group
// per point in CTAs of 128 threads, the point staged in shared memory and the shares added by the step kernels'
// group_sum, so y equals what the step kernels compute at the same point bit for bit.  The engine also takes the
// initial log-likelihoods of its (AoS) state from here.
extern "C" __global__ void __launch_bounds__(128) mcgpu_plugin_loglik(const double *par, int npar, const double *x, double *y, int npset)
{
  using namespace mcgpu::fast;
  __shared__ __align__(16) double sx[128 / PL * PD];
  const int g = threadIdx.x / PL, r = threadIdx.x % PL;
  const long long j0 = (long long)blockIdx.x * (128 / PL) + g;
  const long long j = j0 < npset ? j0 : npset - 1;      // idle groups shadow the last point: every lane reaches the shuffles
  double *s = sx + g * PD;
  s[2 * r] = x[j * PD + 2 * r]; s[2 * r + 1] = x[j * PD + 2 * r + 1];
  __syncwarp();
  const double v = group_sum<PL>(UserLik::partial(s, 1, par, npar, r, PL));
  if (j0 < npset && r == 0) y[j0] = v;
}

extern "C" __device__ int mcgpu_plugin_wide = 1;
extern "C" __device__ int mcgpu_plugin_nch = mcgpu::fast::PNCH;   // chains per lane group: must be the library's (wide_launch)

#else
// ---- thread-per-chain plugin: mh_steps_kernel, one thread per chain, UserLik::eval ---------------------------------
static_assert(MCGPU_PLUGIN_NPARAM >= 2 && MCGPU_PLUGIN_NPARAM <= MCGPU_MAX_D_REG && MCGPU_PLUGIN_NPARAM % 2 == 0,
              "MCGPU_PLUGIN_NPARAM must be even and in 2..16 (thread-per-chain kernels)");

namespace mcgpu { namespace fast {

constexpr int PD = MCGPU_PLUGIN_NPARAM;

// the user functor behind the engine's likelihood id; par = lik_dev (npar = lik_k reals)
template <> struct Lik<MCGPU_DEVICE_PLUGIN, PD> {
  static __device__ __forceinline__ double eval(const double (&x)[PD], const StepParams &p, const MathTables &) {
    return UserLik::eval(x, p.lik_dev, p.lik_k);
  }
};

template __global__ void mh_steps_kernel<MCGPU_DEVICE_PLUGIN, PD, RNG_PHILOX, PH_BURN>(const StepParams);
template __global__ void mh_steps_kernel<MCGPU_DEVICE_PLUGIN, PD, RNG_PHILOX, PH_MIXED>(const StepParams);
template __global__ void mh_steps_kernel<MCGPU_DEVICE_PLUGIN, PD, RNG_PHILOX, PH_LOCAL>(const StepParams);
template __global__ void mh_steps_kernel<MCGPU_DEVICE_PLUGIN, PD, RNG_PHILOX, PH_MIXED_SUM>(const StepParams);
template __global__ void init_loglik_kernel<MCGPU_DEVICE_PLUGIN, PD>(const StepParams);

}}  // namespace mcgpu::fast

// VLFunc::operator()(npset, x, y) for the plugin: x is npset*nparam chain-major (AoS), y is npset
extern "C" __global__ void mcgpu_plugin_loglik(const double *par, int npar, const double *x, double *y, int npset)
{
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= npset) return;
  double xj[mcgpu::fast::PD];
#pragma unroll
  for (int i = 0; i < mcgpu::fast::PD; ++i) xj[i] = x[j * mcgpu::fast::PD + i];
  y[j] = UserLik::eval(xj, par, npar);
}

extern "C" __device__ int mcgpu_plugin_wide = 0;
extern "C" __device__ int mcgpu_plugin_nch = 1;
#endif

// read by the loader before any launch (cudaLibraryGetGlobal)
extern "C" __device__ int mcgpu_plugin_nparam = MCGPU_PLUGIN_NPARAM;
extern "C" __device__ unsigned long long mcgpu_plugin_stamp = MCGPU_KERNEL_STAMP;
