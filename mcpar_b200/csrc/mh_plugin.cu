// mh_plugin.cu -- a device likelihood plugin: the production step kernels instantiated with a user functor.
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
template __global__ void mh_steps_kernel<MCGPU_DEVICE_PLUGIN, PD, RNG_PHILOX, PH_REMOTE>(const StepParams);
template __global__ void mh_steps_kernel<MCGPU_DEVICE_PLUGIN, PD, RNG_PHILOX, PH_MIXED_SUM>(const StepParams);
template __global__ void mh_steps_kernel<MCGPU_DEVICE_PLUGIN, PD, RNG_PHILOX, PH_REMOTE_SUM>(const StepParams);
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

// read by the loader before any launch (cudaLibraryGetGlobal)
extern "C" __device__ int mcgpu_plugin_nparam = MCGPU_PLUGIN_NPARAM;
extern "C" __device__ unsigned long long mcgpu_plugin_stamp = MCGPU_KERNEL_STAMP;
