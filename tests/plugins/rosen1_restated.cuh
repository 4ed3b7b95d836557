// rosen1_restated.cuh -- the built-in Rosenbrock1 (Lik<MCGPU_ROSENBROCK1, D> in mh_kernels.cuh, the reference's
// rosenbrock.cc:4-21) typed in again as a plugin author would.  The plugin's step kernels are the same template
// with the same arithmetic, so a run with this plugin must equal the built-in run bit for bit.
#include "mcgpu_plugin.cuh"
#ifndef MCGPU_PLUGIN_NPARAM
#define MCGPU_PLUGIN_NPARAM 2
#endif

struct UserLik {
  static __device__ __forceinline__ double eval(const double (&x)[MCGPU_PLUGIN_NPARAM], const double *, int) {
    double y = 0.0;
#pragma unroll
    for (int i = 0; i + 1 < MCGPU_PLUGIN_NPARAM; i += 2) {
      const double t1 = 1 - x[i];
      const double t2 = x[i + 1] - x[i] * x[i];
      y -= t1 * t1 + 100.0 * t2 * t2;
    }
    return y;
  }
};
