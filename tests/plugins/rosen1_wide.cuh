// rosen1_wide.cuh -- the built-in wide Rosenbrock1 (wide_loglik<MCGPU_ROSENBROCK1> in mh_wide.cuh, the reference's
// rosenbrock.cc:4-21) typed in again as a wide plugin author would.  Lane `part` of a chain's group returns the term
// of parameter pair `part`; the engine adds the shares in the butterfly order the built-in uses, so a run with this
// plugin must equal the built-in wide run bit for bit (once a chain has accepted a proposal: the initial
// log-likelihoods of the built-in come from another kernel).
#include "mcgpu_plugin.cuh"
#define MCGPU_PLUGIN_WIDE 1
#ifndef MCGPU_PLUGIN_NPARAM
#define MCGPU_PLUGIN_NPARAM 16
#endif

struct UserLik {
  static __device__ __forceinline__ double partial(const double *x, int xs, const double *, int, int part, int) {
    const double x0 = x[(2 * part) * xs], x1 = x[(2 * part + 1) * xs];
    const double t1 = 1 - x0;
    const double t2 = x1 - x0 * x0;
    return -(t1 * t1 + 100.0 * t2 * t2);
  }
};
