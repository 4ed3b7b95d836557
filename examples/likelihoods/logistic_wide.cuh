// logistic_wide.cuh -- Bayesian logistic regression with 31 predictors as a wide device likelihood plugin
// (include/mcgpu_plugin.cuh: MCGPU_PLUGIN_WIDE, d = 32, 16 lanes per chain).
//
// Parameters x = (b0, b1..b31): an intercept and 31 coefficients.  Data and prior come in par:
//   par = [n, 1/sigma^2_prior, X (n x 31, row-major), y (n, 0 or 1)]          npar = 2 + 32 n
// log posterior (up to a constant) = sum_i [y_i eta_i - softplus(eta_i)] - 1/2 (1/sigma^2) sum_k b_k^2,
// eta_i = b0 + sum_k X_ik b_k.  softplus(z) = log(1 + e^z) = max(z, 0) + log1p(e^-|z|) never overflows.
// The data rows are split over the lanes of the chain's group (row i goes to part i % nparts), and each lane adds
// the prior term of its own parameter pair (2 part, 2 part + 1); the engine adds the shares.  Every chain reads the
// same data, so it is read through L1 (__ldg); the point is in shared memory, x[k * xs].
//
//   python -m mcpar_b200.plugin examples/likelihoods/logistic_wide.cuh -o logistic_wide.cubin
#include "mcgpu_plugin.cuh"
#define MCGPU_PLUGIN_WIDE 1
#define MCGPU_PLUGIN_NPARAM 32

struct UserLik {
  static __device__ __forceinline__ double partial(const double *b, int xs, const double *par, int, int part, int nparts) {
    const int n = (int)__ldg(par);
    const double prec = __ldg(par + 1);
    const double *X = par + 2, *y = X + 31 * (size_t)n;
    double s = 0.0;
    for (int i = part; i < n; i += nparts) {
      double eta = b[0];
#pragma unroll
      for (int k = 0; k < 31; ++k) eta += __ldg(X + 31 * (size_t)i + k) * b[(k + 1) * xs];
      const double sp = fmax(eta, 0.0) + log1p(exp(-fabs(eta)));
      s += __ldg(y + i) * eta - sp;
    }
    const double b0 = b[(2 * part) * xs], b1 = b[(2 * part + 1) * xs];
    return s - 0.5 * prec * (b0 * b0 + b1 * b1);
  }
};
