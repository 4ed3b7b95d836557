// logistic.cuh -- Bayesian logistic regression as a device likelihood plugin (include/mcgpu_plugin.cuh).
//
// Parameters x = (b0, b1..b5): an intercept and five coefficients.  Data and prior come in par:
//   par = [n, 1/sigma^2_prior, X (n x 5, row-major), y (n, 0 or 1)]          npar = 2 + 6 n
// log posterior (up to a constant) = sum_i [y_i eta_i - softplus(eta_i)] - 1/2 (1/sigma^2) sum_k b_k^2,
// eta_i = b0 + sum_k X_ik b_k.  softplus(z) = log(1 + e^z) = max(z, 0) + log1p(e^-|z|) never overflows.
// Every chain reads the same data, so it is read through L1 (__ldg).
//
//   python -m mcpar_b200.plugin examples/likelihoods/logistic.cuh -o logistic.cubin
#include "mcgpu_plugin.cuh"
#define MCGPU_PLUGIN_NPARAM 6

struct UserLik {
  static __device__ __forceinline__ double eval(const double (&b)[6], const double *par, int) {
    const int n = (int)__ldg(par);
    const double prec = __ldg(par + 1);
    const double *X = par + 2, *y = X + 5 * (size_t)n;
    double s = 0.0;
    for (int i = 0; i < n; ++i) {
      double eta = b[0];
#pragma unroll
      for (int k = 0; k < 5; ++k) eta += __ldg(X + 5 * i + k) * b[k + 1];
      const double sp = fmax(eta, 0.0) + log1p(exp(-fabs(eta)));
      s += __ldg(y + i) * eta - sp;
    }
    double q = 0.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) q += b[k] * b[k];
    return s - 0.5 * prec * q;
  }
};
