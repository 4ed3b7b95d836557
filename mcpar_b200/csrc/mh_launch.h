// mh_launch.h -- host-visible launcher prototypes of the two kernel translation units.
#pragma once
#include "mcgpu_device.cuh"
namespace mcgpu {
enum { PH_BURN = 0, PH_MIXED = 1, PH_LOCAL = 2, PH_REMOTE = 3, PH_MIXED_SUM = 4, PH_REMOTE_SUM = 5 };   // kernel phases, see mh_kernels.cuh
namespace fast {
bool wide_supported(int lik, int d);
cudaError_t launch_wide(int lik, int d, int phase, const WideParams &p, cudaStream_t st);
WideLaunch wide_launch(int d, long long C);   // the wide kernels' launch rule (built-in likelihoods and plugins)
cudaError_t launch_pool_prep(const double *pool, int M, int mpad, int D, double2 *pmh, double *psd, double *pnb,
                             float2 *pf, float *pnbf, float *pscal,
                             const unsigned long long *arrivals, unsigned long long wait_target, int *xflag,
                             unsigned long long *xstat, cudaStream_t st);
cudaError_t launch_factor_prep(const double *rm, double *cm, int D, int *diag, cudaStream_t st);
size_t cell_table_bytes();       // the d = 2 table of acceptance-ratio bounds (StepParams::cell_tab)
cudaError_t launch_cell_table(const double *pool, int M, float4 *tab, const unsigned long long *arrivals,
                              unsigned long long wait_target, int *xflag, unsigned long long *xstat, cudaStream_t st);
bool steps_supported(int lik, int d);
size_t steps_smem_bytes(int d, int nsteps, int pool_m, bool with_pool);
StepLaunch steps_launch(int d, long long C, int nsteps, int pool_m, int phase);   // the step kernels' launch rule (built-in likelihoods and plugins)
cudaError_t launch_steps(int lik, int d, int rngk, int phase, const StepParams &p, cudaStream_t st);
cudaError_t launch_init_loglik(int lik, int d, const StepParams &p, cudaStream_t st);
cudaError_t launch_tune(unsigned long long *counts, unsigned long long *cum, double *factor, int dd,
                        double armin, double armax, double dfac, double ifac, cudaStream_t st);
}
namespace exact {
bool steps_supported(int lik, int d);
size_t steps_smem_bytes(int d, int nsteps, int pool_m, bool with_pool);
cudaError_t launch_steps(int lik, int d, int rngk, int phase, const StepParams &p, cudaStream_t st);
cudaError_t launch_init_loglik(int lik, int d, const StepParams &p, cudaStream_t st);
cudaError_t launch_tune(unsigned long long *counts, unsigned long long *cum, double *factor, int dd,
                        double armin, double armax, double dfac, double ifac, cudaStream_t st);
cudaError_t launch_verify(const VerifyParams &p, int nranks_local, cudaStream_t st);
cudaError_t launch_hostlik_propose(const HostLikParams &p, cudaStream_t st);
cudaError_t launch_hostlik_accept(const HostLikParams &p, int publish, double pub_winv, cudaStream_t st);
cudaError_t launch_loglik_aos(const LikSpec &L, const double *x, double *y, int npset, cudaStream_t st);
}
}
