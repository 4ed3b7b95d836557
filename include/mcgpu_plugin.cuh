/* include/mcgpu_plugin.cuh -- author contract of a device likelihood plugin.
 *
 * A plugin is a cubin built from ONE user header by `python -m mcpar_b200.plugin mylik.cuh -o mylik.cubin`.
 * It holds the production thread-per-chain step kernels, the initial-log-likelihood kernel and a batched
 * evaluation kernel, all instantiated with the user's functor; mcgpu_set_likelihood_plugin loads it into an
 * engine, which then runs exactly as with a built-in likelihood (counter-based draws, both remote modes,
 * pool lag, burn-in tuning, history and host sinks, checkpoints, peer-to-peer / NCCL exchange, audit mode).
 *
 * The user header defines the parameter count and one functor:
 *
 *   #include "mcgpu_plugin.cuh"                        // optional: this contract
 *   #ifndef MCGPU_PLUGIN_NPARAM                        // the guard lets `plugin.build(..., nparam=n)` override it
 *   #define MCGPU_PLUGIN_NPARAM 6                      // even, 2..16
 *   #endif
 *   struct UserLik {
 *     // x: one chain's point; par: device copy of the par[] given to mcgpu_set_likelihood_plugin (npar reals)
 *     static __device__ __forceinline__ double eval(const double (&x)[MCGPU_PLUGIN_NPARAM], const double *par, int npar);
 *   };
 *
 * Contract of UserLik::eval:
 *  - it returns a LOG-likelihood.  -inf is allowed and is never accepted (as DualGaussian far from its modes);
 *    NaN is never accepted either.
 *  - it runs in one thread per chain inside the step kernel: no shared memory, no barriers, no warp
 *    collectives (chains of one warp take different branches).
 *  - CUDA libm (exp, log, log1p, ...) is available.
 *  - par is read-only and shared by every chain (read it through L1: __ldg); npar is what the caller passed.
 *  - it is called with the same x for the same chain state on every GPU, so a deterministic eval keeps runs
 *    reproducible and independent of how chains are split across GPUs.
 *
 * Limits: thread-per-chain kernels only (even nparam <= 16); NORMAL mode only (not VERIFY or REPLAY_LOCAL).
 * The engine passes its launch parameters to the plugin's kernels by value, so a plugin must be rebuilt
 * whenever the kernel sources change: every plugin carries a stamp of those sources and the engine refuses
 * one whose stamp differs from its own.
 */
#ifndef MCGPU_PLUGIN_CUH_
#define MCGPU_PLUGIN_CUH_
#include <math.h>
#endif
