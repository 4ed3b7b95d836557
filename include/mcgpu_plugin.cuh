/* include/mcgpu_plugin.cuh -- author contract of a device likelihood plugin.
 *
 * A plugin is a cubin built from ONE user header by `python -m mcpar_b200.plugin mylik.cuh -o mylik.cubin`.
 * It holds the production step kernels (thread-per-chain, or with MCGPU_PLUGIN_WIDE the wide ones), the
 * initial-log-likelihood kernel (thread-per-chain) and a batched evaluation kernel, all instantiated with the user's
 * functor; mcgpu_set_likelihood_plugin loads it into an
 * engine, which then runs exactly as with a built-in likelihood (counter-based draws, both remote modes,
 * pool lag, burn-in tuning, history and host sinks, checkpoints, peer-to-peer / NCCL exchange, audit mode).
 *
 * A thread-per-chain plugin's header defines the parameter count and one functor:
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
 * A WIDE plugin runs inside the wide step kernels (mh_wide.cuh), which spread one chain over L = nparam / 2 lanes
 * (two parameters per lane).  Its header declares the kind and returns one share of the log-likelihood per lane:
 *
 *   #include "mcgpu_plugin.cuh"
 *   #define MCGPU_PLUGIN_WIDE 1
 *   #ifndef MCGPU_PLUGIN_NPARAM
 *   #define MCGPU_PLUGIN_NPARAM 32                     // 8, 16, 32 or 64
 *   #endif
 *   struct UserLik {
 *     // One share of one chain's log-likelihood.  Parameter i of the point is x[i * xs] (shared memory, read-only).
 *     // part = 0 .. nparts-1 (nparts = MCGPU_PLUGIN_NPARAM / 2: the lanes of the chain's group).
 *     static __device__ __forceinline__ double partial(const double *x, int xs, const double *par, int npar,
 *                                                      int part, int nparts);
 *   };
 *
 * Contract of UserLik::partial:
 *  - the engine's log-likelihood is the sum of the nparts shares, added in a fixed butterfly order (group_sum of
 *    mh_wide.cuh), the same in the step kernels and in the batched evaluation: it does not depend on how the
 *    chains are split across GPUs, and mcgpu_loglik_plugin returns exactly what the step kernels use.
 *  - no barriers and no warp collectives: the engine does the reduction.
 *  - every lane sees the whole point.
 *  - a model that is a sum over data rows splits the rows over the parts (row r goes to part = r % nparts).
 *  - a model that is not a sum returns everything from part 0 and 0 from the other parts (this wastes lanes).
 *  - -inf is allowed and never accepted; a sum that mixes +inf and -inf is NaN, which is never accepted either.
 *  - par and CUDA libm as for eval above.
 * A wide plugin runs with the job-wide local / remote coin only (mcgpu_config.coin_group = 0; MCPar::coin_group = 0).
 *
 * Limits: thread-per-chain plugins at even nparam <= 16 (any coin_group); wide plugins at nparam 8, 16, 32 or 64
 * with coin_group = 0; NORMAL mode only (not VERIFY or REPLAY_LOCAL).
 * The engine passes its launch parameters to the plugin's kernels by value, so a plugin must be rebuilt
 * whenever the kernel sources change: every plugin carries a stamp of those sources and the engine refuses
 * one whose stamp differs from its own.
 */
#ifndef MCGPU_PLUGIN_CUH_
#define MCGPU_PLUGIN_CUH_
#include <math.h>
#endif
