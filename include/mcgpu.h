/* include/mcgpu.h -- C ABI of the B200-native Metropolis-Hastings step engine.
 *
 * This is the drop-in boundary for MCPar's hot path: everything MCPar::run
 * (reference src/mcpar.cc:17-214) does per step -- proposal generation
 * (genLocal :302-312, genRemote :315-451), the VLFunc likelihood evaluation
 * (src/vlfunc.hh:9-12, src/rosenbrock.cc), the accept test and state update
 * (:65-75, :165-175), burn-in tuning (:78-96), the running moments and their
 * publication (:186-209), the inter-rank exchange (:127-140) and the sample
 * store (MCout::add, src/mcout.cc:129-145) -- runs on the GPU behind these entry
 * points.  Plain pointers and sizes only; no C++ or torch types cross it.
 *
 * Conventions
 *  - every function returns 0 on success or a negative MCGPU_E* code; nothing
 *    throws across the boundary; mcgpu_last_error() gives the text.
 *  - host arrays use the reference's layouts: parameters are chain-major AoS
 *    {a1,b1,c1,a2,b2,c2,...} (src/mcpar.hh:63-64), sample rows are
 *    (p_0..p_{d-1}, logL) (src/mcout.cc:129-145), the (mu,sigma^2) table is
 *    [chain][param][2] (src/mcpar.cc:206-208).
 *  - the engine owns all device memory; the caller owns every host buffer.
 *  - all reals are fp64 (the reference is fp32; see DESIGN.md).
 *  - there is NO CPU fallback: without a CUDA device every compute call fails
 *    with MCGPU_ENODEVICE.
 */
#ifndef MCGPU_H_
#define MCGPU_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCGPU_ABI_VERSION 2

enum {
  MCGPU_OK = 0,
  MCGPU_EINVAL = -1,        /* bad argument / unsupported shape            */
  MCGPU_ENODEVICE = -2,     /* no usable CUDA device                       */
  MCGPU_ECUDA = -3,         /* CUDA runtime error (see mcgpu_last_error)   */
  MCGPU_ESTATE = -4,        /* call out of order                           */
  MCGPU_ENOMEM = -5,
  MCGPU_ESTREAM = -6,       /* a replay stream ran dry                     */
  MCGPU_EPEER = -7          /* a peer GPU did not publish within the bound */
};

/* likelihood functors; replaces the VLFunc subclasses of src/rosenbrock.hh */
enum {
  MCGPU_ROSENBROCK1 = 0,    /* rosenbrock.cc:4-21,   par: none                      */
  MCGPU_ROSENBROCK2 = 1,    /* rosenbrock.cc:25-41,  par: none (verify mode + eval) */
  MCGPU_GAUSSIAN = 2,       /* rosenbrock.cc:44-61,  par: mu[2], sig2[2] (optional) */
  MCGPU_DUALGAUSSIAN = 3,   /* rosenbrock.cc:63-78,  par: w (optional, default 5)   */
  MCGPU_GAUSSMIX = 4,       /* new: par = K, mu[K][d], sig2[K][d], w[K]             */
  MCGPU_HOST_LIKELIHOOD = 100, /* the likelihood is a host callback (a user-written VLFunc, src/vlfunc.hh:9-12):
                               the engine steps with mcgpu_step_propose / mcgpu_step_accept      */
  MCGPU_DEVICE_PLUGIN = 101 /* a user functor compiled into a plugin cubin (include/mcgpu_plugin.cuh):
                               set with mcgpu_set_likelihood_plugin                               */
};

enum {
  MCGPU_MODE_NORMAL = 0,    /* in-kernel Philox4x32-10 keyed on (global chain, step, slot) */
  MCGPU_MODE_VERIFY = 1,    /* the reference's rank-structured algorithm on supplied
                               normal/uniform/int streams (SURVEY.md 8c protocol)    */
  MCGPU_MODE_REPLAY_LOCAL = 2 /* the production kernel, exact arithmetic, reading supplied
                               streams at the reference's offsets; local proposals only
                               (burn-in, or pl >= 1)                                 */
};

typedef struct mcgpu_engine mcgpu_engine;

/* Replaces the MCPar constructor arguments (src/mcpar.hh:32-33, mcpar.cc:216-226). */
typedef struct mcgpu_config {
  int32_t abi_version;      /* MCGPU_ABI_VERSION                                     */
  int32_t device;           /* CUDA ordinal                                          */
  int32_t mode;             /* MCGPU_MODE_*                                          */
  int32_t nparam;           /* np                                                    */
  int64_t nchain;           /* chains hosted by this engine                          */
  int64_t chain0;           /* global id of the first hosted chain (multiple of 32)  */
  int64_t nchain_total;     /* tchains = all chains of the job (mcpar.cc:225)        */
  int32_t chains_per_rank;  /* VERIFY: nc of the emulated MPI ranks; hosted ranks =
                               nchain / chains_per_rank, first = chain0 / chains_per_rank */
  int32_t sync;             /* SYNCSTEP                                              */
  double  pl, armin, armax, dfac, ifac;
  uint64_t seed;            /* Philox key (reference seed 8675309, mcpar.cc:271)     */
  int32_t coin_group;       /* NORMAL: chains sharing the local/remote coin: 0 = one coin per step for the
                               whole job ("one coin per rank", mcpar.cc:106-109, the rank being the job);
                               1..32 (power of 2) = one coin per group of consecutive chains */
  int32_t pool_m;           /* NORMAL: remote-mixture pool size; 0 = all chains      */
  int32_t thin;             /* keep every thin-th main step in the sample history    */
  int32_t trace;            /* VERIFY: steps of per-step accept/trial trace to keep (0 = none) */
  int64_t history_steps;    /* capacity of the device history in kept steps (0 = none).  NORMAL mode keeps
                               a RING of that many kept steps: a run may keep more (nsamp/thin >
                               history_steps); read or drain (mcgpu_history_attach_host*) the rows
                               before the ring overwrites them.  VERIFY holds the whole run.        */
  int32_t remote_mode;      /* NORMAL: how a remote step proposes (replaces MCPar::genRemote, mcpar.cc:315-451)
                               0 = the reference's algorithm: rejection-sample max_i Q_i over the pool,
                                   cfac = max_i Q_i(x)/max_i Q_i(x') with unnormalised Q_i (default);
                               1 = sum-mixture independence proposal: x' ~ (1/M) sum_i N(mu_i, diag sig2_i),
                                   cfac = q(x)/q(x') with normalised components, no rejection loop
                                   (Murray's proposal, SURVEY.md section 7 H1): O(M d) per remote step
                                   and exactly invariant, but not the reference's accept/reject sequence */
  int32_t pool_lag;         /* NORMAL: 0 = window w reads the pool published at the end of window w-1 (the
                               reference's staleness bound, mcpar.cc:127-140); 1 = one window older, which
                               takes the inter-GPU exchange off the critical path (remote steps start at
                               t >= 2 sync)                                                           */
} mcgpu_config;

typedef struct mcgpu_stats {
  int64_t burn_steps, main_steps;       /* steps taken so far                        */
  int64_t accepted, tried;              /* main phase, all hosted chains             */
  int64_t kernel_launches;              /* engine kernels launched since create      */
  int64_t remote_steps;                 /* VERIFY: rank-steps that took the remote branch;
                                           NORMAL: chain-steps of the main phase that did   */
  int64_t remote_iterations;            /* VERIFY: lock-step rejection iterations;
                                           NORMAL: candidates tried by those chain-steps
                                           (iterations of the loop mcpar.cc:331-409)        */
  int64_t history_rows;                 /* rows produced so far (kept steps * chains); the device ring
                                           holds the last history_steps kept steps of them  */
  double  device_ms;                    /* CUDA-event time of burnin+sample calls    */
  int64_t exchange_wait_ns;             /* peer-to-peer exchange: time the window kernels' first CTA spent
                                           waiting for the peers' pool slots (globaltimer)   */
  int64_t exchange_waits;               /* ... and how many launches had to wait at all      */
  int64_t exact_fallbacks;              /* remote candidates / steps whose fp32 bounds did not settle the
                                           decision and were redone exactly in fp64 (DESIGN.md section 3.1) */
} mcgpu_stats;

const char *mcgpu_version(void);
int  mcgpu_device_count(void);
const char *mcgpu_last_error(const mcgpu_engine *e);    /* e may be NULL: last create error */

int  mcgpu_create(const mcgpu_config *cfg, mcgpu_engine **out);
int  mcgpu_destroy(mcgpu_engine *e);

/* Run everything on the caller's CUDA stream (a cudaStream_t passed as void*; NULL is
 * the legacy default stream).  Without this call the engine uses a private
 * non-blocking stream. */
int  mcgpu_set_stream(mcgpu_engine *e, void *cuda_stream);

/* VLFunc &L argument of MCPar::run. */
int  mcgpu_set_likelihood(mcgpu_engine *e, int lik, const double *par, int npar);

/* A user-written likelihood inside the fused step kernels: cubin_path is a plugin built from one user header
 * (include/mcgpu_plugin.cuh, `python -m mcpar_b200.plugin`); par[npar] is copied to the device and handed to
 * the functor unchanged.  The engine then runs as with a built-in likelihood (lik = MCGPU_DEVICE_PLUGIN).
 * NORMAL mode, thread-per-chain kernels (even nparam <= 16).  MCGPU_EINVAL, before any launch, when the file
 * cannot be loaded, the plugin was built for another nparam or from other kernel sources (its stamp), or the
 * mode is VERIFY / REPLAY_LOCAL. */
int  mcgpu_set_likelihood_plugin(mcgpu_engine *e, const char *cubin_path, const double *par, int npar);

/* MCPar::covar_setup (mcpar.cc:454-484): incov is d x d row-major symmetric PD, or
 * NULL for the identity; the lower Cholesky factor is taken on the host (one-off,
 * d <= 64) and becomes the device-resident proposal factor. */
int  mcgpu_set_covariance(mcgpu_engine *e, const double *incov);

/* pinit of MCPar::run (mcpar.cc:47-53): nchain*nparam reals, chain-major; copies
 * them in and evaluates the initial log-likelihoods on the device. */
int  mcgpu_set_state(mcgpu_engine *e, const double *pinit);

/* VERIFY / REPLAY_LOCAL: the pre-generated streams of hosted rank `local_rank`
 * (normals Z, uniforms U in [0,1), ints I in [0,nchain_total)); copied to the device. */
int  mcgpu_set_streams(mcgpu_engine *e, int local_rank, const double *Z, size_t nz,
                       const double *U, size_t nu, const int32_t *I, size_t ni);

/* Burn-in loop of MCPar::run (mcpar.cc:56-97), including acceptance-rate tuning. */
int  mcgpu_burnin(mcgpu_engine *e, int nburn);

/* Main loop of MCPar::run (mcpar.cc:100-210).  begin resets the running moments;
 * sample advances nsteps steps (asynchronously on the engine's stream).  When the
 * engine hosts ALL chains the exchange is internal.  When chains are sharded over
 * several engines (nchain < nchain_total) the caller drives the exchange: a sample
 * call may not cross a multiple of `sync`; at each multiple call exchange_begin,
 * all-gather the returned buffer in place across engines (each engine's own slice
 * is [own_offset, own_offset+own_bytes)), then exchange_end. */
int  mcgpu_sample_begin(mcgpu_engine *e, int nsamp);
int  mcgpu_sample(mcgpu_engine *e, int nsteps);
/* The same for `world` peer-to-peer engines driven by ONE host thread (mcgpu_p2p_attach_local): the
 * windows of all engines are enqueued in turn, one exchange window at a time.  A window kernel that waits
 * for its peers' publications is then never queued in front of the launches that make them; engines
 * attached with attach_local refuse an mcgpu_sample call that would cross a multiple of `sync`. */
int  mcgpu_sample_group(mcgpu_engine *const *engines, int world, int nsteps);
int  mcgpu_exchange_begin(mcgpu_engine *e, void **dev_buffer, size_t *total_bytes,
                          size_t *own_offset, size_t *own_bytes);
int  mcgpu_exchange_end(mcgpu_engine *e);

/* Host-callback likelihood (SURVEY.md 8f: what a user-written VLFunc such as the R-backed RFunc of
 * src/rfunc.cc:48-67 needs).  After mcgpu_set_likelihood(e, MCGPU_HOST_LIKELIHOOD, NULL, 0) the step is split
 * around the plugin call, exactly where MCPar::run makes it (src/mcpar.cc:59-60, :151-160):
 *   mcgpu_set_state_host   pinit AND the caller's L(nchain, pinit, lylast) (mcpar.cc:47-53)
 *   mcgpu_step_propose     one step's trial points -- genLocal / genRemote with the normal mode's counter-based
 *                          draws -- copied to the host, ptrial [nchain][nparam]
 *   (the caller evaluates its VLFunc: L(nchain, ptrial, lytrial))
 *   mcgpu_step_accept      lytrial [nchain] in; accept test, state update, running moments, sample store,
 *                          pool publication; burn-in tuning at its boundaries
 * nburn burn-in steps come first, then mcgpu_sample_begin and nsamp main steps.  One engine hosting every chain
 * (no sharding); any nparam <= 64; both remote modes.  mcgpu_burnin / mcgpu_sample refuse such an engine. */
int  mcgpu_set_state_host(mcgpu_engine *e, const double *pinit, const double *lylast);
int  mcgpu_step_propose(mcgpu_engine *e, double *ptrial);
int  mcgpu_step_accept(mcgpu_engine *e, const double *lytrial);

/* Peer-to-peer exchange between sharded engines (replaces MPI_Allgather(MPI_IN_PLACE),
 * src/mcpar.cc:127-140, without a collective call): after attaching, the window
 * kernels store the published (mu, sigma^2) slots directly into every peer GPU's
 * next pool buffer over NVLink and signal an arrival counter there; the next
 * window's kernel waits for the arrivals on the device.  mcgpu_sample may then
 * cross multiples of `sync` and the exchange_begin/end calls are not used.  All
 * engines must make the same sequence of sample calls.  Engines host equal
 * contiguous blocks (chain0 = rank*nchain).  Attach before the first
 * mcgpu_sample_begin.  mcgpu_synchronize returns MCGPU_EPEER if a window waited
 * longer than ~10 s for a peer.
 *  - one process per GPU: export a handle (cudaIpcMemHandle_t, MCGPU_P2P_HANDLE_BYTES),
 *    all-gather the handles in rank order by any host means, attach;
 *  - one process, several engines (same or different devices): attach_local. */
#define MCGPU_P2P_HANDLE_BYTES 64
int  mcgpu_p2p_export(mcgpu_engine *e, void *handle, size_t nbytes);
int  mcgpu_p2p_attach(mcgpu_engine *e, int world, int rank, const void *handles);
int  mcgpu_p2p_attach_local(mcgpu_engine *const *engines, int world);

/* Burn-in tuning across sharded engines: device address of this engine's
 * {accepted, tried} int64 pair for the current tuning window (sum it across
 * engines between mcgpu_burnin calls that end on a tuning boundary). */
int  mcgpu_tuning_counters(mcgpu_engine *e, void **dev_counts);
/* Sharded burn-in: advance at most nmax steps without crossing a tuning boundary
 * (isamp = 51, 101, ... mcpar.cc:78,95); *tune_pending is set when the call ended on
 * one: all-reduce (sum) the tuning counters across engines, then mcgpu_tune. */
int  mcgpu_burnin_some(mcgpu_engine *e, int nmax, int *ndone, int *tune_pending);
int  mcgpu_tune(mcgpu_engine *e);
/* The same for `world` sharded engines living in ONE process (one per GPU): burn all of
 * them in, summing the counters across engines on the host at each tuning boundary. */
int  mcgpu_burnin_group(mcgpu_engine *const *engines, int world, int nburn);

int  mcgpu_synchronize(mcgpu_engine *e);

/* State export (all optional, host buffers): pvals/mu/sig/psum2 [nchain][nparam],
 * lylast [nchain]. */
int  mcgpu_get_state(mcgpu_engine *e, double *pvals, double *lylast, double *mu, double *sig,
                     double *psum2);
/* the (tuned) proposal factor of hosted rank local_rank, d x d row-major */
int  mcgpu_get_factor(mcgpu_engine *e, int local_rank, double *factor);
/* VERIFY: hosted rank's (mu,sigma^2) table musigall [nchain_total][nparam][2];
 * NORMAL: the current pool [pool_m][nparam][2] (local_rank ignored). */
int  mcgpu_get_musig(mcgpu_engine *e, int local_rank, double *musig);
/* VERIFY trace of hosted rank: accept [T][C] bytes, trial_ly [T][C], trial_p [T][C][d],
 * cfac [T][C], remote [T] bytes, iters [T] int32, cursors [3] (consumed Z,U,I). */
int  mcgpu_get_trace(mcgpu_engine *e, int local_rank, uint8_t *accept, double *trial_ly,
                     double *trial_p, double *cfac, uint8_t *remote, int32_t *iters,
                     int64_t *cursors);

/* Sample history = what MCout holds (src/mcout.cc:129-145): rows (p..., logL), kept
 * step major, then hosted chain.  read copies kept steps [first, first+count) to the
 * host through pinned staging buffers on a side stream. */
int  mcgpu_history_read(mcgpu_engine *e, int64_t first_step, int64_t count, double *rows);
/* Attach a host sink [capacity_steps][nchain][nparam+1] (pinned, or page-locked here):
 * from now on every mcgpu_sample call drains the rows it produced to the sink with
 * asynchronous copies on a side stream, overlapping the next window's compute (what
 * MCout::output/collect do with MPI_Gather, mcout.cc:30-94).  mcgpu_synchronize waits
 * for the drain.  NULL detaches. */
int  mcgpu_history_attach_host(mcgpu_engine *e, double *rows, size_t capacity_steps);
/* The same with fp32 rows -- the element type of the reference's MCout (src/mcout.hh:21-23 holds
 * floats): the rows are narrowed on the device and half the bytes cross PCIe.  The device history
 * (mcgpu_history_read, maxlike, moments) stays fp64. */
int  mcgpu_history_attach_host_f32(mcgpu_engine *e, float *rows, size_t capacity_steps);
/* MCout::maxlike's local part (mcout.cc:96-127): arg-max of logL over the stored
 * history; out = nparam parameters then the value. */
int  mcgpu_history_maxlike(mcgpu_engine *e, double *out);
/* posterior moments accumulated over the stored history on the device:
 * mean[d], cov[d][d] over all rows (for checks that cannot afford the D2H). */
int  mcgpu_history_moments(mcgpu_engine *e, double *mean, double *cov);

/* Checkpoint / restart (NORMAL mode; the reference has none).  The blob holds the chain state, the
 * running moments, the tuned proposal factor, the counters, the exchange pools and the schedule;
 * an engine created with the same configuration and likelihood continues the run bit for bit after
 * load (with a peer-to-peer exchange, all peers restore the same checkpoint).  The sample history
 * is not part of it: rows kept before the checkpoint must have been read or drained (after a load,
 * history_read / maxlike / moments see only rows produced since).  With a peer-to-peer exchange every
 * peer must have finished its load (a barrier) before any peer samples again. */
int  mcgpu_checkpoint_size(mcgpu_engine *e, size_t *bytes);
int  mcgpu_checkpoint_save(mcgpu_engine *e, void *buf, size_t bytes);
int  mcgpu_checkpoint_load(mcgpu_engine *e, const void *buf, size_t bytes);

int  mcgpu_get_stats(mcgpu_engine *e, mcgpu_stats *out);

/* raw device addresses for orchestrators / benchmarks: 0 state x, 1 lylast, 2 mu,
 * 3 psum2, 4 history, 5 pool(current) */
int  mcgpu_device_ptr(mcgpu_engine *e, int which, void **ptr, size_t *bytes);

/* Batched log-likelihood on the device = VLFunc::operator()(npset,x,y)
 * (src/vlfunc.hh:11): x is npset*nparam chain-major, y is npset. */
int  mcgpu_loglik(int device, int lik, int nparam, const double *par, int npar, int npset,
                  const double *x, double *y);
/* The same for a plugin cubin (mcgpu_set_likelihood_plugin); nparam must be the plugin's. */
int  mcgpu_loglik_plugin(int device, const char *cubin_path, int nparam, const double *par, int npar, int npset,
                         const double *x, double *y);

/* mcutil::qriguess (src/mcutil.cc:3-34): Sobol points in the box [plo,phi],
 * rank skip-ahead; pout is npset*nparam chain-major on the host. */
int  mcgpu_qriguess(int device, int rank, int npset, int nparam, const double *plo,
                    const double *phi, double *pout);
/* qriguess straight into the engine (no host round trip): chain g of the job starts at Sobol point
 * `first_point + g` of the nparam-dimensional sequence scaled into the box [plo, phi] -- what
 * qriguess(rank, npset, ...) gives rank = chain0 / npset (mcutil.cc:16-31; first_point = 0).  Replaces
 * mcgpu_set_state for runs of >= 1M chains without a hand-made pinit; nparam <= 64. */
int  mcgpu_set_state_sobol(mcgpu_engine *e, const double *plo, const double *phi, uint64_t first_point);

/* FP64 DFMA micro-benchmark used for the roofline denominator: returns the measured
 * TFLOP/s (2 flops per DFMA) of `iters` dependent-chain DFMAs per thread. */
int  mcgpu_measure_fp64_peak(int device, double *tflops);

#ifdef __cplusplus
}
#endif
#endif
