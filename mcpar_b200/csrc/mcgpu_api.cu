// mcgpu_api.cu -- the extern "C" boundary (include/mcgpu.h) and the host-side engine
// that sequences the fused step kernels: it replaces the control flow of
// MCPar::run (reference src/mcpar.cc:17-214) with device-resident multi-step launches.
//
// There is no CPU compute path in this file: every numerical result comes from a
// kernel in mh_fast.cu / mh_exact.cu, and every entry point fails with
// MCGPU_ENODEVICE / MCGPU_ECUDA when no device is usable.
#include "../../include/mcgpu.h"
#include "mh_launch.h"
#include "mcgpu_sobol.h"
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <string>
#include <vector>
#include <deque>
#include <algorithm>

#ifndef MCGPU_KERNEL_STAMP
#error "build with mcpar_b200/build.py: it passes -DMCGPU_KERNEL_STAMP (the stamp plugins must carry)"
#endif

using namespace mcgpu;

namespace {

thread_local std::string g_create_err;

struct StreamSet { std::vector<double> Z, U; std::vector<int32_t> I; };

}  // namespace

struct mcgpu_engine {
  mcgpu_config cfg;
  int d = 0;
  long long C = 0, ld = 0, N = 0;
  bool sharded = false, verify = false, replay_local = false;
  int dev = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr, side = nullptr;
  std::string err;

  // likelihood
  int lik = -1; int lik_k = 0; double lp[8] = {0}; double *lik_dev = nullptr;
  cudaLibrary_t plugin = nullptr; cudaKernel_t pk[8] = {};   // MCGPU_DEVICE_PLUGIN: the loaded cubin, kernels by PH_* / PK_*

  // NORMAL / REPLAY_LOCAL state (SoA) or VERIFY state (AoS per rank)
  double *x = nullptr, *ly = nullptr, *mu = nullptr, *ps = nullptr;
  double *factor = nullptr;
  unsigned long long *counts = nullptr;   // [0,1] window, [2,3] cumulative, [4,5] main-phase stats, [6,7] remote chain-steps / candidate iterations, [8,9] exchange wait ns / waits, [10] exact-path fallbacks of the bounded tests
  // exchange region (one allocation, IPC-exportable): NPOOL pool buffers [M][d][2] + the arrival counter
  char *xchg = nullptr; size_t pool_bytes = 0, xchg_bytes = 0;
  double *pool[4] = {nullptr, nullptr, nullptr, nullptr}; int M = 0; long long stride = 1; bool pool_in_smem = true;
  long long npub = 0;                      // publications completed since create: publication k lives in pool[k % nbuf]
  int lag = 0, remote_mode = 0;            // cfg.pool_lag, cfg.remote_mode
  bool p2p = false, p2p_local = false; int p2p_world = 0; char **peers_d = nullptr; std::vector<void*> peer_opened; int *xflag_d = nullptr;
  // sample history: a ring of hist_cap kept steps; kept step k lives in ring row k % hist_cap
  double *hist = nullptr; long long hist_cap = 0, hist_kept = 0, hist_valid_from = 0;
  int *overrun = nullptr;
  double *Zd = nullptr, *Ud = nullptr; int *Id = nullptr; long long nz = 0, nu = 0, ni = 0;

  // host-callback likelihood (MCGPU_HOST_LIKELIHOOD): AoS state, one step per propose / accept pair
  bool hostlik = false, proposed = false; double *aux = nullptr, *lytrial_d = nullptr; int *flags_d = nullptr;   // (ptrial: below)
  // wide kernels (d >= 8, job-wide coin): AoS state, column-major factor, prepared pool, transposed GaussMix
  bool wide = false;
  double *factor_cm = nullptr; int *diag_d = nullptr;
  double *pprep = nullptr; int mpad = 0;
  double *gm_t = nullptr; int kpad = 0;

  // VERIFY extras
  int Cr = 0, Rl = 0, R = 0, rank0 = 0;
  double *ptrial = nullptr, *sig = nullptr, *mutrial = nullptr, *sigtrial = nullptr, *musig = nullptr;
  double *snap[2] = {nullptr, nullptr}; int snap_cur = 0;
  long long *soff = nullptr, *cursors = nullptr; int *irate_d = nullptr;
  unsigned long long *rstats = nullptr;
  std::vector<StreamSet> host_streams; bool streams_dirty = false;
  uint8_t *tr_accept = nullptr, *tr_remote = nullptr; double *tr_trial_ly = nullptr, *tr_trial_p = nullptr, *tr_cfac = nullptr;
  int *tr_iters = nullptr; int trace_cap = 0;

  // schedule
  bool have_state = false, have_factor = false, sampling = false, exchange_pending = false, tune_pending = false;
  long long burn_done = 0, t_main = 0; int nsamp = 0; int irate = 50; int nburn_total = 0;
  long long launches = 0;
  std::deque<std::pair<cudaEvent_t, cudaEvent_t>> timers; std::vector<cudaEvent_t> ev_free; double ms_accum = 0.0;

  // pinned staging for history reads
  double *pin[2] = {nullptr, nullptr}; size_t pin_bytes = 0; cudaEvent_t pin_ev[2] = {nullptr, nullptr};

  // host sink of the sample history: rows drain to it on the side stream as windows finish
  double *sink = nullptr; size_t sink_rows_cap = 0; long long sink_sent = 0; bool sink_registered = false;
  bool sink_f32 = false; float *hist_f32 = nullptr;       // fp32 sink (the reference's MCout element type): device mirror of the history
  cudaEvent_t sink_ev = nullptr;
  std::deque<std::pair<long long, cudaEvent_t>> drains;   // (kept steps drained once the event completes, event on the side stream)
};

namespace {

#define CK(call)                                                                         \
  do {                                                                                   \
    cudaError_t _s = (call);                                                             \
    if (_s != cudaSuccess) {                                                             \
      char _b[512];                                                                      \
      snprintf(_b, sizeof _b, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_s)); \
      e->err = _b;                                                                       \
      return _s == cudaErrorMemoryAllocation ? MCGPU_ENOMEM : MCGPU_ECUDA;               \
    }                                                                                    \
  } while (0)

int fail(mcgpu_engine *e, int code, const char *msg) { if (e) e->err = msg; else g_create_err = msg; return code; }

template <class T> int dalloc(mcgpu_engine *e, T **p, size_t n, bool zero = true)
{
  CK(cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T)));
  if (zero) CK(cudaMemsetAsync(*p, 0, std::max<size_t>(n, 1) * sizeof(T), e->stream));
  return 0;
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// device time of the burnin / sample calls: event pairs, harvested without blocking as they complete and recycled
cudaEvent_t event_get(mcgpu_engine *e, unsigned flags = cudaEventDefault)
{
  cudaEvent_t ev = nullptr;
  if (flags == cudaEventDefault && !e->ev_free.empty()) { ev = e->ev_free.back(); e->ev_free.pop_back(); return ev; }
  cudaEventCreateWithFlags(&ev, flags);
  return ev;
}
void timers_harvest(mcgpu_engine *e, bool block)
{
  while (!e->timers.empty()) {
    auto &t = e->timers.front();
    if (block) cudaEventSynchronize(t.second);
    else if (cudaEventQuery(t.second) != cudaSuccess) { cudaGetLastError(); break; }
    float ms = 0;
    if (cudaEventElapsedTime(&ms, t.first, t.second) == cudaSuccess) e->ms_accum += ms; else cudaGetLastError();
    e->ev_free.push_back(t.first); e->ev_free.push_back(t.second);
    e->timers.pop_front();
  }
}
void timer_begin(mcgpu_engine *e)
{
  timers_harvest(e, false);
  cudaEvent_t a = event_get(e), b = event_get(e);
  cudaEventRecord(a, e->stream);
  e->timers.emplace_back(a, b);
}
void timer_end(mcgpu_engine *e) { cudaEventRecord(e->timers.back().second, e->stream); }
void timers_resolve(mcgpu_engine *e) { timers_harvest(e, true); }

// lower Cholesky factor of a row-major SPD matrix in place (replaces spotrf('U') on the
// column-major view, mcpar.cc:475-480); the strict upper triangle keeps its input
int cholesky_lower(int d, double *a)
{
  for (int i = 0; i < d; ++i)
    for (int j = 0; j <= i; ++j) {
      double sum = a[i * d + j];
      for (int k = 0; k < j; ++k) sum -= a[i * d + k] * a[j * d + k];
      if (i == j) { if (!(sum > 0)) return i + 1; a[i * d + i] = sqrt(sum); }
      else a[i * d + j] = sum / a[j * d + j];
    }
  return 0;
}

// Pool buffers rotate with the publication count.  Two suffice when the exchange is stream-ordered (one
// engine, or a caller-driven all-gather).  The peer-to-peer exchange needs three: a GPU that has all of
// publication P may write publication P+1 into its peers while their last CTAs of the window that
// produced P still read pool P-1 -- so P+1 must not alias P-1.  (Every main-phase launch waits for the
// arrivals of the pool it is entitled to read, so no GPU is ever more than one publication ahead.)
// With pool_lag = 1 a window reads the publication BEFORE the newest one, so one more buffer stays live.
enum { NPOOL = 4 };
int pool_nbuf(const mcgpu_engine *e) { return (e->p2p ? 3 : 2) + e->lag; }
long long pool_read_index(const mcgpu_engine *e) { return std::max<long long>(e->npub - e->lag, 0); }
double *pool_cur(const mcgpu_engine *e) { return e->pool[pool_read_index(e) % pool_nbuf(e)]; }       // what this window reads
double *pool_newest(const mcgpu_engine *e) { return e->pool[e->npub % pool_nbuf(e)]; }                 // the latest publication
double *pool_next(const mcgpu_engine *e) { return e->pool[(e->npub + 1) % pool_nbuf(e)]; }
int arrivals_per_slot(const mcgpu_engine *e) { return e->wide ? e->d / 2 : 1; }   // the wide kernel's lanes arrive one by one

// peer-to-peer exchange: where this launch publishes and what it waits for
void fill_p2p(const mcgpu_engine *e, StepParams &p)
{
  if (!e->p2p) return;
  p.peers = e->peers_d; p.npeers = e->p2p_world;
  p.next_off = (long long)(((e->npub + 1) % pool_nbuf(e)) * e->pool_bytes); p.arr_off = (long long)(NPOOL * e->pool_bytes);
  p.arrivals = reinterpret_cast<const unsigned long long*>(e->xchg + NPOOL * e->pool_bytes);
  const unsigned long long per_pub = (unsigned long long)e->M * arrivals_per_slot(e);
  p.wait_target = per_pub * (unsigned long long)pool_read_index(e);     // readers: the publication this window reads
  p.pub_wait_target = per_pub * (unsigned long long)e->npub;            // publishers: never more than one publication ahead
  p.xflag = e->xflag_d;
}

void fill_step_params(mcgpu_engine *e, StepParams &p)
{
  memset(&p, 0, sizeof p);
  p.x = e->x; p.ly = e->ly; p.mu = e->mu; p.ps = e->ps;
  p.C = e->C; p.ld = e->ld; p.chain0 = e->cfg.chain0;
  p.factor = e->factor;
  p.key0 = (uint32_t)e->cfg.seed; p.key1 = (uint32_t)(e->cfg.seed >> 32);
  for (int r = 0; r < 10; ++r) { p.rk[2 * r] = p.key0 + (uint32_t)r * 0x9E3779B9u; p.rk[2 * r + 1] = p.key1 + (uint32_t)r * 0xBB67AE85u; }
  p.sync = e->cfg.sync; p.coin_group = e->cfg.coin_group; p.pl = e->cfg.pl;
  p.first_remote_t = e->cfg.sync * (1 + e->lag);
  p.hist_cap = (int)std::max<long long>(e->hist_cap, 1);
  p.pool_m = e->M; p.pool_stride = e->stride; p.pool_in_smem = e->pool_in_smem;
  p.thin = e->cfg.thin;
  static const int exact_tests = getenv("MCGPU_EXACT_TESTS") ? atoi(getenv("MCGPU_EXACT_TESTS")) : 0;
  p.exact_tests = exact_tests;
  p.Z = e->Zd; p.U = e->Ud; p.nz = e->nz; p.nu = e->nu; p.overrun = e->overrun;
  memcpy(p.lp, e->lp, sizeof p.lp); p.lik_dev = e->lik_dev; p.lik_k = e->lik_k;
  p.nburn_total = e->nburn_total;
}

// ---- device likelihood plugins (mh_plugin.cu compiled per user header into a cubin) --------------------------
enum { PK_INIT = 6, PK_EVAL = 7 };           // plugin kernels beyond the six step phases PH_*

// The one place that knows the plugin's symbol names: mh_plugin.cu instantiates mcgpu::fast::mh_steps_kernel
// <MCGPU_DEVICE_PLUGIN, d, RNG_PHILOX = 0, phase> and init_loglik_kernel<MCGPU_DEVICE_PLUGIN, d>.
std::string plugin_kernel_name(int d, int which)
{
  char b[128];
  if (which == PK_EVAL) return "mcgpu_plugin_loglik";
  if (which == PK_INIT) snprintf(b, sizeof b, "_ZN5mcgpu4fast18init_loglik_kernelILi%dELi%dEEEvNS_10StepParamsE", MCGPU_DEVICE_PLUGIN, d);
  else snprintf(b, sizeof b, "_ZN5mcgpu4fast15mh_steps_kernelILi%dELi%dELi0ELi%dEEEvNS_10StepParamsE", MCGPU_DEVICE_PLUGIN, d, which);
  return b;
}

// Load a plugin cubin into the current device's context and check it before anything launches from it: it must
// have been compiled from the kernel sources this library was (StepParams crosses by value) and for d parameters.
int plugin_open(const char *path, int d, cudaLibrary_t *lib, cudaKernel_t k[8], std::string &err)
{
  *lib = nullptr;
  FILE *f = path ? fopen(path, "rb") : nullptr;
  if (!f) { err = std::string("plugin: cannot open '") + (path ? path : "(null)") + "'"; return MCGPU_EINVAL; }
  fclose(f);
  cudaLibrary_t L = nullptr;
  cudaError_t s = cudaLibraryLoadFromFile(&L, path, nullptr, nullptr, 0, nullptr, nullptr, 0);
  if (s != cudaSuccess) { cudaGetLastError(); err = std::string("plugin: cannot load '") + path + "': " + cudaGetErrorString(s); return MCGPU_EINVAL; }
  void *ps = nullptr, *pn = nullptr; size_t bs = 0, bn = 0;
  unsigned long long stamp = 0; int np = 0;
  if (cudaLibraryGetGlobal(&ps, &bs, L, "mcgpu_plugin_stamp") != cudaSuccess || bs != sizeof stamp ||
      cudaLibraryGetGlobal(&pn, &bn, L, "mcgpu_plugin_nparam") != cudaSuccess || bn != sizeof np ||
      cudaMemcpy(&stamp, ps, sizeof stamp, cudaMemcpyDeviceToHost) != cudaSuccess ||
      cudaMemcpy(&np, pn, sizeof np, cudaMemcpyDeviceToHost) != cudaSuccess) {
    cudaGetLastError(); cudaLibraryUnload(L);
    err = std::string("plugin: '") + path + "' is not a likelihood plugin (no mcgpu_plugin_stamp / mcgpu_plugin_nparam)";
    return MCGPU_EINVAL;
  }
  char b[256];
  if (stamp != (unsigned long long)MCGPU_KERNEL_STAMP) {
    snprintf(b, sizeof b, "plugin: kernel-source stamp %016llx differs from this library's %016llx: rebuild the plugin",
             stamp, (unsigned long long)MCGPU_KERNEL_STAMP);
    cudaLibraryUnload(L); err = b; return MCGPU_EINVAL;
  }
  if (np != d) {
    snprintf(b, sizeof b, "plugin: built for nparam = %d, the engine has nparam = %d", np, d);
    cudaLibraryUnload(L); err = b; return MCGPU_EINVAL;
  }
  for (int w = 0; w < 8; ++w)
    if (cudaLibraryGetKernel(&k[w], L, plugin_kernel_name(d, w).c_str()) != cudaSuccess) {
      cudaGetLastError(); cudaLibraryUnload(L);
      err = "plugin: kernel " + plugin_kernel_name(d, w) + " missing from the cubin";
      return MCGPU_EINVAL;
    }
  *lib = L;
  return MCGPU_OK;
}

void plugin_release(mcgpu_engine *e)
{
  if (e->plugin) cudaLibraryUnload(e->plugin);
  e->plugin = nullptr;
}

cudaError_t launch_plugin(mcgpu_engine *e, int which, const StepParams &p, unsigned grid, unsigned block, size_t smem)
{
  const void *f = reinterpret_cast<const void *>(e->pk[which]);
  if (smem > 48 * 1024) {                            // per launch: the attribute is per device
    cudaError_t s = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (s != cudaSuccess) return s;
  }
  void *args[] = {const_cast<StepParams *>(&p)};
  return cudaLaunchKernel(f, dim3(grid), dim3(block), args, smem, e->stream);
}

// the grid, block and shared-memory rules of launch_lik_d (mh_dispatch.inl)
cudaError_t launch_plugin_steps(mcgpu_engine *e, int phase, const StepParams &p)
{
  const int block = fast::step_block();
  const size_t smem = fast::steps_smem_bytes(e->d, p.nsteps, p.pool_m, phase != PH_BURN && phase != PH_LOCAL);
  return launch_plugin(e, phase, p, (unsigned)((p.C + block - 1) / block), block, smem);
}

// initial log-likelihoods L(nchain, pvals, lylast), mcpar.cc:53, on the SoA state
cudaError_t launch_init_any(mcgpu_engine *e, const StepParams &p)
{
  if (e->lik == MCGPU_DEVICE_PLUGIN) return launch_plugin(e, PK_INIT, p, (unsigned)((p.C + 255) / 256), 256, 0);
  return (e->replay_local ? exact::launch_init_loglik : fast::launch_init_loglik)(e->lik, e->d, p, e->stream);
}

cudaError_t launch_steps_any(mcgpu_engine *e, int phase, const StepParams &p)
{
  ++e->launches;
  if (e->wide) {
    WideParams w; memset(&w, 0, sizeof w);
    w.x = p.x; w.ly = p.ly; w.mu = p.mu; w.ps = p.ps; w.C = p.C; w.chain0 = p.chain0;
    w.factor_cm = e->factor_cm; w.factor_rm = e->factor; w.diagonal = e->diag_d; w.counts = p.counts;
    w.key0 = p.key0; w.key1 = p.key1; memcpy(w.rk, p.rk, sizeof w.rk); w.step0 = p.step0; w.nsteps = p.nsteps; w.t0 = p.t0;
    w.pmh = reinterpret_cast<const double2*>(e->pprep); w.psd = e->pprep + (size_t)2 * e->d * e->mpad;
    w.pool_m = e->M; w.mpad = e->mpad; w.pool_next = p.pool_next; w.pool_stride = p.pool_stride;
    w.peers = p.peers; w.npeers = p.npeers; w.next_off = p.next_off; w.arr_off = p.arr_off;
    w.arrivals = p.arrivals; w.wait_target = p.wait_target; w.pub_wait_target = p.pub_wait_target; w.xflag = p.xflag;   // readers wait in pool_prep, publishers in the kernel
    w.xstat = p.xstat;
    w.hist = p.hist; w.thin = p.thin; w.hist_cap = p.hist_cap; w.hist_ring0 = p.hist_ring0;
    w.pnb = e->pprep + (size_t)3 * e->d * e->mpad; w.summix = e->remote_mode; w.exact_tests = p.exact_tests;
    w.pf = reinterpret_cast<const float2*>(e->pprep + ((size_t)3 * e->d + 1) * e->mpad);        // fp32 copy behind the fp64 arrays
    w.pnbf = reinterpret_cast<const float*>(w.pf + (size_t)e->d * e->mpad); w.pscal = w.pnbf + e->mpad;
    w.gm2 = reinterpret_cast<const double2*>(e->gm_t);
    w.gm_lw = e->gm_t ? e->gm_t + (size_t)2 * e->d * e->kpad : nullptr; w.kpad = e->kpad;
    return fast::launch_wide(e->lik, e->d, phase == PH_REMOTE && e->remote_mode == 1 ? PH_REMOTE_SUM : phase, w, e->stream);
  }
  if (e->replay_local) return exact::launch_steps(e->lik, e->d, 1, phase == PH_BURN ? PH_BURN : PH_LOCAL, p, e->stream);
  if (e->remote_mode == 1) phase = phase == PH_MIXED ? PH_MIXED_SUM : (phase == PH_REMOTE ? PH_REMOTE_SUM : phase);
  if (e->lik == MCGPU_DEVICE_PLUGIN) return launch_plugin_steps(e, phase, p);
  return fast::launch_steps(e->lik, e->d, 0, phase, p, e->stream);
}

// Host copy of the device's Philox4x32-10 (mcgpu_device.cuh): with a job-wide coin the host
// evaluates each step's local/remote draw itself and plans PH_LOCAL / PH_REMOTE launches
// without a device round trip.
double host_coin(const mcgpu_engine *e, uint32_t step)
{
  // the coin is word 2*NP+1 of chain 0's local stream (mcgpu_device.cuh "draws")
  const int np = (e->d + 1) / 2, idx = 2 * np + 1;
  uint32_t c0 = 0, c1 = 0, c2 = step, c3 = (uint32_t)(idx / 4);
  uint32_t k0 = (uint32_t)e->cfg.seed, k1 = (uint32_t)(e->cfg.seed >> 32);
  for (int r = 0; r < 10; ++r) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0, p1 = (unsigned long long)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  const uint32_t w[4] = {c0, c1, c2, c3};
  return (double)w[idx % 4] * (1.0 / 4294967296.0);
}

int upload_streams(mcgpu_engine *e)
{
  if (!e->streams_dirty) return 0;
  const int nr = (int)e->host_streams.size();
  std::vector<long long> soff((size_t)nr * 6);
  size_t tz = 0, tu = 0, ti = 0;
  for (int r = 0; r < nr; ++r) {
    auto &s = e->host_streams[r];
    soff[r * 6 + 0] = (long long)tz; soff[r * 6 + 1] = (long long)s.Z.size(); tz += s.Z.size();
    soff[r * 6 + 2] = (long long)tu; soff[r * 6 + 3] = (long long)s.U.size(); tu += s.U.size();
    soff[r * 6 + 4] = (long long)ti; soff[r * 6 + 5] = (long long)s.I.size(); ti += s.I.size();
  }
  if (e->Zd) cudaFree(e->Zd);
  if (e->Ud) cudaFree(e->Ud);
  if (e->Id) cudaFree(e->Id);
  e->Zd = e->Ud = nullptr; e->Id = nullptr;
  CK(cudaMalloc((void**)&e->Zd, std::max<size_t>(tz, 1) * 8));
  CK(cudaMalloc((void**)&e->Ud, std::max<size_t>(tu, 1) * 8));
  CK(cudaMalloc((void**)&e->Id, std::max<size_t>(ti, 1) * 4));
  for (int r = 0; r < nr; ++r) {
    auto &s = e->host_streams[r];
    if (!s.Z.empty()) CK(cudaMemcpyAsync(e->Zd + soff[r * 6], s.Z.data(), s.Z.size() * 8, cudaMemcpyHostToDevice, e->stream));
    if (!s.U.empty()) CK(cudaMemcpyAsync(e->Ud + soff[r * 6 + 2], s.U.data(), s.U.size() * 8, cudaMemcpyHostToDevice, e->stream));
    if (!s.I.empty()) CK(cudaMemcpyAsync(e->Id + soff[r * 6 + 4], s.I.data(), s.I.size() * 4, cudaMemcpyHostToDevice, e->stream));
  }
  if (e->verify) CK(cudaMemcpyAsync(e->soff, soff.data(), soff.size() * 8, cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->nz = (long long)tz; e->nu = (long long)tu; e->ni = (long long)ti;
  e->streams_dirty = false;
  return 0;
}

void fill_verify_params(mcgpu_engine *e, VerifyParams &p)
{
  memset(&p, 0, sizeof p);
  p.d = e->d; p.C = e->Cr; p.N = (int)e->N; p.rank0 = e->rank0; p.nsamp = e->nsamp;
  p.L.lik = e->lik; p.L.d = e->d; p.L.k = e->lik_k; memcpy(p.L.lp, e->lp, sizeof p.L.lp); p.L.dev = e->lik_dev;
  p.pvals = e->x; p.ptrial = e->ptrial; p.ly = e->ly; p.mu = e->mu; p.sig = e->sig; p.ps = e->ps;
  p.mutrial = e->mutrial; p.sigtrial = e->sigtrial; p.factor = e->factor; p.musig = e->musig;
  p.Z = e->Zd; p.U = e->Ud; p.I = e->Id; p.soff = e->soff; p.cursors = e->cursors;
  p.counts = e->counts; p.irate = e->irate_d;
  p.sync = e->cfg.sync; p.pl = e->cfg.pl; p.armin = e->cfg.armin; p.armax = e->cfg.armax;
  p.dfac = e->cfg.dfac; p.ifac = e->cfg.ifac;
  p.hist = e->hist; p.hist_chains = e->C;
  p.tr_accept = e->tr_accept; p.tr_trial_ly = e->tr_trial_ly; p.tr_trial_p = e->tr_trial_p;
  p.tr_cfac = e->tr_cfac; p.tr_remote = e->tr_remote; p.tr_iters = e->tr_iters; p.trace_cap = e->trace_cap;
  p.overrun = e->overrun; p.rstats = e->rstats;
}

int check_overrun(mcgpu_engine *e)
{
  int flag = 0;
  CK(cudaMemcpyAsync(&flag, e->overrun, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  if (flag) return fail(e, MCGPU_ESTREAM, "a replay stream ran dry (or a remote step was requested in REPLAY_LOCAL mode)");
  return 0;
}

// ---- small utility kernels -------------------------------------------------
// history rows fp64 -> fp32 for the fp32 host sink (grid-stride)
__global__ void narrow_rows_kernel(const double *src, float *dst, size_t n)
{
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = (float)src[i];
}

__global__ void fill_kernel(double *dst, size_t n, double v)
{
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = v;
}

__global__ void argmax_rows_kernel(const double *rows, long long nrows, int ncol, double *best_val, long long *best_row)
{
  __shared__ double sv[256]; __shared__ long long sr[256];
  double bv = -INFINITY; long long br = -1;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (long long)gridDim.x * blockDim.x) {
    const double v = rows[r * ncol + ncol - 1];
    if (v > bv) { bv = v; br = r; }              // strict >: first occurrence wins (mcout.cc:138)
  }
  sv[threadIdx.x] = bv; sr[threadIdx.x] = br;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const double v = sv[threadIdx.x + o]; const long long r = sr[threadIdx.x + o];
      if (r >= 0 && (v > sv[threadIdx.x] || sr[threadIdx.x] < 0 || (v == sv[threadIdx.x] && r < sr[threadIdx.x]))) { sv[threadIdx.x] = v; sr[threadIdx.x] = r; }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { best_val[blockIdx.x] = sv[0]; best_row[blockIdx.x] = sr[0]; }
}

// sums of x_i (pair index < d) and x_i*x_j over all rows; one quantity per blockIdx.y
__global__ void moments_kernel(const double *rows, long long nrows, int d, double *out)
{
  __shared__ double ssum[256];
  const int q = blockIdx.y;
  int ci, cj = -1;
  if (q < d) ci = q;
  else { int k = q - d; ci = 0; while (k >= d - ci) { k -= d - ci; ++ci; } cj = ci + k; }
  double s = 0.0;
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < nrows; r += (long long)gridDim.x * blockDim.x) {
    const double a = rows[r * (d + 1) + ci];
    s += cj < 0 ? a : a * rows[r * (d + 1) + cj];
  }
  ssum[threadIdx.x] = s;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) { if (threadIdx.x < o) ssum[threadIdx.x] += ssum[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) atomicAdd(out + q, ssum[0]);
}

// Scalar q of the output is scalar first_scalar + q of the point-major Sobol stream (what vslSkipAheadStream +
// vsRngUniform deliver, mcutil.cc:22-25) scaled into the box of OUTPUT column q % d (mcutil.cc:28-32).
// ld = 0: chain-major output pout[q] (the host layout); ld > 0: the engine's SoA state pout[(q % d) * ld + q / d].
__global__ void sobol_box_kernel(const uint32_t *dirs, int d, unsigned long long first_scalar, size_t ntot,
                                 const double *plo, const double *phi, double *pout, long long ld)
{
  for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < ntot; q += (size_t)gridDim.x * blockDim.x) {
    const unsigned long long sc = first_scalar + (unsigned long long)q;
    const unsigned long long n = sc / (unsigned long long)d; const int k = (int)(sc % (unsigned long long)d);
    unsigned long long gray = n ^ (n >> 1);
    uint32_t xv = 0;
    for (int b = 0; gray && b < 32; ++b, gray >>= 1) if (gray & 1ull) xv ^= dirs[k * 32 + b];
    const double u = (double)xv * (1.0 / 4294967296.0);
    const int i = (int)(q % (size_t)d);
    const double v = __dadd_rn(plo[i], __dmul_rn(u, __dsub_rn(phi[i], plo[i])));   // mcutil.cc:31, no contraction
    if (ld > 0) pout[(size_t)i * ld + q / (size_t)d] = v; else pout[q] = v;
  }
}

__global__ void dfma_peak_kernel(double *out, int iters, double a, double b)
{
  double v0 = threadIdx.x, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3, v4 = v0 + 4, v5 = v0 + 5, v6 = v0 + 6, v7 = v0 + 7;
  for (int i = 0; i < iters; ++i) {
    v0 = fma(v0, a, b); v1 = fma(v1, a, b); v2 = fma(v2, a, b); v3 = fma(v3, a, b);
    v4 = fma(v4, a, b); v5 = fma(v5, a, b); v6 = fma(v6, a, b); v7 = fma(v7, a, b);
  }
  const double s = v0 + v1 + v2 + v3 + v4 + v5 + v6 + v7;
  if (s == 12345.678) out[0] = s;
}

__global__ void transpose_aos_to_soa(const double *aos, double *soa, long long C, long long ld, int d)
{
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= C) return;
  for (int i = 0; i < d; ++i) soa[i * ld + j] = aos[j * d + i];
}
__global__ void transpose_soa_to_aos(const double *soa, double *aos, long long C, long long ld, int d, double scale)
{
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= C) return;
  for (int i = 0; i < d; ++i) aos[j * d + i] = soa[i * ld + j] * scale;
}

// Sobol direction numbers, Joe & Kuo (2008), dimensions 1..64 (mcgpu_sobol.h, generated by tools/gen_sobol_table.py)
void sobol_dirs(int dim, uint32_t *v)
{
  if (dim == 0) { for (int i = 0; i < 32; ++i) v[i] = 1u << (31 - i); return; }
  const sobol_jk_t &p = SOBOL_JK[dim]; const int s = p.s;
  for (int i = 0; i < 32; ++i) {
    if (i < s) v[i] = p.m[i] << (31 - i);
    else {
      v[i] = v[i - s] ^ (v[i - s] >> s);
      for (int k = 1; k < s; ++k) v[i] ^= (((p.a >> (s - 1 - k)) & 1u) * v[i - k]);
    }
  }
}

int prepare_lik(int lik, int d, const double *par, int npar, double lp[8], std::vector<double> &dev, int &K, std::string &err)
{
  memset(lp, 0, 8 * sizeof(double)); K = 0; dev.clear();
  switch (lik) {
    case MCGPU_ROSENBROCK1:
      if (d < 2 || d % 2) { err = "N for Rosenbrock1 must be even and >= 2"; return MCGPU_EINVAL; }   // rosenbrock.hh:13-16
      return 0;
    case MCGPU_ROSENBROCK2:
      if (d < 2) { err = "N for Rosenbrock2 must be >= 2"; return MCGPU_EINVAL; }                      // rosenbrock.hh:27-30
      return 0;
    case MCGPU_GAUSSIAN:
      if (d != 2) { err = "Invalid specification.  N for Gaussian must == 2."; return MCGPU_EINVAL; }   // rosenbrock.hh:43
      if (par && npar < 4) { err = "Gaussian needs mu[2], sig2[2]"; return MCGPU_EINVAL; }
      for (int k = 0; k < 2; ++k) { lp[k] = par ? par[k] : 0.0; lp[2 + k] = par ? 1.0 / par[2 + k] : 1.0; }  // :44-47
      return 0;
    case MCGPU_DUALGAUSSIAN:
      if (d != 2) { err = "DualGaussian has two parameters"; return MCGPU_EINVAL; }
      lp[0] = (par && npar >= 1) ? par[0] : 5.0;
      lp[1] = log(lp[0]);                                   // the production kernels evaluate the sum in log-sum-exp form
      return 0;
    case MCGPU_GAUSSMIX: {
      if (!par || npar < 1) { err = "GaussMix needs par = K, mu, sig2, w"; return MCGPU_EINVAL; }
      K = (int)par[0];
      if (K < 1 || npar != 1 + 2 * K * d + K) { err = "GaussMix parameter block has the wrong length"; return MCGPU_EINVAL; }
      dev.resize((size_t)2 * K * d + K);
      const double *mu = par + 1, *s2 = mu + (size_t)K * d, *w = s2 + (size_t)K * d;
      for (int i = 0; i < K * d; ++i) { dev[i] = mu[i]; dev[(size_t)K * d + i] = 1.0 / s2[i]; }
      for (int k = 0; k < K; ++k) dev[(size_t)2 * K * d + k] = log(w[k]);
      return 0;
    }
  }
  err = "unknown likelihood id";
  return MCGPU_EINVAL;
}

}  // namespace

// ============================================================================
extern "C" {

const char *mcgpu_version(void) { return "mcpar-b200 0.1 (sm_100a, abi 1)"; }

int mcgpu_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

const char *mcgpu_last_error(const mcgpu_engine *e) { return e ? e->err.c_str() : g_create_err.c_str(); }

int mcgpu_create(const mcgpu_config *cfg, mcgpu_engine **out)
{
  if (!cfg || !out) return fail(nullptr, MCGPU_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->abi_version != MCGPU_ABI_VERSION) return fail(nullptr, MCGPU_EINVAL, "abi_version mismatch");
  if (cfg->nparam < 1 || cfg->nparam > MCGPU_MAX_D) return fail(nullptr, MCGPU_EINVAL, "nparam out of range (1..64)");
  if (cfg->nchain < 1 || cfg->nchain_total < cfg->nchain || cfg->chain0 < 0 || cfg->chain0 + cfg->nchain > cfg->nchain_total)
    return fail(nullptr, MCGPU_EINVAL, "inconsistent chain geometry");
  if (cfg->sync < 1) return fail(nullptr, MCGPU_EINVAL, "sync must be >= 1");
  if (cfg->thin < 1) return fail(nullptr, MCGPU_EINVAL, "thin must be >= 1");
  if (mcgpu_device_count() <= cfg->device || cfg->device < 0) return fail(nullptr, MCGPU_ENODEVICE, "no usable CUDA device (this engine has no CPU path)");

  mcgpu_engine *e = new mcgpu_engine();
  e->cfg = *cfg; e->d = cfg->nparam; e->C = cfg->nchain; e->N = cfg->nchain_total; e->dev = cfg->device;
  e->verify = cfg->mode == MCGPU_MODE_VERIFY; e->replay_local = cfg->mode == MCGPU_MODE_REPLAY_LOCAL;
  e->sharded = cfg->nchain < cfg->nchain_total;
  auto bail = [&](int code, const char *msg) { g_create_err = msg ? msg : e->err; mcgpu_destroy(e); return code; };
  if (cudaSetDevice(e->dev) != cudaSuccess) return bail(MCGPU_ENODEVICE, "cudaSetDevice failed");
  if (cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(MCGPU_ECUDA, "stream create failed");
  if (cudaStreamCreateWithFlags(&e->side, cudaStreamNonBlocking) != cudaSuccess) return bail(MCGPU_ECUDA, "stream create failed");
  e->stream = e->own_stream;
  const int d = e->d;
  int rc = 0;
#define TRY(x) do { rc = (x); if (rc) return bail(rc, nullptr); } while (0)
  TRY(dalloc(e, &e->overrun, 1));
  if (!e->verify) {
    if (cfg->mode != MCGPU_MODE_NORMAL && cfg->mode != MCGPU_MODE_REPLAY_LOCAL) return bail(MCGPU_EINVAL, "unknown mode");
    if (cfg->coin_group < 0 || cfg->coin_group > 32 || (cfg->coin_group & (cfg->coin_group - 1))) return bail(MCGPU_EINVAL, "coin_group must be 0 (job-wide coin) or a power of two in 1..32");
    if (cfg->chain0 % 32) return bail(MCGPU_EINVAL, "chain0 must be a multiple of 32");
    if (cfg->remote_mode != 0 && cfg->remote_mode != 1) return bail(MCGPU_EINVAL, "remote_mode must be 0 (reference max-mixture rejection loop) or 1 (sum-mixture proposal)");
    if (cfg->pool_lag != 0 && cfg->pool_lag != 1) return bail(MCGPU_EINVAL, "pool_lag must be 0 or 1");
    if (e->replay_local && (cfg->remote_mode || cfg->pool_lag)) return bail(MCGPU_EINVAL, "REPLAY_LOCAL takes local steps only: remote_mode / pool_lag do not apply");
    e->remote_mode = cfg->remote_mode; e->lag = cfg->pool_lag;
    if (e->replay_local && e->sharded) return bail(MCGPU_EINVAL, "REPLAY_LOCAL hosts the whole rank");
    e->ld = (e->C + 31) / 32 * 32;
    const bool never_remote = cfg->pl >= 1.0;              // the coin is < 1: rndlocal <= PLOCAL always (mcpar.cc:152)
    e->M = (cfg->pool_m > 0 && cfg->pool_m < e->N) ? cfg->pool_m : (int)std::min<long long>(e->N, 1 << 20);
    if (never_remote && cfg->pool_m <= 0) e->M = 1;        // pool is never read: keep one slot
    if (!never_remote && cfg->pool_m <= 0 && e->N > (1 << 20)) return bail(MCGPU_EINVAL, "pool_m = 0 (all chains) is limited to 2^20 chains; choose a pool size");
    e->stride = e->N / e->M;
    e->pool_in_smem = true;
    TRY(dalloc(e, &e->x, (size_t)d * e->ld)); TRY(dalloc(e, &e->ly, (size_t)e->ld));
    TRY(dalloc(e, &e->mu, (size_t)d * e->ld)); TRY(dalloc(e, &e->ps, (size_t)d * e->ld));
    TRY(dalloc(e, &e->factor, (size_t)d * d)); TRY(dalloc(e, &e->counts, 12));
    e->pool_bytes = ((size_t)e->M * d * 16 + 255) / 256 * 256;
    e->xchg_bytes = NPOOL * e->pool_bytes + 256;
    TRY(dalloc(e, &e->xchg, e->xchg_bytes));
    for (int b = 0; b < NPOOL; ++b) e->pool[b] = reinterpret_cast<double*>(e->xchg + (size_t)b * e->pool_bytes);
    TRY(dalloc(e, &e->xflag_d, 1));
    e->hist_cap = cfg->history_steps;
    if (e->hist_cap > 0) TRY(dalloc(e, &e->hist, (size_t)e->hist_cap * e->C * (d + 1), false));
    e->host_streams.resize(1);
  } else {
    if (cfg->remote_mode || cfg->pool_lag) return bail(MCGPU_EINVAL, "VERIFY runs the reference's own remote proposal: remote_mode / pool_lag must be 0");
    e->Cr = cfg->chains_per_rank;
    if (e->Cr < 1 || e->Cr > 1024) return bail(MCGPU_EINVAL, "VERIFY: chains_per_rank must be 1..1024");
    if (e->C % e->Cr || e->N % e->Cr || cfg->chain0 % e->Cr) return bail(MCGPU_EINVAL, "VERIFY: chain counts must be multiples of chains_per_rank");
    if (cfg->thin != 1) return bail(MCGPU_EINVAL, "VERIFY keeps every step (thin = 1)");
    e->Rl = (int)(e->C / e->Cr); e->R = (int)(e->N / e->Cr); e->rank0 = (int)(cfg->chain0 / e->Cr);
    const size_t nt = (size_t)e->Cr * d, nm = (size_t)2 * e->N * d;
    TRY(dalloc(e, &e->x, e->Rl * nt)); TRY(dalloc(e, &e->ptrial, e->Rl * nt)); TRY(dalloc(e, &e->ly, (size_t)e->C));
    TRY(dalloc(e, &e->mu, e->Rl * nt)); TRY(dalloc(e, &e->sig, e->Rl * nt)); TRY(dalloc(e, &e->ps, e->Rl * nt));
    TRY(dalloc(e, &e->mutrial, e->Rl * nt)); TRY(dalloc(e, &e->sigtrial, e->Rl * nt));
    TRY(dalloc(e, &e->factor, (size_t)e->Rl * d * d)); TRY(dalloc(e, &e->musig, e->Rl * nm));
    TRY(dalloc(e, &e->snap[0], nm)); TRY(dalloc(e, &e->snap[1], nm));
    TRY(dalloc(e, &e->soff, (size_t)e->Rl * 6)); TRY(dalloc(e, &e->cursors, (size_t)e->Rl * 3));
    TRY(dalloc(e, &e->counts, (size_t)e->Rl * 2)); TRY(dalloc(e, &e->irate_d, (size_t)e->Rl)); TRY(dalloc(e, &e->rstats, 4));
    e->hist_cap = cfg->history_steps;
    if (e->hist_cap > 0) TRY(dalloc(e, &e->hist, (size_t)e->hist_cap * e->C * (d + 1), false));
    e->host_streams.resize(e->Rl);
    if (cfg->trace > 0) {                                  // per-step trace of cfg->trace steps
      e->trace_cap = cfg->trace;
      const size_t T = (size_t)e->trace_cap * e->Rl;
      TRY(dalloc(e, &e->tr_accept, T * e->Cr)); TRY(dalloc(e, &e->tr_trial_ly, T * e->Cr));
      TRY(dalloc(e, &e->tr_trial_p, T * e->Cr * d)); TRY(dalloc(e, &e->tr_cfac, T * e->Cr));
      TRY(dalloc(e, &e->tr_remote, T)); TRY(dalloc(e, &e->tr_iters, T));
    }
    std::vector<int> ir(e->Rl, 50);                       // irate = 50, mcpar.cc:57
    if (cudaMemcpyAsync(e->irate_d, ir.data(), ir.size() * sizeof(int), cudaMemcpyHostToDevice, e->stream) != cudaSuccess) return bail(MCGPU_ECUDA, "memcpy failed");
    if (cudaStreamSynchronize(e->stream) != cudaSuccess) return bail(MCGPU_ECUDA, "sync failed");
  }
#undef TRY
  if (cudaStreamSynchronize(e->stream) != cudaSuccess) return bail(MCGPU_ECUDA, "sync failed after allocation");
  *out = e;
  return MCGPU_OK;
}

int mcgpu_destroy(mcgpu_engine *e)
{
  if (!e) return MCGPU_OK;
  cudaSetDevice(e->dev);
  if (e->own_stream) cudaStreamSynchronize(e->own_stream);
  if (e->stream && e->stream != e->own_stream) cudaStreamSynchronize(e->stream);
  if (e->p2p && e->xchg) {
    // peers may still be storing their last publication into this region: wait (bounded, 10 s) until every
    // arrival this engine is owed has landed before the region is freed.  (Peers that imported the region
    // must also have stopped using it: callers put a barrier between their last synchronize and destroy.)
    const unsigned long long want = (unsigned long long)e->M * arrivals_per_slot(e) * (unsigned long long)e->npub;
    for (int i = 0; i < 10000; ++i) {
      unsigned long long got = 0;
      if (cudaMemcpy(&got, e->xchg + NPOOL * e->pool_bytes, sizeof got, cudaMemcpyDeviceToHost) != cudaSuccess || got >= want) break;
      struct timespec ts = {0, 1000000}; nanosleep(&ts, nullptr);
    }
  }
  timers_resolve(e);
  void *ptrs[] = {e->x, e->ly, e->mu, e->ps, e->factor, e->counts, e->xchg, e->xflag_d, e->peers_d, e->hist, e->overrun,
                  e->Zd, e->Ud, e->Id, e->ptrial, e->sig, e->mutrial, e->sigtrial, e->musig, e->snap[0], e->snap[1],
                  e->soff, e->cursors, e->irate_d, e->rstats, e->tr_accept, e->tr_remote, e->tr_trial_ly,
                  e->tr_trial_p, e->tr_cfac, e->tr_iters, e->lik_dev, e->factor_cm, e->diag_d, e->pprep, e->gm_t, e->hist_f32,
                  e->aux, e->lytrial_d, e->flags_d};
  for (void *p : ptrs) if (p) cudaFree(p);
  for (void *q : e->peer_opened) cudaIpcCloseMemHandle(q);
  for (int i = 0; i < 2; ++i) { if (e->pin[i]) cudaFreeHost(e->pin[i]); if (e->pin_ev[i]) cudaEventDestroy(e->pin_ev[i]); }
  if (e->side) cudaStreamSynchronize(e->side);
  plugin_release(e);
  if (e->sink && e->sink_registered) cudaHostUnregister(e->sink);
  if (e->sink_ev) cudaEventDestroy(e->sink_ev);
  for (auto &dr : e->drains) cudaEventDestroy(dr.second);
  for (cudaEvent_t ev : e->ev_free) cudaEventDestroy(ev);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  if (e->side) cudaStreamDestroy(e->side);
  delete e;
  return MCGPU_OK;
}

int mcgpu_set_stream(mcgpu_engine *e, void *cuda_stream)
{
  if (!e) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  CK(cudaStreamSynchronize(e->stream));
  e->stream = (cudaStream_t)cuda_stream;                 // NULL is the legacy default stream
  return MCGPU_OK;
}

int mcgpu_set_likelihood(mcgpu_engine *e, int lik, const double *par, int npar)
{
  if (!e) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  if (lik == MCGPU_HOST_LIKELIHOOD) {                     // the likelihood stays with the caller: mcgpu_step_propose / accept
    if (e->cfg.mode != MCGPU_MODE_NORMAL || e->sharded) return fail(e, MCGPU_EINVAL, "a host likelihood needs one NORMAL-mode engine hosting every chain");
    if (e->have_state && !e->hostlik) return fail(e, MCGPU_ESTATE, "likelihood change would change the state layout: create a new engine");
    if (!e->ptrial) {
      CK(cudaMalloc((void**)&e->ptrial, (size_t)e->C * e->d * 8)); CK(cudaMalloc((void**)&e->aux, (size_t)e->C * 8));
      CK(cudaMalloc((void**)&e->lytrial_d, (size_t)e->C * 8)); CK(cudaMalloc((void**)&e->flags_d, (size_t)e->C * sizeof(int)));
    }
    e->hostlik = true; e->wide = false; e->lik = lik; e->lik_k = 0;
    return MCGPU_OK;
  }
  if (e->hostlik) return fail(e, MCGPU_ESTATE, "this engine was set up for a host likelihood: create a new engine");
  std::vector<double> dev; int K = 0; std::string err;
  int rc = prepare_lik(lik, e->d, par, npar, e->lp, dev, K, err);
  if (rc) { e->err = err; return rc; }
  if (!e->verify) {
    if (lik == MCGPU_ROSENBROCK2) return fail(e, MCGPU_EINVAL, "Rosenbrock2 couples neighbouring chains of a batch (rosenbrock.cc:32-33); available in VERIFY mode and mcgpu_loglik only");
    const bool can_wide = e->cfg.mode == MCGPU_MODE_NORMAL && e->cfg.coin_group == 0 && fast::wide_supported(lik, e->d);
    if (!can_wide && !fast::steps_supported(lik, e->d)) return fail(e, MCGPU_EINVAL, "no step kernel instantiated for this (likelihood, nparam)");
    if (e->have_state && can_wide != e->wide) return fail(e, MCGPU_ESTATE, "likelihood change would change the state layout: create a new engine");
    e->wide = can_wide;
    if (!e->wide && e->cfg.pl < 1.0 && fast::steps_smem_bytes(e->d, e->cfg.sync, e->M, true) > 200 * 1024)
      return fail(e, MCGPU_EINVAL, "remote-mixture pool does not fit in shared memory (40 bytes per slot and parameter + 16 per slot): choose pool_m with pool_m*nparam <= 4800");
  }
  if (e->plugin) { CK(cudaStreamSynchronize(e->stream)); plugin_release(e); }
  if (e->lik_dev) { cudaFree(e->lik_dev); e->lik_dev = nullptr; }
  if (!dev.empty()) {
    CK(cudaMalloc((void**)&e->lik_dev, dev.size() * 8));
    CK(cudaMemcpyAsync(e->lik_dev, dev.data(), dev.size() * 8, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
  }
  e->lik = lik; e->lik_k = K;
  if (e->wide) {
    const int d = e->d, L = d / 2;
    if (!e->factor_cm) { CK(cudaMalloc((void**)&e->factor_cm, (size_t)d * d * 8)); CK(cudaMalloc((void**)&e->diag_d, sizeof(int))); }
    e->mpad = (e->M + L - 1) / L * L;
    // (mu, h) pairs, sigma, n_s in fp64; then the fp32 copy: (g mu, g) pairs, n_s log2 e, 4 scalars
    if (!e->pprep) CK(cudaMalloc((void**)&e->pprep, ((size_t)3 * d + 1) * e->mpad * 8 + ((size_t)2 * d + 1) * e->mpad * 4 + 16));
    if (e->gm_t) { cudaFree(e->gm_t); e->gm_t = nullptr; }
    if (lik == MCGPU_GAUSSMIX) {                        // [d][Kpad] (mu, 1/s2) pairs, then [Kpad] log w; padding has weight 0
      e->kpad = (K + 2 * L - 1) / (2 * L) * (2 * L);
      std::vector<double> t((size_t)2 * d * e->kpad + e->kpad, 0.0);
      // exponent of component k expanded: c_k + sum_i x_i (a_ki x_i + b_ki), a = -1/(2 s2), b = mu/s2,
      // c = log w - 1/2 sum_i mu^2/s2 (two DFMA per component, parameter and chain in wide_loglik)
      for (int k = 0; k < e->kpad; ++k) {
        long double cacc = 0.0L;
        for (int i = 0; i < d; ++i) {
          const double mu = k < K ? dev[(size_t)k * d + i] : 0.0, is2 = k < K ? dev[(size_t)K * d + (size_t)k * d + i] : 0.0;
          t[((size_t)i * e->kpad + k) * 2] = -0.5 * is2;
          t[((size_t)i * e->kpad + k) * 2 + 1] = mu * is2;
          cacc += (long double)mu * mu * is2;
        }
        t[(size_t)2 * d * e->kpad + k] = k < K ? (double)((long double)dev[(size_t)2 * K * d + k] - 0.5L * cacc) : -INFINITY;
      }
      CK(cudaMalloc((void**)&e->gm_t, t.size() * 8));
      CK(cudaMemcpyAsync(e->gm_t, t.data(), t.size() * 8, cudaMemcpyHostToDevice, e->stream));
      CK(cudaStreamSynchronize(e->stream));
    }
  }
  return MCGPU_OK;
}

int mcgpu_set_likelihood_plugin(mcgpu_engine *e, const char *cubin_path, const double *par, int npar)
{
  if (!e) return MCGPU_EINVAL;
  if (npar < 0 || (npar > 0 && !par)) return fail(e, MCGPU_EINVAL, "par must hold npar reals");
  if (e->cfg.mode != MCGPU_MODE_NORMAL) return fail(e, MCGPU_EINVAL, "plugin likelihoods run in NORMAL mode only (not VERIFY or REPLAY_LOCAL)");
  if (e->hostlik) return fail(e, MCGPU_ESTATE, "this engine was set up for a host likelihood: create a new engine");
  if (e->have_state && e->wide) return fail(e, MCGPU_ESTATE, "likelihood change would change the state layout: create a new engine");
  if (e->cfg.pl < 1.0 && fast::steps_smem_bytes(e->d, e->cfg.sync, e->M, true) > 200 * 1024)
    return fail(e, MCGPU_EINVAL, "remote-mixture pool does not fit in shared memory (40 bytes per slot and parameter + 16 per slot): choose pool_m with pool_m*nparam <= 4800");
  DeviceGuard g(e->dev);
  cudaLibrary_t lib = nullptr; cudaKernel_t k[8]; std::string err;
  const int rc = plugin_open(cubin_path, e->d, &lib, k, err);
  if (rc) { e->err = err; return rc; }
  CK(cudaStreamSynchronize(e->stream));                   // nothing of the previous likelihood is in flight
  plugin_release(e);
  e->plugin = lib; memcpy(e->pk, k, sizeof e->pk);
  if (e->lik_dev) { cudaFree(e->lik_dev); e->lik_dev = nullptr; }
  if (npar > 0) {
    CK(cudaMalloc((void**)&e->lik_dev, (size_t)npar * 8));
    CK(cudaMemcpyAsync(e->lik_dev, par, (size_t)npar * 8, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
  }
  memset(e->lp, 0, sizeof e->lp);
  for (int i = 0; i < npar && i < 8; ++i) e->lp[i] = par[i];
  e->lik = MCGPU_DEVICE_PLUGIN; e->lik_k = npar; e->wide = false;   // thread-per-chain kernels only
  return MCGPU_OK;
}

int mcgpu_set_covariance(mcgpu_engine *e, const double *incov)
{
  if (!e) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  const int d = e->d;
  std::vector<double> cov((size_t)d * d, 0.0);
  if (incov) std::copy(incov, incov + (size_t)d * d, cov.begin());     // mcpar.cc:457-459
  else for (int i = 0; i < d; ++i) cov[(size_t)i * (d + 1)] = 1.0;      // :460-467
  (void)cholesky_lower(d, cov.data());                                  // :480 (info unchecked there too)
  const int copies = e->verify ? e->Rl : 1;
  for (int r = 0; r < copies; ++r)
    CK(cudaMemcpyAsync(e->factor + (size_t)r * d * d, cov.data(), cov.size() * 8, cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->have_factor = true;
  return MCGPU_OK;
}

// a fresh run starts here: schedule, tuning counters (window and cumulative) and the pending-boundary flag
static int state_installed(mcgpu_engine *e)
{
  if (!e->verify) CK(cudaMemsetAsync(e->counts, 0, 4 * sizeof(unsigned long long), e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->have_state = true; e->burn_done = 0; e->t_main = 0; e->sampling = false; e->irate = 50; e->tune_pending = false;
  return MCGPU_OK;
}

int mcgpu_set_state(mcgpu_engine *e, const double *pinit)
{
  if (!e || !pinit) return MCGPU_EINVAL;
  if (e->lik < 0) return fail(e, MCGPU_ESTATE, "set_likelihood first");
  if (e->hostlik) return fail(e, MCGPU_ESTATE, "host likelihood: the initial log-likelihoods come from the caller (mcgpu_set_state_host)");
  DeviceGuard g(e->dev);
  const int d = e->d;
  if (e->verify) {
    CK(cudaMemcpyAsync(e->x, pinit, (size_t)e->C * d * 8, cudaMemcpyHostToDevice, e->stream));
    // L(nchain, pvals, lylast) per rank batch (mcpar.cc:53)
    LikSpec L; L.lik = e->lik; L.d = d; L.k = e->lik_k; memcpy(L.lp, e->lp, sizeof L.lp); L.dev = e->lik_dev;
    for (int r = 0; r < e->Rl; ++r) {
      ++e->launches;
      CK(exact::launch_loglik_aos(L, e->x + (size_t)r * e->Cr * d, e->ly + (size_t)r * e->Cr, e->Cr, e->stream));
    }
  } else if (e->wide) {
    CK(cudaMemcpyAsync(e->x, pinit, (size_t)e->C * d * 8, cudaMemcpyHostToDevice, e->stream));
    LikSpec L; L.lik = e->lik; L.d = d; L.k = e->lik_k; memcpy(L.lp, e->lp, sizeof L.lp); L.dev = e->lik_dev;
    ++e->launches;
    CK(exact::launch_loglik_aos(L, e->x, e->ly, (int)e->C, e->stream));   // L(nchain, pvals, lylast), mcpar.cc:53
  } else {
    double *tmp = nullptr;
    CK(cudaMallocAsync((void**)&tmp, (size_t)e->C * d * 8, e->stream));
    CK(cudaMemcpyAsync(tmp, pinit, (size_t)e->C * d * 8, cudaMemcpyHostToDevice, e->stream));
    transpose_aos_to_soa<<<(unsigned)((e->C + 255) / 256), 256, 0, e->stream>>>(tmp, e->x, e->C, e->ld, d);
    CK(cudaGetLastError());
    CK(cudaFreeAsync(tmp, e->stream));
    StepParams p; fill_step_params(e, p);
    e->launches += 2;
    CK(launch_init_any(e, p));
  }
  return state_installed(e);
}

int mcgpu_set_streams(mcgpu_engine *e, int local_rank, const double *Z, size_t nz, const double *U, size_t nu,
                      const int32_t *I, size_t ni)
{
  if (!e) return MCGPU_EINVAL;
  if (!e->verify && !e->replay_local) return fail(e, MCGPU_ESTATE, "streams are only consumed in VERIFY / REPLAY_LOCAL mode");
  if (local_rank < 0 || local_rank >= (int)e->host_streams.size()) return fail(e, MCGPU_EINVAL, "local_rank out of range");
  StreamSet &s = e->host_streams[local_rank];
  s.Z.assign(Z, Z + (Z ? nz : 0)); s.U.assign(U, U + (U ? nu : 0)); s.I.assign(I, I + (I ? ni : 0));
  e->streams_dirty = true;
  return MCGPU_OK;
}

static int ready_to_step(mcgpu_engine *e, bool hostlik_ok = false)
{
  if (!e->have_state) return fail(e, MCGPU_ESTATE, "set_state first");
  if (e->hostlik && !hostlik_ok) return fail(e, MCGPU_ESTATE, "host likelihood: step with mcgpu_step_propose / mcgpu_step_accept");
  if (!e->have_factor) { int rc = mcgpu_set_covariance(e, nullptr); if (rc) return rc; }
  if (e->wide) { ++e->launches; CK(fast::launch_factor_prep(e->factor, e->factor_cm, e->d, e->diag_d, e->stream)); }
  if (e->verify || e->replay_local) { int rc = upload_streams(e); if (rc) return rc; }
  return 0;
}

// advance the burn-in by at most nmax steps without crossing a tuning boundary
static int burnin_some(mcgpu_engine *e, int nmax, int *ndone)
{
  *ndone = 0;
  if (nmax <= 0) return 0;
  if (e->tune_pending) return fail(e, MCGPU_ESTATE, "a tuning boundary is pending: call mcgpu_tune");
  const long long boundary = (long long)e->irate + 2;     // tune after step index irate+1 (isamp > irate, mcpar.cc:78)
  const int n = (int)std::min<long long>(nmax, boundary - e->burn_done);
  StepParams p; fill_step_params(e, p);
  p.counts = e->counts; p.step0 = (uint32_t)e->burn_done; p.nsteps = n; p.t0 = 0;
  CK(launch_steps_any(e, PH_BURN, p));
  e->burn_done += n; *ndone = n;
  if (e->burn_done == boundary) e->tune_pending = true;
  return 0;
}

int mcgpu_tune(mcgpu_engine *e)
{
  if (!e) return MCGPU_EINVAL;
  if (!e->tune_pending) return MCGPU_OK;
  DeviceGuard g(e->dev);
  ++e->launches;
  CK(fast::launch_tune(e->counts, e->counts + 2, e->factor, e->d * e->d, e->cfg.armin, e->cfg.armax, e->cfg.dfac, e->cfg.ifac, e->stream));
  e->irate += 50; e->tune_pending = false;
  if (e->wide) { ++e->launches; CK(fast::launch_factor_prep(e->factor, e->factor_cm, e->d, e->diag_d, e->stream)); }
  return MCGPU_OK;
}

int mcgpu_burnin_some(mcgpu_engine *e, int nmax, int *ndone, int *tune_pending)
{
  if (!e || !ndone) return MCGPU_EINVAL;
  if (e->verify) return fail(e, MCGPU_EINVAL, "VERIFY mode tunes inside the kernel: use mcgpu_burnin");
  DeviceGuard g(e->dev);
  int rc = ready_to_step(e); if (rc) return rc;
  rc = burnin_some(e, nmax, ndone);
  if (tune_pending) *tune_pending = e->tune_pending;
  return rc;
}

int mcgpu_burnin(mcgpu_engine *e, int nburn)
{
  if (!e || nburn < 0) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  int rc = ready_to_step(e); if (rc) return rc;
  if (e->sampling) return fail(e, MCGPU_ESTATE, "burn-in after sampling has begun");
  timer_begin(e);
  if (e->verify) {
    if (nburn > 0) {
      VerifyParams p; fill_verify_params(e, p);
      p.phase = 0; p.s0 = (int)e->burn_done; p.nsteps = nburn; p.trace_base = (int)e->burn_done;
      ++e->launches;
      CK(exact::launch_verify(p, e->Rl, e->stream));
      e->burn_done += nburn;
    }
  } else {
    if (e->sharded) return fail(e, MCGPU_ESTATE, "sharded engines burn in with mcgpu_burnin_some + all-reduce + mcgpu_tune");
    int left = nburn;
    while (left > 0) {
      int done = 0;
      rc = burnin_some(e, left, &done); if (rc) return rc;
      left -= done;
      if (e->tune_pending) { rc = mcgpu_tune(e); if (rc) return rc; }
    }
  }
  timer_end(e);
  e->nburn_total = (int)e->burn_done;
  if (e->verify || e->replay_local) return check_overrun(e);
  return MCGPU_OK;
}

int mcgpu_sample_begin(mcgpu_engine *e, int nsamp)
{
  if (!e || nsamp < 0) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  int rc = ready_to_step(e, true); if (rc) return rc;
  if (e->proposed) return fail(e, MCGPU_ESTATE, "a proposal is pending: call mcgpu_step_accept");
  const int d = e->d;
  CK(cudaStreamSynchronize(e->side));
  e->nsamp = nsamp; e->t_main = 0; e->sampling = true; e->exchange_pending = false; e->hist_kept = 0; e->sink_sent = 0;
  e->hist_valid_from = 0;
  for (auto &dr : e->drains) e->ev_free.push_back(dr.second);
  e->drains.clear();
  e->nburn_total = (int)e->burn_done;
  const long long need = (nsamp + e->cfg.thin - 1) / e->cfg.thin;
  if (e->verify && e->hist && need > e->hist_cap) return fail(e, MCGPU_EINVAL, "history_steps too small for nsamp (VERIFY holds the whole run)");
  // mu = 0, psum2 = FPEPS (mcpar.cc:100-103)
  const size_t n = e->verify ? (size_t)e->C * d : (size_t)d * e->ld;
  CK(cudaMemsetAsync(e->mu, 0, n * 8, e->stream));
  fill_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 148 * 8), 256, 0, e->stream>>>(e->ps, n, MCGPU_FPEPS);
  CK(cudaGetLastError());
  if (!e->verify) CK(cudaMemsetAsync(e->counts + 4, 0, 64, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return MCGPU_OK;
}

// The device history is a ring: before a launch overwrites kept steps that a host sink has not received yet,
// the engine's stream waits for their drain (an event on the side stream).
static int ring_guard(mcgpu_engine *e, long long k_hi)
{
  const long long need = k_hi - e->hist_cap;               // kept steps < need are about to be overwritten
  if (need <= 0 || !e->hist) return 0;
  if (e->sink && e->sink_sent < need) return fail(e, MCGPU_EINVAL, "history_steps is smaller than one exchange window's kept steps: the ring would overwrite rows before they drain");
  while (!e->drains.empty() && e->drains.front().first < need) { e->ev_free.push_back(e->drains.front().second); e->drains.pop_front(); }
  if (!e->drains.empty()) {                                // the first drain that covers `need` (drains complete in order)
    CK(cudaStreamWaitEvent(e->stream, e->drains.front().second, 0));
    e->ev_free.push_back(e->drains.front().second); e->drains.pop_front();
  }
  return 0;
}

// MCout drain: the kept steps [sink_sent, hist_kept) go to the host sink with asynchronous copies on the side
// stream (fp32 sink: narrowed on the device first), ring segment by ring segment.
static int drain_to_sink(mcgpu_engine *e)
{
  if (!e->sink || e->hist_kept <= e->sink_sent) return 0;
  if ((size_t)e->hist_kept > e->sink_rows_cap) return fail(e, MCGPU_EINVAL, "host sink is full: capacity_steps must hold every kept step of the run");
  const size_t row_elems = (size_t)(e->d + 1) * e->C;
  CK(cudaEventRecord(e->sink_ev, e->stream));
  CK(cudaStreamWaitEvent(e->side, e->sink_ev, 0));
  long long k = e->sink_sent;
  while (k < e->hist_kept) {
    const long long ring = k % e->hist_cap, cnt = std::min<long long>(e->hist_kept - k, e->hist_cap - ring);
    const size_t n0 = (size_t)ring * row_elems, n = (size_t)cnt * row_elems;
    if (e->sink_f32) {                                       // narrow on the device, then move half the bytes
      narrow_rows_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 148 * 16), 256, 0, e->side>>>(e->hist + n0, e->hist_f32 + n0, n);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync((float*)(void*)e->sink + (size_t)k * row_elems, e->hist_f32 + n0, n * sizeof(float), cudaMemcpyDeviceToHost, e->side));
    } else
      CK(cudaMemcpyAsync(e->sink + (size_t)k * row_elems, e->hist + n0, n * 8, cudaMemcpyDeviceToHost, e->side));
    k += cnt;
  }
  cudaEvent_t ev = event_get(e);
  CK(cudaEventRecord(ev, e->side));
  e->drains.emplace_back(e->hist_kept, ev);
  e->sink_sent = e->hist_kept;
  return 0;
}

int mcgpu_sample(mcgpu_engine *e, int nsteps)
{
  if (!e || nsteps < 0) return MCGPU_EINVAL;
  if (!e->sampling) return fail(e, MCGPU_ESTATE, "sample_begin first");
  if (e->hostlik) return fail(e, MCGPU_ESTATE, "host likelihood: step with mcgpu_step_propose / mcgpu_step_accept");
  if (e->t_main + nsteps > e->nsamp) return fail(e, MCGPU_EINVAL, "more steps than sample_begin announced");
  DeviceGuard g(e->dev);
  const int sync = e->cfg.sync;
  if (e->p2p_local && nsteps > sync - (e->t_main % sync))
    return fail(e, MCGPU_ESTATE, "engines attached with mcgpu_p2p_attach_local advance one exchange window at a time, in turn: use mcgpu_sample_group");
  timer_begin(e);
  int left = nsteps;
  while (left > 0) {
    if (e->exchange_pending) return fail(e, MCGPU_ESTATE, "exchange pending: call mcgpu_exchange_begin/end at every multiple of sync");
    const long long to_boundary = sync - (e->t_main % sync);
    const int n = (int)std::min<long long>(left, to_boundary);
    if (!e->verify) { int rc = ring_guard(e, (e->t_main + n + e->cfg.thin - 1) / e->cfg.thin); if (rc) return rc; }
    if (e->verify) {
      VerifyParams p; fill_verify_params(e, p);
      p.phase = 1; p.s0 = (int)e->t_main; p.nsteps = n; p.trace_base = (int)(e->nburn_total + e->t_main);
      p.refresh = (e->R > 1) && (e->t_main % sync == 0);
      p.publish = 1;
      p.snap_cur = e->snap[e->snap_cur]; p.snap_next = e->snap[e->snap_cur ^ 1];
      ++e->launches;
      CK(exact::launch_verify(p, e->Rl, e->stream));
    } else {
      StepParams p; fill_step_params(e, p);
      p.counts = e->counts + 4; p.xstat = e->counts + 8;
      p.pool_cur = pool_cur(e);
      fill_p2p(e, p);
      p.hist = e->hist; p.hist_ring0 = e->hist ? (int)((e->t_main / e->cfg.thin) % e->hist_cap) : 0;
      // publish (mu, sigma^2) into the next pool only from the launch that ends the window
      double *const publish = ((e->t_main + n) % sync == 0) ? pool_next(e) : nullptr;
      if (e->cfg.coin_group > 0 || e->replay_local) {       // per-group coins: one mixed launch per window
        p.step0 = (uint32_t)(e->nburn_total + e->t_main); p.nsteps = n; p.t0 = (int)e->t_main;
        p.pool_next = publish;
        CK(launch_steps_any(e, PH_MIXED, p));
      } else {                                               // job-wide coin: runs of local / remote steps
        // wide kernels read the pool as (mu, -1/2sig^2, sig), slot-fastest: prepared right before the window's
        // first remote launch (with a peer-to-peer exchange that kernel also waits for the arrivals, so the
        // window's leading local steps overlap the exchange)
        bool prepped = !e->wide;
        auto pool_prep = [&]() -> cudaError_t {
          prepped = true; ++e->launches;
          return fast::launch_pool_prep(pool_cur(e), e->M, e->mpad, e->d, reinterpret_cast<double2*>(e->pprep),
                                        e->pprep + (size_t)2 * e->d * e->mpad, e->pprep + (size_t)3 * e->d * e->mpad,
                                        reinterpret_cast<float2*>(e->pprep + ((size_t)3 * e->d + 1) * e->mpad),
                                        reinterpret_cast<float*>(e->pprep + ((size_t)3 * e->d + 1) * e->mpad) + (size_t)2 * e->d * e->mpad,
                                        reinterpret_cast<float*>(e->pprep + ((size_t)3 * e->d + 1) * e->mpad) + ((size_t)2 * e->d + 1) * e->mpad,
                                        p.arrivals, p.wait_target, p.xflag, p.xstat, e->stream);
        };
        auto is_remote = [&](long long tt) {
          return tt >= (long long)sync * (1 + e->lag) && !(host_coin(e, (uint32_t)(e->nburn_total + tt)) <= e->cfg.pl);   // mcpar.cc:142-152
        };
        static const int plan = getenv("MCGPU_PLAN") ? atoi(getenv("MCGPU_PLAN")) : 1;
        uint32_t mask = 0;
        for (int k = 0; k < n && k < 32; ++k) if (is_remote(e->t_main + k)) mask |= 1u << k;
        if (plan && !e->wide && n <= 32) {
          // one launch per window: the lean local kernel when no step of the window is remote,
          // otherwise the two-path kernel with the host-drawn plan (uniform branches)
          p.step0 = (uint32_t)(e->nburn_total + e->t_main); p.nsteps = n; p.t0 = (int)e->t_main;
          p.pool_next = publish;
          p.plan_mask = mask; p.plan_valid = 1;
          CK(launch_steps_any(e, mask ? PH_MIXED : PH_LOCAL, p));
        } else {
          int k = 0;
          while (k < n) {
            const long long t = e->t_main + k;
            const bool rem = is_remote(t);
            int len = 1;
            while (k + len < n && is_remote(t + len) == rem) ++len;
            p.step0 = (uint32_t)(e->nburn_total + t); p.nsteps = len; p.t0 = (int)t;
            p.hist_ring0 = e->hist ? (int)((t / e->cfg.thin) % e->hist_cap) : 0;
            p.pool_next = (k + len == n) ? publish : nullptr;
            if (rem && !prepped) CK(pool_prep());
            CK(launch_steps_any(e, rem ? PH_REMOTE : PH_LOCAL, p));
            k += len;
          }
        }
      }
    }
    e->t_main += n; left -= n;
    e->hist_kept = (e->t_main + e->cfg.thin - 1) / e->cfg.thin;
    if (e->hist) { int rc = drain_to_sink(e); if (rc) return rc; }
    if (e->t_main % sync == 0) {
      if (e->sharded && !e->p2p) e->exchange_pending = true;   // caller all-gathers the published slices
      else if (e->verify) e->snap_cur ^= 1;
      else ++e->npub;                                      // one engine, or the kernels exchanged over NVLink themselves
    }
  }
  timer_end(e);
  if ((e->verify || e->replay_local) && e->t_main == e->nsamp) return check_overrun(e);
  return MCGPU_OK;
}

int mcgpu_exchange_begin(mcgpu_engine *e, void **dev_buffer, size_t *total_bytes, size_t *own_offset, size_t *own_bytes)
{
  if (!e || !dev_buffer) return MCGPU_EINVAL;
  const int d = e->d;
  if (e->verify) {
    *dev_buffer = e->snap[e->snap_cur ^ 1];
    if (total_bytes) *total_bytes = (size_t)2 * e->N * d * 8;
    if (own_offset) *own_offset = (size_t)2 * e->cfg.chain0 * d * 8;
    if (own_bytes) *own_bytes = (size_t)2 * e->C * d * 8;
  } else {
    // own pool slots: s with chain0 <= s*stride < chain0 + C
    const long long s0 = (e->cfg.chain0 + e->stride - 1) / e->stride;
    const long long s1 = std::min<long long>(e->M, (e->cfg.chain0 + e->C + e->stride - 1) / e->stride);
    *dev_buffer = pool_next(e);
    if (total_bytes) *total_bytes = (size_t)e->M * d * 16;
    if (own_offset) *own_offset = (size_t)s0 * d * 16;
    if (own_bytes) *own_bytes = (size_t)std::max<long long>(0, s1 - s0) * d * 16;
  }
  return MCGPU_OK;
}

int mcgpu_exchange_end(mcgpu_engine *e)
{
  if (!e) return MCGPU_EINVAL;
  if (!e->exchange_pending) return MCGPU_OK;
  if (e->verify) e->snap_cur ^= 1; else ++e->npub;
  e->exchange_pending = false;
  return MCGPU_OK;
}

// ---- peer-to-peer exchange --------------------------------------------------------------------
// The window kernels of sharded engines store their published (mu, sigma^2) slots straight into
// every GPU's next pool buffer over NVLink and bump that GPU's arrival counter; the next window's
// kernel waits on its own counter.  No host round trip, no separate collective launch: this
// replaces MPI_Allgather(MPI_IN_PLACE) of src/mcpar.cc:127-140 inside the step kernel.
static int p2p_check(mcgpu_engine *e, int world, int rank)
{
  if (e->verify || e->replay_local) return fail(e, MCGPU_ESTATE, "peer-to-peer exchange exists in NORMAL mode only");
  if (e->npub != 0 || e->sampling || e->p2p) return fail(e, MCGPU_ESTATE, "attach peers once, before the first mcgpu_sample_begin");
  if (world < 1 || world > 64 || rank < 0 || rank >= world) return fail(e, MCGPU_EINVAL, "bad world/rank");
  if (e->C * world != e->N || e->cfg.chain0 != rank * e->C) return fail(e, MCGPU_EINVAL, "peers must host equal contiguous blocks of chains: chain0 = rank * nchain");
  return MCGPU_OK;
}

static int p2p_finish(mcgpu_engine *e, int world, const std::vector<char*> &bases)
{
  CK(cudaMalloc((void**)&e->peers_d, sizeof(char*) * world));
  CK(cudaMemcpyAsync(e->peers_d, bases.data(), sizeof(char*) * world, cudaMemcpyHostToDevice, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->p2p = true; e->p2p_world = world;
  return MCGPU_OK;
}

int mcgpu_p2p_export(mcgpu_engine *e, void *handle, size_t nbytes)
{
  if (!e || !handle) return MCGPU_EINVAL;
  if (nbytes < sizeof(cudaIpcMemHandle_t) || sizeof(cudaIpcMemHandle_t) > MCGPU_P2P_HANDLE_BYTES) return fail(e, MCGPU_EINVAL, "handle buffer too small");
  if (!e->xchg) return fail(e, MCGPU_ESTATE, "no exchange region (VERIFY engine)");
  DeviceGuard g(e->dev);
  CK(cudaStreamSynchronize(e->stream));                    // the region is zeroed before anybody maps it
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, e->xchg));
  memset(handle, 0, nbytes); memcpy(handle, &h, sizeof h);
  return MCGPU_OK;
}

int mcgpu_p2p_attach(mcgpu_engine *e, int world, int rank, const void *handles)
{
  if (!e || !handles) return MCGPU_EINVAL;
  int rc = p2p_check(e, world, rank); if (rc) return rc;
  DeviceGuard g(e->dev);
  std::vector<char*> bases(world, nullptr);
  for (int r = 0; r < world; ++r) {
    if (r == rank) { bases[r] = e->xchg; continue; }
    cudaIpcMemHandle_t h; memcpy(&h, (const char*)handles + (size_t)r * MCGPU_P2P_HANDLE_BYTES, sizeof h);
    void *q = nullptr;
    CK(cudaIpcOpenMemHandle(&q, h, cudaIpcMemLazyEnablePeerAccess));
    e->peer_opened.push_back(q); bases[r] = (char*)q;
  }
  return p2p_finish(e, world, bases);
}

int mcgpu_p2p_attach_local(mcgpu_engine *const *engines, int world)
{
  if (!engines || world < 1) return MCGPU_EINVAL;
  for (int r = 0; r < world; ++r) {
    if (!engines[r]) return MCGPU_EINVAL;
    int rc = p2p_check(engines[r], world, r); if (rc) return rc;
    if (engines[r]->M != engines[0]->M || engines[r]->d != engines[0]->d) return fail(engines[r], MCGPU_EINVAL, "peers differ in shape");
  }
  for (int r = 0; r < world; ++r) {
    mcgpu_engine *e = engines[r];
    DeviceGuard g(e->dev);
    std::vector<char*> bases(world, nullptr);
    for (int q = 0; q < world; ++q) {
      bases[q] = engines[q]->xchg;
      if (engines[q]->dev == e->dev) continue;
      int can = 0;
      CK(cudaDeviceCanAccessPeer(&can, e->dev, engines[q]->dev));
      if (!can) return fail(e, MCGPU_ECUDA, "devices cannot access each other's memory");
      cudaError_t s = cudaDeviceEnablePeerAccess(engines[q]->dev, 0);
      if (s != cudaSuccess && s != cudaErrorPeerAccessAlreadyEnabled) CK(s);
      cudaGetLastError();
    }
    CK(cudaStreamSynchronize(e->stream));
    int rc = p2p_finish(e, world, bases); if (rc) return rc;
    e->p2p_local = true;
  }
  return MCGPU_OK;
}

// One host thread drives `world` peer-to-peer engines: their windows are enqueued in turn, one exchange window at
// a time, so that a window kernel waiting for its peers' publications is never queued in front of the launches
// that make them (the launch queue is finite, and engines may share a device).
int mcgpu_sample_group(mcgpu_engine *const *engines, int world, int nsteps)
{
  if (!engines || world < 1 || nsteps < 0) return MCGPU_EINVAL;
  for (int r = 0; r < world; ++r) {
    if (!engines[r]) return MCGPU_EINVAL;
    if (engines[r]->t_main != engines[0]->t_main || engines[r]->cfg.sync != engines[0]->cfg.sync)
      return fail(engines[r], MCGPU_ESTATE, "engines of a group are out of step");
  }
  const int sync = engines[0]->cfg.sync;
  int left = nsteps;
  while (left > 0) {
    const int n = (int)std::min<long long>(left, sync - (engines[0]->t_main % sync));
    for (int r = 0; r < world; ++r) { int rc = mcgpu_sample(engines[r], n); if (rc) return rc; }
    left -= n;
  }
  return MCGPU_OK;
}

// Burn-in of several sharded engines of one process: the window's {accepted, tried} counters are
// summed over the engines before every tuning decision (what sharded.py does with an all-reduce).
int mcgpu_burnin_group(mcgpu_engine *const *engines, int world, int nburn)
{
  if (!engines || world < 1 || nburn < 0) return MCGPU_EINVAL;
  for (int r = 0; r < world; ++r) {
    if (!engines[r]) return MCGPU_EINVAL;
    if (engines[r]->verify) return fail(engines[r], MCGPU_EINVAL, "VERIFY mode tunes inside the kernel: use mcgpu_burnin");
  }
  int left = nburn;
  while (left > 0) {
    int done = 0, pending = 0;
    for (int r = 0; r < world; ++r) {
      int dr = 0, pr = 0;
      int rc = mcgpu_burnin_some(engines[r], left, &dr, &pr); if (rc) return rc;
      if (r > 0 && (dr != done || pr != pending)) return fail(engines[r], MCGPU_ESTATE, "engines of a group are out of step");
      done = dr; pending = pr;
    }
    left -= done;
    if (!pending) continue;
    unsigned long long sum[2] = {0, 0};
    for (int r = 0; r < world; ++r) {
      mcgpu_engine *e = engines[r]; DeviceGuard g(e->dev);
      unsigned long long c[2];
      CK(cudaMemcpyAsync(c, e->counts, sizeof c, cudaMemcpyDeviceToHost, e->stream));
      CK(cudaStreamSynchronize(e->stream));
      sum[0] += c[0]; sum[1] += c[1];
    }
    for (int r = 0; r < world; ++r) {
      mcgpu_engine *e = engines[r]; DeviceGuard g(e->dev);
      CK(cudaMemcpyAsync(e->counts, sum, sizeof sum, cudaMemcpyHostToDevice, e->stream));
      CK(cudaStreamSynchronize(e->stream));              // `sum` is pageable stack memory
      int rc = mcgpu_tune(e); if (rc) return rc;
    }
  }
  for (int r = 0; r < world; ++r) engines[r]->nburn_total = (int)engines[r]->burn_done;
  return MCGPU_OK;
}

// ---- host-callback likelihood: one step = propose (device) -> VLFunc (host) -> accept (device) ------------
int mcgpu_set_state_host(mcgpu_engine *e, const double *pinit, const double *lylast)
{
  if (!e || !pinit || !lylast) return MCGPU_EINVAL;
  if (!e->hostlik) return fail(e, MCGPU_ESTATE, "mcgpu_set_likelihood(e, MCGPU_HOST_LIKELIHOOD, NULL, 0) first");
  DeviceGuard g(e->dev);
  CK(cudaMemcpyAsync(e->x, pinit, (size_t)e->C * e->d * 8, cudaMemcpyHostToDevice, e->stream));     // chain-major, as given
  CK(cudaMemcpyAsync(e->ly, lylast, (size_t)e->C * 8, cudaMemcpyHostToDevice, e->stream));          // L(nchain, pvals, lylast), mcpar.cc:53
  e->proposed = false;
  return state_installed(e);
}

static void fill_hostlik(mcgpu_engine *e, HostLikParams &p)
{
  memset(&p, 0, sizeof p);
  p.x = e->x; p.ly = e->ly; p.mu = e->mu; p.ps = e->ps; p.ptrial = e->ptrial; p.aux = e->aux; p.flags = e->flags_d;
  p.lytrial = e->lytrial_d; p.C = e->C; p.chain0 = e->cfg.chain0; p.d = e->d; p.factor = e->factor;
  p.counts = e->counts; p.mcounts = e->counts + 4;
  p.key0 = (uint32_t)e->cfg.seed; p.key1 = (uint32_t)(e->cfg.seed >> 32);
  p.main_phase = e->sampling ? 1 : 0;
  p.step = (uint32_t)(e->sampling ? e->nburn_total + e->t_main : e->burn_done);
  p.t = (int)e->t_main; p.first_remote_t = e->cfg.sync * (1 + e->lag); p.coin_group = e->cfg.coin_group; p.pl = e->cfg.pl;
  p.pool = pool_cur(e); p.pool_next = pool_next(e); p.pool_m = e->M; p.pool_stride = e->stride; p.remote_mode = e->remote_mode;
  p.hist = e->hist; p.hist_row = -1;
}

int mcgpu_step_propose(mcgpu_engine *e, double *ptrial)
{
  if (!e || !ptrial) return MCGPU_EINVAL;
  if (!e->hostlik) return fail(e, MCGPU_ESTATE, "not a host-likelihood engine");
  if (e->proposed) return fail(e, MCGPU_ESTATE, "a proposal is pending: call mcgpu_step_accept");
  if (e->sampling && e->t_main >= e->nsamp) return fail(e, MCGPU_EINVAL, "more steps than sample_begin announced");
  DeviceGuard g(e->dev);
  int rc = ready_to_step(e, true);
  if (rc) return rc;
  HostLikParams p; fill_hostlik(e, p);
  ++e->launches;
  CK(exact::launch_hostlik_propose(p, e->stream));
  CK(cudaMemcpyAsync(ptrial, e->ptrial, (size_t)e->C * e->d * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  e->proposed = true;
  return MCGPU_OK;
}

int mcgpu_step_accept(mcgpu_engine *e, const double *lytrial)
{
  if (!e || !lytrial) return MCGPU_EINVAL;
  if (!e->hostlik || !e->proposed) return fail(e, MCGPU_ESTATE, "mcgpu_step_propose first");
  DeviceGuard g(e->dev);
  CK(cudaMemcpyAsync(e->lytrial_d, lytrial, (size_t)e->C * 8, cudaMemcpyHostToDevice, e->stream));
  HostLikParams p; fill_hostlik(e, p);
  int publish = 0; double pub_winv = 0.0;
  if (e->sampling) {
    const int thin = e->cfg.thin;
    if (e->hist && e->t_main % thin == 0) {
      int rc = ring_guard(e, e->t_main / thin + 1); if (rc) return rc;
      p.hist_row = (int)((e->t_main / thin) % e->hist_cap);
    }
    publish = (e->t_main + 1) % e->cfg.sync == 0;
    pub_winv = 1.0 / (double)(e->t_main + 1);
  }
  ++e->launches;
  CK(exact::launch_hostlik_accept(p, publish, pub_winv, e->stream));
  CK(cudaStreamSynchronize(e->stream));                   // lytrial is the caller's (pageable) buffer
  e->proposed = false;
  if (!e->sampling) {
    ++e->burn_done;
    e->nburn_total = (int)e->burn_done;
    if (e->burn_done == (long long)e->irate + 2) {         // tune after step index irate+1 (isamp > irate, mcpar.cc:78)
      e->tune_pending = true;
      int rc = mcgpu_tune(e); if (rc) return rc;
    }
  } else {
    ++e->t_main;
    e->hist_kept = (e->t_main + e->cfg.thin - 1) / e->cfg.thin;
    if (e->hist) { int rc = drain_to_sink(e); if (rc) return rc; }
    if (publish) ++e->npub;
  }
  return MCGPU_OK;
}

int mcgpu_tuning_counters(mcgpu_engine *e, void **dev_counts)
{
  if (!e || !dev_counts) return MCGPU_EINVAL;
  *dev_counts = e->counts;
  return MCGPU_OK;
}

int mcgpu_synchronize(mcgpu_engine *e)
{
  if (!e) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  CK(cudaStreamSynchronize(e->stream));
  CK(cudaStreamSynchronize(e->side));
  if (e->p2p) {                                            // did a window give up waiting for a peer's publication?
    int flag = 0;
    CK(cudaMemcpy(&flag, e->xflag_d, sizeof flag, cudaMemcpyDeviceToHost));
    if (flag) return fail(e, MCGPU_EPEER, "peer-to-peer exchange timed out: a peer did not publish its pool slots");
  }
  return MCGPU_OK;
}

static int attach_host_sink(mcgpu_engine *e, void *rows_v, size_t capacity_steps, bool f32);

int mcgpu_history_attach_host(mcgpu_engine *e, double *rows, size_t capacity_steps) { return attach_host_sink(e, rows, capacity_steps, false); }
int mcgpu_history_attach_host_f32(mcgpu_engine *e, float *rows, size_t capacity_steps) { return attach_host_sink(e, rows, capacity_steps, true); }

static int attach_host_sink(mcgpu_engine *e, void *rows_v, size_t capacity_steps, bool f32)
{
  if (!e) return MCGPU_EINVAL;
  double *rows = static_cast<double*>(rows_v);
  DeviceGuard g(e->dev);
  CK(cudaStreamSynchronize(e->side));
  if (e->sink && e->sink_registered) { cudaHostUnregister(e->sink); e->sink_registered = false; }
  e->sink = nullptr; e->sink_rows_cap = 0; e->sink_f32 = false;
  if (!rows) return MCGPU_OK;
  if (!e->hist) return fail(e, MCGPU_ESTATE, "engine was created with history_steps = 0");
  if (capacity_steps < 1) return fail(e, MCGPU_EINVAL, "host sink holds no kept step");
  if (e->hist_cap * e->cfg.thin < e->cfg.sync && !e->verify) return fail(e, MCGPU_EINVAL, "history_steps must hold at least one exchange window's kept steps to drain into a host sink");
  cudaPointerAttributes at;
  const bool pinned = cudaPointerGetAttributes(&at, rows) == cudaSuccess && at.type == cudaMemoryTypeHost;
  cudaGetLastError();
  if (!pinned) {                                           // page-lock the caller's buffer for DMA
    CK(cudaHostRegister(rows, capacity_steps * (size_t)e->C * (e->d + 1) * (f32 ? 4 : 8), cudaHostRegisterDefault));
    e->sink_registered = true;
  }
  if (f32 && !e->hist_f32) CK(cudaMalloc((void**)&e->hist_f32, (size_t)e->hist_cap * e->C * (e->d + 1) * sizeof(float)));
  e->sink_f32 = f32;
  if (!e->sink_ev) CK(cudaEventCreateWithFlags(&e->sink_ev, cudaEventDisableTiming));
  e->sink = rows; e->sink_rows_cap = capacity_steps; e->sink_sent = e->hist_kept;
  return MCGPU_OK;
}

int mcgpu_get_state(mcgpu_engine *e, double *pvals, double *lylast, double *mu, double *sig, double *psum2)
{
  if (!e) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  const int d = e->d;
  const size_t nb = (size_t)e->C * d * 8;
  if (e->verify) {
    if (pvals) CK(cudaMemcpyAsync(pvals, e->x, nb, cudaMemcpyDeviceToHost, e->stream));
    if (mu) CK(cudaMemcpyAsync(mu, e->mu, nb, cudaMemcpyDeviceToHost, e->stream));
    if (sig) CK(cudaMemcpyAsync(sig, e->sig, nb, cudaMemcpyDeviceToHost, e->stream));
    if (psum2) CK(cudaMemcpyAsync(psum2, e->ps, nb, cudaMemcpyDeviceToHost, e->stream));
  } else if (e->wide || e->hostlik) {
    if (pvals) CK(cudaMemcpyAsync(pvals, e->x, nb, cudaMemcpyDeviceToHost, e->stream));
    if (mu) CK(cudaMemcpyAsync(mu, e->mu, nb, cudaMemcpyDeviceToHost, e->stream));
    if (psum2) CK(cudaMemcpyAsync(psum2, e->ps, nb, cudaMemcpyDeviceToHost, e->stream));
    if (sig) {
      CK(cudaMemcpyAsync(sig, e->ps, nb, cudaMemcpyDeviceToHost, e->stream));
      CK(cudaStreamSynchronize(e->stream));
      const double winv = e->t_main > 0 ? 1.0 / (double)e->t_main : 0.0;      // sig = psum2 * winv (mcpar.cc:202)
      for (size_t i = 0; i < (size_t)e->C * d; ++i) sig[i] *= winv;
    }
  } else {
    double *tmp = nullptr;
    CK(cudaMallocAsync((void**)&tmp, nb, e->stream));
    const unsigned grid = (unsigned)((e->C + 255) / 256);
    struct { double *dst; const double *src; double scale; } jobs[4] = {
      {pvals, e->x, 1.0}, {mu, e->mu, 1.0}, {psum2, e->ps, 1.0},
      {sig, e->ps, e->t_main > 0 ? 1.0 / (double)e->t_main : 0.0}};   // sig = psum2 * winv (mcpar.cc:202)
    for (auto &jb : jobs) {
      if (!jb.dst) continue;
      transpose_soa_to_aos<<<grid, 256, 0, e->stream>>>(jb.src, tmp, e->C, e->ld, d, jb.scale);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(jb.dst, tmp, nb, cudaMemcpyDeviceToHost, e->stream));
    }
    CK(cudaFreeAsync(tmp, e->stream));
  }
  if (lylast) CK(cudaMemcpyAsync(lylast, e->ly, (size_t)e->C * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return MCGPU_OK;
}

int mcgpu_get_factor(mcgpu_engine *e, int local_rank, double *factor)
{
  if (!e || !factor) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  const int nr = e->verify ? e->Rl : 1;
  if (local_rank < 0 || local_rank >= nr) return fail(e, MCGPU_EINVAL, "local_rank out of range");
  CK(cudaMemcpyAsync(factor, e->factor + (size_t)local_rank * e->d * e->d, (size_t)e->d * e->d * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return MCGPU_OK;
}

int mcgpu_get_musig(mcgpu_engine *e, int local_rank, double *musig)
{
  if (!e || !musig) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  if (e->verify) {
    if (local_rank < 0 || local_rank >= e->Rl) return fail(e, MCGPU_EINVAL, "local_rank out of range");
    const size_t nm = (size_t)2 * e->N * e->d;
    CK(cudaMemcpyAsync(musig, e->musig + (size_t)local_rank * nm, nm * 8, cudaMemcpyDeviceToHost, e->stream));
  } else {
    CK(cudaMemcpyAsync(musig, pool_newest(e), (size_t)e->M * e->d * 16, cudaMemcpyDeviceToHost, e->stream));
  }
  CK(cudaStreamSynchronize(e->stream));
  return MCGPU_OK;
}

int mcgpu_get_trace(mcgpu_engine *e, int local_rank, uint8_t *accept, double *trial_ly, double *trial_p, double *cfac,
                    uint8_t *remote, int32_t *iters, int64_t *cursors)
{
  if (!e) return MCGPU_EINVAL;
  if (!e->verify) return fail(e, MCGPU_ESTATE, "traces exist in VERIFY mode only");
  if (local_rank < 0 || local_rank >= e->Rl) return fail(e, MCGPU_EINVAL, "local_rank out of range");
  DeviceGuard g(e->dev);
  const size_t T = (size_t)e->trace_cap, C = (size_t)e->Cr, r = (size_t)local_rank;
  if ((accept || trial_ly || trial_p || cfac || remote || iters) && !e->tr_accept) return fail(e, MCGPU_ESTATE, "engine was created with trace = 0");
  if (accept) CK(cudaMemcpyAsync(accept, e->tr_accept + r * T * C, T * C, cudaMemcpyDeviceToHost, e->stream));
  if (trial_ly) CK(cudaMemcpyAsync(trial_ly, e->tr_trial_ly + r * T * C, T * C * 8, cudaMemcpyDeviceToHost, e->stream));
  if (trial_p) CK(cudaMemcpyAsync(trial_p, e->tr_trial_p + r * T * C * e->d, T * C * e->d * 8, cudaMemcpyDeviceToHost, e->stream));
  if (cfac) CK(cudaMemcpyAsync(cfac, e->tr_cfac + r * T * C, T * C * 8, cudaMemcpyDeviceToHost, e->stream));
  if (remote) CK(cudaMemcpyAsync(remote, e->tr_remote + r * T, T, cudaMemcpyDeviceToHost, e->stream));
  if (iters) CK(cudaMemcpyAsync(iters, e->tr_iters + r * T, T * 4, cudaMemcpyDeviceToHost, e->stream));
  if (cursors) CK(cudaMemcpyAsync(cursors, e->cursors + r * 3, 24, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return MCGPU_OK;
}

int mcgpu_history_read(mcgpu_engine *e, int64_t first_step, int64_t count, double *rows)
{
  if (!e || !rows || first_step < 0 || count < 0) return MCGPU_EINVAL;
  if (!e->hist) return fail(e, MCGPU_ESTATE, "engine was created with history_steps = 0");
  if (first_step + count > e->hist_kept) return fail(e, MCGPU_EINVAL, "history range not yet produced");
  if (count > 0 && first_step < std::max(e->hist_valid_from, e->hist_kept - e->hist_cap))
    return fail(e, MCGPU_EINVAL, "history range no longer on the device (the ring holds the last history_steps kept steps; rows before a checkpoint load are not restored)");
  DeviceGuard g(e->dev);
  const size_t row_bytes = (size_t)(e->d + 1) * 8;
  if (count > 0 && first_step % e->hist_cap + count > e->hist_cap) {   // the range wraps around the ring: two reads
    const int64_t c1 = e->hist_cap - first_step % e->hist_cap;
    int rc = mcgpu_history_read(e, first_step, c1, rows); if (rc) return rc;
    return mcgpu_history_read(e, first_step + c1, count - c1, rows + (size_t)c1 * e->C * (e->d + 1));
  }
  const size_t total = (size_t)count * e->C * row_bytes;
  const char *src = (const char*)e->hist + (size_t)(first_step % e->hist_cap) * e->C * row_bytes;
  if (total == 0) return MCGPU_OK;
  {
    cudaPointerAttributes at;
    const bool pinned = cudaPointerGetAttributes(&at, rows) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    if (pinned) {                                          // page-locked destination: one DMA, no staging
      CK(cudaMemcpyAsync(rows, src, total, cudaMemcpyDeviceToHost, e->stream));
      CK(cudaStreamSynchronize(e->stream));
      return MCGPU_OK;
    }
  }
  // drain on the side stream through two pinned staging buffers so the PCIe copy of
  // chunk k overlaps the host memcpy of chunk k-1
  const size_t chunk = (size_t)32 << 20;
  if (!e->pin[0]) {
    for (int i = 0; i < 2; ++i) { CK(cudaMallocHost((void**)&e->pin[i], chunk)); CK(cudaEventCreateWithFlags(&e->pin_ev[i], cudaEventDisableTiming)); }
    e->pin_bytes = chunk;
  }
  cudaEvent_t produced; CK(cudaEventCreateWithFlags(&produced, cudaEventDisableTiming));
  CK(cudaEventRecord(produced, e->stream));
  CK(cudaStreamWaitEvent(e->side, produced, 0));
  CK(cudaEventDestroy(produced));
  const size_t nchunks = (total + chunk - 1) / chunk;
  for (size_t k = 0; k <= nchunks; ++k) {
    if (k < nchunks) {
      const size_t off = k * chunk, nb = std::min(chunk, total - off);
      if (k >= 2) CK(cudaEventSynchronize(e->pin_ev[k & 1]));   // buffer consumed below before reuse
      CK(cudaMemcpyAsync(e->pin[k & 1], src + off, nb, cudaMemcpyDeviceToHost, e->side));
      CK(cudaEventRecord(e->pin_ev[k & 1], e->side));
    }
    if (k >= 1) {
      const size_t pk = k - 1, off = pk * chunk, nb = std::min(chunk, total - off);
      CK(cudaEventSynchronize(e->pin_ev[pk & 1]));
      memcpy((char*)rows + off, e->pin[pk & 1], nb);
    }
  }
  return MCGPU_OK;
}

// the kept steps the device still holds, [max(valid_from, kept - cap), kept), as at most two contiguous ring ranges
namespace {
struct HistSeg { long long ring0, kept0, count; };
int hist_segments(const mcgpu_engine *e, HistSeg seg[2])
{
  const long long lo = std::max(e->hist_valid_from, e->hist_kept - e->hist_cap), hi = e->hist_kept;
  if (hi <= lo) return 0;
  const long long r0 = lo % e->hist_cap, c0 = std::min(hi - lo, e->hist_cap - r0);
  seg[0] = {r0, lo, c0};
  if (c0 == hi - lo) return 1;
  seg[1] = {0, lo + c0, hi - lo - c0};
  return 2;
}
}  // namespace

int mcgpu_history_maxlike(mcgpu_engine *e, double *out)
{
  if (!e || !out) return MCGPU_EINVAL;
  if (!e->hist) return fail(e, MCGPU_ESTATE, "engine was created with history_steps = 0");
  DeviceGuard g(e->dev);
  HistSeg seg[2]; const int nseg = hist_segments(e, seg);
  if (nseg == 0) return fail(e, MCGPU_ESTATE, "history is empty");
  const int nb = 296;
  double *bv = nullptr; long long *br = nullptr;
  CK(cudaMallocAsync((void**)&bv, nb * 8, e->stream)); CK(cudaMallocAsync((void**)&br, nb * 8, e->stream));
  std::vector<double> hv(nb); std::vector<long long> hr(nb);
  long long best = -1, best_abs = -1; double val = -INFINITY;   // best_abs: row index in kept-step order (first occurrence wins, mcout.cc:138)
  for (int sg = 0; sg < nseg; ++sg) {
    ++e->launches;
    argmax_rows_kernel<<<nb, 256, 0, e->stream>>>(e->hist + (size_t)seg[sg].ring0 * e->C * (e->d + 1), seg[sg].count * e->C, e->d + 1, bv, br);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(hv.data(), bv, nb * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(hr.data(), br, nb * 8, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    for (int i = 0; i < nb; ++i) {
      if (hr[i] < 0) continue;
      const long long abs_row = seg[sg].kept0 * e->C + hr[i];
      if (best < 0 || hv[i] > val || (hv[i] == val && abs_row < best_abs)) { best = seg[sg].ring0 * e->C + hr[i]; best_abs = abs_row; val = hv[i]; }
    }
  }
  CK(cudaFreeAsync(bv, e->stream)); CK(cudaFreeAsync(br, e->stream));
  if (best < 0) return fail(e, MCGPU_ESTATE, "history holds no finite log-likelihood");
  CK(cudaMemcpy(out, e->hist + (size_t)best * (e->d + 1), (size_t)(e->d + 1) * 8, cudaMemcpyDeviceToHost));
  return MCGPU_OK;
}

int mcgpu_history_moments(mcgpu_engine *e, double *mean, double *cov)
{
  if (!e || !mean || !cov) return MCGPU_EINVAL;
  if (!e->hist) return fail(e, MCGPU_ESTATE, "engine was created with history_steps = 0");
  DeviceGuard g(e->dev);
  const int d = e->d; const int nq = d + d * (d + 1) / 2;
  HistSeg seg[2]; const int nseg = hist_segments(e, seg);
  if (nseg == 0) return fail(e, MCGPU_ESTATE, "history is empty");
  long long nrows = 0;
  double *acc = nullptr;
  CK(cudaMallocAsync((void**)&acc, nq * 8, e->stream));
  CK(cudaMemsetAsync(acc, 0, nq * 8, e->stream));
  for (int sg = 0; sg < nseg; ++sg) {
    ++e->launches;
    moments_kernel<<<dim3(592, nq), 256, 0, e->stream>>>(e->hist + (size_t)seg[sg].ring0 * e->C * (d + 1), seg[sg].count * e->C, d, acc);
    CK(cudaGetLastError());
    nrows += seg[sg].count * e->C;
  }
  std::vector<double> h(nq);
  CK(cudaMemcpyAsync(h.data(), acc, nq * 8, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaFreeAsync(acc, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  const double n = (double)nrows;
  for (int i = 0; i < d; ++i) mean[i] = h[i] / n;
  int q = d;
  for (int i = 0; i < d; ++i)
    for (int j = i; j < d; ++j, ++q) { const double c = h[q] / n - mean[i] * mean[j]; cov[i * d + j] = c; cov[j * d + i] = c; }
  return MCGPU_OK;
}

// ---- checkpoint / restart ---------------------------------------------------------------------
// Everything a NORMAL-mode engine needs to continue a run bit for bit: chain state, running moments,
// the tuned proposal factor, tuning / statistics counters, the exchange pools and the schedule.
// The sample history is not part of it (rows kept so far must have been read or drained).
namespace {
struct CkptHeader {
  char magic[8]; int32_t abi, d, lik, wide, M, sync, thin, coin_group; int64_t C, N, chain0, ld;
  int64_t burn_done, t_main, npub; int32_t nsamp, irate, nburn_total, sampling, tune_pending, have_factor, remote_mode, pool_lag;
  uint64_t seed; double pl;
};
size_t ckpt_bytes(const mcgpu_engine *e)
{
  return sizeof(CkptHeader) + ((size_t)3 * e->d * e->ld + e->ld + (size_t)e->d * e->d) * 8 + 12 * 8 + NPOOL * e->pool_bytes;
}
}  // namespace

int mcgpu_checkpoint_size(mcgpu_engine *e, size_t *bytes)
{
  if (!e || !bytes) return MCGPU_EINVAL;
  if (e->verify || e->replay_local || e->hostlik) return fail(e, MCGPU_ESTATE, "checkpoints exist in NORMAL mode with a device likelihood only");
  *bytes = ckpt_bytes(e);
  return MCGPU_OK;
}

int mcgpu_checkpoint_save(mcgpu_engine *e, void *buf, size_t bytes)
{
  if (!e || !buf) return MCGPU_EINVAL;
  if (e->verify || e->replay_local) return fail(e, MCGPU_ESTATE, "checkpoints exist in NORMAL mode only");
  if (bytes < ckpt_bytes(e)) return fail(e, MCGPU_EINVAL, "checkpoint buffer too small (mcgpu_checkpoint_size)");
  if (!e->have_state) return fail(e, MCGPU_ESTATE, "nothing to save: set_state first");
  if (e->exchange_pending) return fail(e, MCGPU_ESTATE, "finish the pending exchange first");
  DeviceGuard g(e->dev);
  CkptHeader h; memset(&h, 0, sizeof h);
  memcpy(h.magic, "MCGPUCK2", 8);
  h.abi = MCGPU_ABI_VERSION; h.d = e->d; h.lik = e->lik; h.wide = e->wide; h.M = e->M; h.sync = e->cfg.sync; h.thin = e->cfg.thin;
  h.coin_group = e->cfg.coin_group; h.C = e->C; h.N = e->N; h.chain0 = e->cfg.chain0; h.ld = e->ld;
  h.burn_done = e->burn_done; h.t_main = e->t_main; h.npub = e->npub; h.nsamp = e->nsamp; h.irate = e->irate;
  h.nburn_total = e->nburn_total; h.sampling = e->sampling; h.tune_pending = e->tune_pending; h.have_factor = e->have_factor;
  h.seed = e->cfg.seed; h.pl = e->cfg.pl; h.remote_mode = e->remote_mode; h.pool_lag = e->lag;
  char *q = static_cast<char*>(buf);
  memcpy(q, &h, sizeof h); q += sizeof h;
  const size_t ns = (size_t)e->d * e->ld * 8;
  struct { const void *src; size_t n; } parts[] = {{e->x, ns}, {e->mu, ns}, {e->ps, ns}, {e->ly, (size_t)e->ld * 8},
                                                   {e->factor, (size_t)e->d * e->d * 8}, {e->counts, 96}, {e->xchg, NPOOL * e->pool_bytes}};
  for (auto &pt : parts) { CK(cudaMemcpyAsync(q, pt.src, pt.n, cudaMemcpyDeviceToHost, e->stream)); q += pt.n; }
  CK(cudaStreamSynchronize(e->stream));
  return MCGPU_OK;
}

int mcgpu_checkpoint_load(mcgpu_engine *e, const void *buf, size_t bytes)
{
  if (!e || !buf) return MCGPU_EINVAL;
  if (e->verify || e->replay_local) return fail(e, MCGPU_ESTATE, "checkpoints exist in NORMAL mode only");
  if (e->lik < 0) return fail(e, MCGPU_ESTATE, "set_likelihood first (the likelihood is not part of a checkpoint)");
  if (bytes < ckpt_bytes(e)) return fail(e, MCGPU_EINVAL, "checkpoint truncated");
  CkptHeader h; memcpy(&h, buf, sizeof h);
  if (memcmp(h.magic, "MCGPUCK2", 8) || h.abi != MCGPU_ABI_VERSION) return fail(e, MCGPU_EINVAL, "not a checkpoint of this ABI");
  if (h.d != e->d || h.C != e->C || h.N != e->N || h.chain0 != e->cfg.chain0 || h.ld != e->ld || h.M != e->M || h.lik != e->lik ||
      h.wide != (int)e->wide || h.sync != e->cfg.sync || h.thin != e->cfg.thin || h.coin_group != e->cfg.coin_group ||
      h.seed != e->cfg.seed || h.pl != e->cfg.pl || h.remote_mode != e->remote_mode || h.pool_lag != e->lag)
    return fail(e, MCGPU_EINVAL, "checkpoint was taken by an engine of a different shape / likelihood / seed");
  DeviceGuard g(e->dev);
  CK(cudaStreamSynchronize(e->side));
  const char *q = static_cast<const char*>(buf) + sizeof h;
  const size_t ns = (size_t)e->d * e->ld * 8;
  struct { void *dst; size_t n; } parts[] = {{e->x, ns}, {e->mu, ns}, {e->ps, ns}, {e->ly, (size_t)e->ld * 8},
                                             {e->factor, (size_t)e->d * e->d * 8}, {e->counts, 96}, {e->xchg, NPOOL * e->pool_bytes}};
  for (auto &pt : parts) { CK(cudaMemcpyAsync(pt.dst, q, pt.n, cudaMemcpyHostToDevice, e->stream)); q += pt.n; }
  if (e->p2p) {   // peers restore the same epoch: every publication up to npub counts as arrived
    const unsigned long long arrived = (unsigned long long)e->M * arrivals_per_slot(e) * (unsigned long long)h.npub;
    CK(cudaMemcpyAsync(e->xchg + NPOOL * e->pool_bytes, &arrived, sizeof arrived, cudaMemcpyHostToDevice, e->stream));
  }
  if (e->wide) { ++e->launches; CK(fast::launch_factor_prep(e->factor, e->factor_cm, e->d, e->diag_d, e->stream)); }   // derived copies
  CK(cudaStreamSynchronize(e->stream));
  e->burn_done = h.burn_done; e->t_main = h.t_main; e->npub = h.npub; e->nsamp = h.nsamp; e->irate = h.irate;
  e->nburn_total = h.nburn_total; e->sampling = h.sampling != 0; e->tune_pending = h.tune_pending != 0;
  e->have_factor = h.have_factor != 0; e->have_state = true; e->exchange_pending = false;
  e->hist_kept = (e->t_main + e->cfg.thin - 1) / e->cfg.thin; e->sink_sent = e->hist_kept;
  e->hist_valid_from = e->hist_kept;                       // the history is not part of the blob: earlier rows are not on this device
  for (auto &dr : e->drains) e->ev_free.push_back(dr.second);
  e->drains.clear();
  return MCGPU_OK;
}

int mcgpu_get_stats(mcgpu_engine *e, mcgpu_stats *out)
{
  if (!e || !out) return MCGPU_EINVAL;
  DeviceGuard g(e->dev);
  CK(cudaStreamSynchronize(e->stream));
  timers_resolve(e);
  memset(out, 0, sizeof *out);
  out->burn_steps = e->burn_done; out->main_steps = e->t_main; out->kernel_launches = e->launches;
  out->history_rows = e->hist_kept * e->C; out->device_ms = e->ms_accum;
  unsigned long long h[12] = {0};
  if (e->verify) {
    CK(cudaMemcpy(h, e->rstats, 32, cudaMemcpyDeviceToHost));
    out->remote_steps = (int64_t)h[0]; out->remote_iterations = (int64_t)h[1];
    out->accepted = (int64_t)h[2]; out->tried = (int64_t)h[3];
  } else {
    CK(cudaMemcpy(h, e->counts, 96, cudaMemcpyDeviceToHost));
    out->accepted = (int64_t)h[4]; out->tried = (int64_t)h[5];
    out->remote_steps = (int64_t)h[6]; out->remote_iterations = (int64_t)h[7];
    out->exchange_wait_ns = (int64_t)h[8]; out->exchange_waits = (int64_t)h[9]; out->exact_fallbacks = (int64_t)h[10];
  }
  return MCGPU_OK;
}

int mcgpu_device_ptr(mcgpu_engine *e, int which, void **ptr, size_t *bytes)
{
  if (!e || !ptr) return MCGPU_EINVAL;
  const size_t st = e->verify ? (size_t)e->C * e->d * 8 : (size_t)e->d * e->ld * 8;
  size_t nb = 0;
  switch (which) {
    case 0: *ptr = e->x; nb = st; break;
    case 1: *ptr = e->ly; nb = (size_t)(e->verify ? e->C : e->ld) * 8; break;
    case 2: *ptr = e->mu; nb = st; break;
    case 3: *ptr = e->ps; nb = st; break;
    case 4: *ptr = e->hist; nb = (size_t)e->hist_cap * e->C * (e->d + 1) * 8; break;
    case 5: *ptr = e->verify ? e->snap[e->snap_cur] : pool_newest(e); nb = e->verify ? (size_t)2 * e->N * e->d * 8 : (size_t)e->M * e->d * 16; break;
    default: return fail(e, MCGPU_EINVAL, "unknown buffer id");
  }
  if (bytes) *bytes = nb;
  return MCGPU_OK;
}

// ---- stand-alone entry points (no engine) -----------------------------------
#define CK0(call) do { cudaError_t _s = (call); if (_s != cudaSuccess) { g_create_err = std::string(#call) + " -> " + cudaGetErrorString(_s); return MCGPU_ECUDA; } } while (0)

int mcgpu_loglik(int device, int lik, int nparam, const double *par, int npar, int npset, const double *x, double *y)
{
  if (!x || !y || npset < 0) return fail(nullptr, MCGPU_EINVAL, "null argument");
  if (mcgpu_device_count() <= device || device < 0) return fail(nullptr, MCGPU_ENODEVICE, "no usable CUDA device (this engine has no CPU path)");
  if (npset == 0) return MCGPU_OK;
  DeviceGuard g(device);
  LikSpec L; memset(&L, 0, sizeof L);
  std::vector<double> dev; std::string err;
  int rc = prepare_lik(lik, nparam, par, npar, L.lp, dev, L.k, err);
  if (rc) { g_create_err = err; return rc; }
  L.lik = lik; L.d = nparam;
  double *dx = nullptr, *dy = nullptr, *dp = nullptr;
  CK0(cudaMalloc((void**)&dx, (size_t)npset * nparam * 8)); CK0(cudaMalloc((void**)&dy, (size_t)npset * 8));
  if (!dev.empty()) { CK0(cudaMalloc((void**)&dp, dev.size() * 8)); CK0(cudaMemcpy(dp, dev.data(), dev.size() * 8, cudaMemcpyHostToDevice)); }
  L.dev = dp;
  CK0(cudaMemcpy(dx, x, (size_t)npset * nparam * 8, cudaMemcpyHostToDevice));
  CK0(exact::launch_loglik_aos(L, dx, dy, npset, 0));
  CK0(cudaMemcpy(y, dy, (size_t)npset * 8, cudaMemcpyDeviceToHost));
  cudaFree(dx); cudaFree(dy); if (dp) cudaFree(dp);
  return MCGPU_OK;
}

int mcgpu_loglik_plugin(int device, const char *cubin_path, int nparam, const double *par, int npar, int npset,
                        const double *x, double *y)
{
  if (!x || !y || npset < 0 || npar < 0 || (npar > 0 && !par)) return fail(nullptr, MCGPU_EINVAL, "null argument");
  if (mcgpu_device_count() <= device || device < 0) return fail(nullptr, MCGPU_ENODEVICE, "no usable CUDA device (this engine has no CPU path)");
  DeviceGuard g(device);
  cudaLibrary_t lib = nullptr; cudaKernel_t k[8]; std::string err;
  const int rc = plugin_open(cubin_path, nparam, &lib, k, err);
  if (rc) return fail(nullptr, rc, err.c_str());
  struct Unload { cudaLibrary_t l; ~Unload() { cudaLibraryUnload(l); } } unload = {lib};
  if (npset == 0) return MCGPU_OK;
  double *dx = nullptr, *dy = nullptr, *dp = nullptr;
  CK0(cudaMalloc((void**)&dx, (size_t)npset * nparam * 8)); CK0(cudaMalloc((void**)&dy, (size_t)npset * 8));
  if (npar > 0) CK0(cudaMalloc((void**)&dp, (size_t)npar * 8));
  if (npar > 0) CK0(cudaMemcpyAsync(dp, par, (size_t)npar * 8, cudaMemcpyHostToDevice, 0));
  CK0(cudaMemcpyAsync(dx, x, (size_t)npset * nparam * 8, cudaMemcpyHostToDevice, 0));
  const double *cdp = dp, *cdx = dx;
  void *args[] = {(void *)&cdp, (void *)&npar, (void *)&cdx, (void *)&dy, (void *)&npset};
  CK0(cudaLaunchKernel(reinterpret_cast<const void *>(k[PK_EVAL]), dim3((unsigned)((npset + 255) / 256)), dim3(256), args, 0, 0));
  CK0(cudaMemcpyAsync(y, dy, (size_t)npset * 8, cudaMemcpyDeviceToHost, 0));
  CK0(cudaStreamSynchronize(0));
  cudaFree(dx); cudaFree(dy); if (dp) cudaFree(dp);
  return MCGPU_OK;
}

int mcgpu_qriguess(int device, int rank, int npset, int nparam, const double *plo, const double *phi, double *pout)
{
  if (!plo || !phi || !pout || npset < 0 || rank < 0) return fail(nullptr, MCGPU_EINVAL, "bad argument");
  if (nparam < 1 || nparam > SOBOL_JK_NDIM) return fail(nullptr, MCGPU_EINVAL, "Sobol table covers 1..64 dimensions");
  if (mcgpu_device_count() <= device || device < 0) return fail(nullptr, MCGPU_ENODEVICE, "no usable CUDA device (this engine has no CPU path)");
  const size_t ntot = (size_t)npset * (size_t)nparam;               // mcutil.cc:19 (an int there)
  if (ntot == 0) return MCGPU_OK;
  DeviceGuard g(device);
  std::vector<uint32_t> dirs((size_t)nparam * 32);
  for (int k = 0; k < nparam; ++k) sobol_dirs(k, &dirs[(size_t)k * 32]);
  uint32_t *dd = nullptr; double *dlo = nullptr, *dhi = nullptr, *dout = nullptr;
  CK0(cudaMalloc((void**)&dd, dirs.size() * 4)); CK0(cudaMalloc((void**)&dlo, nparam * 8));
  CK0(cudaMalloc((void**)&dhi, nparam * 8)); CK0(cudaMalloc((void**)&dout, ntot * 8));
  CK0(cudaMemcpy(dd, dirs.data(), dirs.size() * 4, cudaMemcpyHostToDevice));
  CK0(cudaMemcpy(dlo, plo, nparam * 8, cudaMemcpyHostToDevice)); CK0(cudaMemcpy(dhi, phi, nparam * 8, cudaMemcpyHostToDevice));
  const unsigned long long first = rank > 0 ? (unsigned long long)rank * (unsigned long long)ntot : 0ull;   // :22-23
  sobol_box_kernel<<<(unsigned)std::min<size_t>((ntot + 255) / 256, 148 * 32), 256>>>(dd, nparam, first, ntot, dlo, dhi, dout, 0);
  CK0(cudaGetLastError());
  CK0(cudaMemcpy(pout, dout, ntot * 8, cudaMemcpyDeviceToHost));
  cudaFree(dd); cudaFree(dlo); cudaFree(dhi); cudaFree(dout);
  return MCGPU_OK;
}

// qriguess straight into the engine's state: chain g = chain0 + j starts at Sobol point first_point + g.
int mcgpu_set_state_sobol(mcgpu_engine *e, const double *plo, const double *phi, uint64_t first_point)
{
  if (!e || !plo || !phi) return MCGPU_EINVAL;
  if (e->lik < 0) return fail(e, MCGPU_ESTATE, "set_likelihood first");
  if (e->verify) return fail(e, MCGPU_ESTATE, "VERIFY mode takes its initial points from the host (mcgpu_set_state)");
  DeviceGuard g(e->dev);
  const int d = e->d;
  std::vector<uint32_t> dirs((size_t)d * 32);
  for (int k = 0; k < d; ++k) sobol_dirs(k, &dirs[(size_t)k * 32]);
  std::vector<double> box(plo, plo + d); box.insert(box.end(), phi, phi + d);
  uint32_t *dd = nullptr; double *dbox = nullptr;
  CK(cudaMallocAsync((void**)&dd, dirs.size() * 4, e->stream)); CK(cudaMallocAsync((void**)&dbox, box.size() * 8, e->stream));
  CK(cudaMemcpyAsync(dd, dirs.data(), dirs.size() * 4, cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemcpyAsync(dbox, box.data(), box.size() * 8, cudaMemcpyHostToDevice, e->stream));
  const size_t ntot = (size_t)e->C * d;
  const unsigned long long first = ((unsigned long long)first_point + (unsigned long long)e->cfg.chain0) * (unsigned long long)d;
  ++e->launches;
  sobol_box_kernel<<<(unsigned)std::min<size_t>((ntot + 255) / 256, 148 * 32), 256, 0, e->stream>>>(dd, d, first, ntot, dbox, dbox + d, e->x, e->wide ? 0 : e->ld);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(e->stream));                    // dirs / box are host temporaries
  CK(cudaFreeAsync(dd, e->stream)); CK(cudaFreeAsync(dbox, e->stream));
  ++e->launches;
  if (e->wide) {
    LikSpec L; L.lik = e->lik; L.d = d; L.k = e->lik_k; memcpy(L.lp, e->lp, sizeof L.lp); L.dev = e->lik_dev;
    CK(exact::launch_loglik_aos(L, e->x, e->ly, (int)e->C, e->stream));   // L(nchain, pvals, lylast), mcpar.cc:53
  } else {
    StepParams p; fill_step_params(e, p);
    CK(launch_init_any(e, p));
  }
  return state_installed(e);
}

int mcgpu_measure_fp64_peak(int device, double *tflops)
{
  if (!tflops) return MCGPU_EINVAL;
  if (mcgpu_device_count() <= device || device < 0) return fail(nullptr, MCGPU_ENODEVICE, "no usable CUDA device");
  DeviceGuard g(device);
  cudaDeviceProp prop; CK0(cudaGetDeviceProperties(&prop, device));
  double *out = nullptr; CK0(cudaMalloc((void**)&out, 8));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
  cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
  double best = 0;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(a);
    dfma_peak_kernel<<<blocks, threads>>>(out, iters, 1.0000001, 1e-9);
    cudaEventRecord(b);
    CK0(cudaEventSynchronize(b));
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    const double tf = (double)blocks * threads * (double)iters * 8 * 2 / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(out);
  *tflops = best;
  return MCGPU_OK;
}

}  // extern "C"
