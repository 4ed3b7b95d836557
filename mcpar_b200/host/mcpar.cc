// mcpar.cc -- MCPar on the B200 engine.  Same constructor, run() signature, log file and
// output cadence as the reference (src/mcpar.cc:17-214), but the chain loop is a handful
// of calls into the C ABI: the device keeps the state and runs SYNCSTEP-step launches.
#include "mcpar.hh"
#include "../../include/mcgpu.h"
#include <fstream>
#include <sstream>
#include <iomanip>
#include <vector>
#include <new>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <typeinfo>
#include <algorithm>

const Real MCPar::FPEPS = 1.0e-14;

namespace {
void die(mcgpu_engine *e, const char *what, int rc)
{
  fprintf(stderr, "MCPar: %s failed (%d): %s\n", what, rc, mcgpu_last_error(e));
  exit(3);                                   // the reference aborts on MKL/MPI errors (mcpar.hh:93)
}
#define CHECK(call) do { int _rc = (call); if (_rc != MCGPU_OK) die(eng, #call, _rc); } while (0)
}

MCPar::MCPar(int np, int nc, int mpisiz, int mpirank, Real pl, Real armin, Real armax, Real dfac, Real ifac, int sync)
  : TGT_ARATE_MIN(armin), TGT_ARATE_MAX(armax), SCALE_DEC(dfac), SCALE_INC(ifac), PLOCAL(pl), SYNCSTEP(sync),
    logging(false), logstep(1000), device(0), ngpu(1), pool_m(0), thin(1), coin_group(-1), remote_mode(0), pool_lag(0),
    history_bytes(1ll << 30), seed(8675309ull),
    nparam(np), nchain(nc), size(mpisiz < 1 ? 1 : mpisiz), rank(mpirank), mdevice_ms(0), maccept(0), mxwait_ms(0)
{
  tchains = size * nchain;
  if (rank != 0) {
    fprintf(stderr, "rank = %d:  this build hosts every rank in one process; construct MCPar with mpirank 0\n", rank);
    throw("Invalid rank: the B200 engine is single-process");
  }
}

void MCPar::destroy_engines()
{
  for (size_t g = 0; g < engs.size(); ++g) if (engs[g]) mcgpu_destroy(engs[g]);
  engs.clear();
}

MCPar::~MCPar() { destroy_engines(); }

int MCPar::run(int nsamp, int nburn, const Real *pinit, VLFunc &L, MCout &outsamples, Real *incov)
{
  // A likelihood with a device functor runs inside the fused step kernels.  Any other VLFunc (a user-written
  // plugin, src/vlfunc.hh:9-12) is called HERE, on the host, once per step between the engine's propose and
  // accept kernels -- the same place MCPar::run calls it (src/mcpar.cc:60, :160); everything else stays on the GPU.
  DeviceVLFunc *dl = dynamic_cast<DeviceVLFunc *>(&L);
  const bool hostlik = dl == 0;
  if (hostlik && ngpu > 1) {
    fprintf(stderr, "MCPar::run: a host likelihood runs on one engine (ngpu = 1)\n");
    return INVALID;
  }
  // log file, as the reference: rank 0 writes mcpar-log.000.txt in the working directory
  std::stringstream logname;
  logname << "mcpar-log." << std::setfill('0') << std::setw(3) << rank << ".txt";
  std::ofstream logfile(logname.str().c_str());

  try {
    outsamples.newsamps((size_t)((nsamp + thin - 1) / thin) * (size_t)tchains);
  } catch (std::bad_alloc &) {
    logfile << "Unable to allocate space for output samples.  Exiting.\n";
    exit(2);
  }

  // chains sharded over G engines by contiguous blocks of ranks (the musigall slot rule, mcpar.cc:206)
  destroy_engines();
  const int G = ngpu < 1 ? 1 : ngpu;
  const int ndev = mcgpu_device_count();
  if (size % G != 0 || (G > 1 && (((long long)(size / G) * nchain) % 32) != 0)) {
    fprintf(stderr, "MCPar::run: ngpu = %d needs mpisiz %% ngpu == 0 and (mpisiz / ngpu) * nc a multiple of 32\n", G);
    return INVALID;
  }
  const long long cg_chains = (long long)(size / G) * nchain;          // chains per engine
  const int rpg = size / G;                                           // ranks per engine
  // one local/remote coin per rank-sized group of chains (mcpar.cc:106-109,142-159)
  int cg = 1; while (cg * 2 <= nchain && cg < 32) cg *= 2;
  if (coin_group == 0) cg = 0;                                        // one coin per step for the whole job
  mcgpu_engine *eng = 0;                                              // the engine CHECK reports on
  // The device history is a ring of `ring` kept steps, read back into MCout piece by piece: at least one
  // exchange window's worth, at most the whole run, otherwise what fits the byte budget.
  const int outstep = nsamp > 50 ? nsamp / 10 : 5;       // mcpar.cc:110
  const long long kept_total = (nsamp + thin - 1) / thin;
  const long long row_bytes = (long long)cg_chains * (nparam + 1) * (long long)sizeof(Real);
  long long ring = std::max<long long>(history_bytes / std::max<long long>(row_bytes, 1), (SYNCSTEP + thin - 1) / thin + 1);
  ring = std::max<long long>(1, std::min(ring, kept_total));
  const int piece = (int)std::max<long long>(SYNCSTEP, (ring * thin) / SYNCSTEP * SYNCSTEP);   // steps sampled between two reads
  for (int g = 0; g < G; ++g) {
    mcgpu_config cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.abi_version = MCGPU_ABI_VERSION; cfg.device = ndev > 0 ? (device + g) % ndev : device; cfg.mode = MCGPU_MODE_NORMAL;
    cfg.nparam = nparam; cfg.nchain = cg_chains; cfg.chain0 = g * cg_chains; cfg.nchain_total = tchains;
    cfg.sync = SYNCSTEP; cfg.pl = PLOCAL; cfg.armin = TGT_ARATE_MIN; cfg.armax = TGT_ARATE_MAX;
    cfg.dfac = SCALE_DEC; cfg.ifac = SCALE_INC; cfg.seed = seed;
    cfg.coin_group = cg;
    cfg.pool_m = pool_m; cfg.thin = thin; cfg.remote_mode = remote_mode; cfg.pool_lag = pool_lag;
    cfg.history_steps = ring;
    mcgpu_engine *e = 0;
    const int rc = mcgpu_create(&cfg, &e);
    if (rc != MCGPU_OK) die(0, "mcgpu_create", rc);
    engs.push_back(e);
  }
  eng = engs[0];

  static const std::vector<double> nopar;
  const std::vector<double> &par = dl ? dl->params() : nopar;
  // pinit holds np*nc values; every rank starts from the same block (the mains pass the
  // same array on every rank, mcpar-rosen1.cc:43)
  std::vector<Real> p0((size_t)cg_chains * nparam);
  for (int r = 0; r < rpg; ++r) memcpy(&p0[(size_t)r * nchain * nparam], pinit, sizeof(Real) * (size_t)nchain * nparam);
  std::vector<Real> ptrial, lytrial;                                  // host likelihood: one step's trial points and their logL
  // the plugin is called with rank-sized batches, as each MPI rank called it: L(nchain, x, y) (mcpar.cc:53,60,160)
  struct Plugin {
    VLFunc &L; int nchain, nparam, size;
    void operator()(const Real *x, Real *y) { for (int r = 0; r < size; ++r) L(nchain, x + (size_t)r * nchain * nparam, y + (size_t)r * nchain); }
  } plugin = {L, nchain, nparam, size};
  for (int g = 0; g < G; ++g) {
    eng = engs[g];
    if (hostlik) {
      CHECK(mcgpu_set_likelihood(eng, MCGPU_HOST_LIKELIHOOD, 0, 0));
      CHECK(mcgpu_set_covariance(eng, incov));
      ptrial.resize(p0.size()); lytrial.resize((size_t)cg_chains);
      plugin(&p0[0], &lytrial[0]);                                    // L(nchain, pvals, lylast), mcpar.cc:53
      CHECK(mcgpu_set_state_host(eng, &p0[0], &lytrial[0]));
    } else {
      if (dl->plugin_path()) CHECK(mcgpu_set_likelihood_plugin(eng, dl->plugin_path(), par.empty() ? 0 : &par[0], (int)par.size()));
      else CHECK(mcgpu_set_likelihood(eng, dl->lik_id(), par.empty() ? 0 : &par[0], (int)par.size()));
      CHECK(mcgpu_set_covariance(eng, incov));
      CHECK(mcgpu_set_state(eng, &p0[0]));
    }
  }
  eng = engs[0];
  if (G > 1) CHECK(mcgpu_p2p_attach_local(&engs[0], G));

  logfile << "Starting burn-in.  Samples = " << nburn << std::endl;
  if (hostlik) {
    for (int isamp = 0; isamp < nburn; ++isamp) {                     // propose -> plugin -> accept (+ tuning inside accept)
      CHECK(mcgpu_step_propose(eng, &ptrial[0]));
      plugin(&ptrial[0], &lytrial[0]);
      CHECK(mcgpu_step_accept(eng, &lytrial[0]));
    }
  } else if (G > 1) CHECK(mcgpu_burnin_group(&engs[0], G, nburn));     // tuning counters summed over the engines
  else CHECK(mcgpu_burnin(eng, nburn));

  logfile << "Starting main sample loop:  nsamp = " << nsamp << std::endl;
  logfile << "Output after each " << outstep << " steps." << std::endl;
  for (int g = 0; g < G; ++g) { eng = engs[g]; CHECK(mcgpu_sample_begin(eng, nsamp)); }

  // Rows reach MCout in the reference's order: batches of `outstep` steps; inside a batch
  // rank-major blocks; inside a rank block step-major, then chain (mcout.cc:52-94 gathers
  // rank blocks; src/anly/mcpar-analysis.R:80-120 relies on it).
  const int ncol = nparam + 1;
  std::vector<std::vector<Real> > block(G);                // the rows of the current output batch, per engine, kept-step major
  long long batch_kept = 0;                                // kept steps gathered in `block` so far
  int done = 0;
  int next_out = outstep;                                  // outsamples.output() before step outstep, 2 outstep, ... (mcpar.cc:115-119)
  while (done < nsamp) {
    if (done > 0 && done == next_out) {
      logfile << "Beginning output at step " << done << std::endl;
      outsamples.output();
      logfile << "Output finished\n" << std::endl;
      next_out += outstep;
    }
    const int n = std::min(std::min(nsamp - done, next_out - done), piece);   // up to the next output, at most one ring
    if (logging && done % logstep == 0)
      logfile << "sample step " << done << ":\toutsamples size= " << outsamples.size() << "  maxsize = "
              << outsamples.maxsize() << "  ncol= " << outsamples.ncol() << std::endl;
    if (hostlik) {
      for (int k = 0; k < n; ++k) {
        CHECK(mcgpu_step_propose(eng, &ptrial[0]));
        plugin(&ptrial[0], &lytrial[0]);                   // L(nchain, ptrial, lytrial), mcpar.cc:160
        CHECK(mcgpu_step_accept(eng, &lytrial[0]));
      }
    } else if (G == 1) CHECK(mcgpu_sample(eng, n));
    else CHECK(mcgpu_sample_group(&engs[0], G, n));      // one exchange window at a time, engine after engine
    const long long k0 = (done + thin - 1) / thin, k1 = (done + n + thin - 1) / thin;   // kept steps of this piece
    if (k1 > k0) {
      for (int g = 0; g < G; ++g) {
        eng = engs[g];
        block[g].resize((size_t)(batch_kept + k1 - k0) * cg_chains * ncol);
        CHECK(mcgpu_history_read(eng, k0, k1 - k0, &block[g][(size_t)batch_kept * cg_chains * ncol]));
      }
      batch_kept += k1 - k0;
    }
    done += n;
    if ((done == next_out || done == nsamp) && batch_kept > 0) {   // the batch is complete: hand it to MCout rank by rank
      for (int r = 0; r < size; ++r)
        for (long long k = 0; k < batch_kept; ++k)
          outsamples.addrows(&block[r / rpg][((size_t)k * cg_chains + (size_t)(r % rpg) * nchain) * ncol], (size_t)nchain);
      batch_kept = 0;
    }
  }
  outsamples.output();                                   // remaining samples (mcpar.cc:212)

  long long acc = 0, tried = 0, xwait = 0, xwaits = 0;
  mdevice_ms = 0;
  for (int g = 0; g < G; ++g) {
    eng = engs[g];
    CHECK(mcgpu_synchronize(eng));                         // also reports a peer that failed to publish
    mcgpu_stats st;
    CHECK(mcgpu_get_stats(eng, &st));
    acc += st.accepted; tried += st.tried;
    if (st.device_ms > mdevice_ms) mdevice_ms = st.device_ms;
    if (st.exchange_wait_ns > xwait) xwait = st.exchange_wait_ns;
    xwaits += st.exchange_waits;
  }
  maccept = tried ? (double)acc / (double)tried : 0.0;
  mxwait_ms = (double)xwait * 1e-6;
  logfile << "Acceptance rate (main loop) = " << maccept << "  device time = " << mdevice_ms << " ms  ("
          << (double)tchains * (nburn + nsamp) / (mdevice_ms * 1e-3) << " chain-steps/s)" << std::endl;
  if (G > 1)
    logfile << "Exchange wait (slowest engine) = " << mxwait_ms << " ms in " << xwaits << " launches that waited for a peer's pool slots"
            << std::endl;
  return OK;
}
