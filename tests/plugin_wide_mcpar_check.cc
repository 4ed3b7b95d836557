// tests/plugin_wide_mcpar_check.cc -- a wide device likelihood plugin through MCPar::run (built and run by
// tests/test_gpu_plugin_wide.py).  DevicePlugin(<rosen1_wide cubin>, d) is the built-in wide Rosenbrock1 typed in
// again: with coin_group = 0 both run on the wide kernels, so MCPar::run with it must give the parameter columns of
// MCPar::run with Rosenbrock1(d) bit for bit, on one engine or sharded over ngpu engines.  The log-likelihood column
// may differ in the last bits for a chain that never moved (the built-in's initial values come from the exact unit).
// With the default coin_group (one coin per rank) MCPar::run must refuse the plugin and exit with the ABI's message.
// Usage: plugin_wide_mcpar_check <cubin> <d> <ngpu> [remote_mode | refuse].  Prints "ok <rows>".
#include <iostream>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "mcpar.hh"
#include "rosenbrock.hh"
#include "mcout.hh"

int main(int argc, char *argv[])
{
  if (argc < 4) { std::cout << "usage: plugin_wide_mcpar_check <cubin> <d> <ngpu> [remote_mode | refuse]\n"; return 2; }
  const int d = atoi(argv[2]), ngpu = atoi(argv[3]);
  const bool refuse = argc > 4 && !strcmp(argv[4], "refuse");
  const int remote_mode = argc > 4 && !refuse ? atoi(argv[4]) : 0;
  const int ranks = 16, nc = 4, nsamp = 60, nburn = 120;
  std::vector<Real> pinit((size_t)nc * d);
  const Real base[4][2] = {{0.0, 0.0}, {2.0, 2.0}, {0.0, 1.5}, {0.0, -2.0}};
  for (int c = 0; c < nc; ++c)
    for (int i = 0; i < d; ++i) pinit[(size_t)c * d + i] = base[c][i % 2];
  MCout a(d, 0, 0), b(d, 0, 0);
  DevicePlugin P(argv[1], d);
  Rosenbrock1 R(d);
  {
    MCPar m(d, nc, ranks, 0, 0.7);
    m.pool_m = 8; m.remote_mode = remote_mode; m.ngpu = ngpu;
    if (!refuse) m.coin_group = 0;                     // the wide kernels draw one local / remote coin per step for the job
    if (m.run(nsamp, nburn, &pinit[0], P, a) != MCPar::OK) { std::cout << "plugin run failed\n"; return 1; }
    if (refuse) { std::cout << "plugin run with per-rank coins was not refused\n"; return 1; }
  }
  {
    MCPar m(d, nc, ranks, 0, 0.7);
    m.pool_m = 8; m.remote_mode = remote_mode; m.ngpu = ngpu; m.coin_group = 0;
    if (m.run(nsamp, nburn, &pinit[0], R, b) != MCPar::OK) { std::cout << "built-in run failed\n"; return 1; }
  }
  if (a.size() != b.size() || a.size() != nsamp * nc * ranks) { std::cout << "size mismatch " << a.size() << " " << b.size() << "\n"; return 1; }
  long diff = 0, ldiff = 0;
  for (int r = 0; r < a.size(); ++r) {
    const Real *p = a.getpset(r), *q = b.getpset(r);
    for (int i = 0; i < d; ++i) diff += p[i] != q[i];
    ldiff += std::fabs(a.getlval(r) - b.getlval(r)) > 1e-15 * std::fabs(b.getlval(r));
  }
  std::cout << (diff == 0 && ldiff == 0 ? "ok " : "MISMATCH ") << a.size() << " " << diff << " " << ldiff << "\n";
  return 0;
}
