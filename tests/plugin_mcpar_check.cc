// tests/plugin_mcpar_check.cc -- a device likelihood plugin through MCPar::run (built and run by tests/test_gpu_plugin.py).
// DevicePlugin(<rosen1_restated cubin>, 2) is the built-in Rosenbrock1 typed in again as a plugin: its step kernels are
// the same template with the same arithmetic, so MCPar::run with it must give the rows of MCPar::run with
// Rosenbrock1(2) bit for bit, on one engine or sharded over ngpu engines.  The batched operator() of the plugin must
// agree with the built-in's to rounding (the built-in batch evaluation runs without FMA contraction).  Usage: plugin_mcpar_check <cubin> <ngpu> [remote_mode].  Prints "ok <rows>".
#include <iostream>
#include <cmath>
#include <cstdlib>
#include <vector>
#include "mcpar.hh"
#include "rosenbrock.hh"
#include "mcout.hh"

int main(int argc, char *argv[])
{
  if (argc < 3) { std::cout << "usage: plugin_mcpar_check <cubin> <ngpu> [remote_mode]\n"; return 2; }
  const int ngpu = atoi(argv[2]), remote_mode = argc > 3 ? atoi(argv[3]) : 0;
  const int ranks = 16, nc = 4, nsamp = 60, nburn = 120;
  const Real pinit[8] = {0.0, 0.0, 2.0, 2.0, 0.0, 1.5, 0.0, -2.0};
  MCout a(2, 0, 0), b(2, 0, 0);
  DevicePlugin P(argv[1], 2);
  Rosenbrock1 R(2);
  {
    MCPar m(2, nc, ranks, 0, 0.7);
    m.pool_m = 8; m.remote_mode = remote_mode; m.ngpu = ngpu;
    if (m.run(nsamp, nburn, pinit, P, a) != MCPar::OK) { std::cout << "plugin run failed\n"; return 1; }
  }
  {
    MCPar m(2, nc, ranks, 0, 0.7);
    m.pool_m = 8; m.remote_mode = remote_mode; m.ngpu = ngpu;
    if (m.run(nsamp, nburn, pinit, R, b) != MCPar::OK) { std::cout << "built-in run failed\n"; return 1; }
  }
  if (a.size() != b.size() || a.size() != nsamp * nc * ranks) { std::cout << "size mismatch " << a.size() << " " << b.size() << "\n"; return 1; }
  long diff = 0;
  for (int r = 0; r < a.size(); ++r) {
    const Real *p = a.getpset(r), *q = b.getpset(r);
    diff += a.getlval(r) != b.getlval(r) || p[0] != q[0] || p[1] != q[1];
  }
  std::vector<Real> ya(ranks * nc), yb(ranks * nc), x(2 * ranks * nc);
  for (size_t i = 0; i < x.size(); ++i) x[i] = a.getpset((int)(i / 2))[i % 2];
  P(ranks * nc, &x[0], &ya[0]); R(ranks * nc, &x[0], &yb[0]);
  long ydiff = 0;
  for (size_t i = 0; i < ya.size(); ++i) ydiff += std::fabs(ya[i] - yb[i]) > 1e-12 * (1 + std::fabs(yb[i]));   // plugin: FMA contraction on, built-in mcgpu_loglik: off
  std::cout << (diff == 0 && ydiff == 0 ? "ok " : "MISMATCH ") << a.size() << " " << diff << " " << ydiff << "\n";
  return 0;
}
