// likelihoods.cc -- host side of the VLFunc plugin surface: parameter carriers for the
// device functors; the batched operator() is evaluated ON THE GPU through mcgpu_loglik
// (there is deliberately no host arithmetic here).  Constructor checks and messages follow
// src/rosenbrock.hh:13-16,27-30,42-48.
#include "rosenbrock.hh"
#include "../../include/mcgpu.h"
#include <stdio.h>
#include <stdlib.h>

int DeviceVLFunc::operator()(int npset, const Real *x, Real *restrict y)
{
  const std::vector<double> &p = params();
  const int rc = plugin_path()
      ? mcgpu_loglik_plugin(device, plugin_path(), nparam(), p.empty() ? 0 : &p[0], (int)p.size(), npset, x, y)
      : mcgpu_loglik(device, lik_id(), nparam(), p.empty() ? 0 : &p[0], (int)p.size(), npset, x, y);
  if (rc != MCGPU_OK) {                      // no CPU fallback: fail loudly
    fprintf(stderr, "VLFunc: GPU likelihood evaluation failed (%d): %s\n", rc, mcgpu_last_error(0));
    abort();
  }
  return 0;
}

Rosenbrock1::Rosenbrock1(int nc) : n(nc)
{
  if (n < 2 || n % 2 != 0) throw("N for Rosenbrock1 must be even and >= 2");
}
int Rosenbrock1::lik_id() const { return MCGPU_ROSENBROCK1; }

Rosenbrock2::Rosenbrock2(int nc) : n(nc)
{
  if (n < 2) throw("N for Rosenbrock2 must be >= 2");
}
int Rosenbrock2::lik_id() const { return MCGPU_ROSENBROCK2; }

Gaussian::Gaussian(int nc, const Real muin[], const Real sig2[]) : n(nc)
{
  if (nc != 2) throw("Invalid specification.  N for Gaussian must == 2.");
  mpar.resize(4);
  for (int i = 0; i < 2; ++i) { mpar[i] = muin ? muin[i] : 0.0; mpar[2 + i] = sig2 ? sig2[i] : 1.0; }
}
int Gaussian::lik_id() const { return MCGPU_GAUSSIAN; }

DualGaussian::DualGaussian(Real win) { mpar.assign(1, win); }
int DualGaussian::lik_id() const { return MCGPU_DUALGAUSSIAN; }

GaussMix::GaussMix(int nparam, int ncomp, const Real *mu, const Real *sig2, const Real *w) : n(nparam), K(ncomp)
{
  if (n < 1 || K < 1) throw("GaussMix needs nparam >= 1 and ncomp >= 1");
  mpar.reserve(1 + 2 * (size_t)K * n + K);
  mpar.push_back((double)K);
  mpar.insert(mpar.end(), mu, mu + (size_t)K * n);
  mpar.insert(mpar.end(), sig2, sig2 + (size_t)K * n);
  mpar.insert(mpar.end(), w, w + K);
}
int GaussMix::lik_id() const { return MCGPU_GAUSSMIX; }

DevicePlugin::DevicePlugin(const std::string &cubin_path, int nparam, const std::vector<double> &par) : path(cubin_path), n(nparam)
{
  if (n < 2 || n > 16 || n % 2 != 0) throw("a device plugin has an even nparam in 2..16");
  mpar = par;
}
int DevicePlugin::lik_id() const { return MCGPU_DEVICE_PLUGIN; }
