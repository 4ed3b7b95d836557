// vlfunc.hh -- the likelihood plugin surface, kept from the reference (src/vlfunc.hh:9-12):
//   virtual int operator()(int npset, const Real *x, Real *restrict y) = 0;
// x holds npset parameter sets, chain-major {a1,b1,...,a2,b2,...}; y receives npset
// LOG-likelihoods; the functor knows nparam itself; the return code is reserved.
// Real is double here (the reference is float; see DESIGN.md "precision").
#ifndef MCPAR_B200_VLFUNC_HH_
#define MCPAR_B200_VLFUNC_HH_
#include <string>
#include <vector>

#ifndef restrict
#define restrict __restrict__            /* the reference gets this from -Drestrict=__restrict__ (src/Makefile:12) */
#endif

typedef double Real;

class VLFunc {
public:
  virtual int operator()(int npset, const Real *x, Real *restrict y) = 0;
  virtual ~VLFunc() {}
};

// A likelihood the B200 engine can run inside its fused step kernel.  The batched
// operator() is also served by the GPU (mcgpu_loglik); there is no host evaluation.
class DeviceVLFunc : public VLFunc {
public:
  virtual int lik_id() const = 0;                       // MCGPU_* id of the device functor
  virtual int nparam() const = 0;
  virtual const std::vector<double> &params() const { return mpar; }
  virtual const char *plugin_path() const { return 0; }   // a plugin cubin (DevicePlugin) instead of a built-in id
  int operator()(int npset, const Real *x, Real *restrict y);     // evaluates on the GPU
  int device;                                           // CUDA ordinal used by operator()
protected:
  DeviceVLFunc() : device(0) {}
  std::vector<double> mpar;
};

// A user-written likelihood compiled into a plugin cubin (include/mcgpu_plugin.cuh, python -m mcpar_b200.plugin):
// MCPar::run loads it into every engine (mcgpu_set_likelihood_plugin) and operator() evaluates it on the GPU
// (mcgpu_loglik_plugin).  par is handed to the functor unchanged.
class DevicePlugin : public DeviceVLFunc {
  const std::string path; const int n;
public:
  DevicePlugin(const std::string &cubin_path, int nparam, const std::vector<double> &par = std::vector<double>());
  int lik_id() const; int nparam() const { return n; }
  const char *plugin_path() const { return path.c_str(); }
};

#endif
