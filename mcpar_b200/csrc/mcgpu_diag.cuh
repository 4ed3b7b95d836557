// mcgpu_diag.cuh -- device reductions of the sample history for convergence diagnostics (split and nested R-hat,
// multi-chain ESS, MCSE) and exact posterior quantiles (include/mcgpu.h: mcgpu_history_diag_partials,
// mcgpu_history_quantiles): the types and launchers mcgpu_api.cu uses; the kernels are in mcgpu_diag.cu.
//
// The kernels are a translation unit (a device module) of their own: a sampling engine never loads them, and the
// modules a peer-to-peer engine loads up front (DESIGN.md section 6) do not grow with them.
//
// The history is a ring of kept steps [ring step][hosted chain][ncol]; the valid rows are at most two contiguous
// ring ranges (hist_segments).  DiagRows maps a logical row s (0 = oldest valid kept step) to its ring row.
//
// Every floating-point reduction runs in a fixed order (a per-thread sequence, a fixed shuffle tree, a fixed
// sequential sum over a CTA's chains): no floating-point atomics, so a repeated call returns the same bits.
// Integer counters (quantile histograms, NaN counts) use atomics.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

namespace mcgpu_diag {

struct DiagRows {
  const double *p0, *p1;   // ring row of logical rows [0, c0) and of [c0, n)
  long long c0, row;       // row = doubles per kept step (hosted chains * ncol)
  __device__ __forceinline__ const double *at(int s) const { return s < c0 ? p0 + (long long)s * row : p1 + (long long)(s - c0) * row; }
};

// (count, mean, M2) of a set of values plus a plain sum, the min, the max and a count of non-finite values.
// An empty partial has cnt = 0, mn = +inf, mx = -inf.
struct Part { double cnt, mean, m2, sx, mn, mx, nf; };

// Chan et al.'s pairwise update of (count, mean, M2); also used by the host finalize so both sides merge alike
__host__ __device__ inline void chan_merge(double &na, double &ma, double &m2a, double nb, double mb, double m2b)
{
  if (nb == 0) return;
  if (na == 0) { na = nb; ma = mb; m2a = m2b; return; }
  const double n = na + nb, dl = mb - ma;
  ma = ma + dl * (nb / n);
  m2a = m2a + m2b + dl * dl * (na * nb / n);
  na = n;
}

constexpr int DIAG_THREADS = 256;
constexpr int DIAG_LAGS = 8;       // lags accumulated in registers per pass over a split chain

// ---- quantiles: radix select on order-preserving keys ------------------------------------------------------------
__host__ __device__ inline uint64_t diag_key(uint64_t u) { return (u >> 63) ? ~u : u | 0x8000000000000000ull; }
__host__ __device__ inline uint64_t diag_unkey(uint64_t k) { return (k >> 63) ? k & 0x7fffffffffffffffull : ~k; }

constexpr int QSEL_BINS = 256;

// Launchers (mcgpu_diag.cu); each returns the launch's error.  diag_chain: one CTA per DIAG_THREADS / ncol chains.
cudaError_t diag_chain(const DiagRows &rows, long long C, int ncol, int n, int L, Part *chain, Part *split, double *lagp,
                       cudaStream_t st);
cudaError_t diag_group(const Part *in, long long nin, int ncol, long long gs, long long ch, int to_item, Part *out,
                       cudaStream_t st);
cudaError_t diag_sum_rows(const double *in, long long nb, long long nr, double *out, cudaStream_t st);
// one radix pass with `smem` bytes of histograms per CTA, as many CTAs as fit on the device's SMs
cudaError_t diag_radix(const double *rows, long long nrows, int ncol, int j0, int j1, int pass, const uint64_t *prefix,
                       const int *soff, unsigned long long *hist, unsigned long long *nan_count, size_t smem,
                       cudaStream_t st);

}  // namespace mcgpu_diag
