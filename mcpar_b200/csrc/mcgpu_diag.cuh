// mcgpu_diag.cuh -- device reductions of the sample history for convergence diagnostics (split and nested R-hat,
// multi-chain ESS, MCSE), exact posterior quantiles and the rank normalisation of ArviZ's rank diagnostics
// (include/mcgpu.h: mcgpu_history_diag_partials, mcgpu_history_quantiles, mcgpu_history_rank_diag): the types and
// launchers mcgpu_api.cu uses; the kernels are in mcgpu_diag.cu.
//
// The kernels are a translation unit (a device module) of their own: a sampling engine never loads them, and the
// modules a peer-to-peer engine loads up front (DESIGN.md section 6) do not grow with them.
//
// The history is a ring of kept steps [ring step][hosted chain][ncol]; the valid rows are at most two contiguous
// ring ranges (hist_segments).  DiagRows maps a logical row s (0 = oldest valid kept step) to its ring row.
//
// Every floating-point reduction runs in a fixed order (a per-thread sequence, a fixed shuffle tree, a fixed
// sequential sum over a CTA's chains): no floating-point atomics, so a repeated call returns the same bits.
// Integer counters (quantile histograms, NaN counts) use atomics; CUB's radix sort and scan are deterministic.
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

// ---- rank normalisation (mcgpu_history_rank_diag) ----------------------------------------------------------------
// The split draws of one column (S2 = 2CN of them) become the series [2N][C][RANK_COLS]: column 0 the normal scores
// of their ranks, column 1 those of the folded draws |y - median|, columns 2 and 3 the tail indicators.  Position
// i = r C + c is split row r of hosted chain c (rows N..2N-1 are kept steps n-N..n-1).
constexpr int RANK_COLS = 4;
constexpr int RANK_SCORE_LAUNCHES = 5;   // rank_scores: the sort, 3 kernels, the scan

// CUB temp storage rank_scores needs for S2 pairs
cudaError_t rank_temp_bytes(long long S2, size_t *bytes);
// keys, pos := the sort keys and positions of column j's split draws.  mid == nullptr: of the draws; series
// columns 2 and 3 := I(x <= q05), I(x <= q95); *nonfinite += the non-finite draws of all n kept steps.  Else: of the
// folded draws, with mid the sorted keys of the draws (the median is the mean of its middle two).
cudaError_t rank_keys(const DiagRows &rows, long long C, int ncol, int j, int n, const uint64_t *mid, double q05,
                      double q95, uint64_t *keys, uint32_t *pos, double *series, unsigned long long *nonfinite,
                      cudaStream_t st);
// sorts the pairs (keys[0], pos[0]) through the buffers keys[1], pos[1] (on return keys[0], pos[0] name the sorted
// pairs, keys[1] the spare buffer of 8 S2 bytes) and writes series[i][col] = the normal score of the average rank
cudaError_t rank_scores(uint64_t *keys[2], uint32_t *pos[2], long long S2, void *temp, size_t temp_bytes, double *series,
                        int col, cudaStream_t st);

}  // namespace mcgpu_diag
