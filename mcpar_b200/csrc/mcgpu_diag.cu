// mcgpu_diag.cu -- the kernels of the history diagnostics and quantiles and their launchers (mcgpu_diag.cuh).
#include "mcgpu_diag.cuh"
#include <algorithm>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cuda/functional>

namespace mcgpu_diag {

__device__ inline void part_merge(Part &a, const Part &b)
{
  chan_merge(a.cnt, a.mean, a.m2, b.cnt, b.mean, b.m2);
  a.sx += b.sx; a.nf += b.nf; a.mn = fmin(a.mn, b.mn); a.mx = fmax(a.mx, b.mx);
}

// One thread per (hosted chain, column); a CTA holds cpb = DIAG_THREADS / ncol whole chains, so a warp's loads of
// one row are consecutive doubles.  Per thread: pass 1 = the chain's mean, the two split-chain means, min, max and
// the non-finite count; pass 2 = the chain's centred sum of squares; then, DIAG_LAGS lags at a time, the biased
// autocovariances of both split chains, centred on their own means, with a sliding register window.  Outputs:
// chain[j][c] = {1, xbar_c, 0, s2_c, min, max, nonfinite}, split[j][2c + h] = {1, ybar_m, 0, v_m, +inf, -inf, 0},
// lagp[block][j][t] = the CTA's sum over its split chains of gamma_{m,t} (added in chain order).
__global__ void __launch_bounds__(DIAG_THREADS, 2) diag_chain_kernel(DiagRows rows, long long C, int ncol, int n, int L,
                                                                  Part *chain, Part *split, double *lagp)
{
  __shared__ double red[DIAG_LAGS][DIAG_THREADS];
  const int cpb = DIAG_THREADS / ncol, N = n / 2;
  const int ci = threadIdx.x / ncol, j = threadIdx.x % ncol;
  const long long c = (long long)blockIdx.x * cpb + ci;
  const int nblk = (int)min((long long)cpb, C - (long long)blockIdx.x * cpb);
  const bool active = ci < nblk;
  const long long i = c * ncol + j;
  double ybar0 = 0.0, ybar1 = 0.0;
  if (active) {
    double s = 0.0, sh[2] = {0.0, 0.0}, mn = INFINITY, mx = -INFINITY, nf = 0.0;
    for (int k = 0; k < n; ++k) {
      const double x = rows.at(k)[i];
      s += x;
      if (k < N) sh[0] += x;
      if (k >= n - N) sh[1] += x;
      if (!isfinite(x)) nf += 1.0;
      mn = fmin(mn, x); mx = fmax(mx, x);
    }
    const double xbar = s / n;
    ybar0 = sh[0] / N; ybar1 = sh[1] / N;
    double ss = 0.0;
    for (int k = 0; k < n; ++k) { const double z = rows.at(k)[i] - xbar; ss += z * z; }
    chain[(long long)j * C + c] = Part{1.0, xbar, 0.0, ss / (n - 1), mn, mx, nf};
  }
  double v0 = 0.0, v1 = 0.0;
  for (int t0 = 0; t0 <= L; t0 += DIAG_LAGS) {
    double tot[DIAG_LAGS];
#pragma unroll
    for (int k = 0; k < DIAG_LAGS; ++k) tot[k] = 0.0;
    if (active) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int base = h ? n - N : 0; const double yb = h ? ybar1 : ybar0;
        double w[DIAG_LAGS], acc[DIAG_LAGS];
#pragma unroll
        for (int k = 0; k < DIAG_LAGS; ++k) { acc[k] = 0.0; w[k] = t0 + k < N ? rows.at(base + t0 + k)[i] - yb : 0.0; }
#pragma unroll 4
        for (int s = 0; s < N - t0; ++s) {
          const double zs = rows.at(base + s)[i] - yb;
#pragma unroll
          for (int k = 0; k < DIAG_LAGS; ++k) acc[k] = fma(zs, w[k], acc[k]);
#pragma unroll
          for (int k = 0; k < DIAG_LAGS - 1; ++k) w[k] = w[k + 1];
          const int nx = s + t0 + DIAG_LAGS;
          w[DIAG_LAGS - 1] = nx < N ? rows.at(base + nx)[i] - yb : 0.0;
        }
        if (t0 == 0) (h ? v1 : v0) = acc[0] / (N - 1);
#pragma unroll
        for (int k = 0; k < DIAG_LAGS; ++k) tot[k] += acc[k] / N;
      }
    }
#pragma unroll
    for (int k = 0; k < DIAG_LAGS; ++k) red[k][threadIdx.x] = tot[k];
    __syncthreads();
    for (int p = threadIdx.x; p < DIAG_LAGS * ncol; p += blockDim.x) {
      const int k = p / ncol, jj = p % ncol;
      if (t0 + k > L) continue;
      double s = 0.0;
      for (int q = 0; q < nblk; ++q) s += red[k][q * ncol + jj];
      lagp[((long long)blockIdx.x * ncol + jj) * (L + 1) + t0 + k] = s;
    }
    __syncthreads();
  }
  if (active) {
    split[(long long)j * 2 * C + 2 * c] = Part{1.0, ybar0, 0.0, v0, INFINITY, -INFINITY, 0.0};
    split[(long long)j * 2 * C + 2 * c + 1] = Part{1.0, ybar1, 0.0, v1, INFINITY, -INFINITY, 0.0};
  }
}

// One warp per output: merges in[j][g*gs + q*ch + (0 .. min(ch, gs - q*ch)))] (group g, chunk q) into
// out[j][g*nchunk + q], lanes taking every 32nd entry, then a fixed shuffle tree.  to_item (nchunk = 1): the output
// becomes the superchain item {1, mean, 0, Btilde + Wtilde} of nested R-hat, Btilde = M2/(G-1) (0 when G = 1) and
// Wtilde = sum/G.
__global__ void diag_group_kernel(const Part *in, long long nin, int ncol, long long gs, long long ch, int to_item,
                                  Part *out)
{
  const long long nchunk = (gs + ch - 1) / ch, ngroup = nin / gs, nout = ngroup * nchunk;
  const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (wid >= nout * ncol) return;
  const int j = (int)(wid / nout); const long long o = wid % nout, g = o / nchunk, q = o % nchunk;
  const long long lo = g * gs + q * ch, hi = g * gs + min(gs, (q + 1) * ch);
  Part a{0.0, 0.0, 0.0, 0.0, INFINITY, -INFINITY, 0.0};
  for (long long k = lo + lane; k < hi; k += 32) part_merge(a, in[(long long)j * nin + k]);
  for (int off = 1; off < 32; off <<= 1) {
    Part b;
    b.cnt = __shfl_down_sync(0xffffffffu, a.cnt, off); b.mean = __shfl_down_sync(0xffffffffu, a.mean, off);
    b.m2 = __shfl_down_sync(0xffffffffu, a.m2, off); b.sx = __shfl_down_sync(0xffffffffu, a.sx, off);
    b.mn = __shfl_down_sync(0xffffffffu, a.mn, off); b.mx = __shfl_down_sync(0xffffffffu, a.mx, off);
    b.nf = __shfl_down_sync(0xffffffffu, a.nf, off);
    if ((lane & (2 * off - 1)) == 0) part_merge(a, b);
  }
  if (lane) return;
  if (to_item) a = Part{1.0, a.mean, 0.0, (a.cnt > 1 ? a.m2 / (a.cnt - 1) : 0.0) + a.sx / a.cnt, a.mn, a.mx, a.nf};
  out[(long long)j * nout + o] = a;
}

// out[r] = sum over b of in[b * nr + r] (b ascending per lane, then a fixed shuffle tree); one warp per r
__global__ void diag_sum_rows_kernel(const double *in, long long nb, long long nr, double *out)
{
  const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= nr) return;
  double s = 0.0;
  for (long long b = lane; b < nb; b += 32) s += in[b * nr + r];
  for (int off = 1; off < 32; off <<= 1) {
    const double o = __shfl_down_sync(0xffffffffu, s, off);
    if ((lane & (2 * off - 1)) == 0) s += o;
  }
  if (!lane) out[r] = s;
}

// One radix pass (digit `pass` of 8, most significant first) over the elements of columns [j0, j1) of `nrows` kept
// steps starting at `rows`.  Column j has slots [soff[j - j0], soff[j - j0 + 1]), one per distinct prefix (the key's
// 8*pass high bits) still holding a target rank; an element whose prefix matches a slot counts in that slot's bin of
// its next digit.  Pass 0 also counts NaN per column.  Histograms are per-CTA uint32 in shared memory (warp-
// aggregated atomics), then added to hist[slot][256] (uint64).
__global__ void diag_radix_kernel(const double *rows, long long nrows, int ncol, int j0, int j1, int pass,
                                  const uint64_t *prefix, const int *soff, unsigned long long *hist,
                                  unsigned long long *nan_count)
{
  extern __shared__ unsigned int qs[];
  const int nj = j1 - j0, nslot = soff[nj];
  unsigned int *sh = qs, *snan = qs + nslot * QSEL_BINS;
  for (int k = threadIdx.x; k < nslot * QSEL_BINS + nj; k += blockDim.x) qs[k] = 0;
  __syncthreads();
  const int hi_shift = 64 - 8 * pass, dg_shift = 56 - 8 * pass;
  const long long total = nrows * ncol;
  for (long long base = (long long)blockIdx.x * blockDim.x; base < total; base += (long long)gridDim.x * blockDim.x) {
    const long long idx = base + threadIdx.x;
    int bin = -1;
    if (idx < total) {
      const int j = (int)(idx % ncol);
      if (j >= j0 && j < j1) {
        const double x = rows[idx];
        if (pass == 0 && isnan(x)) atomicAdd(snan + (j - j0), 1u);
        const uint64_t key = diag_key((uint64_t)__double_as_longlong(x));
        int slot = soff[j - j0];
        if (pass > 0) {
          const uint64_t pf = key >> hi_shift;
          const int end = soff[j - j0 + 1];
          while (slot < end && prefix[slot] != pf) ++slot;
          if (slot == end) slot = -1;
        }
        if (slot >= 0) bin = slot * QSEL_BINS + (int)((key >> dg_shift) & 0xff);
      }
    }
    const unsigned int peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(sh + bin, (unsigned int)__popc(peers));
  }
  __syncthreads();
  for (int k = threadIdx.x; k < nslot * QSEL_BINS; k += blockDim.x)
    if (sh[k]) atomicAdd(hist + k, (unsigned long long)sh[k]);
  if (pass == 0)
    for (int k = threadIdx.x; k < nj; k += blockDim.x)
      if (snan[k]) atomicAdd(nan_count + j0 + k, (unsigned long long)snan[k]);
}

cudaError_t diag_chain(const DiagRows &rows, long long C, int ncol, int n, int L, Part *chain, Part *split, double *lagp,
                       cudaStream_t st)
{
  const long long cpb = DIAG_THREADS / ncol;
  diag_chain_kernel<<<(unsigned)((C + cpb - 1) / cpb), DIAG_THREADS, 0, st>>>(rows, C, ncol, n, L, chain, split, lagp);
  return cudaGetLastError();
}

cudaError_t diag_group(const Part *in, long long nin, int ncol, long long gs, long long ch, int to_item, Part *out,
                       cudaStream_t st)
{
  const long long nwarp = nin / gs * ((gs + ch - 1) / ch) * ncol, warps = 8;
  diag_group_kernel<<<(unsigned)((nwarp + warps - 1) / warps), 32 * warps, 0, st>>>(in, nin, ncol, gs, ch, to_item, out);
  return cudaGetLastError();
}

cudaError_t diag_sum_rows(const double *in, long long nb, long long nr, double *out, cudaStream_t st)
{
  diag_sum_rows_kernel<<<(unsigned)((nr + 7) / 8), 256, 0, st>>>(in, nb, nr, out);
  return cudaGetLastError();
}

cudaError_t diag_radix(const double *rows, long long nrows, int ncol, int j0, int j1, int pass, const uint64_t *prefix,
                       const int *soff, unsigned long long *hist, unsigned long long *nan_count, size_t smem,
                       cudaStream_t st)
{
  int dev = 0, nsm = 0, occ = 0;
  cudaError_t r = cudaGetDevice(&dev);
  if (r == cudaSuccess) r = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  if (r == cudaSuccess) r = cudaFuncSetAttribute(diag_radix_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (r == cudaSuccess) r = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, diag_radix_kernel, 256, smem);
  if (r != cudaSuccess) return r;
  diag_radix_kernel<<<(unsigned)(std::max(occ, 1) * nsm), 256, smem, st>>>(rows, nrows, ncol, j0, j1, pass, prefix, soff,
                                                                          hist, nan_count);
  return cudaGetLastError();
}

// ---- rank normalisation -------------------------------------------------------------------------------------------
__device__ inline double key_value(uint64_t k) { return __longlong_as_double((long long)diag_unkey(k)); }

// One thread per draw (kept step k, hosted chain c) of column j; see rank_keys in mcgpu_diag.cuh.  -0.0 is keyed as
// +0.0 because rankdata ties them.
__global__ void rank_keys_kernel(DiagRows rows, long long C, int ncol, int j, int n, const uint64_t *mid, double q05,
                                 double q95, uint64_t *keys, uint32_t *pos, double *series,
                                 unsigned long long *nonfinite)
{
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int N = n / 2;
  bool bad = false;
  if (t < (long long)n * C) {
    const int k = (int)(t / C);
    const long long c = t - (long long)k * C;
    double x = rows.at(k)[c * ncol + j];
    bad = !isfinite(x);
    if (k < N || k >= n - N) {
      const long long i = (long long)(k < N ? k : k - (n - 2 * N)) * C + c;
      if (mid) {
        const double med = (key_value(mid[(long long)N * C - 1]) + key_value(mid[(long long)N * C])) / 2;
        x = fabs(x - med);
      } else {
        series[i * RANK_COLS + 2] = x <= q05 ? 1.0 : 0.0;
        series[i * RANK_COLS + 3] = x <= q95 ? 1.0 : 0.0;
      }
      keys[i] = diag_key((uint64_t)__double_as_longlong(x == 0.0 ? 0.0 : x));
      pos[i] = (uint32_t)i;
    }
  }
  if (!mid) {
    const unsigned int m = __ballot_sync(0xffffffffu, bad);
    if (m && (threadIdx.x & 31) == 0) atomicAdd(nonfinite, (unsigned long long)__popc(m));
  }
}

// head[i] = i where a run of equal sorted keys starts, else 0; a running max then gives each entry its run's start
__global__ void rank_heads_kernel(const uint64_t *keys, long long S2, uint32_t *head)
{
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S2) head[i] = (i == 0 || keys[i] != keys[i - 1]) ? (uint32_t)i : 0u;
}

// the last entry of each run stores its index at the run's start: end[start] = the run's last sorted index
__global__ void rank_tails_kernel(const uint64_t *keys, const uint32_t *start, long long S2, uint32_t *end)
{
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S2 && (i == S2 - 1 || keys[i] != keys[i + 1])) end[start[i]] = (uint32_t)i;
}

// a run over sorted indices [a, b] has the average rank (a + b)/2 + 1 (exact in fp64); its normal score
// Phi^-1((rank - 3/8) / (S2 + 1/4)) goes to series[pos][col]
__global__ void rank_scores_kernel(const uint32_t *start, const uint32_t *end, const uint32_t *pos, long long S2,
                                   double *series, int col)
{
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S2) return;
  const uint32_t a = start[i], b = end[a];
  const double rank = ((double)a + (double)b) / 2 + 1.0;
  series[(long long)pos[i] * RANK_COLS + col] = normcdfinv((rank - 0.375) / ((double)S2 + 0.25));
}

cudaError_t rank_temp_bytes(long long S2, size_t *bytes)
{
  cub::DoubleBuffer<uint64_t> kb(nullptr, nullptr);
  cub::DoubleBuffer<uint32_t> pb(nullptr, nullptr);
  size_t sort = 0, scan = 0;
  cudaError_t r = cub::DeviceRadixSort::SortPairs(nullptr, sort, kb, pb, S2, 0, 64);
  if (r == cudaSuccess)
    r = cub::DeviceScan::InclusiveScan(nullptr, scan, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                       cuda::maximum<uint32_t>{}, (uint32_t)S2);
  *bytes = std::max(sort, scan);
  return r;
}

cudaError_t rank_keys(const DiagRows &rows, long long C, int ncol, int j, int n, const uint64_t *mid, double q05,
                      double q95, uint64_t *keys, uint32_t *pos, double *series, unsigned long long *nonfinite,
                      cudaStream_t st)
{
  rank_keys_kernel<<<(unsigned)((n * C + 255) / 256), 256, 0, st>>>(rows, C, ncol, j, n, mid, q05, q95, keys, pos,
                                                                     series, nonfinite);
  return cudaGetLastError();
}

cudaError_t rank_scores(uint64_t *keys[2], uint32_t *pos[2], long long S2, void *temp, size_t temp_bytes, double *series,
                        int col, cudaStream_t st)
{
  cub::DoubleBuffer<uint64_t> kb(keys[0], keys[1]);
  cub::DoubleBuffer<uint32_t> pb(pos[0], pos[1]);
  cudaError_t r = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, kb, pb, S2, 0, 64, st);
  if (r != cudaSuccess) return r;
  keys[0] = kb.Current(); keys[1] = kb.Alternate(); pos[0] = pb.Current(); pos[1] = pb.Alternate();
  uint32_t *start = reinterpret_cast<uint32_t*>(keys[1]), *end = start + S2;   // the spare key buffer, 2 S2 words
  const unsigned nb = (unsigned)((S2 + 255) / 256);
  rank_heads_kernel<<<nb, 256, 0, st>>>(keys[0], S2, end);
  if ((r = cudaGetLastError()) != cudaSuccess) return r;
  r = cub::DeviceScan::InclusiveScan(temp, temp_bytes, (const uint32_t*)end, start, cuda::maximum<uint32_t>{},
                                     (uint32_t)S2, st);
  if (r != cudaSuccess) return r;
  rank_tails_kernel<<<nb, 256, 0, st>>>(keys[0], start, S2, end);
  if ((r = cudaGetLastError()) != cudaSuccess) return r;
  rank_scores_kernel<<<nb, 256, 0, st>>>(start, end, pos[0], S2, series, col);
  return cudaGetLastError();
}

}  // namespace mcgpu_diag
