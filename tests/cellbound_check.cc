// Host check of cell_bounds2 (mcpar_b200/csrc/mcgpu_cellbound.cuh): for pools of several shapes, cells of the grid the
// table kernel lays over them (5 sigma beyond every slot, 64 cells per axis, each dilated by 1/64 of its width), and
// points inside the dilated cells (random, corners, edge midpoints), the acceptance ratio of remote_exact,
//     R(x) = max(FPEPS, max_s Q_s(x)) / (FPEPS + sum_s Q_s(x)),
// evaluated in x86 extended precision must lie in [R_lo, R_hi], and the stored fp32 pair must lie outside that.
// Prints one JSON line per pool shape: points checked, violations, decidable cells and the median relative width.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <random>
#include <vector>
#include "../mcpar_b200/csrc/mcgpu_cellbound.cuh"

static long double ratio_ld(const std::vector<double> &pool, int M, double x0, double x1)
{
  long double qmax = 1.0e-14L, qsum = 1.0e-14L;
  for (int s = 0; s < M; ++s) {
    long double a = 0.0L;
    const double x[2] = {x0, x1};
    for (int i = 0; i < 2; ++i) {
      double m, h; mcgpu::cell_slot(pool.data(), s, i, m, h);     // the doubles the kernels hold
      const long double y = (long double)x[i] - (long double)m;
      a += (long double)h * y * y;
    }
    const long double q = expl(a);
    qsum += q; qmax = q > qmax ? q : qmax;
  }
  return qmax / qsum;
}

struct Shape { const char *name; int M; double mu_scale, sig_lo, sig_hi; int kind; };

int main()
{
  const int G = 64;
  const Shape shapes[] = {
    {"random", 16, 6.0, 0.5, 2.0, 0},
    {"widths_spread_60x", 16, 6.0, 0.05, 3.0, 0},
    {"means_300_sigma_out", 16, 300.0, 0.5, 2.0, 0},
    {"pool_256", 256, 10.0, 0.2, 2.0, 0},
    {"plateau_like", 16, 3.0, 1.0, 1.0, 1},
    {"plateau_like_256", 256, 3.0, 1.0, 1.0, 1},
    {"sigma_1e-7", 16, 1.0, 1.0e-7, 1.0e-7, 2},
  };
  std::mt19937_64 rng(12345);
  std::uniform_real_distribution<double> U01(0.0, 1.0);
  std::normal_distribution<double> N01(0.0, 1.0);
  for (const Shape &sh : shapes) {
    long long points = 0, viol = 0, cells = 0, decidable = 0, store_viol = 0;
    std::vector<double> widths;
    for (int rep = 0; rep < 6; ++rep) {
      const int M = sh.M;
      std::vector<double> pool((size_t)M * 4);
      const double base[2] = {sh.mu_scale * (2 * U01(rng) - 1), sh.mu_scale * (2 * U01(rng) - 1)};
      for (int s = 0; s < M; ++s)
        for (int i = 0; i < 2; ++i) {
          double m, sd;
          if (sh.kind == 1) {                  // running means / variances of chains that adopt each other's moments
            m = base[i] + 0.05 * N01(rng); sd = 1.5 * (1.0 + 0.02 * N01(rng));
          } else if (sh.kind == 2) {           // the first windows: every chain still at its start
            m = base[i] + 1e-6 * N01(rng); sd = sh.sig_lo * (1.0 + 0.5 * U01(rng));
          } else {
            m = sh.mu_scale * (2 * U01(rng) - 1);
            sd = std::exp(std::log(sh.sig_lo) + (std::log(sh.sig_hi) - std::log(sh.sig_lo)) * U01(rng));
          }
          pool[(s * 2 + i) * 2] = m; pool[(s * 2 + i) * 2 + 1] = sd * sd;
        }
      // the grid of the table kernel
      double o[2], inv[2];
      for (int i = 0; i < 2; ++i) {
        double lo = INFINITY, hi = -INFINITY;
        for (int s = 0; s < M; ++s) {
          const double m = pool[(s * 2 + i) * 2], sd = std::sqrt(pool[(s * 2 + i) * 2 + 1]);
          lo = std::min(lo, m - 5.0 * sd); hi = std::max(hi, m + 5.0 * sd);
        }
        o[i] = (double)mcgpu::cell_f32_down(lo);
        inv[i] = (double)(float)((double)G / (hi - o[i]));
      }
      for (int t = 0; t < 400; ++t) {
        const int gx = (int)(U01(rng) * G), gy = (int)(U01(rng) * G);
        const double iw[2] = {1.0 / inv[0], 1.0 / inv[1]};
        const double c0 = o[0] + (gx + 0.5) * iw[0], c1 = o[1] + (gy + 0.5) * iw[1];
        const double w0 = (0.5 + 1.0 / 64.0) * iw[0] * (1.0 + 1e-12), w1 = (0.5 + 1.0 / 64.0) * iw[1] * (1.0 + 1e-12);
        double rlo, rhi;
        mcgpu::cell_bounds2(pool.data(), M, c0, c1, w0, w1, 0, 1, mcgpu::CellRedSelf(), rlo, rhi);
        float flo, fhi;
        mcgpu::cell_store_bounds(rlo, rhi, flo, fhi);
        ++cells;
        if (rhi <= 1.0) { ++decidable; widths.push_back((rhi - rlo) / std::max(rhi, 1e-300)); }
        if (!((double)flo <= rlo && (double)fhi >= std::min(rhi, 1.0))) ++store_viol;
        for (int q = 0; q < 16; ++q) {
          double x0, x1;
          if (q < 4) { x0 = c0 + ((q & 1) ? w0 : -w0); x1 = c1 + ((q & 2) ? w1 : -w1); }          // corners
          else if (q < 8) { const int e = q - 4; x0 = c0 + (e == 0 ? w0 : e == 1 ? -w0 : 0.0); x1 = c1 + (e == 2 ? w1 : e == 3 ? -w1 : 0.0); }
          else { x0 = c0 + w0 * (2 * U01(rng) - 1); x1 = c1 + w1 * (2 * U01(rng) - 1); }
          const long double R = ratio_ld(pool, M, x0, x1);
          ++points;
          if (!(R >= (long double)rlo && R <= (long double)rhi)) ++viol;
        }
      }
    }
    std::sort(widths.begin(), widths.end());
    const double med = widths.empty() ? -1.0 : widths[widths.size() / 2];
    printf("{\"shape\": \"%s\", \"points\": %lld, \"violations\": %lld, \"store_violations\": %lld, \"cells\": %lld, "
           "\"decidable\": %lld, \"median_rel_width\": %.6g}\n", sh.name, points, viol, store_viol, cells, decidable, med);
  }
  return 0;
}
