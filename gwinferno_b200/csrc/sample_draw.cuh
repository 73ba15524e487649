// Per-sample population log-weights and weighted draws from them, on the device (gwi_sample_log_weights /
// gwi_draw_samples, include/gwi.h): the population-reweighted event posteriors and the posterior-predictive check of the
// reference (gwinferno/pipeline/analysis.py:321-355: numpyro's random.choice(p = w / sum w) per event and over the found
// injections).  Not on the likelihood path: nothing here is launched by the likelihood calls.
//
//   sample_logw_kernel    one thread per padded stream position: the full log-weight of its sample (static column, spline
//                         pieces, linear and parametric terms, every normaliser) scattered to its catalog position through
//                         the plan's sample index;
//   draw_tile_max_kernel  per tile of DRAW_TILE catalog-order samples: max;
//   draw_seg_max_kernel   per segment (one warp): max over its tiles;
//   draw_tile_sum_kernel  per tile: sum of exp(x - segment max) in sample order;
//   draw_scan_kernel      per segment: inclusive prefix over its tiles in tile order;
//   draw_kernel           per draw: u from Philox4x32-10, r = u total, binary search over the tile prefixes, then a scan in
//                         sample order inside the one tile.
// Everything after the log-weight pass runs on catalog-order arrays with a fixed tiling, so the draws do not depend on the
// plan geometry (kernel, chunk length, deep dims, builder).
//
// Part of the kernels.cu translation unit (included at its end), like the other launch helpers that api.cu calls.
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <vector>

#include "dev_structs.h"
#include "philox.h"
#include "stream.cuh"

namespace gwi {
namespace {

__global__ void __launch_bounds__(256) fill_kernel(double* __restrict__ out, int64_t n, double v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = v;
}

// the word layout of the plan (plan.cpp): word(col, p) = columns[(p/64) n_columns 64 + col 64 + p%64]; the arithmetic is the
// stream kernels' (stream.cuh: eval, param_terms), one sample per thread
__global__ void __launch_bounds__(256) sample_logw_kernel(const ModelDev* __restrict__ Mp, const uint32_t* __restrict__ index, double* __restrict__ out) {
  const ModelDev& M = Mp[0];
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= M.n_padded) return;
  const uint32_t c = index[p];
  if (c == SAMPLE_INDEX_PAD) return;  // lane padding
  const uint64_t* q = M.columns + (size_t)(p >> 6) * (size_t)M.n_columns * 64 + (size_t)(p & 63);
  double x = __longlong_as_double((long long)q[(size_t)M.col_static * 64]);
  for (int d = 0; d < M.n_dims; ++d) {
    const unsigned long long word = q[(size_t)d * 64];
    const int J = (int)((unsigned)word & 63u);
    const double w = __longlong_as_double((long long)word);  // the word IS w (J rides in its 6 low mantissa bits)
    const double* a = M.tables + (size_t)(M.dims[d].row_off + J) * 4;
    double v = fma(fma(a[3], w, a[2]), w * w, fma(a[1], w, a[0]));
    if ((M.liny_mask >> d) & 1) v = v > 1e-300 ? log(v) : -INFINITY;  // spline density: log of the cubic
    x += v;
  }
  x = param_terms_x<false>(x, 0, M.n_kops, M.kops, M.kc, q, nullptr, 0);
  double K = M.Ksum[0];  // the constant finish_segment adds: scalar normalisers minus the grid normalisers
  for (int g = 0; g < M.n_groups; ++g) K -= M.logZ[g];
  out[c] = x + K;
}

__device__ __forceinline__ void tile_range(const DrawScratch& D, int t, int& s, int64_t& b, int64_t& e) {
  s = D.tile_seg[t];
  b = D.seg_off[s] + (int64_t)(t - D.tile_off[s]) * DRAW_TILE;
  e = b + DRAW_TILE < D.seg_off[s + 1] ? b + DRAW_TILE : D.seg_off[s + 1];
}

__global__ void __launch_bounds__(256) draw_tile_max_kernel(const DrawScratch D) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= D.n_tiles) return;
  int s;
  int64_t b, e;
  tile_range(D, t, s, b, e);
  double mx = -INFINITY;
  for (int64_t i = b; i < e; ++i) mx = fmax(mx, D.logw[i]);
  D.tile_max[t] = mx;
}

__global__ void __launch_bounds__(256) draw_seg_max_kernel(const DrawScratch D) {
  const int s = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (s >= D.n_seg) return;  // (whole warps)
  double mx = -INFINITY;
  for (int t = D.tile_off[s] + lane; t < D.tile_off[s + 1]; t += 32) mx = fmax(mx, D.tile_max[t]);
  mx = wmax(mx);
  if (lane == 0) D.seg_max[s] = mx;
}

__global__ void __launch_bounds__(256) draw_tile_sum_kernel(const DrawScratch D) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= D.n_tiles) return;
  int s;
  int64_t b, e;
  tile_range(D, t, s, b, e);
  const double m = D.seg_max[s];
  double acc = 0.0;
  if (m > -INFINITY && m < INFINITY)
    for (int64_t i = b; i < e; ++i) acc += exp(D.logw[i] - m);
  D.tile_cum[t] = acc;  // the tile's own sum; draw_scan_kernel turns it into the inclusive prefix
}

__global__ void __launch_bounds__(256) draw_scan_kernel(const DrawScratch D) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= D.n_seg) return;
  double acc = 0.0;
  for (int t = D.tile_off[s]; t < D.tile_off[s + 1]; ++t) {
    acc += D.tile_cum[t];
    D.tile_cum[t] = acc;
  }
}

__global__ void __launch_bounds__(256) draw_kernel(const DrawScratch D, uint64_t seed, int E, int dpe, int dinj, int64_t* __restrict__ out) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_pe_draws = (int64_t)E * dpe;
  if (g >= n_pe_draws + dinj) return;
  const int s = g < n_pe_draws ? (int)(g / dpe) : E;
  const uint32_t k = (uint32_t)(g < n_pe_draws ? g - (int64_t)s * dpe : g - n_pe_draws);
  const int t0 = D.tile_off[s], t1 = D.tile_off[s + 1];
  const double m = D.seg_max[s];
  const double total = t1 > t0 ? D.tile_cum[t1 - 1] : 0.0;
  if (!(m > -INFINITY && m < INFINITY) || !(total > 0.0 && total < INFINITY)) {
    out[g] = -1;  // no weight in this segment
    return;
  }
  const U4 rn = philox4x32_10(U4{k, (uint32_t)s, 0u, 0u}, (uint32_t)seed, (uint32_t)(seed >> 32));
  double r = u01(rn.x, rn.y) * total;
  if (!(r < total)) r = nextafter(total, 0.0);  // u total rounded up to the total
  int lo = t0, hi = t1 - 1;  // first tile whose inclusive prefix exceeds r
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (D.tile_cum[mid] > r) hi = mid; else lo = mid + 1;
  }
  int s_;
  int64_t b, e;
  tile_range(D, lo, s_, b, e);
  double acc = lo > t0 ? D.tile_cum[lo - 1] : 0.0;
  int64_t pick = -1, last = -1;
  for (int64_t i = b; i < e; ++i) {
    const double w = exp(D.logw[i] - m);
    if (w > 0.0) {
      last = i;
      acc += w;
      if (acc > r) {
        pick = i;
        break;
      }
    }
  }
  // (the scan inside the tile re-adds what the tile sum added in another association: if rounding leaves r just above its
  // end, the tile's last sample with weight is the one whose interval holds r)
  if (pick < 0) pick = last;
  out[g] = pick - D.seg_off[s];
}

}  // namespace

void launch_sample_log_weights(const ModelDev* Md, int64_t n_padded, const uint32_t* index, double* out, int64_t n_cat, cudaStream_t st) {
  if (n_cat > 0) GWI_LAUNCH(fill_kernel, dim3((unsigned)((n_cat + 255) / 256)), dim3(256), 0, st)(out, n_cat, -INFINITY);  // samples the plan dropped
  if (n_padded > 0) GWI_LAUNCH(sample_logw_kernel, dim3((unsigned)((n_padded + 255) / 256)), dim3(256), 0, st)(Md, index, out);
}

void launch_draws(const DrawScratch& D, uint64_t seed, int E, int dpe, int dinj, int64_t* out, cudaStream_t st) {
  const unsigned tb = (unsigned)((D.n_tiles + 255) / 256);
  if (D.n_tiles > 0) {
    GWI_LAUNCH(draw_tile_max_kernel, dim3(tb), dim3(256), 0, st)(D);
    GWI_LAUNCH(draw_seg_max_kernel, dim3((unsigned)((D.n_seg + 7) / 8)), dim3(256), 0, st)(D);
    GWI_LAUNCH(draw_tile_sum_kernel, dim3(tb), dim3(256), 0, st)(D);
    GWI_LAUNCH(draw_scan_kernel, dim3((unsigned)((D.n_seg + 255) / 256)), dim3(256), 0, st)(D);
  }
  const int64_t n = (int64_t)E * dpe + dinj;
  if (n > 0) GWI_LAUNCH(draw_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st)(D, seed, E, dpe, dinj, out);
}

// tiles of the catalog-order segments (host, once per model): tile_off[s] = first tile of segment s, tile_seg[t] = segment
void draw_tiles(const std::vector<int64_t>& seg_off, std::vector<int32_t>& tile_off, std::vector<int32_t>& tile_seg) {
  const int n_seg = (int)seg_off.size() - 1;
  tile_off.assign(n_seg + 1, 0);
  tile_seg.clear();
  for (int s = 0; s < n_seg; ++s) {
    const int64_t nt = (seg_off[s + 1] - seg_off[s] + DRAW_TILE - 1) / DRAW_TILE;
    tile_off[s + 1] = tile_off[s] + (int32_t)nt;
    tile_seg.insert(tile_seg.end(), (size_t)nt, s);
  }
}

}  // namespace gwi
