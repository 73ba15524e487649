// Device-side plan builder (SURVEY.md section 8 row f3): what the reference does at model construction on the host
// -- masks + dense design matrices over every sample, gwinferno/models/bsplines/single.py:54-57, interpolation.py:128-149,
// dVc/dz per sample, cosmology.py:95-120 -- done by four kernels on the catalog's own GPU:
//   key     one thread per sample: validity (masks, cuts, finite features) + sort key {segment | piece indices}
//   sort    stable LSD radix sort of (key, sample index) pairs over the used key bits (cub::DeviceRadixSort)
//   bounds  segment boundaries in the sorted order + sampled piece-change rates per segment and dim (from the key bits)
//   fill    one thread per padded stream position: inverse of the lane-run layout -> sorted rank -> sample index ->
//           gather of the raw coordinates -> packed spline words, features, static log-weight, written block-interleaved
//           straight into the plan's device array; per-chunk statistics (max static weight, occupied pieces, feature ranges)
// The stages between them (deep-dim choice, slices, chunks, reduction tree: O(segments + chunks)) stay on the host and are
// the SAME code as the host builder's (plan.cpp: plan_classify / plan_geometry / plan_tree), so both builders produce the
// same plan; the per-sample arithmetic is shared too (plan_sample.h).  The catalog columns may already be device-resident
// (gwi_catalog_desc.columns_on_device): then nothing crosses PCIe but the few KB of chunk descriptors.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <numeric>
#include <thread>

#ifndef GWI_HOST_EMULATION
#include <cub/device/device_radix_sort.cuh>
#endif

#include "dev_structs.h"
#include "plan_sample.h"

namespace gwi {

namespace {

constexpr int PD_MAX_COLS = 16;   // catalog columns a model may use on this path
constexpr int PD_MAX_FEATS = 20;  // static / per-sample-operation features
constexpr int PD_MAX_CUTS = 24;

// everything the kernels need of the model, passed by value (< 4 KB of parameter space)
struct PdParams {
  const double* pe[PD_MAX_COLS];   // by COMPACT column index (position in PlanInputs::used_cols)
  const double* inj[PD_MAX_COLS];
  int used_cols[PD_MAX_COLS];      // identity: 0..n_used-1
  int n_used;
  int n_cuts;
  RangeCut cuts[PD_MAX_CUTS];
  SplineGeom geom[MAX_SPLINE_DIMS];
  int key_shift[MAX_SPLINE_DIMS];
  int NS;
  int n_static;
  Feat static_feats[PD_MAX_FEATS];
  Feat kop_feats[PD_MAX_FEATS];
  int n_kf;
  int n_kops;
  int lin_feat[MAX_KOPS];          // kop q is KOP_LIN: index of its feature among kop_feats, else -1
  CosmoView cv;                    // Dc table in device memory
  const int64_t* pe_offsets;       // device copy, n_events + 1
  int n_events;
  int key_bits, seg_bits;
  int64_t n_pe, n_all;             // combined sample index j: [0, n_pe) = PE samples, [n_pe, n_all) = injections
};

struct PdChunk {
  int64_t first;   // first padded stream position
  int64_t src0;    // position of the chunk's first sample in the globally sorted order
  int64_t n_c;     // valid samples
  int32_t steps;
  int32_t segment;
};

struct PdChunkStat {  // order-encoded doubles (see enc_double) so that integer atomics apply
  unsigned long long max_static;
  unsigned long long occ[MAX_SPLINE_DIMS];
  unsigned long long fmin[MAX_KOPS], fmax[MAX_KOPS];
};

// monotone map double -> uint64 (a < b  <=>  enc(a) < enc(b) for non-NaN values)
GWI_HD inline unsigned long long enc_double(double x) {
  unsigned long long b;
  memcpy(&b, &x, 8);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
GWI_HD inline double dec_double(unsigned long long e) {
  const unsigned long long b = (e >> 63) ? (e & 0x7fffffffffffffffull) : ~e;
  double x;
  memcpy(&x, &b, 8);
  return x;
}

__device__ inline const double* const* pd_cols(const PdParams& A, int64_t j, int64_t& jj) {
  const bool is_pe = j < A.n_pe;
  jj = is_pe ? j : j - A.n_pe;
  return is_pe ? A.pe : A.inj;
}

// ---- key: validity + {segment | piece indices} per sample ------------------------------------------------------------
__global__ void __launch_bounds__(256) pd_key_kernel(const __grid_constant__ PdParams A, uint64_t* __restrict__ keys, uint32_t* __restrict__ idx) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= A.n_all) return;
  int64_t jj;
  const double* const* cols = pd_cols(A, j, jj);
  uint64_t k = sample_key(cols, jj, A.used_cols, A.n_used, A.cuts, A.n_cuts, A.geom, A.key_shift, A.NS, A.static_feats, A.n_static, A.kop_feats, A.n_kf, A.cv);
  if (k != PLAN_KEY_INVALID) {
    uint64_t seg = 0;  // injections
    if (j < A.n_pe) {  // event e owns [off[e], off[e+1]): e = (first i with off[i] > j) - 1
      int lo = 0, hi = A.n_events + 1;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (A.pe_offsets[mid] > j) hi = mid; else lo = mid + 1;
      }
      seg = (uint64_t)lo;  // = e + 1
    }
    k |= seg << A.key_bits;
  }
  keys[j] = k;
  idx[j] = (uint32_t)j;
}

// ---- bounds: seg_begin[s] = first sorted position of segment s (s = 0..n_seg; dropped samples sort behind every segment) ----
__global__ void __launch_bounds__(256) pd_bounds_kernel(const uint64_t* __restrict__ keys, int64_t n_all, int key_bits, int seg_bits, int n_seg, int64_t* __restrict__ seg_begin) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n_all) return;
  const uint64_t seg_mask = (1ull << seg_bits) - 1;
  auto seg_of = [&](int64_t q) -> int64_t {
    if (q < 0) return -1;
    if (q >= n_all) return n_seg;
    const uint64_t s = (keys[q] >> key_bits) & seg_mask;
    return s >= (uint64_t)n_seg ? (int64_t)n_seg : (int64_t)s;
  };
  const int64_t here = seg_of(i), prev = seg_of(i - 1);
  for (int64_t s = prev + 1; s <= here; ++s) seg_begin[s] = i;
}

// ---- rates: how often does each dim's piece index change between consecutive sorted samples (sampled with the host
// builder's stride: pairs (i, i+1), i = 0, stride, 2 stride, ...)?  counts[s][d] ----------------------------------------
__global__ void __launch_bounds__(256) pd_rate_kernel(const uint64_t* __restrict__ keys, const int64_t* __restrict__ seg_begin, const __grid_constant__ PdParams A, unsigned* __restrict__ counts) {
  __shared__ unsigned sh[MAX_SPLINE_DIMS];
  if (threadIdx.x < MAX_SPLINE_DIMS) sh[threadIdx.x] = 0;
  __syncthreads();
  const int s = blockIdx.y;
  const int64_t b = seg_begin[s], n = seg_begin[s + 1] - b;
  const int64_t stride = n / 50000 > 1 ? n / 50000 : 1;
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * stride;
  if (i + 1 < n) {
    const uint64_t x = keys[b + i] ^ keys[b + i + 1];
    for (int d = 0; d < A.NS; ++d)
      if ((x >> A.key_shift[d]) & 63) atomicAdd(&sh[d], 1u);
  }
  __syncthreads();
  if (threadIdx.x < A.NS && sh[threadIdx.x]) atomicAdd(&counts[s * MAX_SPLINE_DIMS + threadIdx.x], sh[threadIdx.x]);
}

// ---- fill: one thread per padded stream position -----------------------------------------------------------------------
// stream layout (plan.cpp): blocks of 64 consecutive padded samples, word(col, p) = [p/64][col][p%64]; inside a chunk the
// sub-chunk of main warp w is [first + w steps 32, ...), lane l owns the sorted run [l steps, (l+1) steps) of that
// sub-chunk, and step k of lane l sits at (k/UNROLL)(32 UNROLL) + l UNROLL + k%UNROLL
__global__ void __launch_bounds__(256) pd_fill_kernel(const __grid_constant__ PdParams A, const PdChunk* __restrict__ chunks, int n_chunks, const uint32_t* __restrict__ idx, int64_t n_padded,
                                                      int n_columns, uint64_t* __restrict__ columns, PdChunkStat* __restrict__ stats, uint32_t* __restrict__ sample_index) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_padded) return;  // n_padded is a multiple of 64: whole warps leave
  int lo = 0, hi = n_chunks - 1;
  while (lo < hi) {  // last chunk with first <= p
    const int mid = (lo + hi + 1) >> 1;
    if (chunks[mid].first <= p) lo = mid; else hi = mid - 1;
  }
  const PdChunk C = chunks[lo];
  const int64_t q = p - C.first;
  const int64_t per_warp = (int64_t)C.steps * LANES;
  const int64_t w = q / per_warp, q2 = q - w * per_warp;
  const int64_t blk = q2 / (LANES * UNROLL);
  const int r2 = (int)(q2 - blk * (LANES * UNROLL));
  const int lane = r2 / UNROLL, kk = r2 % UNROLL;
  const int64_t run = w * LANES + lane;
  const int64_t r = run * C.steps + blk * UNROLL + kk;
  const bool valid = r < C.n_c;
  // lane padding: a copy of the chunk's last valid sample (every term evaluates to finite values and no piece index
  // changes) with static log-weight -inf => weight 0
  const int64_t j = (int64_t)idx[C.src0 + (valid ? r : C.n_c - 1)];
  if (sample_index) sample_index[p] = valid ? (uint32_t)j : SAMPLE_INDEX_PAD;  // j: the catalog position (PE samples, then injections)
  int64_t jj;
  const double* const* cols = pd_cols(A, j, jj);
  const size_t base = ((size_t)(p >> 6) * (size_t)n_columns) * 64 + (size_t)(p & 63);
  unsigned long long occ[MAX_SPLINE_DIMS];
  for (int d = 0; d < A.NS; ++d) {
    int J = 0;
    double u = 0.0;
    spline_locate(A.geom[d], cols[A.geom[d].col][jj], J, u);
    columns[base + (size_t)d * 64] = pack_word(J, u);
    occ[d] = valid ? 1ull << J : 0ull;
  }
  for (int f = 0; f < A.n_kf; ++f) {
    const double v = eval_feat(A.kop_feats[f], cols, jj, A.cv);
    uint64_t b;
    memcpy(&b, &v, 8);
    columns[base + (size_t)(A.NS + f) * 64] = b;
  }
  double sw = 0.0;
  for (int i = 0; i < A.n_static; ++i) sw += eval_feat(A.static_feats[i], cols, jj, A.cv);
  const double NEG_INF = -plan_inf();
  if (!valid) sw = NEG_INF;
  {
    uint64_t b;
    memcpy(&b, &sw, 8);
    columns[base + (size_t)(A.NS + A.n_kf) * 64] = b;
  }
  // per-chunk statistics: the 32 positions of a warp belong to one chunk (chunk boundaries are multiples of 64)
  PdChunkStat* S = stats + lo;
  const unsigned lane_id = threadIdx.x & 31u;
  unsigned long long m = enc_double(sw);  // -inf for the padding lanes
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
    m = t > m ? t : m;
  }
  if (lane_id == 0 && m > S->max_static) atomicMax(&S->max_static, m);
  for (int d = 0; d < A.NS; ++d) {
    unsigned long long v = occ[d];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v |= __shfl_xor_sync(0xffffffffu, v, o);
    if (lane_id == 0 && (v & ~S->occ[d])) atomicOr(&S->occ[d], v);
  }
  for (int qk = 0; qk < A.n_kops; ++qk) {
    const int f = A.lin_feat[qk];
    if (f < 0) continue;  // (uniform across the warp)
    const double v = eval_feat(A.kop_feats[f], cols, jj, A.cv);
    unsigned long long mn = valid ? enc_double(v) : ~0ull, mx = valid ? enc_double(v) : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long a = __shfl_xor_sync(0xffffffffu, mn, o), b = __shfl_xor_sync(0xffffffffu, mx, o);
      mn = a < mn ? a : mn;
      mx = b > mx ? b : mx;
    }
    if (lane_id == 0) {
      if (mn < S->fmin[qk]) atomicMin(&S->fmin[qk], mn);
      if (mx > S->fmax[qk]) atomicMax(&S->fmax[qk], mx);
    }
  }
}

struct DevBuf {  // frees what the build allocated unless released
  std::vector<void*> ptrs;
  ~DevBuf() {
    for (void* p : ptrs)
      if (p) cudaFree(p);
  }
  template <class T>
  bool alloc(T** out, size_t count) {
    void* p = nullptr;
    if (cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) {
      cudaGetLastError();
      *out = nullptr;
      return false;
    }
    ptrs.push_back(p);
    *out = (T*)p;
    return true;
  }
  void release(void* p) {
    for (auto& q : ptrs)
      if (q == p) q = nullptr;
  }
  void free_now(void* p) {
    for (auto& q : ptrs)
      if (q == p && p) {
        cudaFree(p);
        q = nullptr;
      }
  }
};

// Host columns -> device through pinned staging buffers filled by worker threads (a pageable cudaMemcpy stages through ONE
// driver thread: ~6 GB/s; several memcpy threads + asynchronous copies run at the PCIe rate)
bool upload_columns(const std::vector<std::pair<const double*, double*>>& jobs_src_dst, const std::vector<int64_t>& counts, int device) {
  constexpr size_t STAGE = (size_t)32 << 20;  // bytes per staging buffer
  struct Piece {
    const char* src;
    char* dst;
    size_t bytes;
  };
  std::vector<Piece> pieces;
  for (size_t i = 0; i < jobs_src_dst.size(); ++i) {
    const char* s = (const char*)jobs_src_dst[i].first;
    char* d = (char*)jobs_src_dst[i].second;
    size_t left = (size_t)counts[i] * 8;
    while (left > 0) {
      const size_t n = std::min(left, STAGE);
      pieces.push_back(Piece{s, d, n});
      s += n;
      d += n;
      left -= n;
    }
  }
  if (pieces.empty()) return true;
  size_t total = 0;
  for (auto& p : pieces) total += p.bytes;
  if (total < ((size_t)64 << 20)) {  // small catalogs: not worth the pinned allocations
    for (auto& p : pieces)
      if (cudaMemcpy(p.dst, p.src, p.bytes, cudaMemcpyHostToDevice) != cudaSuccess) return false;
    return true;
  }
  const int T = (int)std::min<size_t>(8, std::max(1u, std::thread::hardware_concurrency()));
  std::atomic<size_t> next{0};
  std::atomic<bool> ok{true};
  auto work = [&]() {
    void* stage[2] = {nullptr, nullptr};
    cudaStream_t st = nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    if (cudaSetDevice(device) != cudaSuccess ||  // (the current device is per thread)
        cudaMallocHost(&stage[0], STAGE) != cudaSuccess || cudaMallocHost(&stage[1], STAGE) != cudaSuccess || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming) != cudaSuccess) {
      ok = false;
    } else {
      int b = 0;
      bool used[2] = {false, false};
      for (;;) {
        const size_t i = next.fetch_add(1);
        if (i >= pieces.size() || !ok) break;
        if (used[b]) cudaEventSynchronize(ev[b]);  // the copy that last read this buffer has finished
        std::memcpy(stage[b], pieces[i].src, pieces[i].bytes);
        if (cudaMemcpyAsync(pieces[i].dst, stage[b], pieces[i].bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) ok = false;
        cudaEventRecord(ev[b], st);
        used[b] = true;
        b ^= 1;
      }
      if (cudaStreamSynchronize(st) != cudaSuccess) ok = false;
    }
    for (int k = 0; k < 2; ++k) {
      if (stage[k]) cudaFreeHost(stage[k]);
      if (ev[k]) cudaEventDestroy(ev[k]);
    }
    if (st) cudaStreamDestroy(st);
  };
  std::vector<std::thread> th;
  for (int t = 0; t < T; ++t) th.emplace_back(work);
  for (auto& t : th) t.join();
  return ok;
}

double seconds_since(std::chrono::steady_clock::time_point& t0) {
  const auto now = std::chrono::steady_clock::now();
  const double s = std::chrono::duration<double>(now - t0).count();
  t0 = now;
  return s;
}

}  // namespace

// Returns GWI_OK, an error, or PLAN_DEVICE_FALLBACK (the model does not fit this path's fixed-size tables: the caller uses the
// host builder if the catalog is on the host).  On success *d_columns_out is the plan's device array (cudaMalloc'd; the
// caller owns it) and plan.columns stays empty.  stats_seconds[4] = raw-column upload, keys + sort + bounds, host geometry, fill.
int build_plan_device(const CatalogView& cat, const gwi_model_desc& desc, int sm_count, Plan& plan, uint64_t** d_columns_out, uint32_t** d_index_out,
                      double* stats_seconds) {
  *d_columns_out = nullptr;
  *d_index_out = nullptr;
  const bool timing = std::getenv("GWI_PLAN_TIMING") != nullptr;
  auto t0 = std::chrono::steady_clock::now();
  double secs[4] = {0, 0, 0, 0};
  PlanInputs in;
  int rc = plan_classify(cat.n_columns, desc, plan, in);
  if (rc != GWI_OK) return rc;
  rc = plan_begin_segments(cat, plan);
  if (rc != GWI_OK) return rc;
  const int NS = (int)plan.dims.size();
  const int E = cat.n_events, n_seg = E + 1;
  const int64_t n_pe = plan.n_samples_pe, n_inj = plan.n_samples_inj, n_all = n_pe + n_inj;
  int seg_bits = 1;
  while (((1ull << seg_bits) - 1) < (uint64_t)n_seg) ++seg_bits;  // the all-ones segment field is reserved for dropped samples
  if ((int)in.used_cols.size() > PD_MAX_COLS || (int)in.static_feats.size() > PD_MAX_FEATS || (int)in.kop_feats.size() > PD_MAX_FEATS ||
      (int)in.cuts.size() > PD_MAX_CUTS || in.key_bits + seg_bits > 64)
    return PLAN_DEVICE_FALLBACK;

  DevBuf buf;
#define PD_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      set_error(std::string("device plan build: " #expr " failed: ") + cudaGetErrorString(e_));    \
      return e_ == cudaErrorMemoryAllocation ? GWI_ERR_ALLOC : GWI_ERR_CUDA;                       \
    }                                                                                              \
  } while (0)
#define PD_ALLOC(ptr, count)                                                                        \
  do {                                                                                             \
    if (!buf.alloc(&(ptr), (size_t)(count))) {                                                     \
      set_error("device plan build: out of device memory");                                        \
      return GWI_ERR_ALLOC;                                                                        \
    }                                                                                              \
  } while (0)

  // ---- model tables -----------------------------------------------------------------------------------------------
  PdParams A{};
  std::vector<int> compact(cat.n_columns, -1);
  A.n_used = (int)in.used_cols.size();
  for (int i = 0; i < A.n_used; ++i) {
    compact[in.used_cols[i]] = i;
    A.used_cols[i] = i;
  }
  auto cc = [&](int c) { return c >= 0 ? compact[c] : c; };
  A.n_cuts = (int)in.cuts.size();
  for (int i = 0; i < A.n_cuts; ++i) {
    A.cuts[i] = in.cuts[i];
    A.cuts[i].col[0] = cc(in.cuts[i].col[0]);
    A.cuts[i].col[1] = cc(in.cuts[i].col[1]);
  }
  A.NS = NS;
  for (int d = 0; d < NS; ++d) {
    A.geom[d] = in.geom[d];
    A.geom[d].col = cc(in.geom[d].col);
    A.key_shift[d] = in.key_shift[d];
    if (in.geom[d].n_pieces > 0) {  // explicit knot vector: the piece tables go to device memory
      const int np = in.geom[d].n_pieces;
      double* dp;
      PD_ALLOC(dp, 3 * (size_t)np);
      PD_CUDA(cudaMemcpy(dp, in.geom[d].piece_lo, sizeof(double) * np, cudaMemcpyHostToDevice));
      PD_CUDA(cudaMemcpy(dp + np, in.geom[d].piece_origin, sizeof(double) * np, cudaMemcpyHostToDevice));
      PD_CUDA(cudaMemcpy(dp + 2 * np, in.geom[d].piece_inv_h, sizeof(double) * np, cudaMemcpyHostToDevice));
      A.geom[d].piece_lo = dp;
      A.geom[d].piece_origin = dp + np;
      A.geom[d].piece_inv_h = dp + 2 * np;
    }
  }
  auto copy_feats = [&](const std::vector<Feat>& src, Feat* dst) {
    for (size_t i = 0; i < src.size(); ++i) {
      dst[i] = src[i];
      dst[i].col[0] = cc(src[i].col[0]);
      dst[i].col[1] = cc(src[i].col[1]);
    }
  };
  A.n_static = (int)in.static_feats.size();
  copy_feats(in.static_feats, A.static_feats);
  A.n_kf = (int)in.kop_feats.size();
  copy_feats(in.kop_feats, A.kop_feats);
  A.n_kops = (int)plan.kops.size();
  for (int q = 0; q < A.n_kops; ++q) A.lin_feat[q] = plan.kops[q].kind == KOP_LIN ? plan.kops[q].col[0] - NS : -1;
  A.n_events = E;
  A.key_bits = in.key_bits;
  A.seg_bits = seg_bits;
  A.n_pe = n_pe;
  A.n_all = n_all;
  {
    const CosmoView hv = cosmo_view_host();
    double* d_dc;
    PD_ALLOC(d_dc, hv.n);
    PD_CUDA(cudaMemcpy(d_dc, hv.Dc, sizeof(double) * hv.n, cudaMemcpyHostToDevice));
    A.cv = CosmoView{d_dc, hv.n, hv.c_over_Ho};
    int64_t* d_off;
    PD_ALLOC(d_off, E + 1);
    PD_CUDA(cudaMemcpy(d_off, cat.pe_offsets.data(), sizeof(int64_t) * (E + 1), cudaMemcpyHostToDevice));
    A.pe_offsets = d_off;
  }
  // ---- raw columns on the device ------------------------------------------------------------------------------------
  std::vector<double*> raw_owned;
  if (cat.on_device) {
    for (int i = 0; i < A.n_used; ++i) {
      A.pe[i] = cat.pe_columns[in.used_cols[i]];
      A.inj[i] = cat.inj_columns[in.used_cols[i]];
    }
  } else {
    std::vector<std::pair<const double*, double*>> jobs;
    std::vector<int64_t> counts;
    for (int i = 0; i < A.n_used; ++i) {
      double* d;
      PD_ALLOC(d, n_all);
      raw_owned.push_back(d);
      A.pe[i] = d;
      A.inj[i] = d + n_pe;
      if (n_pe > 0) {
        jobs.push_back({cat.pe_columns[in.used_cols[i]], d});
        counts.push_back(n_pe);
      }
      if (n_inj > 0) {
        jobs.push_back({cat.inj_columns[in.used_cols[i]], d + n_pe});
        counts.push_back(n_inj);
      }
    }
    if (!upload_columns(jobs, counts, cat.device)) {
      set_error(std::string("device plan build: upload of the catalog columns failed: ") + cudaGetErrorString(cudaGetLastError()));
      return GWI_ERR_CUDA;
    }
  }
  secs[0] = seconds_since(t0);

  // ---- keys, sort, segment bounds, rates ----------------------------------------------------------------------------
  uint64_t *d_keys = nullptr, *d_keys2 = nullptr;
  uint32_t *d_idx = nullptr, *d_idx2 = nullptr;
  int64_t* d_seg_begin = nullptr;
  unsigned* d_counts = nullptr;
  PD_ALLOC(d_keys, n_all);
  PD_ALLOC(d_idx, n_all);
  PD_ALLOC(d_seg_begin, n_seg + 1);
  PD_ALLOC(d_counts, (size_t)n_seg * MAX_SPLINE_DIMS);
  PD_CUDA(cudaMemset(d_counts, 0, sizeof(unsigned) * (size_t)n_seg * MAX_SPLINE_DIMS));
  const int TB = 256;
  if (n_all > 0) GWI_LAUNCH(pd_key_kernel, dim3((unsigned)((n_all + TB - 1) / TB)), dim3(TB), 0, 0)(A, d_keys, d_idx);
  PD_CUDA(cudaGetLastError());
  const int end_bit = in.key_bits + seg_bits;
  const uint64_t* keys_sorted = d_keys;
  const uint32_t* idx_sorted = d_idx;
  if (n_all > 1) {
#ifdef GWI_HOST_EMULATION
    // (test infrastructure: the emulator's device memory is host memory) the same stable sort on the low end_bit bits
    const uint64_t mask = end_bit >= 64 ? ~0ull : ((1ull << end_bit) - 1);
    std::vector<uint32_t> perm((size_t)n_all);
    std::iota(perm.begin(), perm.end(), 0u);
    std::stable_sort(perm.begin(), perm.end(), [&](uint32_t a, uint32_t b) { return (d_keys[a] & mask) < (d_keys[b] & mask); });
    PD_ALLOC(d_keys2, n_all);
    PD_ALLOC(d_idx2, n_all);
    for (int64_t i = 0; i < n_all; ++i) {
      d_keys2[i] = d_keys[perm[i]];
      d_idx2[i] = d_idx[perm[i]];
    }
    keys_sorted = d_keys2;
    idx_sorted = d_idx2;
#else
    PD_ALLOC(d_keys2, n_all);
    PD_ALLOC(d_idx2, n_all);
    cub::DoubleBuffer<uint64_t> kb(d_keys, d_keys2);
    cub::DoubleBuffer<uint32_t> ib(d_idx, d_idx2);
    size_t temp_bytes = 0;
    PD_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, kb, ib, (long long)n_all, 0, end_bit, (cudaStream_t)0));
    char* d_temp;
    PD_ALLOC(d_temp, temp_bytes);
    PD_CUDA(cub::DeviceRadixSort::SortPairs(d_temp, temp_bytes, kb, ib, (long long)n_all, 0, end_bit, (cudaStream_t)0));
    keys_sorted = kb.Current();
    idx_sorted = ib.Current();
    PD_CUDA(cudaDeviceSynchronize());
    buf.free_now(d_temp);
    buf.free_now(kb.Alternate());
    buf.free_now(ib.Alternate());
#endif
  }
  GWI_LAUNCH(pd_bounds_kernel, dim3((unsigned)((n_all + 1 + TB - 1) / TB)), dim3(TB), 0, 0)(keys_sorted, n_all, in.key_bits, seg_bits, n_seg, d_seg_begin);
  PD_CUDA(cudaGetLastError());
  std::vector<int64_t> seg_begin(n_seg + 1);
  PD_CUDA(cudaMemcpy(seg_begin.data(), d_seg_begin, sizeof(int64_t) * (n_seg + 1), cudaMemcpyDeviceToHost));
  int64_t max_pairs = 0;
  for (int s = 0; s < n_seg; ++s) {
    const int64_t n = seg_begin[s + 1] - seg_begin[s];
    plan.segments[s].n_total = s == 0 ? n_inj : cat.pe_offsets[s] - cat.pe_offsets[s - 1];
    plan.segments[s].n_valid = n;
    const int64_t stride = std::max<int64_t>(1, n / 50000);
    if (n >= 2) max_pairs = std::max(max_pairs, (n - 1 + stride - 1) / stride);
  }
  for (int s = 1; s < n_seg; ++s) plan.n_valid_pe += plan.segments[s].n_valid;
  plan.n_valid_inj = plan.segments[0].n_valid;
  std::vector<std::vector<double>> rate(n_seg, std::vector<double>(NS, 0.0));
  if (max_pairs > 0) {
    for (int s0 = 0; s0 < n_seg; s0 += 32768) {  // (grid.y limit)
      const int ns = std::min(32768, n_seg - s0);
      GWI_LAUNCH(pd_rate_kernel, dim3((unsigned)((max_pairs + TB - 1) / TB), (unsigned)ns), dim3(TB), 0, 0)(keys_sorted, d_seg_begin + s0, A, d_counts + (size_t)s0 * MAX_SPLINE_DIMS);
    }
    PD_CUDA(cudaGetLastError());
    std::vector<unsigned> counts((size_t)n_seg * MAX_SPLINE_DIMS);
    PD_CUDA(cudaMemcpy(counts.data(), d_counts, sizeof(unsigned) * counts.size(), cudaMemcpyDeviceToHost));
    for (int s = 0; s < n_seg; ++s) {
      const int64_t n = plan.segments[s].n_valid;
      const int64_t stride = std::max<int64_t>(1, n / 50000);
      const double pairs = n >= 2 ? (double)((n - 1 + stride - 1) / stride) : 0.0;
      for (int d = 0; d < NS; ++d) rate[s][d] = pairs > 0 ? (double)counts[(size_t)s * MAX_SPLINE_DIMS + d] / pairs : 0.0;
    }
  }
  buf.free_now((void*)keys_sorted);
  secs[1] = seconds_since(t0);

  // ---- geometry (host; the same code as the host builder) ------------------------------------------------------------
  std::vector<int64_t> chunk_r0, chunk_nc;
  rc = plan_geometry(desc, sm_count, in, rate, plan, chunk_r0, chunk_nc);
  if (rc != GWI_OK) return rc;
  const int n_chunks = (int)plan.chunks.size();
  secs[2] = seconds_since(t0);

  // ---- fill ----------------------------------------------------------------------------------------------------------
  uint64_t* d_columns;
  {
    void* p = nullptr;
    const size_t words = (size_t)plan.n_columns * (size_t)std::max<int64_t>(1, plan.n_padded);
    if (cudaMalloc(&p, words * 8) != cudaSuccess) {
      cudaGetLastError();
      set_error("device plan build: out of device memory for the plan (" + std::to_string(words * 8) + " bytes)");
      return GWI_ERR_ALLOC;
    }
    d_columns = (uint64_t*)p;
    buf.ptrs.push_back(p);
  }
  uint32_t* d_index = nullptr;
  if (plan.keep_index) {
    if (!buf.alloc(&d_index, (size_t)std::max<int64_t>(1, plan.n_padded))) {
      set_error("device plan build: out of device memory for the sample index");
      return GWI_ERR_ALLOC;
    }
  }
  std::vector<PdChunkStat> cstat(n_chunks);
  if (n_chunks > 0) {
    std::vector<PdChunk> pc(n_chunks);
    for (int c = 0; c < n_chunks; ++c) {
      const Chunk& C = plan.chunks[c];
      pc[c] = PdChunk{C.first, seg_begin[C.segment] + chunk_r0[c], chunk_nc[c], C.steps, C.segment};
      PdChunkStat& st = cstat[c];
      st.max_static = enc_double(-std::numeric_limits<double>::infinity());
      for (int d = 0; d < MAX_SPLINE_DIMS; ++d) st.occ[d] = 0;
      for (int k = 0; k < MAX_KOPS; ++k) {
        st.fmin[k] = enc_double(std::numeric_limits<double>::infinity());
        st.fmax[k] = enc_double(-std::numeric_limits<double>::infinity());
      }
    }
    PdChunk* d_pc;
    PdChunkStat* d_stat;
    PD_ALLOC(d_pc, n_chunks);
    PD_ALLOC(d_stat, n_chunks);
    PD_CUDA(cudaMemcpy(d_pc, pc.data(), sizeof(PdChunk) * n_chunks, cudaMemcpyHostToDevice));
    PD_CUDA(cudaMemcpy(d_stat, cstat.data(), sizeof(PdChunkStat) * n_chunks, cudaMemcpyHostToDevice));
    GWI_LAUNCH(pd_fill_kernel, dim3((unsigned)((plan.n_padded + TB - 1) / TB)), dim3(TB), 0, 0)(A, d_pc, n_chunks, idx_sorted, plan.n_padded, plan.n_columns, d_columns, d_stat, d_index);
    PD_CUDA(cudaGetLastError());
    PD_CUDA(cudaMemcpy(cstat.data(), d_stat, sizeof(PdChunkStat) * n_chunks, cudaMemcpyDeviceToHost));
  }
  for (int c = 0; c < n_chunks; ++c) {
    Segment& S = plan.segments[plan.chunks[c].segment];
    S.max_static = std::max(S.max_static, dec_double(cstat[c].max_static));
    for (int d = 0; d < NS; ++d) S.occ[d] |= cstat[c].occ[d];
    for (size_t q = 0; q < plan.kops.size(); ++q) {
      S.fmin[q] = std::min(S.fmin[q], dec_double(cstat[c].fmin[q]));
      S.fmax[q] = std::max(S.fmax[q], dec_double(cstat[c].fmax[q]));
    }
  }
  PD_CUDA(cudaDeviceSynchronize());
  secs[3] = seconds_since(t0);
  plan_tree(plan);
  buf.release(d_columns);
  *d_columns_out = d_columns;
  if (d_index) {
    buf.release(d_index);
    *d_index_out = d_index;
  }
  if (stats_seconds)
    for (int i = 0; i < 4; ++i) stats_seconds[i] = secs[i];
  if (timing)
    std::fprintf(stderr, "[gwi plan] device build: columns %s %.3f s | keys + sort + bounds %.3f s | geometry (host) %.3f s | fill %.3f s\n",
                 cat.on_device ? "(device-resident)" : "upload", secs[0], secs[1], secs[2], secs[3]);
#undef PD_CUDA
#undef PD_ALLOC
  return GWI_OK;
}

}  // namespace gwi
