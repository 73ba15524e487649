// C-ABI entry points of libgwi.so (include/gwi.h): handle management, plan upload, and the
// per-evaluation launch sequence.  No CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <new>
#include <string>
#include <map>
#include <vector>

#include "dev_structs.h"
#include "plan_sample.h"
#include "smem_layout.h"

namespace gwi {

static thread_local std::string g_error;
void set_error(const std::string& msg) { g_error = msg; }

typedef void (*stream_fn)(const ModelDev*);
stream_fn pick_stream_kernel(int ns, int ndeep, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_cta_kernel(int ns, int ndeep, int nlin);  // CTA-cooperative kernel (stream_cta.cuh)
stream_fn pick_stream_cta_max_kernel();
void launch_prologue_tables(const ModelDev* Md, const double* lam, int n_groups, int n_seg, bool two_pass, int nc, cudaStream_t st, int use_learned_shift);
void launch_segmax_learn(const ModelDev* Md, int n_seg, int nc, cudaStream_t st);
void launch_prologue_groups(const ModelDev* Md, const double* lam, int n_groups, int max_grid, int nc, cudaStream_t aux);
void launch_reduce(const ModelDev* Md, int level, int n_tasks, int rec, int nc, cudaStream_t st);
void launch_segmax(const ModelDev* Md, int n_seg, int nc, cudaStream_t st);
void launch_finish(const ModelDev* Md, int n_seg, int rec_doubles, int nc, cudaStream_t st);
void launch_export(const ModelDev* Md, const gwi_outputs& out, cudaStream_t st);
void launch_partial(const ModelDev* Md, double* rec, int n_params, int nc, cudaStream_t st);
void launch_combine(const ModelDev* Md, const double* recs, int R, const gwi_like_opts& o, double* out, int nc, cudaStream_t st);
void launch_partial_tail(const ModelDev* Md, double* rec, int n_params, int tail, const gwi_like_opts& o, double* out, const CommDev& C, unsigned long long epoch, int nc,
                         cudaStream_t st);
void launch_exchange(const ModelDev* Md, const double* rec_local, const CommDev& C, unsigned long long epoch, int mode, const gwi_like_opts& o, double* out, cudaStream_t st);
void launch_sample_log_weights(const ModelDev* Md, int64_t n_padded, const uint32_t* index, double* out, int64_t n_cat, cudaStream_t st);
void launch_draws(const DrawScratch& D, uint64_t seed, int E, int dpe, int dinj, int64_t* out, cudaStream_t st);
void draw_tiles(const std::vector<int64_t>& seg_off, std::vector<int32_t>& tile_off, std::vector<int32_t>& tile_seg);

}  // namespace gwi

using namespace gwi;

// nothing may throw across the C boundary: the plan builder allocates several arrays of the
// catalog's size on the host
static int build_plan_noexcept(const CatalogView& cat, const gwi_model_desc& desc, int sm_count, int n_workers, Plan& plan) {
  try {
    return build_plan(cat, desc, sm_count, n_workers, plan);
  } catch (const std::bad_alloc&) {
    set_error("out of host memory building the plan");
    return GWI_ERR_ALLOC;
  } catch (const std::exception& e) {
    set_error(std::string("plan builder failed: ") + e.what());
    return GWI_ERR_INVALID;
  }
}

static int build_plan_device_noexcept(const CatalogView& cat, const gwi_model_desc& desc, int sm_count, Plan& plan, uint64_t** d_cols, uint32_t** d_index, double* secs) {
  try {
    return build_plan_device(cat, desc, sm_count, plan, d_cols, d_index, secs);
  } catch (const std::bad_alloc&) {
    set_error("out of host memory building the plan");
    return GWI_ERR_ALLOC;
  } catch (const std::exception& e) {
    set_error(std::string("device plan builder failed: ") + e.what());
    return GWI_ERR_INVALID;
  }
}

struct gwi_catalog {
  CatalogView view;
};

struct gwi_plan {
  Plan plan;
};

struct gwi_model {
  int device = 0;
  Plan plan;  // columns are released after the upload
  ModelDev host{};      // host copy of the device descriptor
  ModelDev* dev = nullptr;
  std::vector<void*> allocs;
  std::vector<std::pair<ReduceTask*, int>> level_tasks;  // device task arrays (static, shared by all chains)
  int n_chain_alloc = 1;                                  // descriptors / scratch sets allocated (chain batch)
  bool force_exact_shift = false;                         // gwi_model_set_exact_shift
  // gwi_loglike_host replays ONE (GWI_GRAPH=0 switches it off)
  // captured CUDA graph (H2D copy of Lambda, every kernel of the evaluation with its aux-stream fork /
  // join, D2H copy of the result) instead of issuing ~10 stream operations per call
  bool use_graph = false;
  cudaGraphExec_t graph_exec = nullptr;
  gwi_like_opts graph_opts{};
  double* partial_batch = nullptr;                        // [n_chain_alloc][PR_HEADER + 3P]
  int stream_grid_x = 1;
  bool cta = false;        // the CTA-cooperative stream kernel runs this model (plan.cta_mode)
  int stream_block = 0;    // threads per block of the full pass
  int max_grid_x = 1, max_block = 0;  // launch geometry of the max-only pass
  stream_fn k_full = nullptr, k_max = nullptr;
  size_t smem_full = 0, smem_max = 0;
  // speculative shift (GWI_SPECULATIVE_SHIFT=0 turns it off; host call only, one chain): models that need
  // the exact per-segment maximum take it from the previous evaluation's full pass instead of a max-only pass
  bool spec_shift = false;      // switch
  bool spec_learned = false;    // shift_next holds maxima of an earlier evaluation
  bool spec_allowed_now = false;  // set by gwi_loglike_host around its first attempt
  int max_grid = 0;
  int launches_per_eval = 0;
  // scratch for the host-buffer call and single-rank likelihood
  double* lam_dev = nullptr;
  double* out_dev = nullptr;
  double* partial_dev = nullptr;
  double* lam_pinned = nullptr;
  double* out_pinned = nullptr;
  // gwi_loglike_batch_host: staging for `batch_cap` chains and one captured graph per batch size in use
  int batch_cap = 0;
  double* lam_pinned_b = nullptr;
  double* out_pinned_b = nullptr;
  double* lam_dev_b = nullptr;
  double* out_dev_b = nullptr;
  std::map<int, cudaGraphExec_t> batch_graphs;
  gwi_like_opts batch_graph_opts{};
  cudaStream_t own_stream = nullptr;
  cudaStream_t aux_stream = nullptr;  // grid normalisers run here, concurrently with the stream kernel
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int64_t bytes_per_eval = 0;
  bool plan_on_device = false;  // built by plan_device.cu
  double plan_seconds[5] = {0, 0, 0, 0, 0};
  // GWI_PHASE_TIMING=1 (diagnostic): CUDA events between the kernels of every single-chain evaluation; the mean device
  // time of each phase is printed to stderr when the model is destroyed (this serialises consecutive evaluations)
  bool phase_timing = false;
  cudaEvent_t ph_ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  double ph_sum[5] = {0, 0, 0, 0, 0};
  int64_t ph_n = 0;
  bool ph_pending = false;
  // library-owned multi-GPU exchange (gwi_comm_*): this rank's buffer {flags [2][R] | slots [2][R][stride]},
  // the peers' buffers as opened here, and the number of sharded evaluations so far (the epoch)
  void* comm_base = nullptr;
  std::vector<void*> comm_opened;  // IPC mappings to close
  CommDev comm{};
  bool comm_connected = false;
  unsigned long long comm_epoch = 0, comm_pushed = 0;
  // optional timing of the stream kernel (ring of event pairs)
  bool timing = false;
  std::vector<cudaEvent_t> ev0, ev1;
  int64_t n_timed = 0;
  // gwi_model_desc.keep_sample_index: catalog position per padded stream position (device memory, in allocs)
  uint32_t* sample_index = nullptr;
  DrawScratch draw{};  // gwi_draw_samples: allocated on first use (in allocs)
};

static void phase_mark(gwi_model* m, int i, cudaStream_t st) {
  if (m->phase_timing) cudaEventRecord(m->ph_ev[i], st);
}
static void phase_collect(gwi_model* m) {
  if (!m->phase_timing || !m->ph_pending) return;
  cudaEventSynchronize(m->ph_ev[5]);
  for (int i = 0; i < 5; ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, m->ph_ev[i], m->ph_ev[i + 1]);
    m->ph_sum[i] += ms;
  }
  ++m->ph_n;
  m->ph_pending = false;
}

#define CUDA_TRY(expr)                                                                                 \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess) {                                                                           \
      set_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e));                            \
      return GWI_ERR_CUDA;                                                                             \
    }                                                                                                  \
  } while (0)

extern "C" {

const char* gwi_last_error(void) { return g_error.c_str(); }
int gwi_version(void) { return GWI_VERSION; }

int gwi_catalog_create(const gwi_catalog_desc* d, gwi_catalog** out) {
  if (!d || !out) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  if (d->n_columns <= 0 || d->n_events < 0 || d->n_inj < 0 || (d->n_events > 0 && (!d->pe_offsets || !d->pe_columns)) || (d->n_inj > 0 && !d->inj_columns)) {
    set_error("catalog description is incomplete");
    return GWI_ERR_INVALID;
  }
  if (!(d->total_inj > 0.0) || d->total_inj < (double)d->n_inj) {
    set_error("total_inj must be positive and at least the number of found injections");
    return GWI_ERR_INVALID;
  }
  // the plan builder indexes samples with 32 bits (a rank's shard; 180 GB of HBM hold ~2.5e9 samples)
  if (d->n_inj > (int64_t)UINT32_MAX || (d->n_events > 0 && d->pe_offsets && d->pe_offsets[d->n_events] > (int64_t)UINT32_MAX)) {
    set_error("more than 2^32 - 1 samples in one catalog shard: split it across ranks");
    return GWI_ERR_UNSUPPORTED;
  }
  gwi_catalog* c = new (std::nothrow) gwi_catalog();
  if (!c) return GWI_ERR_ALLOC;
  c->view.n_columns = d->n_columns;
  c->view.n_events = d->n_events;
  c->view.n_inj = d->n_inj;
  c->view.total_inj = d->total_inj;
  c->view.device = d->device;
  c->view.on_device = d->columns_on_device != 0;
  c->view.pe_offsets.assign(1, 0);
  if (d->n_events > 0) {
    c->view.pe_offsets.assign(d->pe_offsets, d->pe_offsets + d->n_events + 1);
    for (int e = 0; e < d->n_events; ++e)
      if (c->view.pe_offsets[e + 1] < c->view.pe_offsets[e] || c->view.pe_offsets[0] != 0) {
        delete c;
        set_error("pe_offsets must start at 0 and be non-decreasing");
        return GWI_ERR_INVALID;
      }
  }
  for (int k = 0; k < d->n_columns; ++k) {
    const double* p = d->n_events > 0 ? d->pe_columns[k] : nullptr;
    const double* q = d->n_inj > 0 ? d->inj_columns[k] : nullptr;
    if ((d->n_events > 0 && c->view.pe_offsets.back() > 0 && !p) || (d->n_inj > 0 && !q)) {
      delete c;
      set_error("null column pointer");
      return GWI_ERR_INVALID;
    }
    c->view.pe_columns.push_back(p);
    c->view.inj_columns.push_back(q);
  }
  *out = c;
  return GWI_OK;
}

void gwi_catalog_destroy(gwi_catalog* c) { delete c; }

int gwi_debug_plan_build(const gwi_catalog* cat, const gwi_model_desc* desc, int32_t n_workers, gwi_plan** out) {
  if (!cat || !desc || !out) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  gwi_plan* p = new (std::nothrow) gwi_plan();
  if (!p) return GWI_ERR_ALLOC;
  const int rc = build_plan_noexcept(cat->view, *desc, 148, n_workers, p->plan);
  if (rc != GWI_OK) {
    delete p;
    return rc;
  }
  *out = p;
  return GWI_OK;
}
void gwi_debug_plan_destroy(gwi_plan* p) { delete p; }

static int64_t plan_read(const Plan& p, int32_t what, void* dst, int64_t cap);
int64_t gwi_debug_plan_read(const gwi_plan* pp, int32_t what, void* dst, int64_t cap) {
  if (!pp) return GWI_ERR_INVALID;
  return plan_read(pp->plan, what, dst, cap);
}
int64_t gwi_debug_model_read(const gwi_model* m, int32_t what, void* dst, int64_t cap) {
  if (!m) return GWI_ERR_INVALID;
  if (what == 1) {
    const int64_t n = (int64_t)m->plan.n_columns * m->plan.n_padded;
    if (dst) {
      if (cap < n) return GWI_ERR_INVALID;
      if (n > 0 && cudaMemcpy(dst, m->host.columns, (size_t)n * 8, cudaMemcpyDeviceToHost) != cudaSuccess) {
        set_error("cudaMemcpy of the plan columns failed");
        return GWI_ERR_CUDA;
      }
    }
    return n;
  }
  if (what == 7) {
    const int64_t n = m->sample_index ? m->plan.n_padded : 0;
    if (dst && n > 0) {
      if (cap < n) return GWI_ERR_INVALID;
      std::vector<uint32_t> h((size_t)n);
      if (cudaMemcpy(h.data(), m->sample_index, (size_t)n * 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
        set_error("cudaMemcpy of the sample index failed");
        return GWI_ERR_CUDA;
      }
      int64_t* d = (int64_t*)dst;
      for (int64_t i = 0; i < n; ++i) d[i] = h[i] == SAMPLE_INDEX_PAD ? -1 : (int64_t)h[i];
    }
    return n;
  }
  return plan_read(m->plan, what, dst, cap);
}

static int64_t plan_read(const Plan& p, int32_t what, void* dst, int64_t cap) {
  std::vector<int64_t> v;
  const void* src = nullptr;
  int64_t n = 0;
  switch (what) {
    case 0:
      v = {p.n_columns, p.n_padded, (int64_t)p.chunks.size(), (int64_t)p.segments.size(), (int64_t)p.dims.size(), (int64_t)p.kops.size(),
           p.rows_total, p.n_deep, (int64_t)p.n_gslots, p.rec_doubles, p.cta_mode ? p.cta_main_warps : 1};
      break;
    case 1:
      src = p.columns.data();
      n = (int64_t)p.n_columns * p.n_padded;
      break;
    case 2:
      for (auto& c : p.chunks) {
        v.push_back(c.segment);
        v.push_back(c.first);
        v.push_back(c.steps);
        v.push_back(c.record_slot);
      }
      break;
    case 3:
      for (auto& s : p.segments) {
        v.push_back(s.n_total);
        v.push_back(s.n_valid);
        v.push_back(s.first_chunk);
        v.push_back(s.n_chunks);
      }
      break;
    case 4:
      for (auto& d : p.dims) {
        v.push_back(d.term);
        v.push_back(d.rows);
        v.push_back(d.row_off);
        v.push_back(d.deep);
      }
      break;
    case 5:
      for (auto& k : p.kops) {
        int64_t bits;
        std::memcpy(&bits, &k.cst[0], 8);
        v.push_back(k.kind);
        v.push_back(k.col[0]);
        v.push_back(k.col[1]);
        v.push_back(k.slot[0]);
        v.push_back(k.slot[1]);
        v.push_back(k.slot[2]);
        v.push_back(k.slot[3]);
        v.push_back(bits);
      }
      break;
    case 6:  // per-segment statistics behind the a-priori shift: max static weight, occupied pieces, LIN feature ranges (bit patterns)
      for (auto& sg : p.segments) {
        int64_t bits;
        std::memcpy(&bits, &sg.max_static, 8);
        v.push_back(bits);
        for (int d = 0; d < MAX_SPLINE_DIMS; ++d) v.push_back((int64_t)sg.occ[d]);
        for (int q = 0; q < MAX_KOPS; ++q) {
          std::memcpy(&bits, &sg.fmin[q], 8);
          v.push_back(bits);
        }
        for (int q = 0; q < MAX_KOPS; ++q) {
          std::memcpy(&bits, &sg.fmax[q], 8);
          v.push_back(bits);
        }
      }
      break;
    case 7:  // catalog position per padded stream position, -1 = lane padding
      if (p.keep_index)
        for (uint32_t c : p.sample_index) v.push_back(c == SAMPLE_INDEX_PAD ? -1 : (int64_t)c);
      if (p.n_padded == 0) v.clear();  // (the builder keeps one element for an empty plan)
      break;
    default:
      return GWI_ERR_INVALID;
  }
  if (!src) {
    src = v.data();
    n = (int64_t)v.size();
  }
  if (dst) {
    if (cap < n) return GWI_ERR_INVALID;
    std::memcpy(dst, src, (size_t)n * 8);
  }
  return n;
}

}  // extern "C"

// -------------------------------------------------------------------------------------------------
template <class T>
static int upload(gwi_model* m, const T* src, size_t count, T** dst) {
  *dst = nullptr;
  const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    set_error(std::string("cudaMalloc of ") + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e));
    return GWI_ERR_ALLOC;
  }
  m->allocs.push_back(p);
  if (src && count) {
    e = cudaMemcpy(p, src, count * sizeof(T), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      set_error(std::string("cudaMemcpy H2D failed: ") + cudaGetErrorString(e));
      return GWI_ERR_CUDA;
    }
  } else {
    cudaMemset(p, 0, bytes);
  }
  *dst = (T*)p;
  return GWI_OK;
}

// per-evaluation scratch of ONE chain (tables, normalisers, records, per-segment results)
static int alloc_chain_scratch(gwi_model* m, ModelDev& H) {
  const Plan& p = m->plan;
  const int P = p.n_params, nseg = (int)p.segments.size();
  int rc;
#define UPS(expr)                \
  do {                           \
    rc = (expr);                 \
    if (rc != GWI_OK) return rc; \
  } while (0)
  UPS(upload<double>(m, nullptr, (size_t)p.rows_total * 4, &H.tables));
  UPS(upload<double>(m, nullptr, (size_t)p.rows_total, &H.piece_ub));
  UPS(upload<double>(m, nullptr, (size_t)std::max(1, H.n_kops) * KC_STRIDE, &H.kc));
  UPS(upload<double>(m, nullptr, (size_t)nseg, &H.shift));
  UPS(upload<double>(m, nullptr, (size_t)std::max(1, H.n_groups), &H.logZ));
  UPS(upload<double>(m, nullptr, (size_t)std::max(1, H.n_groups) * P, &H.dlogZ));
  UPS(upload<double>(m, nullptr, (size_t)P + 1, &H.Ksum));
  UPS(upload<double>(m, nullptr, (size_t)std::max(1, H.n_chunks), &H.chunk_max));
  UPS(upload<int32_t>(m, nullptr, (size_t)2, &H.slice_counter));
  UPS(upload<double>(m, nullptr, (size_t)std::max(1, p.n_records0) * p.rec_doubles, &H.records0));
  UPS(upload<double>(m, nullptr, (size_t)nseg * 4, &H.seg_out));
  UPS(upload<double>(m, nullptr, (size_t)nseg * P, &H.seg_J1));
  UPS(upload<double>(m, nullptr, (size_t)nseg * P, &H.seg_Jn));
  UPS(upload<double>(m, nullptr, (size_t)3 + 2 * P, &H.inj_raw));
  UPS(upload<double>(m, nullptr, (size_t)nseg, &H.shift_next));
  UPS(upload<double>(m, nullptr, (size_t)nseg, &H.spec_bad));
  UPS(upload<int32_t>(m, nullptr, (size_t)1, &H.tail_counter));
  H.n_levels = (int)p.levels.size();
  for (int l = 0; l < 6; ++l) {
    H.level_buf[l] = nullptr;
    H.level_tasks[l] = nullptr;
    H.level_ntasks[l] = 0;
  }
  for (int l = 0; l < H.n_levels; ++l) {
    H.level_tasks[l] = m->level_tasks[l].first;
    H.level_ntasks[l] = m->level_tasks[l].second;
    if (l + 1 < H.n_levels) UPS(upload<double>(m, nullptr, p.levels[l].size() * (size_t)p.rec_doubles, &H.level_buf[l]));
  }
#undef UPS
  return GWI_OK;
}

// make sure descriptors + scratch exist for `n` chains (chain 0 always exists)
static int ensure_chains(gwi_model* m, int n) {
  if (n <= m->n_chain_alloc) return GWI_OK;
  std::vector<ModelDev> all(n);
  // existing descriptors are re-read from the device (they hold the scratch pointers)
  if (cudaMemcpy(all.data(), m->dev, sizeof(ModelDev) * m->n_chain_alloc, cudaMemcpyDeviceToHost) != cudaSuccess) {
    set_error("cudaMemcpy of the chain descriptors failed");
    return GWI_ERR_CUDA;
  }
  for (int c = m->n_chain_alloc; c < n; ++c) {
    all[c] = m->host;
    const int rc = alloc_chain_scratch(m, all[c]);
    if (rc != GWI_OK) return rc;
  }
  ModelDev* d = nullptr;
  int rc = upload(m, all.data(), (size_t)n, &d);
  if (rc != GWI_OK) return rc;
  double* pb = nullptr;
  rc = upload<double>(m, nullptr, (size_t)n * (PR_HEADER + 3 * m->plan.n_params), &pb);
  if (rc != GWI_OK) return rc;
  m->dev = d;  // the old (smaller) descriptor array stays in m->allocs until destroy
  m->partial_batch = pb;
  m->n_chain_alloc = n;
  return GWI_OK;
}

extern "C" {

void gwi_model_destroy(gwi_model* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  if (m->phase_timing) {
    phase_collect(m);
    if (m->ph_n > 0)
      std::fprintf(stderr, "[gwi phases] %lld evaluations, mean device ms: prologue %.4f | stream %.4f | reduce %.4f | finish (+ join) %.4f | partial + combine %.4f\n",
                   (long long)m->ph_n, m->ph_sum[0] / m->ph_n, m->ph_sum[1] / m->ph_n, m->ph_sum[2] / m->ph_n, m->ph_sum[3] / m->ph_n, m->ph_sum[4] / m->ph_n);
    for (auto e : m->ph_ev)
      if (e) cudaEventDestroy(e);
  }
#ifndef GWI_HOST_EMULATION
  for (void* p : m->comm_opened) cudaIpcCloseMemHandle(p);
#endif
  for (void* p : m->allocs) cudaFree(p);
  if (m->lam_pinned) cudaFreeHost(m->lam_pinned);
  if (m->out_pinned) cudaFreeHost(m->out_pinned);
  if (m->lam_pinned_b) cudaFreeHost(m->lam_pinned_b);
  if (m->out_pinned_b) cudaFreeHost(m->out_pinned_b);
  for (auto& g : m->batch_graphs)
    if (g.second) cudaGraphExecDestroy(g.second);
  if (m->own_stream) cudaStreamDestroy(m->own_stream);
  if (m->aux_stream) cudaStreamDestroy(m->aux_stream);
  if (m->ev_fork) cudaEventDestroy(m->ev_fork);
  if (m->ev_join) cudaEventDestroy(m->ev_join);
  if (m->graph_exec) cudaGraphExecDestroy(m->graph_exec);
  for (auto e : m->ev0) cudaEventDestroy(e);
  for (auto e : m->ev1) cudaEventDestroy(e);
  delete m;
}

int gwi_model_create(gwi_catalog* cat, const gwi_model_desc* desc, gwi_model** out) {
  if (!cat || !desc || !out) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    set_error("no CUDA device available: libgwi has no CPU fallback");
    return GWI_ERR_CUDA;
  }
  if (cat->view.device < 0 || cat->view.device >= ndev) {
    set_error("bad device ordinal");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(cat->view.device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, cat->view.device));
  for (int g = 0; g < desc->n_groups; ++g)
    if (desc->groups[g].n_grid > 5000) {
      set_error("norm grids are limited to 5000 points");
      return GWI_ERR_UNSUPPORTED;
    }
  gwi_model* m = new (std::nothrow) gwi_model();
  if (!m) return GWI_ERR_ALLOC;
  m->device = cat->view.device;
  // the plan is built on the GPU (plan_device.cu) unless GWI_PLAN_DEVICE=0 asks for the host builder; the host warp
  // emulator of the CPU test suite defaults to the host builder (GWI_PLAN_DEVICE=1 runs the device builder's kernels there)
#ifdef GWI_HOST_EMULATION
  bool dev_build = false;
#else
  bool dev_build = true;
#endif
  if (const char* e = std::getenv("GWI_PLAN_DEVICE")) dev_build = e[0] != '0';
  if (cat->view.on_device) dev_build = true;
  const auto t_plan0 = std::chrono::steady_clock::now();
  uint64_t* d_cols_built = nullptr;
  uint32_t* d_index_built = nullptr;
  int rc = GWI_OK;
  if (dev_build) {
    rc = build_plan_device_noexcept(cat->view, *desc, prop.multiProcessorCount, m->plan, &d_cols_built, &d_index_built, m->plan_seconds + 1);
    if (rc == PLAN_DEVICE_FALLBACK) {
      if (cat->view.on_device) {
        set_error("model too large for the device plan builder's tables and the catalog columns are device-resident");
        rc = GWI_ERR_UNSUPPORTED;
      } else {
        dev_build = false;
      }
    } else if (rc == GWI_ERR_ALLOC && !cat->view.on_device) {
      // the device builder holds the raw columns, the sort buffers AND the plan at its peak (~2.2x the plan): a shard that
      // only just fits the GPU is built on the host instead (the plan alone is uploaded)
      cudaGetLastError();
      dev_build = false;
    }
  }
  if (!dev_build) rc = build_plan_noexcept(cat->view, *desc, prop.multiProcessorCount, 0, m->plan);
  if (rc != GWI_OK) {
    delete m;
    return rc;
  }
  m->plan_on_device = dev_build;
  if (d_cols_built) m->allocs.push_back(d_cols_built);
  if (d_index_built) m->allocs.push_back(d_index_built);
  m->sample_index = d_index_built;
  Plan& p = m->plan;
  ModelDev& H = m->host;
  const int P = p.n_params, NS = (int)p.dims.size(), nseg = (int)p.segments.size();
  H.n_params = P;
  H.n_dims = NS;
  H.n_deep = p.n_deep;
  H.n_kops = (int)p.kops.size();
  H.n_gslots = p.n_gslots;
  H.n_sops = (int)p.sops.size();
  H.n_groups = (int)p.groups.size();
  H.n_segments = nseg;
  H.rows_total = p.rows_total;
  H.rec_doubles = p.rec_doubles;
  H.n_columns = p.n_columns;
  H.col_static = p.col_static;
  H.g2 = p.g2 ? 1 : 0;
  H.n_chunks = (int)p.chunks.size();
  H.n_padded = p.n_padded;
  H.cta_main_warps = p.cta_mode ? p.cta_main_warps : 0;
  H.cta_lead_doubles = 0;
  H.total_inj = p.total_inj;
  H.two_pass = 0;
  H.liny_mask = 0;
  const int mom = p.g2 ? 2 : 1;
  int deep_rows = 0;
  for (int d = 0; d < NS; ++d) {
    const SplineDim& D = p.dims[d];
    const gwi_term& t = desc->terms[D.term];
    DimDev& X = H.dims[d];
    X.rows = D.rows;
    X.row_off = D.row_off;
    X.slot = D.slot;
    X.n_splines = D.n_splines;
    X.deep = D.deep;
    X.deep_off = D.deep ? deep_rows * 2 * mom : 0;  // first double2 accumulator (smem_layout.h): (row, moment set, pair)
    if (D.deep) deep_rows += D.rows;
    X.norm_group = D.norm_group;
    X.grid_off = D.grid_off;
    X.grid_aux = D.grid_aux;
    X.liny = D.liny;
    if (D.liny) {
      H.liny_mask |= 1 << d;
      H.two_pass = 1;  // no a-priori bound through the log of the spline: exact max first
    }
    X.basis_off = D.basis_off;
    X.first_off = D.first_off;
    X.floor_off = D.floor_off;
    X.pad_ = 0;
    X.xi_lo = t.xi_lo;
    X.inv_dxi = (double)(D.rows - 1) / (t.xi_hi - t.xi_lo);
  }
  H.deep_rows = deep_rows;
  if (p.cta_mode) {
    // what a main warp of the CTA-cooperative kernel writes of its record: {S1, S2}, the linear-term slots and the rows of
    // the leading dims (the dims are in sort-key order, the deep ones last)
    int lead_rows = 0;
    for (int d = 0; d < NS - p.n_deep; ++d) lead_rows += p.dims[d].rows;
    H.cta_lead_doubles = 2 + p.n_gslots + lead_rows * 4;
  }
  for (int q = 0; q < H.n_kops; ++q) {
    const Kop& K = p.kops[q];
    KopDev& X = H.kops[q];
    X.kind = K.kind;
    X.col0 = K.col[0];
    X.col1 = K.col[1];
    X.gslot = K.gslot;
    X.n_gslots = K.n_gslots;
    X.norm_group = K.norm_group;
    X.grid_off = K.grid_off;
    for (int i = 0; i < 6; ++i) X.slot[i] = K.slot[i];
    for (int i = 0; i < 4; ++i) X.cst[i] = K.cst[i];
    for (int i = 0; i < K.n_gslots; ++i) H.gslot_slot[K.gslot + i] = K.slot[i];
    if (K.kind != KOP_LIN) H.two_pass = 1;  // no a-priori bound for the non-linear terms: exact max first
  }
  // up to 2 linear terms are register-resident in the stream kernel; any other non-spline term
  // selects the generic-term variant, which then handles ALL non-spline terms
  const bool param = H.n_kops > std::min(p.n_lin, 2) || H.liny_mask != 0;
  H.n_lin_fast = param ? 0 : std::min(p.n_lin, 2);
  for (int q = 0; q < H.n_sops; ++q) {
    const Sop& S = p.sops[q];
    H.sops[q] = SopDev{S.kind, S.slot[0], S.slot[1], 0, S.cst[0], S.cst[1]};
    // A Beta term's two linear features, log x and log(s - x), peak at opposite ends of its support, so the sum of
    // their separate maxima overshoots the largest weight by up to ~(a + b - 2) log 2: ~690 at a = b = 500, where every
    // weight more than e^-16 below the largest one fell under the stream kernel's underflow cut.  Exact max first.
    if (S.kind == SOP_BETA_NORM) H.two_pass = 1;
  }
  m->max_grid = 1;
  std::vector<GroupDev> groups;
  for (auto& g : p.groups) {
    groups.push_back(GroupDev{g.n_grid, g.logw_off});
    m->max_grid = std::max(m->max_grid, g.n_grid);
  }
  std::vector<SegDev> segs(nseg);
  for (int s = 0; s < nseg; ++s) {
    const Segment& S = p.segments[s];
    SegDev& X = segs[s];
    X.n_total = (double)S.n_total;
    X.max_static = S.max_static;
    for (int d = 0; d < MAX_SPLINE_DIMS; ++d) X.occ[d] = S.occ[d];
    for (int q = 0; q < MAX_KOPS; ++q) {
      X.fmin[q] = S.fmin[q];
      X.fmax[q] = S.fmax[q];
    }
    X.first_chunk = S.first_chunk;
    X.n_chunks = S.n_chunks;
  }

#define UP(expr)            \
  do {                      \
    rc = (expr);            \
    if (rc != GWI_OK) {     \
      gwi_model_destroy(m); \
      return rc;            \
    }                       \
  } while (0)

  uint64_t* d_cols = d_cols_built;
  if (!d_cols) {
    UP(upload(m, p.columns.data(), p.columns.size(), &d_cols));
    std::vector<uint64_t>().swap(p.columns);  // host copy no longer needed
  }
  if (p.keep_index && !m->sample_index) {  // host builder
    UP(upload(m, p.sample_index.data(), p.sample_index.size(), &m->sample_index));
    std::vector<uint32_t>().swap(p.sample_index);
  }
  m->bytes_per_eval = (int64_t)p.n_columns * p.n_padded * 8;
  H.columns = d_cols;
  Chunk* d_chunks;
  UP(upload(m, p.chunks.data(), p.chunks.size(), &d_chunks));
  H.chunks = d_chunks;
  int32_t* d_slices;
  UP(upload(m, p.slice_begin.data(), p.slice_begin.size(), &d_slices));
  H.slice_begin = d_slices;
  H.n_slices = (int)p.slice_begin.size() - 1;
  SegDev* d_segs;
  UP(upload(m, segs.data(), segs.size(), &d_segs));
  H.segs = d_segs;
  GroupDev* d_groups;
  UP(upload(m, groups.data(), groups.size(), &d_groups));
  H.groups = d_groups;
  double* d_pool;
  UP(upload(m, p.grid_pool.data(), p.grid_pool.size(), &d_pool));
  H.grid_pool = d_pool;
  if (p.levels.size() > 6) {
    set_error("internal: reduction tree deeper than 6 levels");
    gwi_model_destroy(m);
    return GWI_ERR_UNSUPPORTED;
  }
  for (size_t l = 0; l < p.levels.size(); ++l) {
    ReduceTask* d_t;
    UP(upload(m, p.levels[l].data(), p.levels[l].size(), &d_t));
    m->level_tasks.push_back({d_t, (int)p.levels[l].size()});
  }
  UP(alloc_chain_scratch(m, H));
  UP(upload(m, &H, 1, &m->dev));
  UP(upload<double>(m, nullptr, (size_t)P, &m->lam_dev));
  UP(upload<double>(m, nullptr, (size_t)GWI_LIKE_HEADER + P, &m->out_dev));
  UP(upload<double>(m, nullptr, (size_t)PR_HEADER + 3 * P, &m->partial_dev));
#undef UP
  if (cudaMallocHost((void**)&m->lam_pinned, sizeof(double) * P) != cudaSuccess ||
      cudaMallocHost((void**)&m->out_pinned, sizeof(double) * (GWI_LIKE_HEADER + P)) != cudaSuccess ||
      cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&m->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    set_error("pinned host allocation / stream creation failed");
    gwi_model_destroy(m);
    return GWI_ERR_ALLOC;
  }

  // ---- kernels + shared memory ----
  m->cta = p.cta_mode;
  if (m->cta) {
    m->k_full = pick_stream_cta_kernel(NS, p.n_deep, H.n_lin_fast);
    m->k_max = pick_stream_cta_max_kernel();
  } else {
    m->k_full = pick_stream_kernel(NS, p.n_deep, H.n_lin_fast, p.g2, param, false);
    m->k_max = pick_stream_kernel(NS, p.n_deep, 0, p.g2, true, true);
  }
  if (!m->k_full || !m->k_max) {
    set_error("no stream kernel instantiated for this (spline dims, deep dims) combination");
    gwi_model_destroy(m);
    return GWI_ERR_UNSUPPORTED;
  }
  bool aligned = true;
  if (m->cta) {
    const CtaLayout L = cta_layout(p.cta_main_warps, p.n_columns, p.rows_total, deep_rows);
    aligned = L.aligned16();
    m->smem_full = L.total;
    m->smem_max = 0;
    m->stream_block = (p.cta_main_warps + p.n_deep) * 32;
    m->max_block = 256;
  } else {
    m->smem_full = one_role_smem_bytes(p.rows_total, deep_rows, mom, H.n_kops, p.n_gslots, p.warps_per_block);
    m->smem_max = m->smem_full;
    m->stream_block = p.warps_per_block * 32;
    m->max_block = p.warps_per_block * 32;
  }
  if (!aligned || m->smem_full > (size_t)prop.sharedMemPerBlockOptin) {
    set_error("internal: plan geometry does not fit the device's shared memory");
    gwi_model_destroy(m);
    return GWI_ERR_UNSUPPORTED;
  }
  if (cudaFuncSetAttribute((const void*)m->k_full, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m->smem_full) != cudaSuccess ||
      cudaFuncSetAttribute((const void*)m->k_max, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m->smem_max) != cudaSuccess) {
    set_error(std::string("cudaFuncSetAttribute(shared memory) failed: ") + cudaGetErrorString(cudaGetLastError()));
    gwi_model_destroy(m);
    return GWI_ERR_CUDA;
  }
  {
    if (const char* pt = std::getenv("GWI_PHASE_TIMING")) {
      m->phase_timing = pt[0] == '1';
      if (m->phase_timing)
        for (auto& e : m->ph_ev) cudaEventCreate(&e);
    }
    const char* g = std::getenv("GWI_GRAPH");
    m->use_graph = !(g && g[0] == '0') && !m->phase_timing;  // on by default (r02: +9 % e2e evals/s at config-2 size, bitwise-equal results)
    const char* sp = std::getenv("GWI_SPECULATIVE_SHIFT");
    m->spec_shift = H.two_pass && !(sp && sp[0] == '0');  // on by default (r02 call 37: cfg1 host call 308 -> 211 us, equal results)
    if (m->spec_shift) m->use_graph = false;  // the launch sequence differs from call to call
  }
  m->stream_grid_x = std::max(1, std::min(p.grid_blocks, ((int)p.slice_begin.size() - 1 + p.warps_per_block - 1) / p.warps_per_block));
  m->max_grid_x = m->stream_grid_x;
  if (m->cta) {
    m->stream_grid_x = std::max(1, std::min(p.grid_blocks, (int)p.slice_begin.size() - 1));
    m->max_grid_x = std::max(1, std::min(4 * p.grid_blocks, (int)p.chunks.size()));
  }
  m->launches_per_eval = 2 + (H.two_pass ? 2 : 0) + 1 + ((int)p.levels.size() - 1) + 1 + 1;
  CUDA_TRY(cudaDeviceSynchronize());
  m->plan_seconds[0] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_plan0).count();
  *out = m;
  return GWI_OK;
}

// launches prologue .. finish for `nc` chains on `st` (lam_dev: [nc][P])
static int run_eval(gwi_model* m, const double* lam_dev, int nc, cudaStream_t st, bool exact_shift = false) {
  const ModelDev& H = m->host;
  phase_collect(m);
  phase_mark(m, 0, st);
  // fork: the grid normalisers (needed only by finish_kernel) overlap with the stream kernel
  cudaEventRecord(m->ev_fork, st);
  cudaStreamWaitEvent(m->aux_stream, m->ev_fork, 0);
  launch_prologue_groups(m->dev, lam_dev, H.n_groups, m->max_grid, nc, m->aux_stream);
  cudaEventRecord(m->ev_join, m->aux_stream);
  const bool speculate = m->spec_shift && m->spec_allowed_now && m->spec_learned && nc == 1 && !exact_shift && !m->force_exact_shift;
  launch_prologue_tables(m->dev, lam_dev, H.n_groups, H.n_segments, H.two_pass != 0, nc, st, speculate ? 1 : 0);
  phase_mark(m, 1, st);
  const dim3 grid(m->stream_grid_x, nc), block(m->stream_block);
  if (H.n_chunks > 0) {
    if ((H.two_pass && !speculate) || exact_shift || m->force_exact_shift) {
      // exact per-segment maximum first (always for models with non-linear terms; as a fallback when
      // the a-priori bound was so loose that every weight of a segment underflowed)
      GWI_LAUNCH(m->k_max, dim3(m->max_grid_x, nc), dim3(m->max_block), m->smem_max, st)(m->dev);
      launch_segmax(m->dev, H.n_segments, nc, st);
    }
    if (m->timing) cudaEventRecord(m->ev0[m->n_timed % 64], st);
    GWI_LAUNCH_PDL(m->k_full, grid, block, m->smem_full, st)(m->dev);
    if (m->timing) cudaEventRecord(m->ev1[m->n_timed++ % 64], st);
    if (m->spec_shift && nc == 1) {
      launch_segmax_learn(m->dev, H.n_segments, nc, st);  // next evaluation's shift; flags this one if its shift was off
      m->spec_learned = true;
    }
  }
  phase_mark(m, 2, st);
  const int n_levels = (int)m->level_tasks.size();
  for (int l = 0; l + 1 < n_levels; ++l) launch_reduce(m->dev, l, m->level_tasks[l].second, H.rec_doubles, nc, st);
  phase_mark(m, 3, st);
  cudaStreamWaitEvent(st, m->ev_join, 0);  // join
  // the last reduction level (one task per segment) is fused into finish_kernel
  launch_finish(m->dev, H.n_segments, H.rec_doubles, nc, st);
  phase_mark(m, 4, st);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

// the per-sample log-weights into out_dev (catalog order): the prologue's tables and kernel constants on `st`, the grid
// normalisers on the aux stream, joined before the pass.  No stream kernel, no reduction: the per-segment results, the
// speculative shift and the captured graphs of the likelihood calls are untouched (the a-priori shift blocks of the prologue
// are not launched either).
static int sample_log_weights(gwi_model* m, const double* lam_dev, double* out_dev, cudaStream_t st) {
  const ModelDev& H = m->host;
  cudaEventRecord(m->ev_fork, st);
  cudaStreamWaitEvent(m->aux_stream, m->ev_fork, 0);
  launch_prologue_groups(m->dev, lam_dev, H.n_groups, m->max_grid, 1, m->aux_stream);
  cudaEventRecord(m->ev_join, m->aux_stream);
  launch_prologue_tables(m->dev, lam_dev, H.n_groups, H.n_segments, true, 1, st, 0);
  cudaStreamWaitEvent(st, m->ev_join, 0);  // the pass reads logZ
  launch_sample_log_weights(m->dev, H.n_padded, m->sample_index, out_dev, m->plan.n_samples_pe + m->plan.n_samples_inj, st);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

static int check_sample_call(gwi_model* m, const double* lambda_dev, const void* out_dev) {
  if (!m || !lambda_dev || !out_dev) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  if (!m->sample_index) {
    set_error("per-sample weights and draws need a model created with keep_sample_index = 1");
    return GWI_ERR_UNSUPPORTED;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  return GWI_OK;
}

int gwi_sample_log_weights(gwi_model* m, const double* lambda_dev, double* out_dev, void* stream) {
  const int rc = check_sample_call(m, lambda_dev, out_dev);
  if (rc != GWI_OK) return rc;
  return sample_log_weights(m, lambda_dev, out_dev, (cudaStream_t)stream);
}

int gwi_draw_samples(gwi_model* m, const double* lambda_dev, uint64_t seed, int32_t draws_per_event, int32_t draws_inj, int64_t* out_dev, void* stream) {
  if (draws_per_event < 0 || draws_inj < 0) {
    set_error("negative number of draws");
    return GWI_ERR_INVALID;
  }
  int rc = check_sample_call(m, lambda_dev, out_dev);
  if (rc != GWI_OK) return rc;
  const Plan& p = m->plan;
  const int E = (int)p.segments.size() - 1;
  DrawScratch& D = m->draw;
  if (!D.logw) {
    // segments in catalog order: the events (plan segments 1..E), then the injections (plan segment 0)
    std::vector<int64_t> seg_off(E + 2, 0);
    for (int i = 0; i < E; ++i) seg_off[i + 1] = seg_off[i] + p.segments[i + 1].n_total;
    seg_off[E + 1] = seg_off[E] + p.segments[0].n_total;
    std::vector<int32_t> tile_off, tile_seg;
    draw_tiles(seg_off, tile_off, tile_seg);
    DrawScratch N{};
    N.n_seg = E + 1;
    N.n_tiles = (int32_t)tile_seg.size();
    N.n_cat = seg_off[E + 1];
    int64_t* d_off;
    int32_t *d_toff, *d_tseg;
    if ((rc = upload(m, seg_off.data(), seg_off.size(), &d_off)) != GWI_OK || (rc = upload(m, tile_off.data(), tile_off.size(), &d_toff)) != GWI_OK ||
        (rc = upload(m, tile_seg.data(), tile_seg.size(), &d_tseg)) != GWI_OK || (rc = upload<double>(m, nullptr, (size_t)N.n_cat, &N.logw)) != GWI_OK ||
        (rc = upload<double>(m, nullptr, (size_t)N.n_tiles, &N.tile_max)) != GWI_OK || (rc = upload<double>(m, nullptr, (size_t)N.n_tiles, &N.tile_cum)) != GWI_OK ||
        (rc = upload<double>(m, nullptr, (size_t)N.n_seg, &N.seg_max)) != GWI_OK)
      return rc;  // (what was allocated stays in m->allocs until gwi_model_destroy)
    N.seg_off = d_off;
    N.tile_off = d_toff;
    N.tile_seg = d_tseg;
    D = N;
  }
  cudaStream_t st = (cudaStream_t)stream;
  rc = sample_log_weights(m, lambda_dev, D.logw, st);
  if (rc != GWI_OK) return rc;
  launch_draws(D, seed, E, draws_per_event, draws_inj, out_dev, st);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

int gwi_eval(gwi_model* m, const double* lambda_dev, const gwi_outputs* out, void* stream) {
  if (!m || !lambda_dev || !out) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  if ((out->J_logNeff || out->J_logNeff_inj) && !m->plan.g2) {
    set_error("N_eff Jacobians requested but the model was created without need_neff_grad");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = run_eval(m, lambda_dev, 1, st);
  if (rc != GWI_OK) return rc;
  launch_export(m->dev, *out, st);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

int64_t gwi_partial_size(const gwi_model* m) { return m ? (int64_t)PR_HEADER + 3 * (int64_t)m->plan.n_params : (int64_t)GWI_ERR_INVALID; }

int gwi_partial(gwi_model* m, const double* lambda_dev, double* record_dev, void* stream) {
  if (!m || !lambda_dev || !record_dev) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = run_eval(m, lambda_dev, 1, st);
  if (rc != GWI_OK) return rc;
  launch_partial(m->dev, record_dev, m->plan.n_params, 1, st);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

int gwi_combine(gwi_model* m, const double* records_dev, int32_t n_ranks, const gwi_like_opts* opts, double* out_dev, void* stream) {
  if (!m || !records_dev || !opts || !out_dev || n_ranks < 1) {
    set_error("bad argument");
    return GWI_ERR_INVALID;
  }
  if (opts->marginalize_selection && !m->plan.g2) {
    set_error("marginalize_selection needs a model created with need_neff_grad");
    return GWI_ERR_INVALID;
  }
  if (opts->max_variance_cut && (opts->marginalize_selection || opts->min_neff_cut)) {
    set_error("max_variance_cut requires marginalize_selection and min_neff_cut to be off (analysis.py:237-244)");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  launch_combine(m->dev, records_dev, n_ranks, *opts, out_dev, 1, (cudaStream_t)stream);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

int gwi_loglike(gwi_model* m, const double* lambda_dev, const gwi_like_opts* opts, double* out_dev, void* stream) {
  if (!m) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  if (!lambda_dev || !opts || !out_dev) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  if (opts->marginalize_selection && !m->plan.g2) {
    set_error("marginalize_selection needs a model created with need_neff_grad");
    return GWI_ERR_INVALID;
  }
  if (opts->max_variance_cut && (opts->marginalize_selection || opts->min_neff_cut)) {
    set_error("max_variance_cut requires marginalize_selection and min_neff_cut to be off (analysis.py:237-244)");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = run_eval(m, lambda_dev, 1, st);
  if (rc != GWI_OK) return rc;
  // partial record + single-rank combine in one launch (the last block to finish its rows combines)
  launch_partial_tail(m->dev, m->partial_dev, m->plan.n_params, 1, *opts, out_dev, m->comm, 0ull, 1, st);
  phase_mark(m, 5, st);
  m->ph_pending = m->phase_timing;
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

// ---- library-owned multi-GPU exchange ------------------------------------------------------------------
static size_t comm_flag_bytes(int R) { return ((size_t)2 * R * sizeof(unsigned long long) + 255) / 256 * 256; }

int gwi_comm_local_handle(gwi_model* m, int32_t n_ranks, gwi_ipc_handle* out) {
  if (!m || !out || n_ranks < 1 || n_ranks > MAX_RANKS) {
    set_error("bad argument (1 <= n_ranks <= 16)");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  const size_t stride = (size_t)PR_HEADER + 3 * (size_t)m->plan.n_params;
  if (m->comm_base && m->comm.n_ranks != n_ranks) {
    set_error("the exchange buffer of this model was created for another number of ranks");
    return GWI_ERR_INVALID;
  }
  if (!m->comm_base) {
    const size_t bytes = comm_flag_bytes(n_ranks) + (size_t)2 * n_ranks * stride * sizeof(double);
    void* p = nullptr;
    CUDA_TRY(cudaMalloc(&p, bytes));
    m->allocs.push_back(p);
    CUDA_TRY(cudaMemset(p, 0, bytes));
    CUDA_TRY(cudaDeviceSynchronize());
    m->comm_base = p;
    m->comm.n_ranks = n_ranks;
  }
  std::memset(out->bytes, 0, sizeof(out->bytes));
#ifndef GWI_HOST_EMULATION
  cudaIpcMemHandle_t h;
  CUDA_TRY(cudaIpcGetMemHandle(&h, m->comm_base));
  static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
  std::memcpy(out->bytes, &h, 64);
#endif
  const long long pid = (long long)getpid();
  std::memcpy(out->bytes + 64, &pid, 8);
  std::memcpy(out->bytes + 72, &m->comm_base, 8);
  return GWI_OK;
}

int gwi_comm_connect(gwi_model* m, const gwi_ipc_handle* handles, int32_t rank, int32_t n_ranks) {
  if (!m || !handles || n_ranks < 1 || n_ranks > MAX_RANKS || rank < 0 || rank >= n_ranks) {
    set_error("bad argument");
    return GWI_ERR_INVALID;
  }
  if (!m->comm_base || m->comm.n_ranks != n_ranks) {
    set_error("call gwi_comm_local_handle(m, n_ranks, ...) first");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  const size_t fb = comm_flag_bytes(n_ranks);
  for (int p = 0; p < n_ranks; ++p) {
    void* base = nullptr;
    long long pid = 0;
    std::memcpy(&pid, handles[p].bytes + 64, 8);
    if (p == rank) {
      base = m->comm_base;
    } else if (pid == (long long)getpid()) {
      std::memcpy(&base, handles[p].bytes + 72, 8);  // same process: the pointer itself
#ifndef GWI_HOST_EMULATION
      cudaPointerAttributes attr;
      if (cudaPointerGetAttributes(&attr, base) == cudaSuccess && attr.device != m->device) {
        const cudaError_t e = cudaDeviceEnablePeerAccess(attr.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
          set_error(std::string("cudaDeviceEnablePeerAccess failed: ") + cudaGetErrorString(e));
          return GWI_ERR_CUDA;
        }
        cudaGetLastError();
      }
#endif
    } else {
#ifndef GWI_HOST_EMULATION
      cudaIpcMemHandle_t h;
      std::memcpy(&h, handles[p].bytes, 64);
      const cudaError_t e = cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        set_error(std::string("cudaIpcOpenMemHandle of rank ") + std::to_string(p) + " failed: " + cudaGetErrorString(e));
        return GWI_ERR_CUDA;
      }
      m->comm_opened.push_back(base);
#else
      set_error("the host emulator has no inter-process exchange");
      return GWI_ERR_UNSUPPORTED;
#endif
    }
    m->comm.peer_flags[p] = reinterpret_cast<unsigned long long*>(base);
    m->comm.peer_slots[p] = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(base) + fb);
  }
  m->comm.rank = rank;
  m->comm_connected = true;
  return GWI_OK;
}

static int sharded_checks(gwi_model* m, const gwi_like_opts* opts) {
  if (!m->comm_connected) {
    set_error("gwi_comm_connect has not been called on this model");
    return GWI_ERR_INVALID;
  }
  if (opts) {
    if (opts->marginalize_selection && !m->plan.g2) {
      set_error("marginalize_selection needs a model created with need_neff_grad");
      return GWI_ERR_INVALID;
    }
    if (opts->max_variance_cut && (opts->marginalize_selection || opts->min_neff_cut)) {
      set_error("max_variance_cut requires marginalize_selection and min_neff_cut to be off (analysis.py:237-244)");
      return GWI_ERR_INVALID;
    }
  }
  return GWI_OK;
}

int gwi_loglike_sharded(gwi_model* m, const double* lambda_dev, const gwi_like_opts* opts, double* out_dev, void* stream) {
  if (!m || !lambda_dev || !opts || !out_dev) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  int rc = sharded_checks(m, opts);
  if (rc != GWI_OK) return rc;
  CUDA_TRY(cudaSetDevice(m->device));
  rc = run_eval(m, lambda_dev, 1, (cudaStream_t)stream);
  if (rc != GWI_OK) return rc;
  m->comm_pushed = ++m->comm_epoch;
  // partial record, push to every rank, wait for every rank, combine: one launch
  launch_partial_tail(m->dev, m->partial_dev, m->plan.n_params, 2, *opts, out_dev, m->comm, m->comm_epoch, 1, (cudaStream_t)stream);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

int gwi_sharded_push(gwi_model* m, const double* lambda_dev, void* stream) {
  if (!m || !lambda_dev) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  int rc = sharded_checks(m, nullptr);
  if (rc != GWI_OK) return rc;
  rc = gwi_partial(m, lambda_dev, m->partial_dev, stream);
  if (rc != GWI_OK) return rc;
  m->comm_pushed = ++m->comm_epoch;
  gwi_like_opts none{};
  launch_exchange(m->dev, m->partial_dev, m->comm, m->comm_epoch, 1, none, nullptr, (cudaStream_t)stream);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

int gwi_sharded_combine(gwi_model* m, const gwi_like_opts* opts, double* out_dev, void* stream) {
  if (!m || !opts || !out_dev) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  const int rc = sharded_checks(m, opts);
  if (rc != GWI_OK) return rc;
  if (m->comm_pushed != m->comm_epoch || m->comm_epoch == 0) {
    set_error("gwi_sharded_combine without a preceding gwi_sharded_push");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  m->comm_pushed = 0;
  launch_exchange(m->dev, m->partial_dev, m->comm, m->comm_epoch, 2, *opts, out_dev, (cudaStream_t)stream);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

int gwi_loglike_batch(gwi_model* m, const double* lambda_dev, int32_t n_chains, const gwi_like_opts* opts, double* out_dev, void* stream) {
  if (!m || !lambda_dev || !out_dev || !opts || n_chains < 1 || n_chains > 65535) {
    set_error("bad argument (1 <= n_chains <= 65535)");
    return GWI_ERR_INVALID;
  }
  if (opts->marginalize_selection && !m->plan.g2) {
    set_error("marginalize_selection needs a model created with need_neff_grad");
    return GWI_ERR_INVALID;
  }
  if (opts->max_variance_cut && (opts->marginalize_selection || opts->min_neff_cut)) {
    set_error("max_variance_cut requires marginalize_selection and min_neff_cut to be off (analysis.py:237-244)");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  if (n_chains == 1) return gwi_loglike(m, lambda_dev, opts, out_dev, stream);
  int rc = ensure_chains(m, n_chains);
  if (rc != GWI_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  // ONE launch of every kernel covers all chains (chain = a grid coordinate): the whole machine works
  // on the batch instead of one small catalog at a time
  rc = run_eval(m, lambda_dev, n_chains, st);
  if (rc != GWI_OK) return rc;
  launch_partial_tail(m->dev, m->partial_batch, m->plan.n_params, 1, *opts, out_dev, m->comm, 0ull, n_chains, st);
  CUDA_TRY(cudaGetLastError());
  return GWI_OK;
}

int gwi_loglike_host(gwi_model* m, const double* lambda_host, const gwi_like_opts* opts, double* out_host) {
  if (!m || !lambda_host || !out_host) {
    set_error("null argument");
    return GWI_ERR_INVALID;
  }
  CUDA_TRY(cudaSetDevice(m->device));
  const int P = m->plan.n_params;
  std::memcpy(m->lam_pinned, lambda_host, sizeof(double) * P);
  m->spec_allowed_now = m->spec_shift;
  struct SpecGuard {
    gwi_model* m;
    ~SpecGuard() { m->spec_allowed_now = false; }
  } spec_guard{m};
  if (m->use_graph && opts && !m->timing && !m->force_exact_shift) {
    // the kernels take `opts` by value: a graph is valid for the options it was captured with
    if (m->graph_exec && std::memcmp(&m->graph_opts, opts, sizeof(gwi_like_opts)) != 0) {
      cudaGraphExecDestroy(m->graph_exec);
      m->graph_exec = nullptr;
    }
    if (!m->graph_exec) {
      cudaGraph_t graph = nullptr;
      CUDA_TRY(cudaStreamBeginCapture(m->own_stream, cudaStreamCaptureModeThreadLocal));
      cudaMemcpyAsync(m->lam_dev, m->lam_pinned, sizeof(double) * P, cudaMemcpyHostToDevice, m->own_stream);
      const int rc_cap = gwi_loglike(m, m->lam_dev, opts, m->out_dev, m->own_stream);
      cudaMemcpyAsync(m->out_pinned, m->out_dev, sizeof(double) * (GWI_LIKE_HEADER + P), cudaMemcpyDeviceToHost, m->own_stream);
      const cudaError_t e_end = cudaStreamEndCapture(m->own_stream, &graph);  // always ends the capture, also after an error
      bool graph_ok = rc_cap == GWI_OK && e_end == cudaSuccess && graph != nullptr;  // (a genuine argument error shows again on the eager path)
      if (graph_ok) {
        const cudaError_t e_inst = cudaGraphInstantiate(&m->graph_exec, graph, 0);
        graph_ok = e_inst == cudaSuccess;
        if (!graph_ok) m->graph_exec = nullptr;
      }
      if (graph) cudaGraphDestroy(graph);
      if (!graph_ok) {
        // this driver cannot capture the launch sequence (e.g. programmatic dependent launches inside a capture): eager launches
        // from now on -- same results, a few microseconds more host latency per call
        cudaGetLastError();
        m->use_graph = false;
      } else {
        m->graph_opts = *opts;
      }
    }
  }
  if (m->use_graph && m->graph_exec && opts && !m->timing && !m->force_exact_shift) {
    CUDA_TRY(cudaGraphLaunch(m->graph_exec, m->own_stream));
  } else {
    CUDA_TRY(cudaMemcpyAsync(m->lam_dev, m->lam_pinned, sizeof(double) * P, cudaMemcpyHostToDevice, m->own_stream));
    const int rc = gwi_loglike(m, m->lam_dev, opts, m->out_dev, m->own_stream);
    if (rc != GWI_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(m->out_pinned, m->out_dev, sizeof(double) * (GWI_LIKE_HEADER + P), cudaMemcpyDeviceToHost, m->own_stream));
  }
  CUDA_TRY(cudaStreamSynchronize(m->own_stream));
  std::memcpy(out_host, m->out_pinned, sizeof(double) * (GWI_LIKE_HEADER + P));
  if (out_host[GWI_LIKE_STATUS] != 0.0 && (!m->host.two_pass || m->spec_shift) && !m->force_exact_shift) {
    m->spec_allowed_now = false;
    // the a-priori shift bound was too loose for this Lambda (all weights of a segment
    // underflowed): repeat once with the exact per-segment maximum
    m->force_exact_shift = true;
    const int rc2 = gwi_loglike(m, m->lam_dev, opts, m->out_dev, m->own_stream);
    m->force_exact_shift = false;
    if (rc2 != GWI_OK) return rc2;
    CUDA_TRY(cudaMemcpyAsync(m->out_pinned, m->out_dev, sizeof(double) * (GWI_LIKE_HEADER + P), cudaMemcpyDeviceToHost, m->own_stream));
    CUDA_TRY(cudaStreamSynchronize(m->own_stream));
    std::memcpy(out_host, m->out_pinned, sizeof(double) * (GWI_LIKE_HEADER + P));
  }
  if (out_host[GWI_LIKE_STATUS] != 0.0) {
    set_error("a segment's weights all under/overflowed the fp64 range");
    return GWI_ERR_RANGE;
  }
  return GWI_OK;
}

int gwi_loglike_batch_host(gwi_model* m, const double* lambda_host, int32_t n_chains, const gwi_like_opts* opts, double* out_host) {
  if (!m || !lambda_host || !out_host || !opts || n_chains < 1 || n_chains > 65535) {
    set_error("bad argument (1 <= n_chains <= 65535)");
    return GWI_ERR_INVALID;
  }
  const int P = m->plan.n_params;
  const size_t row_out = (size_t)GWI_LIKE_HEADER + P;
  if (n_chains == 1) return gwi_loglike_host(m, lambda_host, opts, out_host);
  CUDA_TRY(cudaSetDevice(m->device));
  if (n_chains > m->batch_cap) {
    // staging grows to the largest batch seen (the old, smaller device buffers stay in m->allocs until destroy)
    for (auto& g : m->batch_graphs)
      if (g.second) cudaGraphExecDestroy(g.second);
    m->batch_graphs.clear();
    if (m->lam_pinned_b) cudaFreeHost(m->lam_pinned_b);
    if (m->out_pinned_b) cudaFreeHost(m->out_pinned_b);
    m->lam_pinned_b = m->out_pinned_b = nullptr;
    m->batch_cap = 0;
    if (cudaMallocHost((void**)&m->lam_pinned_b, sizeof(double) * P * n_chains) != cudaSuccess ||
        cudaMallocHost((void**)&m->out_pinned_b, sizeof(double) * row_out * n_chains) != cudaSuccess) {
      set_error("cudaMallocHost failed");
      return GWI_ERR_ALLOC;
    }
    int rc = upload<double>(m, nullptr, (size_t)P * n_chains, &m->lam_dev_b);
    if (rc != GWI_OK) return rc;
    rc = upload<double>(m, nullptr, row_out * n_chains, &m->out_dev_b);
    if (rc != GWI_OK) return rc;
    m->batch_cap = n_chains;
  }
  {
    const int rc = ensure_chains(m, n_chains);  // (outside any capture: it allocates)
    if (rc != GWI_OK) return rc;
  }
  std::memcpy(m->lam_pinned_b, lambda_host, sizeof(double) * P * n_chains);
  const bool want_graph = m->use_graph && !m->timing && !m->force_exact_shift;
  if (want_graph && !m->batch_graphs.empty() && std::memcmp(&m->batch_graph_opts, opts, sizeof(gwi_like_opts)) != 0) {
    for (auto& g : m->batch_graphs)
      if (g.second) cudaGraphExecDestroy(g.second);
    m->batch_graphs.clear();
  }
  cudaGraphExec_t exec = nullptr;
  if (want_graph) {
    auto it = m->batch_graphs.find(n_chains);
    if (it != m->batch_graphs.end()) {
      exec = it->second;
    } else if (m->batch_graphs.size() < 64) {
      cudaGraph_t graph = nullptr;
      CUDA_TRY(cudaStreamBeginCapture(m->own_stream, cudaStreamCaptureModeThreadLocal));
      cudaMemcpyAsync(m->lam_dev_b, m->lam_pinned_b, sizeof(double) * P * n_chains, cudaMemcpyHostToDevice, m->own_stream);
      const int rc_cap = gwi_loglike_batch(m, m->lam_dev_b, n_chains, opts, m->out_dev_b, m->own_stream);
      cudaMemcpyAsync(m->out_pinned_b, m->out_dev_b, sizeof(double) * row_out * n_chains, cudaMemcpyDeviceToHost, m->own_stream);
      const cudaError_t e_end = cudaStreamEndCapture(m->own_stream, &graph);
      bool ok = rc_cap == GWI_OK && e_end == cudaSuccess && graph != nullptr;
      if (ok) ok = cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess;
      if (graph) cudaGraphDestroy(graph);
      if (!ok) {
        cudaGetLastError();
        exec = nullptr;
        m->use_graph = false;  // eager launches from now on (same results)
      } else {
        m->batch_graphs[n_chains] = exec;
        m->batch_graph_opts = *opts;
      }
    }
  }
  if (exec) {
    CUDA_TRY(cudaGraphLaunch(exec, m->own_stream));
  } else {
    CUDA_TRY(cudaMemcpyAsync(m->lam_dev_b, m->lam_pinned_b, sizeof(double) * P * n_chains, cudaMemcpyHostToDevice, m->own_stream));
    const int rc = gwi_loglike_batch(m, m->lam_dev_b, n_chains, opts, m->out_dev_b, m->own_stream);
    if (rc != GWI_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(m->out_pinned_b, m->out_dev_b, sizeof(double) * row_out * n_chains, cudaMemcpyDeviceToHost, m->own_stream));
  }
  CUDA_TRY(cudaStreamSynchronize(m->own_stream));
  std::memcpy(out_host, m->out_pinned_b, sizeof(double) * row_out * n_chains);
  // a chain whose a-priori shift bound was too loose (status != 0) is repeated alone: the single-chain call falls back to
  // the exact per-segment maximum; GWI_ERR_RANGE only if that fails too (the chain's row then keeps its non-zero status)
  int rc_all = GWI_OK;
  for (int c = 0; c < n_chains; ++c) {
    double* row = out_host + (size_t)c * row_out;
    if (row[GWI_LIKE_STATUS] == 0.0) continue;
    const int rc = gwi_loglike_host(m, lambda_host + (size_t)c * P, opts, row);
    if (rc == GWI_ERR_RANGE)
      rc_all = GWI_ERR_RANGE;
    else if (rc != GWI_OK)
      return rc;
  }
  return rc_all;
}

int gwi_model_batch_hint(const gwi_model* m) { return m ? std::max(1, m->plan.batch_hint) : (int)GWI_ERR_INVALID; }

int gwi_model_set_exact_shift(gwi_model* m, int32_t on) {
  if (!m) return GWI_ERR_INVALID;
  m->force_exact_shift = on != 0;
  return GWI_OK;
}

int gwi_model_set_timing(gwi_model* m, int32_t on) {
  if (!m) return GWI_ERR_INVALID;
  CUDA_TRY(cudaSetDevice(m->device));
  if (on && m->ev0.empty()) {
    m->ev0.resize(64);
    m->ev1.resize(64);
    for (int i = 0; i < 64; ++i) {
      CUDA_TRY(cudaEventCreate(&m->ev0[i]));
      CUDA_TRY(cudaEventCreate(&m->ev1[i]));
    }
  }
  m->timing = on != 0;
  m->n_timed = 0;
  return GWI_OK;
}

int gwi_model_stream_times(gwi_model* m, float* ms_out, int32_t cap) {
  if (!m || !ms_out || cap <= 0) return GWI_ERR_INVALID;
  CUDA_TRY(cudaSetDevice(m->device));
  const int64_t n = std::min<int64_t>(std::min<int64_t>(m->n_timed, 64), cap);
  for (int64_t i = 0; i < n; ++i) {
    const int64_t k = (m->n_timed - n + i) % 64;
    CUDA_TRY(cudaEventSynchronize(m->ev1[k]));
    CUDA_TRY(cudaEventElapsedTime(&ms_out[i], m->ev0[k], m->ev1[k]));
  }
  return (int)n;
}

int64_t gwi_model_last_sites(gwi_model* m, double* dst_host, int64_t cap) {
  if (!m) return GWI_ERR_INVALID;
  const int64_t n = 4 * (int64_t)m->plan.segments.size();
  if (!dst_host) return n;
  if (cap < n) {
    set_error("gwi_model_last_sites: destination too small");
    return GWI_ERR_INVALID;
  }
  if (cudaSetDevice(m->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess ||
      cudaMemcpy(dst_host, m->host.seg_out, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost) != cudaSuccess) {
    set_error(std::string("gwi_model_last_sites: ") + cudaGetErrorString(cudaGetLastError()));
    return GWI_ERR_CUDA;
  }
  return n;
}

int gwi_model_get_info(const gwi_model* m, gwi_model_info* info) {
  if (!m || !info) return GWI_ERR_INVALID;
  const Plan& p = m->plan;
  std::memset(info, 0, sizeof(*info));
  info->n_samples_pe = p.n_samples_pe;
  info->n_samples_inj = p.n_samples_inj;
  info->n_valid_pe = p.n_valid_pe;
  info->n_valid_inj = p.n_valid_inj;
  info->n_padded = p.n_padded;
  info->bytes_per_eval = m->bytes_per_eval * (m->host.two_pass ? 2 : 1);
  info->n_chunks = (int)p.chunks.size();
  info->n_stream_columns = p.n_columns;
  info->n_spline_dims = (int)p.dims.size();
  info->n_deep = p.n_deep;
  info->n_linear = 0;
  for (auto& k : p.kops) (k.kind == KOP_LIN ? info->n_linear : info->n_param_terms)++;
  info->grid_blocks = p.grid_blocks;
  info->block_threads = m->stream_block;
  info->kernel_launches_per_eval = m->launches_per_eval;
  info->active_switches = 0 | (m->use_graph ? 2 : 0) | (m->cta ? 4 : 0) | (m->spec_shift ? 8 : 0);
  info->plan_on_device = m->plan_on_device ? 1 : 0;
  for (int i = 0; i < 5; ++i) info->plan_seconds[i] = m->plan_seconds[i];
  return GWI_OK;
}

}  // extern "C"
