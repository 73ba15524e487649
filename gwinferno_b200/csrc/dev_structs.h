// Device-visible, trivially copyable mirrors of the plan (passed to kernels by value / pointer).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdlib>

#include "gwi_internal.h"

// kernel<<<grid, block, dynamic shared bytes, stream>>>(args...).  The only other expansion is the
// host warp emulator of the CPU test suite (tests/emu/cuda_runtime.h: test infrastructure that
// compiles these same kernel sources with g++; it is never part of libgwi.so).
#ifdef GWI_HOST_EMULATION
#define GWI_LAUNCH(kernel, grid, block, smem, stream) GWI_EMU_LAUNCH(kernel, grid, block, smem, stream)
#define GWI_LAUNCH_PDL(kernel, grid, block, smem, stream) GWI_EMU_LAUNCH(kernel, grid, block, smem, stream)
#define GWI_PDL_WAIT() ((void)0)
#define GWI_PDL_TRIGGER() ((void)0)
#else
#define GWI_LAUNCH(kernel, grid, block, smem, stream) kernel<<<(grid), (block), (smem), (stream)>>>
// Programmatic dependent launch: the kernels of one evaluation form a chain of small dependent launches (~8 us each in
// situ, mostly launch latency + ramp + dependent loads).  A kernel launched with the programmatic-serialisation attribute may
// be SCHEDULED as soon as every block of its predecessor has executed GWI_PDL_TRIGGER(); it runs its preamble (descriptor
// staging, task lookup, shared-memory initialisation -- static data only) and blocks in GWI_PDL_WAIT() until the predecessor
// grid has completed and its writes are visible.  GWI_PDL=0 launches everything with plain stream order (A/B measurement).
namespace gwi {
inline bool pdl_enabled() {
  static const bool on = [] {
    const char* e = std::getenv("GWI_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}
template <class... KArgs>
struct PdlLauncher {
  void (*kernel)(KArgs...);
  dim3 grid, block;
  size_t smem;
  cudaStream_t stream;
  template <class... A>
  void operator()(A... args) const {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
  }
};
template <class... KArgs>
PdlLauncher<KArgs...> make_pdl_launcher(void (*k)(KArgs...), dim3 g, dim3 b, size_t s, cudaStream_t st) {
  return PdlLauncher<KArgs...>{k, g, b, s, st};
}
}  // namespace gwi
#define GWI_LAUNCH_PDL(kernel, grid, block, smem, stream) gwi::make_pdl_launcher((kernel), dim3(grid), dim3(block), (size_t)(smem), (stream))
#define GWI_PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
#define GWI_PDL_TRIGGER() asm volatile("griddepcontrol.launch_dependents;" ::: "memory")
#endif

// Speculative shift (on by default; run-time switch GWI_SPECULATIVE_SHIFT=0 turns it off): models without an
// a-priori bound of their log-weights (parametric terms, spline densities) need the exact per-segment maximum as the
// log-sum-exp shift -- a max-only pass before the full pass.  Instead the full pass of the generic-term stream kernel also
// records every chunk's max x, and the NEXT evaluation of gwi_loglike_host takes its shift from THIS evaluation's exact maxima;
// an evaluation whose maxima moved by more than SPEC_SHIFT_TOL from the shift it used is flagged and repeated with the exact
// maximum by the host call.  Measured on B200 (cfg1, profiles/r02_call37_speculative_shift.txt): host call 308 -> 211 us per
// evaluation, results equal; the recording costs the spline-only kernels nothing (compiled into the PARAM variants only).

namespace gwi {

constexpr double SPEC_SHIFT_TOL = 300.0;  // p = e^(x - shift) within e^+-300 at the maximum: p and p^2 (N_eff sums) stay far from the fp64 limits

// Power-law normaliser (distributions.py:111-116), shared by the prologue (SOP_POWERLAW_NORM, KOP_PLPEAK) and the stream
// kernel (KOP_PLRATIO, per sample): lognorm = -log int_lo^hi x^(a1-1) dx and d lognorm / d a1, given log lo, L = log(hi/lo)
// and inv_a1 = 1/a1 (0 at a1 = 0; the stream kernel takes it from the prologue instead of dividing per sample).
// With z = a1 L the integral is lo^a1 L expm1(z)/z = lo^a1 expm1(z)/a1, so lognorm = -a1 log lo - log(expm1(z)/a1) (-log L at
// z = 0) and the derivative is -log lo - L g(z), g(z) = 1/(1 - e^-z) - 1/z, i.e. 1/a1 - log hi - L/expm1(z).  No difference of
// powers and no switch near a1 = 0 (alpha = -1).  The direct form of g loses ~eps/|z| to cancellation, so below |z| = 0.1 g is
// its series (Bernoulli numbers; the first omitted term is < 3e-17 there).
__device__ __forceinline__ void powerlaw_lognorm(double a1, double inv_a1, double loglo, double L, double& lognorm, double& dnorm) {
  const double z = a1 * L;
  const double em1 = expm1(z);
  lognorm = -a1 * loglo - log(z != 0.0 ? em1 * inv_a1 : L);
  const double z2 = z * z;
  dnorm = fabs(z) < 0.1 ? -loglo - L * (0.5 + z * (1.0 / 12.0 + z2 * (-1.0 / 720.0 + z2 * (1.0 / 30240.0 - z2 * (1.0 / 1209600.0)))))
                        : inv_a1 - (loglo + L) - L / em1;
}

struct DimDev {
  int32_t rows, row_off, slot, n_splines;
  int32_t deep, deep_off;  // deep_off: first double2 entry of this dim in the lane-private deep block
  int32_t norm_group, grid_off;
  int32_t grid_aux, liny;  // derived grid taps (see SplineDim::grid_aux); liny: SplineDim::liny
  int32_t basis_off, first_off;  // SplineDim::basis_off / first_off (-1: uniform cubic pieces)
  int32_t floor_off, pad_;
  double xi_lo, inv_dxi;
};

struct KopDev {
  int32_t kind, col0, col1, gslot;
  int32_t n_gslots, norm_group, grid_off, pad;
  int32_t slot[6], pad2[2];
  double cst[4];
};

struct SopDev {
  int32_t kind, slot0, slot1, pad;
  double cst0, cst1;
};

struct SegDev {
  double n_total;     // Monte-Carlo denominator (events); injections use total_inj
  double max_static;
  uint64_t occ[MAX_SPLINE_DIMS];
  double fmin[MAX_KOPS], fmax[MAX_KOPS];
  int32_t first_chunk, n_chunks;
};

struct GroupDev {
  int32_t n_grid, logw_off;
};

// everything the kernels need, resident in device global memory: one descriptor per CHAIN (the
// static pointers are shared, the per-evaluation scratch pointers differ); kernels index the
// descriptor array with their chain coordinate of the grid
struct ModelDev {
  int32_t n_params, n_dims, n_deep, n_kops, n_gslots, n_sops, n_groups, n_segments;
  int32_t rows_total, rec_doubles, n_columns, col_static, g2, two_pass, n_chunks, deep_rows;  // deep_rows: table rows of the deep dims
  int32_t n_lin_fast, n_slices;  // leading LIN kops handled in registers by the stream kernel
  int64_t n_padded;
  double total_inj;
  DimDev dims[MAX_SPLINE_DIMS];
  KopDev kops[MAX_KOPS];
  SopDev sops[MAX_SOPS];
  int32_t gslot_slot[MAX_GSLOTS];  // generic gradient slot -> Lambda slot
  // static arrays
  const uint64_t* columns;  // [n_padded/64][n_columns][64]
  const Chunk* chunks;
  const int32_t* slice_begin;  // [n_slices + 1]
  const SegDev* segs;
  const GroupDev* groups;
  const double* grid_pool;
  // per-evaluation scratch
  double* tables;     // [rows_total*4] polynomial pieces in w = u - 1/2
  double* piece_ub;   // [rows_total]   max of the 4 coefficients of each piece
  double* kc;         // [n_kops*KC_STRIDE]
  double* shift;      // [n_segments]
  double* logZ;       // [n_groups]
  double* dlogZ;      // [n_groups*P]
  double* Ksum;       // [1 + P] : K = sum(sops) - sum(logZ), then dK
  double* chunk_max;  // [n_chunks] (two-pass mode)
  int32_t* slice_counter;  // [2] dynamic slice scheduling: [0] full pass, [1] max-only pass; reset by the prologue
  double* records0;   // [n_records0 * rec]
  double* level_buf[6];              // output of reduction level l (the last level is fused into finish)
  const ReduceTask* level_tasks[6];  // static task lists
  int32_t level_ntasks[6];
  int32_t n_levels, liny_mask;  // bit d: spline dim d is a linear-in-y density
  double* seg_out;    // [n_segments * 4] {logmean, logneff, var, status}
  double* seg_J1;     // [n_segments * P]
  double* seg_Jn;     // [n_segments * P]
  double* inj_raw;    // [3 + 2P] {shift, S1, S2, G1raw[P], G2raw[P]}
  // speculative shift: maxima learned from the last full pass; 1.0 where the shift used was too far off
  double* shift_next;  // [n_segments]
  double* spec_bad;    // [n_segments], zero unless a speculative evaluation has to be repeated
  // CTA-cooperative stream kernel (stream_cta.cuh): main warps per CTA (0 = the one-role kernel's geometry)
  int32_t cta_main_warps, cta_lead_doubles;  // cta_lead_doubles: header + linear slots + leading rows of a record (what a main warp writes)
  int32_t* tail_counter;  // arrival counter of partial_tail_kernel (zero between evaluations)
};

// posterior-predictive draws (sample_draw.cuh) over the catalog-order log-weights: segment s = event s (s < E) or the injection
// set (s = E) covers catalog positions [seg_off[s], seg_off[s+1]) and is cut into tiles of DRAW_TILE samples that never
// straddle segments (tiles [tile_off[s], tile_off[s+1]) of segment s).  Allocated on the first draw, owned by the model.
constexpr int DRAW_TILE = 256;
struct DrawScratch {
  double* logw = nullptr;       // [n_cat] log-weights, catalog order
  double* tile_max = nullptr;   // [n_tiles]
  double* tile_cum = nullptr;   // [n_tiles] inclusive prefix over the segment's tiles of sum exp(x - seg_max)
  double* seg_max = nullptr;    // [n_seg]
  const int64_t* seg_off = nullptr;   // [n_seg + 1]
  const int32_t* tile_off = nullptr;  // [n_seg + 1]
  const int32_t* tile_seg = nullptr;  // [n_tiles]
  int32_t n_seg = 0, n_tiles = 0;
  int64_t n_cat = 0;
};

// multi-GPU exchange (exchange_kernel): the exchange buffers of every rank as seen from this rank (peer
// memory), passed to the kernel by value
constexpr int MAX_RANKS = 16;
struct CommDev {
  double* peer_slots[MAX_RANKS];              // rank p's slots  [2 parities][n_ranks][PR_HEADER + 3P]
  unsigned long long* peer_flags[MAX_RANKS];  // rank p's flags  [2 parities][n_ranks]: epoch of the record in the slot
  int32_t rank, n_ranks;
};

// partial (per-rank) likelihood record: 8 header doubles + 3P
enum { PR_SHIFT = 0, PR_S1 = 1, PR_S2 = 2, PR_SUM_LOGBF = 3, PR_MIN_LOGNEFF = 4, PR_SUM_VAR = 5, PR_N_EVENTS = 6, PR_STATUS = 7, PR_HEADER = 8 };

}  // namespace gwi
