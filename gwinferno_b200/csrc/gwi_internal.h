// Internal structures shared by the host plan builder (plan.cpp), the kernels (kernels.cu) and
// the C-ABI glue (api.cu).  Not part of the public interface (include/gwi.h).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "gwi.h"

// host + device functions (the plan builders' per-sample arithmetic, the shared-memory layouts); plain functions in
// the host warp emulator's g++ build.  GWI_HD_INLINE: inlined before the caller is optimised, so that the caller compiles
// as if the body were written out in it.
#if defined(__CUDACC__) && !defined(GWI_HOST_EMULATION)
#define GWI_HD __host__ __device__
#define GWI_HD_INLINE __host__ __device__ __forceinline__
#else
#define GWI_HD
#define GWI_HD_INLINE inline
#endif

namespace gwi {

constexpr int MAX_SPLINE_DIMS = 8;  // spline dimensions per model
constexpr int MAX_ROWS = 62;        // polynomial pieces per dimension incl. the dummy row (12-bit field, 64-bit occupancy mask)
constexpr int MAX_KOPS = 16;        // non-spline per-sample operations
constexpr int MAX_GSLOTS = 32;      // gradient slots of the non-spline operations
constexpr int MAX_SOPS = 16;        // scalar (sample-independent) normaliser operations
constexpr int KC_STRIDE = 12;       // doubles of per-eval constants per kop
constexpr int LANES = 32;
constexpr uint32_t SAMPLE_INDEX_PAD = 0xFFFFFFFFu;  // Plan::sample_index of lane padding
constexpr int UNROLL = 2;           // samples per lane per load (16-byte vector loads)
// copies of the deep accumulators per warp: lanes l and l+16 share a slot (two update phases, half the
// shared memory of fully lane-private copies)
constexpr int DEEP_LANES = 16;

// ---- packed spline word: the fp64 value w = u - 1/2 (u in [0,1): offset inside the polynomial piece)
// with its 6 least significant mantissa bits replaced by the piece index J.  The kernels use the word
// AS the double w (no unpack arithmetic; the J bits perturb w by < 2^-46 |w|, i.e. the sample's
// coordinate by < 1e-14 of a knot spacing, the same for the value and for the gradient) and take
// J = low word & 63.
constexpr uint64_t J_MASK = 63ull;
static_assert(MAX_ROWS <= 64, "the piece index must fit the 6 low mantissa bits of the packed word");

// per-sample operation executed by the stream kernel besides the spline dimensions
enum KopKind : int32_t {
  KOP_LIN = 1,       // x += theta * F                       gslots: theta
  KOP_PLRATIO = 2,   // powerlaw in q with per-sample lower bound: cols (log q, log lo)   gslots: beta
  KOP_PLPEAK = 3,    // cols (log m1, m1)                     gslots: alpha, mu, sigma, lam [, delta]
  KOP_ISOALIGN = 4,  // col (cos tilt)                        gslots: xi, sigma
  KOP_QUAD = 5,      // truncated normal body: col (x)        gslots: mu, sigma
  KOP_SMOOTH = 6,    // low-mass window: col (x - xmin)       gslots: delta
  KOP_ISOALIGN2 = 7  // cols (cos tilt 1, cos tilt 2)         gslots: xi, sigma
};

struct Kop {
  int32_t kind;
  int32_t col[2];     // stream-column indices of its features
  int32_t gslot;      // first generic gradient slot
  int32_t n_gslots;
  int32_t slot[6];    // Lambda slots
  double cst[4];      // LIN: cst[0] = offset added to Lambda[slot]; PLPEAK/QUAD: lo, hi
  int32_t norm_group; // LIN only
  int32_t grid_off;   // offset of its grid feature in the grid pool (doubles), -1 none
};

// scalar normaliser operation (prologue): K += value, dK[slot] += derivative
enum SopKind : int32_t {
  SOP_POWERLAW_NORM = 1,  // log[(1+a)/(hi^(1+a) - lo^(1+a))]
  SOP_BETA_NORM = 2,      // -betaln(a,b) - (a+b-1) log s
  SOP_TRUNCNORM_NORM = 3  // -log(sigma) - log sqrt(2 pi) - log(Phi(b) - Phi(a))
};
struct Sop {
  int32_t kind;
  int32_t slot[2];
  double cst[2];
};

struct SplineDim {
  int32_t term;      // index in the model description
  int32_t n_splines;
  int32_t rows;      // n_splines - 2 : pieces 0..rows-2 are real, piece rows-1 is the all-zero dummy
  int32_t row_off;   // first row in the concatenated tables
  int32_t slot;      // first coefficient in Lambda
  int32_t column;    // stream column
  int32_t deep;      // accumulated in lane-private shared memory
  int32_t norm_group;
  int32_t grid_off;  // offset of its grid xi array in the grid pool, -1 none
  int32_t grid_aux;  // offset of the derived per-grid-point taps: W[4G], J[G], then lo[n], hi[n] per basis
  int32_t outside;
  int32_t liny;      // GWI_TERM_SPLINE_LINEAR: the spline is the density (log-weight = log of the cubic)
  // explicit knot vector / order (gwi_term.knots): per-piece tables in the grid pool, -1 = default uniform cubic pieces
  int32_t basis_off;  // [rows-1][4][4]: basis first[J]+k on piece J = sum_n basis[J][k][n] w^n
  int32_t first_off;  // [rows-1]: first coefficient a piece uses (stored as doubles)
  int32_t floor_off;  // [rows-1]: 0 where the piece's bases do not sum to one (spline <= max(max c, 0)), else -inf
};

struct NormGroup {
  int32_t n_grid;
  int32_t logw_off;  // offset in the grid pool
};

struct Chunk {
  int32_t segment;
  int32_t steps;        // samples per lane (multiple of 2*UNROLL)
  int64_t first;        // first padded sample index (multiple of 32*UNROLL)
  int32_t record_slot;  // level-0 record receiving this chunk's sums
  int32_t pad;          // (every chunk writes and clears its own record)
};

struct Segment {
  int64_t n_total;      // samples given (denominator of the Monte-Carlo mean)
  int64_t n_valid;
  int32_t first_chunk, n_chunks;
  double max_static;    // max_j of the static log-weight
  uint64_t occ[MAX_SPLINE_DIMS];  // occupied pieces per spline dim
  double fmin[MAX_KOPS], fmax[MAX_KOPS];  // LIN feature range (for the shift bound)
};

struct ReduceTask {
  int32_t out_slot;  // slot in the output buffer of this level
  int32_t in_first;  // first slot in the input buffer
  int32_t in_count;
  int32_t src;       // where the inputs are: -1 = the level-0 records of the stream kernel, l >= 0 = the output buffer of level l
};

// Host-side evaluation plan ("what the stream kernel reads")
struct Plan {
  // model structure
  int n_params = 0, n_terms = 0;
  bool g2 = false;
  std::vector<SplineDim> dims;   // in SORT-KEY order; the last n_deep are "deep"
  int n_deep = 0;
  int rows_total = 0;
  std::vector<Kop> kops;         // LIN kops first
  int n_lin = 0;                 // number of leading LIN kops
  int n_gslots = 0;
  std::vector<Sop> sops;
  std::vector<NormGroup> groups;
  std::vector<double> grid_pool;  // all grid arrays back to back
  // sample streams
  int n_columns = 0;              // spline columns, then kop feature columns, then the static log-weight
  int col_static = 0;
  int64_t n_padded = 0;
  std::vector<uint64_t> columns;  // [n_padded/64][n_columns][64]: blocks of one warp iteration
  // gwi_model_desc.keep_sample_index: catalog position of the sample at every padded position (PE samples in event order,
  // then the injections), SAMPLE_INDEX_PAD for lane padding.  Host builder only (the device builder writes device memory).
  bool keep_index = false;
  std::vector<uint32_t> sample_index;
  std::vector<Chunk> chunks;
  std::vector<int32_t> slice_begin;  // slice i = chunks [slice_begin[i], slice_begin[i+1]); warp = i % W
  std::vector<Segment> segments;  // segment 0 = injections, 1..E = events
  // level-0 records and the reduction tree
  int rec_doubles = 0;
  int n_records0 = 0;
  // levels.back() has one task per segment (slot = segment; executed by finish_kernel); the earlier levels only hold
  // tasks of the segments that still have more than one fan-in of inputs (a 10 000-sample event goes straight from its
  // few records to the last level instead of being copied through every level)
  std::vector<std::vector<ReduceTask>> levels;
  // launch geometry (fixed at plan time: the chunk -> warp assignment depends on it)
  int grid_blocks = 0, warps_per_block = 0;
  int chunk_steps = 0;
  // CTA-cooperative geometry (stream_cta.cuh): a chunk is processed by ALL `cta_main_warps` main warps of one
  // CTA (its padded range = cta_main_warps sub-chunks of steps x 32 samples) and owns cta_main_warps + 1 records
  bool cta_mode = false;
  int batch_hint = 1;  // chains per launch the geometry was laid out for (gwi_model_desc.batch_hint)
  int cta_main_warps = 0;
  double total_inj = 0.0;
  int64_t n_samples_pe = 0, n_samples_inj = 0, n_valid_pe = 0, n_valid_inj = 0;
};

struct CatalogView {
  int n_columns = 0;
  int n_events = 0;
  std::vector<int64_t> pe_offsets;
  std::vector<const double*> pe_columns, inj_columns;
  int64_t n_inj = 0;
  double total_inj = 0.0;
  int device = 0;
  bool on_device = false;  // the column pointers are device pointers (gwi_catalog_desc.columns_on_device)
};

// record layout helpers --------------------------------------------------------------------------
// [0]=S1 [1]=S2 | g1[n_gslots] | g2[n_gslots] (g2 only) | M1[rows_total*4] | M2[rows_total*4] (g2 only)
inline int rec_off_g1() { return 2; }
inline int rec_off_g2(int ngs) { return 2 + ngs; }
inline int rec_off_m1(int ngs, bool g2) { return 2 + ngs * (g2 ? 2 : 1); }
inline int rec_off_m2(int ngs, bool g2, int rows_total) { return rec_off_m1(ngs, g2) + rows_total * 4; }
inline int rec_size(int ngs, bool g2, int rows_total) { return 2 + (ngs + rows_total * 4) * (g2 ? 2 : 1); }

void set_error(const std::string& msg);
int build_plan(const CatalogView& cat, const gwi_model_desc& desc, int sm_count, int n_workers, Plan& plan);
// flat LCDM Planck15-LVK dVc/dz (cosmology.py:48-120)
double log_dvcdz(double z);

}  // namespace gwi
