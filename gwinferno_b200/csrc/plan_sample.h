// Per-sample arithmetic of the plan builders, shared by the host builder (plan.cpp) and the device builder
// (plan_device.cu): validity (model masks, single.py:54-55; cuts), the polynomial piece + local coordinate of a
// spline coordinate (interpolation.py:98-106,128-149 for uniform knots), the packed word, the static features
// (log dVc/dz of cosmology.py:95-120, logs of the coordinates).  Every function is host + device.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
#include <memory>
#include <vector>

#include "gwi_internal.h"

namespace gwi {

GWI_HD inline double plan_nan() {
  const uint64_t b = 0x7ff8000000000000ull;
  double d;
  memcpy(&d, &b, 8);
  return d;
}
GWI_HD inline double plan_inf() {
  const uint64_t b = 0x7ff0000000000000ull;
  double d;
  memcpy(&d, &b, 8);
  return d;
}
GWI_HD inline bool plan_finite(double x) { return ::fabs(x) <= 1.7976931348623157e308; }  // false for NaN

// ---- cosmology: flat LCDM, Planck15-LVK constants (gwinferno/cosmology.py:19-22); the comoving-distance table
// (sequential trapezoid on z = arange(0, 10, 1e-3), cosmology.py:48-77) is built once on the host (plan.cpp)
struct CosmoView {
  const double* Dc;  // Dc[i] at z = i * 1e-3
  int n;
  double c_over_Ho;
};
constexpr double COSMO_OM = 0.3065;
constexpr double COSMO_OL = 1.0 - 0.3065;
constexpr double COSMO_DZ = 1e-3;

GWI_HD inline double cosmo_dDcdz(const CosmoView& c, double zz) {
  const double opz = 1.0 + zz;
  return c.c_over_Ho / ::sqrt(COSMO_OL + COSMO_OM * opz * opz * opz);
}
// Dc by linear interpolation in the table (cosmology.py:111-120)
GWI_HD inline double cosmo_interp_Dc(const CosmoView& c, double zz) {
  if (!(zz >= 0.0)) return plan_nan();
  const int n = c.n;
  if (zz >= (double)(n - 1) * COSMO_DZ) return plan_nan();  // beyond the table (z < 10)
  int i = (int)(zz / COSMO_DZ);
  if (i > n - 2) i = n - 2;
  while (i > 0 && (double)i * COSMO_DZ > zz) --i;
  while (i < n - 2 && (double)(i + 1) * COSMO_DZ <= zz) ++i;
  const double z0 = (double)i * COSMO_DZ, z1 = (double)(i + 1) * COSMO_DZ;
  const double f = (zz - z0) / (z1 - z0);
  return c.Dc[i] + f * (c.Dc[i + 1] - c.Dc[i]);
}
// log of dVc/dz = 4 pi Dc^2 (c/H0)/E(z)  (cosmology.py:95-101)
GWI_HD inline double cosmo_log_dvcdz(const CosmoView& c, double z) {
  const double Dc = cosmo_interp_Dc(c, z);
  return ::log(4.0 * 3.14159265358979323846 * Dc * Dc * cosmo_dDcdz(c, z));
}

// ---- per-sample features -------------------------------------------------------------------------
enum FeatKind : int { F_LOG1P = 1, F_LOG = 2, F_LOG_RATIO = 3, F_LOG_DVDZ = 4, F_NEG_LOG = 5, F_RAW = 6, F_LOG_C_OVER = 7, F_LOG_S_MINUS = 8, F_NEG_LOG1P = 9, F_CONST = 10, F_MINUS_C = 11, F_PROD_MINUS_C = 12 };
struct Feat {
  int kind;
  int col[2];
  double cst;
};

GWI_HD inline double eval_feat(const Feat& f, const double* const* cols, int64_t j, const CosmoView& cv) {
  const double a = cols[f.col[0]][j];
  switch (f.kind) {
    case F_LOG1P: return ::log(1.0 + a);
    case F_LOG: return ::log(a);
    case F_LOG_RATIO: return ::log(a / cols[f.col[1]][j]);
    case F_LOG_DVDZ: return cosmo_log_dvcdz(cv, a);
    case F_NEG_LOG: return -::log(a);
    case F_NEG_LOG1P: return -::log(1.0 + a);
    case F_CONST: return f.cst;
    case F_MINUS_C: return a - f.cst;
    case F_PROD_MINUS_C: return a * cols[f.col[1]][j] - f.cst;
    case F_RAW: return a;
    case F_LOG_C_OVER: return ::log(f.cst / a);
    case F_LOG_S_MINUS: return ::log(f.cst - a);
  }
  return plan_nan();
}

struct RangeCut {
  int kind;  // 1 range, 2 ratio range, 3 open range (lo < x < hi), 4 q >= c/m1 && q <= 1 && c/m1 < 1
  int col[2];
  double lo, hi;
};

GWI_HD inline bool pass_cut(const RangeCut& c, const double* const* cols, int64_t j) {
  const double a = cols[c.col[0]][j];
  switch (c.kind) {
    case 1: return a >= c.lo && a <= c.hi;
    case 2: {
      const double r = a / cols[c.col[1]][j];
      return r >= c.lo && r <= c.hi;
    }
    case 3: return a > c.lo && a < c.hi;
    case 4: {
      const double lo = c.lo / cols[c.col[1]][j];
      return a >= lo && a <= 1.0 && lo < 1.0;
    }
  }
  return false;
}

struct SplineGeom {
  int col;
  int logx;
  int outside;
  int rows;
  double x_lo, x_hi, xi_lo, xi_hi, inv_dxi;
  // explicit knot vector (gwi_term.knots): piece J covers [piece_lo[J], piece_lo[J+1]) of the spline coordinate and its
  // local coordinate is u = (xi - piece_origin[J]) * piece_inv_h[J] (origin and width of the knot SPAN the piece lies in).
  // n_pieces == 0: the default uniform pieces.  Host pointers in the host builder, device pointers in the device builder.
  int n_pieces;
  int pad_;
  const double* piece_lo;
  const double* piece_origin;
  const double* piece_inv_h;
};

// piece index and local coordinate u in [0,1) of one sample; returns false if the sample must be
// dropped (GWI_OUTSIDE_DROP and outside the mask)
GWI_HD inline bool spline_locate(const SplineGeom& g, double x, int& J, double& u) {
  const bool inside = (x >= g.x_lo) && (x <= g.x_hi);
  if (!inside) {
    if (g.outside == GWI_OUTSIDE_DROP) return false;
    J = g.rows - 1;  // dummy all-zero piece: bases are 0 outside the range (interpolation.py:175)
    u = 0.0;
    return x == x;  // NaN coordinate => drop
  }
  double xi = g.logx ? ::log(x) : x;
  if (xi < g.xi_lo) xi = g.xi_lo;
  if (xi > g.xi_hi) xi = g.xi_hi;
  const double top = 1.0 - 0x1p-52;  // 1 + top = 2 - 2^-52 is the largest double below 2
  int j;
  double uu;
  if (g.n_pieces > 0) {
    // half-open spans as in the reference's order-1 indicator (interpolation.py:143-146): the last piece whose
    // lower edge is <= xi
    int lo = 0, hi = g.n_pieces - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (g.piece_lo[mid] <= xi) lo = mid; else hi = mid - 1;
    }
    j = lo;
    uu = (xi - g.piece_origin[j]) * g.piece_inv_h[j];
  } else {
    const double t = (xi - g.xi_lo) * g.inv_dxi;
    j = (int)::floor(t);
    if (j < 0) j = 0;
    if (j > g.rows - 2) j = g.rows - 2;
    uu = t - (double)j;
  }
  if (uu < 0.0) uu = 0.0;
  if (uu > top) uu = top;
  J = j;
  u = uu;
  return true;
}

GWI_HD inline uint64_t pack_word(int J, double u) {
  const double w = u - 0.5;  // [-1/2, 1/2): the variable of the per-piece polynomials
  uint64_t b;
  memcpy(&b, &w, 8);
  return (b & ~J_MASK) | (uint64_t)J;
}

// ---- what both builders derive from the model description (plan_classify) -------------------------
constexpr uint64_t PLAN_KEY_INVALID = ~0ull;
// per-piece tables of a spline term with an explicit knot vector (plan.cpp: build_piece_table)
struct PieceTable {
  std::vector<double> lo, inv_h;  // [n]: lower edge of the piece; origin / inverse width of its knot span
  std::vector<double> origin;     // [n]: origin of the local coordinate (the span's lower knot)
  std::vector<double> floor_;     // [n]: 0 where the bases do not sum to one on the piece, else -inf
  std::vector<int> first;         // [n]: first coefficient used
  std::vector<double> basis;      // [n][4][4]
  int n() const { return (int)lo.size(); }
};

struct PlanInputs {
  std::vector<std::shared_ptr<PieceTable>> piece_tables;  // keeps SplineGeom::piece_* alive
  std::vector<SplineGeom> geom;  // parallel to plan.dims (sort-key order)
  std::vector<Feat> kop_feats;   // feature columns of the kops, in stream-column order
  std::vector<Feat> static_feats;
  std::vector<RangeCut> cuts;
  std::vector<int> used_cols;
  int key_shift[MAX_SPLINE_DIMS] = {0, 0, 0, 0, 0, 0, 0, 0};
  int key_bits = 0;
};

// sort key of one sample = its piece indices, most pieces = most significant; PLAN_KEY_INVALID = dropped
GWI_HD inline uint64_t sample_key(const double* const* cols, int64_t j, const int* used_cols, int n_used, const RangeCut* cuts, int n_cuts, const SplineGeom* geom,
                                  const int* key_shift, int NS, const Feat* static_feats, int n_static, const Feat* kop_feats, int n_kf, const CosmoView& cv) {
  for (int i = 0; i < n_used; ++i) {
    const double v = cols[used_cols[i]][j];
    if (!(v == v)) return PLAN_KEY_INVALID;
  }
  for (int i = 0; i < n_cuts; ++i)
    if (!pass_cut(cuts[i], cols, j)) return PLAN_KEY_INVALID;
  uint64_t key = 0;
  for (int d = 0; d < NS; ++d) {
    int J;
    double u;
    if (!spline_locate(geom[d], cols[geom[d].col][j], J, u)) return PLAN_KEY_INVALID;
    key |= (uint64_t)J << key_shift[d];
  }
  double st = 0.0;
  for (int i = 0; i < n_static; ++i) st += eval_feat(static_feats[i], cols, j, cv);
  if (!plan_finite(st)) return PLAN_KEY_INVALID;
  for (int i = 0; i < n_kf; ++i)
    if (!plan_finite(eval_feat(kop_feats[i], cols, j, cv))) return PLAN_KEY_INVALID;
  return key;
}

// stages of the plan build (plan.cpp); build_plan = classify -> order (host sort) -> geometry -> fill (host) -> tree,
// build_plan_device (plan_device.cu) replaces the order and fill stages by kernels
int plan_classify(int n_cat_columns, const gwi_model_desc& desc, Plan& plan, PlanInputs& in);
int plan_geometry(const gwi_model_desc& desc, int sm_count, const PlanInputs& in, const std::vector<std::vector<double>>& rate, Plan& plan,
                  std::vector<int64_t>& chunk_r0, std::vector<int64_t>& chunk_nc);
void plan_tree(Plan& plan);
int plan_begin_segments(const CatalogView& cat, Plan& plan);
CosmoView cosmo_view_host();
// plan_device.cu: the order and fill stages as kernels on the catalog's GPU; *d_columns_out = the plan's device array,
// *d_index_out = its sample index (desc.keep_sample_index; nullptr otherwise)
constexpr int PLAN_DEVICE_FALLBACK = 1;  // the model exceeds the device builder's fixed tables: use the host builder
int build_plan_device(const CatalogView& cat, const gwi_model_desc& desc, int sm_count, Plan& plan, uint64_t** d_columns_out, uint32_t** d_index_out,
                      double* stats_seconds);

}  // namespace gwi
