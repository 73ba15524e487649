// Host-side plan builder: turns the borrowed catalog columns + model description into the static
// device-resident evaluation plan.  This replaces the reference's model construction
// (gwinferno/models/bsplines/single.py:35-58 -- masks + dense Cox-de Boor design matrices,
// gwinferno/interpolation.py:128-149) with, per sample and spline dimension, ONE 8-byte word
// (w = u - 1/2 as fp64 with the piece index J in its 6 low mantissa bits) so that the kernel re-creates the 4 non-zero basis weights on
// the fly.  Samples whose population density is identically zero (outside the model masks,
// single.py:54-55,90-92; z > zmax, spline_perturbation.py:368-372; non-finite static weight) are
// dropped here; the Monte-Carlo denominators keep the full sample counts.
//
// Samples of every segment (injection set, each event) are sorted lexicographically by their
// piece indices so that consecutive samples of one GPU lane share polynomial pieces: the kernel
// keeps the per-piece gradient moments in registers and only spills when a piece index changes.
#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <numeric>
#include <thread>

#include "gwi_internal.h"
#include "plan_sample.h"
#include "smem_layout.h"

namespace gwi {

// ---------------------------------------------------------------------------------------------
// cosmology: flat LCDM, Planck15-LVK constants (gwinferno/cosmology.py:19-22), comoving-distance
// table by sequential trapezoid on z = arange(0, 10, 1e-3) (cosmology.py:48-77); dVc/dz with Dc
// linearly interpolated (cosmology.py:95-120) is in plan_sample.h (host + device).
// ---------------------------------------------------------------------------------------------
namespace {
struct Cosmo {
  static constexpr double C_SI = 299792458.0;
  static constexpr double Ho = 67.90 / 1e-3;
  double c_over_Ho;
  std::vector<double> Dc;
  Cosmo() {
    c_over_Ho = C_SI / Ho;
    const int n = (int)std::ceil(10.0 / COSMO_DZ);
    Dc.resize(n);
    const CosmoView v{nullptr, n, c_over_Ho};
    Dc[0] = 0.0;
    for (int i = 0; i + 1 < n; ++i) {
      const double zi = i * COSMO_DZ;  // numpy arange(0, 10, 1e-3): start + i*step
      Dc[i + 1] = Dc[i] + 0.5 * (cosmo_dDcdz(v, zi) + cosmo_dDcdz(v, zi + COSMO_DZ)) * COSMO_DZ;
    }
  }
};
const Cosmo& cosmo() {
  static Cosmo c;
  return c;
}
}  // namespace

CosmoView cosmo_view_host() {
  const Cosmo& c = cosmo();
  return CosmoView{c.Dc.data(), (int)c.Dc.size(), c.c_over_Ho};
}

double log_dvcdz(double z) { return cosmo_log_dvcdz(cosmo_view_host(), z); }

// ---------------------------------------------------------------------------------------------
namespace {

template <class F>
void parallel_for(int64_t n, int n_workers, F&& fn, int64_t min_n = 4096) {
  if (n_workers <= 1 || n < min_n) {
    fn(0, n, 0);
    return;
  }
  std::vector<std::thread> th;
  const int64_t per = (n + n_workers - 1) / n_workers;
  for (int w = 0; w < n_workers; ++w) {
    const int64_t a = w * per, b = std::min<int64_t>(n, a + per);
    if (a >= b) break;
    th.emplace_back([=, &fn] { fn(a, b, w); });
  }
  for (auto& t : th) t.join();
}

// LSD radix sort of (key, index) pairs by the low `bits` bits of the key, 11-bit digits
void radix_sort_pairs(std::vector<uint64_t>& keys, std::vector<uint32_t>& idx, int bits, int n_workers = 1) {
  const size_t n = keys.size();
  if (n < 2) return;
  if (n < 4096) {
    std::vector<uint32_t> perm(n);
    std::iota(perm.begin(), perm.end(), 0u);
    std::stable_sort(perm.begin(), perm.end(), [&](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
    std::vector<uint64_t> k2(n);
    std::vector<uint32_t> i2(n);
    for (size_t i = 0; i < n; ++i) {
      k2[i] = keys[perm[i]];
      i2[i] = idx[perm[i]];
    }
    keys.swap(k2);
    idx.swap(i2);
    return;
  }
  constexpr int RB = 11, NB = 1 << RB;
  std::vector<uint64_t> k2(n);
  std::vector<uint32_t> i2(n);
  // every pass: per-thread histograms of contiguous blocks, one exclusive scan over
  // (bucket, thread), then a stable scatter of every block (the result does not depend on T)
  const int T = (n_workers > 1 && n >= (size_t)1 << 20) ? n_workers : 1;
  const size_t per = (n + T - 1) / T;
  std::vector<size_t> cnt((size_t)T * NB);
  for (int shift = 0; shift < bits; shift += RB) {
    std::fill(cnt.begin(), cnt.end(), 0);
    parallel_for((int64_t)T, T, [&](int64_t ta, int64_t tb, int) {
      for (int64_t t = ta; t < tb; ++t) {
        size_t* c = cnt.data() + (size_t)t * NB;
        const size_t a = (size_t)t * per, b = std::min(n, a + per);
        for (size_t i = a; i < b; ++i) ++c[(keys[i] >> shift) & (NB - 1)];
      }
    }, 1);
    size_t acc = 0;
    for (int b = 0; b < NB; ++b)
      for (int t = 0; t < T; ++t) {
        const size_t c = cnt[(size_t)t * NB + b];
        cnt[(size_t)t * NB + b] = acc;
        acc += c;
      }
    parallel_for((int64_t)T, T, [&](int64_t ta, int64_t tb, int) {
      for (int64_t t = ta; t < tb; ++t) {
        size_t* c = cnt.data() + (size_t)t * NB;
        const size_t a = (size_t)t * per, b = std::min(n, a + per);
        for (size_t i = a; i < b; ++i) {
          const size_t p = c[(keys[i] >> shift) & (NB - 1)]++;
          k2[p] = keys[i];
          i2[p] = idx[i];
        }
      }
    }, 1);
    keys.swap(k2);
    idx.swap(i2);
  }
}

}  // namespace

namespace {
// GWI_PLAN_TIMING=1: print the wall time of every build phase to stderr
struct PlanTimer {
  bool on = std::getenv("GWI_PLAN_TIMING") != nullptr;
  std::chrono::steady_clock::time_point last = std::chrono::steady_clock::now();
  void tick(const char* what) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[gwi plan] %-28s %8.3f s\n", what, std::chrono::duration<double>(now - last).count());
    last = now;
  }
};
}  // namespace

namespace {
// Per-piece polynomial form of the canonical B-spline basis of an explicit knot vector, restating the reference's
// Cox-de Boor recursion (gwinferno/interpolation.py:128-149: M-spline recursion with half-open order-1 indicators and the
// "support shorter than 1e-6 => zero" guard at every level; :268-278: rescaled by (t[i+k]-t[i])/k to canonical
// B-splines) with polynomials in w = u - 1/2 instead of numbers, u = (x - t[m]) / (t[m+1] - t[m]) on the knot span m.
// Pieces = the spans that meet [x0, x1] (bases are zeroed outside the range, interpolation.py:175), clipped to it; a span
// that STARTS at x1 is kept as a piece that only x1 itself falls into (half-open spans).  Where no span covers part of
// the range the piece has no basis (the spline is 0 there).
using Poly = std::array<double, 4>;
struct SpanPoly {
  const double* t;
  int m, n_knots;
  double xa, xb;  // x(w) = xa + xb w on span m
  Poly M(int i, int kk) const {
    Poly z{0.0, 0.0, 0.0, 0.0};
    if (i < 0 || i + kk > n_knots - 1) return z;
    if (t[i + kk] - t[i] < 1e-6) return z;  // interpolation.py:141
    if (kk == 1) {
      if (i == m) z[0] = 1.0 / (t[i + 1] - t[i]);  // :143-146 (on span m only the indicator of [t_m, t_m+1) is 1)
      return z;
    }
    const Poly a = M(i, kk - 1), b = M(i + 1, kk - 1);
    // (x - t_i) a + (t_{i+kk} - x) b   (:148)
    const double a0 = xa - t[i], b0 = t[i + kk] - xa;
    Poly v{0.0, 0.0, 0.0, 0.0};
    for (int n = 0; n < 4; ++n) {
      v[n] += a0 * a[n] + b0 * b[n];
      if (n + 1 < 4) v[n + 1] += xb * a[n] - xb * b[n];
    }
    const double f = (double)kk / ((double)(kk - 1) * (t[i + kk] - t[i]));  // :149
    for (int n = 0; n < 4; ++n) v[n] *= f;
    return v;
  }
};

int build_piece_table(const double* t, int n_knots, int order, int N, double x0, double x1, PieceTable& T) {
  const double NEG_INF = -std::numeric_limits<double>::infinity();
  auto add_piece = [&](double lo, double origin, double inv_h, int first, const double* basis16, double floor_) {
    T.lo.push_back(lo);
    T.origin.push_back(origin);
    T.inv_h.push_back(inv_h);
    T.first.push_back(first);
    T.floor_.push_back(floor_);
    for (int i = 0; i < 16; ++i) T.basis.push_back(basis16 ? basis16[i] : 0.0);
  };
  for (int m = 0; m + 1 < n_knots; ++m)
    if (!(t[m + 1] >= t[m])) return GWI_ERR_INVALID;  // must be non-decreasing (NaN fails too)
  if (t[0] > x0) add_piece(x0, x0, 1.0, 0, nullptr, 0.0);  // below the first knot: every basis is 0
  for (int m = 0; m + 1 < n_knots; ++m) {
    const double h = t[m + 1] - t[m];
    if (!(h > 0.0) || !(t[m + 1] > x0) || !(t[m] <= x1)) continue;
    SpanPoly sp{t, m, n_knots, t[m] + 0.5 * h, h};
    const int first = std::max(0, std::min(m - order + 1, N - 4));
    double B[16] = {0};
    double sum[4] = {0, 0, 0, 0};
    for (int i = std::max(0, m - order + 1); i <= std::min(N - 1, m); ++i) {
      Poly Mi = sp.M(i, order);
      const double scale = (t[i + order] - t[i]) / (double)order;  // :278
      for (int n = 0; n < 4; ++n) {
        B[(i - first) * 4 + n] = scale * Mi[n];
        sum[n] += scale * Mi[n];
      }
    }
    const bool unity = std::fabs(sum[0] - 1.0) < 1e-9 && std::fabs(sum[1]) < 1e-9 && std::fabs(sum[2]) < 1e-9 && std::fabs(sum[3]) < 1e-9;
    add_piece(std::max(t[m], x0), t[m], 1.0 / h, first, B, unity ? NEG_INF : 0.0);
  }
  if (t[n_knots - 1] <= x1) add_piece(t[n_knots - 1], t[n_knots - 1], 1.0, 0, nullptr, 0.0);  // at / beyond the last knot: 0
  if (T.n() == 0 || T.n() > MAX_ROWS - 1) return GWI_ERR_UNSUPPORTED;
  return GWI_OK;
}

}  // namespace

// stage 1 (host, O(model)): terms -> spline dims / per-sample operations / cuts / grids; sort-key layout
int plan_classify(int n_cat_columns, const gwi_model_desc& desc, Plan& plan, PlanInputs& in) {
  if (desc.n_terms <= 0 || !desc.terms || desc.n_params <= 0) {
    set_error("model description needs at least one term and one parameter");
    return GWI_ERR_INVALID;
  }
  plan = Plan();
  plan.keep_index = desc.keep_sample_index != 0;
  plan.n_params = desc.n_params;
  plan.n_terms = desc.n_terms;
  plan.g2 = desc.need_neff_grad != 0;
  auto col_ok = [&](int c) { return c >= 0 && c < n_cat_columns; };
  auto slot_ok = [&](int s, int n) { return s >= 0 && s + n <= desc.n_params; };
  // ---- norm groups --------------------------------------------------------------------------
  for (int g = 0; g < desc.n_groups; ++g) {
    const gwi_norm_group& G = desc.groups[g];
    if (G.n_grid < 2 || !G.log_w) {
      set_error("norm group needs >= 2 grid points and a log_w array");
      return GWI_ERR_INVALID;
    }
    NormGroup ng;
    ng.n_grid = G.n_grid;
    ng.logw_off = (int)plan.grid_pool.size();
    plan.grid_pool.insert(plan.grid_pool.end(), G.log_w, G.log_w + G.n_grid);
    plan.groups.push_back(ng);
  }
  auto add_grid = [&](const gwi_term& t, int& off) -> bool {
    off = -1;
    if (t.norm_group < 0) return true;
    if (t.norm_group >= desc.n_groups || !t.grid) return false;
    off = (int)plan.grid_pool.size();
    const int n = desc.groups[t.norm_group].n_grid;
    plan.grid_pool.insert(plan.grid_pool.end(), t.grid, t.grid + n);
    return true;
  };

  // ---- classify terms -----------------------------------------------------------------------
  in = PlanInputs();
  std::vector<SplineGeom>& geom = in.geom;  // parallel to plan.dims (before ordering)
  std::vector<Feat>& kop_feats = in.kop_feats;
  std::vector<Feat>& static_feats = in.static_feats;
  std::vector<RangeCut>& cuts = in.cuts;
  std::vector<int>& used_cols = in.used_cols;
  auto use_col = [&](int c) {
    if (std::find(used_cols.begin(), used_cols.end(), c) == used_cols.end()) used_cols.push_back(c);
  };
  auto add_feat = [&](int kind, int c0, int c1, double cst) {
    kop_feats.push_back(Feat{kind, {c0, c1}, cst});
    return (int)kop_feats.size() - 1;  // index among kop features (stream column assigned later)
  };
  auto add_kop = [&](int kind, int f0, int f1, int n_gs, const int* slots, const double* cst, int group, int grid_off) -> bool {
    if ((int)plan.kops.size() >= MAX_KOPS || plan.n_gslots + n_gs > MAX_GSLOTS) return false;
    Kop k{};
    k.kind = kind;
    k.col[0] = f0;
    k.col[1] = f1;
    k.gslot = plan.n_gslots;
    k.n_gslots = n_gs;
    for (int i = 0; i < 6; ++i) k.slot[i] = i < n_gs ? slots[i] : -1;
    for (int i = 0; i < 4; ++i) k.cst[i] = cst ? cst[i] : 0.0;
    k.norm_group = group;
    k.grid_off = grid_off;
    plan.n_gslots += n_gs;
    plan.kops.push_back(k);
    return true;
  };

  for (int ti = 0; ti < desc.n_terms; ++ti) {
    const gwi_term& t = desc.terms[ti];
    if (!col_ok(t.col[0])) {
      set_error("term " + std::to_string(ti) + ": bad column index");
      return GWI_ERR_INVALID;
    }
    use_col(t.col[0]);
    bool ok = true;
    switch (t.kind) {
      case GWI_TERM_SPLINE:
      case GWI_TERM_SPLINE_LINEAR: {
        if (t.kind == GWI_TERM_SPLINE_LINEAR && t.outside != GWI_OUTSIDE_DROP) {
          set_error("term " + std::to_string(ti) + ": a spline density must drop the samples outside its range");
          return GWI_ERR_INVALID;
        }
        const bool general = t.knots != nullptr;
        if (t.n_splines < 4 || (!general && t.n_splines - 2 > MAX_ROWS) || !slot_ok(t.slot[0], t.n_splines) || !(t.xi_hi > t.xi_lo)) {
          set_error("term " + std::to_string(ti) + ": bad spline description");
          return GWI_ERR_INVALID;
        }
        if ((int)plan.dims.size() >= MAX_SPLINE_DIMS) {
          set_error("too many spline dimensions");
          return GWI_ERR_UNSUPPORTED;
        }
        std::shared_ptr<PieceTable> table;
        if (general) {
          if (t.order < 1 || t.order > 4 || t.n_knots != t.n_splines + t.order) {
            set_error("term " + std::to_string(ti) + ": an explicit knot vector needs order 1..4 (degree <= 3) and n_knots == n_splines + order");
            return t.order > 4 ? GWI_ERR_UNSUPPORTED : GWI_ERR_INVALID;
          }
          table = std::make_shared<PieceTable>();
          const int rc = build_piece_table(t.knots, t.n_knots, t.order, t.n_splines, t.xi_lo, t.xi_hi, *table);
          if (rc != GWI_OK) {
            set_error("term " + std::to_string(ti) + (rc == GWI_ERR_UNSUPPORTED ? ": more than 61 polynomial pieces inside the range" : ": the knot vector must be non-decreasing"));
            return rc;
          }
          in.piece_tables.push_back(table);
        }
        SplineDim d{};
        d.term = ti;
        d.n_splines = t.n_splines;
        d.rows = general ? table->n() + 1 : t.n_splines - 2;
        d.basis_off = d.first_off = d.floor_off = -1;
        if (general) {
          d.basis_off = (int)plan.grid_pool.size();
          plan.grid_pool.insert(plan.grid_pool.end(), table->basis.begin(), table->basis.end());
          d.first_off = (int)plan.grid_pool.size();
          for (int f : table->first) plan.grid_pool.push_back((double)f);
          d.floor_off = (int)plan.grid_pool.size();
          plan.grid_pool.insert(plan.grid_pool.end(), table->floor_.begin(), table->floor_.end());
        }
        d.slot = t.slot[0];
        d.norm_group = t.norm_group;
        d.outside = t.outside;
        d.liny = t.kind == GWI_TERM_SPLINE_LINEAR ? 1 : 0;
        if (!add_grid(t, d.grid_off)) ok = false;
        plan.dims.push_back(d);
        SplineGeom g{};
        g.col = t.col[0];
        g.logx = t.logx != 0;
        g.outside = t.outside;
        g.x_lo = t.x_lo;
        g.x_hi = t.x_hi;
        g.xi_lo = t.xi_lo;
        g.xi_hi = t.xi_hi;
        g.rows = d.rows;
        g.inv_dxi = (double)(d.rows - 1) / (t.xi_hi - t.xi_lo);
        if (general) {
          g.n_pieces = table->n();
          g.piece_lo = table->lo.data();
          g.piece_origin = table->origin.data();
          g.piece_inv_h = table->inv_h.data();
        }
        geom.push_back(g);
        break;
      }
      case GWI_TERM_LINEAR: {
        if (!slot_ok(t.slot[0], 1)) ok = false;
        int fk = 0;
        switch (t.feature) {
          case GWI_FEAT_LOG1P: fk = F_LOG1P; break;
          case GWI_FEAT_LOG: fk = F_LOG; break;
          case GWI_FEAT_LOG_RATIO: fk = F_LOG_RATIO; break;
          case GWI_FEAT_LOG_DVDZ: fk = F_LOG_DVDZ; break;
          case GWI_FEAT_NEG_LOG: fk = F_NEG_LOG; break;
          case GWI_FEAT_NEG_LOG1P: fk = F_NEG_LOG1P; break;
          default: ok = false;
        }
        if (fk == F_LOG_RATIO) {
          if (!col_ok(t.col[1])) ok = false; else use_col(t.col[1]);
        }
        int goff;
        if (!add_grid(t, goff)) ok = false;
        if (ok) {
          const int f = add_feat(fk, t.col[0], t.col[1], 0.0);
          const double cst[4] = {t.cst[0], 0, 0, 0};
          ok = add_kop(KOP_LIN, f, -1, 1, t.slot, cst, t.norm_group, goff);
        }
        break;
      }
      case GWI_TERM_STATIC: {
        int fk = 0;
        switch (t.feature) {
          case GWI_FEAT_LOG1P: fk = F_LOG1P; break;
          case GWI_FEAT_LOG: fk = F_LOG; break;
          case GWI_FEAT_LOG_RATIO: fk = F_LOG_RATIO; break;
          case GWI_FEAT_LOG_DVDZ: fk = F_LOG_DVDZ; break;
          case GWI_FEAT_NEG_LOG: fk = F_NEG_LOG; break;
          case GWI_FEAT_NEG_LOG1P: fk = F_NEG_LOG1P; break;
          case GWI_FEAT_CONST: fk = F_CONST; break;
          default: ok = false;
        }
        if (fk == F_LOG_RATIO) {
          if (!col_ok(t.col[1])) ok = false; else use_col(t.col[1]);
        }
        if (ok) static_feats.push_back(Feat{fk, {t.col[0], t.col[1]}, t.cst[0]});
        break;
      }
      case GWI_TERM_POWERLAW: {
        if (!slot_ok(t.slot[0], 1) || !(t.cst[0] > 0.0) || !(t.cst[1] > t.cst[0])) ok = false;
        if (ok) {
          const int f = add_feat(F_LOG, t.col[0], -1, 0.0);
          const double cst[4] = {0, 0, 0, 0};
          ok = add_kop(KOP_LIN, f, -1, 1, t.slot, cst, -1, -1);
          if ((int)plan.sops.size() >= MAX_SOPS) ok = false;
          plan.sops.push_back(Sop{SOP_POWERLAW_NORM, {t.slot[0], -1}, {t.cst[0], t.cst[1]}});
          cuts.push_back(RangeCut{1, {t.col[0], -1}, t.cst[0], t.cst[1]});
        }
        break;
      }
      case GWI_TERM_POWERLAW_RATIO: {
        if (!slot_ok(t.slot[0], 1) || !col_ok(t.col[1]) || !(t.cst[0] > 0.0)) ok = false;
        if (ok) {
          use_col(t.col[1]);
          const int f0 = add_feat(F_LOG, t.col[0], -1, 0.0);
          const int f1 = add_feat(F_LOG_C_OVER, t.col[1], -1, t.cst[0]);
          ok = add_kop(KOP_PLRATIO, f0, f1, 1, t.slot, nullptr, -1, -1);
          cuts.push_back(RangeCut{4, {t.col[0], t.col[1]}, t.cst[0], 1.0});
        }
        break;
      }
      case GWI_TERM_PLPEAK: {
        for (int i = 0; i < 4; ++i)
          if (!slot_ok(t.slot[i], 1)) ok = false;
        if (!(t.cst[0] > 0.0) || !(t.cst[1] > t.cst[0])) ok = false;
        const bool tapered = t.slot[4] >= 0;  // delta_m given: PL part x smooth(delta, m1, mmin)
        if (tapered && !slot_ok(t.slot[4], 1)) ok = false;
        if (ok) {
          const int f0 = add_feat(F_LOG, t.col[0], -1, 0.0);
          const int f1 = add_feat(F_RAW, t.col[0], -1, 0.0);
          const double cst[4] = {t.cst[0], t.cst[1], 0, 0};
          ok = add_kop(KOP_PLPEAK, f0, f1, tapered ? 5 : 4, t.slot, cst, -1, -1);
          cuts.push_back(RangeCut{1, {t.col[0], -1}, t.cst[0], t.cst[1]});
        }
        break;
      }
      case GWI_TERM_SMOOTH: {
        if (!slot_ok(t.slot[0], 1)) ok = false;
        const bool prod = t.col[1] >= 0;
        if (prod && !col_ok(t.col[1])) ok = false;
        if (ok) {
          if (prod) use_col(t.col[1]);
          const int f0 = add_feat(prod ? F_PROD_MINUS_C : F_MINUS_C, t.col[0], prod ? t.col[1] : -1, t.cst[0]);
          ok = add_kop(KOP_SMOOTH, f0, -1, 1, t.slot, nullptr, -1, -1);
        }
        break;
      }
      case GWI_TERM_BETA: {
        if (!slot_ok(t.slot[0], 1) || !slot_ok(t.slot[1], 1) || !(t.cst[0] > 0.0)) ok = false;
        if (ok) {
          const int f0 = add_feat(F_LOG, t.col[0], -1, 0.0);
          const int f1 = add_feat(F_LOG_S_MINUS, t.col[0], -1, t.cst[0]);
          const double cst[4] = {-1.0, 0, 0, 0};
          ok = add_kop(KOP_LIN, f0, -1, 1, &t.slot[0], cst, -1, -1) && add_kop(KOP_LIN, f1, -1, 1, &t.slot[1], cst, -1, -1);
          if ((int)plan.sops.size() >= MAX_SOPS) ok = false;
          plan.sops.push_back(Sop{SOP_BETA_NORM, {t.slot[0], t.slot[1]}, {t.cst[0], 0.0}});
          cuts.push_back(RangeCut{3, {t.col[0], -1}, 0.0, t.cst[0]});
        }
        break;
      }
      case GWI_TERM_ISOALIGN: {
        if (!slot_ok(t.slot[0], 1) || !slot_ok(t.slot[1], 1)) ok = false;
        if (ok) {
          const int f0 = add_feat(F_RAW, t.col[0], -1, 0.0);
          ok = add_kop(KOP_ISOALIGN, f0, -1, 2, t.slot, nullptr, -1, -1);
          cuts.push_back(RangeCut{1, {t.col[0], -1}, -1.0, 1.0});
        }
        break;
      }
      case GWI_TERM_ISOALIGN_PAIR: {
        if (!slot_ok(t.slot[0], 1) || !slot_ok(t.slot[1], 1) || !col_ok(t.col[1])) ok = false;
        if (ok) {
          use_col(t.col[1]);
          const int f0 = add_feat(F_RAW, t.col[0], -1, 0.0);
          const int f1 = add_feat(F_RAW, t.col[1], -1, 0.0);
          ok = add_kop(KOP_ISOALIGN2, f0, f1, 2, t.slot, nullptr, -1, -1);
          cuts.push_back(RangeCut{1, {t.col[0], -1}, -1.0, 1.0});
          cuts.push_back(RangeCut{1, {t.col[1], -1}, -1.0, 1.0});
        }
        break;
      }
      case GWI_TERM_TRUNCNORM: {
        if (!slot_ok(t.slot[0], 1) || !slot_ok(t.slot[1], 1) || !(t.cst[1] > t.cst[0])) ok = false;
        if (ok) {
          const int f0 = add_feat(F_RAW, t.col[0], -1, 0.0);
          const double cst[4] = {t.cst[0], t.cst[1], 0, 0};
          ok = add_kop(KOP_QUAD, f0, -1, 2, t.slot, cst, -1, -1);
          if ((int)plan.sops.size() >= MAX_SOPS) ok = false;
          plan.sops.push_back(Sop{SOP_TRUNCNORM_NORM, {t.slot[0], t.slot[1]}, {t.cst[0], t.cst[1]}});
          cuts.push_back(RangeCut{1, {t.col[0], -1}, t.cst[0], t.cst[1]});
        }
        break;
      }
      default:
        ok = false;
    }
    if (!ok) {
      set_error("term " + std::to_string(ti) + ": invalid or unsupported description (kind " + std::to_string(t.kind) + ")");
      return GWI_ERR_INVALID;
    }
  }
  for (int c = 0; c < desc.n_cuts; ++c) {
    const gwi_cut& k = desc.cuts[c];
    if (!col_ok(k.col[0]) || (k.kind == GWI_CUT_RATIO_RANGE && !col_ok(k.col[1])) || (k.kind != GWI_CUT_RANGE && k.kind != GWI_CUT_RATIO_RANGE)) {
      set_error("bad cut description");
      return GWI_ERR_INVALID;
    }
    use_col(k.col[0]);
    if (k.kind == GWI_CUT_RATIO_RANGE) use_col(k.col[1]);
    cuts.push_back(RangeCut{k.kind == GWI_CUT_RANGE ? 1 : 2, {k.col[0], k.col[1]}, k.lo, k.hi});
  }

  // ---- linear terms first (the stream kernel keeps the leading ones in registers) --------------
  {
    std::stable_partition(plan.kops.begin(), plan.kops.end(), [](const Kop& k) { return k.kind == KOP_LIN; });
    int gs = 0;
    plan.n_lin = 0;
    for (auto& k : plan.kops) {
      k.gslot = gs;
      gs += k.n_gslots;
      if (k.kind == KOP_LIN) ++plan.n_lin;
    }
  }

  // a spline density's normaliser is linear in its coefficients: its group holds that term alone
  for (const SplineDim& D : plan.dims) {
    if (!D.liny || D.norm_group < 0) continue;
    int members = 0;
    for (const SplineDim& O : plan.dims) members += O.norm_group == D.norm_group;
    for (const Kop& k : plan.kops) members += k.norm_group == D.norm_group;
    if (members != 1) {
      set_error("the norm group of a SPLINE_LINEAR term must not have other members");
      return GWI_ERR_INVALID;
    }
  }
  // ---- order the spline dims: most pieces first (sort key most significant), deep dims last ----
  const int NS = (int)plan.dims.size();
  {
    std::vector<int> order(NS);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return plan.dims[a].rows > plan.dims[b].rows; });
    std::vector<SplineDim> d2;
    std::vector<SplineGeom> g2;
    for (int i : order) {
      d2.push_back(plan.dims[i]);
      g2.push_back(geom[i]);
    }
    plan.dims.swap(d2);
    geom.swap(g2);
  }
  int row_off = 0;
  for (int d = 0; d < NS; ++d) {
    plan.dims[d].row_off = row_off;
    plan.dims[d].column = d;
    row_off += plan.dims[d].rows;
  }
  plan.rows_total = row_off;
  // ---- static taps of the normalisation grids (the grid never changes between evaluations) ----
  for (int d = 0; d < NS; ++d) {
    SplineDim& D = plan.dims[d];
    D.grid_aux = -1;
    if (D.grid_off < 0) continue;
    const int G = plan.groups[D.norm_group].n_grid;
    const int n = D.n_splines;
    std::vector<double> aux((size_t)G * 5 + 2 * n, 0.0);
    std::vector<int> Jg(G, -1);
    bool monotone = true;
    int lastJ = -1;
    for (int i = 0; i < G; ++i) {
      const double xi = plan.grid_pool[D.grid_off + i];
      if (!(xi == xi)) {
        aux[(size_t)4 * G + i] = -1.0;
        continue;
      }
      int J;
      if (geom[d].n_pieces > 0) {
        // explicit knot vector: the piece of the (clamped) grid coordinate, its 4 tap weights from the per-piece
        // polynomials, and the FIRST coefficient of the piece in the J field
        const SplineGeom& g = geom[d];
        const double xc = std::min(std::max(xi, g.xi_lo), g.xi_hi);
        int lo = 0, hi = g.n_pieces - 1;
        while (lo < hi) {
          const int mid = (lo + hi + 1) >> 1;
          if (g.piece_lo[mid] <= xc) lo = mid; else hi = mid - 1;
        }
        double u = (xc - g.piece_origin[lo]) * g.piece_inv_h[lo];
        u = std::min(std::max(u, 0.0), 1.0);
        const double* b16 = plan.grid_pool.data() + D.basis_off + (size_t)lo * 16;
        const double w = u - 0.5;
        for (int k = 0; k < 4; ++k) aux[(size_t)4 * i + k] = ((b16[k * 4 + 3] * w + b16[k * 4 + 2]) * w + b16[k * 4 + 1]) * w + b16[k * 4 + 0];
        J = (int)plan.grid_pool[D.first_off + lo];
      } else {
        const double t = (xi - geom[d].xi_lo) * geom[d].inv_dxi;
        J = (int)std::floor(t);
        J = std::max(0, std::min(J, D.rows - 2));
        const double u = t - (double)J, omu = 1.0 - u;
        aux[(size_t)4 * i + 0] = omu * omu * omu * (1.0 / 6.0);
        aux[(size_t)4 * i + 1] = (3.0 * u * u * u - 6.0 * u * u + 4.0) * (1.0 / 6.0);
        aux[(size_t)4 * i + 2] = (-3.0 * u * u * u + 3.0 * u * u + 3.0 * u + 1.0) * (1.0 / 6.0);
        aux[(size_t)4 * i + 3] = u * u * u * (1.0 / 6.0);
      }
      aux[(size_t)4 * G + i] = (double)J;
      Jg[i] = J;
      if (J < lastJ) monotone = false;
      lastJ = J;
    }
    for (int k = 0; k < n; ++k) {
      int lo = G, hi = 0;
      if (monotone) {
        for (int i = 0; i < G; ++i)
          if (Jg[i] >= 0 && k - Jg[i] >= 0 && k - Jg[i] <= 3) {
            lo = std::min(lo, i);
            hi = std::max(hi, i + 1);
          }
        if (lo > hi) lo = hi = 0;
      } else {
        lo = 0;
        hi = G;
      }
      aux[(size_t)5 * G + k] = (double)lo;
      aux[(size_t)5 * G + n + k] = (double)hi;
    }
    D.grid_aux = (int)plan.grid_pool.size();
    plan.grid_pool.insert(plan.grid_pool.end(), aux.begin(), aux.end());
  }

  const int NK = (int)kop_feats.size();
  plan.n_columns = NS + NK + 1;
  plan.col_static = NS + NK;
  for (auto& k : plan.kops) {
    k.col[0] = NS + k.col[0];
    if (k.col[1] >= 0) k.col[1] = NS + k.col[1];
  }
  plan.rec_doubles = rec_size(plan.n_gslots, plan.g2, plan.rows_total);

  {
    int sh = 0;
    for (int d = NS - 1; d >= 0; --d) {
      in.key_shift[d] = sh;
      sh += 6;
    }
    in.key_bits = sh;
  }
  return GWI_OK;
}

namespace {
// stage 2, host form: validity + sort key per sample, order-preserving compaction, stable LSD radix sort per segment;
// piece-change rates along the sorted order (sampled)
void plan_order_host(const CatalogView& cat, const PlanInputs& in, int n_workers, Plan& plan, std::vector<std::vector<uint32_t>>& order,
                     std::vector<std::vector<double>>& rate, PlanTimer& tm) {
  const int NS = (int)plan.dims.size();
  const std::vector<SplineGeom>& geom = in.geom;
  const CosmoView cv = cosmo_view_host();
  const int E = cat.n_events;
  const int64_t n_inj = cat.n_inj;
  const int key_bits = in.key_bits;
  constexpr uint64_t INVALID = PLAN_KEY_INVALID;
  auto sample_key_ = [&](const double* const* cols, int64_t j) -> uint64_t {
    return sample_key(cols, j, in.used_cols.data(), (int)in.used_cols.size(), in.cuts.data(), (int)in.cuts.size(), geom.data(), in.key_shift, NS, in.static_feats.data(),
                      (int)in.static_feats.size(), in.kop_feats.data(), (int)in.kop_feats.size(), cv);
  };
  const int n_seg = E + 1;
  order.assign(n_seg, {});
  {
    // injections
    std::vector<uint64_t> keys(n_inj);
    parallel_for(n_inj, n_workers, [&](int64_t a, int64_t b, int) {
      for (int64_t j = a; j < b; ++j) keys[j] = sample_key_(cat.inj_columns.data(), j);
    });
    // compaction of the valid samples, order-preserving: per-block counts, scan, per-block copy
    std::vector<uint64_t> vk;
    std::vector<uint32_t>& vi = order[0];
    {
      const int T = std::max(1, n_workers);
      const int64_t per = (n_inj + T - 1) / T;
      std::vector<int64_t> cnt(T + 1, 0);
      parallel_for((int64_t)T, T, [&](int64_t ta, int64_t tb, int) {
        for (int64_t t = ta; t < tb; ++t) {
          int64_t n = 0;
          for (int64_t j = t * per; j < std::min(n_inj, (t + 1) * per); ++j) n += keys[j] != INVALID;
          cnt[t + 1] = n;
        }
      }, 1);
      for (int t = 0; t < T; ++t) cnt[t + 1] += cnt[t];
      vk.resize(cnt[T]);
      vi.resize(cnt[T]);
      parallel_for((int64_t)T, T, [&](int64_t ta, int64_t tb, int) {
        for (int64_t t = ta; t < tb; ++t) {
          int64_t o = cnt[t];
          for (int64_t j = t * per; j < std::min(n_inj, (t + 1) * per); ++j)
            if (keys[j] != INVALID) {
              vk[o] = keys[j];
              vi[o++] = (uint32_t)j;
            }
        }
      }, 1);
    }
    keys.clear();
    keys.shrink_to_fit();
    tm.tick("injection keys + compaction");
    radix_sort_pairs(vk, vi, key_bits, n_workers);
    tm.tick("injection sort");
    plan.segments[0].n_total = n_inj;
    plan.segments[0].n_valid = (int64_t)vi.size();
  }
  {
    std::atomic<int> next{0};
    auto work = [&]() {
      for (;;) {
        const int e = next.fetch_add(1);
        if (e >= E) break;
        const int64_t a = cat.pe_offsets[e], b = cat.pe_offsets[e + 1];
        std::vector<uint64_t> vk;
        std::vector<uint32_t>& vi = order[e + 1];
        for (int64_t j = a; j < b; ++j) {
          const uint64_t k = sample_key_(cat.pe_columns.data(), j);
          if (k != INVALID) {
            vk.push_back(k);
            vi.push_back((uint32_t)j);
          }
        }
        radix_sort_pairs(vk, vi, key_bits);
        plan.segments[e + 1].n_total = b - a;
        plan.segments[e + 1].n_valid = (int64_t)vi.size();
      }
    };
    std::vector<std::thread> th;
    for (int w = 0; w < std::min(n_workers, std::max(1, E)); ++w) th.emplace_back(work);
    for (auto& t : th) t.join();
  }
  for (int s = 1; s < n_seg; ++s) plan.n_valid_pe += plan.segments[s].n_valid;
  plan.n_valid_inj = plan.segments[0].n_valid;

  tm.tick("event keys + sorts");
  {
    // per segment: fraction of consecutive sorted samples whose piece index differs, per dim
    rate.assign(n_seg, std::vector<double>(NS, 0.0));
    std::atomic<int> next_seg{0};
    auto rate_work = [&]() {
      for (;;) {
        const int s = next_seg.fetch_add(1);
        if (s >= n_seg) break;
        const double* const* cols = s == 0 ? cat.inj_columns.data() : cat.pe_columns.data();
        const std::vector<uint32_t>& ord = order[s];
        const size_t n = ord.size();
        const size_t stride = std::max<size_t>(1, n / 50000);  // sample long segments
        double pairs = 0.0;
        for (size_t i = 0; i + 1 < n; i += stride) {
          for (int d = 0; d < NS; ++d) {
            int J0 = 0, J1 = 0;  // (every sample of the plan is inside the support: spline_locate succeeds)
            double u = 0.0;
            spline_locate(geom[d], cols[geom[d].col][ord[i]], J0, u);
            spline_locate(geom[d], cols[geom[d].col][ord[i + 1]], J1, u);
            if (J0 != J1) rate[s][d] += 1.0;
          }
          pairs += 1.0;
        }
        for (int d = 0; d < NS; ++d) rate[s][d] = pairs > 0 ? rate[s][d] / pairs : 0.0;
      }
    };
    {
      std::vector<std::thread> th;
      for (int w = 0; w < std::min(n_workers, n_seg); ++w) th.emplace_back(rate_work);
      for (auto& t : th) t.join();
    }
  }
}
}  // namespace

// stage 3 (host, O(segments + chunks)): deep dims from the piece-change rates, kernel choice, launch geometry, slices and chunks.
// Needs only plan.segments[s].n_valid and the rates.
int plan_geometry(const gwi_model_desc& desc, int sm_count, const PlanInputs& in, const std::vector<std::vector<double>>& rate, Plan& plan,
                  std::vector<int64_t>& chunk_r0, std::vector<int64_t>& chunk_nc) {
  PlanTimer tm;
  const bool timing = tm.on;
  const int NS = (int)plan.dims.size();
  const int n_seg = (int)plan.segments.size();
  chunk_r0.clear();
  chunk_nc.clear();
  bool want_cta = false;  // the CTA-cooperative stream kernel is the better one for this plan (decided below)
  {
    // cost model (issue slots per sample): a register-resident dim pays the warp-wide spill path
    // whenever ANY of its 32 lanes changes piece (~60 slots incl. the shared-memory atomics); a
    // deep dim pays ~17 extra slots on every sample.  Deep dims must be a suffix of the sort order.
    // Which stream kernel?  Measured on B200 after the one-role kernel's chunk flush became fire-and-forget reductions (r02c17 /
    // r02c18, stream-kernel ms, one-role / CTA-cooperative): cfg3 1.03e8 samples 1.52 / 1.79, 4-way shard (2.6e7) 0.420 / 0.471,
    // cfg5 (2.2e7) 0.434 / 0.462, 8-way shard (1.3e7) 0.237 / 0.256, 16-way (6.4e6) 0.142 / 0.148, 32-way (3.2e6) 0.085 / 0.094,
    // 64-way (1.6e6) 0.062 / 0.052, cfg2 (7.8e5) 0.043 / 0.035, the 1024-chain batch 45.8k / 50.6k chain-evals/s: the
    // CTA-cooperative kernel (no per-warp accumulators to set up and flush, one slice per CTA) wins on SMALL catalogs and
    // on chain batches, the one-role kernel everywhere else.  GWI_CTA_KERNEL=0 / 1 forces the choice.
    {
      int64_t n_valid_all = 0;
      for (int s = 0; s < n_seg; ++s) n_valid_all += plan.segments[s].n_valid;
      want_cta = n_valid_all < 2400000 || desc.batch_hint > 1;
      if (const char* e = std::getenv("GWI_CTA_KERNEL")) want_cta = e[0] != '0';
      bool ok = !plan.g2 && (int)plan.kops.size() == plan.n_lin && plan.n_lin <= 2;
      for (const SplineDim& D : plan.dims) ok = ok && !D.liny;
      want_cta = want_cta && ok;
    }
    // r02 calibration (B200, unified pair path + RED spills + conflict-free deep tables; both kernels are bound by
    // shared-memory wavefronts now): a deep dim costs ~22 slot-equivalents per sample; a register-resident dim costs ~12
    // whenever any lane of the warp changes piece plus ~60 per changing lane.  cfg3: the 5th key (piece change every ~27
    // samples) is better kept in registers (1.573 vs 1.726 ms), the 6th (every ~3 samples) is not.
    // In the CTA-cooperative kernel the deep dims belong to dedicated warps: cheaper (cfg5 0.469 ms with 3 deep dims, 0.522 with 2).
    const double COST_WARP = 12.0, COST_LANE = 60.0, COST_DEEP = want_cta ? 13.0 : 22.0;
    int want = desc.n_deep;
    int nd = 0;
    if (want < 0) {
      double best = -1.0;
      for (int cand = 0; cand <= std::min(NS, 4); ++cand) {
        double cost = 0.0;
        for (int s = 0; s < n_seg; ++s) {
          const double n = (double)plan.segments[s].n_valid;
          for (int d = 0; d < NS - cand; ++d) cost += n * (std::min(1.0, 32.0 * rate[s][d]) * COST_WARP + rate[s][d] * COST_LANE);
          cost += n * cand * COST_DEEP;
        }
        if (timing) {
          double ci = 0.0, cp = 0.0, np_ = 0.0;
          for (int s = 0; s < n_seg; ++s) {
            const double n = (double)plan.segments[s].n_valid;
            double c = cand * COST_DEEP;
            for (int d = 0; d < NS - cand; ++d) c += std::min(1.0, 32.0 * rate[s][d]) * COST_WARP + rate[s][d] * COST_LANE;
            if (s == 0) ci = c; else { cp += n * c; np_ += n; }
          }
          std::fprintf(stderr, "[gwi plan] n_deep=%d: modelled extra issue slots per sample: injections %.1f, events %.1f\n", cand, ci, np_ > 0 ? cp / np_ : 0.0);
        }
        if (best < 0.0 || cost < best) {
          best = cost;
          nd = cand;
        }
      }
    } else {
      nd = want;
    }
    nd = std::min(std::min(nd, NS), 4);
    // shared-memory budget: keep at least 4 warps per CTA
    const int mom_ = plan.g2 ? 2 : 1;
    for (;;) {
      int64_t bytes = (int64_t)plan.rows_total * 4 * mom_ * 8;
      for (int d = NS - nd; d < NS; ++d) bytes += (int64_t)plan.dims[d].rows * 4 * mom_ * DEEP_LANES * 8;
      if (nd == 0 || bytes * 4 <= 200 * 1024) break;
      --nd;
    }
    plan.n_deep = nd;
    for (int d = 0; d < NS; ++d) plan.dims[d].deep = d >= NS - nd;
  }
  // ---- launch geometry + chunking -----------------------------------------------------------
  // the most warps whose exact shared-memory layout (smem_layout.h) fits SMEM_BUDGET, 225 of the 227 KB an sm_100 CTA
  // may use.  The warp counts fix the chunking, hence the summation order: another budget moves results in the last bits.
  constexpr unsigned SMEM_BUDGET = 225 * 1024;
  const int mom = plan.g2 ? 2 : 1;
  int rows_deep = 0;
  for (int d = 0; d < NS; ++d)
    if (plan.dims[d].deep) rows_deep += plan.dims[d].rows;
  int wpb = 8;
  while (wpb > 1 && one_role_smem_bytes(plan.rows_total, rows_deep, mom, (int)plan.kops.size(), plan.n_gslots, wpb) > SMEM_BUDGET) --wpb;
  plan.warps_per_block = wpb;
  plan.grid_blocks = std::max(1, sm_count);
  // CTA-cooperative geometry (stream_cta.cuh) for spline models with at most 2 linear terms and no N_eff
  // gradient: main warps stage their blocks with bulk copies, one dedicated warp per deep dim accumulates
  // that dim's moments for the whole CTA.  GWI_CTA_KERNEL=0 keeps the one-role kernel (tuning / bisection).
  if (want_cta && plan.n_deep >= 1) {
    int nw = CTA_MAX_WARPS - plan.n_deep;
    while (nw >= 2 && cta_layout(nw, plan.n_columns, plan.rows_total, rows_deep).total > SMEM_BUDGET) --nw;
    if (nw >= 2) {
      plan.cta_mode = true;
      plan.cta_main_warps = nw;
    }
  }
  const int LW = plan.cta_mode ? plan.cta_main_warps : 1;  // warps that share a chunk
  const int LPC = LANES * LW;                              // lane runs per chunk
  // gwi_model_desc.batch_hint = n (default 1): the model will be evaluated for ~n chains per launch
  // (gwi_loglike_batch), so the machine is filled by chains and ONE chain only needs W/n warps:
  // slices get n times longer (up to the cap), i.e. fewer record flushes and longer piece-sorted lane
  // runs.  The emulator's path statistics for the config-2 catalog: 2 701 chunks of 8 steps and 88 % of
  // the warp iterations with lanes on the piece-change path at n = 1.
  const int batch_hint = std::max(1, (int)desc.batch_hint);
  plan.batch_hint = batch_hint;
  const int W = plan.cta_mode ? std::max(1, plan.grid_blocks / batch_hint) : std::max(plan.warps_per_block, plan.grid_blocks * plan.warps_per_block / batch_hint);
  // Balanced slicing: the piece-sorted sample stream of all segments (the events first, then the
  // injections) is cut into SLICES of L steps (32 samples per step); slice i belongs to warp i % W.
  // By default L = ceil(total steps / W): every warp gets exactly one slice, i.e. the same amount
  // of work.  A slice is split into CHUNKS at segment boundaries; the lanes of the warp own
  // contiguous sorted runs inside each chunk.  (desc.chunk_steps > 0 caps L: tests use it to force
  // many slices per warp.)
  const int Q = plan.cta_mode ? UNROLL : 2 * UNROLL;  // chunk steps are a multiple of the kernel's load pipeline depth
  auto roundQ = [Q](int64_t v) { return (v + Q - 1) / Q * Q; };
  int64_t total_steps = 0;
  for (int s = 0; s < n_seg; ++s) total_steps += roundQ((plan.segments[s].n_valid + LPC - 1) / LPC);
  // Slices are pulled dynamically by the warps (stream.cuh), so they only need to be small enough
  // for a good tail (>= ~4 per warp when the problem allows) and large enough to amortise the
  // per-chunk record flush and the piece changes at every lane-run start: 64..768 steps
  // (measured optimum 64-128 on a 1.3e7-sample shard; on 1e8 samples 256 -> 2.40 ms, 512 -> 2.34,
  // 768 -> 2.33, 1024 -> 2.32 with the guided shrink below taking care of the tail).
  const int64_t per_warp = (total_steps + W - 1) / W;
  // slices per warp the one-role kernel aims for: 4 on long catalogs, 2 where a warp only has a few hundred steps (an 8-way cfg3
  // shard, 330 steps per warp: 4308 instead of 5764 chunks, step 0.304 -> 0.296 ms; cfg3 itself 1.600 vs 1.624 ms the other way:
  // profiles/r02_call29_slices.txt).
  const int64_t spw = per_warp < 512 ? 2 : 4;
  int64_t L = roundQ(std::max<int64_t>(per_warp < 64 ? 32 : 64, std::min<int64_t>(768, per_warp / spw)));
  L = std::max<int64_t>(L, 8 * Q);
  bool fixed_L = false;  // one slice per CTA: no guided shrink
  if (plan.cta_mode) {
    // a slice is L steps of ALL main warps of a CTA: >= ~4 slices per CTA for the dynamic balance, but never
    // fewer slices than CTAs on a small catalog
    // r02 sweeps (B200, ms/step at div = 1 / 2 / 3 / 4): 8-way cfg3 shard 0.390 / 0.327 / 0.325 / 0.331, cfg5 - / 0.531 / 0.539 / 0.539
    const int64_t div = 2;
    L = roundQ(std::min<int64_t>(768, std::max<int64_t>(16, per_warp / div)));
    if (L > per_warp) L = roundQ(std::max<int64_t>(Q, per_warp));
    // Small catalogs (a few blocks per warp: the kernel is latency, not throughput): every slice costs a counter round trip,
    // a pipeline fill and a record flush, so give every CTA exactly ONE slice -- the shortest L whose slice count still fits
    // the grid (cfg2, 70 events of 18 steps + 2232 injection steps on 148 CTAs: L = 30 -> 145 slices / 145 chunks instead of
    // L = 16 -> 280 chunks, where every event was cut into a 16-step and a 2-step chunk).
    if (per_warp < 64) {
      auto n_slices_for = [&](int64_t Lt) {
        int64_t slices = 1, fill_t = 0;
        for (int si = 0; si < n_seg; ++si) {
          const int sg = (si + 1) % n_seg;
          int64_t left = plan.segments[sg].n_valid;
          bool first = true;
          while (left > 0) {
            const int64_t want = roundQ((left + LPC - 1) / LPC);
            if (Lt - fill_t < Q || (first && fill_t > 0 && want > Lt - fill_t)) {
              ++slices;
              fill_t = 0;
            }
            const int64_t steps = std::min<int64_t>(Lt - fill_t, want);
            left -= std::min<int64_t>(left, steps * LPC);
            fill_t += steps;
            first = false;
          }
        }
        return slices;
      };
      for (int64_t Lt = roundQ(std::max<int64_t>(Q, per_warp)); Lt <= 4 * per_warp + 4 * Q; Lt += Q)
        if (n_slices_for(Lt) <= W) {
          L = Lt;
          fixed_L = true;
          break;
        }
    }
  }
  if (desc.chunk_steps > 0) {  // explicit slice length (tests force tiny slices)
    L = roundQ(desc.chunk_steps);
    fixed_L = false;
  }
  plan.chunk_steps = (int)L;
  plan.slice_begin.clear();
  plan.slice_begin.push_back(0);
  // Guided scheduling: the warps pull slices in order, so the slices shrink towards the end of
  // the stream (guided self-scheduling: slice = remaining work / W, clamped to [L_MIN, L]) to keep
  // the tail short.
  const int64_t L_full = L;
  // one warp step takes ~2500 cycles of latency (8 resident warps/SM), so a 32-step final slice is a
  // 40 us tail; 8-step slices at the very end cut it to ~10 us for ~2W extra record flushes
  // r02 measurements (B200): DIV 1 / LMIN 32 instead of 2 / 8 cut the chunks of an 8-way cfg3 shard from 10 044 to 5 764 and its
  // stream kernel from 0.427 to 0.372 ms, the full catalog from 15 167 to 8 477 chunks and 1.807 to 1.752 ms (fewer record
  // flushes and records to reduce; the tail stays short because the final slices are still small)
  const int64_t L_MIN = fixed_L ? L : roundQ(32);
  const int64_t GUIDED_DIV = 1;  // slice = remaining / (DIV * W)
  int64_t done_steps = 0;
  int64_t pos = 0, fill = 0;
  for (int si = 0; si < n_seg; ++si) {
    // events first, the injection set (segment 0) last: the small final slices of the guided
    // schedule are then cheap injection slices, not spill-heavy PE slices (shorter tail)
    const int s = (si + 1) % n_seg;
    Segment& S = plan.segments[s];
    S.first_chunk = (int)plan.chunks.size();
    int64_t left = S.n_valid, r0 = 0;
    while (left > 0) {

      // slice full -- or a new segment that does not fit into the rest of this slice: start it on a
      // fresh slice instead of fragmenting it (every chunk boundary costs a record flush)
      if (L - fill < Q || (r0 == 0 && fill > 0 && roundQ((left + LPC - 1) / LPC) > L - fill)) {
        plan.slice_begin.push_back((int)plan.chunks.size());
        fill = 0;
        {
          const int64_t remaining = std::max<int64_t>(0, total_steps - done_steps);
          L = std::max<int64_t>(std::min<int64_t>(L_MIN, L_full), std::min<int64_t>(L_full, roundQ(remaining / (GUIDED_DIV * (int64_t)W))));
        }
      }
      const int64_t steps = std::min<int64_t>(L - fill, roundQ((left + LPC - 1) / LPC));
      const int64_t n_c = std::min<int64_t>(left, steps * LPC);
      Chunk c{};
      c.segment = s;
      c.steps = (int)steps;
      c.first = pos;
      plan.chunks.push_back(c);
      chunk_r0.push_back(r0);
      chunk_nc.push_back(n_c);
      pos += steps * LPC;
      fill += steps;
      done_steps += steps;
      left -= n_c;
      r0 += n_c;
    }
    S.n_chunks = (int)plan.chunks.size() - S.first_chunk;
    S.max_static = -std::numeric_limits<double>::infinity();
    for (int k = 0; k < MAX_KOPS; ++k) {
      S.fmin[k] = std::numeric_limits<double>::infinity();
      S.fmax[k] = -std::numeric_limits<double>::infinity();
    }
  }
  plan.slice_begin.push_back((int)plan.chunks.size());
  plan.n_padded = pos;

  return GWI_OK;
}

namespace {
// stage 4, host form: gather the sorted samples chunk by chunk and write the stream columns + per-segment statistics
int plan_fill_host(const CatalogView& cat, const PlanInputs& in, const std::vector<std::vector<uint32_t>>& order, const std::vector<int64_t>& chunk_r0,
                   const std::vector<int64_t>& chunk_nc, int n_workers, Plan& plan, PlanTimer& tm) {
  const bool timing = tm.on;
  const int NS = (int)plan.dims.size();
  const int NK = (int)in.kop_feats.size();
  const int n_chunks = (int)plan.chunks.size();
  const std::vector<SplineGeom>& geom = in.geom;
  const std::vector<Feat>& kop_feats = in.kop_feats;
  const std::vector<Feat>& static_feats = in.static_feats;
  const std::vector<int>& used_cols = in.used_cols;
  const CosmoView cv = cosmo_view_host();
  const int LW = plan.cta_mode ? plan.cta_main_warps : 1;
  const int LPC = LANES * LW;
  // ---- pass 2: fill the stream columns ------------------------------------------------------
  try {
    plan.columns.assign((size_t)plan.n_columns * (size_t)std::max<int64_t>(1, plan.n_padded), 0ull);
    if (plan.keep_index) plan.sample_index.assign((size_t)std::max<int64_t>(1, plan.n_padded), SAMPLE_INDEX_PAD);
  } catch (const std::bad_alloc&) {
    set_error("out of host memory building the plan");
    return GWI_ERR_ALLOC;
  }
  const double NEG_INF = -std::numeric_limits<double>::infinity();
  // stream layout: blocks of 64 consecutive padded samples (one warp iteration: 32 lanes x UNROLL),
  // inside a block the columns follow each other: word(col, p) = [p/64][col][p%64]
  const size_t ncol_ = (size_t)plan.n_columns;
  auto col_index = [ncol_](int col, int64_t p) -> size_t { return ((size_t)(p >> 6) * ncol_ + (size_t)col) * 64 + (size_t)(p & 63); };
  struct SegStat {
    double max_static;
    uint64_t occ[MAX_SPLINE_DIMS];
    double fmin[MAX_KOPS], fmax[MAX_KOPS];
  };
  std::vector<SegStat> cstat(n_chunks);
  std::atomic<int64_t> gather_seconds{0};  // (microseconds, summed over the workers; timing only)
  {
    std::atomic<int> next{0};
    auto work = [&]() {
      // The sorted order gathers from random rows of the caller's columns.  Gather first, in tight
      // loops with nothing but independent loads (many cache/TLB misses in flight), into a
      // chunk-local copy in sorted order; everything below then reads sequentially.
      std::vector<std::vector<double>> gathered(cat.n_columns);
      std::vector<const double*> tcols(cat.n_columns, nullptr);
      double t_gather = 0.0;
      for (;;) {
        const int c = next.fetch_add(1);
        if (c >= n_chunks) break;
        const auto tg0 = std::chrono::steady_clock::now();
        const Chunk& C = plan.chunks[c];
        const int s = C.segment;
        const double* const* src = s == 0 ? cat.inj_columns.data() : cat.pe_columns.data();
        const std::vector<uint32_t>& ord = order[s];
        const int64_t r0 = chunk_r0[c];  // first sorted rank of this chunk
        const int64_t n_c = chunk_nc[c];
        // catalog position = the row in the PE columns (event order), or n_samples_pe + the row in the injection columns
        const uint32_t cat_base = s == 0 ? (uint32_t)plan.n_samples_pe : 0u;
        for (int cc : used_cols) {
          std::vector<double>& g = gathered[cc];
          if ((int64_t)g.size() < n_c) g.resize(n_c);
          const double* sc = src[cc];
          const uint32_t* o = ord.data() + r0;
          double* gp = g.data();
          for (int64_t r = 0; r < n_c; ++r) gp[r] = sc[o[r]];
          tcols[cc] = gp;
        }
        if (timing) t_gather += std::chrono::duration<double>(std::chrono::steady_clock::now() - tg0).count();
        const double* const* cols = tcols.data();
        SegStat st;
        st.max_static = NEG_INF;
        for (int d = 0; d < MAX_SPLINE_DIMS; ++d) st.occ[d] = 0;
        for (int k = 0; k < MAX_KOPS; ++k) {
          st.fmin[k] = std::numeric_limits<double>::infinity();
          st.fmax[k] = -std::numeric_limits<double>::infinity();
        }
        for (int run = 0; run < LPC; ++run) {
          const int lane = run % LANES;
          const int64_t sub = C.first + (int64_t)(run / LANES) * C.steps * LANES;  // sub-chunk of warp run / 32
          for (int k = 0; k < C.steps; ++k) {
            const int64_t r = (int64_t)run * C.steps + k;
            const int64_t p = sub + (int64_t)(k / UNROLL) * (LANES * UNROLL) + lane * UNROLL + (k % UNROLL);
            if (r < n_c) {
              const int64_t j = r;  // row of the chunk-local sorted copy
              if (plan.keep_index) plan.sample_index[p] = cat_base + ord[r0 + r];
              for (int d = 0; d < NS; ++d) {
                int J = 0;
                double u = 0.0;
                spline_locate(geom[d], cols[geom[d].col][j], J, u);
                plan.columns[col_index(d, p)] = pack_word(J, u);
                st.occ[d] |= 1ull << J;
              }
              for (int f = 0; f < NK; ++f) {
                const double v = eval_feat(kop_feats[f], cols, j, cv);
                std::memcpy(&plan.columns[col_index(NS + f, p)], &v, 8);
              }
              double sw = 0.0;
              for (const Feat& f : static_feats) sw += eval_feat(f, cols, j, cv);
              std::memcpy(&plan.columns[col_index(plan.col_static, p)], &sw, 8);
              st.max_static = std::max(st.max_static, sw);
              for (size_t q = 0; q < plan.kops.size(); ++q)
                if (plan.kops[q].kind == KOP_LIN) {
                  double v;
                  std::memcpy(&v, &plan.columns[col_index(plan.kops[q].col[0], p)], 8);
                  st.fmin[q] = std::min(st.fmin[q], v);
                  st.fmax[q] = std::max(st.fmax[q], v);
                }
            } else {
              // lane padding: a copy of the chunk's last valid sample (so every term evaluates to
              // finite values and no piece index changes) with static log-weight -inf => weight 0
              const int64_t j = n_c - 1;
              for (int d = 0; d < NS; ++d) {
                int J = 0;
                double u = 0.0;
                spline_locate(geom[d], cols[geom[d].col][j], J, u);
                plan.columns[col_index(d, p)] = pack_word(J, u);
              }
              for (int f = 0; f < NK; ++f) {
                const double v = eval_feat(kop_feats[f], cols, j, cv);
                std::memcpy(&plan.columns[col_index(NS + f, p)], &v, 8);
              }
              std::memcpy(&plan.columns[col_index(plan.col_static, p)], &NEG_INF, 8);
            }
          }
        }
        cstat[c] = st;
      }
      if (timing) gather_seconds.fetch_add((int64_t)(t_gather * 1e6));
    };
    std::vector<std::thread> th;
    for (int w = 0; w < std::min(n_workers, std::max(1, n_chunks)); ++w) th.emplace_back(work);
    for (auto& t : th) t.join();
  }
  for (int c = 0; c < n_chunks; ++c) {
    Segment& S = plan.segments[plan.chunks[c].segment];
    S.max_static = std::max(S.max_static, cstat[c].max_static);
    for (int d = 0; d < NS; ++d) S.occ[d] |= cstat[c].occ[d];
    for (size_t q = 0; q < plan.kops.size(); ++q) {
      S.fmin[q] = std::min(S.fmin[q], cstat[c].fmin[q]);
      S.fmax[q] = std::max(S.fmax[q], cstat[c].fmax[q]);
    }
  }

  tm.tick("column fill");
  if (timing) std::fprintf(stderr, "[gwi plan]   of which gather (thread-seconds) %8.3f s over %d workers\n", gather_seconds.load() * 1e-6, n_workers);
  return GWI_OK;
}
}  // namespace

// stage 5 (host): level-0 records and the fixed-order reduction tree
void plan_tree(Plan& plan) {
  const int n_chunks = (int)plan.chunks.size();
  const int n_seg = (int)plan.segments.size();
  const int LW = plan.cta_mode ? plan.cta_main_warps : 1;
  // ---- level-0 records: one per chunk (the chunks, hence the records, of a segment are
  //      consecutive); fixed-order tree reduction afterwards
  {
    const int RPC = plan.cta_mode ? LW + 1 : 1;  // records per chunk (CTA mode: one per main warp + the deep warps')
    plan.n_records0 = n_chunks * RPC;
    std::vector<int> cnt(n_seg, 0), first(n_seg, 0);
    for (int c = 0; c < n_chunks; ++c) {
      plan.chunks[c].record_slot = c * RPC;
      cnt[plan.chunks[c].segment] += RPC;
    }
    for (int s = 0; s < n_seg; ++s) first[s] = plan.segments[s].first_chunk * RPC;  // chunks (hence records) of a segment are consecutive
    // reduction tree, fan-in 64: per segment, levels are added only while it has more than LAST = 64 inputs (what
    // finish_kernel sums itself).  A larger fan-in (128 / 256) would bring cfg3's
    // 8477 records down in ONE level instead of two, i.e. one dependent launch less -- measured SLOWER on B200
    // (profiles/r02_call31_reduce_fan.txt: everything-but-the-stream-kernel per evaluation 76.7 us with two levels of 64 against
    // 99-108 us with one level of 128 / 256 on cfg3, 69.6 against 78-83 us on an 8-way shard, 76 against 89-96 us on cfg5:
    // finish_kernel's injection block then sums 34-67 inputs itself, which costs more than the extra launch).  64 it stays.
    constexpr int LAST = 64, FAN = 64;  // FAN: reduce_kernel's fixed fan-in
    std::vector<int> src(n_seg, -1);  // where the segment's current inputs are (-1 = level-0 records)
    for (;;) {
      int max_cnt = 0;
      for (int s = 0; s < n_seg; ++s) max_cnt = std::max(max_cnt, cnt[s]);
      if (max_cnt <= LAST) break;
      const int lvl = (int)plan.levels.size();
      std::vector<ReduceTask> tasks;
      for (int s = 0; s < n_seg; ++s) {
        if (cnt[s] <= LAST) continue;
        const int nt = (cnt[s] + FAN - 1) / FAN;
        const int out0 = (int)tasks.size();
        for (int t = 0; t < nt; ++t) {
          ReduceTask T{};
          T.out_slot = out0 + t;
          T.in_first = first[s] + t * FAN;
          T.in_count = std::min(FAN, cnt[s] - t * FAN);
          T.src = src[s];
          tasks.push_back(T);
        }
        first[s] = out0;
        cnt[s] = nt;
        src[s] = lvl;
      }
      plan.levels.push_back(tasks);
    }
    {
      std::vector<ReduceTask> tasks(n_seg);
      for (int s = 0; s < n_seg; ++s) {
        tasks[s].out_slot = s;
        tasks[s].in_first = first[s];
        tasks[s].in_count = std::max(0, cnt[s]);
        tasks[s].src = src[s];
      }
      plan.levels.push_back(tasks);
    }
  }
}

// segments: 0 = injections, 1..E = events
int plan_begin_segments(const CatalogView& cat, Plan& plan) {
  const int E = cat.n_events;
  const int64_t n_pe = E > 0 ? cat.pe_offsets[E] : 0;
  plan.total_inj = cat.total_inj;
  plan.n_samples_pe = n_pe;
  plan.n_samples_inj = cat.n_inj;
  if (n_pe + cat.n_inj >= (int64_t)0xFFFFFFF0u) {
    set_error("more than 2^32 samples per process are not supported");
    return GWI_ERR_UNSUPPORTED;
  }
  plan.segments.assign(E + 1, Segment{});
  return GWI_OK;
}

// ---------------------------------------------------------------------------------------------
int build_plan(const CatalogView& cat, const gwi_model_desc& desc, int sm_count, int n_workers, Plan& plan) {
  if (cat.on_device) {
    set_error("the host plan builder cannot read device-resident catalog columns");
    return GWI_ERR_INVALID;
  }
  if (n_workers <= 0) n_workers = (int)std::max(1u, std::thread::hardware_concurrency());
  n_workers = std::min(n_workers, 64);
  PlanTimer tm;
  PlanInputs in;
  int rc = plan_classify(cat.n_columns, desc, plan, in);
  if (rc != GWI_OK) return rc;
  rc = plan_begin_segments(cat, plan);
  if (rc != GWI_OK) return rc;
  tm.tick("terms, grids");
  std::vector<std::vector<uint32_t>> order;  // sorted valid sample indices per segment
  std::vector<std::vector<double>> rate;
  plan_order_host(cat, in, n_workers, plan, order, rate, tm);
  tm.tick("piece-change rates");
  std::vector<int64_t> chunk_r0, chunk_nc;  // first sorted rank / valid samples of every chunk
  rc = plan_geometry(desc, sm_count, in, rate, plan, chunk_r0, chunk_nc);
  if (rc != GWI_OK) return rc;
  tm.tick("slicing");
  rc = plan_fill_host(cat, in, order, chunk_r0, chunk_nc, n_workers, plan, tm);
  if (rc != GWI_OK) return rc;
  plan_tree(plan);
  return GWI_OK;
}

}  // namespace gwi
