/*
 * TEST INFRASTRUCTURE ONLY (the oracle) -- never linked into or called by the product path.
 *
 * Plain-C restatement of the reference's hierarchical population likelihood path, straight from the
 * raw sample coordinates: no plan, no sorting, no packing -- per sample, evaluate every term of the
 * model description once, take a running log-sum-exp per segment and scatter the 4-tap gradients
 * directly.
 * It consumes the SAME descriptors as the C-ABI of the product (include/gwi.h: gwi_catalog_desc,
 * gwi_model_desc), so tests hand identical inputs to both.  Independent of oracle/popmodel.py
 * (NumPy) and of gwinferno_b200/csrc (CUDA): a third implementation for three-way agreement, and
 * the multi-threaded CPU baseline of bench.py.
 *
 * Reference lines followed (relative to /root/reference):
 *   uniform cubic B-spline bases      gwinferno/interpolation.py:98-106,128-149,163-175,268-278
 *   projections + grid normalisers    gwinferno/interpolation.py:280-317,335-357,375-407,425-449
 *   1-D models, masks                 gwinferno/models/bsplines/single.py:35-58,77-128
 *   redshift models                   gwinferno/models/spline_perturbation.py:304-372,
 *                                     gwinferno/models/parametric/parametric.py:112-145,
 *                                     gwinferno/models/bsplines/single.py:398-492
 *   parametric densities              gwinferno/distributions.py:16-21,100-162,
 *                                     gwinferno/models/parametric/parametric.py:27-102
 *   dVc/dz                            gwinferno/cosmology.py:48-120 (LVK Planck15 constants :19-22)
 *   per-event / injection reductions  gwinferno/pipeline/analysis.py:50-136
 * Pinning: tests/test_c_oracle.py checks it against every golden vector in tests/golden/ (outputs
 * of the reference's own code) to 1e-12 / 1e-9.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "gwi.h"

#define MAXD 8 /* derivative entries one term can produce per sample */

/* ---------------------------------------------------------------- cosmology (cosmology.py:48-120) */
#define NZ 10000
static double g_Dc[NZ];
static int g_cosmo_ready = 0;
static pthread_mutex_t g_cosmo_lock = PTHREAD_MUTEX_INITIALIZER;
static const double C_OVER_HO = 299792458.0 / (67.90 / 1e-3), OM = 0.3065, OL = 1.0 - 0.3065, DZ = 1e-3;

static double dDcdz(double z) {
  const double opz = 1.0 + z;
  return C_OVER_HO / sqrt(OL + OM * opz * opz * opz);
}
static void cosmo_init(void) {
  pthread_mutex_lock(&g_cosmo_lock);
  if (!g_cosmo_ready) {
    g_Dc[0] = 0.0;
    for (int i = 1; i < NZ; ++i) {
      const double zl = (i - 1) * DZ; /* np.arange(0, 10, 1e-3)[i-1] */
      g_Dc[i] = g_Dc[i - 1] + 0.5 * (dDcdz(zl) + dDcdz(zl + DZ)) * DZ;
    }
    g_cosmo_ready = 1;
  }
  pthread_mutex_unlock(&g_cosmo_lock);
}
static double dVcdz(double z) { /* linear interpolation of Dc on the table, clamped like np.interp */
  double Dc;
  if (!(z > 0.0)) Dc = g_Dc[0];
  else if (z >= (NZ - 1) * DZ) Dc = g_Dc[NZ - 1];
  else {
    int i = (int)floor(z / DZ);
    if (i > NZ - 2) i = NZ - 2;
    while (i > 0 && i * DZ > z) --i;
    while (i < NZ - 2 && (i + 1) * DZ <= z) ++i;
    const double z0 = i * DZ, z1 = (i + 1) * DZ;
    Dc = g_Dc[i] + (g_Dc[i + 1] - g_Dc[i]) * ((z - z0) / (z1 - z0));
  }
  return 4.0 * M_PI * Dc * Dc * dDcdz(z);
}

/* ---------------------------------------------------------------- small special functions */
static double digamma(double x) {
  double r = 0.0;
  while (x < 10.0) {
    r -= 1.0 / x;
    x += 1.0;
  }
  const double f = 1.0 / (x * x);
  const double t = f * (-1.0 / 12.0 + f * (1.0 / 120.0 + f * (-1.0 / 252.0 + f * (1.0 / 240.0 + f * (-1.0 / 132.0 + f * (691.0 / 32760.0 + f * (-1.0 / 12.0)))))));
  return r + log(x) - 0.5 / x + t;
}
static double phi(double x) { return exp(-0.5 * x * x) / sqrt(2.0 * M_PI); }

/* Phi(b) - Phi(a), formed where it keeps its relative accuracy: a series for an interval narrow against the curvature
 * of phi (2h phi(m) sum_k He_2k(m) h^2k / (2k+1)!, half-width h, midpoint m), the difference of erfc when both bounds
 * lie in one tail, else the difference of erf */
static double normal_interval(double lo, double hi, double mu, double sig) {
  const double a = (lo - mu) / sig, b = (hi - mu) / sig;
  const double h = 0.5 * (hi - lo) / sig, m = (0.5 * (lo + hi) - mu) / sig;
  if (h * fmax(fabs(m), 1.0) < 0.01) {
    const double m2 = m * m, h2 = h * h;
    return 2.0 * h * phi(m) * (1.0 + h2 * ((m2 - 1.0) / 6.0 + h2 * ((m2 * (m2 - 6.0) + 3.0) / 120.0 + h2 * (((m2 - 15.0) * m2 + 45.0) * m2 - 15.0) / 5040.0)));
  }
  if (a >= 0.0) return 0.5 * (erfc(a / M_SQRT2) - erfc(b / M_SQRT2));
  if (b <= 0.0) return 0.5 * (erfc(-b / M_SQRT2) - erfc(-a / M_SQRT2));
  return 0.5 * (erf(b / M_SQRT2) - erf(a / M_SQRT2));
}
/* log truncnorm_pdf and its (mu, sigma) derivatives (distributions.py:122-143) */
static double truncnorm_logpdf(double x, double mu, double sig, double lo, double hi, double* dmu, double* dsig) {
  const double a = (lo - mu) / sig, b = (hi - mu) / sig;
  const double D = normal_interval(lo, hi, mu, sig);
  const double dD_dmu = (-phi(b) + phi(a)) / sig, dD_dsig = (-b * phi(b) + a * phi(a)) / sig;
  *dmu = (x - mu) / (sig * sig) - dD_dmu / D;
  *dsig = (x - mu) * (x - mu) / (sig * sig * sig) - 1.0 / sig - dD_dsig / D;
  return -(x - mu) * (x - mu) / (2.0 * sig * sig) - log(sig) - 0.5 * log(2.0 * M_PI) - log(D);
}
/* log of the power-law normalisation and d/dalpha (distributions.py:111-116), without the difference of powers that
 * cancels near alpha = -1: with L = log(hi/lo) and z = (1+alpha) L the integral is lo^(1+alpha) L expm1(z)/z, and
 * d/dalpha = -log lo - L g(z), g(z) = 1/(1 - e^-z) - 1/z (its series below |z| = 0.1) */
static double powerlaw_lognorm(double alpha, double lo, double hi, double* d) {
  const double a1 = 1.0 + alpha, loglo = log(lo), L = log(hi / lo), z = a1 * L, em1 = expm1(z), z2 = z * z;
  const double g = fabs(z) < 0.1 ? 0.5 + z * (1.0 / 12.0 + z2 * (-1.0 / 720.0 + z2 * (1.0 / 30240.0 - z2 / 1209600.0)))
                                 : 1.0 + 1.0 / em1 - 1.0 / z;
  *d = -loglo - L * g;
  return -a1 * loglo - log(z != 0.0 ? L * (em1 / z) : L);
}
/* the low-mass window as the reference evaluates it (distributions.py:16-21): its second where()
 * condition is always true, so the result is 1/(1 + exp(d/y + d/(y-d))) for every y = x - xmin */
static double smooth_window(double d, double y, double* dlog) {
  const double t = d / y + d / (y - d);
  const double win = 1.0 / (1.0 + exp(t));
  *dlog = win > 0.0 ? -(1.0 - win) * (1.0 / y + y / ((y - d) * (y - d))) : 0.0;
  return win;
}

/* ---------------------------------------------------------------- features and splines */
static double feature(const gwi_term* t, const double* const* cols, int64_t j) {
  const double a = cols[t->col[0]][j];
  switch (t->feature) {
    case GWI_FEAT_LOG1P: return log(1.0 + a);
    case GWI_FEAT_LOG: return log(a);
    case GWI_FEAT_LOG_RATIO: return log(a / cols[t->col[1]][j]);
    case GWI_FEAT_LOG_DVDZ: return log(dVcdz(a));
    case GWI_FEAT_NEG_LOG: return -log(a);
    case GWI_FEAT_NEG_LOG1P: return -log(1.0 + a);
    case GWI_FEAT_CONST: return t->cst[0];
  }
  return NAN;
}
/* M-spline basis i of order k at x on an explicit knot vector: the reference's recursion, number for number
 * (gwinferno/interpolation.py:128-149: support shorter than 1e-6 => 0; order 1 = half-open indicator / width) */
static double mspline(const double* t, int i, int k, double x) {
  if (t[i + k] - t[i] < 1e-6) return 0.0;
  if (k == 1) return (x >= t[i] && x < t[i + 1]) ? 1.0 / (t[i + 1] - t[i]) : 0.0;
  const double v = (x - t[i]) * mspline(t, i, k - 1, x) + (t[i + k] - x) * mspline(t, i + 1, k - 1, x);
  return (v * k) / ((k - 1) * (t[i + k] - t[i]));
}
/* first tap index and the 4 tap weights of the basis at spline coordinate xi (clamped to the range):
 * explicit knot vector (gwi_term.knots; canonical B-splines = M-splines x (t[i+k]-t[i])/k, interpolation.py:278),
 * else the closed form of the default uniform cubic basis */
static int spline_taps(const gwi_term* t, double xi, double w[4]) {
  if (t->knots) {
    const double* kn = t->knots;
    const int k = t->order, N = t->n_splines;
    if (xi < t->xi_lo) xi = t->xi_lo;
    if (xi > t->xi_hi) xi = t->xi_hi;
    int m = -1; /* last knot <= xi */
    for (int q = 0; q < t->n_knots; ++q)
      if (kn[q] <= xi) m = q;
    int j = m - k + 1;
    if (j > N - 4) j = N - 4;
    if (j < 0) j = 0;
    for (int q = 0; q < 4; ++q) w[q] = (kn[j + q + k] - kn[j + q]) / k * mspline(kn, j + q, k, xi);
    return j;
  }
  const int n_int = t->n_splines - 2;
  const double dx = (t->xi_hi - t->xi_lo) / (n_int - 1);
  if (xi < t->xi_lo) xi = t->xi_lo;
  if (xi > t->xi_hi) xi = t->xi_hi;
  const double tt = (xi - t->xi_lo) / dx;
  int j = (int)floor(tt);
  if (j < 0) j = 0;
  if (j > n_int - 2) j = n_int - 2;
  const double u = tt - j, omu = 1.0 - u;
  w[0] = omu * omu * omu / 6.0;
  w[1] = (3.0 * u * u * u - 6.0 * u * u + 4.0) / 6.0;
  w[2] = (-3.0 * u * u * u + 3.0 * u * u + 3.0 * u + 1.0) / 6.0;
  w[3] = u * u * u / 6.0;
  return j;
}

/* One term at one sample: returns its log-density contribution (NAN/-inf = the sample has zero weight)
 * and up to MAXD derivative entries (slot, d f / d Lambda[slot]). */
static double term_eval(const gwi_term* t, const double* const* cols, int64_t j, const double* L, int* nd, int* ds, double* dv) {
  *nd = 0;
  const double x = cols[t->col[0]][j];
  switch (t->kind) {
    case GWI_TERM_SPLINE:
    case GWI_TERM_SPLINE_LINEAR: {
      const int in = x >= t->x_lo && x <= t->x_hi; /* model mask on the raw coordinate (single.py:54-55) */
      if (!in) return t->outside == GWI_OUTSIDE_DROP ? -INFINITY : 0.0;
      double w[4];
      const int J = spline_taps(t, t->logx ? log(x) : x, w);
      const double* c = L + t->slot[0] + J;
      const double s = w[0] * c[0] + w[1] * c[1] + w[2] * c[2] + w[3] * c[3];
      if (t->kind == GWI_TERM_SPLINE) {
        for (int k = 0; k < 4; ++k) { ds[k] = t->slot[0] + J + k; dv[k] = w[k]; }
        *nd = 4;
        return s;
      }
      if (!(s > 0.0)) return -INFINITY; /* the spline IS the density (interpolation.py:293-317) */
      for (int k = 0; k < 4; ++k) { ds[k] = t->slot[0] + J + k; dv[k] = w[k] / s; }
      *nd = 4;
      return log(s);
    }
    case GWI_TERM_LINEAR: {
      const double F = feature(t, cols, j);
      if (!isfinite(F)) return -INFINITY;
      ds[0] = t->slot[0]; dv[0] = F; *nd = 1;
      return (L[t->slot[0]] + t->cst[0]) * F;
    }
    case GWI_TERM_STATIC: {
      const double F = feature(t, cols, j);
      return isfinite(F) ? F : -INFINITY;
    }
    case GWI_TERM_POWERLAW: {
      const double lo = t->cst[0], hi = t->cst[1];
      if (!(x >= lo && x <= hi)) return -INFINITY;
      double dn;
      const double ln = powerlaw_lognorm(L[t->slot[0]], lo, hi, &dn);
      ds[0] = t->slot[0]; dv[0] = log(x) + dn; *nd = 1;
      return L[t->slot[0]] * log(x) + ln;
    }
    case GWI_TERM_POWERLAW_RATIO: {
      const double lo = t->cst[0] / cols[t->col[1]][j];
      if (!(x >= lo && x <= 1.0 && lo < 1.0)) return -INFINITY;
      double dn;
      const double ln = powerlaw_lognorm(L[t->slot[0]], lo, 1.0, &dn);
      ds[0] = t->slot[0]; dv[0] = log(x) + dn; *nd = 1;
      return L[t->slot[0]] * log(x) + ln;
    }
    case GWI_TERM_PLPEAK: {
      const double lo = t->cst[0], hi = t->cst[1];
      if (!(x >= lo && x <= hi)) return -INFINITY;
      const double alpha = L[t->slot[0]], mpp = L[t->slot[1]], sig = L[t->slot[2]], lam = L[t->slot[3]];
      double dn, dmu, dsig, dwin = 0.0;
      const double ln = powerlaw_lognorm(alpha, lo, hi, &dn);
      double PL = exp(alpha * log(x) + ln);
      const double TN = exp(truncnorm_logpdf(x, mpp, sig, lo, hi, &dmu, &dsig));
      if (t->slot[4] >= 0) PL *= smooth_window(L[t->slot[4]], x - lo, &dwin); /* parametric.py:52-53 */
      const double A = (1.0 - lam) * PL, B = lam * TN, tot = A + B;
      if (!(tot > 0.0)) return -INFINITY;
      ds[0] = t->slot[0]; dv[0] = A * (log(x) + dn) / tot;
      ds[1] = t->slot[1]; dv[1] = B * dmu / tot;
      ds[2] = t->slot[2]; dv[2] = B * dsig / tot;
      ds[3] = t->slot[3]; dv[3] = (TN - PL) / tot;
      *nd = 4;
      if (t->slot[4] >= 0) { ds[4] = t->slot[4]; dv[4] = A * dwin / tot; *nd = 5; }
      return log(tot);
    }
    case GWI_TERM_BETA: {
      const double s = t->cst[0], a = L[t->slot[0]], b = L[t->slot[1]];
      if (!(x > 0.0 && x < s)) return -INFINITY;
      const double l1 = log(x), l2 = log(s - x), ls = log(s), pab = digamma(a + b);
      ds[0] = t->slot[0]; dv[0] = l1 - ls - (digamma(a) - pab);
      ds[1] = t->slot[1]; dv[1] = l2 - ls - (digamma(b) - pab);
      *nd = 2;
      return (a - 1.0) * l1 + (b - 1.0) * l2 - (a + b - 1.0) * ls - (lgamma(a) + lgamma(b) - lgamma(a + b));
    }
    case GWI_TERM_ISOALIGN: {
      if (!(x >= -1.0 && x <= 1.0)) return -INFINITY;
      const double xi = L[t->slot[0]], sg = L[t->slot[1]];
      double dmu, dsig;
      const double TN = exp(truncnorm_logpdf(x, 1.0, sg, -1.0, 1.0, &dmu, &dsig));
      const double B = xi * TN, tot = (1.0 - xi) / 2.0 + B;
      ds[0] = t->slot[0]; dv[0] = (TN - 0.5) / tot;
      ds[1] = t->slot[1]; dv[1] = B * dsig / tot;
      *nd = 2;
      return log(tot);
    }
    case GWI_TERM_ISOALIGN_PAIR: {
      const double x2 = cols[t->col[1]][j];
      if (!(x >= -1.0 && x <= 1.0 && x2 >= -1.0 && x2 <= 1.0)) return -INFINITY;
      const double xi = L[t->slot[0]], sg = L[t->slot[1]];
      double dmu, d1, d2;
      const double TN = exp(truncnorm_logpdf(x, 1.0, sg, -1.0, 1.0, &dmu, &d1) + truncnorm_logpdf(x2, 1.0, sg, -1.0, 1.0, &dmu, &d2));
      const double B = xi * TN, tot = (1.0 - xi) / 4.0 + B;
      ds[0] = t->slot[0]; dv[0] = (TN - 0.25) / tot;
      ds[1] = t->slot[1]; dv[1] = B * (d1 + d2) / tot;
      *nd = 2;
      return log(tot);
    }
    case GWI_TERM_TRUNCNORM: {
      const double lo = t->cst[0], hi = t->cst[1];
      if (!(x >= lo && x <= hi)) return -INFINITY;
      double dmu, dsig;
      const double f = truncnorm_logpdf(x, L[t->slot[0]], L[t->slot[1]], lo, hi, &dmu, &dsig);
      ds[0] = t->slot[0]; dv[0] = dmu;
      ds[1] = t->slot[1]; dv[1] = dsig;
      *nd = 2;
      return f;
    }
    case GWI_TERM_SMOOTH: {
      const double xx = t->col[1] >= 0 ? x * cols[t->col[1]][j] : x;
      double dwin;
      const double win = smooth_window(L[t->slot[0]], xx - t->cst[0], &dwin);
      if (!(win > 0.0)) return -INFINITY;
      ds[0] = t->slot[0]; dv[0] = dwin; *nd = 1;
      return log(win);
    }
  }
  return NAN;
}

static int cuts_pass(const gwi_model_desc* m, const double* const* cols, int64_t j) {
  for (int c = 0; c < m->n_cuts; ++c) {
    const gwi_cut* q = &m->cuts[c];
    double v = cols[q->col[0]][j];
    if (q->kind == GWI_CUT_RATIO_RANGE) v = v / cols[q->col[1]][j];
    if (!(v >= q->lo && v <= q->hi)) return 0;
  }
  return 1;
}

/* log-weight of one sample (-inf = zero weight) and its derivative entries (slot, dx/dLambda[slot]) */
static double sample_logw(const gwi_model_desc* m, const double* const* cols, int64_t j, const double* L, int* ne, int* es, double* ev) {
  *ne = 0;
  if (!cuts_pass(m, cols, j)) return -INFINITY;
  double x = 0.0;
  int n = 0;
  for (int k = 0; k < m->n_terms; ++k) {
    int nd;
    const double f = term_eval(&m->terms[k], cols, j, L, &nd, es + n, ev + n);
    if (!isfinite(f)) return -INFINITY;
    x += f;
    n += nd;
  }
  *ne = n;
  return isfinite(x) ? x : -INFINITY;
}

/* ---------------------------------------------------------------- grid normalisers */
static void normalisers(const gwi_model_desc* m, const double* L, double* logZ, double* dlogZ /* [G*P] */) {
  const int P = m->n_params;
  for (int g = 0; g < m->n_groups; ++g) {
    const int G = m->groups[g].n_grid;
    double* li = (double*)malloc(sizeof(double) * G);
    double* dz = dlogZ + (size_t)g * P;
    memset(dz, 0, sizeof(double) * P);
    int liny = 0;
    for (int k = 0; k < m->n_terms; ++k)
      if (m->terms[k].norm_group == g && m->terms[k].kind == GWI_TERM_SPLINE_LINEAR) liny = 1;
    if (liny) { /* BSpline.norm (interpolation.py:280-291): Z = trapezoid(sum_k B_k c_k), linear in c */
      double Z = 0.0;
      double* a = (double*)calloc(P, sizeof(double));
      for (int k = 0; k < m->n_terms; ++k) {
        const gwi_term* t = &m->terms[k];
        if (t->norm_group != g) continue;
        for (int i = 0; i < G; ++i) {
          if (!(t->grid[i] == t->grid[i]) || !isfinite(m->groups[g].log_w[i])) continue;
          double w[4];
          const int J = spline_taps(t, t->grid[i], w);
          const double wq = exp(m->groups[g].log_w[i]);
          for (int q = 0; q < 4; ++q) a[t->slot[0] + J + q] += wq * w[q];
        }
      }
      for (int i = 0; i < P; ++i) Z += a[i] * L[i];
      logZ[g] = log(Z);
      for (int i = 0; i < P; ++i) dz[i] = a[i] / Z;
      free(a);
      free(li);
      continue;
    }
    for (int i = 0; i < G; ++i) li[i] = m->groups[g].log_w[i];
    for (int k = 0; k < m->n_terms; ++k) {
      const gwi_term* t = &m->terms[k];
      if (t->norm_group != g) continue;
      for (int i = 0; i < G; ++i) {
        if (t->kind == GWI_TERM_SPLINE) {
          if (!(t->grid[i] == t->grid[i])) continue; /* NaN: outside the basis range, contributes 0 */
          double w[4];
          const int J = spline_taps(t, t->grid[i], w);
          const double* c = L + t->slot[0] + J;
          li[i] += w[0] * c[0] + w[1] * c[1] + w[2] * c[2] + w[3] * c[3];
        } else if (t->kind == GWI_TERM_LINEAR) {
          li[i] += (L[t->slot[0]] + t->cst[0]) * t->grid[i];
        }
      }
    }
    double mx = -INFINITY, S = 0.0;
    for (int i = 0; i < G; ++i) mx = fmax(mx, li[i]);
    for (int i = 0; i < G; ++i) {
      li[i] = exp(li[i] - mx);
      S += li[i];
    }
    logZ[g] = mx + log(S);
    for (int k = 0; k < m->n_terms; ++k) {
      const gwi_term* t = &m->terms[k];
      if (t->norm_group != g) continue;
      for (int i = 0; i < G; ++i) {
        if (t->kind == GWI_TERM_SPLINE) {
          if (!(t->grid[i] == t->grid[i])) continue;
          double w[4];
          const int J = spline_taps(t, t->grid[i], w);
          for (int q = 0; q < 4; ++q) dz[t->slot[0] + J + q] += li[i] / S * w[q];
        } else if (t->kind == GWI_TERM_LINEAR) {
          dz[t->slot[0]] += li[i] / S * t->grid[i];
        }
      }
    }
    free(li);
  }
}

/* ---------------------------------------------------------------- segments */
typedef struct {
  double m, S1, S2; /* running maximum and sums of e^{x-m}, e^{2(x-m)} */
  double *G1, *G2;  /* [P] sum e^{x-m} dx, sum e^{2(x-m)} dx */
} SegSums;

static void sums_rescale(SegSums* s, double new_max, int P, int want_jac) {
  if (!(new_max > s->m)) return;
  const double f = s->m > -INFINITY ? exp(s->m - new_max) : 0.0;
  s->S1 *= f;
  s->S2 *= f * f;
  if (want_jac)
    for (int i = 0; i < P; ++i) {
      s->G1[i] *= f;
      s->G2[i] *= f * f;
    }
  s->m = new_max;
}

/* One pass over samples [a, b) in tiles: evaluate every term once per sample, then accumulate the tile
 * relative to the running maximum (log-sum-exp with rescaling when the maximum grows). */
#define TILE 512
static void block_sums(const gwi_model_desc* md, const double* const* cols, int64_t a, int64_t b, const double* L, int want_jac, SegSums* out) {
  const int P = md->n_params, cap = md->n_terms * MAXD;
  double* x = (double*)malloc(sizeof(double) * TILE);
  int* ne = (int*)malloc(sizeof(int) * TILE);
  int* es = (int*)malloc(sizeof(int) * (size_t)TILE * cap);
  double* ev = (double*)malloc(sizeof(double) * (size_t)TILE * cap);
  out->m = -INFINITY;
  out->S1 = out->S2 = 0.0;
  for (int64_t t0 = a; t0 < b; t0 += TILE) {
    const int n = (int)((b - t0 < TILE) ? b - t0 : TILE);
    double tmax = -INFINITY;
    for (int i = 0; i < n; ++i) {
      x[i] = sample_logw(md, cols, t0 + i, L, &ne[i], es + (size_t)i * cap, ev + (size_t)i * cap);
      tmax = fmax(tmax, x[i]);
    }
    if (!(tmax > -INFINITY)) continue;
    sums_rescale(out, tmax, P, want_jac);
    for (int i = 0; i < n; ++i) {
      if (!(x[i] > -INFINITY)) continue;
      const double p = exp(x[i] - out->m), p2 = p * p;
      out->S1 += p;
      out->S2 += p2;
      if (want_jac == 1)
        for (int k = 0; k < ne[i]; ++k) out->G1[es[(size_t)i * cap + k]] += p * ev[(size_t)i * cap + k];
      else if (want_jac)
        for (int k = 0; k < ne[i]; ++k) {
          out->G1[es[(size_t)i * cap + k]] += p * ev[(size_t)i * cap + k];
          out->G2[es[(size_t)i * cap + k]] += p2 * ev[(size_t)i * cap + k];
        }
    }
  }
  free(x);
  free(ne);
  free(es);
  free(ev);
}

typedef struct {
  const gwi_catalog_desc* cat;
  const gwi_model_desc* md;
  const double* L;
  int want_jac, n_threads, tid;
  /* events: dynamic assignment */
  int* next_event;
  pthread_mutex_t* lock;
  double *logBF, *logNeff, *J_logBF, *J_logNeff;
  double sumZ;
  const double* dsumZ;
  /* injections: block [a, b) */
  int64_t a, b;
  SegSums sums;
} Work;

static void* events_worker(void* arg) {
  Work* w = (Work*)arg;
  const int P = w->md->n_params, E = w->cat->n_events;
  double* G1 = (double*)malloc(sizeof(double) * P);
  double* G2 = (double*)malloc(sizeof(double) * P);
  for (;;) {
    pthread_mutex_lock(w->lock);
    const int e = (*w->next_event)++;
    pthread_mutex_unlock(w->lock);
    if (e >= E) break;
    const int64_t a = w->cat->pe_offsets[e], b = w->cat->pe_offsets[e + 1];
    memset(G1, 0, sizeof(double) * P);
    memset(G2, 0, sizeof(double) * P);
    SegSums s = {0, 0, 0, G1, G2};
    block_sums(w->md, w->cat->pe_columns, a, b, w->L, w->want_jac, &s);
    if (!(s.m > -INFINITY)) {
      w->logBF[e] = -INFINITY;
      w->logNeff[e] = NAN;
      if (w->want_jac) {
        memset(w->J_logBF + (size_t)e * P, 0, sizeof(double) * P);
        if (w->J_logNeff) memset(w->J_logNeff + (size_t)e * P, 0, sizeof(double) * P);
      }
      continue;
    }
    /* analysis.py:50-88 */
    w->logBF[e] = s.m + log(s.S1) - log((double)(b - a)) - w->sumZ;
    w->logNeff[e] = 2.0 * log(s.S1) - log(s.S2);
    if (w->want_jac)
      for (int i = 0; i < P; ++i) {
        w->J_logBF[(size_t)e * P + i] = G1[i] / s.S1 - w->dsumZ[i];
        if (w->J_logNeff) w->J_logNeff[(size_t)e * P + i] = 2.0 * G1[i] / s.S1 - 2.0 * G2[i] / s.S2;
      }
  }
  free(G1);
  free(G2);
  return NULL;
}

static void* inj_worker(void* arg) {
  Work* w = (Work*)arg;
  block_sums(w->md, w->cat->inj_columns, w->a, w->b, w->L, w->want_jac, &w->sums);
  return NULL;
}

/* Forward + Jacobians of the hot path.  Any output pointer may be NULL; the Jacobians are computed
 * when J_log_mu != NULL (the N_eff Jacobians only if one of their pointers is given).  Returns 0, or -1 on a bad argument / allocation failure. */
int gwio_evaluate(const gwi_catalog_desc* cat, const gwi_model_desc* md, const double* lam, int n_threads, double* logBF, double* logNeff, double* log_mu,
                  double* logNeff_inj, double* J_logBF, double* J_logNeff, double* J_log_mu, double* J_logNeff_inj, double* logZ_out) {
  if (!cat || !md || !lam || n_threads < 1) return -1;
  cosmo_init();
  const int P = md->n_params, E = cat->n_events, T = n_threads;
  /* 0: values only; 1: first-order sums (J_logBF, J_log_mu); 2: also the N_eff Jacobians */
  const int want_jac = J_log_mu == NULL ? 0 : ((J_logNeff || J_logNeff_inj) ? 2 : 1);
  double* logZ = (double*)calloc((size_t)(md->n_groups > 0 ? md->n_groups : 1), sizeof(double));
  double* dlogZ = (double*)calloc((size_t)(md->n_groups > 0 ? md->n_groups : 1) * P, sizeof(double));
  double* dsumZ = (double*)calloc(P, sizeof(double));
  if (!logZ || !dlogZ || !dsumZ) return -1;
  normalisers(md, lam, logZ, dlogZ);
  double sumZ = 0.0;
  for (int g = 0; g < md->n_groups; ++g) {
    sumZ += logZ[g];
    if (logZ_out) logZ_out[g] = logZ[g];
    for (int i = 0; i < P; ++i) dsumZ[i] += dlogZ[(size_t)g * P + i];
  }
  pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * T);
  Work* wk = (Work*)calloc(T, sizeof(Work));
  /* ---- events ---- */
  if (E > 0 && logBF && logNeff) {
    int next = 0;
    pthread_mutex_t lock = PTHREAD_MUTEX_INITIALIZER;
    for (int t = 0; t < T; ++t) {
      wk[t] = (Work){cat, md, lam, J_logBF ? want_jac : 0, T, t, &next, &lock, logBF, logNeff, J_logBF, J_logNeff, sumZ, dsumZ};
      pthread_create(&th[t], NULL, events_worker, &wk[t]);
    }
    for (int t = 0; t < T; ++t) pthread_join(th[t], NULL);
  }
  /* ---- injections: blocks in index order, merged in block order (deterministic) ---- */
  if (log_mu && logNeff_inj) {
    const int64_t I = cat->n_inj, per = (I + T - 1) / T;
    double gmax = -INFINITY;
    for (int t = 0; t < T; ++t) {
      memset(&wk[t], 0, sizeof(Work));
      wk[t].cat = cat; wk[t].md = md; wk[t].L = lam; wk[t].want_jac = want_jac;
      wk[t].a = t * per < I ? t * per : I;
      wk[t].b = (t + 1) * per < I ? (t + 1) * per : I;
      wk[t].sums.G1 = (double*)calloc(P, sizeof(double));
      wk[t].sums.G2 = (double*)calloc(P, sizeof(double));
      pthread_create(&th[t], NULL, inj_worker, &wk[t]);
    }
    for (int t = 0; t < T; ++t) {
      pthread_join(th[t], NULL);
      gmax = fmax(gmax, wk[t].sums.m);
    }
    double S1 = 0.0, S2 = 0.0;
    double* G1 = (double*)calloc(P, sizeof(double));
    double* G2 = (double*)calloc(P, sizeof(double));
    for (int t = 0; t < T; ++t) { /* merge in block order, relative to the global maximum */
      if (!(wk[t].sums.m > -INFINITY)) continue;
      sums_rescale(&wk[t].sums, gmax, P, want_jac);
      S1 += wk[t].sums.S1;
      S2 += wk[t].sums.S2;
      for (int i = 0; i < P; ++i) {
        G1[i] += wk[t].sums.G1[i];
        G2[i] += wk[t].sums.G2[i];
      }
    }
    /* analysis.py:91-136: mu = S1/N, var = S2/N^2 - mu^2/N, N_eff = mu^2/var */
    const double N = cat->total_inj, den = S2 - S1 * S1 / N;
    *log_mu = gmax + log(S1) - log(N) - sumZ;
    *logNeff_inj = 2.0 * log(S1) - log(den);
    if (want_jac)
      for (int i = 0; i < P; ++i) {
        const double n1 = G1[i] / S1;
        J_log_mu[i] = n1 - dsumZ[i];
        if (J_logNeff_inj) J_logNeff_inj[i] = 2.0 * n1 - (2.0 * G2[i] - 2.0 * S1 * S1 / N * n1) / den;
      }
    for (int t = 0; t < T; ++t) {
      free(wk[t].sums.G1);
      free(wk[t].sums.G2);
    }
    free(G1);
    free(G2);
  }
  free(th);
  free(wk);
  free(logZ);
  free(dlogZ);
  free(dsumZ);
  return 0;
}

int gwio_version(void) { return GWI_VERSION; }
