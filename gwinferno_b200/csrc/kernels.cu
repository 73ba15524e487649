// sm_100a kernels of the population-likelihood path.
//
//   prologue_kernel   per evaluation, from Lambda: polynomial pieces of every spline dimension,
//                     grid normalisers log Z_g and their gradients (interpolation.py:290;
//                     spline_perturbation.py:323-336), scalar normalisers, per-segment shift.
//   stream_kernel     THE hot kernel: one pass over the plan columns.  Per sample: unpack the
//                     (piece, offset) words, Horner-evaluate every spline dimension, add the
//                     non-spline terms and the static log-weight, p = exp(x - shift), and
//                     accumulate (sum p, sum p^2) plus the gradient moments sum p w^n per piece.
//                     Moments of the leading ("shallow") dimensions live in registers and are
//                     spilled only when the piece index changes (samples are piece-sorted); the
//                     trailing ("deep") dimensions use lane-private shared-memory accumulators.
//   reduce_kernel     fixed-order tree sum of the per-warp records.
//   finish_kernel     per segment: log-mean, log N_eff, Jacobian rows (moments -> coefficients).
//   partial/combine   likelihood glue (analysis.py:257-319) split around the multi-GPU exchange.
#include <cuda_runtime.h>

#include <cfloat>
#include <cmath>

#include "dev_structs.h"

// The small kernels read dozens of ModelDev fields, each a dependent global load if read in place (the cold
// prologue took 33 us under ncu, mostly load latency).  So a block first copies its chain's descriptor (~3 KB)
// into shared memory with coalesced 8-byte loads and works from that copy.
#define GWI_STAGED_DESC(M, src)                                                                              \
  __shared__ __align__(16) unsigned long long gwi_desc_stage[(sizeof(ModelDev) + 7) / 8];                    \
  {                                                                                                          \
    const unsigned long long* gwi_desc_src = reinterpret_cast<const unsigned long long*>(&(src));            \
    for (unsigned i = threadIdx.x; i < (sizeof(ModelDev) + 7) / 8; i += blockDim.x) gwi_desc_stage[i] = gwi_desc_src[i]; \
    __syncthreads();                                                                                         \
  }                                                                                                          \
  const ModelDev& M = *reinterpret_cast<const ModelDev*>(gwi_desc_stage)

namespace gwi {

// cubic B-spline piece basis in w = u - 1/2 :  b_k(u) = sum_n BETA[k][n] w^n
__constant__ double BETA[4][4] = {{1.0 / 48.0, -1.0 / 8.0, 1.0 / 4.0, -1.0 / 6.0},
                                  {23.0 / 48.0, -5.0 / 8.0, -1.0 / 4.0, 1.0 / 2.0},
                                  {23.0 / 48.0, 5.0 / 8.0, -1.0 / 4.0, -1.0 / 2.0},
                                  {1.0 / 48.0, 1.0 / 8.0, 1.0 / 4.0, 1.0 / 6.0}};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// deterministic block reductions (blockDim.x multiple of 32, <= 1024); scratch: 32 doubles
__device__ double block_sum(double v, double* scratch) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) scratch[w] = v;
  __syncthreads();
  double r = 0.0;
  for (int i = 0; i < nw; ++i) r += scratch[i];
  return r;
}
__device__ double block_max(double v, double* scratch) {
  v = warp_max(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) scratch[w] = v;
  __syncthreads();
  double r = -INFINITY;
  for (int i = 0; i < nw; ++i) r = fmax(r, scratch[i]);
  return r;
}

__device__ __forceinline__ void tap_weights(double u, double w[4]) {
  const double omu = 1.0 - u;
  w[0] = omu * omu * omu * (1.0 / 6.0);
  w[1] = (3.0 * u * u * u - 6.0 * u * u + 4.0) * (1.0 / 6.0);
  w[2] = (-3.0 * u * u * u + 3.0 * u * u + 3.0 * u + 1.0) * (1.0 / 6.0);
  w[3] = u * u * u * (1.0 / 6.0);
}

__device__ double digamma_dev(double x) {
  double r = 0.0;
  while (x < 10.0) {
    r -= 1.0 / x;
    x += 1.0;
  }
  const double f = 1.0 / (x * x);
  // asymptotic series: ln x - 1/2x - sum B_2n / (2n x^2n)
  const double t = f * (-1.0 / 12.0 + f * (1.0 / 120.0 + f * (-1.0 / 252.0 + f * (1.0 / 240.0 + f * (-1.0 / 132.0 + f * (691.0 / 32760.0 + f * (-1.0 / 12.0)))))));
  return r + log(x) - 0.5 / x + t;
}

__device__ __forceinline__ double norm_pdf(double x) { return exp(-0.5 * x * x) * 0.3989422804014327; }

// log-normalisation of the truncated normal and the two ratios its gradient needs
// (distributions.py:122-143): D = Phi(b) - Phi(a), formed where it keeps its relative accuracy:
//   - an interval narrow against the curvature of phi (half-width h, midpoint m): the series
//     D = 2h phi(m) sum_k He_2k(m) h^2k / (2k+1)!  (He: Hermite polynomials; terms after h^6 are < 1e-17 there);
//   - both bounds in one tail: the difference of erfc of that tail (the difference of two CDFs near 1 loses
//     everything once the interval lies ~8 sigma out);
//   - otherwise the difference of erf (no "1 +" to round away a small D).
__device__ void truncnorm_consts(double mu, double sig, double lo, double hi, double& lognorm, double& dDmu_D, double& dDsig_D) {
  const double a = (lo - mu) / sig, b = (hi - mu) / sig;
  const double h = 0.5 * (hi - lo) / sig, m = (0.5 * (lo + hi) - mu) / sig;
  const double r = 0.7071067811865476;
  double D;
  if (h * fmax(fabs(m), 1.0) < 0.01) {
    const double m2 = m * m, h2 = h * h;
    D = 2.0 * h * norm_pdf(m) * (1.0 + h2 * ((m2 - 1.0) * (1.0 / 6.0) + h2 * ((m2 * (m2 - 6.0) + 3.0) * (1.0 / 120.0) + h2 * (((m2 - 15.0) * m2 + 45.0) * m2 - 15.0) * (1.0 / 5040.0))));
  } else if (a >= 0.0) {
    D = 0.5 * (erfc(a * r) - erfc(b * r));
  } else if (b <= 0.0) {
    D = 0.5 * (erfc(-b * r) - erfc(-a * r));
  } else {
    D = 0.5 * (erf(b * r) - erf(a * r));
  }
  lognorm = -log(sig) - 0.9189385332046727 - log(D);
  dDmu_D = (-norm_pdf(b) + norm_pdf(a)) / sig / D;
  dDsig_D = (-b * norm_pdf(b) + a * norm_pdf(a)) / sig / D;
}

// Upper bound of the spline on polynomial piece J of dim D (convex-hull property: the bases are >= 0 and sum to <= 1):
// the maximum of the coefficients the piece uses.  Default pieces: c[J..J+3]; explicit knot vector: the coefficients whose
// basis polynomial on the piece is not identically zero, floored at 0 where the bases do not sum to one.
__device__ __forceinline__ double piece_upper_bound(const ModelDev& M, const DimDev& D, int J, const double* __restrict__ Lam) {
  if (J >= D.rows - 1) return 0.0;  // the dummy all-zero piece
  if (D.basis_off < 0) {
    const double* c = Lam + D.slot + J;
    return fmax(fmax(c[0], c[1]), fmax(c[2], c[3]));
  }
  const double* Bm = M.grid_pool + D.basis_off + J * 16;
  const double* c = Lam + D.slot + (int)M.grid_pool[D.first_off + J];
  double ub = M.grid_pool[D.floor_off + J];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const double* b = Bm + k * 4;
    if (b[0] != 0.0 || b[1] != 0.0 || b[2] != 0.0 || b[3] != 0.0) ub = fmax(ub, c[k]);
  }
  return ub == -INFINITY ? 0.0 : ub;  // a piece without any basis: the spline is 0 there
}

// =================================================================================================
// prologue
// =================================================================================================
__global__ void __launch_bounds__(256) prologue_kernel(const ModelDev* __restrict__ Mp, const double* __restrict__ Lam0, int role_off, int use_learned_shift) {
  GWI_PDL_TRIGGER();  // the stream kernel may be scheduled (it waits for this grid before it reads the tables)
  GWI_STAGED_DESC(M, Mp[blockIdx.y]);  // blockIdx.y = chain
  const double* __restrict__ Lam = Lam0 + (size_t)blockIdx.y * M.n_params;
  extern __shared__ double sm[];
  __shared__ double scratch[32];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int P = M.n_params;
  const int role = (int)blockIdx.x + role_off;  // [0, n_groups): one norm group each; n_groups: tables + shifts
  if (role < M.n_groups) {
    // ---------------- one norm group ----------------
    const int g = role;
    const int G = M.groups[g].n_grid;
    const double* logw = M.grid_pool + M.groups[g].logw_off;
    double* li = sm;  // [G]
    bool liny = false;
    for (int d = 0; d < M.n_dims; ++d) liny = liny || (M.dims[d].norm_group == g && M.dims[d].liny);
    if (liny) {
      // spline density (BSpline.norm, interpolation.py:280-291): Z = sum_i w_i sum_k B_k(x_i) c_k
      double s = 0.0;
      for (int i = tid; i < G; i += nt) {
        const double wq = exp(logw[i]);
        double sv = 0.0;
        for (int d = 0; d < M.n_dims; ++d) {
          const DimDev& D = M.dims[d];
          if (D.norm_group != g) continue;
          const double* aux = M.grid_pool + D.grid_aux;
          const int J = (int)aux[4 * G + i];
          if (J >= 0) {
            const double* w = aux + 4 * i;
            const double* c = Lam + D.slot + J;
            sv += w[0] * c[0] + w[1] * c[1] + w[2] * c[2] + w[3] * c[3];
          }
        }
        li[i] = wq;
        s += wq * sv;
      }
      s = block_sum(s, scratch);
      if (tid == 0) M.logZ[g] = log(s);
      const double inv = 1.0 / s;
      for (int i = tid; i < P; i += nt) M.dlogZ[(size_t)g * P + i] = 0.0;
      __syncthreads();
      for (int d = 0; d < M.n_dims; ++d) {
        const DimDev& D = M.dims[d];
        if (D.norm_group != g) continue;
        const double* aux = M.grid_pool + D.grid_aux;
        for (int k = tid >> 5; k < D.n_splines; k += nt >> 5) {
          double acc = 0.0;
          const int lo = (int)aux[5 * G + k], hi = (int)aux[5 * G + D.n_splines + k];
          for (int i = lo + (tid & 31); i < hi; i += 32) {
            const int J = (int)aux[4 * G + i];
            const int kk = k - J;
            if (J < 0 || kk < 0 || kk > 3) continue;
            acc += li[i] * aux[4 * i + kk];
          }
          acc = warp_sum(acc);
          if ((tid & 31) == 0) M.dlogZ[(size_t)g * P + D.slot + k] += acc * inv;
        }
        __syncthreads();
      }
      return;
    }
    for (int i = tid; i < G; i += nt) {
      double v = logw[i];
      for (int d = 0; d < M.n_dims; ++d) {
        const DimDev& D = M.dims[d];
        if (D.norm_group != g) continue;
        const double* aux = M.grid_pool + D.grid_aux;  // W[4G] | J[G] | lo[n] | hi[n]
        const int J = (int)aux[4 * G + i];
        if (J >= 0) {
          const double* w = aux + 4 * i;
          const double* c = Lam + D.slot + J;
          v += w[0] * c[0] + w[1] * c[1] + w[2] * c[2] + w[3] * c[3];
        }
      }
      for (int q = 0; q < M.n_kops; ++q) {
        const KopDev& K = M.kops[q];
        if (K.kind == KOP_LIN && K.norm_group == g) v += (Lam[K.slot[0]] + K.cst[0]) * M.grid_pool[K.grid_off + i];
      }
      li[i] = v;
    }
    __syncthreads();
    double mx = -INFINITY;
    for (int i = tid; i < G; i += nt) mx = fmax(mx, li[i]);
    mx = block_max(mx, scratch);
    double s = 0.0;
    for (int i = tid; i < G; i += nt) {
      const double e = exp(li[i] - mx);
      li[i] = e;
      s += e;
    }
    s = block_sum(s, scratch);
    if (tid == 0) M.logZ[g] = mx + log(s);
    const double inv = 1.0 / s;
    for (int i = tid; i < P; i += nt) M.dlogZ[(size_t)g * P + i] = 0.0;
    __syncthreads();
    for (int d = 0; d < M.n_dims; ++d) {
      const DimDev& D = M.dims[d];
      if (D.norm_group != g) continue;
      const double* aux = M.grid_pool + D.grid_aux;
      // one warp per basis function, lanes stride over the grid points in its support
      for (int k = tid >> 5; k < D.n_splines; k += nt >> 5) {
        double acc = 0.0;
        const int lo = (int)aux[5 * G + k], hi = (int)aux[5 * G + D.n_splines + k];
        for (int i = lo + (tid & 31); i < hi; i += 32) {
          const int J = (int)aux[4 * G + i];
          const int kk = k - J;
          if (J < 0 || kk < 0 || kk > 3) continue;
          acc += li[i] * aux[4 * i + kk];
        }
        acc = warp_sum(acc);
        if ((tid & 31) == 0) M.dlogZ[(size_t)g * P + D.slot + k] += acc * inv;
      }
      __syncthreads();
    }
    for (int q = 0; q < M.n_kops; ++q) {
      const KopDev& K = M.kops[q];
      if (K.kind != KOP_LIN || K.norm_group != g) continue;
      double acc = 0.0;
      for (int i = tid; i < G; i += nt) acc += li[i] * M.grid_pool[K.grid_off + i];
      acc = block_sum(acc, scratch);
      if (tid == 0) M.dlogZ[(size_t)g * P + K.slot[0]] += acc * inv;
      __syncthreads();
    }
    return;
  }
  // ---------------- per-segment shifts: blocks role > n_groups, 256 segments each ----------------
  // (independent of the tables block: the per-piece bounds max(c_J..c_J+3) and the linear coefficients are
  // recomputed from Lambda here, so that the ~300 segments of a catalog do not wait behind the serial table
  // fill of ONE block -- the stream kernel starts after the slowest block of this launch)
  if (role > M.n_groups) {
    if (M.two_pass) return;
    __shared__ double ub_s[MAX_SPLINE_DIMS * MAX_ROWS];
    for (int r = tid; r < M.rows_total; r += nt) {
      int d = 0;
      while (d + 1 < M.n_dims && r >= M.dims[d + 1].row_off) ++d;
      const DimDev& D = M.dims[d];
      ub_s[r] = piece_upper_bound(M, D, r - D.row_off, Lam);
    }
    __syncthreads();
    const int s = (role - M.n_groups - 1) * nt + tid;
    if (s >= M.n_segments) return;
    const SegDev& S = M.segs[s];
    double sh = S.max_static;
    unsigned long long occ_all[MAX_SPLINE_DIMS];
#pragma unroll
    for (int d = 0; d < MAX_SPLINE_DIMS; ++d) occ_all[d] = S.occ[d];  // independent loads, issued together
#pragma unroll
    for (int d = 0; d < MAX_SPLINE_DIMS; ++d) {
      if (d >= M.n_dims) break;
      const DimDev& D = M.dims[d];
      // Maximum of the piece bounds over the OCCUPIED pieces: walk the set bits four at a time -- the bit extraction is
      // ALU-only, the four shared-memory loads are independent.  Measured prologue (eager, us, cfg3 / cfg2): one-at-a-time
      // walk 27.5 / 21.1, ALL rows with a predicate 47.8 / 18.1, four at a time 29.1 / 21.5, width-adaptive mix 74.2 / 21.6
      // (divergence inside the injection segment's warp).
      double mx = -INFINITY;
      unsigned long long occ = occ_all[d];
      const double* ub = ub_s + D.row_off;
      while (occ) {
        const int J0 = __ffsll((long long)occ) - 1;
        occ &= occ - 1;
        const int J1 = occ ? __ffsll((long long)occ) - 1 : J0;
        occ &= occ - 1;
        const int J2 = occ ? __ffsll((long long)occ) - 1 : J0;
        occ &= occ - 1;
        const int J3 = occ ? __ffsll((long long)occ) - 1 : J0;
        occ &= occ - 1;
        const double v0 = ub[J0], v1 = ub[J1], v2 = ub[J2], v3 = ub[J3];
        mx = fmax(fmax(mx, fmax(v0, v1)), fmax(v2, v3));
      }
      if (mx > -INFINITY) sh += mx;
    }
    for (int q = 0; q < M.n_kops; ++q) {
      const KopDev& K = M.kops[q];
      if (K.kind != KOP_LIN) continue;
      const double th = Lam[K.slot[0]] + K.cst[0];
      if (S.fmax[q] >= S.fmin[q]) sh += fmax(th * S.fmin[q], th * S.fmax[q]);
    }
    M.shift[s] = (sh == sh && sh > -INFINITY && sh < INFINITY) ? sh : 0.0;
    return;
  }
  // ---------------- tables, kop constants, scalar normalisers ----------------
  if (tid == 0) {
    M.slice_counter[0] = 0;
    M.slice_counter[1] = 0;
  }
  if (use_learned_shift)  // speculative shift: the maxima of the previous evaluation's full pass
    for (int sg = tid; sg < M.n_segments; sg += nt) M.shift[sg] = M.shift_next[sg];
  for (int r = tid; r < M.rows_total; r += nt) {
    int d = 0;
    while (d + 1 < M.n_dims && r >= M.dims[d + 1].row_off) ++d;
    const DimDev& D = M.dims[d];
    const int J = r - D.row_off;
    double a[4] = {0.0, 0.0, 0.0, 0.0};
    const double ub = piece_upper_bound(M, D, J, Lam);
    if (J < D.rows - 1) {
      if (D.basis_off < 0) {  // default uniform cubic pieces
        const double* c = Lam + D.slot + J;
#pragma unroll
        for (int n = 0; n < 4; ++n) a[n] = c[0] * BETA[0][n] + c[1] * BETA[1][n] + c[2] * BETA[2][n] + c[3] * BETA[3][n];
      } else {  // explicit knot vector / order: per-piece basis polynomials
        const double* Bm = M.grid_pool + D.basis_off + J * 16;
        const double* c = Lam + D.slot + (int)M.grid_pool[D.first_off + J];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
          for (int n = 0; n < 4; ++n) a[n] += c[k] * Bm[k * 4 + n];
      }
    }
#pragma unroll
    for (int n = 0; n < 4; ++n) M.tables[r * 4 + n] = a[n];
    M.piece_ub[r] = ub;
  }
  for (int q = tid; q < M.n_kops; q += nt) {
    const KopDev& K = M.kops[q];
    double* kc = M.kc + q * KC_STRIDE;
    for (int i = 0; i < KC_STRIDE; ++i) kc[i] = 0.0;
    if (K.kind == KOP_LIN) {
      kc[0] = Lam[K.slot[0]] + K.cst[0];
    } else if (K.kind == KOP_PLRATIO) {
      kc[0] = Lam[K.slot[0]];
      kc[1] = 1.0 + kc[0];
      kc[2] = kc[1] != 0.0 ? 1.0 / kc[1] : 0.0;
    } else if (K.kind == KOP_PLPEAK) {
      const double alpha = Lam[K.slot[0]], mu = Lam[K.slot[1]], sig = Lam[K.slot[2]], lam = Lam[K.slot[3]];
      double ln, dn, lt, dmu, dsg;
      const double a1 = 1.0 + alpha;
      powerlaw_lognorm(a1, a1 != 0.0 ? 1.0 / a1 : 0.0, log(K.cst[0]), log(K.cst[1] / K.cst[0]), ln, dn);
      truncnorm_consts(mu, sig, K.cst[0], K.cst[1], lt, dmu, dsg);
      kc[0] = alpha; kc[1] = ln; kc[2] = mu; kc[3] = 0.5 / (sig * sig); kc[4] = lt; kc[5] = lam;
      kc[6] = dn; kc[7] = sig; kc[8] = dmu; kc[9] = dsg;
      kc[10] = K.slot[4] >= 0 ? Lam[K.slot[4]] : 0.0;  // delta_m (0 = no low-mass window)
      kc[11] = K.cst[0];                                // mmin
    } else if (K.kind == KOP_ISOALIGN || K.kind == KOP_ISOALIGN2) {
      const double xi = Lam[K.slot[0]], sig = Lam[K.slot[1]];
      double lt, dmu, dsg;
      truncnorm_consts(1.0, sig, -1.0, 1.0, lt, dmu, dsg);
      kc[0] = xi; kc[1] = sig; kc[2] = lt; kc[3] = 0.5 / (sig * sig); kc[4] = dsg;
    } else if (K.kind == KOP_QUAD) {
      const double mu = Lam[K.slot[0]], sig = Lam[K.slot[1]];
      kc[0] = mu; kc[1] = sig; kc[2] = 0.5 / (sig * sig);
    } else if (K.kind == KOP_SMOOTH) {
      kc[0] = Lam[K.slot[0]];
    }
  }
  for (int i = tid; i < P + 1; i += nt) M.Ksum[i] = 0.0;
  __syncthreads();
  if (tid == 0) {
    double K = 0.0;
    for (int q = 0; q < M.n_sops; ++q) {
      const SopDev& S = M.sops[q];
      if (S.kind == SOP_POWERLAW_NORM) {
        double ln, dn;
        const double a1 = 1.0 + Lam[S.slot0];
        powerlaw_lognorm(a1, a1 != 0.0 ? 1.0 / a1 : 0.0, log(S.cst0), log(S.cst1 / S.cst0), ln, dn);
        K += ln;
        M.Ksum[1 + S.slot0] += dn;
      } else if (S.kind == SOP_BETA_NORM) {
        const double a = Lam[S.slot0], b = Lam[S.slot1], ls = log(S.cst0);
        K += -(lgamma(a) + lgamma(b) - lgamma(a + b)) - (a + b - 1.0) * ls;
        const double pab = digamma_dev(a + b);
        M.Ksum[1 + S.slot0] += -(digamma_dev(a) - pab) - ls;
        M.Ksum[1 + S.slot1] += -(digamma_dev(b) - pab) - ls;
      } else if (S.kind == SOP_TRUNCNORM_NORM) {
        double lt, dmu, dsg;
        const double sig = Lam[S.slot1];
        truncnorm_consts(Lam[S.slot0], sig, S.cst0, S.cst1, lt, dmu, dsg);
        K += lt;
        M.Ksum[1 + S.slot0] += -dmu;
        M.Ksum[1 + S.slot1] += -1.0 / sig - dsg;
      }
    }
    M.Ksum[0] = K;
  }
}

// =================================================================================================
// reductions
// =================================================================================================
// element i of the sum of the task's input records.  Eight independent partial sums (inputs r, r+8, ...: eight loads
// in flight instead of a chain of <= 64 dependent load->add steps, which made these kernels latency-bound), combined in
// a fixed order.  Level-0 records of the CTA-cooperative stream kernel are sparse by construction -- the NW main-warp
// records of a chunk hold the header + leading rows, the chunk's last record holds the deep rows, everything else is
// zero for ever -- so only the records that can be non-zero at element i are read.
__device__ __forceinline__ double reduce_element(const ModelDev& M, const ReduceTask& T, int i) {
  const int rec = M.rec_doubles;
  const double* __restrict__ in = T.src < 0 ? M.records0 : M.level_buf[T.src];
  const double* __restrict__ p = in + (size_t)T.in_first * rec + i;
  double a[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  const int NW = M.cta_main_warps;
  if (T.src < 0 && NW > 0) {
    const int RPC = NW + 1;
    if (i >= M.cta_lead_doubles) {  // deep rows: only the last record of every chunk
      int k = 0;
      for (int r = (NW + RPC - T.in_first % RPC) % RPC; r < T.in_count; r += RPC, k = (k + 1) & 7) a[k] += p[(size_t)r * rec];
    } else {  // header + leading rows: the main-warp records
      int ph = T.in_first % RPC, r = 0;
      for (; r + 8 <= T.in_count; r += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          if (ph != NW) a[k] += p[(size_t)(r + k) * rec];
          ph = ph == NW ? 0 : ph + 1;
        }
      }
      for (int k = 0; r + k < T.in_count; ++k) {
        if (ph != NW) a[k] += p[(size_t)(r + k) * rec];
        ph = ph == NW ? 0 : ph + 1;
      }
    }
  } else {
    int r = 0;
    for (; r + 8 <= T.in_count; r += 8) {
#pragma unroll
      for (int k = 0; k < 8; ++k) a[k] += p[(size_t)(r + k) * rec];
    }
    for (int k = 0; r + k < T.in_count; ++k) a[k] += p[(size_t)(r + k) * rec];
  }
  return ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
}

// One block = one task x 32 record elements; the 8 warps split the task's <= 64 inputs (warp g takes inputs g, g+8, ...:
// at most K = 8 independent loads per thread, ONE memory round trip) and the partial sums are combined through shared memory in
// the same fixed order as reduce_element's.  (A thread per element walking all 64 inputs needed 8 dependent rounds: ~20 us per
// level whatever the number of tasks.)
__global__ void __launch_bounds__(256) reduce_kernel(const ModelDev* __restrict__ Mp, int level) {
  constexpr int K = 8;  // loads per thread: fan-in 64 / 8 warps
  GWI_PDL_TRIGGER();
  const ModelDev& M = Mp[blockIdx.z];  // blockIdx.z = chain
  const ReduceTask T = M.level_tasks[level][blockIdx.x];  // (static data: read before the dependency wait)
  const int rec = M.rec_doubles;
  const int j = threadIdx.x & 31, g = threadIdx.x >> 5;
  GWI_PDL_WAIT();  // the producer of the input records has completed
  const int i = blockIdx.y * 32 + j;
  __shared__ double part[8][33];
  double acc = 0.0;
  if (i < rec) {
    const double* __restrict__ in = T.src < 0 ? M.records0 : M.level_buf[T.src];
    const double* __restrict__ p = in + (size_t)T.in_first * rec + i;
    const int NW = M.cta_main_warps;
    const bool sparse = T.src < 0 && NW > 0;
    const int RPC = NW + 1;
    const bool want_deep = sparse && i >= M.cta_lead_doubles;
    double v[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int r = g + 8 * k;
      bool use = r < T.in_count;
      if (use && sparse) use = (((T.in_first + r) % RPC) == NW) == want_deep;
      v[k] = use ? p[(size_t)r * rec] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) acc += v[k];
  }
  part[g][j] = acc;
  __syncthreads();
  if (g == 0 && i < rec)
    M.level_buf[level][(size_t)T.out_slot * rec + i] = ((part[0][j] + part[1][j]) + (part[2][j] + part[3][j])) + ((part[4][j] + part[5][j]) + (part[6][j] + part[7][j]));
}

__global__ void __launch_bounds__(256) segmax_kernel(const ModelDev* __restrict__ Mp) {
  const ModelDev& M = Mp[blockIdx.y];
  __shared__ double scratch[32];
  const int s = blockIdx.x;
  const SegDev& S = M.segs[s];
  double mx = -INFINITY;
  for (int c = threadIdx.x; c < S.n_chunks; c += blockDim.x) mx = fmax(mx, M.chunk_max[S.first_chunk + c]);
  mx = block_max(mx, scratch);
  if (threadIdx.x == 0) M.shift[s] = (mx > -INFINITY && mx < INFINITY) ? mx : 0.0;
}

// after a full pass that recorded the chunk maxima (speculative shift): learn the next evaluation's shift and
// flag the segments whose maximum is too far from the shift this evaluation used
__global__ void __launch_bounds__(256) segmax_learn_kernel(const ModelDev* __restrict__ Mp) {
  const ModelDev& M = Mp[blockIdx.y];
  __shared__ double scratch[32];
  const int s = blockIdx.x;
  const SegDev& S = M.segs[s];
  double mx = -INFINITY;
  for (int c = threadIdx.x; c < S.n_chunks; c += blockDim.x) mx = fmax(mx, M.chunk_max[S.first_chunk + c]);
  mx = block_max(mx, scratch);
  if (threadIdx.x == 0) {
    const bool finite = mx > -INFINITY && mx < INFINITY;
    M.shift_next[s] = finite ? mx : 0.0;
    M.spec_bad[s] = (finite && !(fabs(mx - M.shift[s]) < SPEC_SHIFT_TOL)) ? 1.0 : 0.0;
  }
}

// =================================================================================================
// finish: per segment
// =================================================================================================
// per-segment results from the segment's summed record `rec` (in shared memory): all threads of the block
__device__ void finish_segment(const ModelDev& M, int s, const double* rec) {
  const int P = M.n_params;
  const double S1 = rec[0], S2 = rec[1];
  const double shift = M.shift[s];
  const int ngs = M.n_gslots;
  const bool g2 = M.g2 != 0;
  const double* g1 = rec + 2;
  const double* g2v = rec + 2 + ngs;
  const double* M1 = rec + 2 + ngs * (g2 ? 2 : 1);
  const double* M2 = M1 + M.rows_total * 4;
  double K = M.Ksum[0];
  for (int g = 0; g < M.n_groups; ++g) K -= M.logZ[g];
  bool ok = (S1 > 0.0) && (S1 < INFINITY) && (S2 > 0.0) && (S2 < INFINITY);
  ok = ok && M.spec_bad[s] == 0.0;  // the learned shift was too far from this evaluation's maximum
  const double N = M.total_inj;
  const double den_inj = S2 - S1 * S1 / N;
  if (threadIdx.x == 0) {
    double* o = M.seg_out + (size_t)s * 4;
    const SegDev& S = M.segs[s];
    if (s == 0) {
      o[0] = shift + log(S1) - log(N) + K;
      o[1] = 2.0 * log(S1) - log(den_inj);
      o[2] = 1.0 / exp(o[1]) - 1.0 / N;
      M.inj_raw[0] = shift;
      M.inj_raw[1] = S1;
      M.inj_raw[2] = S2;
    } else {
      o[0] = shift + log(S1) - log(S.n_total) + K;
      o[1] = 2.0 * log(S1) - log(S2);
      o[2] = 1.0 / exp(o[1]) - 1.0 / S.n_total;
    }
    o[3] = ok ? 0.0 : 1.0;
  }
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    double G1 = 0.0, G2s = 0.0;
    for (int d = 0; d < M.n_dims; ++d) {
      const DimDev& D = M.dims[d];
      const int k = i - D.slot;
      if (k < 0 || k >= D.n_splines) continue;
      if (D.basis_off >= 0) {  // explicit knot vector: every piece whose 4 coefficients include k
        for (int J = 0; J < D.rows - 1; ++J) {
          const int kk = k - (int)M.grid_pool[D.first_off + J];
          if (kk < 0 || kk > 3) continue;
          const double* b = M.grid_pool + D.basis_off + J * 16 + kk * 4;
          const double* m1 = M1 + (D.row_off + J) * 4;
          G1 += b[0] * m1[0] + b[1] * m1[1] + b[2] * m1[2] + b[3] * m1[3];
          if (g2) {
            const double* m2 = M2 + (D.row_off + J) * 4;
            G2s += b[0] * m2[0] + b[1] * m2[1] + b[2] * m2[2] + b[3] * m2[3];
          }
        }
        continue;
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const int J = k - kk;
        if (J < 0 || J > D.rows - 2) continue;
        const double* m1 = M1 + (D.row_off + J) * 4;
        G1 += BETA[kk][0] * m1[0] + BETA[kk][1] * m1[1] + BETA[kk][2] * m1[2] + BETA[kk][3] * m1[3];
        if (g2) {
          const double* m2 = M2 + (D.row_off + J) * 4;
          G2s += BETA[kk][0] * m2[0] + BETA[kk][1] * m2[1] + BETA[kk][2] * m2[2] + BETA[kk][3] * m2[3];
        }
      }
    }
    for (int g = 0; g < ngs; ++g)
      if (M.gslot_slot[g] == i) {
        G1 += g1[g];
        if (g2) G2s += g2v[g];
      }
    double dK = M.Ksum[1 + i];
    for (int g = 0; g < M.n_groups; ++g) dK -= M.dlogZ[(size_t)g * P + i];
    const double n1 = ok ? G1 / S1 : 0.0;
    M.seg_J1[(size_t)s * P + i] = n1 + dK;
    if (s == 0) {
      M.inj_raw[3 + i] = G1;
      M.inj_raw[3 + P + i] = G2s;
      M.seg_Jn[(size_t)s * P + i] = (ok && g2) ? 2.0 * n1 - (2.0 * G2s - 2.0 * S1 * S1 / N * n1) / den_inj : 0.0;
    } else {
      M.seg_Jn[(size_t)s * P + i] = (ok && g2) ? 2.0 * n1 - 2.0 * G2s / S2 : 0.0;
    }
  }
}

__global__ void __launch_bounds__(256) finish_kernel(const ModelDev* __restrict__ Mp) {
  GWI_PDL_TRIGGER();
  GWI_STAGED_DESC(M, Mp[blockIdx.y]);
  const ReduceTask* __restrict__ tasks = M.level_tasks[M.n_levels - 1];
  const int s = blockIdx.x;
  const ReduceTask T = tasks[s];  // (static data: read before the dependency wait)
  GWI_PDL_WAIT();
  // last level of the record reduction (task s sums the <= 64 remaining inputs of segment s), fused in here
  extern __shared__ double srec[];
  {
    for (int i = threadIdx.x; i < M.rec_doubles; i += blockDim.x) srec[i] = reduce_element(M, T, i);
    __syncthreads();
  }
  finish_segment(M, s, srec);
}

// gather the per-segment results into the caller's gwi_outputs buffers
__global__ void export_kernel(const ModelDev* __restrict__ Mp, gwi_outputs out) {
  const ModelDev& M = Mp[0];
  const int P = M.n_params, E = M.n_segments - 1;
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  for (int e = tid; e < E; e += nt) {
    if (out.logBF) out.logBF[e] = M.seg_out[(size_t)(e + 1) * 4 + 0];
    if (out.logNeff) out.logNeff[e] = M.seg_out[(size_t)(e + 1) * 4 + 1];
  }
  if (tid == 0) {
    if (out.log_mu) out.log_mu[0] = M.seg_out[0];
    if (out.logNeff_inj) out.logNeff_inj[0] = M.seg_out[1];
  }
  for (int g = tid; g < M.n_groups; g += nt)
    if (out.logZ) out.logZ[g] = M.logZ[g];
  for (size_t i = tid; i < (size_t)E * P; i += nt) {
    if (out.J_logBF) out.J_logBF[i] = M.seg_J1[(size_t)P + i];
    if (out.J_logNeff) out.J_logNeff[i] = M.seg_Jn[(size_t)P + i];
  }
  for (int i = tid; i < P; i += nt) {
    if (out.J_log_mu) out.J_log_mu[i] = M.seg_J1[i];
    if (out.J_logNeff_inj) out.J_logNeff_inj[i] = M.seg_Jn[i];
  }
}

// =================================================================================================
// likelihood: per-rank partial record, then the rank-ordered combine (analysis.py:257-319)
// =================================================================================================
template <bool CG>
__device__ __forceinline__ double ldd(const double* p) {
  return CG ? __ldcg(p) : *p;
}

// The rank's partial record.  Warp `gwarp` of `n_gwarps` takes the hyper-parameters gwarp, gwarp +
// n_gwarps, ...; warp 0 also writes the header.  CG: the per-segment results were written by other
// blocks of the SAME kernel (fused epilogue) and must be read through L2.
template <bool CG>
__device__ __forceinline__ void partial_rows(const ModelDev& M, double* recd, int gwarp, int n_gwarps) {
  const int P = M.n_params, E = M.n_segments - 1;
  const int lane = threadIdx.x & 31;
  if (gwarp == 0) {
    // header: fixed-order (lane-strided, then butterfly) sums over this rank's events
    double sum_logBF = 0.0, min_ln = INFINITY, sum_var = 0.0, status = 0.0;
    for (int e = 1 + lane; e <= E; e += 32) {
      const double* o = M.seg_out + (size_t)e * 4;
      sum_logBF += ldd<CG>(o + 0);
      double ln = ldd<CG>(o + 1);  // analysis.py:296: min over nan_to_num(logn_effs)
      if (ln != ln) ln = 0.0;
      ln = fmin(fmax(ln, -DBL_MAX), DBL_MAX);
      min_ln = fmin(min_ln, ln);
      sum_var += ldd<CG>(o + 2);
      status = fmax(status, ldd<CG>(o + 3));
    }
    sum_logBF = warp_sum(sum_logBF);
    sum_var = warp_sum(sum_var);
    min_ln = -warp_max(-min_ln);
    status = warp_max(status);
    if (lane == 0) {
      recd[PR_SHIFT] = ldd<CG>(M.inj_raw + 0);
      recd[PR_S1] = ldd<CG>(M.inj_raw + 1);
      recd[PR_S2] = ldd<CG>(M.inj_raw + 2);
      recd[PR_SUM_LOGBF] = sum_logBF;
      recd[PR_MIN_LOGNEFF] = min_ln;
      recd[PR_SUM_VAR] = sum_var;
      recd[PR_N_EVENTS] = (double)E;
      recd[PR_STATUS] = status;  // events only: a rank may legitimately hold no (valid) injections;
                                 // the merged injection sum is checked in combine_kernel
    }
  }
  // one warp per hyper-parameter: sum_e J_logBF[e][i]
  for (int i = gwarp; i < P; i += n_gwarps) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;  // four independent chains (the loads of 128 events are in flight together)
    int e = 1 + lane;
    for (; e + 96 <= E; e += 128) {
      a0 += ldd<CG>(M.seg_J1 + (size_t)e * P + i);
      a1 += ldd<CG>(M.seg_J1 + (size_t)(e + 32) * P + i);
      a2 += ldd<CG>(M.seg_J1 + (size_t)(e + 64) * P + i);
      a3 += ldd<CG>(M.seg_J1 + (size_t)(e + 96) * P + i);
    }
    for (; e <= E; e += 32) a0 += ldd<CG>(M.seg_J1 + (size_t)e * P + i);
    double acc = warp_sum((a0 + a1) + (a2 + a3));
    if (lane == 0) {
      recd[PR_HEADER + i] = ldd<CG>(M.inj_raw + 3 + i);
      recd[PR_HEADER + P + i] = ldd<CG>(M.inj_raw + 3 + P + i);
      recd[PR_HEADER + 2 * P + i] = acc;
    }
  }
}

__global__ void __launch_bounds__(256) partial_kernel(const ModelDev* __restrict__ Mp, double* __restrict__ recd0) {
  const ModelDev& M = Mp[blockIdx.y];
  double* __restrict__ recd = recd0 + (size_t)blockIdx.y * (PR_HEADER + 3 * M.n_params);
  const int warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  partial_rows<false>(M, recd, blockIdx.x * wpb + warp, gridDim.x * wpb);
}

// rank-ordered merge of R partial records + the likelihood glue: all threads of one block.  CG: the
// records were written by OTHER GPUs through peer memory while this kernel was running (exchange_kernel):
// read them through L2.
template <bool CG>
__device__ void combine_records(const ModelDev& M, const double* recs, int R, const gwi_like_opts& opts, double* out) {
  const int P = M.n_params;
  const int stride = PR_HEADER + 3 * P;
  const double N = M.total_inj;
  const double SENT = -DBL_MAX;  // nan_to_num(-inf)
  // injection sums of all ranks on a common shift
  double m = -INFINITY;
  for (int r = 0; r < R; ++r)
    if (ldd<CG>(&recs[(size_t)r * stride + PR_S1]) > 0.0) m = fmax(m, ldd<CG>(&recs[(size_t)r * stride + PR_SHIFT]));
  double S1 = 0.0, S2 = 0.0, sum_logBF = 0.0, min_ln = INFINITY, sum_var = 0.0, status = 0.0;
  for (int r = 0; r < R; ++r) {
    const double* q = recs + (size_t)r * stride;
    if (ldd<CG>(&q[PR_S1]) > 0.0) {
      const double f = exp(ldd<CG>(&q[PR_SHIFT]) - m);
      S1 += ldd<CG>(&q[PR_S1]) * f;
      S2 += ldd<CG>(&q[PR_S2]) * f * f;
    }
    sum_logBF += ldd<CG>(&q[PR_SUM_LOGBF]);
    min_ln = fmin(min_ln, ldd<CG>(&q[PR_MIN_LOGNEFF]));
    sum_var += ldd<CG>(&q[PR_SUM_VAR]);
    status = fmax(status, ldd<CG>(&q[PR_STATUS]));
  }
  if (!(S1 > 0.0) || !(S1 < INFINITY)) status = 1.0;  // no injection weight survived on any rank
  double K = M.Ksum[0];
  for (int g = 0; g < M.n_groups; ++g) K -= M.logZ[g];
  const double den = S2 - S1 * S1 / N;
  const double log_mu = m + log(S1) - log(N) + K;
  const double logneff_inj = 2.0 * log(S1) - log(den);
  const double neff_inj = exp(logneff_inj);
  const double var_inj = 1.0 / neff_inj - 1.0 / N;
  const double Nobs = (double)opts.Nobs;
  double log_det = log_mu;
  if (opts.marginalize_selection) log_det -= (3.0 + Nobs) / (2.0 * neff_inj);
  bool passed = true;
  if (opts.min_neff_cut && !(logneff_inj >= log(4.0 * Nobs))) {
    log_det = INFINITY;
    passed = false;
  }
  const double sel = isinf(log_det) ? SENT : -Nobs * log_det;
  double log_l = sel + sum_logBF;
  if (log_l != log_l) log_l = SENT;
  log_l = fmin(fmax(log_l, -DBL_MAX), DBL_MAX);
  if (opts.min_neff_cut && exp(min_ln) <= Nobs) {
    log_l = SENT;
    passed = false;
  }
  const double variance = Nobs * Nobs * var_inj + sum_var;
  if (opts.max_variance_cut && !(variance <= 1.0)) {
    log_l = SENT;
    passed = false;
  }
  if (status != 0.0) passed = false;
  if (threadIdx.x == 0) {
    out[GWI_LIKE_LOG_L] = log_l;
    out[GWI_LIKE_PASSED] = passed ? 1.0 : 0.0;
    out[GWI_LIKE_LOG_MU] = log_mu;
    out[GWI_LIKE_LOGNEFF_INJ] = logneff_inj;
    out[GWI_LIKE_MIN_LOGNEFF] = min_ln;
    out[GWI_LIKE_SUM_LOGBF] = sum_logBF;
    out[GWI_LIKE_VARIANCE] = variance;
    out[GWI_LIKE_STATUS] = status;
  }
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    double G1 = 0.0, G2s = 0.0, sumJ = 0.0;
    for (int r = 0; r < R; ++r) {
      const double* q = recs + (size_t)r * stride;
      if (ldd<CG>(&q[PR_S1]) > 0.0) {
        const double f = exp(ldd<CG>(&q[PR_SHIFT]) - m);
        G1 += ldd<CG>(&q[PR_HEADER + i]) * f;
        G2s += ldd<CG>(&q[PR_HEADER + P + i]) * f * f;
      }
      sumJ += ldd<CG>(&q[PR_HEADER + 2 * P + i]);
    }
    double dK = M.Ksum[1 + i];
    for (int g = 0; g < M.n_groups; ++g) dK -= M.dlogZ[(size_t)g * P + i];
    const double n1 = G1 / S1;
    double g_det = n1 + dK;
    if (opts.marginalize_selection) {
      const double Jn = 2.0 * n1 - (2.0 * G2s - 2.0 * S1 * S1 / N * n1) / den;
      g_det += (3.0 + Nobs) / (2.0 * neff_inj) * Jn;
    }
    out[GWI_LIKE_HEADER + i] = passed ? (-Nobs * g_det + sumJ) : 0.0;
  }
}

// blockIdx.x = chain: chain c combines the R records at recs0 + c*R*stride into out0 + c*(HEADER+P)
__global__ void __launch_bounds__(256) combine_kernel(const ModelDev* __restrict__ Mp, const double* recs0, int R, gwi_like_opts opts, double* __restrict__ out0) {
  GWI_STAGED_DESC(M, Mp[blockIdx.x]);
  const int P = M.n_params;
  const int stride = PR_HEADER + 3 * P;
  combine_records<false>(M, recs0 + (size_t)blockIdx.x * R * stride, R, opts, out0 + (size_t)blockIdx.x * (GWI_LIKE_HEADER + P));
}

// =================================================================================================
// multi-GPU exchange owned by the library: every rank PUSHES its partial record into the exchange slots of
// every rank (its own included) with plain stores through NVLink peer memory, publishes it with a
// system-scope release of the slot's flag (the evaluation's epoch number), and the block that pushed into
// the rank's OWN slots goes on to wait for the flags of all ranks and runs the rank-ordered combine -- one
// launch, no collective library, no host in the loop.  Slots and flags are double-buffered by epoch parity:
// a rank can only be one evaluation ahead of the slowest rank (its combine of epoch e needs everybody's
// push of epoch e), so the slots of epoch e are never overwritten (epoch e + 2) while somebody still reads
// them.  mode 0 = push + wait + combine, 1 = push only, 2 = wait + combine only (single-process tests).
// =================================================================================================
__device__ __forceinline__ void store_release_sys(unsigned long long* p, unsigned long long v) {
#ifdef GWI_HOST_EMULATION
  __atomic_store_n(p, v, __ATOMIC_RELEASE);
#else
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
#endif
}
__device__ __forceinline__ unsigned long long load_acquire_sys(const unsigned long long* p) {
#ifdef GWI_HOST_EMULATION
  return __atomic_load_n(p, __ATOMIC_ACQUIRE);
#else
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
#endif
}

// push this rank's record into peer `b`'s slots and publish it (all threads of the block)
__device__ __forceinline__ void exchange_push(const CommDev& C, const double* rec_local, int stride, int par, unsigned long long epoch, int b) {
  double* dst = C.peer_slots[b] + (size_t)(par * C.n_ranks + C.rank) * stride;
  for (int i = threadIdx.x; i < stride; i += blockDim.x) dst[i] = rec_local[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) store_release_sys(C.peer_flags[b] + par * C.n_ranks + C.rank, epoch);
}

// wait for the records of all ranks in this rank's own slots, then the rank-ordered combine (all threads of the block)
__device__ void exchange_wait_combine(const ModelDev& M, const CommDev& C, int stride, int par, unsigned long long epoch, const gwi_like_opts& opts, double* out) {
  const int R = C.n_ranks;
  __shared__ int timed_out;
  if (threadIdx.x == 0) timed_out = 0;
  __syncthreads();
  if ((int)threadIdx.x < R) {
    const unsigned long long* f = C.peer_flags[C.rank] + par * R + threadIdx.x;
#ifdef GWI_HOST_EMULATION
    if (load_acquire_sys(f) != epoch) timed_out = 1;  // the emulated launches are sequential: the pushes must have happened
#else
    const long long t0 = clock64();
    while (load_acquire_sys(f) != epoch) {
      if (clock64() - t0 > 20000000000ll) {  // ~10 s: a peer died; report instead of hanging the GPU
        timed_out = 1;
        break;
      }
      __nanosleep(64);
    }
#endif
  }
  __syncthreads();
  if (timed_out) {
    if (threadIdx.x == 0) {
      out[GWI_LIKE_LOG_L] = -DBL_MAX;
      out[GWI_LIKE_PASSED] = 0.0;
      out[GWI_LIKE_STATUS] = 3.0;  // exchange timed out
    }
    return;
  }
  __threadfence_system();
  combine_records<true>(M, C.peer_slots[C.rank] + (size_t)par * R * stride, R, opts, out);
}

__global__ void __launch_bounds__(256) exchange_kernel(const ModelDev* __restrict__ Mp, const double* __restrict__ rec_local, CommDev C, unsigned long long epoch, int mode,
                                                       gwi_like_opts opts, double* __restrict__ out) {
  const ModelDev& M = Mp[0];
  const int stride = PR_HEADER + 3 * M.n_params;
  const int par = (int)(epoch & 1ull);
  const int b = blockIdx.x;  // the peer this block pushes to
  if (mode != 2) exchange_push(C, rec_local, stride, par, epoch, b);
  if (b != C.rank || mode == 1) return;
  exchange_wait_combine(M, C, stride, par, epoch, opts, out);
}

// partial record + what follows it, in ONE launch: the blocks compute the rows of the rank's record; the block that
// finishes last (arrival counter) goes on -- tail 1: single-rank combine; tail 2: push to every rank, wait, combine.
// blockIdx.y = chain (tail 2: one chain).
__global__ void __launch_bounds__(256) partial_tail_kernel(const ModelDev* __restrict__ Mp, double* recd0, int tail, gwi_like_opts opts, double* out0, CommDev C,
                                                           unsigned long long epoch) {
  GWI_PDL_TRIGGER();
  GWI_STAGED_DESC(M, Mp[blockIdx.y]);
  const int P = M.n_params, stride = PR_HEADER + 3 * P;
  double* recd = recd0 + (size_t)blockIdx.y * stride;
  GWI_PDL_WAIT();  // finish_kernel has completed
  const int warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  partial_rows<false>(M, recd, blockIdx.x * wpb + warp, gridDim.x * wpb);
  __shared__ int last_s;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int k = atomicAdd(M.tail_counter, 1);
    last_s = k == (int)gridDim.x - 1;
    if (last_s) *M.tail_counter = 0;  // nobody else touches it in this evaluation
  }
  __syncthreads();
  if (!last_s) return;
  __threadfence();
  double* out = out0 + (size_t)blockIdx.y * (GWI_LIKE_HEADER + P);
  if (tail == 1) {
    combine_records<true>(M, recd, 1, opts, out);
    return;
  }
  const int par = (int)(epoch & 1ull);
  for (int b = 0; b < C.n_ranks; ++b) {
    double* dst = C.peer_slots[b] + (size_t)(par * C.n_ranks + C.rank) * stride;
    for (int i = threadIdx.x; i < stride; i += blockDim.x) dst[i] = __ldcg(recd + i);
  }
  __threadfence_system();
  __syncthreads();
  if ((int)threadIdx.x < C.n_ranks) store_release_sys(C.peer_flags[threadIdx.x] + par * C.n_ranks + C.rank, epoch);
  exchange_wait_combine(M, C, stride, par, epoch, opts, out);
}

// =================================================================================================
// host-side launch helpers (called from api.cu)
// =================================================================================================
// tables + shifts (what the stream kernel needs) on `st`; the grid normalisers (only needed by
// finish_kernel) on `aux`, concurrently with the stream kernel.  `nc` = number of chains.
void launch_prologue_tables(const ModelDev* Md, const double* lam, int n_groups, int n_seg, bool two_pass, int nc, cudaStream_t st, int use_learned_shift) {
  const int shift_blocks = two_pass ? 0 : (n_seg + 255) / 256;  // block 0: tables; blocks 1..: per-segment shifts
  GWI_LAUNCH(prologue_kernel, dim3(1 + shift_blocks, nc), 256, 0, st)(Md, lam, n_groups, use_learned_shift);
}
void launch_segmax_learn(const ModelDev* Md, int n_seg, int nc, cudaStream_t st) { GWI_LAUNCH(segmax_learn_kernel, dim3(n_seg, nc), 256, 0, st)(Md); }
void launch_prologue_groups(const ModelDev* Md, const double* lam, int n_groups, int max_grid, int nc, cudaStream_t aux) {
  if (n_groups > 0) GWI_LAUNCH(prologue_kernel, dim3(n_groups, nc), 256, (size_t)max_grid * sizeof(double), aux)(Md, lam, 0, 0);
}
void launch_reduce(const ModelDev* Md, int level, int n_tasks, int rec, int nc, cudaStream_t st) {
  GWI_LAUNCH_PDL(reduce_kernel, dim3(n_tasks, (rec + 31) / 32, nc), 256, 0, st)(Md, level);
}
void launch_segmax(const ModelDev* Md, int n_seg, int nc, cudaStream_t st) { GWI_LAUNCH(segmax_kernel, dim3(n_seg, nc), 256, 0, st)(Md); }
void launch_finish(const ModelDev* Md, int n_seg, int rec_doubles, int nc, cudaStream_t st) {
  GWI_LAUNCH_PDL(finish_kernel, dim3(n_seg, nc), 256, (size_t)rec_doubles * sizeof(double), st)(Md);
}
void launch_export(const ModelDev* Md, const gwi_outputs& out, cudaStream_t st) { GWI_LAUNCH(export_kernel, 64, 256, 0, st)(Md, out); }
void launch_partial(const ModelDev* Md, double* rec, int n_params, int nc, cudaStream_t st) {
  GWI_LAUNCH(partial_kernel, dim3((n_params + 7) / 8, nc), 256, 0, st)(Md, rec);
}
void launch_exchange(const ModelDev* Md, const double* rec_local, const CommDev& C, unsigned long long epoch, int mode, const gwi_like_opts& o, double* out, cudaStream_t st) {
  GWI_LAUNCH(exchange_kernel, C.n_ranks, 256, 0, st)(Md, rec_local, C, epoch, mode, o, out);
}
void launch_partial_tail(const ModelDev* Md, double* rec, int n_params, int tail, const gwi_like_opts& o, double* out, const CommDev& C, unsigned long long epoch, int nc,
                         cudaStream_t st) {
  GWI_LAUNCH_PDL(partial_tail_kernel, dim3((n_params + 7) / 8, nc), 256, 0, st)(Md, rec, tail, o, out, C, epoch);
}
void launch_combine(const ModelDev* Md, const double* recs, int R, const gwi_like_opts& o, double* out, int nc, cudaStream_t st) {
  GWI_LAUNCH(combine_kernel, nc, 256, 0, st)(Md, recs, R, o, out);
}

}  // namespace gwi

// per-sample log-weights and posterior-predictive draws (gwi_sample_log_weights / gwi_draw_samples)
#include "sample_draw.cuh"
