// CTA-cooperative stream kernel (the headline path for spline models: B-spline terms + <= 2 linear
// terms, gradient of the means only).
//
// One persistent CTA per SM with two warp roles:
//   * NW "main" warps.  A chunk (a contiguous piece of ONE segment of the piece-sorted sample stream)
//     is split into NW sub-chunks; lane l of main warp w owns a contiguous sorted run.  Per iteration
//     a main warp takes ONE 64-sample block ([column][64] words, 512 B per column), staged into shared
//     memory by a bulk asynchronous copy (cp.async.bulk + mbarrier: one instruction of one lane moves the
//     whole 4.6 KB block, no register staging, ring of CTA_NSTAGE stages per warp), evaluates the cubics
//     of all dims, p = exp(x - shift), the sums S1 / S2, the linear-term gradients and the gradient
//     moments of the LEADING dims (register-resident per piece, spilled with fire-and-forget
//     red.global.add.f64 into the warp's own record when the piece changes), and publishes the two
//     weights p of every lane next to the staged block.
//   * NDEEP "deep" warps, one per trailing ("deep") dim, whose piece index changes with every sample.
//     A deep warp consumes the staged words of ITS dim + the published weights of every main warp in a
//     fixed order and accumulates the moments sum p w^n into lane-private shared-memory accumulators
//     [piece][moment pair][32 lanes] -- ONE set per dim and CTA, single phase, bank-conflict-free -- and
//     writes them to the chunk's deep record when the chunk ends.
// This takes the shared-memory read-modify-write chain (half of the stall samples of the one-role kernel,
// profiles/r01_final_cfg3_stream_kernel_stalls_by_line.txt) out of the main warps' dependency chain
// and the ~20 KB of accumulators per warp out of the occupancy equation.
// Records: every chunk owns NW + 1 consecutive level-0 records (main warp w -> slot + w: S1, S2, linear
// gradients, leading rows; deep warps -> slot + NW: deep rows); the fixed-order reduction tree does the
// rest, so results do not depend on which CTA processed which slice.
#pragma once
#include "stream.cuh"

namespace gwi {

// ---- mbarrier + bulk-copy primitives ------------------------------------------------------------
#ifdef GWI_HOST_EMULATION
#include <cstdio>
#include <cstdlib>
// CPU test build (tests/emu): an mbarrier is a word {completed phases : 32 | expected : 16 | pending : 16};
// the threads of a block are fibers of ONE OS thread, so plain accesses + a yield in the wait loop do.
typedef unsigned long long* mbar_t;
__device__ inline mbar_t mbar_at(unsigned char* base, unsigned off) { return reinterpret_cast<unsigned long long*>(base + off); }
__device__ inline mbar_t mbar_idx(mbar_t first, int i) { return first + i; }
__device__ inline void mbar_init(mbar_t b, unsigned count) { *b = ((unsigned long long)count << 16) | count; }
__device__ inline void mbar_fence_init() {}
__device__ inline void mbar_arrive(mbar_t b) {
  unsigned long long v = *b;
  unsigned pending = (unsigned)(v & 0xFFFFu) - 1u;
  const unsigned expected = (unsigned)((v >> 16) & 0xFFFFu);
  unsigned long long phases = v >> 32;
  if (pending == 0u) {
    pending = expected;
    ++phases;
  }
  *b = (phases << 32) | ((unsigned long long)expected << 16) | pending;
}
__device__ inline void mbar_arrive_expect_tx(mbar_t b, unsigned) { mbar_arrive(b); }  // the emulated copy is synchronous
__device__ inline void mbar_wait(mbar_t b, unsigned parity) {
  unsigned long long spins = 0;
  while ((((*(volatile unsigned long long*)b) >> 32) & 1ull) == (unsigned long long)parity) {
    gwi_emu::warp_yield();
    if (++spins == 40000000ull) {  // a protocol error in the emulated run: say where instead of hanging the test
      extern thread_local double sm[];
      std::fprintf(stderr, "gwi_emu: mbarrier wait stuck: block %u thread %u barrier +%ld parity %u value %llx\n", blockIdx.x, threadIdx.x,
                   (long)((unsigned char*)b - (unsigned char*)sm), parity, *b);
      std::abort();
    }
  }
}
__device__ inline void bulk_copy_g2s(void* dst, const void* src, unsigned bytes, mbar_t) { std::memcpy(dst, src, bytes); }
#else
typedef unsigned mbar_t;  // shared-window address
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ mbar_t mbar_at(unsigned char* base, unsigned off) { return smem_u32(base + off); }
__device__ __forceinline__ mbar_t mbar_idx(mbar_t first, int i) { return first + 8u * (unsigned)i; }
__device__ __forceinline__ void mbar_init(mbar_t b, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(mbar_t b) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(b) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(mbar_t b, unsigned bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(b), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(mbar_t b, unsigned parity) {
  unsigned ok;
  // the hint lets the hardware SUSPEND the warp (no issue slots burnt) until the phase completes or ~the hint elapses
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(b), "r"(parity), "r"(20000u) : "memory");
  return ok != 0u;
}
// all 32 lanes call this together (warp-uniform control flow: a lone lane spinning here while the others run ahead would
// split the warp for the rest of the loop body -- measured: every main-loop instruction issued twice)
__device__ __forceinline__ void mbar_wait(mbar_t b, unsigned parity) {
  unsigned tries = 0;
  while (!mbar_try_wait(b, parity)) {
    if (++tries > (1u << 22)) __trap();  // a protocol error must end in a launch failure, not in a hung GPU
  }
  __syncwarp();
}
// one lane moves `bytes` (multiple of 16) from global to shared memory; completion is signalled on `bar`
__device__ __forceinline__ void bulk_copy_g2s(void* dst, const void* src, unsigned bytes, mbar_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(__cvta_generic_to_global(src)), "r"(bytes),
               "r"(bar)
               : "memory");
}
#endif

__device__ __forceinline__ void red_add_global(double* p, double v) {
#ifdef GWI_HOST_EMULATION
  atomicAdd(p, v);
#else
  asm volatile("red.global.add.f64 [%0], %1;" ::"l"(__cvta_generic_to_global(p)), "d"(v) : "memory");
#endif
}

// record-time flush of the register moments of one leading dim (all 32 lanes, converged): segmented
// shuffle scan over maximal runs of lanes on the same row, then the last lane of each run adds into the
// warp's own record (global reduction: equal rows may recur non-adjacently)
__device__ __forceinline__ void flush_moments_red(double* recM, int row, int lane, double (&a1)[4]) {
  const int prev = __shfl_up_sync(0xffffffffu, row, 1);
  const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || prev != row);
  const int head = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
  const int next = __shfl_down_sync(0xffffffffu, row, 1);
  const bool tail = lane == 31 || next != row;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const bool take = lane - off >= head;
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      const double u = __shfl_up_sync(0xffffffffu, a1[n], off);
      if (take) a1[n] += u;
    }
  }
  if (tail && row >= 0) {
#pragma unroll
    for (int n = 0; n < 4; ++n) red_add_global(&recM[row * 4 + n], a1[n]);
  }
#pragma unroll
  for (int n = 0; n < 4; ++n) a1[n] = 0.0;
}

template <int NS, int NDEEP, int NLIN>
__global__ void __launch_bounds__(CTA_MAX_WARPS * 32, 1) stream_cta_kernel(const ModelDev* __restrict__ Mp) {
  GWI_PDL_TRIGGER();  // the record reduction may be scheduled behind this grid (it waits for it to complete)
  const ModelDev& M = Mp[blockIdx.y];  // blockIdx.y = chain
  constexpr int NSH = NS - NDEEP;
  constexpr int NSHd = NSH > 0 ? NSH : 1;
  constexpr int NLd = NLIN > 0 ? NLIN : 1;
  extern __shared__ __align__(16) double sm[];
  unsigned char* const smb = reinterpret_cast<unsigned char*>(sm);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int NW = M.cta_main_warps;
  const int ncol = M.n_columns, rows_total = M.rows_total, n_gs = M.n_gslots;
  const CtaLayout L = cta_layout(NW, ncol, rows_total, M.deep_rows);  // smem_layout.h
  double* const tables = reinterpret_cast<double*>(smb + L.tables);
  volatile int* const ctl = reinterpret_cast<volatile int*>(smb + L.ctl);
  // Synchronisation (all mbarriers, phases = uses of a stage):
  //   full[w][s]  the bulk copy of main warp w's block has landed in stage s            (waited by main warp w)
  //   ready[s]    ALL main warps have published the weights of their block in stage s   (count NW; waited by the deep warps)
  //   free[s]     ALL deep warps have read every block + weights of stage s             (count NDEEP; waited by the main warps
  //               before they stage their next block there)
  // so the main warps advance in lock-step within the ring depth and a deep warp synchronises ONCE per iteration for a
  // burst of NW blocks (one wait per block made the deep warps the bottleneck: ~490 cycles per block, r02c3 profile).
  const mbar_t bars0 = mbar_at(smb, L.bars);
  auto bar_full = [&](int w, int s) { return mbar_idx(bars0, w * CTA_NSTAGE + s); };
  auto bar_ready = [&](int s) { return mbar_idx(bars0, NW * CTA_NSTAGE + s); };
  auto bar_free = [&](int s) { return mbar_idx(bars0, (NW + 1) * CTA_NSTAGE + s); };
  auto stage_ptr = [&](int w, int s) { return smb + L.stages + (unsigned)(w * CTA_NSTAGE + s) * L.stage_bytes; };

  {
    double2* dz = reinterpret_cast<double2*>(smb + L.deep);
    for (int i = threadIdx.x; i < M.deep_rows * 64; i += blockDim.x) dz[i] = make_double2(0.0, 0.0);  // [row][moment pair][32 lanes]
  }
  if (threadIdx.x == 0) {
    for (int s = 0; s < CTA_NSTAGE; ++s) {
      for (int w = 0; w < NW; ++w) mbar_init(bar_full(w, s), 1);
      mbar_init(bar_ready(s), NW);
      mbar_init(bar_free(s), NDEEP);
    }
    mbar_fence_init();
  }
  __syncthreads();
  // ---- everything above touches static data only; now wait for prologue_kernel's tables / shifts / counters ----
  GWI_PDL_WAIT();  // prologue_kernel (tables, shifts, slice counters) has completed
  for (int i = threadIdx.x; i < rows_total * 4; i += blockDim.x) tables[i] = M.tables[i];
  double2* const dtab = reinterpret_cast<double2*>(smb + L.dtab);
  {
    int dro = 0;
    for (int d = NSH; d < NS; ++d) {
      const int rows = M.dims[d].rows, ro = M.dims[d].row_off;
      for (int i = threadIdx.x; i < rows * 16; i += blockDim.x) {
        const int h = i / (rows * 8), r = (i >> 3) % rows;  // [h][r][copy]
        dtab[dro * 16 + i] = make_double2(M.tables[(ro + r) * 4 + 2 * h], M.tables[(ro + r) * 4 + 2 * h + 1]);
      }
      dro += rows;
    }
  }
  __syncthreads();

  const uint64_t* __restrict__ cols = M.columns;
  const size_t blk_words = (size_t)ncol * 64;
  unsigned ring_s = 0, ring_ph = 0;  // stage / phase parity of this warp's NEXT iteration (identical for all warps: every chunk runs on all NW main warps)
  unsigned ring_g = 0;               // iterations done so far

  // ---- main-warp state ----
  double S1 = 0.0, S2 = 0.0;
  int cur[NSHd];
  double cf[NSHd][4], m1[NSHd][4];
  const double* tab_d[NS];
  const double2* dt01[NS];  // deep dims: conflict-free replicated half-rows (see CtaLayout::dtab)
  int dt23_off[NS];
  int row_off[NS];
  {
    int dro = 0;
#pragma unroll
    for (int d = 0; d < NS; ++d) {
      row_off[d] = M.dims[d].row_off;
      tab_d[d] = tables + row_off[d] * 4;
      dt01[d] = dtab + dro * 16 + (lane & 7);
      dt23_off[d] = 0;
      if (d >= NSH) {
        dt23_off[d] = M.dims[d].rows * 8;
        dro += M.dims[d].rows;
      }
    }
  }
#pragma unroll
  for (int d = 0; d < NSH; ++d) {
    cur[d] = -1;
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      cf[d][n] = 0.0;
      m1[d][n] = 0.0;
    }
  }
  double theta[NLd], gl1[NLd];
  int lin_off[NLd];
#pragma unroll
  for (int l = 0; l < NLIN; ++l) {
    theta[l] = M.kc[l * KC_STRIDE];
    lin_off[l] = M.kops[l].col0 * 512 + lane * 16;
    gl1[l] = 0.0;
  }
  const int st_off = M.col_static * 512 + lane * 16;
  const int lead_doubles = M.cta_lead_doubles;  // {S1, S2}, linear slots, leading rows (they come first in a record)

  for (;;) {
    if (threadIdx.x == 0) ctl[0] = atomicAdd(M.slice_counter, 1);
    __syncthreads();
    const int sl = ctl[0];
    __syncthreads();  // everybody has read the slice id before thread 0 fetches the next one
    if (sl >= M.n_slices) break;
    const int c_begin = M.slice_begin[sl], c_end = M.slice_begin[sl + 1];
    if (warp < NW) {
      // ================================ main warp ================================
      for (int c = c_begin; c < c_end; ++c) {
        const Chunk C = M.chunks[c];
        const double shift = M.shift[C.segment];
        const int iters = C.steps >> 1;
        double* const rec = M.records0 + (size_t)(C.record_slot + warp) * M.rec_doubles;
        double* const recM = rec + 2 + n_gs;
        for (int i = lane; i < lead_doubles; i += 32) rec[i] = 0.0;
        __syncwarp();  // the zeroing is ordered before every lane's reductions
        const uint64_t* const src = cols + ((size_t)(C.first >> 6) + (size_t)warp * iters) * blk_words;
        const unsigned g0 = ring_g;  // ring position of this chunk's first block
        auto issue = [&](int t) {  // ALL lanes (uniform control flow); lane 0 stages block t of this sub-chunk
          const unsigned g = g0 + (unsigned)t;
          const unsigned s = g % CTA_NSTAGE, use = g / CTA_NSTAGE;
          if (use > 0) mbar_wait(bar_free(s), (use - 1u) & 1u);  // the deep warps are done with the previous blocks in this stage
          if (lane == 0) {
            const mbar_t fb = bar_full(warp, s);
            mbar_arrive_expect_tx(fb, L.blk_bytes);
            bulk_copy_g2s(stage_ptr(warp, s), src + (size_t)t * blk_words, L.blk_bytes, fb);
          }
        };
        for (int t = 0; t < CTA_NSTAGE - 1 && t < iters; ++t) issue(t);
        for (int it = 0; it < iters; ++it) {
          mbar_wait(bar_full(warp, ring_s), ring_ph);
          const unsigned char* const stg = stage_ptr(warp, ring_s);
          // ---- the two samples of this lane: words are w = u - 1/2 with J in the 6 low mantissa bits ----
          double w0[NS], w1[NS];
          int J0[NS], J1[NS];
#pragma unroll
          for (int d = 0; d < NS; ++d) {
            const ulonglong2 q = *reinterpret_cast<const ulonglong2*>(stg + d * 512 + lane * 16);
            J0[d] = (int)((unsigned)q.x & 63u);
            J1[d] = (int)((unsigned)q.y & 63u);
            w0[d] = __longlong_as_double((long long)q.x);
            w1[d] = __longlong_as_double((long long)q.y);
          }
          const double2 stat = *reinterpret_cast<const double2*>(stg + st_off);
          double2 fl[NLd];
#pragma unroll
          for (int l = 0; l < NLIN; ++l) fl[l] = *reinterpret_cast<const double2*>(stg + lin_off[l]);
          // ---- sample 0: spill finished pieces + fetch coefficients where a leading piece changed ----
          if (NSH > 0) {
            int chg0 = 0;
#pragma unroll
            for (int d = 0; d < NSH; ++d) chg0 |= J0[d] ^ cur[d];
            if (chg0 != 0) {
#pragma unroll
              for (int d = 0; d < NSH; ++d) {
                if (J0[d] != cur[d]) {
                  if (cur[d] >= 0) {
#pragma unroll
                    for (int n = 0; n < 4; ++n) {
                      red_add_global(&recM[(row_off[d] + cur[d]) * 4 + n], m1[d][n]);
                      m1[d][n] = 0.0;
                    }
                  }
                  cur[d] = J0[d];
                  const double2 a01 = *reinterpret_cast<const double2*>(tab_d[d] + J0[d] * 4);
                  const double2 a23 = *reinterpret_cast<const double2*>(tab_d[d] + J0[d] * 4 + 2);
                  cf[d][0] = a01.x;
                  cf[d][1] = a01.y;
                  cf[d][2] = a23.x;
                  cf[d][3] = a23.y;
                }
              }
            }
          }
          double x0 = stat.x, x1 = stat.y;
#pragma unroll
          for (int d = 0; d < NS; ++d) {
            const double w = w0[d];
            if (d < NSH) {
              x0 += fma(fma(cf[d][3], w, cf[d][2]), w * w, fma(cf[d][1], w, cf[d][0]));
            } else {
              const double2 a01 = dt01[d][J0[d] * 8];
              const double2 a23 = dt01[d][dt23_off[d] + J0[d] * 8];
              x0 += fma(fma(a23.y, w, a23.x), w * w, fma(a01.y, w, a01.x));
            }
          }
          // ---- sample 1: its leading pieces may differ from sample 0's: fetch ITS coefficients now; the
          //      moments of sample 0's pieces stay in the registers until sample 0 has been accumulated ----
          int dif = 0;
          if (NSH > 0) {
#pragma unroll
            for (int d = 0; d < NSH; ++d) dif |= J1[d] ^ J0[d];
            if (dif != 0) {
#pragma unroll
              for (int d = 0; d < NSH; ++d) {
                if (J1[d] != J0[d]) {
                  const double2 a01 = *reinterpret_cast<const double2*>(tab_d[d] + J1[d] * 4);
                  const double2 a23 = *reinterpret_cast<const double2*>(tab_d[d] + J1[d] * 4 + 2);
                  cf[d][0] = a01.x;
                  cf[d][1] = a01.y;
                  cf[d][2] = a23.x;
                  cf[d][3] = a23.y;
                }
              }
            }
          }
#pragma unroll
          for (int d = 0; d < NS; ++d) {
            const double w = w1[d];
            if (d < NSH) {
              x1 += fma(fma(cf[d][3], w, cf[d][2]), w * w, fma(cf[d][1], w, cf[d][0]));
            } else {
              const double2 a01 = dt01[d][J1[d] * 8];
              const double2 a23 = dt01[d][dt23_off[d] + J1[d] * 8];
              x1 += fma(fma(a23.y, w, a23.x), w * w, fma(a01.y, w, a01.x));
            }
          }
#pragma unroll
          for (int l = 0; l < NLIN; ++l) {
            x0 = fma(theta[l], fl[l].x, x0);
            x1 = fma(theta[l], fl[l].y, x1);
          }
          const double p0 = exp_nonpos(x0 - shift), p1 = exp_nonpos(x1 - shift);
          // ---- publish the weights for the deep warps ----
          *reinterpret_cast<double2*>(const_cast<unsigned char*>(stg) + L.blk_bytes + lane * 16) = make_double2(p0, p1);
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_ready(ring_s));
          // ---- register-resident sums ----
          S1 += p0;
          S2 = fma(p0, p0, S2);
#pragma unroll
          for (int l = 0; l < NLIN; ++l) gl1[l] = fma(p0, fl[l].x, gl1[l]);
#pragma unroll
          for (int d = 0; d < NSH; ++d) {
            const double w = w0[d], w2 = w * w, w3 = w2 * w;
            m1[d][0] += p0;
            m1[d][1] = fma(p0, w, m1[d][1]);
            m1[d][2] = fma(p0, w2, m1[d][2]);
            m1[d][3] = fma(p0, w3, m1[d][3]);
          }
          if (NSH > 0 && dif != 0) {
            // the moments follow the coefficients
#pragma unroll
            for (int d = 0; d < NSH; ++d) {
              if (J1[d] != cur[d]) {
#pragma unroll
                for (int n = 0; n < 4; ++n) {
                  red_add_global(&recM[(row_off[d] + cur[d]) * 4 + n], m1[d][n]);
                  m1[d][n] = 0.0;
                }
                cur[d] = J1[d];
              }
            }
          }
          S1 += p1;
          S2 = fma(p1, p1, S2);
#pragma unroll
          for (int l = 0; l < NLIN; ++l) gl1[l] = fma(p1, fl[l].y, gl1[l]);
#pragma unroll
          for (int d = 0; d < NSH; ++d) {
            const double w = w1[d], w2 = w * w, w3 = w2 * w;
            m1[d][0] += p1;
            m1[d][1] = fma(p1, w, m1[d][1]);
            m1[d][2] = fma(p1, w2, m1[d][2]);
            m1[d][3] = fma(p1, w3, m1[d][3]);
          }
          ++ring_g;
          if (++ring_s == CTA_NSTAGE) {
            ring_s = 0;
            ring_ph ^= 1u;
          }
          // stage the block NSTAGE - 1 iterations ahead into the stage of iteration it - 1: the deep warps have had this whole
          // iteration to read that one (waiting for it at the TOP of the iteration put their burst on every iteration's
          // critical path: r02c4 profile, 28 % of the samples in this wait); the copy still has NSTAGE - 2 iterations to land
          if (it + CTA_NSTAGE - 1 < iters) issue(it + CTA_NSTAGE - 1);
        }
        // ---- this warp's record of the chunk ----
        __syncwarp();
#pragma unroll
        for (int d = 0; d < NSH; ++d) {
          flush_moments_red(recM, cur[d] >= 0 ? row_off[d] + cur[d] : -1, lane, m1[d]);
          cur[d] = -1;  // the moments are zero now: nothing to spill at the next piece change
        }
        const double s1 = wsum(S1), s2 = wsum(S2);
        S1 = 0.0;
        S2 = 0.0;
        if (lane == 0) {
          rec[0] = s1;
          rec[1] = s2;
        }
#pragma unroll
        for (int l = 0; l < NLIN; ++l) {
          const double a = wsum(gl1[l]);
          gl1[l] = 0.0;
          if (lane == 0) rec[2 + l] = a;
        }
      }
    } else {
      // ================================ deep warp ================================
      const int dd = NSH + (warp - NW);  // my dim (uniform in the warp)
      int dim_row_off = 0, dim_rows = 0, dim_deep_off = 0;
#pragma unroll
      for (int d = NSH; d < NS; ++d)
        if (d == dd) {
          dim_row_off = M.dims[d].row_off;
          dim_rows = M.dims[d].rows;
          dim_deep_off = M.dims[d].deep_off;
        }
      double2* const acc = reinterpret_cast<double2*>(smb + L.deep) + (size_t)dim_deep_off * 32 + lane;  // [J][pair][32 lanes]
      const int w_off = dd * 512 + lane * 16;
      for (int c = c_begin; c < c_end; ++c) {
        const Chunk C = M.chunks[c];
        const int iters = C.steps >> 1;
        for (int it = 0; it < iters; ++it) {
          mbar_wait(bar_ready(ring_s), ring_ph);  // every main warp has published the weights of its block in this stage
          const unsigned char* stg = stage_ptr(0, ring_s);
          for (int w = 0; w < NW; ++w, stg += CTA_NSTAGE * L.stage_bytes) {
            const ulonglong2 q = *reinterpret_cast<const ulonglong2*>(stg + w_off);
            const double2 pp = *reinterpret_cast<const double2*>(stg + L.blk_bytes + lane * 16);
            if (w == NW - 1) {
              __syncwarp();  // every lane has read the last block: the stage may be refilled
              if (lane == 0) mbar_arrive(bar_free(ring_s));
            }
            // accumulators of both samples first (independent unless the pieces coincide)
            const unsigned Ja = (unsigned)q.x & 63u, Jb = (unsigned)q.y & 63u;
            double2* const ea = acc + (size_t)Ja * 64;
            double2* const eb = acc + (size_t)Jb * 64;
            double2 a0 = ea[0], a1 = ea[32], b0 = eb[0], b1 = eb[32];
            {
              const double wv = __longlong_as_double((long long)q.x), w2 = wv * wv, w3 = w2 * wv;
              a0.x += pp.x;
              a0.y = fma(pp.x, wv, a0.y);
              a1.x = fma(pp.x, w2, a1.x);
              a1.y = fma(pp.x, w3, a1.y);
            }
            if (Ja == Jb) {  // same piece: the second sample continues from the first one's sums
              b0 = a0;
              b1 = a1;
            }
            {
              const double wv = __longlong_as_double((long long)q.y), w2 = wv * wv, w3 = w2 * wv;
              b0.x += pp.y;
              b0.y = fma(pp.y, wv, b0.y);
              b1.x = fma(pp.y, w2, b1.x);
              b1.y = fma(pp.y, w3, b1.y);
            }
            ea[0] = a0;
            ea[32] = a1;
            eb[0] = b0;  // (after the stores of sample a: if the pieces coincide these are the final values)
            eb[32] = b1;
          }
          ++ring_g;
          if (++ring_s == CTA_NSTAGE) {
            ring_s = 0;
            ring_ph ^= 1u;
          }
        }
        // ---- the deep rows of this chunk: sum the 32 lane copies (rotated start: conflict-free, fixed order) ----
        __syncwarp();
        double* const recM = M.records0 + (size_t)(C.record_slot + NW) * M.rec_doubles + 2 + n_gs;
        double2* const base = reinterpret_cast<double2*>(smb + L.deep) + (size_t)dim_deep_off * 32;
        const int ne = dim_rows * 2;  // double2 entries: (J, moment pair)
        for (int e = lane; e < ne; e += 32) {
          double2* row = base + (size_t)e * 32;
          double ax = 0.0, ay = 0.0;
          for (int i = 0; i < 32; ++i) {
            const int l = (i + lane) & 31;
            const double2 v = row[l];
            ax += v.x;
            ay += v.y;
            row[l] = make_double2(0.0, 0.0);
          }
          recM[dim_row_off * 4 + e * 2] = ax;
          recM[dim_row_off * 4 + e * 2 + 1] = ay;
        }
        __syncwarp();
      }
    }
    if (warp < NW) {
      // (main warps fall through to the slice fetch; nothing to do)
    }
  }
}

// forward-only pass for the exact per-segment maximum of x (fallback when the a-priori shift bound of a
// spline model was too loose): one block per chunk, plain loads.
template <int DUMMY>
__global__ void __launch_bounds__(256) stream_cta_max_kernel(const ModelDev* __restrict__ Mp) {
  const ModelDev& M = Mp[blockIdx.y];
  __shared__ double red[8];
  const int ncol = M.n_columns, NS = M.n_dims, nlin = M.n_lin_fast;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = blockIdx.x; c < M.n_chunks; c += gridDim.x) {
    const Chunk C = M.chunks[c];
    const long long n = (long long)C.steps * 32 * M.cta_main_warps;
    double mx = -INFINITY;
    for (long long j = threadIdx.x; j < n; j += blockDim.x) {
      const long long p = C.first + j;
      const uint64_t* q = M.columns + (size_t)(p >> 6) * ncol * 64 + (size_t)(p & 63);
      double x = __longlong_as_double((long long)q[(size_t)M.col_static * 64]);
      for (int d = 0; d < NS; ++d) {
        const unsigned long long word = q[(size_t)d * 64];
        const int J = (int)((unsigned)word & 63u);
        const double w = __longlong_as_double((long long)word);
        const double* a = M.tables + (size_t)(M.dims[d].row_off + J) * 4;
        x += fma(fma(a[3], w, a[2]), w * w, fma(a[1], w, a[0]));
      }
      for (int l = 0; l < nlin; ++l) x = fma(M.kc[l * KC_STRIDE], __longlong_as_double((long long)q[(size_t)M.kops[l].col0 * 64]), x);
      mx = fmax(mx, x);
    }
    mx = wmax(mx);
    __syncthreads();
    if (lane == 0) red[warp] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
      double m = red[0];
      for (int i = 1; i < 8; ++i) m = fmax(m, red[i]);
      M.chunk_max[c] = m;
    }
  }
}

template <int NS>
stream_fn pick_stream_cta_for_ns(int nd, int nlin) {
#define GWI_PICK_CTA(ND)                                                  \
  if (nd == ND) {                                                         \
    if (nlin == 0) return (stream_fn)stream_cta_kernel<NS, ND, 0>;        \
    if (nlin == 1) return (stream_fn)stream_cta_kernel<NS, ND, 1>;        \
    if (nlin == 2) return (stream_fn)stream_cta_kernel<NS, ND, 2>;        \
  }
  if (NS >= 1) { GWI_PICK_CTA((NS >= 1 ? 1 : 1)) }
  if (NS >= 2) { GWI_PICK_CTA((NS >= 2 ? 2 : 1)) }
  if (NS >= 3) { GWI_PICK_CTA((NS >= 3 ? 3 : 1)) }
  if (NS >= 4) { GWI_PICK_CTA((NS >= 4 ? 4 : 1)) }
#undef GWI_PICK_CTA
  return nullptr;
}

}  // namespace gwi
