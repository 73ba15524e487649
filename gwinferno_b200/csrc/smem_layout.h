// Shared-memory layouts of the two stream kernels, one function each: the kernel carves its dynamic shared memory with
// it, plan_geometry picks the warp count with it and gwi_model_create sizes the launch with it, so a layout change is
// made here and nowhere else.
#pragma once
#include <cuda_runtime.h>

#include "dev_structs.h"

namespace gwi {

// ---- one-role stream kernel (stream.cuh) ---------------------------------------------------------
// tables[rows_total][4] double | dtab: the deep dims' coefficient half-rows replicated 8x, [h][row][lane & 7] double2 |
// kc[n_kops][KC_STRIDE] double | kops[n_kops] KopDev | per warp {
//   msh[mom][rows_total][4] double | deep[deep_rows][mom][2][DEEP_LANES] double2 | gscr[n_gslots][32] double |
//   gacc[mom][n_gslots][32] double }
// Every region is a multiple of 16 bytes (16-byte vector accesses).
// One function for both users: with Ptr = SmemPtr it returns the kernel's region pointers, stepped with typed pointer
// arithmetic (the kernel compiles to the address arithmetic of carving by hand); with Ptr = SmemOffset, byte offsets.
template <class T>
using SmemPtr = T*;
template <class T>
struct SmemOffset {
  size_t bytes;
  GWI_HD SmemOffset operator+(long long n) const { return {bytes + sizeof(T) * (size_t)n}; }
};
template <class T, class U>
GWI_HD_INLINE T* smem_cast(U* p) { return reinterpret_cast<T*>(p); }
template <class T, class U>
GWI_HD inline SmemOffset<T> smem_cast(SmemOffset<U> p) { return {p.bytes}; }

template <template <class> class Ptr>
struct OneRoleLayout {
  Ptr<double> tables;
  Ptr<double2> dtab;
  Ptr<double> kc;
  Ptr<KopDev> kops;
  Ptr<double> msh;  // the region of warp `warp`
  Ptr<double2> deep;
  Ptr<double> gscr, gacc;
  int warp_doubles;  // size of one warp's region
};
static_assert(sizeof(KopDev) % 16 == 0, "KopDev copies must keep the shared layout 16-byte aligned");
template <template <class> class Ptr>
GWI_HD_INLINE OneRoleLayout<Ptr> one_role_layout(Ptr<double> base, int rows_total, int deep_rows, int mom, int n_kops, int n_gslots, int warp) {
  const int deep_entries = deep_rows * 2 * mom;  // double2 accumulators: (row, moment set, pair)
  OneRoleLayout<Ptr> L;
  L.tables = base;
  L.dtab = smem_cast<double2>(L.tables + rows_total * 4);
  L.kc = L.tables + rows_total * 4 + deep_rows * 32;
  L.kops = smem_cast<KopDev>(L.kc + n_kops * KC_STRIDE);
  L.warp_doubles = rows_total * 4 * mom + deep_entries * 2 * DEEP_LANES + n_gslots * 32 * (1 + mom);
  L.msh = smem_cast<double>(L.kops + n_kops) + (size_t)warp * L.warp_doubles;
  L.deep = smem_cast<double2>(L.msh + rows_total * 4 * mom);
  L.gscr = smem_cast<double>(L.deep + deep_entries * DEEP_LANES);
  L.gacc = L.gscr + n_gslots * 32;
  return L;
}
// dynamic shared memory of a block of `warps` warps: where the region of warp `warps` would begin
inline size_t one_role_smem_bytes(int rows_total, int deep_rows, int mom, int n_kops, int n_gslots, int warps) {
  return one_role_layout<SmemOffset>({0}, rows_total, deep_rows, mom, n_kops, n_gslots, warps).msh.bytes;
}

// ---- CTA-cooperative stream kernel (stream_cta.cuh) ----------------------------------------------
constexpr int CTA_NSTAGE = 4;      // staged 64-sample blocks per main warp
constexpr int CTA_MAX_WARPS = 12;  // main + deep warps (launch bound 384 threads => 168 registers; 13 warps make ptxas fall back to 128 + spills)

struct CtaLayout {
  unsigned bars, ctl, tables, dtab, stages, stage_bytes, blk_bytes, deep, total;
  // 16-byte vector accesses everywhere (tables, staged blocks, accumulators)
  GWI_HD bool aligned16() const { return ((ctl | tables | stages | stage_bytes | blk_bytes | deep) & 15u) == 0u; }
};
GWI_HD inline CtaLayout cta_layout(int nw, int ncol, int rows_total, int deep_rows) {
  CtaLayout L;
  L.bars = 0;  // mbarriers: full[nw][NSTAGE] (one per staged block) | ready[NSTAGE] (count nw) | free[NSTAGE] (count n_deep)
  L.ctl = (L.bars + ((unsigned)nw + 2u) * CTA_NSTAGE * 8u + 15u) & ~15u;  // 16 B: slice id broadcast (16-byte aligned: the tables follow)
  L.tables = L.ctl + 16u;
  L.blk_bytes = (unsigned)ncol * 512u;
  L.stage_bytes = L.blk_bytes + 512u;              // + the 64 weights p of the block
  L.dtab = L.tables + (unsigned)rows_total * 32u;  // deep-dim half-rows replicated 8x: [h][r][lane & 7] double2 (conflict-free LDS.128)
  L.stages = (L.dtab + (unsigned)deep_rows * 256u + 127u) & ~127u;
  L.deep = L.stages + (unsigned)nw * CTA_NSTAGE * L.stage_bytes;
  L.total = L.deep + (unsigned)deep_rows * 2u * 32u * 16u;  // double2 [row][moment pair][32 lanes]
  return L;
}

}  // namespace gwi
