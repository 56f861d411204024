// push_dist.cu -- the fused particle-kernel instantiations of ONE equilibrium distribution (iptcldist), selected
// with -DPIC1DP_DIST=0..3 (0 Maxwellian, 1 two-stream1, 2 two-stream2, 3 bump-on-tail; the tmp2 branches of
// /root/reference/src/pic1dp_interaction.F90:275-326).  Built four times, in parallel, by pic1dp_b200/build.py.
#ifndef PIC1DP_DIST
#error "compile with -DPIC1DP_DIST=0..3"
#endif
#include "push_tables.hpp"

namespace pic1dp {
namespace {
constexpr int DIST = PIC1DP_DIST;

template <bool IRK2, int CFG, bool RC>
PushKernel pick_dep(int dep) {
  switch (dep) {
    case DEP_SMEM_ATOMIC: return k_push<DIST, IRK2, DEP_SMEM_ATOMIC, true, CFG, RC>;
    case DEP_GLOBAL_RED: return k_push<DIST, IRK2, DEP_GLOBAL_RED, true, CFG, RC>;
    case DEP_FIXED: return k_push<DIST, IRK2, DEP_FIXED, true, CFG, RC>;
    default: return k_push<DIST, IRK2, DEP_WARP_PRIVATE, true, CFG, RC>;
  }
}
template <bool IRK2, bool RC>
PushKernel pick_cfg(int dep, int cfg) {
  if (cfg == 1) return pick_dep<IRK2, 1, RC>(dep);
  if (cfg == 9) return pick_dep<IRK2, 9, RC>(dep);
  if (cfg == 25) return pick_dep<IRK2, 25, RC>(dep);
#if PIC1DP_DIST == 2 || PIC1DP_DIST == 3
  if (cfg == 33) return pick_dep<IRK2, 33, RC>(dep);   // PIC1DP_ARITH_TOLERANCE
  if (cfg == 57) return pick_dep<IRK2, 57, RC>(dep);
#endif
  return pick_dep<IRK2, -1, RC>(dep);
}
template <bool IRK2, int CFG>
PushKernel pick_tma_dep(int dep) {
  switch (dep) {
    case DEP_SMEM_ATOMIC: return k_push_tma<DIST, IRK2, DEP_SMEM_ATOMIC, CFG>;
    case DEP_GLOBAL_RED: return k_push_tma<DIST, IRK2, DEP_GLOBAL_RED, CFG>;
    default: return k_push_tma<DIST, IRK2, DEP_WARP_PRIVATE, CFG>;
  }
}
template <bool IRK2, int CFG>
PushKernel pick_cpa_dep(int dep) {
  switch (dep) {
    case DEP_SMEM_ATOMIC: return k_push_cpa<DIST, IRK2, DEP_SMEM_ATOMIC, CFG>;
    case DEP_GLOBAL_RED: return k_push_cpa<DIST, IRK2, DEP_GLOBAL_RED, CFG>;
    default: return k_push_cpa<DIST, IRK2, DEP_WARP_PRIVATE, CFG>;
  }
}
}  // namespace

#define PIC1DP_CAT2(a, b) a##b
#define PIC1DP_CAT(a, b) PIC1DP_CAT2(a, b)

PushKernel PIC1DP_CAT(pick_push_dist, PIC1DP_DIST)(int dep, bool irk2, bool fused, int cfg, bool rc) {
  if (!fused) return irk2 ? k_push<DIST, true, DEP_SMEM_ATOMIC, false, -1> : k_push<DIST, false, DEP_SMEM_ATOMIC, false, -1>;
  if (rc) return irk2 ? pick_cfg<true, true>(dep, cfg) : pick_cfg<false, true>(dep, cfg);
  return irk2 ? pick_cfg<true, false>(dep, cfg) : pick_cfg<false, false>(dep, cfg);
}
PushKernel PIC1DP_CAT(pick_tma_dist, PIC1DP_DIST)(int dep, bool irk2, int cfg) {
  if (cfg == 25) return irk2 ? pick_tma_dep<true, 25>(dep) : pick_tma_dep<false, 25>(dep);
  if (cfg == 9) return irk2 ? pick_tma_dep<true, 9>(dep) : pick_tma_dep<false, 9>(dep);
  return irk2 ? pick_tma_dep<true, 1>(dep) : pick_tma_dep<false, 1>(dep);
}
PushKernel PIC1DP_CAT(pick_cpa_dist, PIC1DP_DIST)(int dep, bool irk2, int cfg) {
  if (cfg == 25) return irk2 ? pick_cpa_dep<true, 25>(dep) : pick_cpa_dep<false, 25>(dep);
  if (cfg == 9) return irk2 ? pick_cpa_dep<true, 9>(dep) : pick_cpa_dep<false, 9>(dep);
  return irk2 ? pick_cpa_dep<true, 1>(dep) : pick_cpa_dep<false, 1>(dep);
}

}  // namespace pic1dp
