// push_tables.hpp -- dispatch tables of the fused particle kernels.
//
// The instantiations of k_push / k_push_tma / k_push_cpa (particle_kernels.cuh) for one iptcldist live in one
// translation unit (push_dist.cu compiled with -DPIC1DP_DIST=0..3), so the four equilibria build in parallel.
// Each unit exports three look-up functions; pic1dp_gpu.cu selects the unit by the run-time iptcldist.
#pragma once
#include "particle_kernels.cuh"

namespace pic1dp {

typedef void (*PushKernel)(const ParticleArgs);

// cfg: -1 generic (switches read at run time), 1 = delta-f nonlinear shape 3/4, 9 = same with power-of-two
// divisors, 25 = same with T = T2 = m = 1 (the reference default input); + 32 = TOLERANCE arithmetic (w path only).
// rc: the recomputed-midpoint forms of step() (fused only; k_push with RC = true)
#define PIC1DP_DECLARE_DIST(D)                                                       \
  PushKernel pick_push_dist##D(int dep, bool irk2, bool fused, int cfg, bool rc);    \
  PushKernel pick_tma_dist##D(int dep, bool irk2, int cfg);                 \
  PushKernel pick_cpa_dist##D(int dep, bool irk2, int cfg);
PIC1DP_DECLARE_DIST(0)
PIC1DP_DECLARE_DIST(1)
PIC1DP_DECLARE_DIST(2)
PIC1DP_DECLARE_DIST(3)
#undef PIC1DP_DECLARE_DIST

inline PushKernel pick_push(int dist, int dep, bool irk2, bool fused, int cfg, bool rc) {
  switch (dist) {
    case 1: return pick_push_dist1(dep, irk2, fused, cfg, rc);
    case 2: return pick_push_dist2(dep, irk2, fused, cfg, rc);
    case 3: return pick_push_dist3(dep, irk2, fused, cfg, rc);
    default: return pick_push_dist0(dep, irk2, fused, cfg, rc);
  }
}
// TMA-pipelined kernels (delta-f nonlinear, fused): cfg in {1, 9, 25}
inline PushKernel pick_tma(int dist, int dep, bool irk2, int cfg) {
  switch (dist) {
    case 1: return pick_tma_dist1(dep, irk2, cfg);
    case 2: return pick_tma_dist2(dep, irk2, cfg);
    case 3: return pick_tma_dist3(dep, irk2, cfg);
    default: return pick_tma_dist0(dep, irk2, cfg);
  }
}
// cp.async-staged kernels (delta-f nonlinear, fused): cfg in {1, 9, 25}
inline PushKernel pick_cpa(int dist, int dep, bool irk2, int cfg) {
  switch (dist) {
    case 1: return pick_cpa_dist1(dep, irk2, cfg);
    case 2: return pick_cpa_dist2(dep, irk2, cfg);
    case 3: return pick_cpa_dist3(dep, irk2, cfg);
    default: return pick_cpa_dist0(dep, irk2, cfg);
  }
}

}  // namespace pic1dp
