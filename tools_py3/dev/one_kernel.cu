#include "../../pic1dp_b200/csrc/particle_kernels.cuh"
using namespace pic1dp;
// the flagship instantiations (bump-on-tail, default fixed-point deposit, unit constants): the stored-midpoint pair of
// the per-substep entry points, then the recomputed-midpoint pair of step()
template __global__ void pic1dp::k_push<3, false, DEP_FIXED, true, 25>(const ParticleArgs);
template __global__ void pic1dp::k_push<3, true, DEP_FIXED, true, 25>(const ParticleArgs);
template __global__ void pic1dp::k_push<3, false, DEP_FIXED, true, 25, true>(const ParticleArgs);
template __global__ void pic1dp::k_push<3, true, DEP_FIXED, true, 25, true>(const ParticleArgs);
