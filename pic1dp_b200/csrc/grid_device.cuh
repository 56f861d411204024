// grid_device.cuh -- device-side building blocks of the grid (density / field) work: the argument block, the peer-memory
// all-reduce helpers, rho finalisation and the partial-DFT field solve.  The __global__ kernels built from them are in
// field_kernels.cuh.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "fp_strict.cuh"

namespace pic1dp {


struct GridArgs {
  int nx, nmode, nspecies, ngrids;  // ngrids = CTAs of the particle kernel (private grids per species)
  int deltaf, matrix_path, zero_partials;
  double lx, rnx;
  double Z[4], n[4];
  double *partial;        // [nspecies][ngrids][nx]
  double *red;            // [nred][nx], nred = matrix_path ? nspecies : 1
  double *rho, *E, *mode_re, *mode_im;
  const double *F_re, *F_im, *ginv;  // [nx*nmode] row-major, [nmode]
  const double *F_reT, *F_imT;       // [nmode*nx]: column-major copies read by k_field_synth (many-mode path only)
  double a_im, a_re;      // -1.0/nx, 1.0/nx  (src/pic1dp_field.F90:234, :239)
  double nx_over_lx;      // input_nx / input_lx (src/pic1dp_interaction.F90:77)
  double *energy;
  // peer-memory all-reduce of `red` fused into the reduce kernel (scatter) and the finalize / solve kernels (gather);
  // p2p_nranks == 0: off (single rank, or ncclAllReduce between the kernels)
  int p2p_nranks, p2p_rank;
  unsigned long long *p2p_peer[8];  // exchange buffer of every rank: flags[2][nranks] (padded to 256 B) | data[2][nranks][count]
  unsigned int *p2p_counter;        // local: CTAs of the reduce kernel that have stored their part
  unsigned long long *p2p_timeouts; // local error counter
  // The all-reduce epoch lives in device memory (not in a kernel argument) so that a captured CUDA graph of the step
  // can be replayed: the reduce kernel works on epoch *p2p_epoch_dev + 1 and its last CTA stores that value back
  // after publishing; the gather side, later in stream order, reads the stored value.  Slot parity = epoch & 1.
  unsigned long long *p2p_epoch_dev;
  // optional trace of the rendezvous (pic1dp_gpu_p2p_trace): %globaltimer at publish, wait entry and wait exit,
  // 3 stamps per epoch in a ring of p2p_stamp_cap entries
  unsigned long long *p2p_stamps;
  int p2p_stamp_cap;
};

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ double *p2p_data(unsigned long long *base, int nranks, int count, int parity, int r) {
  const size_t flag_bytes = ((size_t)2 * nranks * 8 + 255) & ~(size_t)255;
  return reinterpret_cast<double *>(reinterpret_cast<char *>(base) + flag_bytes) + ((size_t)parity * nranks + r) * count;
}

// scatter side, end of the kernel: the last CTA publishes this rank's epoch flag in every rank's buffer
__device__ __forceinline__ void p2p_publish(const GridArgs &g, unsigned long long epoch) {
  __threadfence_system();  // my stores are visible system-wide before the counter / flag
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned prev = atomicAdd(g.p2p_counter, 1u);
    if (prev == gridDim.x - 1) {
      *g.p2p_counter = 0;
      __threadfence_system();
      const int parity = (int)(epoch & 1);
      for (int r = 0; r < g.p2p_nranks; r++) {
        unsigned long long *flag = g.p2p_peer[r] + (size_t)parity * g.p2p_nranks + g.p2p_rank;
        asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(epoch) : "memory");
      }
      *g.p2p_epoch_dev = epoch;  // every CTA of this kernel has read the old value by now (it arrived at the counter)
      if (g.p2p_stamps) g.p2p_stamps[(size_t)(epoch % g.p2p_stamp_cap) * 3] = globaltimer_ns();
    }
  }
}

// gather side, start of the kernel: wait (bounded) until every rank's flag shows this epoch; returns false on timeout
__device__ __forceinline__ bool p2p_wait(const GridArgs &g, unsigned long long epoch) {
  __shared__ int s_ok;
  if (threadIdx.x == 0) {
    s_ok = 1;
    if (g.p2p_stamps && blockIdx.x == 0) g.p2p_stamps[(size_t)(epoch % g.p2p_stamp_cap) * 3 + 1] = globaltimer_ns();
  }
  __syncthreads();
  if ((int)threadIdx.x < g.p2p_nranks) {
    const unsigned long long *flag = g.p2p_peer[g.p2p_rank] + (size_t)(epoch & 1) * g.p2p_nranks + threadIdx.x;
    unsigned long long seen = 0;
    long long spins = 0;
    for (;;) {
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(flag) : "memory");
      if (seen >= epoch) break;
      if (++spins > 200000000LL) {  // seconds: a peer died; report instead of hanging the GPU
        s_ok = 0;
        if (blockIdx.x == 0) atomicAdd(g.p2p_timeouts, 1ULL);
        break;
      }
      __nanosleep(20);
    }
  }
  __syncthreads();
  if (g.p2p_stamps && blockIdx.x == 0 && threadIdx.x == 0)
    g.p2p_stamps[(size_t)(epoch % g.p2p_stamp_cap) * 3 + 2] = globaltimer_ns();
  return s_ok != 0;
}

// gather side: the all-reduced value = sum over ranks in rank order (bitwise identical on every rank)
__device__ __forceinline__ double p2p_sum(const GridArgs &g, int idx, int parity) {
  const int count = (g.matrix_path ? g.nspecies : 1) * g.nx;
  double t = p2p_data(g.p2p_peer[g.p2p_rank], g.p2p_nranks, count, parity, 0)[idx];
  for (int r = 1; r < g.p2p_nranks; r++)
    t = dadd(t, p2p_data(g.p2p_peer[g.p2p_rank], g.p2p_nranks, count, parity, r)[idx]);
  return t;
}

// rho from the (all-)reduced grid: charge1 * nx / lx and the full-f offset (:140-148); matrix path :64-78
__device__ __forceinline__ double red_value(const GridArgs &g, int idx, int parity) {
  if (!g.p2p_nranks) return g.red[idx];
  const double t = p2p_sum(g, idx, parity);  // MPI_Allreduce (:132-133), gather half
  g.red[idx] = t;
  return t;
}

__device__ __forceinline__ double finalize_rho(const GridArgs &g, int j, int parity) {
  double rho;
  if (!g.matrix_path) {
    rho = ddiv(dmul(red_value(g, j, parity), g.rnx), g.lx);  // :140-141
    if (!g.deltaf)
      for (int s = 0; s < g.nspecies; s++) rho = dsub(rho, dmul(g.Z[s], g.n[s]));  // :142-148
  } else {
    rho = 0.0;  // :47
    for (int s = 0; s < g.nspecies; s++) {
      double t = red_value(g, s * g.nx + j, parity);
      if (!g.deltaf) t = dsub(t, ddiv(dmul(g.n[s], g.lx), g.rnx));  // :67
      rho = dadd(rho, dmul(g.Z[s], t));                              // VecAXPY :71
    }
    rho = dmul(rho, g.nx_over_lx);  // VecScale :77
  }
  return rho;
}

// Single CTA, 1024 threads.  smem: rho[nx] + 2*nmode mode values.
// SEQ=true : thread m walks j = 0..nx-1 in order (bit-identical to sequential-AIJ MatMultTranspose).
// SEQ=false: one or more warps per mode, lanes stride j, fixed shuffle tree + warp-ordered sum (deterministic).
// FINALIZE: also does k_finalize_rho's work first (one launch less per substep inside step()).
template <bool SEQ, bool FINALIZE>
__device__ __forceinline__ void field_solve_body(const GridArgs &g, double *smem) {
  double *s_rho = smem;
  double *s_re = smem + g.nx;
  double *s_im = s_re + g.nmode;
  const int M = g.nmode, nx = g.nx;
  const unsigned long long epoch = (FINALIZE && g.p2p_nranks) ? *g.p2p_epoch_dev : 0;
  const bool p2p_ok = (FINALIZE && g.p2p_nranks) ? p2p_wait(g, epoch) : true;
  for (int j = threadIdx.x; j < nx; j += blockDim.x) {
    double r;
    if (FINALIZE) {
      r = p2p_ok ? finalize_rho(g, j, (int)(epoch & 1)) : __longlong_as_double(0x7ff8000000000000LL);
      g.rho[j] = r;
    } else {
      r = g.rho[j];
    }
    s_rho[j] = r;
  }
  __syncthreads();
  if (SEQ) {
    for (int m = threadIdx.x; m < M; m += blockDim.x) {
      double sim = 0.0, sre = 0.0;
      for (int j = 0; j < nx; j++) {
        sim = dadd(sim, dmul(g.F_re[(size_t)j * M + m], s_rho[j]));  // MatMultTranspose(F_re, rho) :231
        sre = dadd(sre, dmul(g.F_im[(size_t)j * M + m], s_rho[j]));  // MatMultTranspose(F_im, rho) :236
      }
      s_im[m] = dmul(dmul(sim, g.a_im), g.ginv[m]);  // :234, :246
      s_re[m] = dmul(dmul(sre, g.a_re), g.ginv[m]);  // :239, :243
    }
  } else {
    // G warps share one mode (G = largest power of two <= warps / modes, 1 when there are more modes than warps): with
    // the reference's single kept mode the whole CTA projects it instead of one warp walking all nx cells.  Lanes
    // stride j, fixed shuffle tree per warp, then the G warp sums are added in warp order: a fixed summation tree.
    __shared__ double s_part[32][2];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int G = 1;
    while (2 * G * M <= nw) G *= 2;
    const int per_pass = nw / G, grp = wid / G, sub = wid % G;
    for (int mb = 0; mb < M; mb += per_pass) {
      const int m = mb + grp;
      double sim = 0.0, sre = 0.0;
      if (m < M && grp < per_pass) {
        for (int j = sub * 32 + lane; j < nx; j += 32 * G) {
          sim = dadd(sim, dmul(g.F_re[(size_t)j * M + m], s_rho[j]));
          sre = dadd(sre, dmul(g.F_im[(size_t)j * M + m], s_rho[j]));
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sim = dadd(sim, __shfl_xor_sync(0xffffffffu, sim, o));
        sre = dadd(sre, __shfl_xor_sync(0xffffffffu, sre, o));
      }
      if (lane == 0) {
        s_part[wid][0] = sim;
        s_part[wid][1] = sre;
      }
      __syncthreads();
      if (lane == 0 && sub == 0 && m < M && grp < per_pass) {
        for (int q = 1; q < G; q++) {
          sim = dadd(sim, s_part[wid + q][0]);
          sre = dadd(sre, s_part[wid + q][1]);
        }
        s_im[m] = dmul(dmul(sim, g.a_im), g.ginv[m]);
        s_re[m] = dmul(dmul(sre, g.a_re), g.ginv[m]);
      }
      __syncthreads();
    }
  }
  __syncthreads();
  for (int m = threadIdx.x; m < M; m += blockDim.x) {
    g.mode_re[m] = s_re[m];
    g.mode_im[m] = s_im[m];
  }
  // E = 2 * (F_re . mode_re + F_im . mode_im): MatMult then MatMultAdd, row sums left to right (:251-256)
  for (int j = threadIdx.x; j < nx; j += blockDim.x) {
    double sum = 0.0;
    for (int m = 0; m < M; m++) sum = dadd(sum, dmul(g.F_re[(size_t)j * M + m], s_re[m]));
    for (int m = 0; m < M; m++) sum = dadd(sum, dmul(g.F_im[(size_t)j * M + m], s_im[m]));
    g.E[j] = dmul(sum, 2.0);
  }
}

// (A single-CTA "tail" -- reduce + solve run by the last CTA of the fused particle kernel, one launch per substep -- was
// built and measured in round 2: slower at every size (6.4e6 markers, nx = 192: 0.200 vs 0.177 ms per step; nx = 4096:
// 0.45 vs 0.25 ms): one CTA reading 148 private grids is slower than the 6 .. 128 CTAs of k_reduce_charge plus two
// launch boundaries inside a replayed graph, and its registers spilled in the marker loop.)

}  // namespace pic1dp
