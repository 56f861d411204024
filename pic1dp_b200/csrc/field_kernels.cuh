// field_kernels.cuh -- grid-side kernels of the PIC1D hot path for sm_100a.
//
//  k_reduce_charge : fixed-order sum of the per-CTA private grids + species charge
//                    (/root/reference/src/pic1dp_interaction.F90:81, :126-127; matrix path :52-59)
//  k_finalize_rho  : scale to charge density + full-f offset after the all-reduce (:140-148; matrix path :64-78)
//  k_field_solve   : mode-filtered partial DFT, 1/k, inverse (/root/reference/src/pic1dp_field.F90:231-256).
//                    There is no KSP / tridiagonal solve in the reference: only the kept modes survive.
//  k_field_energy  : |E|_2^2 * lx / nx (/root/reference/src/pic1dp_output.F90:120-123)
//
// The grid is tiny (nx <= a few thousand): these are single- or few-CTA kernels, latency- not bandwidth-bound.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "grid_device.cuh"

namespace pic1dp {

// CTA = 32 cells x 8 warps.  Warp q sums the private grids q, q+8, q+16, ... of its 32 cells in that order (4 loads
// in flight), then warp 0 adds the 8 partial sums in warp order: a fixed summation tree, hence deterministic.
// Peer-memory all-reduce, scatter half: the CTA's reduced values (32 cells x nred grids) are staged in shared memory
// and warp q stores them into slot [parity][my rank] of rank q's exchange buffer -- one coalesced 256-byte NVLink
// store per peer and grid, all peers in parallel (8 warps = the 8 ranks the exchange supports).
__global__ void __launch_bounds__(256) k_reduce_charge(const GridArgs g) {
  __shared__ double s_part[8][33];
  __shared__ double s_out[4][32];  // reduced values of this CTA: [grid (species on the matrix path)][cell]
  const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + lane;
  const unsigned long long epoch = g.p2p_nranks ? *g.p2p_epoch_dev + 1 : 0;  // a new all-reduce
  double c2 = 0.0;
  for (int s = 0; s < g.nspecies; s++) {
    double c1 = 0.0;
    if (j < g.nx) {
      double *ps = g.partial + (size_t)s * g.ngrids * g.nx + j;
      int k = wq;
      for (; k + 24 < g.ngrids; k += 32) {
        const double t0 = ps[(size_t)k * g.nx], t1 = ps[(size_t)(k + 8) * g.nx];
        const double t2 = ps[(size_t)(k + 16) * g.nx], t3 = ps[(size_t)(k + 24) * g.nx];
        c1 = dadd(dadd(dadd(dadd(c1, t0), t1), t2), t3);
      }
      for (; k < g.ngrids; k += 8) c1 = dadd(c1, ps[(size_t)k * g.nx]);
      if (g.zero_partials)
        for (k = wq; k < g.ngrids; k += 8) ps[(size_t)k * g.nx] = 0.0;
    }
    s_part[wq][lane] = c1;
    __syncthreads();
    if (wq == 0 && j < g.nx) {
      double t = s_part[0][lane];
#pragma unroll
      for (int q = 1; q < 8; q++) t = dadd(t, s_part[q][lane]);
      if (g.matrix_path) {  // field_tmp = S^T w per species (:52-59)
        if (g.p2p_nranks) s_out[s][lane] = t;
        else g.red[(size_t)s * g.nx + j] = t;
      } else {
        c2 = dadd(c2, dmul(t, g.Z[s]));   // charge2 += charge1 * Z (:126-127)
      }
    }
    __syncthreads();
  }
  if (wq == 0 && j < g.nx && !g.matrix_path) {
    if (g.p2p_nranks) s_out[0][lane] = c2;
    else g.red[j] = c2;
  }
  if (g.p2p_nranks) {  // MPI_Allreduce (:132-133), scatter half
    __syncthreads();
    const int nred = g.matrix_path ? g.nspecies : 1, count = nred * g.nx, parity = (int)(epoch & 1);
    if (wq < g.p2p_nranks && j < g.nx) {
      double *dst = p2p_data(g.p2p_peer[wq], g.p2p_nranks, count, parity, g.p2p_rank);
      for (int q = 0; q < nred; q++) dst[(size_t)q * g.nx + j] = s_out[q][lane];
    }
    p2p_publish(g, epoch);
  }
}

__global__ void __launch_bounds__(128) k_finalize_rho(const GridArgs g) {
  const unsigned long long epoch = g.p2p_nranks ? *g.p2p_epoch_dev : 0;  // stored by the reduce kernel before this launch
  const bool ok = g.p2p_nranks ? p2p_wait(g, epoch) : true;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < g.nx) g.rho[j] = ok ? finalize_rho(g, j, (int)(epoch & 1)) : __longlong_as_double(0x7ff8000000000000LL);
}

template <bool SEQ, bool FINALIZE>
__global__ void __launch_bounds__(1024) k_field_solve(const GridArgs g) {
  extern __shared__ __align__(16) double smem[];
  field_solve_body<SEQ, FINALIZE>(g, smem);
}

// ---- many-mode field solve (nmode > PIC1DP_FIELD_CTA_MODES): the same arithmetic as k_field_solve<true, *> spread
// over CTAs.  rho is formed beforehand (k_finalize_rho, or set_field / collect_charge).  Both passes keep the
// sequential order of the reference's SeqAIJ products, so TREE and SEQUENTIAL coincide here.  One warp per CTA, so a
// few hundred modes or cells still spread over as many SMs as there are warps.
constexpr int FIELD_MC_THREADS = 32;

// projection: thread m walks j = 0..nx-1 in order (MatMultTranspose, src/pic1dp_field.F90:231, :236); the warp reads
// 32 consecutive entries of a table row per j (coalesced), rho[j] is a broadcast
__global__ void __launch_bounds__(FIELD_MC_THREADS) k_field_project(const GridArgs g) {
  const int m = blockIdx.x * FIELD_MC_THREADS + threadIdx.x;
  if (m >= g.nmode) return;
  const size_t M = (size_t)g.nmode;
  const double *fr = g.F_re + m, *fi = g.F_im + m, *rho = g.rho;
  double sim = 0.0, sre = 0.0;
#pragma unroll 8
  for (int j = 0; j < g.nx; j++) {
    const double r = __ldg(rho + j);
    sim = dadd(sim, dmul(__ldg(fr + j * M), r));
    sre = dadd(sre, dmul(__ldg(fi + j * M), r));
  }
  g.mode_im[m] = dmul(dmul(sim, g.a_im), g.ginv[m]);  // :234, :246
  g.mode_re[m] = dmul(dmul(sre, g.a_re), g.ginv[m]);  // :239, :243
}

// synthesis: thread j sums its row left to right (MatMult then MatMultAdd, :251-256) from the column-major copies, so
// the warp's reads of one column are coalesced; mode_re[m] / mode_im[m] are broadcasts
__global__ void __launch_bounds__(FIELD_MC_THREADS) k_field_synth(const GridArgs g) {
  const int j = blockIdx.x * FIELD_MC_THREADS + threadIdx.x;
  if (j >= g.nx) return;
  const size_t nx = (size_t)g.nx;
  const double *fr = g.F_reT + j, *fi = g.F_imT + j;
  double sum = 0.0;
#pragma unroll 8
  for (int m = 0; m < g.nmode; m++) sum = dadd(sum, dmul(__ldg(fr + m * nx), __ldg(g.mode_re + m)));
#pragma unroll 8
  for (int m = 0; m < g.nmode; m++) sum = dadd(sum, dmul(__ldg(fi + m * nx), __ldg(g.mode_im + m)));
  g.E[j] = dmul(sum, 2.0);
}

// single CTA of 1024 threads
__global__ void __launch_bounds__(1024) k_field_energy(const GridArgs g) {
  __shared__ double s_part[32];
  double s = 0.0;
  for (int j = threadIdx.x; j < g.nx; j += blockDim.x) s = dadd(s, dmul(g.E[j], g.E[j]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s = dadd(s, __shfl_xor_sync(0xffffffffu, s, o));
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = (threadIdx.x < (blockDim.x >> 5)) ? s_part[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s = dadd(s, __shfl_xor_sync(0xffffffffu, s, o));
    if (threadIdx.x == 0) {
      const double nrm = sqrt(s);  // VecNorm(NORM_2)
      *g.energy = ddiv(dmul(dmul(nrm, nrm), g.lx), g.rnx);
    }
  }
}


}  // namespace pic1dp
