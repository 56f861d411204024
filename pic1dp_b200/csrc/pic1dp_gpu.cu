// pic1dp_gpu.cu -- C ABI (include/pic1dp_gpu.h) and device-resident state of the B200-native PIC1D hot path.
//
// The handle plays the role of the module-global PETSc state of pic1dp_particle / pic1dp_field
// (/root/reference/src/pic1dp_particle.F90:26-58, /root/reference/src/pic1dp_field.F90:27-48):
//   markers : SoA fp64 x, v, w in two buffer sets (A/B) + p.  The RK2 "backup" (VecCopy x3,
//             src/pic1dp_interaction.F90:181-187) is a buffer rotation: substep 1 reads A and writes B,
//             substep 2 reads A (start-of-step) and B (midpoint) and overwrites A.
//   grid    : E, rho, mode_re, mode_im, cos / -sin partial-DFT tables, 1/k -- replicated on every GPU.
//   deposit : per-CTA private grids, reduced in fixed order; one ncclAllReduce(nx doubles) per substep.
// No matrix is ever materialised; no CPU fallback exists.
#include "../../include/pic1dp_gpu.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <nccl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <string>
#include <vector>

#include "diag_kernels.cuh"
#include "field_kernels.cuh"
#include "loader_kernels.cuh"
#include "optimize_host.hpp"
#include "optimize_kernels.cuh"
#include "particle_kernels.cuh"
#include "push_tables.hpp"
#include "rng_kernels.cuh"

using namespace pic1dp;

// LOAD_AUTO: which substeps use the TMA ring (measured, see profiles/r01_ab_experiments.md)
#ifndef PIC1DP_TMA_AUTO_IRK1
#define PIC1DP_TMA_AUTO_IRK1 0
#endif
#ifndef PIC1DP_TMA_AUTO_IRK2
#define PIC1DP_TMA_AUTO_IRK2 0
#endif
static const bool PIC1DP_TMA_AUTO_IRK[2] = {PIC1DP_TMA_AUTO_IRK1 != 0, PIC1DP_TMA_AUTO_IRK2 != 0};
// LOAD_AUTO: which substeps use the cp.async-staged kernel when its ring fits beside the deposit grids
#ifndef PIC1DP_CPA_AUTO_IRK1
#define PIC1DP_CPA_AUTO_IRK1 0
#endif
#ifndef PIC1DP_CPA_AUTO_IRK2
#define PIC1DP_CPA_AUTO_IRK2 0
#endif
static const bool PIC1DP_CPA_AUTO_IRK[2] = {PIC1DP_CPA_AUTO_IRK1 != 0, PIC1DP_CPA_AUTO_IRK2 != 0};

// ------------------------------------------------------------------------------------------------------------
// NCCL is bound at run time (dlopen) and only when nranks > 1, so a single-GPU process never needs it and a
// process that already loaded torch's bundled libnccl.so.2 reuses that copy.
// ------------------------------------------------------------------------------------------------------------
namespace {
struct NcclApi {
  void *so = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) =
      nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  std::string err;
  bool load() {
    if (so) return true;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
      so = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (so) break;
    }
    if (!so) {
      err = std::string("dlopen(libnccl.so.2) failed: ") + dlerror();
      return false;
    }
#define BIND(field, sym)                                           \
  *(void **)(&field) = dlsym(so, sym);                             \
  if (!field) {                                                    \
    err = std::string("dlsym failed: ") + sym;                     \
    return false;                                                  \
  }
    BIND(GetUniqueId, "ncclGetUniqueId");
    BIND(CommInitRank, "ncclCommInitRank");
    BIND(AllReduce, "ncclAllReduce");
    BIND(CommDestroy, "ncclCommDestroy");
    BIND(GetErrorString, "ncclGetErrorString");
#undef BIND
    return true;
  }
};
NcclApi g_nccl;
std::string g_create_err;
}  // namespace

struct Species {
  double *x[2] = {nullptr, nullptr}, *v[2] = {nullptr, nullptr}, *w[2] = {nullptr, nullptr};
  double *p = nullptr;
  int cur = 0;       // buffer set holding the current state
  int bak = 0;       // buffer set holding the start-of-step state (valid between irk=1 and irk=2)
  int64_t np = 0;
  bool loaded = false;
  bool wmax_valid = false;   // d_wmax_hi[s] covers the current deposit source (fixed-point deposit)
  bool pmax_valid = false;   // d_diag_max[2 s] holds max |p| of the current markers (limb histograms)
  SpeciesConst c;
};

struct pic1dp_gpu {
  pic1dp_params p;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t pev[7] = {};
  // launch timing of the fused particle kernels inside step() / push() (pic1dp_gpu_launch_timing_*)
  bool lt_on = false;
  std::vector<cudaEvent_t> lt_ev;   // pairs (before, after)
  std::vector<int> lt_irk;          // irk of each recorded pair
  Species sp[PIC1DP_MAX_SPECIES];
  double *d_E = nullptr, *d_rho = nullptr, *d_mre = nullptr, *d_mim = nullptr;
  double *d_E_start = nullptr;   // field of step()'s first substep, kept for the recomputed midpoint (ParticleArgs::E_start)
  double *d_Fre = nullptr, *d_Fim = nullptr, *d_ginv = nullptr;
  double *d_partial = nullptr, *d_red = nullptr, *d_energy = nullptr;
  void *d_kiss_tab = nullptr;   // KissTables: jump-ahead tables of the device KISS64 (allocated on first use)
  uint64_t *d_sk_state = nullptr;   // SuperKISS64 table + carry advanced by k_superkiss64_table (allocated on first use)
  uint64_t *d_sk_round = nullptr;   // copy of d_sk_state at the start of the current Gaussian round
  // Gaussian marker stream (allocated on first use): one round of raw words, per-CTA accept counts, GaussCtl
  double *d_gauss_words = nullptr;
  unsigned *d_gauss_bcount = nullptr;
  void *d_gauss_ctl = nullptr;
  int64_t gauss_draws = 0, gauss_rounds = 0, gauss_regenerated = 0;   // of the last Gaussian load
  unsigned long long *d_noob = nullptr;
  unsigned *d_wmax_hi = nullptr;              // [species] running max |deposit source| (high words), DEP_FIXED
  unsigned long long *d_dep_overflow = nullptr, *h_dep_overflow = nullptr;  // conversion overflows (+ pinned mirror)

  std::vector<double> h_Fre, h_Fim, h_ginv;
  // diagnostics scratch (allocated on first use)
  double *d_diag_part = nullptr, *d_diag_sums = nullptr, *d_hist = nullptr, *d_hist_out = nullptr;
  int diag_grid = 0, hist_cells = 0, hist_copies = 16, hist_smem_set = -1;
  double *d_hist_all = nullptr;   // output_all: reduced histograms of all species
  __int128 *d_hist_tab = nullptr;   // limb histograms: one 128-bit integer table per CTA, [nsm][3][ncell]
  unsigned *d_diag_max = nullptr;   // [species][2] high words of max |p|, max |w|
  int hist_tab_cells = 0, limb_smem_set = -1;
  bool limb_enabled = true;         // PIC1DP_DIAG_CAS=1: the round-2 CAS.128 histogram kernel instead
  size_t hist_all_cap = 0;
  // marker optimisation (allocated on first use): device scratch of compute_dist_pertb_abs_v, its host copy
  // particle_dist_pertb_abs_v(ispecies, 0:nv-1), and the pinned staging arrays of merge / remove / split
  double *d_dist_part = nullptr;
  int dist_grid = 0, dist_threads = 0, dist_smem_set = -1, dist_cap = 0;
  std::vector<double> h_dist;
  int opt_nv = 0;
  double opt_vmax = 0.0;
  double *stage[4] = {nullptr, nullptr, nullptr, nullptr};
  bool stage_pinned[4] = {false, false, false, false};  // pageable fallback when the pinned allocation is refused
  size_t max_smem = 0;
  int grid = 0, threads = 512, smem_push = 0, smem_dep = 0, dep = 0, nsm = 0, cfg = -1;
  bool use_tma[2] = {false, false};  // per substep (irk = 1, 2)
  int tma_smem[2] = {0, 0};  // dynamic shared memory of the TMA kernels, irk = 1, 2
  bool use_cpa[2] = {false, false};  // cp.async-staged kernel per substep
  int cpa_smem[2] = {0, 0};
  // step() runs the recomputed-midpoint kernel pair (k_push with RC = true): substep 1 stores only w', substep 2 rebuilds
  // x' and v' from the start-of-step state and E_start.  40 + 64 instead of 56 + 80 bytes per marker and step.
  bool recompute = false;
  int smem_rc = 0;   // dynamic shared memory of the RC irk = 2 kernel (second field table)
  bool partial_valid = false;  // a fused push has already deposited into d_partial
  int nred = 1;
  ncclComm_t comm = nullptr;
  // peer-memory all-reduce
  unsigned long long *d_xchg = nullptr;       // my exchange buffer (flags + data), exported over IPC
  unsigned long long *peer_base[8] = {};      // mapped buffers of all ranks (peer_base[rank] == d_xchg)
  unsigned int *d_p2p_counter = nullptr;
  unsigned long long *d_p2p_timeouts = nullptr;
  unsigned long long *d_p2p_epoch = nullptr;  // all-reduce epoch, advanced on the device by k_reduce_charge
  unsigned long long *h_p2p_timeouts = nullptr;  // pinned mirror of d_p2p_timeouts, refreshed by synchronising calls
  unsigned long long *d_p2p_stamps = nullptr; // rendezvous trace ring (pic1dp_gpu_p2p_trace), 3 stamps per epoch
  int p2p_stamp_cap = 0;
  bool p2p_ready = false;
  int64_t p2p_calls = 0;
  // one timestep {push, reduce, solve} x 2 captured as a CUDA graph (pic1dp_gpu_step): valid for the marker counts and
  // buffer rotation it was captured with
  cudaGraphExec_t step_graph = nullptr;
  bool graph_enabled = true;

  int graph_cur[PIC1DP_MAX_SPECIES] = {};
  int64_t graph_np[PIC1DP_MAX_SPECIES] = {};
  int64_t graph_launches = 0, graph_nccl = 0, graph_p2p = 0, graph_replays = 0;
  int64_t launches = 0, nccl_calls = 0, h2d = 0, d2h = 0;
  std::string err;
};

static const char *kErrText[] = {"ok",
                                 "invalid argument or parameter combination",
                                 "CUDA runtime error",
                                 "NCCL error",
                                 "out of memory",
                                 "invalid call sequence",
                                 "marker count exceeds capacity",
                                 "no CUDA device (this library has no CPU fallback)",
                                 "mode not supported for these parameters"};

#define CK(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t e_ = (call);                                                                           \
    if (e_ != cudaSuccess) {                                                                           \
      h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                     \
      return (e_ == cudaErrorMemoryAllocation) ? PIC1DP_ENOMEM : PIC1DP_ECUDA;                         \
    }                                                                                                  \
  } while (0)

#define CKL(h)                                                                                         \
  do {                                                                                                 \
    cudaError_t e_ = cudaGetLastError();                                                               \
    if (e_ != cudaSuccess) {                                                                           \
      (h)->err = std::string("kernel launch: ") + cudaGetErrorString(e_);                              \
      return PIC1DP_ECUDA;                                                                             \
    }                                                                                                  \
    (h)->launches++;                                                                                   \
  } while (0)

static bool is_pow2(double c) {
  if (!(c > 0.0) || !isfinite(c)) return false;
  int e;
  return frexp(c, &e) == 0.5;
}

static void species_const(const pic1dp_params &p, int s, SpeciesConst &c) {
  const double T = p.temperature[s], T2 = p.temperature2[s], m = p.mass[s];
  c.Z = p.charge[s];
  c.m = m;
  c.T = T;
  c.n = p.density[s];
  c.omn = 1.0 - p.density[s];
  c.v0 = p.v0[s];
  c.Tm = T / m;
  c.T2m = T2 / m;
  c.twoTm = 2.0 * T / m;
  c.twoT2m = 2.0 * T2 / m;
  c.sqTm = sqrt(T / m);
  c.sqT2m = sqrt(T2 / m);
  const double divs[8] = {c.m, c.T, c.Tm, c.T2m, c.twoTm, c.twoT2m, c.sqTm, c.sqT2m};
  bool all = true;
  for (double d : divs) all = all && is_pow2(d);
  c.pow2 = all ? 1 : 0;
  c.unit = (c.m == 1.0 && c.T == 1.0 && c.Tm == 1.0 && c.T2m == 1.0 && c.twoTm == 2.0 && c.twoT2m == 2.0 &&
            c.sqTm == 1.0 && c.sqT2m == 1.0) ? 1 : 0;
  // PIC1DP_ARITH_TOLERANCE coefficients
  c.tolA = c.n / (c.Tm * c.sqTm);
  c.tolB = c.omn / (c.T2m * c.sqT2m);
  c.tolC = c.n / c.sqTm;
  c.tolD = c.omn / c.sqT2m;
  c.tolh1 = 1.0 / c.twoTm;
  c.tolh2 = 1.0 / c.twoT2m;
  c.tolk2 = 2.0 * c.v0 / c.Tm;
  c.tolmT = c.m / c.T;
  c.Zm = c.Z / c.m;
  c.i_m = 1.0 / c.m;
  c.i_T = 1.0 / c.T;
  c.i_Tm = 1.0 / c.Tm;
  c.i_T2m = 1.0 / c.T2m;
  c.i_twoTm = 1.0 / c.twoTm;
  c.i_twoT2m = 1.0 / c.twoT2m;
  c.i_sqTm = 1.0 / c.sqTm;
  c.i_sqT2m = 1.0 / c.sqT2m;
}

// ---- kernel dispatch tables: the fused-kernel instantiations live in push_dist.cu, compiled once per iptcldist
// (4 translation units built in parallel); see push_tables.hpp ----
static PushKernel pick_deposit(int dep, bool deposit) {
  if (!deposit) return k_deposit<DEP_SMEM_ATOMIC, false>;
  switch (dep) {
    case DEP_SMEM_ATOMIC: return k_deposit<DEP_SMEM_ATOMIC, true>;
    case DEP_GLOBAL_RED: return k_deposit<DEP_GLOBAL_RED, true>;
    case DEP_FIXED: return k_deposit<DEP_FIXED, true>;
    default: return k_deposit<DEP_WARP_PRIVATE, true>;
  }
}

// shared-memory deposit grids of nx doubles each (the atomic deposit keeps one grid of {left, right} pairs)
static int dep_grids(int dep, int threads) {
  return dep == DEP_WARP_PRIVATE ? threads / 32 : ((dep == DEP_SMEM_ATOMIC || dep == DEP_FIXED) ? 2 : 0);
}

// ---- public API -----------------------------------------------------------------------------------------
extern "C" {

int pic1dp_gpu_abi_version(void) { return PIC1DP_ABI_VERSION; }

const char *pic1dp_gpu_strerror(int code) {
  if (code < 0 || code > PIC1DP_EUNSUPPORTED) return "unknown error";
  return kErrText[code];
}

const char *pic1dp_gpu_last_error(const pic1dp_gpu_t *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

void pic1dp_gpu_params_default(pic1dp_params *p) {
  memset(p, 0, sizeof(*p));
  p->abi_version = PIC1DP_ABI_VERSION;
  p->struct_bytes = (int32_t)sizeof(pic1dp_params);
  p->nx = 192;
  p->nmode = 1;
  p->modes[0] = 1;
  p->lx = 2.0 * 3.1415926535897932384626 / 0.36;
  p->dt = 0.05;
  p->nspecies = 1;
  p->charge[0] = -1.0;
  p->mass[0] = 1.0;
  p->temperature[0] = 1.0;
  p->temperature2[0] = 1.0;
  p->density[0] = 0.9;
  p->v0[0] = 5.0;
  p->iptcldist = 3;
  p->deltaf = 1;
  p->linear = 0;
  p->iptclshape = 4;
  p->capacity = 6400000;
  p->device = 0;
  p->rank = 0;
  p->nranks = 1;
  p->deposit_mode = PIC1DP_DEPOSIT_AUTO;
  p->field_mode = PIC1DP_FIELD_TREE;
  p->fuse = 1;
}

static int validate(const pic1dp_params *p, std::string &err) {
  if (!p) { err = "params is NULL"; return PIC1DP_EINVAL; }
  if (p->abi_version != PIC1DP_ABI_VERSION || p->struct_bytes != (int32_t)sizeof(pic1dp_params)) {
    err = "ABI mismatch: fill params with pic1dp_gpu_params_default() of this library";
    return PIC1DP_EINVAL;
  }
  if (p->nx < 2 || p->nx > (1 << 20)) { err = "nx out of range"; return PIC1DP_EINVAL; }
  if (p->nmode < 1 || p->nmode > PIC1DP_MAX_MODES) { err = "nmode out of range"; return PIC1DP_EINVAL; }
  for (int m = 0; m < p->nmode; m++)
    if (p->modes[m] == 0) { err = "mode number 0 has no 1/k"; return PIC1DP_EINVAL; }
  if (p->nspecies < 1 || p->nspecies > PIC1DP_MAX_SPECIES) { err = "nspecies out of range"; return PIC1DP_EINVAL; }
  if (!(p->lx > 0.0) || !(p->dt > 0.0)) { err = "lx and dt must be positive"; return PIC1DP_EINVAL; }
  if (p->iptcldist < 0 || p->iptcldist > 3) { err = "iptcldist must be 0..3"; return PIC1DP_EINVAL; }
  if (p->iptclshape < 1 || p->iptclshape > 4) { err = "iptclshape must be 1..4"; return PIC1DP_EINVAL; }
  if ((p->deltaf != 0 && p->deltaf != 1) || (p->linear != 0 && p->linear != 1)) {
    err = "deltaf and linear must be 0 or 1";
    return PIC1DP_EINVAL;
  }
  // src/pic1dp_input.F90:301-307
  if (p->linear == 1 && p->deltaf == 0) { err = "case of input_linear = 1 and input_deltaf = 0 not implemented"; return PIC1DP_EINVAL; }
  if (p->capacity < 1) { err = "capacity must be >= 1"; return PIC1DP_EINVAL; }
  if (p->nranks < 1 || p->rank < 0 || p->rank >= p->nranks) { err = "bad rank/nranks"; return PIC1DP_EINVAL; }
  for (int s = 0; s < p->nspecies; s++)
    if (!(p->mass[s] > 0.0) || !(p->temperature[s] > 0.0) || !(p->temperature2[s] > 0.0)) {
      err = "mass and temperatures must be positive";
      return PIC1DP_EINVAL;
    }
  if (p->deposit_mode < 0 || p->deposit_mode > 4 || p->field_mode < 0 || p->field_mode > 1 || p->load_path < 0 ||
      p->load_path > 3 || p->arith_mode < 0 || p->arith_mode > 1) {
    err = "bad deposit_mode / field_mode / load_path / arith_mode";
    return PIC1DP_EINVAL;
  }
  return PIC1DP_OK;
}

int pic1dp_gpu_destroy(pic1dp_gpu_t *h) {
  if (!h) return PIC1DP_OK;
  cudaSetDevice(h->p.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
  for (int s = 0; s < PIC1DP_MAX_SPECIES; s++) {
    Species &S = h->sp[s];
    for (int b = 0; b < 2; b++) {
      if (S.x[b]) cudaFree(S.x[b]);
      if (S.v[b] && (b == 0 || S.v[1] != S.v[0])) cudaFree(S.v[b]);
      if (S.w[b] && (b == 0 || S.w[1] != S.w[0])) cudaFree(S.w[b]);
    }
    if (S.p) cudaFree(S.p);
  }
  double *bufs[] = {h->d_E, h->d_E_start, h->d_rho, h->d_mre, h->d_mim, h->d_Fre, h->d_Fim, h->d_ginv, h->d_partial, h->d_red, h->d_energy,
                    h->d_diag_part, h->d_diag_sums, h->d_hist, h->d_hist_out, h->d_dist_part, h->d_hist_all};
  for (double *b : bufs)
    if (b) cudaFree(b);
  for (int q = 0; q < 4; q++)
    if (h->stage[q]) {
      if (h->stage_pinned[q]) cudaFreeHost(h->stage[q]);
      else free(h->stage[q]);
    }
  if (h->d_noob) cudaFree(h->d_noob);
  if (h->d_kiss_tab) cudaFree(h->d_kiss_tab);
  if (h->d_sk_state) cudaFree(h->d_sk_state);
  if (h->d_sk_round) cudaFree(h->d_sk_round);
  if (h->d_gauss_words) cudaFree(h->d_gauss_words);
  if (h->d_gauss_bcount) cudaFree(h->d_gauss_bcount);
  if (h->d_gauss_ctl) cudaFree(h->d_gauss_ctl);
  if (h->d_wmax_hi) cudaFree(h->d_wmax_hi);
  if (h->d_dep_overflow) cudaFree(h->d_dep_overflow);
  if (h->d_hist_tab) cudaFree(h->d_hist_tab);
  if (h->d_diag_max) cudaFree(h->d_diag_max);

  if (h->h_dep_overflow) cudaFreeHost(h->h_dep_overflow);
  for (int r = 0; r < 8; r++)
    if (h->peer_base[r] && h->peer_base[r] != h->d_xchg) cudaIpcCloseMemHandle(h->peer_base[r]);
  if (h->d_xchg) cudaFree(h->d_xchg);
  if (h->d_p2p_counter) cudaFree(h->d_p2p_counter);
  if (h->d_p2p_timeouts) cudaFree(h->d_p2p_timeouts);
  if (h->d_p2p_epoch) cudaFree(h->d_p2p_epoch);
  if (h->h_p2p_timeouts) cudaFreeHost(h->h_p2p_timeouts);
  if (h->d_p2p_stamps) cudaFree(h->d_p2p_stamps);
  if (h->step_graph) cudaGraphExecDestroy(h->step_graph);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  for (cudaEvent_t e : h->pev)
    if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : h->lt_ev) cudaEventDestroy(e);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return PIC1DP_OK;
}

static int create_impl(pic1dp_gpu_t *h) {
  const pic1dp_params &p = h->p;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    h->err = "no CUDA device visible";
    return PIC1DP_ENODEVICE;
  }
  if (p.device < 0 || p.device >= ndev) {
    h->err = "device ordinal out of range";
    return PIC1DP_EINVAL;
  }
  CK(cudaSetDevice(p.device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, p.device));
  h->nsm = prop.multiProcessorCount;
  h->graph_enabled = p.no_step_graph == 0 && !getenv("PIC1DP_NO_GRAPH");
  h->limb_enabled = !getenv("PIC1DP_DIAG_CAS");

  CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CK(cudaEventCreate(&h->ev0));
  CK(cudaEventCreate(&h->ev1));
  for (int i = 0; i < 7; i++) CK(cudaEventCreate(&h->pev[i]));

  const int nx = p.nx, M = p.nmode;
  const size_t max_smem = prop.sharedMemPerBlockOptin;
  h->max_smem = max_smem;
  // ---- deposit strategy and launch geometry ----
  // Kernels are compiled for <= 64 registers (launch bound 1024 threads), so an SM holds up to 1024 threads =
  // 32 warps.  Shared/global-atomic deposits run 2 CTAs x 512 threads; the warp-private deposit needs one grid
  // per warp in shared memory, so its CTA is as large as fits (multiple of 4 warps, <= 32).
  int dep = p.deposit_mode;
  auto smem_need = [&](int d, int thr) { return (size_t)8 * (((nx + 1) & ~1) + (size_t)nx * dep_grids(d, thr)); };
  auto warp_private_threads = [&]() {
    int w = (int)((max_smem - 8) / ((size_t)nx * 8)) - 1;
    if (w > PIC1DP_MAXTHREADS / 32) w = PIC1DP_MAXTHREADS / 32;
    if (w >= 4) w &= ~3;
    return w * 32;
  };
  if (dep == PIC1DP_DEPOSIT_AUTO) {
    // measured on B200 (profiles/r01_config_sweep.md): the warp-private deposit wins on small grids (nx <= 256: more
    // intra-CTA contention for the CAS loop, and 32 private grids still fit), the 128-bit-CAS deposit elsewhere;
    // RED.ADD.F64 to L2 only when the pair grid does not fit in shared memory.
    // Round 2 (profiles/r02_ab_experiments.md, calls r02x / r02y / r02z / r02h): the fixed-point deposit with native
    // 32-bit adds beats the CAS deposit (strict arithmetic, 1e8 markers, nx = 1024: 2.135 vs 2.25 ms per step) and, on
    // small grids, the warp-private one (6.4e6 markers, nx = 192: 0.162 vs 0.177 ms; the native add resolves collisions
    // in the unit instead of in a retry loop), and it is bitwise reproducible.  With the tolerance arithmetic the CAS
    // deposit is 2 % ahead in a 20-step burst at nx = 1024 (2.18 vs 2.22 ms) but 8 % behind once the part runs under
    // its power cap, which is where a real run lives (500 steps: 2.27 vs 2.47 ms): fewer instructions win there.
    // The fixed-point quantum grows with the markers a CTA handles, so AUTO keeps it to <= 2^20 markers per CTA
    // (1.5e8 per GPU).
    const bool fixed_ok = smem_need(DEP_FIXED, 512) <= max_smem && p.capacity <= ((int64_t)1 << 20) * h->nsm &&
                          !getenv("PIC1DP_AUTO_NO_FIXED");
    if (fixed_ok)
      dep = DEP_FIXED;
    else if (nx <= 256 && warp_private_threads() >= 1024)
      dep = DEP_WARP_PRIVATE;
    else if (smem_need(DEP_SMEM_ATOMIC, 512) <= max_smem)
      dep = DEP_SMEM_ATOMIC;
    else
      dep = DEP_GLOBAL_RED;
  }
  // the warp-private deposit needs one nx-sized shared-memory grid per warp; when fewer than 8 warps fit (nx >~ 2900)
  // the request degrades to the other bitwise-deterministic strategy, the fixed-point pair grid, instead of failing
  if (dep == DEP_WARP_PRIVATE && warp_private_threads() < 256) dep = DEP_FIXED;
  // atomic deposits: one CTA of 1024 threads per SM measured 0.7% faster than 2 x 512 at nx = 1024 (half as many
  // private grids to reduce); small grids keep 2 x 512 to halve the contention on each shared grid
  h->threads = (dep == DEP_WARP_PRIVATE) ? warp_private_threads()
                                         : (nx >= 512 ? PIC1DP_MAXTHREADS : PIC1DP_MAXTHREADS / 2);
  // large grids: when only one CTA's shared memory fits per SM, make that CTA as large as the SM allows
  if (dep != DEP_WARP_PRIVATE &&
      2 * (smem_need(dep, h->threads) + 1024) > (size_t)prop.sharedMemPerMultiprocessor)
    h->threads = PIC1DP_MAXTHREADS;
  if (p.load_path == PIC1DP_LOAD_TMA && dep != DEP_WARP_PRIVATE && dep != DEP_FIXED && h->threads > 512)
    h->threads = 512;  // the TMA-ring kernels are 512-thread CTAs and share the persistent grid with the direct ones
  if (const char *e = getenv("PIC1DP_EXP_THREADS")) {  // experiment hook: CTA size of the atomic-deposit kernels
    const int t = atoi(e);
    if (dep != DEP_WARP_PRIVATE && t >= 64 && t <= PIC1DP_MAXTHREADS && t % 32 == 0) h->threads = t;
  }
  if (h->threads < 32 || smem_need(dep, h->threads) > max_smem) {
    h->err = "shared-memory grid does not fit for this nx with the requested deposit_mode";
    return PIC1DP_EUNSUPPORTED;
  }
  h->dep = dep;
  h->smem_push = (int)smem_need(dep, h->threads);
  h->smem_dep = (int)((size_t)nx * 8 * dep_grids(dep, h->threads));
  h->cfg = (p.deltaf == 1 && p.linear == 0 && p.iptclshape >= 3) ? 1 : -1;
  {
    int per_sm_min = 1 << 30;
    // recomputed-midpoint pair of step(): its irk = 2 kernel holds the field of both substeps.  Used where the rest of the
    // substep is as in the reference's shape-4 loop (no compute_shape_x between the substeps reads the midpoint x) and
    // where the second table keeps the residency of the stored-midpoint kernels (not at nx = 8192 with the pair grid).
    h->smem_rc = h->smem_push + 8 * ((nx + 1) & ~1);
    bool rc_ok = p.fuse != 0 && p.iptclshape == 4 && (size_t)h->smem_rc <= max_smem;
    int per_sm_rc = 1 << 30;
    const int cfgs[6] = {-1, 1, 9, 25, 33, 57};
    for (int irk2 = 0; irk2 < 2; irk2++)
      for (int fused = 0; fused < 2; fused++)
        for (int ci = 0; ci < 6; ci++) {
          PushKernel k = pick_push(p.iptcldist, dep, irk2 == 1, fused == 1, cfgs[ci], false);
          CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_push));
          int per_sm = 0;
          CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, h->threads, h->smem_push));
          if (fused && per_sm < per_sm_min) per_sm_min = per_sm;
          if (fused && rc_ok) {
            const int sm = irk2 ? h->smem_rc : h->smem_push;
            k = pick_push(p.iptcldist, dep, irk2 == 1, true, cfgs[ci], true);
            CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, sm));
            CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, h->threads, sm));
            if (per_sm < per_sm_rc) per_sm_rc = per_sm;
          }
        }
    if (per_sm_min < 1) per_sm_min = 1;
    // TMA-pipelined variant (2-stage ring of 2*threads markers): usable when it reaches the same residency.
    // load_path TMA uses it for both substeps, AUTO only where it measured faster (profiles/r01_ab_experiments.md).
    h->use_tma[0] = h->use_tma[1] = false;
    if (h->cfg == 1 && p.load_path != PIC1DP_LOAD_DIRECT && dep != DEP_WARP_PRIVATE && dep != DEP_FIXED && h->threads == 512) {
      const int tthr = 512;
      for (int irk2 = 0; irk2 < 2; irk2++) {
        const size_t ring = (size_t)2 * (irk2 ? 7 : 4) * (2 * tthr) * 8 + 64;
        const size_t need = 8 * (((size_t)(nx + 1) & ~(size_t)1) + (((size_t)nx * dep_grids(dep, tthr) + 1) & ~(size_t)1)) + ring;
        h->tma_smem[irk2] = (int)need;
        bool ok = need <= max_smem;
        const int cfgs3[3] = {1, 9, 25};
        for (int ci = 0; ci < 3 && ok; ci++) {
          PushKernel k = pick_tma(p.iptcldist, dep, irk2 == 1, cfgs3[ci]);
          CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
          int per_sm = 0;
          CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, tthr, need));
          if (per_sm < per_sm_min) ok = false;  // fewer resident CTAs than the direct kernel: not worth it
        }
        const bool want = (p.load_path == PIC1DP_LOAD_TMA) || (p.load_path == PIC1DP_LOAD_AUTO && PIC1DP_TMA_AUTO_IRK[irk2]);
        h->use_tma[irk2] = ok && want;
      }
      if (p.load_path == PIC1DP_LOAD_TMA && !h->use_tma[0] && !h->use_tma[1]) {
        h->err = "load_path = TMA: the shared-memory ring does not fit beside the deposit grids for this nx";
        return PIC1DP_EUNSUPPORTED;
      }
    } else if (p.load_path == PIC1DP_LOAD_TMA) {
      h->err = "load_path = TMA needs a delta-f nonlinear run with an atomic deposit mode";
      return PIC1DP_EUNSUPPORTED;
    }
    // cp.async-staged variant: same CTA shape as the direct kernel plus a ring of 2 stages x NARR x threads x 16 B
    h->use_cpa[0] = h->use_cpa[1] = false;
    if (h->cfg == 1 && dep != DEP_FIXED && (p.load_path == PIC1DP_LOAD_CPASYNC || p.load_path == PIC1DP_LOAD_AUTO)) {
      for (int irk2 = 0; irk2 < 2; irk2++) {
        const size_t ring = (size_t)2 * (irk2 ? 7 : 4) * h->threads * 16;
        const size_t need = 8 * (((size_t)(nx + 1) & ~(size_t)1) + (((size_t)nx * dep_grids(dep, h->threads) + 1) & ~(size_t)1)) + ring;
        h->cpa_smem[irk2] = (int)need;
        bool ok = need <= max_smem;
        const int cfgs3[3] = {1, 9, 25};
        for (int ci = 0; ci < 3 && ok; ci++) {
          PushKernel k = pick_cpa(p.iptcldist, dep, irk2 == 1, cfgs3[ci]);
          CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
          int per_sm = 0;
          CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, h->threads, need));
          if (per_sm < per_sm_min) ok = false;
        }
        const bool want = (p.load_path == PIC1DP_LOAD_CPASYNC) || PIC1DP_CPA_AUTO_IRK[irk2];
        h->use_cpa[irk2] = ok && want;
      }
      if (p.load_path == PIC1DP_LOAD_CPASYNC && !h->use_cpa[0] && !h->use_cpa[1]) {
        h->err = "load_path = CPASYNC: the shared-memory ring does not fit beside the deposit grids for this nx";
        return PIC1DP_EUNSUPPORTED;
      }
    } else if (p.load_path == PIC1DP_LOAD_CPASYNC) {
      h->err = "load_path = CPASYNC needs a delta-f nonlinear run";
      return PIC1DP_EUNSUPPORTED;
    }
    h->grid = h->nsm * per_sm_min;  // persistent grid: every CTA resident, private grid per CTA
    // the RC pair replaces the direct kernels only (the TMA / cp.async rings keep the stored midpoint)
    h->recompute = rc_ok && per_sm_rc >= per_sm_min && !h->use_tma[0] && !h->use_tma[1] && !h->use_cpa[0] && !h->use_cpa[1];
  }
  CK(cudaFuncSetAttribute(pick_deposit(dep, true), cudaFuncAttributeMaxDynamicSharedMemorySize,
                          h->smem_dep > 0 ? h->smem_dep : 8));
  CK(cudaFuncSetAttribute(k_field_solve<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (nx + 2 * M) * 8));
  CK(cudaFuncSetAttribute(k_field_solve<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (nx + 2 * M) * 8));
  CK(cudaFuncSetAttribute(k_field_solve<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (nx + 2 * M) * 8));
  CK(cudaFuncSetAttribute(k_field_solve<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (nx + 2 * M) * 8));

  // ---- markers ----
  const size_t cap = ((size_t)p.capacity + 1) & ~(size_t)1;  // even, for 128-bit accesses
  for (int s = 0; s < p.nspecies; s++) {
    Species &S = h->sp[s];
    species_const(p, s, S.c);
    CK(cudaMalloc(&S.x[0], cap * 8));
    CK(cudaMalloc(&S.x[1], cap * 8));
    CK(cudaMalloc(&S.v[0], cap * 8));
    if (p.linear) S.v[1] = S.v[0]; else CK(cudaMalloc(&S.v[1], cap * 8));  // linear: v is never written (:335)
    CK(cudaMalloc(&S.w[0], cap * 8));
    if (!p.deltaf) S.w[1] = S.w[0]; else CK(cudaMalloc(&S.w[1], cap * 8));  // full-f: w is never written (:266)
    CK(cudaMalloc(&S.p, cap * 8));
  }
  // ---- grid ----
  h->nred = (p.iptclshape <= 2) ? p.nspecies : 1;
  CK(cudaMalloc(&h->d_E, (size_t)nx * 8));
  CK(cudaMalloc(&h->d_E_start, (size_t)nx * 8));
  CK(cudaMalloc(&h->d_rho, (size_t)nx * 8));
  CK(cudaMalloc(&h->d_mre, (size_t)M * 8));
  CK(cudaMalloc(&h->d_mim, (size_t)M * 8));
  CK(cudaMalloc(&h->d_Fre, (size_t)nx * M * 8));
  CK(cudaMalloc(&h->d_Fim, (size_t)nx * M * 8));
  CK(cudaMalloc(&h->d_ginv, (size_t)M * 8));
  CK(cudaMalloc(&h->d_partial, (size_t)p.nspecies * h->grid * nx * 8));
  CK(cudaMalloc(&h->d_red, (size_t)h->nred * nx * 8));
  CK(cudaMalloc(&h->d_energy, 8));
  CK(cudaMalloc(&h->d_noob, 8));
  CK(cudaMalloc(&h->d_wmax_hi, PIC1DP_MAX_SPECIES * 4));
  CK(cudaMemsetAsync(h->d_wmax_hi, 0, PIC1DP_MAX_SPECIES * 4, h->stream));
  CK(cudaMalloc(&h->d_dep_overflow, 8));
  CK(cudaMemsetAsync(h->d_dep_overflow, 0, 8, h->stream));
  CK(cudaMallocHost(&h->h_dep_overflow, 8));
  *h->h_dep_overflow = 0;

  // ---- field operators (src/pic1dp_field.F90:158-210), evaluated on the host with libm exactly as written ----
  const double PETSC_PI = 3.14159265358979323846264338327950288419716939937510582;
  h->h_Fre.resize((size_t)nx * M);
  h->h_Fim.resize((size_t)nx * M);
  h->h_ginv.resize(M);
  for (int m = 0; m < M; m++) h->h_ginv[m] = 1.0 / (2.0 * PETSC_PI / p.lx * (double)p.modes[m]);  // :166
  for (int j = 0; j < nx; j++)
    for (int m = 0; m < M; m++) {
      const double arg = 2.0 * PETSC_PI / (double)nx * (double)p.modes[m] * (double)j;  // :188, :196
      h->h_Fre[(size_t)j * M + m] = cos(arg);
      h->h_Fim[(size_t)j * M + m] = -sin(arg);
    }
  CK(cudaMemcpyAsync(h->d_Fre, h->h_Fre.data(), (size_t)nx * M * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_Fim, h->h_Fim.data(), (size_t)nx * M * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->d_ginv, h->h_ginv.data(), (size_t)M * 8, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return PIC1DP_OK;
}

int pic1dp_gpu_create(const pic1dp_params *p, pic1dp_gpu_t **out) {
  if (!out) { g_create_err = "out is NULL"; return PIC1DP_EINVAL; }
  *out = nullptr;
  int rc = validate(p, g_create_err);
  if (rc) return rc;
  pic1dp_gpu_t *h = new pic1dp_gpu();
  h->p = *p;
  rc = create_impl(h);
  if (rc) {
    g_create_err = h->err;
    pic1dp_gpu_destroy(h);
    return rc;
  }
  *out = h;
  return PIC1DP_OK;
}

int pic1dp_gpu_comm_unique_id(uint8_t id[PIC1DP_UNIQUE_ID_BYTES]) {
  if (!id) return PIC1DP_EINVAL;
  if (!g_nccl.load()) { g_create_err = g_nccl.err; return PIC1DP_ENCCL; }
  ncclUniqueId u;
  static_assert(sizeof(ncclUniqueId) == PIC1DP_UNIQUE_ID_BYTES, "ncclUniqueId size");
  ncclResult_t r = g_nccl.GetUniqueId(&u);
  if (r != ncclSuccess) { g_create_err = g_nccl.GetErrorString(r); return PIC1DP_ENCCL; }
  memcpy(id, &u, sizeof(u));
  return PIC1DP_OK;
}

int pic1dp_gpu_comm_init(pic1dp_gpu_t *h, const uint8_t id[PIC1DP_UNIQUE_ID_BYTES]) {
  if (!h || !id) return PIC1DP_EINVAL;
  if (h->p.nranks == 1) return PIC1DP_OK;
  if (!g_nccl.load()) { h->err = g_nccl.err; return PIC1DP_ENCCL; }
  CK(cudaSetDevice(h->p.device));
  ncclUniqueId u;
  memcpy(&u, id, sizeof(u));
  ncclResult_t r = g_nccl.CommInitRank(&h->comm, h->p.nranks, u, h->p.rank);
  if (r != ncclSuccess) { h->err = std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r); return PIC1DP_ENCCL; }
  // NCCL sets up its channels lazily on the first collective (hundreds of ms): do that here, not inside a timestep
  r = g_nccl.AllReduce(h->d_energy, h->d_energy, 1, ncclDouble, ncclSum, h->comm, h->stream);
  if (r != ncclSuccess) { h->err = std::string("ncclAllReduce (warm-up): ") + g_nccl.GetErrorString(r); return PIC1DP_ENCCL; }
  CK(cudaStreamSynchronize(h->stream));
  return PIC1DP_OK;
}

static size_t xchg_bytes(const pic1dp_gpu_t *h) {
  const size_t flag_bytes = ((size_t)2 * h->p.nranks * 8 + 255) & ~(size_t)255;
  return flag_bytes + (size_t)2 * h->p.nranks * h->nred * h->p.nx * 8;
}

int pic1dp_gpu_p2p_export(pic1dp_gpu_t *h, uint8_t handle[PIC1DP_IPC_HANDLE_BYTES]) {
  if (!h || !handle) return PIC1DP_EINVAL;
  if (h->p.nranks < 2 || h->p.nranks > 8) { h->err = "p2p all-reduce needs 2..8 ranks"; return PIC1DP_EUNSUPPORTED; }
  CK(cudaSetDevice(h->p.device));
  if (!h->d_xchg) {
    CK(cudaMalloc(&h->d_xchg, xchg_bytes(h)));
    CK(cudaMemset(h->d_xchg, 0, xchg_bytes(h)));
    CK(cudaMalloc(&h->d_p2p_counter, 4));
    CK(cudaMemset(h->d_p2p_counter, 0, 4));
    CK(cudaMalloc(&h->d_p2p_timeouts, 8));
    CK(cudaMemset(h->d_p2p_timeouts, 0, 8));
    CK(cudaMalloc(&h->d_p2p_epoch, 8));
    CK(cudaMemset(h->d_p2p_epoch, 0, 8));
    CK(cudaMallocHost(&h->h_p2p_timeouts, 8));
    *h->h_p2p_timeouts = 0;
  }
  static_assert(sizeof(cudaIpcMemHandle_t) == PIC1DP_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
  cudaIpcMemHandle_t ipc;
  CK(cudaIpcGetMemHandle(&ipc, h->d_xchg));
  memcpy(handle, &ipc, sizeof(ipc));
  return PIC1DP_OK;
}

int pic1dp_gpu_p2p_import(pic1dp_gpu_t *h, const uint8_t *all_handles) {
  if (!h || !all_handles) return PIC1DP_EINVAL;
  if (!h->d_xchg) { h->err = "p2p_import before p2p_export"; return PIC1DP_ESTATE; }
  CK(cudaSetDevice(h->p.device));
  for (int r = 0; r < h->p.nranks; r++) {
    if (r == h->p.rank) {
      h->peer_base[r] = h->d_xchg;
      continue;
    }
    cudaIpcMemHandle_t ipc;
    memcpy(&ipc, all_handles + (size_t)r * PIC1DP_IPC_HANDLE_BYTES, sizeof(ipc));
    void *ptr = nullptr;
    CK(cudaIpcOpenMemHandle(&ptr, ipc, cudaIpcMemLazyEnablePeerAccess));
    h->peer_base[r] = (unsigned long long *)ptr;
  }
  h->p2p_ready = true;
  return PIC1DP_OK;
}

// A peer whose flag never arrives makes the gather side fill rho / E with NaN and bump d_p2p_timeouts.  Every call that
// synchronises queues a copy of that counter before its sync and turns a non-zero count into PIC1DP_ENCCL, so a dead
// peer is reported by the next get_field / output_* / sync instead of silently poisoning the markers.
static void p2p_queue_timeout_read(pic1dp_gpu_t *h) {
  if (h->p2p_ready && h->h_p2p_timeouts)
    cudaMemcpyAsync(h->h_p2p_timeouts, h->d_p2p_timeouts, 8, cudaMemcpyDeviceToHost, h->stream);
  if (h->dep == DEP_FIXED)
    cudaMemcpyAsync(h->h_dep_overflow, h->d_dep_overflow, 8, cudaMemcpyDeviceToHost, h->stream);
}
static int p2p_check_timeouts(pic1dp_gpu_t *h, const char *who) {
  if (h->dep == DEP_FIXED && *h->h_dep_overflow != 0) {
    h->err = std::string(who) + ": fixed-point deposit overflow -- the deposit source grew by more than 8x within one "
             "substep (" + std::to_string(*h->h_dep_overflow) + " warps): the headroom of the integer slots is exhausted "
             "and rho may be invalid.  Use another deposit_mode for this input";
    return PIC1DP_ESTATE;
  }
  if (h->p2p_ready && h->h_p2p_timeouts && *h->h_p2p_timeouts != 0) {
    h->err = std::string(who) + ": the peer-memory density all-reduce timed out (" + std::to_string(*h->h_p2p_timeouts) +
             " flag waits expired: a peer rank died or never reached the substep); rho and E hold NaN";
    return PIC1DP_ENCCL;
  }
  return PIC1DP_OK;
}

// The markers changed behind a fused push: its deposit must not be collected.  The shared-memory deposits overwrite
// their CTA grid at the next flush; the RED deposit accumulates into the L2 grids, which therefore have to be cleared.
static int invalidate_partials(pic1dp_gpu_t *h) {
  if (h->partial_valid && h->dep == DEP_GLOBAL_RED)
    CK(cudaMemsetAsync(h->d_partial, 0, (size_t)h->p.nspecies * h->grid * h->p.nx * 8, h->stream));
  h->partial_valid = false;
  return PIC1DP_OK;
}

// H2D of one species into buffer set 0; the marker count becomes np
static int upload_species(pic1dp_gpu_t *h, int isp, int64_t np, const double *x, const double *v, const double *p,
                          const double *w) {
  CK(cudaSetDevice(h->p.device));
  Species &S = h->sp[isp];
  S.cur = 0;
  S.bak = 0;
  S.np = np;
  const size_t b = (size_t)np * 8;
  CK(cudaMemcpyAsync(S.x[0], x, b, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.v[0], v, b, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.p, p, b, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.w[0], w, b, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));  // host buffers are only borrowed for the call
  h->h2d += 4 * (int64_t)b;
  S.loaded = true;
  S.wmax_valid = false;
  S.pmax_valid = false;
  return invalidate_partials(h);
}

int pic1dp_gpu_set_markers(pic1dp_gpu_t *h, int32_t isp, int64_t np, const double *x, const double *v,
                           const double *p, const double *w) {
  if (!h || isp < 0 || isp >= h->p.nspecies || np < 0 || !x || !v || !p || !w) {
    if (h) h->err = "set_markers: bad argument";
    return PIC1DP_EINVAL;
  }
  if (np > h->p.capacity) { h->err = "set_markers: np exceeds capacity"; return PIC1DP_ECAPACITY; }
  return upload_species(h, isp, np, x, v, p, w);
}

static int load_check_args(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init, double v_max,
                           int32_t init_nmode, const int32_t *init_mode, const double *init_mode_cos,
                           const double *init_mode_sin) {
  if (!h || isp < 0 || isp >= h->p.nspecies || np < 0 || nparticle_init < 1 || !(v_max > 0.0) ||
      init_nmode < 0 || init_nmode > 8 || (init_nmode > 0 && (!init_mode || !init_mode_cos || !init_mode_sin))) {
    if (h) h->err = "load_markers: bad argument (at most 8 initial modes)";
    return PIC1DP_EINVAL;
  }
  if (np > h->p.capacity) { h->err = "load_markers: np exceeds capacity"; return PIC1DP_ECAPACITY; }
  return PIC1DP_OK;
}

// the loader arithmetic on the uniforms (or Gaussians) that already sit in v[0] and x[0] of the species
static int load_markers_finish(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init, double v_max,
                               int32_t init_nmode, const int32_t *init_mode, const double *init_mode_cos,
                               const double *init_mode_sin, int imarker) {
  Species &S = h->sp[isp];
  S.cur = 0;
  S.bak = 0;
  S.np = np;
  LoadArgs a;
  memset(&a, 0, sizeof(a));
  a.x = S.x[0];
  a.v = S.v[0];
  a.p = S.p;
  a.w = S.w[0];
  a.np = np;
  a.lx = h->p.lx;
  a.v_max = v_max;
  a.ninit = (double)nparticle_init;
  a.c = S.c;
  a.T2 = h->p.temperature2[isp];
  a.dist = h->p.iptcldist;
  a.linear = h->p.linear;
  a.imarker = imarker;
  a.init_nmode = init_nmode;
  for (int i = 0; i < init_nmode; i++) {
    a.init_mode[i] = init_mode[i];
    a.init_cos[i] = init_mode_cos[i];
    a.init_sin[i] = init_mode_sin[i];
  }
  k_load_markers<<<h->nsm * 8, 256, 0, h->stream>>>(a);
  CKL(h);
  CK(cudaStreamSynchronize(h->stream));  // host buffers are only borrowed for the call
  S.loaded = true;
  S.wmax_valid = false;
  S.pmax_valid = false;
  return invalidate_partials(h);
}

static int load_markers_impl(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init, const double *rand_v,
                             const double *rand_x, double v_max, int32_t init_nmode, const int32_t *init_mode,
                             const double *init_mode_cos, const double *init_mode_sin, int imarker) {
  int rc = load_check_args(h, isp, np, nparticle_init, v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin);
  if (rc) return rc;
  if (!rand_v || !rand_x) { h->err = "load_markers: NULL stream"; return PIC1DP_EINVAL; }
  CK(cudaSetDevice(h->p.device));
  Species &S = h->sp[isp];
  const size_t b = (size_t)np * 8;
  CK(cudaMemcpyAsync(S.v[0], rand_v, b, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(S.x[0], rand_x, b, cudaMemcpyHostToDevice, h->stream));
  h->h2d += 2 * (int64_t)b;
  return load_markers_finish(h, isp, np, nparticle_init, v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin,
                             imarker);
}

// ---- device-side random streams (rng_kernels.cuh) ----
static int kiss_tables(pic1dp_gpu_t *h) {
  if (h->d_kiss_tab) return PIC1DP_OK;
  KissTables *t = new KissTables;
  memcpy(t->lcg, kiss_lcg_jump, sizeof(t->lcg));
  memcpy(t->mwc, kiss_mwc_jump, sizeof(t->mwc));
  memcpy(t->xs, kiss_xs_jump, sizeof(t->xs));
  cudaError_t e = cudaMalloc(&h->d_kiss_tab, sizeof(KissTables));
  if (e == cudaSuccess) e = cudaMemcpy(h->d_kiss_tab, t, sizeof(KissTables), cudaMemcpyHostToDevice);
  delete t;
  if (e != cudaSuccess) { h->err = std::string("kiss tables: ") + cudaGetErrorString(e); return PIC1DP_ECUDA; }
  return PIC1DP_OK;
}

// raw: the 64-bit outputs themselves (bits in the double slots) instead of the uniforms
static int kiss64_fill_device(pic1dp_gpu_t *h, const uint64_t seeds[4], int64_t offset, int64_t n, double *d_out,
                              bool raw = false) {
  int rc = kiss_tables(h);
  if (rc) return rc;
  if (n == 0) return PIC1DP_OK;
  Kiss64 s0 = {seeds[0], seeds[1], seeds[2], seeds[3]};
  const int chunk = 512;   // a multiple of 32 (the tile protocol of k_kiss64_fill)
  const int64_t nchunks = (n + chunk - 1) / chunk;
  int blocks = (int)((nchunks + 127) / 128);
  if (blocks > h->nsm * 16) blocks = h->nsm * 16;
  if (raw)
    k_kiss64_fill<true><<<blocks, 128, 0, h->stream>>>(s0, (uint64_t)offset, n, chunk, (const KissTables *)h->d_kiss_tab,
                                                       d_out);
  else
    k_kiss64_fill<<<blocks, 128, 0, h->stream>>>(s0, (uint64_t)offset, n, chunk, (const KissTables *)h->d_kiss_tab, d_out);
  CKL(h);
  return PIC1DP_OK;
}

int pic1dp_gpu_load_markers_kiss64(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init,
                                   const uint64_t seeds[4], int64_t offset_v, int64_t offset_x, double v_max,
                                   int32_t init_nmode, const int32_t *init_mode, const double *init_mode_cos,
                                   const double *init_mode_sin) {
  int rc = load_check_args(h, isp, np, nparticle_init, v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin);
  if (rc) return rc;
  if (!seeds || offset_v < 0 || offset_x < 0) { h->err = "load_markers_kiss64: bad stream argument"; return PIC1DP_EINVAL; }
  CK(cudaSetDevice(h->p.device));
  Species &S = h->sp[isp];
  if ((rc = kiss64_fill_device(h, seeds, offset_v, np, S.v[0]))) return rc;   // multirand_real_array(pv), :180
  if ((rc = kiss64_fill_device(h, seeds, offset_x, np, S.x[0]))) return rc;   // multirand_real_array(px), :222
  return load_markers_finish(h, isp, np, nparticle_init, v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin, 2);
}

int pic1dp_gpu_load_markers_counter(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init, uint64_t seed,
                                    int64_t first_index, double v_max, int32_t init_nmode, const int32_t *init_mode,
                                    const double *init_mode_cos, const double *init_mode_sin) {
  int rc = load_check_args(h, isp, np, nparticle_init, v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin);
  if (rc) return rc;
  if (first_index < 0) { h->err = "load_markers_counter: bad first_index"; return PIC1DP_EINVAL; }
  CK(cudaSetDevice(h->p.device));
  Species &S = h->sp[isp];
  if (np > 0) {
    k_counter_fill<<<h->nsm * 8, 256, 0, h->stream>>>(seed, (uint32_t)isp, (uint64_t)first_index, np, S.v[0], S.x[0]);
    CKL(h);
  }
  return load_markers_finish(h, isp, np, nparticle_init, v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin, 2);
}

int pic1dp_gpu_kiss64_uniforms(pic1dp_gpu_t *h, const uint64_t seeds[4], int64_t offset, int64_t n, double *out) {
  if (!h || !seeds || offset < 0 || n < 0 || !out) { if (h) h->err = "kiss64_uniforms: bad argument"; return PIC1DP_EINVAL; }
  if (n == 0) return PIC1DP_OK;
  CK(cudaSetDevice(h->p.device));
  double *d = nullptr;
  CK(cudaMalloc(&d, (size_t)n * 8));
  int rc = kiss64_fill_device(h, seeds, offset, n, d);
  cudaError_t e = cudaSuccess;
  if (!rc) {
    e = cudaMemcpyAsync(out, d, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    h->d2h += n * 8;
  }
  cudaFree(d);
  if (rc) return rc;
  if (e != cudaSuccess) { h->err = std::string("kiss64_uniforms: ") + cudaGetErrorString(e); return PIC1DP_ECUDA; }
  return PIC1DP_OK;
}

// the same generator on the host (no GPU): what a host does to keep its own multirand state in step with the numbers
// the device consumed, and what the CPU tests use to check the jump tables
int pic1dp_host_kiss64_jump(uint64_t seeds[4], int64_t n) {
  if (!seeds || n < 0) return PIC1DP_EINVAL;
  Kiss64 s = {seeds[0], seeds[1], seeds[2], seeds[3]};
  kiss64_jump_host(s, (uint64_t)n);
  seeds[0] = s.x; seeds[1] = s.xs; seeds[2] = s.z; seeds[3] = s.c;
  return PIC1DP_OK;
}

int pic1dp_host_kiss64_fill(uint64_t seeds[4], int64_t n, double *out) {
  if (!seeds || n < 0 || (n > 0 && !out)) return PIC1DP_EINVAL;
  Kiss64 s = {seeds[0], seeds[1], seeds[2], seeds[3]};
  for (int64_t i = 0; i < n; i++) out[i] = int2real64(kiss64_next(s));
  seeds[0] = s.x; seeds[1] = s.xs; seeds[2] = s.z; seeds[3] = s.c;
  return PIC1DP_OK;
}

// ---- SuperKISS64 on the device (rng_kernels.cuh) ----
static bool sk_bad_state(const uint64_t *seeds, const int32_t *iseed) {
  return !seeds || !iseed || *iseed < 0 || *iseed > PIC1DP_SK_N;
}

// table position after ntot draws from position i0 (a refill happens lazily, at the draw that finds iseed = N)
static int32_t sk_iseed_after(int32_t i0, int64_t ntot) {
  const int64_t rest = PIC1DP_SK_N - i0;
  if (ntot <= rest) return (int32_t)(i0 + ntot);
  return (int32_t)((ntot - rest - 1) % PIC1DP_SK_N + 1);
}

// io[i] = the finished draw offset + i, i < n, from its raw table word (k_superkiss64_finish); (lcg0, xs0) = the LCG and
// xorshift before draw 0; raw: the 64-bit outputs instead of the uniforms
static int superkiss64_finish_device(pic1dp_gpu_t *h, uint64_t lcg0, uint64_t xs0, int64_t offset, int64_t n, double *io,
                                     bool raw = false) {
  if (n == 0) return PIC1DP_OK;
  const int chunk = 512;   // a multiple of 32 (the tile protocol of k_superkiss64_finish)
  const int64_t nchunks = (n + chunk - 1) / chunk;
  int blocks = (int)((nchunks + 127) / 128);
  if (blocks > h->nsm * 16) blocks = h->nsm * 16;
  const KissTables *tab = (const KissTables *)h->d_kiss_tab;
  if (raw)
    k_superkiss64_finish<true><<<blocks, 128, 0, h->stream>>>(lcg0, xs0, (uint64_t)offset, n, chunk, tab, io);
  else
    k_superkiss64_finish<<<blocks, 128, 0, h->stream>>>(lcg0, xs0, (uint64_t)offset, n, chunk, tab, io);
  CKL(h);
  return PIC1DP_OK;
}

static int superkiss64_table_device(pic1dp_gpu_t *h, int32_t i0, int64_t ntot, double *d_a, int64_t na, double *d_b,
                                    int64_t pb, int64_t nb) {
  const int smem = PIC1DP_SK_N * sizeof(uint64_t);
  CK(cudaFuncSetAttribute(k_superkiss64_table, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  k_superkiss64_table<<<1, PIC1DP_SK_THREADS, smem, h->stream>>>(h->d_sk_state, i0, ntot, d_a, na, d_b, pb, nb);
  CKL(h);
  return PIC1DP_OK;
}

// draws [0, ntot) of the stream at (seeds, *iseed): draw p becomes the uniform d_a[p] (p < na) or d_b[p - pb]
// (0 <= p - pb < nb), the others are discarded.  seeds / *iseed are advanced past all ntot draws (synchronous D2H of
// the table), so the host generator continues the same stream.
static int superkiss64_fill_device(pic1dp_gpu_t *h, uint64_t *seeds, int32_t *iseed, int64_t ntot, double *d_a,
                                   int64_t na, double *d_b, int64_t pb, int64_t nb) {
  int rc = kiss_tables(h);
  if (rc) return rc;
  if (ntot == 0) return PIC1DP_OK;
  const size_t state_bytes = (PIC1DP_SK_N + 1) * sizeof(uint64_t);
  if (!h->d_sk_state) CK(cudaMalloc(&h->d_sk_state, state_bytes));
  const uint64_t lcg0 = seeds[PIC1DP_SK_N + 1], xs0 = seeds[PIC1DP_SK_N + 2];
  CK(cudaMemcpyAsync(h->d_sk_state, seeds, state_bytes, cudaMemcpyHostToDevice, h->stream));
  h->h2d += state_bytes;
  if ((rc = superkiss64_table_device(h, *iseed, ntot, d_a, na, d_b, pb, nb))) return rc;
  if ((rc = superkiss64_finish_device(h, lcg0, xs0, 0, na, d_a))) return rc;
  if ((rc = superkiss64_finish_device(h, lcg0, xs0, pb, nb, d_b))) return rc;
  CK(cudaMemcpyAsync(seeds, h->d_sk_state, state_bytes, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->d2h += state_bytes;
  seeds[PIC1DP_SK_N + 1] = sk_lcg_jump(lcg0, (uint64_t)ntot);
  seeds[PIC1DP_SK_N + 2] = sk_xs_jump(xs0, (uint64_t)ntot, kiss_xs_jump);
  *iseed = sk_iseed_after(*iseed, ntot);
  return PIC1DP_OK;
}

int pic1dp_gpu_load_markers_superkiss64(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nlocal,
                                        int64_t nparticle_init, uint64_t seeds[PIC1DP_SUPERKISS64_NSEED], int32_t *iseed,
                                        double v_max, int32_t init_nmode, const int32_t *init_mode,
                                        const double *init_mode_cos, const double *init_mode_sin) {
  int rc = load_check_args(h, isp, np, nparticle_init, v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin);
  if (rc) return rc;
  if (sk_bad_state(seeds, iseed) || nlocal < np) {
    h->err = "load_markers_superkiss64: bad stream argument (iseed in [0, 20632], nlocal >= np)";
    return PIC1DP_EINVAL;
  }
  CK(cudaSetDevice(h->p.device));
  Species &S = h->sp[isp];
  // multirand_real_array(pv) over the whole local array (:180), then multirand_real_array(px) (:222)
  if ((rc = superkiss64_fill_device(h, seeds, iseed, 2 * nlocal, S.v[0], np, S.x[0], nlocal, np))) return rc;
  return load_markers_finish(h, isp, np, nparticle_init, v_max, init_nmode, init_mode, init_mode_cos, init_mode_sin, 2);
}

int pic1dp_gpu_superkiss64_uniforms(pic1dp_gpu_t *h, uint64_t seeds[PIC1DP_SUPERKISS64_NSEED], int32_t *iseed, int64_t n,
                                    double *out) {
  if (!h || sk_bad_state(seeds, iseed) || n < 0 || (n > 0 && !out)) {
    if (h) h->err = "superkiss64_uniforms: bad argument";
    return PIC1DP_EINVAL;
  }
  if (n == 0) return PIC1DP_OK;
  CK(cudaSetDevice(h->p.device));
  double *d = nullptr;
  CK(cudaMalloc(&d, (size_t)n * 8));
  int rc = superkiss64_fill_device(h, seeds, iseed, n, d, n, nullptr, 0, 0);
  cudaError_t e = cudaSuccess;
  if (!rc) {
    e = cudaMemcpyAsync(out, d, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    h->d2h += n * 8;
  }
  cudaFree(d);
  if (rc) return rc;
  if (e != cudaSuccess) { h->err = std::string("superkiss64_uniforms: ") + cudaGetErrorString(e); return PIC1DP_ECUDA; }
  return PIC1DP_OK;
}

int pic1dp_host_superkiss64_fill(uint64_t seeds[PIC1DP_SUPERKISS64_NSEED], int32_t *iseed, int64_t n, double *out) {
  if (sk_bad_state(seeds, iseed) || n < 0 || (n > 0 && !out)) return PIC1DP_EINVAL;
  const int N = PIC1DP_SK_N;
  int32_t i = *iseed;
  uint64_t z = seeds[N + 1], xs = seeds[N + 2];
  for (int64_t k = 0; k < n; k++) {
    if (i >= N) {
      seeds[N] = sk_chunk_rewrite(seeds, 0, N, seeds[N]);
      i = 0;
    }
    z = sk_lcg_next(z);
    xs = sk_xs_next(xs);
    out[k] = int2real64(seeds[i++] + z + xs);
  }
  seeds[N + 1] = z;
  seeds[N + 2] = xs;
  *iseed = i;
  return PIC1DP_OK;
}

int pic1dp_host_superkiss64_refill(uint64_t seeds[PIC1DP_SUPERKISS64_NSEED], int32_t nchunks) {
  const int N = PIC1DP_SK_N;
  if (!seeds || nchunks < 1 || nchunks > N) return PIC1DP_EINVAL;
  const int K = (N + nchunks - 1) / nchunks;
  std::vector<unsigned> m(nchunks), prev;
  std::vector<uint64_t> left(nchunks, 0);
  const uint64_t c0 = seeds[N];
  for (int k = 0; k < nchunks; k++) {
    const int s = std::min(k * K, N), e = std::min(s + K, N);
    m[k] = sk_chunk_map(seeds, s, e, c0);
    if (s > 0 && s < e) left[k] = seeds[s - 1];
  }
  for (int d = 1; d < nchunks; d <<= 1) {   // inclusive scan of the chunk maps (Hillis-Steele, as across warp lanes)
    prev = m;
    for (int k = d; k < nchunks; k++) m[k] = sk_compose(prev[k], prev[k - d]);
  }
  for (int k = 0; k < nchunks; k++) {
    const int s = std::min(k * K, N), e = std::min(s + K, N);
    if (s >= e) continue;
    const uint64_t cout = sk_chunk_rewrite(seeds, s, e, s == 0 ? c0 : sk_hi(left[k]) + sk_apply(m[k - 1], 0));
    if (e == N) seeds[N] = cout;
  }
  return PIC1DP_OK;
}

// ---- Maxwellian markers: multirand_gaussian_array(pv) on the device (rng_kernels.cuh) ----
static_assert(PIC1DP_GAUSS_ROUND == PIC1DP_GAUSS_ROUND_DRAWS && PIC1DP_GAUSS_ROUND % 2 == 0, "Gaussian round size");
struct GaussResult {
  int64_t cut = 0;       // draws the Gaussian call consumed: the x stream starts here
  int32_t filled = 0;    // the one-slot buffer after the call
  double buf = 0.0;
};

// gaussian_array(pv, nlocal) from the raw-word stream that produce(a, d) writes (words [a, a + PIC1DP_GAUSS_ROUND) from
// the call's first draw, into d), in rounds: words, accept counts, compaction into d_v (elements < np kept), then one
// read of the running count.  The first round whose count reaches the attempts needed holds the cut.  (filled, buf) is
// the caller's buffer on entry; the result carries it out, the caller's copy is left alone.
static int gauss_stream_device(pic1dp_gpu_t *h, int64_t np, int64_t nlocal, int32_t filled, double buf, double *d_v,
                               GaussResult &out, const std::function<int(int64_t, double *)> &produce) {
  out = GaussResult();
  out.filled = filled;
  out.buf = buf;
  h->gauss_rounds = 0;
  if (nlocal == 0) return PIC1DP_OK;
  int64_t lo = 0;
  if (filled) {   // the buffered value is element 0; no draw for it
    if (np > 0) {
      CK(cudaMemcpyAsync(d_v, &buf, 8, cudaMemcpyHostToDevice, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      h->h2d += 8;
    }
    lo = 1;
  }
  const int64_t need = (nlocal - lo + 1) / 2;   // accepted attempts
  out.filled = (int32_t)((nlocal - lo) & 1);
  if (need == 0) return PIC1DP_OK;
  const int64_t R = PIC1DP_GAUSS_ROUND, npairs = R / 2, nblk = (npairs + PIC1DP_GAUSS_TILE - 1) / PIC1DP_GAUSS_TILE;
  if (!h->d_gauss_words) CK(cudaMalloc(&h->d_gauss_words, (size_t)R * 8));
  if (!h->d_gauss_bcount) CK(cudaMalloc(&h->d_gauss_bcount, (size_t)nblk * sizeof(unsigned)));
  if (!h->d_gauss_ctl) CK(cudaMalloc(&h->d_gauss_ctl, sizeof(GaussCtl)));
  GaussCtl *ctl = (GaussCtl *)h->d_gauss_ctl;
  GaussCtl c = {0ULL, -1LL, 0.0};
  CK(cudaMemcpyAsync(ctl, &c, sizeof(c), cudaMemcpyHostToDevice, h->stream));
  h->h2d += sizeof(c);
  const double2 *words = (const double2 *)h->d_gauss_words;
  for (int64_t a = 0;; a += R) {
    int rc = produce(a, h->d_gauss_words);
    if (rc) return rc;
    const int64_t base = (int64_t)c.total;
    k_gauss_count<<<(unsigned)nblk, PIC1DP_GAUSS_THREADS, 0, h->stream>>>(words, npairs, h->d_gauss_bcount, ctl);
    CKL(h);
    k_gauss_scatter<<<(unsigned)nblk, PIC1DP_GAUSS_THREADS, 0, h->stream>>>(words, npairs, h->d_gauss_bcount, base, a, lo,
                                                                          need, np, nlocal, d_v, ctl);
    CKL(h);
    CK(cudaMemcpyAsync(&c, ctl, sizeof(c), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->d2h += sizeof(c);
    h->gauss_rounds++;
    if ((int64_t)c.total >= need) break;
  }
  out.cut = c.cut;
  if (out.filled) out.buf = c.spare;
  return PIC1DP_OK;
}

static int maxwellian_check_args(pic1dp_gpu_t *h, const char *who, int32_t isp, int64_t np, int64_t nlocal,
                                 int64_t nparticle_init, const void *seeds, const int32_t *gauss_filled,
                                 const double *gauss_buf, int32_t init_nmode, const int32_t *init_mode,
                                 const double *init_mode_cos, const double *init_mode_sin) {
  int rc = load_check_args(h, isp, np, nparticle_init, 1.0, init_nmode, init_mode, init_mode_cos, init_mode_sin);
  if (rc) return rc;
  if (h->p.iptcldist != 0) {  // input_init: "case of input_iptcldist >= 1 and input_imarker = 1 not implemented yet"
    h->err = std::string(who) + ": input_imarker = 1 supports only iptcldist = 0 (src/pic1dp_input.F90:291-299)";
    return PIC1DP_EINVAL;
  }
  if (!seeds || !gauss_filled || !gauss_buf || nlocal < np) {
    h->err = std::string(who) + ": bad stream argument (NULL state or nlocal < np)";
    return PIC1DP_EINVAL;
  }
  return PIC1DP_OK;
}

int pic1dp_gpu_load_markers_maxwellian_kiss64(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nlocal,
                                              int64_t nparticle_init, uint64_t seeds[4], int32_t *gauss_filled,
                                              double *gauss_buf, int32_t init_nmode, const int32_t *init_mode,
                                              const double *init_mode_cos, const double *init_mode_sin) {
  int rc = maxwellian_check_args(h, "load_markers_maxwellian_kiss64", isp, np, nlocal, nparticle_init, seeds,
                                 gauss_filled, gauss_buf, init_nmode, init_mode, init_mode_cos, init_mode_sin);
  if (rc) return rc;
  CK(cudaSetDevice(h->p.device));
  Species &S = h->sp[isp];
  GaussResult g;
  rc = gauss_stream_device(h, np, nlocal, *gauss_filled, *gauss_buf, S.v[0], g, [&](int64_t a, double *d) -> int {
    return kiss64_fill_device(h, seeds, a, PIC1DP_GAUSS_ROUND, d, true);
  });
  if (rc) return rc;
  // multirand_real_array(px) (:222): from the first draw after the last attempt; its unloaded tail is not generated
  if ((rc = kiss64_fill_device(h, seeds, g.cut, np, S.x[0]))) return rc;
  if ((rc = load_markers_finish(h, isp, np, nparticle_init, 1.0, init_nmode, init_mode, init_mode_cos, init_mode_sin, 1)))
    return rc;
  Kiss64 s = {seeds[0], seeds[1], seeds[2], seeds[3]};
  kiss64_jump_host(s, (uint64_t)(g.cut + nlocal));
  seeds[0] = s.x; seeds[1] = s.xs; seeds[2] = s.z; seeds[3] = s.c;
  *gauss_filled = g.filled;
  *gauss_buf = g.buf;
  h->gauss_draws = g.cut;
  h->gauss_regenerated = 0;
  return PIC1DP_OK;
}

int pic1dp_gpu_load_markers_maxwellian_superkiss64(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nlocal,
                                                   int64_t nparticle_init, uint64_t seeds[PIC1DP_SUPERKISS64_NSEED],
                                                   int32_t *iseed, int32_t *gauss_filled, double *gauss_buf,
                                                   int32_t init_nmode, const int32_t *init_mode,
                                                   const double *init_mode_cos, const double *init_mode_sin) {
  int rc = maxwellian_check_args(h, "load_markers_maxwellian_superkiss64", isp, np, nlocal, nparticle_init, seeds,
                                 gauss_filled, gauss_buf, init_nmode, init_mode, init_mode_cos, init_mode_sin);
  if (rc) return rc;
  if (sk_bad_state(seeds, iseed)) {
    h->err = "load_markers_maxwellian_superkiss64: table position outside [0, 20632]";
    return PIC1DP_EINVAL;
  }
  CK(cudaSetDevice(h->p.device));
  if ((rc = kiss_tables(h))) return rc;
  Species &S = h->sp[isp];
  const size_t state_bytes = (PIC1DP_SK_N + 1) * sizeof(uint64_t);
  if (!h->d_sk_state) CK(cudaMalloc(&h->d_sk_state, state_bytes));
  if (!h->d_sk_round) CK(cudaMalloc(&h->d_sk_round, state_bytes));
  const uint64_t lcg0 = seeds[PIC1DP_SK_N + 1], xs0 = seeds[PIC1DP_SK_N + 2];
  CK(cudaMemcpyAsync(h->d_sk_state, seeds, state_bytes, cudaMemcpyHostToDevice, h->stream));
  h->h2d += state_bytes;
  // the table cannot be jumped back: each round starts from a copy of it, from which the x stream is regenerated
  int64_t round_start = 0;
  int32_t round_pos = *iseed;
  bool saved = false;
  GaussResult g;
  rc = gauss_stream_device(h, np, nlocal, *gauss_filled, *gauss_buf, S.v[0], g, [&](int64_t a, double *d) -> int {
    CK(cudaMemcpyAsync(h->d_sk_round, h->d_sk_state, state_bytes, cudaMemcpyDeviceToDevice, h->stream));
    saved = true;
    round_start = a;
    round_pos = sk_iseed_after(*iseed, a);
    int rc2 = superkiss64_table_device(h, round_pos, PIC1DP_GAUSS_ROUND, d, PIC1DP_GAUSS_ROUND, nullptr, 0, 0);
    return rc2 ? rc2 : superkiss64_finish_device(h, lcg0, xs0, a, PIC1DP_GAUSS_ROUND, d, true);
  });
  if (rc) return rc;
  // multirand_real_array(px) (:222): rerun the table from the start of the cut's round over the rest of that round's
  // attempts and the nlocal draws of px, keeping the first np of them
  if (saved) CK(cudaMemcpyAsync(h->d_sk_state, h->d_sk_round, state_bytes, cudaMemcpyDeviceToDevice, h->stream));
  const int64_t skip = g.cut - round_start;
  if (skip + nlocal > 0 && (rc = superkiss64_table_device(h, round_pos, skip + nlocal, nullptr, 0, S.x[0], skip, np)))
    return rc;
  if ((rc = superkiss64_finish_device(h, lcg0, xs0, g.cut, np, S.x[0]))) return rc;
  if ((rc = load_markers_finish(h, isp, np, nparticle_init, 1.0, init_nmode, init_mode, init_mode_cos, init_mode_sin, 1)))
    return rc;
  CK(cudaMemcpyAsync(seeds, h->d_sk_state, state_bytes, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->d2h += state_bytes;
  const int64_t ntot = g.cut + nlocal;
  seeds[PIC1DP_SK_N + 1] = sk_lcg_jump(lcg0, (uint64_t)ntot);
  seeds[PIC1DP_SK_N + 2] = sk_xs_jump(xs0, (uint64_t)ntot, kiss_xs_jump);
  *iseed = sk_iseed_after(*iseed, ntot);
  *gauss_filled = g.filled;
  *gauss_buf = g.buf;
  h->gauss_draws = g.cut;
  h->gauss_regenerated = skip;
  return PIC1DP_OK;
}

int pic1dp_gpu_last_gaussian_load(pic1dp_gpu_t *h, int64_t *draws, int64_t *rounds, int64_t *regenerated) {
  if (!h || !draws || !rounds || !regenerated) return PIC1DP_EINVAL;
  *draws = h->gauss_draws;
  *rounds = h->gauss_rounds;
  *regenerated = h->gauss_regenerated;
  return PIC1DP_OK;
}

void pic1dp_host_counter_uniforms(uint64_t seed, int32_t stream, int64_t first_index, int64_t n, double *u_v, double *u_x) {
  for (int64_t i = 0; i < n; i++) counter_uniforms(seed, (uint32_t)stream, (uint64_t)(first_index + i), u_v[i], u_x[i]);
}

int pic1dp_gpu_load_markers(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init, const double *rand_v,
                            const double *rand_x, double v_max, int32_t init_nmode, const int32_t *init_mode,
                            const double *init_mode_cos, const double *init_mode_sin) {
  return load_markers_impl(h, isp, np, nparticle_init, rand_v, rand_x, v_max, init_nmode, init_mode, init_mode_cos,
                           init_mode_sin, 2);
}

int pic1dp_gpu_load_markers_maxwellian(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init,
                                       const double *gauss_v, const double *rand_x, int32_t init_nmode,
                                       const int32_t *init_mode, const double *init_mode_cos,
                                       const double *init_mode_sin) {
  if (h && h->p.iptcldist != 0) {  // input_init: "case of input_iptcldist >= 1 and input_imarker = 1 not implemented yet"
    h->err = "load_markers_maxwellian: input_imarker = 1 supports only iptcldist = 0 (src/pic1dp_input.F90:291-299)";
    return PIC1DP_EINVAL;
  }
  return load_markers_impl(h, isp, np, nparticle_init, gauss_v, rand_x, 1.0, init_nmode, init_mode, init_mode_cos,
                           init_mode_sin, 1);
}

int pic1dp_gpu_get_markers(pic1dp_gpu_t *h, int32_t isp, double *x, double *v, double *p, double *w, int64_t *np) {
  if (!h || isp < 0 || isp >= h->p.nspecies) return PIC1DP_EINVAL;
  Species &S = h->sp[isp];
  if (!S.loaded) { h->err = "get_markers before set_markers"; return PIC1DP_ESTATE; }
  CK(cudaSetDevice(h->p.device));
  const size_t b = (size_t)S.np * 8;
  if (x) { CK(cudaMemcpyAsync(x, S.x[S.cur], b, cudaMemcpyDeviceToHost, h->stream)); h->d2h += b; }
  if (v) { CK(cudaMemcpyAsync(v, S.v[S.cur], b, cudaMemcpyDeviceToHost, h->stream)); h->d2h += b; }
  if (p) { CK(cudaMemcpyAsync(p, S.p, b, cudaMemcpyDeviceToHost, h->stream)); h->d2h += b; }
  if (w) { CK(cudaMemcpyAsync(w, S.w[S.cur], b, cudaMemcpyDeviceToHost, h->stream)); h->d2h += b; }
  CK(cudaStreamSynchronize(h->stream));
  if (np) *np = S.np;
  return PIC1DP_OK;
}

static void fill_grid_args(pic1dp_gpu_t *h, GridArgs &g) {
  const pic1dp_params &p = h->p;
  memset(&g, 0, sizeof(g));
  g.nx = p.nx;
  g.nmode = p.nmode;
  g.nspecies = p.nspecies;
  g.ngrids = h->grid;
  g.deltaf = p.deltaf;
  g.matrix_path = p.iptclshape <= 2;
  g.zero_partials = h->dep == DEP_GLOBAL_RED;
  g.lx = p.lx;
  g.rnx = (double)p.nx;
  for (int s = 0; s < p.nspecies; s++) {
    g.Z[s] = p.charge[s];
    g.n[s] = p.density[s];
  }
  g.partial = h->d_partial;
  g.red = h->d_red;
  g.rho = h->d_rho;
  g.E = h->d_E;
  g.mode_re = h->d_mre;
  g.mode_im = h->d_mim;
  g.F_re = h->d_Fre;
  g.F_im = h->d_Fim;
  g.ginv = h->d_ginv;
  g.a_im = -1.0 / (double)p.nx;
  g.a_re = 1.0 / (double)p.nx;
  g.nx_over_lx = (double)p.nx / p.lx;
  g.energy = h->d_energy;
  if (p.nranks > 1 && h->p2p_ready) {
    g.p2p_nranks = p.nranks;
    g.p2p_rank = p.rank;
    for (int r = 0; r < p.nranks; r++) g.p2p_peer[r] = h->peer_base[r];
    g.p2p_counter = h->d_p2p_counter;
    g.p2p_timeouts = h->d_p2p_timeouts;
    g.p2p_epoch_dev = h->d_p2p_epoch;
    g.p2p_stamps = h->d_p2p_stamps;
    g.p2p_stamp_cap = h->p2p_stamp_cap;
  }
}

static void fill_particle_args(pic1dp_gpu_t *h, int s, ParticleArgs &a) {
  const pic1dp_params &p = h->p;
  Species &S = h->sp[s];
  memset(&a, 0, sizeof(a));
  a.p = S.p;
  a.E = h->d_E;
  a.E_start = h->d_E_start;
  a.dth = 0.5 * p.dt;
  a.partial = h->d_partial + (size_t)s * h->grid * p.nx;
  a.noob = h->d_noob;
  a.dep_wmax_hi = h->d_wmax_hi + s;
  a.dep_overflow = h->d_dep_overflow;
  a.np = S.np;
  a.nx = p.nx;
  a.lx = p.lx;
  a.rlx = 1.0 / p.lx;
  a.rnx = (double)p.nx;
  a.c = S.c;
  a.deltaf = p.deltaf;
  a.linear = p.linear;
  a.right_frac = p.iptclshape <= 2;
}

static int check_loaded(pic1dp_gpu_t *h, const char *who) {
  for (int s = 0; s < h->p.nspecies; s++)
    if (!h->sp[s].loaded) {
      h->err = std::string(who) + ": markers of every species must be set first";
      return PIC1DP_ESTATE;
    }
  return PIC1DP_OK;
}

// fixed-point deposit: the scale of a launch comes from the running maximum of |deposit source| (w for delta-f, p for
// full-f).  The fused kernels keep it up to date; after the markers were replaced it is recomputed here.
static int ensure_wmax(pic1dp_gpu_t *h) {
  if (h->dep != DEP_FIXED) return PIC1DP_OK;
  for (int s = 0; s < h->p.nspecies; s++) {
    Species &S = h->sp[s];
    if (S.wmax_valid || !S.loaded) continue;
    CK(cudaMemsetAsync(h->d_wmax_hi + s, 0, 4, h->stream));
    if (S.np > 0) {
      k_absmax_hi<<<h->nsm * 8, 256, 0, h->stream>>>(h->p.deltaf ? S.w[S.cur] : S.p, S.np, h->d_wmax_hi + s);
      CKL(h);
    }
    S.wmax_valid = true;
  }
  return PIC1DP_OK;
}

// wrap (+ deposit) pass over all species
static int run_deposit_pass(pic1dp_gpu_t *h, bool deposit) {
  if (deposit) {
    const int rc = ensure_wmax(h);
    if (rc) return rc;
  }
  PushKernel k = pick_deposit(h->dep, deposit);
  for (int s = 0; s < h->p.nspecies; s++) {
    Species &S = h->sp[s];
    ParticleArgs a;
    fill_particle_args(h, s, a);
    a.x_cur = S.x[S.cur];
    a.x_out = S.x[S.cur];
    a.dep_src = h->p.deltaf ? S.w[S.cur] : S.p;
    k<<<h->grid, h->threads, deposit ? h->smem_dep : 0, h->stream>>>(a);
    CKL(h);
  }
  return PIC1DP_OK;
}

int pic1dp_gpu_compute_shape_x(pic1dp_gpu_t *h) {
  if (!h) return PIC1DP_EINVAL;
  int rc = check_loaded(h, "compute_shape_x");
  if (rc) return rc;
  if (h->p.iptclshape == 4) return PIC1DP_OK;  // src/pic1dp.F90:65, :86
  if (h->partial_valid) return PIC1DP_OK;      // fused push already wrapped x
  CK(cudaSetDevice(h->p.device));
  return run_deposit_pass(h, false);
}

int pic1dp_gpu_get_shape_x(pic1dp_gpu_t *h, int32_t isp, int32_t *indexes, double *values_left,
                           double *values_right) {
  if (!h || isp < 0 || isp >= h->p.nspecies) return PIC1DP_EINVAL;
  Species &S = h->sp[isp];
  if (!S.loaded) { h->err = "get_shape_x before set_markers"; return PIC1DP_ESTATE; }
  if (S.np == 0) return PIC1DP_OK;
  CK(cudaSetDevice(h->p.device));
  int *d_ix = nullptr;
  double *d_sl = nullptr, *d_sr = nullptr;
  const size_t n = (size_t)S.np;
  CK(cudaMalloc(&d_ix, n * 4));
  CK(cudaMalloc(&d_sl, n * 8));
  CK(cudaMalloc(&d_sr, n * 8));
  ParticleArgs a;
  fill_particle_args(h, isp, a);
  a.x_cur = S.x[S.cur];
  k_shape_x<<<h->nsm * 4, 256, 0, h->stream>>>(a, d_ix, d_sl, d_sr);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) {
    h->launches++;
    if (indexes) e = cudaMemcpyAsync(indexes, d_ix, n * 4, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess && values_left) e = cudaMemcpyAsync(values_left, d_sl, n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess && values_right) e = cudaMemcpyAsync(values_right, d_sr, n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  }
  cudaFree(d_ix);
  cudaFree(d_sl);
  cudaFree(d_sr);
  if (e != cudaSuccess) { h->err = std::string("get_shape_x: ") + cudaGetErrorString(e); return PIC1DP_ECUDA; }
  return PIC1DP_OK;
}

// sum of the private grids (+ species charge), all-reduce over ranks, optionally rho = ... (k_finalize_rho)
static int reduce_charge(pic1dp_gpu_t *h, bool finalize) {
  GridArgs g;
  fill_grid_args(h, g);
  k_reduce_charge<<<(h->p.nx + 31) / 32, 256, 0, h->stream>>>(g);
  CKL(h);
  if (h->p.nranks > 1 && h->p2p_ready) {
    // all-reduce through peer memory: the reduce kernel above already scattered (it was launched with the p2p
    // arguments), the finalize / solve kernel gathers
    h->p2p_calls++;
  } else if (h->p.nranks > 1) {
    if (!h->comm) { h->err = "collect_charge: nranks > 1 but comm_init was not called"; return PIC1DP_ESTATE; }
    ncclResult_t r = g_nccl.AllReduce(h->d_red, h->d_red, (size_t)h->nred * h->p.nx, ncclDouble, ncclSum, h->comm,
                                      h->stream);  // MPI_Allreduce, src/pic1dp_interaction.F90:132-133
    if (r != ncclSuccess) { h->err = std::string("ncclAllReduce: ") + g_nccl.GetErrorString(r); return PIC1DP_ENCCL; }
    h->nccl_calls++;
  }
  if (finalize) {
    k_finalize_rho<<<(h->p.nx + 127) / 128, 128, 0, h->stream>>>(g);
    CKL(h);
  }
  return PIC1DP_OK;
}

static int collect_charge_impl(pic1dp_gpu_t *h, bool finalize) {
  int rc = check_loaded(h, "collect_charge");
  if (rc) return rc;
  CK(cudaSetDevice(h->p.device));
  if (!h->partial_valid) {
    rc = run_deposit_pass(h, true);
    if (rc) return rc;
  }
  h->partial_valid = false;
  return reduce_charge(h, finalize);
}

int pic1dp_gpu_collect_charge(pic1dp_gpu_t *h) {
  if (!h) return PIC1DP_EINVAL;
  return collect_charge_impl(h, true);
}

// finalize_first: rho has not been formed yet (step() skips k_finalize_rho and lets the solve kernel do it)
static int solve_field_impl(pic1dp_gpu_t *h, bool finalize_first) {
  CK(cudaSetDevice(h->p.device));
  GridArgs g;
  fill_grid_args(h, g);
  const int smem = (h->p.nx + 2 * h->p.nmode) * 8;
  const bool seq = h->p.field_mode == PIC1DP_FIELD_SEQUENTIAL;
  if (seq && finalize_first) k_field_solve<true, true><<<1, 1024, smem, h->stream>>>(g);
  else if (seq) k_field_solve<true, false><<<1, 1024, smem, h->stream>>>(g);
  else if (finalize_first) k_field_solve<false, true><<<1, 1024, smem, h->stream>>>(g);
  else k_field_solve<false, false><<<1, 1024, smem, h->stream>>>(g);
  CKL(h);
  return PIC1DP_OK;
}

int pic1dp_gpu_solve_field(pic1dp_gpu_t *h) {
  if (!h) return PIC1DP_EINVAL;
  return solve_field_impl(h, false);
}

// recompute: the RC kernel pair of step() (h->recompute).  Its irk = 1 leaves the midpoint set's x and v unwritten, so
// it must be followed by the RC irk = 2 before anything reads the markers; the public per-substep push stores them.
static int push_impl(pic1dp_gpu_t *h, int32_t irk, bool recompute) {
  int rc = check_loaded(h, "push");
  if (rc) return rc;
  CK(cudaSetDevice(h->p.device));
  const pic1dp_params &p = h->p;
  const bool fused = p.fuse != 0;
  if (fused && (rc = ensure_wmax(h))) return rc;
  if (fused && h->partial_valid && h->dep == DEP_GLOBAL_RED)  // a previous fused deposit was never collected
    CK(cudaMemsetAsync(h->d_partial, 0, (size_t)p.nspecies * h->grid * p.nx * 8, h->stream));
  for (int s = 0; s < p.nspecies; s++) {
    Species &S = h->sp[s];
    ParticleArgs a;
    fill_particle_args(h, s, a);
    int out;
    if (irk == 1) {
      S.bak = S.cur;       // VecCopy x,v,w -> *_bak (:181-187) without moving a byte
      out = S.cur ^ 1;
      a.dt = a.dth;        // 0.5 * dt, :179
    } else {
      out = S.bak;         // overwrite the start-of-step set
      a.dt = p.dt;         // :192
    }
    a.x_cur = S.x[S.cur];
    a.v_cur = S.v[S.cur];
    a.w_cur = S.w[S.cur];
    a.x_bak = S.x[S.bak];
    a.v_bak = S.v[S.bak];
    a.w_bak = S.w[S.bak];
    a.x_out = S.x[out];
    a.v_out = S.v[out];
    a.w_out = S.w[out];

    int cfg = (h->cfg == 1) ? (S.c.unit ? 25 : S.c.pow2 ? 9 : 1) : -1;
    if (cfg > 0 && fused && p.arith_mode == PIC1DP_ARITH_TOLERANCE && (p.iptcldist == 2 || p.iptcldist == 3))
      cfg = (S.c.unit ? 25 : 1) + 32;   // the tolerance form has no constant divisors left, so pow2 needs no variant
    const bool timed = h->lt_on && h->lt_irk.size() < 8192;
    if (timed) {
      if (h->lt_ev.size() < 2 * (h->lt_irk.size() + 1)) {
        cudaEvent_t e0, e1;
        CK(cudaEventCreate(&e0));
        CK(cudaEventCreate(&e1));
        h->lt_ev.push_back(e0);
        h->lt_ev.push_back(e1);
      }
      CK(cudaEventRecord(h->lt_ev[2 * h->lt_irk.size()], h->stream));
    }
    if (fused && h->use_cpa[irk - 1] && cfg > 0) {
      PushKernel k = pick_cpa(p.iptcldist, h->dep, irk == 2, cfg);
      k<<<h->grid, h->threads, h->cpa_smem[irk - 1], h->stream>>>(a);
    } else if (fused && h->use_tma[irk - 1] && cfg > 0) {
      PushKernel k = pick_tma(p.iptcldist, h->dep, irk == 2, cfg);
      k<<<h->grid, 512, h->tma_smem[irk - 1], h->stream>>>(a);
    } else if (recompute) {
      PushKernel k = pick_push(p.iptcldist, h->dep, irk == 2, true, cfg, true);
      k<<<h->grid, h->threads, irk == 2 ? h->smem_rc : h->smem_push, h->stream>>>(a);
    } else {
      PushKernel k = pick_push(p.iptcldist, h->dep, irk == 2, fused, cfg, false);
      k<<<h->grid, h->threads, h->smem_push, h->stream>>>(a);
    }
    CKL(h);
    if (timed) {
      CK(cudaEventRecord(h->lt_ev[2 * h->lt_irk.size() + 1], h->stream));
      h->lt_irk.push_back(irk);
    }
    S.cur = out;
  }
  h->partial_valid = fused;
  return PIC1DP_OK;
}

int pic1dp_gpu_push(pic1dp_gpu_t *h, int32_t irk) {
  if (!h || (irk != 1 && irk != 2)) { if (h) h->err = "push: irk must be 1 or 2"; return PIC1DP_EINVAL; }
  return push_impl(h, irk, false);
}

int pic1dp_gpu_launch_timing_start(pic1dp_gpu_t *h) {
  if (!h) return PIC1DP_EINVAL;
  h->lt_irk.clear();
  h->lt_on = true;
  return PIC1DP_OK;
}

int pic1dp_gpu_launch_timing_stop(pic1dp_gpu_t *h, double ms_sum[2], int64_t launches[2]) {
  if (!h || !ms_sum || !launches) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  h->lt_on = false;
  CK(cudaStreamSynchronize(h->stream));
  ms_sum[0] = ms_sum[1] = 0.0;
  launches[0] = launches[1] = 0;
  for (size_t k = 0; k < h->lt_irk.size(); k++) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->lt_ev[2 * k], h->lt_ev[2 * k + 1]));
    ms_sum[h->lt_irk[k] - 1] += (double)ms;
    launches[h->lt_irk[k] - 1]++;
  }
  h->lt_irk.clear();
  return PIC1DP_OK;
}

// one timestep with individual launches: src/pic1dp.F90:79-90
static int step_direct(pic1dp_gpu_t *h) {
  for (int irk = 1; irk <= 2; irk++) {
    int rc = push_impl(h, irk, h->recompute);
    if (rc) return rc;
    if (h->p.iptclshape < 4) {
      rc = pic1dp_gpu_compute_shape_x(h);
      if (rc) return rc;
    }
    rc = collect_charge_impl(h, false);   // rho is formed inside the solve kernel: one launch less
    if (rc) return rc;
    rc = solve_field_impl(h, true);
    if (rc) return rc;
  }
  return PIC1DP_OK;
}

// The launches of one timestep are the same every step: the buffer rotation returns to its starting set after two
// substeps, and the all-reduce epoch is device-resident.  They are captured once into a CUDA graph and replayed, which
// removes ~6 launch gaps per step (decisive at the reference's default size, src/pic1dp_input.F90:113).  The graph
// is re-captured when the marker counts or the rotation differ from the captured ones.
static bool step_graph_usable(pic1dp_gpu_t *h) {
  if (!h->graph_enabled || h->lt_on || h->partial_valid || h->p.fuse == 0) return false;
  if (h->p.nranks > 1 && !h->p2p_ready) return false;   // ncclAllReduce between the kernels stays a direct launch
  return true;
}

static bool step_graph_matches(pic1dp_gpu_t *h) {
  if (!h->step_graph) return false;
  for (int s = 0; s < h->p.nspecies; s++)
    if (h->graph_cur[s] != h->sp[s].cur || h->graph_np[s] != h->sp[s].np) return false;
  return true;
}

static int step_graph_capture(pic1dp_gpu_t *h) {
  if (h->step_graph) {
    cudaGraphExecDestroy(h->step_graph);
    h->step_graph = nullptr;
  }
  const int64_t l0 = h->launches, n0 = h->nccl_calls, p0 = h->p2p_calls;
  for (int s = 0; s < h->p.nspecies; s++) {
    h->graph_cur[s] = h->sp[s].cur;
    h->graph_np[s] = h->sp[s].np;
  }
  CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
  const int rc = step_direct(h);   // records the launches; nothing executes
  cudaGraph_t graph = nullptr;
  const cudaError_t e = cudaStreamEndCapture(h->stream, &graph);
  h->graph_launches = h->launches - l0;
  h->graph_nccl = h->nccl_calls - n0;
  h->graph_p2p = h->p2p_calls - p0;
  h->launches = l0;
  h->nccl_calls = n0;
  h->p2p_calls = p0;
  if (rc || e != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    if (!rc) h->err = std::string("step graph capture: ") + cudaGetErrorString(e);
    return rc ? rc : PIC1DP_ECUDA;
  }
  const cudaError_t e2 = cudaGraphInstantiate(&h->step_graph, graph, 0);
  cudaGraphDestroy(graph);
  if (e2 != cudaSuccess) {
    h->step_graph = nullptr;
    h->err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e2);
    return PIC1DP_ECUDA;
  }
  return PIC1DP_OK;
}

int pic1dp_gpu_step(pic1dp_gpu_t *h, int32_t nsteps) {
  if (!h || nsteps < 0) return PIC1DP_EINVAL;
  if (nsteps == 0) return PIC1DP_OK;
  int rc = check_loaded(h, "step");
  if (rc) return rc;
  CK(cudaSetDevice(h->p.device));
  if ((rc = ensure_wmax(h))) return rc;   // outside the captured graph
  if (step_graph_usable(h)) {
    if (!step_graph_matches(h) && (rc = step_graph_capture(h))) return rc;
    for (int it = 0; it < nsteps; it++) {
      CK(cudaGraphLaunch(h->step_graph, h->stream));
      h->launches += h->graph_launches;
      h->nccl_calls += h->graph_nccl;
      h->p2p_calls += h->graph_p2p;
      h->graph_replays++;
    }
    return PIC1DP_OK;   // the rotation is back at the captured set after a whole step
  }
  for (int it = 0; it < nsteps; it++)
    if ((rc = step_direct(h))) return rc;
  return PIC1DP_OK;
}

int pic1dp_gpu_profile_step(pic1dp_gpu_t *h, float ms[6]) {
  if (!h || !ms) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  int e = 0;
  CK(cudaEventRecord(h->pev[e++], h->stream));
  for (int irk = 1; irk <= 2; irk++) {
    int rc = push_impl(h, irk, h->recompute);   // the kernels of step()
    if (rc) return rc;
    CK(cudaEventRecord(h->pev[e++], h->stream));
    if (h->p.iptclshape < 4) {
      rc = pic1dp_gpu_compute_shape_x(h);
      if (rc) return rc;
    }
    rc = pic1dp_gpu_collect_charge(h);
    if (rc) return rc;
    CK(cudaEventRecord(h->pev[e++], h->stream));
    rc = pic1dp_gpu_solve_field(h);
    if (rc) return rc;
    CK(cudaEventRecord(h->pev[e++], h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  for (int i = 0; i < 6; i++) CK(cudaEventElapsedTime(&ms[i], h->pev[i], h->pev[i + 1]));
  return PIC1DP_OK;
}

int pic1dp_gpu_get_field(pic1dp_gpu_t *h, double *electric, double *chargeden, double *mode_re, double *mode_im) {
  if (!h) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  const size_t nb = (size_t)h->p.nx * 8, mb = (size_t)h->p.nmode * 8;
  if (electric) { CK(cudaMemcpyAsync(electric, h->d_E, nb, cudaMemcpyDeviceToHost, h->stream)); h->d2h += nb; }
  if (chargeden) { CK(cudaMemcpyAsync(chargeden, h->d_rho, nb, cudaMemcpyDeviceToHost, h->stream)); h->d2h += nb; }
  if (mode_re) { CK(cudaMemcpyAsync(mode_re, h->d_mre, mb, cudaMemcpyDeviceToHost, h->stream)); h->d2h += mb; }
  if (mode_im) { CK(cudaMemcpyAsync(mode_im, h->d_mim, mb, cudaMemcpyDeviceToHost, h->stream)); h->d2h += mb; }
  p2p_queue_timeout_read(h);
  CK(cudaStreamSynchronize(h->stream));
  return p2p_check_timeouts(h, "get_field");
}

int pic1dp_gpu_set_field(pic1dp_gpu_t *h, const double *electric, const double *chargeden) {
  if (!h) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  const size_t nb = (size_t)h->p.nx * 8;
  if (electric) { CK(cudaMemcpyAsync(h->d_E, electric, nb, cudaMemcpyHostToDevice, h->stream)); h->h2d += nb; }
  if (chargeden) { CK(cudaMemcpyAsync(h->d_rho, chargeden, nb, cudaMemcpyHostToDevice, h->stream)); h->h2d += nb; }
  CK(cudaStreamSynchronize(h->stream));
  return PIC1DP_OK;
}

int pic1dp_gpu_get_operators(pic1dp_gpu_t *h, double *F_re, double *F_im, double *grad_inv) {
  if (!h) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  const size_t fb = (size_t)h->p.nx * h->p.nmode * 8;
  if (F_re) CK(cudaMemcpy(F_re, h->d_Fre, fb, cudaMemcpyDeviceToHost));
  if (F_im) CK(cudaMemcpy(F_im, h->d_Fim, fb, cudaMemcpyDeviceToHost));
  if (grad_inv) CK(cudaMemcpy(grad_inv, h->d_ginv, (size_t)h->p.nmode * 8, cudaMemcpyDeviceToHost));
  return PIC1DP_OK;
}

int pic1dp_gpu_field_energy(pic1dp_gpu_t *h, double *energy) {
  if (!h || !energy) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  GridArgs g;
  fill_grid_args(h, g);
  k_field_energy<<<1, 1024, 0, h->stream>>>(g);
  CKL(h);
  CK(cudaMemcpyAsync(energy, h->d_energy, 8, cudaMemcpyDeviceToHost, h->stream));
  p2p_queue_timeout_read(h);
  CK(cudaStreamSynchronize(h->stream));
  h->d2h += 8;
  return p2p_check_timeouts(h, "field_energy");
}

static int allreduce_inplace(pic1dp_gpu_t *h, double *buf, size_t count) {
  if (h->p.nranks == 1) return PIC1DP_OK;
  if (!h->comm) { h->err = "nranks > 1 but comm_init was not called"; return PIC1DP_ESTATE; }
  ncclResult_t r = g_nccl.AllReduce(buf, buf, count, ncclDouble, ncclSum, h->comm, h->stream);
  if (r != ncclSuccess) { h->err = std::string("ncclAllReduce: ") + g_nccl.GetErrorString(r); return PIC1DP_ENCCL; }
  h->nccl_calls++;
  return PIC1DP_OK;
}

static int diag_setup(pic1dp_gpu_t *h, int ncell) {
  if (!h->d_diag_part) {
    h->diag_grid = h->nsm * 4;
    CK(cudaMalloc(&h->d_diag_part, (size_t)h->diag_grid * 3 * 8));
    CK(cudaMalloc(&h->d_diag_sums, (size_t)3 * PIC1DP_MAX_SPECIES * 8));
  }
  if (ncell > h->hist_cells) {
    if (h->d_hist) cudaFree(h->d_hist);
    if (h->d_hist_out) cudaFree(h->d_hist_out);
    h->d_hist = h->d_hist_out = nullptr;
    CK(cudaMalloc(&h->d_hist, (size_t)h->hist_copies * 3 * ncell * 8));
    CK(cudaMalloc(&h->d_hist_out, (size_t)3 * ncell * 8));
    CK(cudaMemsetAsync(h->d_hist, 0, (size_t)h->hist_copies * 3 * ncell * 8, h->stream));
    h->hist_cells = ncell;
  }
  return PIC1DP_OK;
}

static void fill_diag_args(pic1dp_gpu_t *h, int s, DiagArgs &a) {
  Species &S = h->sp[s];
  memset(&a, 0, sizeof(a));
  a.x = S.x[S.cur];
  a.v = S.v[S.cur];
  a.p = S.p;
  a.w = S.w[S.cur];
  a.np = S.np;
  a.deltaf = h->p.deltaf;
  a.sum_partial = h->d_diag_part;
  a.lx = h->p.lx;
  a.hist = h->d_hist;
  a.ncopies = h->hist_copies;
}

// scalars of output_field from the per-species device sums (src/pic1dp_output.F90:126-172)
static void output_field_scalars(const pic1dp_params &p, const double *sums, double *scalars) {
  for (int s = 0; s < p.nspecies; s++) {
    const double vv = sums[3 * s], vvp = sums[3 * s + 1], vvw = sums[3 * s + 2];
    scalars[1 + 3 * s] = vv;       // :135
    scalars[2 + 3 * s] = vvp;      // :143
    double energy;
    if (p.deltaf == 1) {
      energy = vvw;                                              // :150
      if (p.linear == 1) scalars[2 + 3 * s] = vvp + energy;      // :154
    } else {
      energy = vvp;  // "at this point energy is total energy"   // :157
      if (p.iptcldist == 1) energy = energy - 3.0 * p.density[s] * p.lx;                                   // :160
      else if (p.iptcldist == 0) energy = energy - p.temperature[s] / p.mass[s] * p.density[s] * p.lx;     // :166-168
    }
    scalars[3 + 3 * s] = energy;   // :171
  }
}

int pic1dp_gpu_output_field(pic1dp_gpu_t *h, double *scalars) {
  if (!h || !scalars) return PIC1DP_EINVAL;
  int rc = check_loaded(h, "output_field");
  if (rc) return rc;
  CK(cudaSetDevice(h->p.device));
  rc = diag_setup(h, 0);
  if (rc) return rc;
  const pic1dp_params &p = h->p;
  for (int s = 0; s < p.nspecies; s++) {
    DiagArgs a;
    fill_diag_args(h, s, a);
    k_diag<true, false><<<h->diag_grid, 512, 0, h->stream>>>(a);
    CKL(h);
    k_diag_sums_final<<<1, 32, 0, h->stream>>>(h->d_diag_part, h->diag_grid, h->d_diag_sums + 3 * s);
    CKL(h);
  }
  rc = allreduce_inplace(h, h->d_diag_sums, (size_t)3 * p.nspecies);  // VecSum is collective
  if (rc) return rc;
  GridArgs g;
  fill_grid_args(h, g);
  k_field_energy<<<1, 1024, 0, h->stream>>>(g);
  CKL(h);
  double sums[3 * PIC1DP_MAX_SPECIES];
  CK(cudaMemcpyAsync(sums, h->d_diag_sums, (size_t)3 * p.nspecies * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(&scalars[0], h->d_energy, 8, cudaMemcpyDeviceToHost, h->stream));
  p2p_queue_timeout_read(h);
  CK(cudaStreamSynchronize(h->stream));
  if ((rc = p2p_check_timeouts(h, "output_field"))) return rc;
  h->d2h += 8 + 3 * p.nspecies * 8;
  output_field_scalars(p, sums, scalars);
  return PIC1DP_OK;
}

// histogram pass of one species into d_hist_out[3][ncell] (+ the output_field sums into d_diag_sums[3 isp] when
// with_sums): one fused kernel when the private grid fits in shared memory, RED.ADD.F64 to L2 otherwise
static int launch_hist(pic1dp_gpu_t *h, int isp, int nx_opd, int nv_opd, double v_max, bool with_sums, double *d_out) {
  const int ncell = nx_opd * nv_opd;
  DiagArgs a;
  fill_diag_args(h, isp, a);
  a.nx_opd = nx_opd;
  a.nv_opd = nv_opd;
  a.v_max = v_max;
  const size_t hs = (size_t)4 * nx_opd * (nv_opd + 1) * 8;
  const size_t ls = (size_t)PIC1DP_LIMB_W * nx_opd * (nv_opd + 1) * 4;   // limb counters: [cells + spare row][PIC1DP_LIMB_W words]
  Species &S = h->sp[isp];
  if (h->limb_enabled && ls <= h->max_smem && S.np > 0) {
    // exact fixed-point histograms with native 32-bit shared-memory adds (k_diag_limb)
    if (!h->d_diag_max) {
      CK(cudaMalloc(&h->d_diag_max, (size_t)2 * PIC1DP_MAX_SPECIES * 4));
      CK(cudaMemsetAsync(h->d_diag_max, 0, (size_t)2 * PIC1DP_MAX_SPECIES * 4, h->stream));
    }
    if (ncell > h->hist_tab_cells) {
      if (h->d_hist_tab) cudaFree(h->d_hist_tab);
      h->d_hist_tab = nullptr;
      CK(cudaMalloc(&h->d_hist_tab, (size_t)h->nsm * 3 * ncell * 16));
      h->hist_tab_cells = ncell;
    }
    if (h->limb_smem_set != (int)ls) {
      CK(cudaFuncSetAttribute(k_diag_limb<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ls));
      CK(cudaFuncSetAttribute(k_diag_limb<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ls));
      h->limb_smem_set = (int)ls;
    }
    // the tables are laid out with stride 3 * ncell of THIS call
    CK(cudaMemsetAsync(h->d_hist_tab, 0, (size_t)h->nsm * 3 * ncell * 16, h->stream));
    unsigned *mx = h->d_diag_max + 2 * isp;
    if (!S.pmax_valid) {   // p does not change between marker replacements
      CK(cudaMemsetAsync(mx, 0, 4, h->stream));
      k_absmax_hi<<<h->nsm * 8, 256, 0, h->stream>>>(S.p, S.np, mx);
      CKL(h);
      S.pmax_valid = true;
    }
    // bound on |w|: the fixed-point deposit already keeps a running maximum of its source (w in delta-f runs) on the
    // device, raised by every fused kernel; otherwise one 8 B/marker pass (0.12 ms at 1e8 markers)
    const unsigned *mw = mx + 1;
    if (h->p.deltaf && h->dep == DEP_FIXED && h->p.fuse != 0 && S.wmax_valid) {   // fused: every push tracks it
      mw = h->d_wmax_hi + isp;
    } else {
      CK(cudaMemsetAsync(mx + 1, 0, 4, h->stream));
      if (h->p.deltaf) {
        k_absmax_hi<<<h->nsm * 8, 256, 0, h->stream>>>(S.w[S.cur], S.np, mx + 1);
        CKL(h);
      }
    }
    a.tab = h->d_hist_tab;
    a.max_p_hi = mx;
    a.max_w_hi = mw;
    if (with_sums) k_diag_limb<true><<<h->nsm, 1024, ls, h->stream>>>(a);
    else k_diag_limb<false><<<h->nsm, 1024, ls, h->stream>>>(a);
    CKL(h);
    if (with_sums) {
      k_diag_sums_final<<<1, 32, 0, h->stream>>>(h->d_diag_part, h->nsm, h->d_diag_sums + 3 * isp);
      CKL(h);
    }
    k_diag_limb_final<<<(3 * ncell + 63) / 64, 256, 0, h->stream>>>(h->d_hist_tab, h->nsm, ncell, mx, mw, d_out);
    CKL(h);
    return PIC1DP_OK;
  }
  if (hs <= h->max_smem) {
    if (h->hist_smem_set != (int)hs) {
      CK(cudaFuncSetAttribute(k_diag_fused<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hs));
      CK(cudaFuncSetAttribute(k_diag_fused<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hs));
      h->hist_smem_set = (int)hs;
    }
    // one CTA per SM (at most diag_grid CTAs: the sum partials are sized for that)
    if (with_sums) k_diag_fused<true><<<h->nsm, PIC1DP_DIAG_THREADS, hs, h->stream>>>(a);
    else k_diag_fused<false><<<h->nsm, PIC1DP_DIAG_THREADS, hs, h->stream>>>(a);
    CKL(h);
    if (with_sums) {
      k_diag_sums_final<<<1, 32, 0, h->stream>>>(h->d_diag_part, h->nsm, h->d_diag_sums + 3 * isp);
      CKL(h);
    }
  } else {
    if (with_sums) {
      k_diag<true, false><<<h->diag_grid, 512, 0, h->stream>>>(a);
      CKL(h);
      k_diag_sums_final<<<1, 32, 0, h->stream>>>(h->d_diag_part, h->diag_grid, h->d_diag_sums + 3 * isp);
      CKL(h);
    }
    k_diag<false, true><<<h->diag_grid, 512, 0, h->stream>>>(a);
    CKL(h);
  }
  // the private copies are laid out with stride 3*ncell of THIS call; the reduction also clears them for the next use
  k_diag_hist_final<<<(3 * ncell + 255) / 256, 256, 0, h->stream>>>(h->d_hist, h->hist_copies, 3 * ncell, d_out);
  CKL(h);
  return PIC1DP_OK;
}

// host half of output_ptcldist (src/pic1dp_output.F90:297-455) on the reduced raw histograms raw[3][ncell]
static void ptcldist_finish(const pic1dp_params &p, int isp, int nx_opd, int nv_opd, double v_max, double *raw,
                            double *markr_xv, double *total_xv, double *pertb_xv, double *markr_v, double *total_v,
                            double *pertb_v) {
  const int ncell = nx_opd * nv_opd;
  double *m_xv = raw, *t_xv = m_xv + ncell, *p_xv = t_xv + ncell;
  std::vector<double> m_v(nv_opd, 0.0), t_v(nv_opd, 0.0), p_v(nv_opd, 0.0);
  for (int iv = 0; iv < nv_opd; iv++)  // v-only histograms = sums over x of the x-v ones (sx + (1-sx) = 1)
    for (int ix = 0; ix < nx_opd; ix++) {
      m_v[iv] += m_xv[iv * nx_opd + ix];
      t_v[iv] += t_xv[iv * nx_opd + ix];
      p_v[iv] += p_xv[iv * nx_opd + ix];
    }
  if (p.linear == 1) {  // :326-329
    for (int c = 0; c < ncell; c++) t_xv[c] = t_xv[c] + p_xv[c];
    for (int iv = 0; iv < nv_opd; iv++) t_v[iv] = t_v[iv] + p_v[iv];
  }
  const double delv_inv = (double)(nv_opd - 1) / (2.0 * v_max);  // :207-208
  const double delx_inv = (double)nx_opd / p.lx;                 // :209
  for (int c = 0; c < ncell; c++) {                              // :362-363
    m_xv[c] = m_xv[c] * delx_inv * delv_inv;
    t_xv[c] = t_xv[c] * delx_inv * delv_inv;
  }
  for (int iv = 0; iv < nv_opd; iv++) {                          // :364-365
    m_v[iv] = m_v[iv] * delv_inv;
    t_v[iv] = t_v[iv] * delv_inv;
  }
  if (p.deltaf == 1) {                                           // :366-369
    for (int c = 0; c < ncell; c++) p_xv[c] = p_xv[c] * delx_inv * delv_inv;
    for (int iv = 0; iv < nv_opd; iv++) p_v[iv] = p_v[iv] * delv_inv;
  } else {                                                       // :371-455: subtract the equilibrium
    const double PETSC_PI = 3.14159265358979323846264338327950288419716939937510582;
    const double n = p.density[isp], v0 = p.v0[isp], T = p.temperature[isp], T2 = p.temperature2[isp], m = p.mass[isp];
    for (int iv = 0; iv < nv_opd; iv++) {
      const double sv = ((double)iv / (double)(nv_opd - 1) * 2.0 - 1.0) * v_max;  // :374-375
      double f0;
      if (p.iptcldist == 1)
        f0 = n * (sv * sv) * exp(-(sv * sv) / 2.0) / sqrt(2.0 * PETSC_PI);
      else if (p.iptcldist == 2)
        f0 = n * (exp(-((sv + v0) * (sv + v0)) / (2.0 * T / m)) + exp(-((sv - v0) * (sv - v0)) / (2.0 * T / m))) /
             (sqrt(8.0 * PETSC_PI) * T / m);
      else if (p.iptcldist == 3)
        f0 = n * exp(-(sv * sv) / (2.0 * T / m)) / (sqrt(2.0 * PETSC_PI) * T / m) +
             (1.0 - n) * exp(-((sv - v0) * (sv - v0)) / (2.0 * T2 / m)) / (sqrt(2.0 * PETSC_PI) * T2 / m);
      else
        f0 = n * exp(-((sv - v0) * (sv - v0)) / (2.0 * T / m)) / (sqrt(2.0 * PETSC_PI) * T / m);
      for (int ix = 0; ix < nx_opd; ix++) p_xv[iv * nx_opd + ix] = t_xv[iv * nx_opd + ix] - f0;
      p_v[iv] = t_v[iv] - p.lx * f0;
    }
  }
  if (markr_xv) memcpy(markr_xv, m_xv, (size_t)ncell * 8);
  if (total_xv) memcpy(total_xv, t_xv, (size_t)ncell * 8);
  if (pertb_xv) memcpy(pertb_xv, p_xv, (size_t)ncell * 8);
  if (markr_v) memcpy(markr_v, m_v.data(), (size_t)nv_opd * 8);
  if (total_v) memcpy(total_v, t_v.data(), (size_t)nv_opd * 8);
  if (pertb_v) memcpy(pertb_v, p_v.data(), (size_t)nv_opd * 8);
}

static int ptcldist_check(pic1dp_gpu_t *h, int32_t nx_opd, int32_t nv_opd, double v_max, const char *who) {
  if (nx_opd < 1 || nv_opd < 2 || !(v_max > 0.0) || (int64_t)nx_opd * nv_opd > (1 << 22)) {
    h->err = std::string(who) + ": bad argument";
    return PIC1DP_EINVAL;
  }
  return check_loaded(h, who);
}

int pic1dp_gpu_output_ptcldist(pic1dp_gpu_t *h, int32_t isp, int32_t nx_opd, int32_t nv_opd, double v_max,
                               double *markr_xv, double *total_xv, double *pertb_xv, double *markr_v,
                               double *total_v, double *pertb_v) {
  if (!h || isp < 0 || isp >= h->p.nspecies) { if (h) h->err = "output_ptcldist: bad species"; return PIC1DP_EINVAL; }
  int rc = ptcldist_check(h, nx_opd, nv_opd, v_max, "output_ptcldist");
  if (rc) return rc;
  CK(cudaSetDevice(h->p.device));
  const int ncell = nx_opd * nv_opd;
  if ((rc = diag_setup(h, ncell))) return rc;
  if ((rc = launch_hist(h, isp, nx_opd, nv_opd, v_max, false, h->d_hist_out))) return rc;
  rc = allreduce_inplace(h, h->d_hist_out, (size_t)3 * ncell);  // MPI_Reduce :333-357 (every rank gets the sum)
  if (rc) return rc;
  std::vector<double> raw((size_t)3 * ncell);
  CK(cudaMemcpyAsync(raw.data(), h->d_hist_out, (size_t)3 * ncell * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->d2h += (int64_t)3 * ncell * 8;
  ptcldist_finish(h->p, isp, nx_opd, nv_opd, v_max, raw.data(), markr_xv, total_xv, pertb_xv, markr_v, total_v, pertb_v);
  return PIC1DP_OK;
}

int pic1dp_gpu_output_all(pic1dp_gpu_t *h, int32_t nx_opd, int32_t nv_opd, double v_max, double *scalars, double *dist) {
  if (!h || !scalars || !dist) { if (h) h->err = "output_all: NULL output"; return PIC1DP_EINVAL; }
  int rc = ptcldist_check(h, nx_opd, nv_opd, v_max, "output_all");
  if (rc) return rc;
  CK(cudaSetDevice(h->p.device));
  const pic1dp_params &p = h->p;
  const int ncell = nx_opd * nv_opd;
  if ((rc = diag_setup(h, ncell))) return rc;
  if ((size_t)3 * ncell * p.nspecies > h->hist_all_cap) {   // reduced histograms of all species side by side
    if (h->d_hist_all) cudaFree(h->d_hist_all);
    h->d_hist_all = nullptr;
    CK(cudaMalloc(&h->d_hist_all, (size_t)3 * ncell * p.nspecies * 8));
    h->hist_all_cap = (size_t)3 * ncell * p.nspecies;
  }
  for (int s = 0; s < p.nspecies; s++)   // ONE pass over the markers of each species: sums + histograms
    if ((rc = launch_hist(h, s, nx_opd, nv_opd, v_max, true, h->d_hist_all + (size_t)3 * ncell * s))) return rc;
  if ((rc = allreduce_inplace(h, h->d_diag_sums, (size_t)3 * p.nspecies))) return rc;        // VecSum
  if ((rc = allreduce_inplace(h, h->d_hist_all, (size_t)3 * ncell * p.nspecies))) return rc;  // MPI_Reduce :333-357
  GridArgs g;
  fill_grid_args(h, g);
  k_field_energy<<<1, 1024, 0, h->stream>>>(g);
  CKL(h);
  double sums[3 * PIC1DP_MAX_SPECIES];
  std::vector<double> raw((size_t)3 * ncell * p.nspecies);
  CK(cudaMemcpyAsync(sums, h->d_diag_sums, (size_t)3 * p.nspecies * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(&scalars[0], h->d_energy, 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(raw.data(), h->d_hist_all, raw.size() * 8, cudaMemcpyDeviceToHost, h->stream));
  p2p_queue_timeout_read(h);
  CK(cudaStreamSynchronize(h->stream));
  if ((rc = p2p_check_timeouts(h, "output_all"))) return rc;
  h->d2h += 8 + 3 * p.nspecies * 8 + (int64_t)raw.size() * 8;
  output_field_scalars(p, sums, scalars);
  const size_t per = (size_t)3 * ncell + 3 * nv_opd;
  for (int s = 0; s < p.nspecies; s++) {
    double *o = dist + per * s;
    ptcldist_finish(p, s, nx_opd, nv_opd, v_max, raw.data() + (size_t)3 * ncell * s, o, o + ncell, o + 2 * ncell,
                    o + 3 * ncell, o + 3 * ncell + nv_opd, o + 3 * ncell + 2 * nv_opd);
  }
  return PIC1DP_OK;
}

// ---- marker optimisation (src/pic1dp_particle.F90:356-813) ----

int pic1dp_gpu_compute_dist_pertb_abs_v(pic1dp_gpu_t *h, int32_t nv, double v_max, double *dist) {
  if (!h || nv < 2 || nv > (1 << 20) || !(v_max > 0.0)) {
    if (h) h->err = "compute_dist_pertb_abs_v: bad argument";
    return PIC1DP_EINVAL;
  }
  int rc = check_loaded(h, "compute_dist_pertb_abs_v");
  if (rc) return rc;
  CK(cudaSetDevice(h->p.device));
  const pic1dp_params &p = h->p;
  // one private (nv + 1)-cell grid per warp in shared memory; fewer warps per CTA for large grids
  int threads = 512;
  while (threads > 32 && (size_t)(threads / 32) * (nv + 1) * 8 > h->max_smem) threads >>= 1;
  const size_t smem = (size_t)(threads / 32) * (nv + 1) * 8;
  if (smem > h->max_smem) { h->err = "compute_dist_pertb_abs_v: nv too large for a shared-memory grid"; return PIC1DP_EUNSUPPORTED; }
  if (h->dist_smem_set != (int)smem || h->dist_threads != threads) {
    CK(cudaFuncSetAttribute(k_dist_pertb_abs_v, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_dist_pertb_abs_v, threads, smem));
    h->dist_grid = h->nsm * (per_sm < 1 ? 1 : per_sm);
    h->dist_threads = threads;
    h->dist_smem_set = (int)smem;
  }
  const int need = h->dist_grid * nv + p.nspecies * nv;
  if (need > h->dist_cap) {
    if (h->d_dist_part) cudaFree(h->d_dist_part);
    h->d_dist_part = nullptr;
    CK(cudaMalloc(&h->d_dist_part, (size_t)need * 8));
    h->dist_cap = need;
  }
  double *d_out = h->d_dist_part + (size_t)h->dist_grid * nv;  // [nspecies][nv]
  for (int s = 0; s < p.nspecies; s++) {
    Species &S = h->sp[s];
    DistArgs a;
    a.v = S.v[S.cur];
    a.w = S.w[S.cur];
    a.np = S.np;
    a.nv = nv;
    a.v_max = v_max;
    a.partial = h->d_dist_part;
    k_dist_pertb_abs_v<<<h->dist_grid, threads, smem, h->stream>>>(a);
    CKL(h);
    k_dist_final<<<(nv + 255) / 256, 256, 0, h->stream>>>(h->d_dist_part, h->dist_grid, nv, d_out + (size_t)s * nv);
    CKL(h);
  }
  rc = allreduce_inplace(h, d_out, (size_t)p.nspecies * nv);  // MPI_Allreduce :392-395
  if (rc) return rc;
  h->h_dist.assign((size_t)p.nspecies * nv, 0.0);
  CK(cudaMemcpyAsync(h->h_dist.data(), d_out, (size_t)p.nspecies * nv * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->d2h += (int64_t)p.nspecies * nv * 8;
  h->opt_nv = nv;
  h->opt_vmax = v_max;
  if (dist) memcpy(dist, h->h_dist.data(), (size_t)p.nspecies * nv * 8);
  return PIC1DP_OK;
}

// D2H of the current x, v, p, w of one species into the pinned staging arrays (allocated on first use)
static int stage_species(pic1dp_gpu_t *h, int isp, const char *who) {
  if (h->opt_nv == 0) { h->err = std::string(who) + ": compute_dist_pertb_abs_v must be called first"; return PIC1DP_ESTATE; }
  CK(cudaSetDevice(h->p.device));
  const size_t bytes = (size_t)(h->p.capacity > 0 ? h->p.capacity : 1) * 8;
  for (int q = 0; q < 4; q++) {
    if (h->stage[q]) continue;
    if (cudaMallocHost(&h->stage[q], bytes) == cudaSuccess) {
      h->stage_pinned[q] = true;
    } else {  // 4 x capacity x 8 B of pinned memory can be refused on a large handle: pageable staging still works
      cudaGetLastError();
      h->stage[q] = static_cast<double *>(malloc(bytes));
      h->stage_pinned[q] = false;
      if (!h->stage[q]) { h->err = std::string(who) + ": host staging allocation failed"; return PIC1DP_ENOMEM; }
    }
  }
  return pic1dp_gpu_get_markers(h, isp, h->stage[0], h->stage[1], h->stage[2], h->stage[3], nullptr);
}

int pic1dp_gpu_particle_merge(pic1dp_gpu_t *h, double thsh, int64_t *np_out) {
  if (!h) return PIC1DP_EINVAL;
  int rc = check_loaded(h, "particle_merge");
  if (rc) return rc;
  for (int s = 0; s < h->p.nspecies; s++) {
    if ((rc = stage_species(h, s, "particle_merge"))) return rc;
    const hostopt::Markers m = {h->stage[0], h->stage[1], h->stage[2], h->stage[3]};
    const int64_t n = hostopt::merge(m, h->sp[s].np, h->h_dist.data() + (size_t)s * h->opt_nv, h->opt_nv, h->opt_vmax,
                                     thsh, h->p.nx, h->p.lx);
    if ((rc = upload_species(h, s, n, m.x, m.v, m.p, m.w))) return rc;
    if (np_out) np_out[s] = n;
  }
  return PIC1DP_OK;
}

int pic1dp_gpu_particle_remove(pic1dp_gpu_t *h, double thsh, int32_t typeremove, double remove_frac,
                               pic1dp_real64_fn dice, void *rng_ctx, int64_t *np_out) {
  if (!h || !dice || (typeremove != 1 && typeremove != 2)) {
    if (h) h->err = "particle_remove: bad argument";
    return PIC1DP_EINVAL;
  }
  int rc = check_loaded(h, "particle_remove");
  if (rc) return rc;
  for (int s = 0; s < h->p.nspecies; s++) {
    if ((rc = stage_species(h, s, "particle_remove"))) return rc;
    const hostopt::Markers m = {h->stage[0], h->stage[1], h->stage[2], h->stage[3]};
    const int64_t n = hostopt::remove(m, h->sp[s].np, h->h_dist.data() + (size_t)s * h->opt_nv, h->opt_nv, h->opt_vmax,
                                      thsh, typeremove, remove_frac, dice, rng_ctx);
    if ((rc = upload_species(h, s, n, m.x, m.v, m.p, m.w))) return rc;
    if (np_out) np_out[s] = n;
  }
  return PIC1DP_OK;
}

int pic1dp_gpu_particle_split(pic1dp_gpu_t *h, double thsh, int32_t ngroup, double dv_sig_frac,
                              pic1dp_gaussian_array_fn gauss, void *rng_ctx, int64_t *np_out) {
  if (!h || !gauss || ngroup < 1) {
    if (h) h->err = "particle_split: bad argument";
    return PIC1DP_EINVAL;
  }
  int rc = check_loaded(h, "particle_split");
  if (rc) return rc;
  for (int s = 0; s < h->p.nspecies; s++) {
    if ((rc = stage_species(h, s, "particle_split"))) return rc;
    const hostopt::Markers m = {h->stage[0], h->stage[1], h->stage[2], h->stage[3]};
    const int64_t n = hostopt::split(m, h->sp[s].np, h->p.capacity, h->h_dist.data() + (size_t)s * h->opt_nv, h->opt_nv,
                                     h->opt_vmax, thsh, ngroup, dv_sig_frac, h->p.deltaf, gauss, rng_ctx);
    if ((rc = upload_species(h, s, n, m.x, m.v, m.p, m.w))) return rc;
    if (np_out) np_out[s] = n;
  }
  return PIC1DP_OK;
}

// host halves on caller-owned arrays (no GPU involved)
int64_t pic1dp_host_particle_merge(int64_t np, double *x, double *v, double *p, double *w, const double *dist,
                                   int32_t nv, double v_max, double thsh, int32_t nx, double lx) {
  const hostopt::Markers m = {x, v, p, w};
  return hostopt::merge(m, np, dist, nv, v_max, thsh, nx, lx);
}

int64_t pic1dp_host_particle_remove(int64_t np, double *x, double *v, double *p, double *w, const double *dist,
                                    int32_t nv, double v_max, double thsh, int32_t typeremove, double remove_frac,
                                    pic1dp_real64_fn dice, void *rng_ctx) {
  const hostopt::Markers m = {x, v, p, w};
  return hostopt::remove(m, np, dist, nv, v_max, thsh, typeremove, remove_frac, dice, rng_ctx);
}

int64_t pic1dp_host_particle_split(int64_t np, int64_t capacity, double *x, double *v, double *p, double *w,
                                   const double *dist, int32_t nv, double v_max, double thsh, int32_t ngroup,
                                   double dv_sig_frac, int32_t deltaf, pic1dp_gaussian_array_fn gauss, void *rng_ctx) {
  const hostopt::Markers m = {x, v, p, w};
  return hostopt::split(m, np, capacity, dist, nv, v_max, thsh, ngroup, dv_sig_frac, deltaf, gauss, rng_ctx);
}

int pic1dp_gpu_p2p_trace(pic1dp_gpu_t *h, int32_t capacity) {
  if (!h || capacity < 0 || capacity > (1 << 20)) return PIC1DP_EINVAL;
  if (!h->p2p_ready) { h->err = "p2p_trace: the peer-memory all-reduce is not set up"; return PIC1DP_ESTATE; }
  CK(cudaSetDevice(h->p.device));
  CK(cudaStreamSynchronize(h->stream));
  if (h->d_p2p_stamps) cudaFree(h->d_p2p_stamps);
  h->d_p2p_stamps = nullptr;
  h->p2p_stamp_cap = 0;
  if (h->step_graph) {  // the captured kernels hold the old trace pointer
    cudaGraphExecDestroy(h->step_graph);
    h->step_graph = nullptr;
  }
  if (capacity > 0) {
    CK(cudaMalloc(&h->d_p2p_stamps, (size_t)capacity * 3 * 8));
    CK(cudaMemset(h->d_p2p_stamps, 0, (size_t)capacity * 3 * 8));
    h->p2p_stamp_cap = capacity;
  }
  return PIC1DP_OK;
}

int pic1dp_gpu_p2p_trace_read(pic1dp_gpu_t *h, uint64_t *stamps, int64_t *last_epoch) {
  if (!h || !stamps || !last_epoch) return PIC1DP_EINVAL;
  if (!h->d_p2p_stamps) { h->err = "p2p_trace_read: tracing is off"; return PIC1DP_ESTATE; }
  CK(cudaSetDevice(h->p.device));
  CK(cudaStreamSynchronize(h->stream));
  unsigned long long ep = 0;
  CK(cudaMemcpy(&ep, h->d_p2p_epoch, 8, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(stamps, h->d_p2p_stamps, (size_t)h->p2p_stamp_cap * 3 * 8, cudaMemcpyDeviceToHost));
  *last_epoch = (int64_t)ep;
  return PIC1DP_OK;
}

int pic1dp_gpu_sync(pic1dp_gpu_t *h) {
  if (!h) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  p2p_queue_timeout_read(h);
  CK(cudaStreamSynchronize(h->stream));
  return p2p_check_timeouts(h, "sync");
}

int pic1dp_gpu_timer_start(pic1dp_gpu_t *h) {
  if (!h) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  CK(cudaEventRecord(h->ev0, h->stream));
  return PIC1DP_OK;
}

int pic1dp_gpu_timer_stop(pic1dp_gpu_t *h, float *milliseconds) {
  if (!h || !milliseconds) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  CK(cudaEventRecord(h->ev1, h->stream));
  CK(cudaEventSynchronize(h->ev1));
  CK(cudaEventElapsedTime(milliseconds, h->ev0, h->ev1));
  return PIC1DP_OK;
}

int pic1dp_gpu_get_counters(pic1dp_gpu_t *h, pic1dp_counters *c) {
  if (!h || !c) return PIC1DP_EINVAL;
  CK(cudaSetDevice(h->p.device));
  unsigned long long noob = 0;
  CK(cudaMemcpyAsync(&noob, h->d_noob, 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  c->kernel_launches = h->launches;
  c->nccl_calls = h->nccl_calls;
  c->p2p_allreduces = h->p2p_calls;
  c->p2p_timeouts = 0;
  if (h->d_p2p_timeouts) {
    unsigned long long t = 0;
    CK(cudaMemcpy(&t, h->d_p2p_timeouts, 8, cudaMemcpyDeviceToHost));
    c->p2p_timeouts = (int64_t)t;
  }
  c->oob_markers = (int64_t)noob;
  c->h2d_bytes = h->h2d;
  c->d2h_bytes = h->d2h;
  c->deposit_mode = h->dep;
  c->grid_ctas = h->grid;
  c->cta_threads = h->threads;
  c->smem_bytes = h->smem_push;
  c->graph_replays = h->graph_replays;
  return PIC1DP_OK;
}

}  // extern "C"
