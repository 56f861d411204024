/*
 * include/pic1dp_gpu.h -- C ABI of the B200-native PIC1D hot path (libpic1dp_b200.so).
 *
 * This is the drop-in boundary for the per-timestep vector-matrix PIC cycle of PIC1D-PETSc
 * (wenjundeng/pic1dp).  The reference has no plugin registry: the path sits behind argument-less Fortran
 * module procedures over module-global PETSc Vec/Mat state.  Each entry point below cites the reference
 * interface it replaces (file:line into the reference tree); fortran/pic1dp_gpu_shim.F90 shows the
 * ISO_C_BINDING side a maintainer adds inside pic1dp_particle / pic1dp_field / pic1dp_interaction
 * (INTEGRATION.md walks through it).
 *
 * Conventions
 *  - Plain C: pointers, sizes, POD structs.  No torch / CUDA types in any signature.
 *  - Every call returns int: 0 = PIC1DP_OK, otherwise a PIC1DP_E* code; the Fortran shim stores it into
 *    global_ierr and applies CHKERRQ exactly as it does after PETSc calls (src/pic1dp_global.F90:59).
 *    pic1dp_gpu_strerror() maps a code to text; pic1dp_gpu_last_error() returns the detailed message of
 *    the last failure on that handle.
 *  - The library owns all device memory from create to destroy.  Host pointers are borrowed for the
 *    duration of one call.  Marker arrays held by the host go stale between get_markers calls.
 *  - One host thread <-> one handle <-> one GPU <-> one CUDA stream.  Calls are asynchronous on that stream
 *    and ordered; calls that return data to the host synchronise.  Not thread-safe per handle (neither is the
 *    reference: module save state, src/multirand.F90:43-44).
 *  - All marker and grid data are fp64 (PetscScalar real double, src/pic1dp_global.F90:28-30); cell indices
 *    int32 (PetscInt).
 */
#ifndef PIC1DP_GPU_H
#define PIC1DP_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIC1DP_ABI_VERSION 2
#define PIC1DP_MAX_SPECIES 4
#define PIC1DP_MAX_MODES 64
#define PIC1DP_UNIQUE_ID_BYTES 128

/* error codes */
enum {
  PIC1DP_OK = 0,
  PIC1DP_EINVAL = 1,      /* bad argument / parameter combination (input_init checks, src/pic1dp_input.F90:292-307) */
  PIC1DP_ECUDA = 2,       /* CUDA runtime error (message in last_error) */
  PIC1DP_ENCCL = 3,       /* NCCL error or NCCL library not loadable */
  PIC1DP_ENOMEM = 4,      /* device/host allocation failed */
  PIC1DP_ESTATE = 5,      /* call sequence error (e.g. push before markers were set) */
  PIC1DP_ECAPACITY = 6,   /* marker count exceeds the capacity given at create */
  PIC1DP_ENODEVICE = 7,   /* no CUDA device: this library has no CPU fallback */
  PIC1DP_EUNSUPPORTED = 8 /* requested mode not available for these parameters (e.g. smem grid too large) */
};

/* deposit (S^T w) strategies; all give the same sum up to fp64 summation order */
enum {
  PIC1DP_DEPOSIT_AUTO = 0,       /* fastest strategy that fits: FIXED (native 32-bit shared-memory adds; up to 2^20 markers
                                    per CTA), else WARP_PRIVATE for nx <= 256, SMEM_ATOMIC, else GLOBAL_RED */
  PIC1DP_DEPOSIT_SMEM_ATOMIC = 1,/* per-CTA shared-memory grid of {left,right} pairs, 128-bit CAS; CTA partials reduced
                                    in fixed order */
  PIC1DP_DEPOSIT_GLOBAL_RED = 2, /* RED.ADD.F64 into an L2-resident per-CTA private grid */
  PIC1DP_DEPOSIT_WARP_PRIVATE = 3,/* per-warp private shared-memory grid, lane-ordered duplicate merge: bitwise
                                    run-to-run deterministic ("deterministic deposition"); needs >= 8 nx-sized grids in
                                    shared memory (nx <~ 2900) and degrades to FIXED beyond that */
  PIC1DP_DEPOSIT_FIXED = 4       /* per-CTA grid of 64-bit FIXED-POINT left / right sums (value * 2^e, e from the running
                                    max |w|), each add = two native 32-bit shared-memory adds (low word, high word +
                                    carry): integer adds are order-independent, so the density is bitwise reproducible
                                    for any nx the grid fits (<~ 9600), within ~1e-14 max|w| per contribution of the
                                    fp64 sum */
};

/* how the fused kernel reads marker arrays */
enum {
  PIC1DP_LOAD_AUTO = 0,
  PIC1DP_LOAD_DIRECT = 1, /* 128-bit streaming loads into registers, 2 markers per thread */
  PIC1DP_LOAD_TMA = 2,    /* cp.async.bulk tiles into a shared-memory ring (mbarrier pipeline) */
  PIC1DP_LOAD_CPASYNC = 3 /* per-thread cp.async (LDGSTS.128) into thread-private slots of a 2-stage shared-memory ring:
                             next tile in flight during the current one, no barrier; used where the ring fits */
};

/*
 * arithmetic of the weight push (src/pic1dp_interaction.F90:266-331).  Cell index, weights, gather, x and v are
 * evaluated in the reference's operation order in BOTH modes and are bit-identical to it given the same inputs.
 */
enum {
  PIC1DP_ARITH_STRICT = 0,   /* tmp2 = -d ln f0/dv exactly as written at :275-326: two exponentials, every division and
                                rounding of the reference (w then differs from glibc only through exp, <= 1 ulp) */
  PIC1DP_ARITH_TOLERANCE = 1 /* two-stream2 / bump-on-tail: numerator and denominator divided through by the first
                                exponential, so ONE exponential of the difference of the two arguments and fused
                                multiply-adds; algebraically identical, w agrees with STRICT to a few ulp
                                (tested <= 1e-14 of max|w| per substep; north_star bar 1e-12) */
};

/* field-solve summation order for the partial-DFT projections */
enum {
  PIC1DP_FIELD_TREE = 0,      /* fixed-shape block tree reduction (deterministic, fast) */
  PIC1DP_FIELD_SEQUENTIAL = 1 /* j = 0..nx-1 in order: bit-identical to sequential-AIJ MatMultTranspose on one rank */
};

/*
 * Run-time copy of the reference's compile-time parameters that the hot path reads
 * (src/pic1dp_input.F90:32-256), plus placement.  Fill with pic1dp_gpu_params_default() first.
 */
typedef struct pic1dp_params {
  int32_t abi_version;                      /* PIC1DP_ABI_VERSION */
  int32_t struct_bytes;                     /* sizeof(pic1dp_params) */
  /* grid and field (src/pic1dp_input.F90:47, :75-80, :128) */
  int32_t nx;                               /* input_nx */
  int32_t nmode;                            /* input_nmode */
  int32_t modes[PIC1DP_MAX_MODES];          /* input_modes */
  double lx;                                /* input_lx */
  double dt;                                /* input_dt (:109) */
  /* species (:57-72) */
  int32_t nspecies;                         /* input_nspecies */
  double charge[PIC1DP_MAX_SPECIES];        /* input_species_charge */
  double mass[PIC1DP_MAX_SPECIES];          /* input_species_mass */
  double temperature[PIC1DP_MAX_SPECIES];   /* input_species_temperature */
  double temperature2[PIC1DP_MAX_SPECIES];  /* input_species_temperature2 */
  double density[PIC1DP_MAX_SPECIES];       /* input_species_density */
  double v0[PIC1DP_MAX_SPECIES];            /* input_species_v0 */
  /* model switches */
  int32_t iptcldist;                        /* input_iptcldist (:54) 0 Maxwellian 1 two-stream1 2 two-stream2 3 bump-on-tail */
  int32_t deltaf;                           /* input_deltaf (:106) */
  int32_t linear;                           /* input_linear (:43) */
  int32_t iptclshape;                       /* input_iptclshape (:138): 1,2 -> right weight `frac` and matrix-path
                                               scaling (src/pic1dp_particle.F90:322-323, interaction.F90:46-78);
                                               3,4 -> right weight 1-(1-frac), array-path scaling (:79-151) */
  /* placement */
  int64_t capacity;                         /* local marker capacity per species (this rank's share of input_nparticle_max) */
  int32_t device;                           /* CUDA device ordinal */
  int32_t rank;                             /* global_mype */
  int32_t nranks;                           /* global_npe */
  /* implementation choices */
  int32_t deposit_mode;                     /* PIC1DP_DEPOSIT_* */
  int32_t field_mode;                       /* PIC1DP_FIELD_* */
  int32_t fuse;                             /* 1: push also wraps x and deposits (collect_charge then only reduces);
                                               0: each call has exactly the reference's side effects */
  int32_t load_path;                        /* PIC1DP_LOAD_*: how marker tiles reach the SM (delta-f nonlinear kernels) */
  int32_t arith_mode;                       /* PIC1DP_ARITH_*: evaluation of -d ln f0/dv on the w path */
  int32_t no_step_graph;                    /* 1: pic1dp_gpu_step launches its kernels one by one instead of replaying a
                                               captured CUDA graph of the timestep */
  int32_t reserved[5];
} pic1dp_params;

typedef struct pic1dp_gpu pic1dp_gpu_t; /* opaque handle: the module-global state of the three Fortran modules */

/* defaults of src/pic1dp_input.F90 (electron bump-on-tail, nx=192, 1 mode, dt=0.05, delta-f nonlinear, shape 4) */
void pic1dp_gpu_params_default(pic1dp_params *p);

/* library / ABI identification */
int pic1dp_gpu_abi_version(void);
const char *pic1dp_gpu_strerror(int code);
const char *pic1dp_gpu_last_error(const pic1dp_gpu_t *h); /* h may be NULL: last create() failure */

/*
 * create: replaces particle_init (src/pic1dp_particle.F90:66-139: VecCreate/VecDuplicate of x,v,p,w,*_bak) and
 * field_init (src/pic1dp_field.F90:55-212: field Vecs, 1/k operator :158-174, partial-DFT matrices :176-210).
 * Validates parameters like input_init (src/pic1dp_input.F90:287-308).  Fails with PIC1DP_ENODEVICE when no
 * GPU is present -- there is no CPU fallback.
 */
int pic1dp_gpu_create(const pic1dp_params *p, pic1dp_gpu_t **out);

/* destroy: replaces particle_final (src/pic1dp_particle.F90:819-858) and field_final (src/pic1dp_field.F90:315-348) */
int pic1dp_gpu_destroy(pic1dp_gpu_t *h);

/*
 * Multi-GPU: replaces MPI_COMM_WORLD as used by MPI_Allreduce at src/pic1dp_interaction.F90:132-133.
 * Rank 0 calls comm_unique_id, the host broadcasts the 128 bytes (MPI_Bcast in the Fortran host,
 * torch.distributed in bench.py), every rank calls comm_init.  With nranks == 1 neither call is needed and
 * NCCL is never loaded.
 */
int pic1dp_gpu_comm_unique_id(uint8_t id[PIC1DP_UNIQUE_ID_BYTES]);
int pic1dp_gpu_comm_init(pic1dp_gpu_t *h, const uint8_t id[PIC1DP_UNIQUE_ID_BYTES]);

/*
 * Optional peer-memory all-reduce (one process per GPU, NVLink/NVSwitch): instead of ncclAllReduce, the reduce kernel
 * of every rank stores its partial density straight into an exchange buffer on every peer GPU and raises a flag; the
 * next kernel waits for all flags and sums the nranks partial grids in rank order, so the density is bitwise
 * identical on every rank and run-to-run.  Each rank exports a 64-byte IPC handle of its exchange buffer, the host
 * all-gathers the handles (MPI_Allgather / torch.distributed), every rank imports all nranks*64 bytes.
 * comm_init is still required (it is the fallback and is used by the diagnostics).  Processes only: IPC handles cannot
 * be opened by the process that exported them.
 */
#define PIC1DP_IPC_HANDLE_BYTES 64
int pic1dp_gpu_p2p_export(pic1dp_gpu_t *h, uint8_t handle[PIC1DP_IPC_HANDLE_BYTES]);
int pic1dp_gpu_p2p_import(pic1dp_gpu_t *h, const uint8_t *all_handles /* nranks * PIC1DP_IPC_HANDLE_BYTES */);

/*
 * Rendezvous trace of the peer-memory all-reduce (measurement aid): with capacity > 0 the kernels stamp %globaltimer
 * (ns) when this rank publishes its partial density, when its gather kernel starts waiting and when the wait ends --
 * 3 stamps per all-reduce in a ring of `capacity` entries indexed by epoch % capacity; capacity = 0 turns it off.
 * trace_read copies the ring (capacity * 3 values) and the epoch of the last all-reduce.  (wait_end - publish) of the
 * rank that arrived last is the exchange latency; for the others the excess is arrival skew.
 */
int pic1dp_gpu_p2p_trace(pic1dp_gpu_t *h, int32_t capacity);
int pic1dp_gpu_p2p_trace_read(pic1dp_gpu_t *h, uint64_t *stamps, int64_t *last_epoch);

/*
 * set_markers: H2D of one species after particle_load (src/pic1dp_particle.F90:145-269 fills x,v,p,w through
 * VecGetArrayF90).  np = particle_np(ispecies) (:248).  isp is 0-based.
 */
int pic1dp_gpu_set_markers(pic1dp_gpu_t *h, int32_t isp, int64_t np, const double *x, const double *v,
                           const double *p, const double *w);

/*
 * load_markers: the arithmetic of particle_load for uniform-v markers (input_imarker = 2,
 * src/pic1dp_particle.F90:179-264) on the device.  The host keeps the RNG (multirand is sequential) and passes the
 * two uniform [0, 1] streams in the order particle_load draws them: rand_v (multirand_real_array(pv), :180) and rand_x
 * (:222).  On the device: v = (rand_v - 0.5) * 2 * v_max (:181), p = f0(v) * lx * 2 v_max / nparticle_init (:182-218),
 * x = rand_x * lx (:223), w = sum over init modes of cos/sin (:225-232) * p * pertb_shape (= 1, :235-236), and
 * p = p + w for nonlinear runs (:260-263).  Halves the host-to-device traffic of set_markers (16 instead of 32 B per
 * marker).  np = markers of this rank, nparticle_init = input_species_nparticle_init (all ranks together).
 */
int pic1dp_gpu_load_markers(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init, const double *rand_v,
                            const double *rand_x, double v_max, int32_t init_nmode, const int32_t *init_mode,
                            const double *init_mode_cos, const double *init_mode_sin);

/*
 * load_markers_maxwellian: the same for input_imarker = 1 (src/pic1dp_particle.F90:172-178, iptcldist = 0 only, as
 * input_init enforces, src/pic1dp_input.F90:291-299): gauss_v is the multirand_gaussian_array(pv) stream (:174), the
 * device forms v = gauss_v * sqrt(T/m) + v0 (:175-176) and p = n * lx / nparticle_init (:177-178); x, w and the
 * nonlinear p = p + w as in load_markers.
 */
int pic1dp_gpu_load_markers_maxwellian(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init,
                                       const double *gauss_v, const double *rand_x, int32_t init_nmode,
                                       const int32_t *init_mode, const double *init_mode_cos,
                                       const double *init_mode_sin);

/*
 * ---- device-side random streams: particle_load without a marker-sized host-to-device copy ----
 *
 * load_markers_kiss64: load_markers with the two uniform streams generated ON THE DEVICE by Marsaglia's 64-bit KISS,
 * the generator multirand_al_int = 1 selects (src/multirand.F90:921-945), bit for bit.  seeds = multirand_seeds(0:3)
 * as multirand_init leaves them (any seed_type; :256-381 stay on the host: a few dozen generator calls), offset_v /
 * offset_x = how many 64-bit outputs the host generator would have produced before the first element of this rank's
 * pv / px arrays (particle_load draws the whole local Vec: offset_v = 2 * isp * nlocal, offset_x = offset_v + nlocal,
 * nlocal = particle_ip_high - particle_ip_low, :180, :222).  Each device thread jumps the three recurrences of KISS64
 * (LCG, xorshift, multiply-with-carry) to its chunk in O(log offset) and then runs the sequential generator; the
 * uniforms are INT2REAL64 of its outputs (:49).  Afterwards the host advances its own state with
 * pic1dp_host_kiss64_jump(seeds, 2 * nlocal * nspecies) so that later draws (particle_remove, particle_split)
 * continue the same stream.  SuperKISS64 (al_int = 3) has its own loader below, and both generators have a
 * Maxwellian loader (input_imarker = 1) below; MT19937-64 (al_int = 2) streams keep coming from the host through
 * load_markers / load_markers_maxwellian.
 */
int pic1dp_gpu_load_markers_kiss64(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init,
                                   const uint64_t seeds[4], int64_t offset_v, int64_t offset_x, double v_max,
                                   int32_t init_nmode, const int32_t *init_mode, const double *init_mode_cos,
                                   const double *init_mode_sin);

/*
 * load_markers_counter: the same with a counter-based generator (Philox-4x32-10) for synthetic markers that need no
 * reference stream: the uniforms of marker i depend only on (seed, isp, first_index + i), so any decomposition over
 * ranks loads the same global marker set (first_index = global index of this rank's first marker).
 */
int pic1dp_gpu_load_markers_counter(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nparticle_init, uint64_t seed,
                                    int64_t first_index, double v_max, int32_t init_nmode, const int32_t *init_mode,
                                    const double *init_mode_cos, const double *init_mode_sin);

/*
 * load_markers_superkiss64: load_markers with the two uniform streams generated ON THE DEVICE by Marsaglia's 64-bit
 * SuperKISS, the generator multirand_al_int = 3 selects (the reference's default input, src/multirand.F90:1004-1039),
 * bit for bit.  seeds = multirand_seeds(0:20634) and *iseed = the table position (0 .. 20632), both as multirand_init
 * (or earlier draws) left them.  The device draws in particle_load's order: nlocal numbers for pv (:180), then nlocal
 * for px (:222), nlocal = particle_ip_high - particle_ip_low >= np; the unloaded tail of each array (nlocal > np) is
 * generated and discarded.  Its lag-20632 multiply-with-carry table has no practical jump: one CTA advances it
 * sequentially in shared memory, each refill a parallel scan over the carry chain; a grid-wide kernel adds the LCG
 * and xorshift parts, jumped per chunk.  Before returning, seeds and *iseed are overwritten with the state after the
 * 2 * nlocal draws (a synchronous 165 KB device-to-host copy), so later host draws (particle_remove, particle_split)
 * continue the same stream.  PIC1DP_EINVAL for *iseed outside [0, 20632], nlocal < np or NULL pointers.
 */
#define PIC1DP_SUPERKISS64_NSEED 20635 /* multirand_nseed: 20632 table words, carry, LCG, xorshift */
int pic1dp_gpu_load_markers_superkiss64(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nlocal,
                                        int64_t nparticle_init, uint64_t seeds[PIC1DP_SUPERKISS64_NSEED],
                                        int32_t *iseed, double v_max, int32_t init_nmode, const int32_t *init_mode,
                                        const double *init_mode_cos, const double *init_mode_sin);

/*
 * load_markers_maxwellian_kiss64 / _superkiss64: load_markers_maxwellian (input_imarker = 1, iptcldist = 0,
 * src/pic1dp_particle.F90:172-178) with BOTH of particle_load's streams generated ON THE DEVICE from the generator's
 * state: multirand_gaussian_array(pv, nlocal) (:174; Marsaglia's polar method, src/multirand.F90:838-872), then
 * multirand_real_array(px, nlocal) (:222), nlocal = particle_ip_high - particle_ip_low >= np; elements past np are drawn
 * and discarded.  The Gaussian call's one-slot buffer is part of the state: *gauss_filled / *gauss_buf = the value
 * a previous gaussian_array left buffered (it becomes element 0 without a draw), and on return the value the call leaves
 * buffered when it needs an odd number of values after that (element nlocal).  Attempts are pairs of draws; whether one
 * is accepted depends on its own two words and is decided with the reference's IEEE operations, so the draws consumed,
 * the x stream and the returned state are exact; the Gaussian values x * sqrt(-2 log(w) / w) go through the device log
 * and match the host's to a few ulp.  The device works in rounds of PIC1DP_GAUSS_ROUND_DRAWS draws (32 MB of scratch)
 * and reads one count per round.  State in / out: KISS64 seeds = multirand_seeds(0:3); SuperKISS64 seeds =
 * multirand_seeds(0:20634) and *iseed = the table position (its x stream is regenerated from a copy of the table taken
 * at the start of the round that holds the last attempt, at most one round of draws).  On success the state is the one
 * after all draws of both calls, so later host draws (particle_remove, particle_split's gaussian_array) continue the
 * same stream.  PIC1DP_EINVAL for iptcldist != 0, nlocal < np, *iseed outside [0, 20632] or NULL pointers,
 * PIC1DP_ECAPACITY for np > capacity; a refused call leaves the state untouched.
 */
#define PIC1DP_GAUSS_ROUND_DRAWS 4194304
int pic1dp_gpu_load_markers_maxwellian_kiss64(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nlocal,
                                              int64_t nparticle_init, uint64_t seeds[4], int32_t *gauss_filled,
                                              double *gauss_buf, int32_t init_nmode, const int32_t *init_mode,
                                              const double *init_mode_cos, const double *init_mode_sin);
int pic1dp_gpu_load_markers_maxwellian_superkiss64(pic1dp_gpu_t *h, int32_t isp, int64_t np, int64_t nlocal,
                                                   int64_t nparticle_init, uint64_t seeds[PIC1DP_SUPERKISS64_NSEED],
                                                   int32_t *iseed, int32_t *gauss_filled, double *gauss_buf,
                                                   int32_t init_nmode, const int32_t *init_mode,
                                                   const double *init_mode_cos, const double *init_mode_sin);
/* the last Maxwellian load of this handle: draws its Gaussian call consumed, rounds it ran, and the SuperKISS64 draws
 * it generated a second time for the x stream (0 for KISS64) */
int pic1dp_gpu_last_gaussian_load(pic1dp_gpu_t *h, int64_t *draws, int64_t *rounds, int64_t *regenerated);

/* debug / parity: n uniforms of the device KISS64 stream starting at `offset`, copied to the host */
int pic1dp_gpu_kiss64_uniforms(pic1dp_gpu_t *h, const uint64_t seeds[4], int64_t offset, int64_t n, double *out);

/* the same generator code on the host (no handle, no GPU): jump advances multirand_seeds(0:3) by n outputs in
 * O(log n); fill writes n uniforms (multirand_real_array) and advances the state; counter_uniforms = the two streams
 * of load_markers_counter */
int pic1dp_host_kiss64_jump(uint64_t seeds[4], int64_t n);
int pic1dp_host_kiss64_fill(uint64_t seeds[4], int64_t n, double *out);

/* parity: n uniforms of the device SuperKISS64 stream from (seeds, *iseed), copied to the host; the state is advanced
 * past them like load_markers_superkiss64 does */
int pic1dp_gpu_superkiss64_uniforms(pic1dp_gpu_t *h, uint64_t seeds[PIC1DP_SUPERKISS64_NSEED], int32_t *iseed,
                                    int64_t n, double *out);
/* no handle, no GPU: fill = the sequential SuperKISS64 generator (n uniforms of multirand_real_array, state advanced);
 * refill = one table refill done the way the device does it, as a scan over the carry maps of nchunks chunks
 * (1024 = the kernel's chunking), for checking the device algorithm against the sequential recurrence */
int pic1dp_host_superkiss64_fill(uint64_t seeds[PIC1DP_SUPERKISS64_NSEED], int32_t *iseed, int64_t n, double *out);
int pic1dp_host_superkiss64_refill(uint64_t seeds[PIC1DP_SUPERKISS64_NSEED], int32_t nchunks);
void pic1dp_host_counter_uniforms(uint64_t seed, int32_t stream, int64_t first_index, int64_t n, double *u_v,
                                  double *u_x);

/*
 * get_markers: D2H refresh of the host Vecs before pic1dp_output reads them (src/pic1dp_output.F90:128-150,
 * :228-237) or before particle_optimize.  Any of x,v,p,w may be NULL.  *np receives particle_np.
 */
int pic1dp_gpu_get_markers(pic1dp_gpu_t *h, int32_t isp, double *x, double *v, double *p, double *w, int64_t *np);

/*
 * compute_shape_x: replaces particle_compute_shape_x (src/pic1dp_particle.F90:275-350) for iptclshape 1-3:
 * wraps x in place (:308-310).  No matrix or (index, weight) array is materialised -- weights are recomputed
 * on the fly with the rounding that iptclshape selects.  No-op for iptclshape 4, as in the reference driver
 * (src/pic1dp.F90:65, :86).
 */
int pic1dp_gpu_compute_shape_x(pic1dp_gpu_t *h);

/*
 * get_shape_x: the (index, weight) arrays that particle_compute_shape_x stores for iptclshape 3
 * (particle_shape_x_indexes / particle_shape_x_values, src/pic1dp_particle.F90:47-48, :331-332) and the two
 * matrix values of a row for iptclshape 1,2 (:320-323), computed from the current x without modifying it:
 * indexes[i] = left cell ix1, values_left[i] = 1-frac, values_right[i] = frac (shape 1,2) or 1-(1-frac) (3,4).
 * Debug / parity interface: the hot path never stores these.  Any output pointer may be NULL.
 */
int pic1dp_gpu_get_shape_x(pic1dp_gpu_t *h, int32_t isp, int32_t *indexes, double *values_left,
                           double *values_right);

/*
 * collect_charge: replaces interaction_collect_charge (src/pic1dp_interaction.F90:33-155): wrap x (:102-104),
 * deposit S^T w (:96-114), species charge (:126-127), all-reduce over ranks (:132-133), scale to density
 * (:140-148).  Result: field_chargeden on every rank.
 */
int pic1dp_gpu_collect_charge(pic1dp_gpu_t *h);

/*
 * solve_field: replaces field_solve_electric (src/pic1dp_field.F90:218-270): partial DFT of rho onto the kept
 * modes, 1/k, inverse.  Results: field_electric, field_mode_re, field_mode_im.  Solved redundantly on every rank
 * (replaces the E all-gather VecScatter at src/pic1dp_interaction.F90:197-206).
 */
int pic1dp_gpu_solve_field(pic1dp_gpu_t *h);

/*
 * push: replaces interaction_push_particle (src/pic1dp_interaction.F90:161-370) for global_irk = irk (1 or 2):
 * backup (:178-189, done by buffer rotation, no copy), gather S.E (:243-257), push x (:261), w (:266-331),
 * v (:335-338).  With params.fuse == 1 the wrap + deposit of the following collect_charge is folded in.
 */
int pic1dp_gpu_push(pic1dp_gpu_t *h, int32_t irk);

/*
 * step: nsteps iterations of the reference time loop body (src/pic1dp.F90:79-93):
 * do irk = 1,2 { push; [compute_shape_x]; collect_charge; solve_field }.  Same results as the individual calls.
 */
int pic1dp_gpu_step(pic1dp_gpu_t *h, int32_t nsteps);

/* field access: field_electric, field_chargeden, field_mode_re, field_mode_im (src/pic1dp_field.F90:27-31);
 * any pointer may be NULL.  get synchronises. */
int pic1dp_gpu_get_field(pic1dp_gpu_t *h, double *electric, double *chargeden, double *mode_re, double *mode_im);
/* set field_chargeden / field_electric from the host (what field_test does with VecSetValues,
 * src/pic1dp_field.F90:286-297); either may be NULL */
int pic1dp_gpu_set_field(pic1dp_gpu_t *h, const double *electric, const double *chargeden);

/* the partial-DFT operators built at create (src/pic1dp_field.F90:158-210): F_re, F_im row-major [j*nmode+m],
 * grad_inv[nmode]; any may be NULL */
int pic1dp_gpu_get_operators(pic1dp_gpu_t *h, double *F_re, double *F_im, double *grad_inv);

/* field energy |E|_2^2 * lx / nx (src/pic1dp_output.F90:120-123), reduced on the device */
int pic1dp_gpu_field_energy(pic1dp_gpu_t *h, double *energy);

/*
 * output_field: the scalars output_field writes per record (src/pic1dp_output.F90:117-172), reduced on the device
 * and over ranks (VecNorm / VecSum are collective): scalars[0] = |E|^2*lx/nx, then per species s:
 * scalars[1+3s] = sum v^2, scalars[2+3s] = sum v^2 p (+ sum v^2 w when linear, :152-155),
 * scalars[3+3s] = sum v^2 w (delta-f) or the full-f perturbed energy (:156-170).  1 + 3*nspecies doubles.
 * Replaces the host-side VecPointwiseMult/VecSum over marker Vecs: no marker leaves the GPU.
 */
int pic1dp_gpu_output_field(pic1dp_gpu_t *h, double *scalars);

/*
 * output_ptcldist: the six arrays output_ptcldist writes per species (src/pic1dp_output.F90:196-477): bilinear x-v
 * histograms of markers g, total f and perturbed delta f on an nx_opd x nv_opd grid ([iv*nx_opd + ix]) and their
 * v-only counterparts, binned on the device, summed over ranks (MPI_Reduce, :333-357; here every rank receives the
 * result), scaled by 1/(dx dv) (:362-371) and, for full-f, reduced by the equilibrium (:372-455).
 * markers with |v| >= v_max are skipped (:241).  Any output pointer may be NULL.
 */
int pic1dp_gpu_output_ptcldist(pic1dp_gpu_t *h, int32_t isp, int32_t nx_opd, int32_t nv_opd, double v_max,
                               double *markr_xv, double *total_xv, double *pertb_xv, double *markr_v,
                               double *total_v, double *pertb_v);

/*
 * output_all: what one call of output_all does on the marker side (src/pic1dp_output.F90:488-520: output_field, then
 * output_ptcldist for every species) in ONE pass over x, v, p, w per species: the fused kernel accumulates the
 * output_field sums and the x-v histograms together, so an output step reads each marker once.  scalars as in
 * output_field (1 + 3*nspecies); dist = per species [markr_xv | total_xv | pertb_xv | markr_v | total_v | pertb_v]
 * (3*nx_opd*nv_opd + 3*nv_opd doubles each), same definitions as output_ptcldist.
 */
int pic1dp_gpu_output_all(pic1dp_gpu_t *h, int32_t nx_opd, int32_t nv_opd, double v_max, double *scalars, double *dist);

/*
 * ---- marker optimisation: particle_optimize's workers (src/pic1dp_particle.F90:356-746) ----
 * particle_optimize itself (:752-813) is schedule logic (input_tmerge / _tremove / _tsplit against global_time, only at
 * global_irk == 2, delta-f only) and stays in the host; it is called between push and collect_charge
 * (src/pic1dp.F90:82), so a host that optimises must drive that substep with the individual entry points
 * (push, [optimise], collect_charge, solve_field) instead of step().
 *
 * compute_dist_pertb_abs_v: replaces particle_compute_dist_pertb_abs_v (:356-403): per species
 * dist[iv] = sum over markers with |v| < v_max of |w| x linear weight on the nv-point v grid, reduced on the device and
 * over ranks (MPI_Allreduce, :392-395).  dist (may be NULL) receives particle_dist_pertb_abs_v as [nspecies][nv]; the
 * handle keeps a copy for the three routines below.  nv = input_nv, v_max = input_v_max.
 */
int pic1dp_gpu_compute_dist_pertb_abs_v(pic1dp_gpu_t *h, int32_t nv, double v_max, double *dist);

/* RNG call-backs: the host owns the generator (multirand is sequential and rank-seeded, src/multirand.F90).
 * real64 = multirand_real64() (:644-650); gaussian_array fills a[0..n) like multirand_gaussian_array (:838-872). */
typedef double (*pic1dp_real64_fn)(void *rng_ctx);
typedef void (*pic1dp_gaussian_array_fn)(void *rng_ctx, double *a, int32_t n);

/*
 * particle_merge / particle_remove / particle_split (src/pic1dp_particle.F90:411-522, :530-627, :635-746) for every
 * species of this rank, thsh = thsh_frac_dist_pertb_abs_v.  The three algorithms are sequential by definition (a freed
 * slot is refilled by the LAST marker and examined again; pairs form in visiting order; one RNG stream is consumed in
 * visiting order), so each call stages x, v, p, w in pinned host memory, runs the reference's visiting order there and
 * copies the survivors back (32 B/marker each way, a few events per run).  They use the dist of the last
 * compute_dist_pertb_abs_v call (PIC1DP_ESTATE without one).  np_out (may be NULL) receives particle_np per species.
 * remove: typeremove = input_typeremove (1 or 2), remove_frac = input_remove_frac.
 * split: ngroup = input_split_ngroup, dv_sig_frac = input_split_dv_sig_frac; capacity given at create bounds growth.
 */
int pic1dp_gpu_particle_merge(pic1dp_gpu_t *h, double thsh, int64_t *np_out);
int pic1dp_gpu_particle_remove(pic1dp_gpu_t *h, double thsh, int32_t typeremove, double remove_frac,
                               pic1dp_real64_fn dice, void *rng_ctx, int64_t *np_out);
int pic1dp_gpu_particle_split(pic1dp_gpu_t *h, double thsh, int32_t ngroup, double dv_sig_frac,
                              pic1dp_gaussian_array_fn gauss, void *rng_ctx, int64_t *np_out);

/* The same host halves on caller-owned arrays (no handle, no GPU): for a host that already holds fresh marker arrays,
 * and for testing the visiting order without a device.  Return the new particle_np.  split: arrays hold `capacity`. */
int64_t pic1dp_host_particle_merge(int64_t np, double *x, double *v, double *p, double *w, const double *dist,
                                   int32_t nv, double v_max, double thsh, int32_t nx, double lx);
int64_t pic1dp_host_particle_remove(int64_t np, double *x, double *v, double *p, double *w, const double *dist,
                                    int32_t nv, double v_max, double thsh, int32_t typeremove, double remove_frac,
                                    pic1dp_real64_fn dice, void *rng_ctx);
int64_t pic1dp_host_particle_split(int64_t np, int64_t capacity, double *x, double *v, double *p, double *w,
                                   const double *dist, int32_t nv, double v_max, double thsh, int32_t ngroup,
                                   double dv_sig_frac, int32_t deltaf, pic1dp_gaussian_array_fn gauss, void *rng_ctx);

/* block until all queued work of this handle is done; surfaces asynchronous CUDA errors */
int pic1dp_gpu_sync(pic1dp_gpu_t *h);

/* ---- instrumentation (replaces the wtimer slots global_iwt_push_particle / _collect_charge / _mpiallredu /
 * _field_electric, src/pic1dp_global.F90:38-50, with CUDA events on the handle's stream) ---- */
int pic1dp_gpu_timer_start(pic1dp_gpu_t *h);
int pic1dp_gpu_timer_stop(pic1dp_gpu_t *h, float *milliseconds); /* synchronises */

typedef struct pic1dp_counters {
  int64_t kernel_launches;   /* kernels of this library launched on this handle so far */
  int64_t nccl_calls;        /* ncclAllReduce calls issued */
  int64_t p2p_allreduces;    /* density all-reduces done through peer memory instead of NCCL */
  int64_t p2p_timeouts;      /* peer flags that never arrived (bounded spin): results are invalid when non-zero */
  int64_t oob_markers;       /* markers whose wrapped x was exactly lx (ix == nx; the reference writes out of
                                bounds there, src/pic1dp_interaction.F90:104-113); deposited as ix=0, s=1 */
  int64_t h2d_bytes;         /* bytes copied host->device by this handle */
  int64_t d2h_bytes;         /* bytes copied device->host */
  int32_t deposit_mode;      /* resolved PIC1DP_DEPOSIT_* */
  int32_t grid_ctas;         /* CTAs of the particle kernels */
  int32_t cta_threads;
  int32_t smem_bytes;        /* dynamic shared memory of the fused kernel */
  int64_t graph_replays;     /* timesteps executed by replaying the captured CUDA graph of the step */
} pic1dp_counters;
int pic1dp_gpu_get_counters(pic1dp_gpu_t *h, pic1dp_counters *c);

/* per-kernel device time of one profiled timestep (each launch bracketed by events; slower than step()):
 * ms[0] push+deposit irk=1, ms[1] reduce+allreduce irk=1, ms[2] field irk=1, ms[3..5] same for irk=2 */
int pic1dp_gpu_profile_step(pic1dp_gpu_t *h, float ms[6]);

/* launch timing: between start and stop every fused particle-kernel launch of push() / step() is bracketed by a pair
 * of CUDA events on the handle's stream (up to 8192 launches).  stop synchronises and returns, per substep
 * (index 0: irk = 1, index 1: irk = 2), the summed device time in ms and the number of launches -- the per-launch
 * average over a whole timed region rather than over one separately profiled step. */
int pic1dp_gpu_launch_timing_start(pic1dp_gpu_t *h);
int pic1dp_gpu_launch_timing_stop(pic1dp_gpu_t *h, double ms_sum[2], int64_t launches[2]);

#ifdef __cplusplus
}
#endif
#endif /* PIC1DP_GPU_H */
