// host/pic1dp_host.cpp -- C++ host side above the C ABI (include/pic1dp_gpu.h).
//
// The reference host is Fortran 2003; no Fortran compiler exists in this image, so the host side is restated in
// C++ with the reference's own structure and names: the argument-less procedures of pic1dp_particle /
// pic1dp_field / pic1dp_interaction over module-global state, the RNG module multirand that feeds particle_load,
// and the driver sequence of `program pic1dp` (/root/reference/src/pic1dp.F90:43-125).  Every procedure forwards
// to libpic1dp_b200.so and leaves its status in global_ierr, checked by CHKERRQ like the reference does after every
// PETSc call.  One host thread per GPU ("rank"); ranks rendezvous through the library's NCCL communicator.
//
// Build:  g++ -O2 -std=c++17 -pthread -Iinclude host/pic1dp_host.cpp -Lpic1dp_b200 -lpic1dp_b200 \
//             -Wl,-rpath,'$ORIGIN/../pic1dp_b200' -o host/pic1dp_host
// Run:    host/pic1dp_host nparticle_max=6400000 nx=192 time_max=50 ngpus=1 seed_type=1 out=run.txt
//
// This is product code: it never touches oracle/.
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <time.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "pic1dp_gpu.h"

// ===================================================================================================== global
namespace pic1dp_global {
// src/pic1dp_global.F90:57-64
struct RankState {
  int global_mype = 0, global_npe = 1;
  int global_ierr = 0;
  int global_irk = 1;
  int global_itime = 0;
  double global_time = 0.0;
};
const double PETSC_PI = 3.14159265358979323846264338327950288419716939937510582;
const double PETSC_SQRT_MACHINE_EPSILON = 1.490116119384766e-08;
}  // namespace pic1dp_global

#define CHKERRQ(st, h)                                                                              \
  do {                                                                                              \
    if ((st).global_ierr) {                                                                         \
      fprintf(stderr, "[%d] %s:%d error %d (%s): %s\n", (st).global_mype, __FILE__, __LINE__,       \
              (st).global_ierr, pic1dp_gpu_strerror((st).global_ierr), pic1dp_gpu_last_error(h));   \
      exit(1);                                                                                      \
    }                                                                                               \
  } while (0)

// ====================================================================================================== input
namespace pic1dp_input {
// run-time version of the compile-time parameters of src/pic1dp_input.F90:32-256 (same names, same defaults)
struct Input {
  int64_t input_ntime_max = 900000;
  double input_time_max = 500.0;
  int input_linear = 0;
  double input_lx = 2.0 * 3.1415926535897932384626 / 0.36;
  int input_iptcldist = 3;
  int input_nspecies = 1;
  double input_species_charge = -1.0, input_species_mass = 1.0, input_species_temperature = 1.0,
         input_species_temperature2 = 1.0, input_species_density = 0.9, input_species_v0 = 5.0;
  int input_nmode = 1;
  int input_modes[PIC1DP_MAX_MODES] = {1};
  int input_init_nmode = 1;
  int input_init_mode[PIC1DP_MAX_MODES] = {1};
  double input_init_mode_cos[PIC1DP_MAX_MODES] = {0.0}, input_init_mode_sin[PIC1DP_MAX_MODES] = {1e-5};
  int input_deltaf = 1;
  double input_dt = 0.05;
  int64_t input_nparticle_max = 6400000;
  int input_imarker = 2;
  double input_v_max = 8.0;
  int input_nx = 192;
  int input_iptclshape = 4;
  int input_multirand_al_int = 3, input_multirand_seed_type = 3, input_multirand_warmup = 5;
  bool input_multirand_selftest = true;
  double input_output_interval = 0.5;
  // placement / implementation (not in the reference)
  int ngpus = 1, deposit_mode = 0, field_mode = 0, fuse = 1;
  int device_rng = 1;  // 1: KISS64 / SuperKISS64 marker streams are generated on the device; 0: host streams
  std::string out = "pic1dp_energy.txt";
  std::string petsc_out;          // when set: also write the reference's binary output file (pic1dp.out layout)
  int input_nv = 128, input_nx_opd = 64, input_nv_opd = 64;  // src/pic1dp_input.F90:131, :253-256
  // marker optimisation (src/pic1dp_input.F90:117, :146-206).  The reference hard-codes the schedules as
  // t_i = 50 + 0.5 i and the thresholds as 0.1 i / n (merge, remove) and 1 - 0.9 i / n (split); start and spacing of
  // the schedule are run-time values here (opt_t0, opt_dt), the formulas are the reference's.
  int64_t input_species_nparticle_init = -1;  // -1: input_nparticle_max (:117)
  int input_nmerge = 0, input_nremove = 0, input_nsplit = 0;
  double opt_t0 = 50.0, opt_dt = 0.5;
  int input_typeremove = 2;
  double input_remove_frac = 0.9;
  int input_split_ngroup = 5;
  double input_split_dv_sig_frac = 0.1;
  std::string markers_out;  // when set: rank 0 dumps its final x, v, p, w (raw doubles) for inspection / tests
  double input_tmerge(int i) const { return opt_t0 + i * opt_dt; }                                      // :150
  double input_thshmerge(int i) const { return 0.1 / (input_nmerge > 1 ? input_nmerge : 1) * (double)i; }   // :157
  double input_tremove(int i) const { return opt_t0 + i * opt_dt; }                                     // :166
  double input_thshremove(int i) const { return 0.1 / (input_nremove > 1 ? input_nremove : 1) * (double)i; }  // :179
  double input_tsplit(int i) const { return opt_t0 + i * opt_dt; }                                      // :192
  double input_thshsplit(int i) const { return 1.0 - 0.9 / (input_nsplit > 1 ? input_nsplit : 1) * (double)i; }  // :199
};

static bool parse(Input &in, int argc, char **argv) {
  for (int i = 1; i < argc; i++) {
    std::string a(argv[i]);
    size_t eq = a.find('=');
    if (eq == std::string::npos) return false;
    std::string k = a.substr(0, eq), v = a.substr(eq + 1);
    double d = atof(v.c_str());
    if (k == "nparticle_max") in.input_nparticle_max = (int64_t)d;
    else if (k == "nx") in.input_nx = (int)d;
    else if (k == "time_max") in.input_time_max = d;
    else if (k == "ntime_max") in.input_ntime_max = (int64_t)d;
    else if (k == "dt") in.input_dt = d;
    else if (k == "lx") in.input_lx = d;
    else if (k == "linear") in.input_linear = (int)d;
    else if (k == "deltaf") in.input_deltaf = (int)d;
    else if (k == "iptcldist") in.input_iptcldist = (int)d;
    else if (k == "iptclshape") in.input_iptclshape = (int)d;
    else if (k == "density") in.input_species_density = d;
    else if (k == "v0") in.input_species_v0 = d;
    else if (k == "temperature") in.input_species_temperature = d;
    else if (k == "temperature2") in.input_species_temperature2 = d;
    else if (k == "mass") in.input_species_mass = d;
    else if (k == "charge") in.input_species_charge = d;
    else if (k == "v_max") in.input_v_max = d;
    else if (k == "init_sin") in.input_init_mode_sin[0] = d;
    else if (k == "init_cos") in.input_init_mode_cos[0] = d;
    else if (k == "al_int") in.input_multirand_al_int = (int)d;
    else if (k == "seed_type") in.input_multirand_seed_type = (int)d;
    else if (k == "warmup") in.input_multirand_warmup = (int)d;
    else if (k == "output_interval") in.input_output_interval = d;
    else if (k == "ngpus") in.ngpus = (int)d;
    else if (k == "deposit_mode") in.deposit_mode = (int)d;
    else if (k == "field_mode") in.field_mode = (int)d;
    else if (k == "fuse") in.fuse = (int)d;
    else if (k == "out") in.out = v;
    else if (k == "petsc_out") in.petsc_out = v;
    else if (k == "nparticle_init") in.input_species_nparticle_init = (int64_t)d;
    else if (k == "nmerge") in.input_nmerge = (int)d;
    else if (k == "nremove") in.input_nremove = (int)d;
    else if (k == "nsplit") in.input_nsplit = (int)d;
    else if (k == "opt_t0") in.opt_t0 = d;
    else if (k == "opt_dt") in.opt_dt = d;
    else if (k == "typeremove") in.input_typeremove = (int)d;
    else if (k == "remove_frac") in.input_remove_frac = d;
    else if (k == "split_ngroup") in.input_split_ngroup = (int)d;
    else if (k == "split_dv_sig_frac") in.input_split_dv_sig_frac = d;
    else if (k == "markers_out") in.markers_out = v;
    else if (k == "imarker") in.input_imarker = (int)d;
    else if (k == "device_rng") in.device_rng = (int)d;
    else return false;
  }
  return true;
}

// input_init (src/pic1dp_input.F90:287-308)
static void input_init(const Input &in) {
  if (in.input_iptcldist >= 1 && in.input_imarker == 1) {
    fprintf(stderr, "Error: case of input_iptcldist >= 1 and input_imarker = 1 not implemented yet.\n");
    exit(1);
  }
  if (in.input_linear == 1 && in.input_deltaf == 0) {
    fprintf(stderr, "Error: case of input_linear = 1 and input_deltaf = 0 not implemented yet.\n");
    exit(1);
  }
  if (in.input_species_nparticle_init > in.input_nparticle_max || in.input_species_nparticle_init == 0 ||
      (in.input_typeremove != 1 && in.input_typeremove != 2) || in.input_split_ngroup < 1) {
    fprintf(stderr, "Error: bad marker-optimisation input.\n");
    exit(1);
  }
}
}  // namespace pic1dp_input

// ================================================================================================== multirand
// Product-side RNG with the reference's three engines and seeding rules (src/multirand.F90).  Self test against
// the reference's known-answer values runs at start-up like input_multirand_selftest = .true. does.
namespace multirand {
struct Generator {
  enum { NSEED = 20635 };
  std::vector<uint64_t> s = std::vector<uint64_t>(NSEED, 0);
  int iseed = 0, al = 3;

  uint64_t kiss() {  // :921-945
    uint64_t t = (s[0] << 58) + s[3];
    const uint64_t c0 = s[0] >> 63;
    s[3] = (c0 == (t >> 63)) ? (s[0] >> 6) + c0 : (s[0] >> 6) - ((s[0] + t) >> 63) + 1;
    s[0] += t;
    s[1] ^= s[1] << 13;
    s[1] ^= s[1] >> 17;
    s[1] ^= s[1] << 43;
    s[2] = 6906969069ULL * s[2] + 1234567ULL;
    return s[0] + s[1] + s[2];
  }
  uint64_t mt() {  // :952-997
    const int nn = 312, mm = 156;
    const uint64_t um = 0xFFFFFFFF80000000ULL, lm = 0x7FFFFFFFULL, mag[2] = {0, 0xB5026F5AA96619E9ULL};
    if (iseed >= nn) {
      for (int i = 0; i < nn; i++) {
        const uint64_t x = (s[i] & um) | (s[(i + 1) % nn] & lm);
        s[i] = s[(i + mm) % nn] ^ (x >> 1) ^ mag[x & 1];
      }
      iseed = 0;
    }
    uint64_t x = s[iseed++];
    x ^= (x >> 29) & 0x5555555555555555ULL;
    x ^= (x << 17) & 0x71D67FFFEDA60000ULL;
    x ^= (x << 37) & 0xFFF7EEE000000000ULL;
    return x ^ (x >> 43);
  }
  uint64_t superkiss() {  // :1004-1039
    const int nn = 20632;
    if (iseed >= nn) {
      for (int i = 0; i < nn; i++) {
        const uint64_t h = s[nn] & 1, z = ((s[i] << 41) >> 1) + ((s[i] << 39) >> 1) + (s[nn] >> 1);
        s[nn] = (s[i] >> 23) + (s[i] >> 25) + (z >> 63);
        s[i] = ~((z << 1) + h);
      }
      iseed = 0;
    }
    s[nn + 1] = s[nn + 1] * 6906969069ULL + 123;
    s[nn + 2] ^= s[nn + 2] << 13;
    s[nn + 2] ^= s[nn + 2] >> 17;
    s[nn + 2] ^= s[nn + 2] << 43;
    return s[iseed++] + s[nn + 1] + s[nn + 2];
  }
  int64_t int64() { return (int64_t)(al == 2 ? mt() : al == 3 ? superkiss() : kiss()); }
  double real64() { return (double)int64() / 18446744073709551615.0 + 0.5; }  // INT2REAL64, :49

  void default_seeds(int al_) {  // :476-518
    al = al_;
    std::fill(s.begin(), s.end(), 0);
    iseed = 0;
    if (al == 2) {
      s[0] = 5489;
      for (int i = 1; i < 312; i++) s[i] = 6364136223846793005ULL * (s[i - 1] ^ (s[i - 1] >> 62)) + (uint64_t)i;
      iseed = 312;
    } else if (al == 3) {
      s[20632] = 36243678541ULL;
      s[20633] = 12367890123456ULL;
      s[20634] = 521288629546311ULL;
      for (int i = 0; i < 20632; i++) {
        s[20633] = s[20633] * 6906969069ULL + 123;
        s[20634] ^= s[20634] << 13;
        s[20634] ^= s[20634] >> 17;
        s[20634] ^= s[20634] << 43;
        s[i] = s[20633] + s[20634];
      }
      iseed = 20632;
    } else {
      s[0] = 1234567890987654321ULL;
      s[1] = 362436362436362436ULL;
      s[2] = 1066149217761810ULL;
      s[3] = 123456123456123456ULL;
    }
  }
  bool selftest(int al_) {  // first known-answer value of each engine, :396-419
    default_seeds(al_);
    const int64_t first = int64();
    return first == (al_ == 2 ? -3932459287431434586LL : al_ == 3 ? 6140839658375754198LL : 8932985056925012148LL);
  }
  // multirand_init, seed types 1 (constant) and 3 (/dev/urandom): :244-381
  void init(int al_, int seed_type, int mype, int warmup) {
    static const int64_t primes1[100] = {
        15484219, 15484223, 15484243, 15484247, 15484279, 15484333, 15484363, 15484387, 15484393, 15484409, 15484421,
        15484453, 15484457, 15484459, 15484471, 15484489, 15484517, 15484519, 15484549, 15484559, 15484591, 15484627,
        15484631, 15484643, 15484661, 15484697, 15484709, 15484723, 15484769, 15484771, 15484783, 15484817, 15484823,
        15484873, 15484877, 15484879, 15484901, 15484919, 15484939, 15484951, 15484961, 15484999, 15485039, 15485053,
        15485059, 15485077, 15485083, 15485143, 15485161, 15485179, 15485191, 15485221, 15485243, 15485251, 15485257,
        15485273, 15485287, 15485291, 15485293, 15485299, 15485311, 15485321, 15485339, 15485341, 15485357, 15485363,
        15485383, 15485389, 15485401, 15485411, 15485429, 15485441, 15485447, 15485471, 15485473, 15485497, 15485537,
        15485539, 15485543, 15485549, 15485557, 15485567, 15485581, 15485609, 15485611, 15485621, 15485651, 15485653,
        15485669, 15485677, 15485689, 15485711, 15485737, 15485747, 15485761, 15485773, 15485783, 15485801, 15485807,
        15485837};
    static const int64_t primes2[100] = {
        7001, 7013, 7019, 7027, 7039, 7043, 7057, 7069, 7079, 7103, 7109, 7121, 7127, 7129, 7151, 7159, 7177, 7187, 7193,
        7207, 7211, 7213, 7219, 7229, 7237, 7243, 7247, 7253, 7283, 7297, 7307, 7309, 7321, 7331, 7333, 7349, 7351, 7369,
        7393, 7411, 7417, 7433, 7451, 7457, 7459, 7477, 7481, 7487, 7489, 7499, 7507, 7517, 7523, 7529, 7537, 7541, 7547,
        7549, 7559, 7561, 7573, 7577, 7583, 7589, 7591, 7603, 7607, 7621, 7639, 7643, 7649, 7669, 7673, 7681, 7687, 7691,
        7699, 7703, 7717, 7723, 7727, 7741, 7753, 7757, 7759, 7789, 7793, 7817, 7823, 7829, 7841, 7853, 7867, 7873, 7877,
        7879, 7883, 7901, 7907, 7919};
    al = al_;
    const int nseed = al == 2 ? 312 : al == 3 ? 20635 : 4;
    std::fill(s.begin(), s.end(), 0);
    bool seeded = false;
    if (seed_type == 3) {  // :256-300: /dev/urandom, re-reading the words that must not be zero
      FILE *f = fopen("/dev/urandom", "rb");
      if (f && fread(s.data(), 8, nseed, f) == (size_t)nseed) {
        seeded = true;
        auto again = [&](uint64_t &word) { return fread(&word, 8, 1, f) == 1; };
        if (al == 1) {
          while (seeded && s[1] == 0) seeded = again(s[1]);
          while (seeded && s[0] == 0 && s[3] == 0) seeded = again(s[0]) && again(s[3]);
        } else if (al == 3) {
          while (seeded && s[20634] == 0) seeded = again(s[20634]);
        }
      }
      if (f) fclose(f);
      if (!seeded) {  // the reference falls back to system_clock seeds with a warning (:257-276)
        fprintf(stderr, "[multirand_init] Warning: /dev/urandom unusable, falling back to system_clock seeds\n");
        seed_type = 2;
        std::fill(s.begin(), s.end(), 0);
      }
    }
    if (!seeded) {  // clock (seed_type 2, :303) or constant (seed_type 1, :305) seeds, rank dependent (:301-350)
      auto iabs = [](int64_t a) { return a < 0 ? -a : a; };
      int64_t clock = primes1[1];
      if (seed_type == 2) {  // system_clock(count): a monotonic tick counter
        struct timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        clock = (int64_t)ts.tv_sec * 1000 + ts.tv_nsec / 1000000;
      } else if (seed_type != 1) {
        fprintf(stderr, "[multirand_init] Error: seed_type must be 1 (constant), 2 (system_clock) or 3 (/dev/urandom)\n");
        exit(1);
      }
      int64_t k4[4];
      for (int i = 0; i < 4; i++) k4[i] = clock + primes1[iabs(clock + primes2[iabs(clock) % 100] * mype) % 100] * mype;
      for (int i = 0; i < 4; i++) k4[i] += primes2[iabs(k4[i] + primes1[iabs(clock) % 100] * i) % 100] * i;
      for (int i = 0; i < 4; i++) s[i] = (uint64_t)k4[i];
      std::vector<uint64_t> tmp(NSEED, 0);
      for (int i = 0; i < 20; i++) tmp[0] = kiss();
      for (int i = 1; i < nseed; i++) tmp[i] = kiss();
      if (al == 1) {
        while (tmp[1] == 0) tmp[1] = kiss();
        while (tmp[0] == 0 && tmp[3] == 0) {
          tmp[0] = kiss();
          tmp[3] = kiss();
        }
      }
      s = tmp;
    }
    iseed = al == 2 ? 312 : al == 3 ? 20632 : 0;
    for (int64_t i = 0; i < (int64_t)warmup * nseed; i++) (void)int64();
  }
  void real_array(double *a, int64_t n) {
    for (int64_t i = 0; i < n; i++) a[i] = real64();
  }
  // multirand_gaussian_array64 (:838-872): Marsaglia's polar method, two values per accepted point; an odd tail
  // leaves the second value in the one-slot buffer that the next call consumes first
  double spare = 0.0;
  bool has_spare = false;
  void gaussian_array(double *a, int64_t n) {
    int64_t k = 0;
    if (has_spare && n > 0) {
      a[k++] = spare;
      has_spare = false;
    }
    while (k < n) {
      double gx, gy, r2;
      do {
        gx = (double)int64() / 9223372036854775807.0;
        gy = (double)int64() / 9223372036854775807.0;
        r2 = gx * gx + gy * gy;
      } while (!(r2 > 0.0 && r2 < 1.0));
      const double f = sqrt((-2.0 * log(r2)) / r2);
      a[k++] = gx * f;
      if (k < n) {
        a[k++] = gy * f;
      } else {
        spare = gy * f;
        has_spare = true;
      }
    }
  }
};
}  // namespace multirand

// ================================================================================= per-rank "module" state
struct Rank {
  pic1dp_global::RankState g;
  const pic1dp_input::Input *in = nullptr;
  pic1dp_gpu_t *h = nullptr;
  int64_t particle_ip_low = 0, particle_ip_high = 0, particle_np = 0;
  std::vector<double> x, v;        // host scratch for the two uniform streams of particle_load
  multirand::Generator rng;        // module state of multirand (seeded in particle_load, drawn again by remove / split)
  int particle_imerge = 0, particle_iremove = 0, particle_isplit = 0;  // src/pic1dp_particle.F90:26, :73-87
  double marker_steps = 0.0;       // sum over timesteps of particle_np (throughput report)
  std::vector<double> field_electric, field_chargeden, field_mode_re, field_mode_im;
};

namespace pic1dp_particle {
// particle_init (src/pic1dp_particle.F90:66-139) + field_init (src/pic1dp_field.F90:55-212)
static void particle_init(Rank &r, const uint8_t *uid) {
  const pic1dp_input::Input &in = *r.in;
  const int64_t n = in.input_nparticle_max, npe = r.g.global_npe, me = r.g.global_mype;
  r.particle_ip_low = (n / npe) * me + (me < n % npe ? me : n % npe);  // PETSC_DECIDE split, :91, :129
  r.particle_ip_high = r.particle_ip_low + n / npe + (me < n % npe ? 1 : 0);
  pic1dp_params p;
  pic1dp_gpu_params_default(&p);
  p.nx = in.input_nx;
  p.nmode = in.input_nmode;
  for (int m = 0; m < in.input_nmode; m++) p.modes[m] = in.input_modes[m];
  p.lx = in.input_lx;
  p.dt = in.input_dt;
  p.nspecies = 1;
  p.charge[0] = in.input_species_charge;
  p.mass[0] = in.input_species_mass;
  p.temperature[0] = in.input_species_temperature;
  p.temperature2[0] = in.input_species_temperature2;
  p.density[0] = in.input_species_density;
  p.v0[0] = in.input_species_v0;
  p.iptcldist = in.input_iptcldist;
  p.deltaf = in.input_deltaf;
  p.linear = in.input_linear;
  p.iptclshape = in.input_iptclshape;
  p.capacity = r.particle_ip_high - r.particle_ip_low;
  p.device = (int)me;
  p.rank = (int)me;
  p.nranks = (int)npe;
  p.deposit_mode = in.deposit_mode;
  p.field_mode = in.field_mode;
  p.fuse = in.fuse;
  r.g.global_ierr = pic1dp_gpu_create(&p, &r.h);
  CHKERRQ(r.g, (pic1dp_gpu_t *)nullptr);
  if (npe > 1) {
    r.g.global_ierr = pic1dp_gpu_comm_init(r.h, uid);
    CHKERRQ(r.g, r.h);
  }
  r.particle_imerge = in.input_nmerge > 0 ? 1 : 0;    // :73-77
  r.particle_iremove = in.input_nremove > 0 ? 1 : 0;  // :78-82
  r.particle_isplit = in.input_nsplit > 0 ? 1 : 0;    // :83-87
  r.field_electric.resize(in.input_nx);
  r.field_chargeden.resize(in.input_nx);
  r.field_mode_re.resize(in.input_nmode);
  r.field_mode_im.resize(in.input_nmode);
}

// particle_load (src/pic1dp_particle.F90:145-269): the RNG (multirand, a sequential generator) keeps the reference's
// draw order -- the whole local array for v first (:174 / :180), then for x (:222) -- and the loader arithmetic
// (:172-237, :260-263) runs on the device.  With KISS64 (al_int = 1) or SuperKISS64 (al_int = 3, the default) the device
// also generates both streams from the generator's state -- uniform v (input_imarker = 2) or the Gaussian v of
// Maxwellian markers (input_imarker = 1) -- and the generator (with the Gaussian one-slot buffer) continues after them,
// so nothing marker-sized crosses PCIe.  With MT19937-64, or device_rng=0, the host draws the streams and they cross
// PCIe (pic1dp_gpu_load_markers / _maxwellian).  The same markers either way: bit for bit for uniform v, and for
// Gaussian v to a few ulp (the device log is not glibc's; every accept decision and every other stream is exact).
static void particle_load(Rank &r) {
  const pic1dp_input::Input &in = *r.in;
  multirand::Generator &rng = r.rng;
  if (in.input_multirand_selftest && !rng.selftest(in.input_multirand_al_int))
    fprintf(stderr, "[%d][multirand_selftest] Warning: unexpected head sequence.\n", r.g.global_mype);
  rng.init(in.input_multirand_al_int, in.input_multirand_seed_type, r.g.global_mype, in.input_multirand_warmup);
  const int64_t n = r.particle_ip_high - r.particle_ip_low;
  // unload not used particles (:240-248): the tail of the local array stays free for particle_split
  const int64_t ninit = in.input_species_nparticle_init > 0 ? in.input_species_nparticle_init : in.input_nparticle_max;
  int64_t nparticle_unload = (in.input_nparticle_max - ninit) / r.g.global_npe;
  if (r.g.global_mype == 0) nparticle_unload += (in.input_nparticle_max - ninit) % r.g.global_npe;
  r.particle_np = n - nparticle_unload;
  const int al = in.input_multirand_al_int;
  if (in.device_rng && (al == 1 || al == 3)) {
    int32_t iseed = rng.iseed, filled = rng.has_spare ? 1 : 0;
    double spare = rng.spare;
    if (in.input_imarker == 1 && al == 3)
      r.g.global_ierr = pic1dp_gpu_load_markers_maxwellian_superkiss64(
          r.h, 0, r.particle_np, n, ninit, rng.s.data(), &iseed, &filled, &spare, in.input_init_nmode, in.input_init_mode,
          in.input_init_mode_cos, in.input_init_mode_sin);
    else if (in.input_imarker == 1)
      r.g.global_ierr = pic1dp_gpu_load_markers_maxwellian_kiss64(r.h, 0, r.particle_np, n, ninit, rng.s.data(), &filled,
                                                                  &spare, in.input_init_nmode, in.input_init_mode,
                                                                  in.input_init_mode_cos, in.input_init_mode_sin);
    else if (al == 3)
      r.g.global_ierr = pic1dp_gpu_load_markers_superkiss64(r.h, 0, r.particle_np, n, ninit, rng.s.data(), &iseed,
                                                            in.input_v_max, in.input_init_nmode, in.input_init_mode,
                                                            in.input_init_mode_cos, in.input_init_mode_sin);
    else   // KISS64 jumps: pv is draws [0, n), px draws [n, 2n); the host generator then skips both
      r.g.global_ierr = pic1dp_gpu_load_markers_kiss64(r.h, 0, r.particle_np, ninit, rng.s.data(), 0, n, in.input_v_max,
                                                       in.input_init_nmode, in.input_init_mode, in.input_init_mode_cos,
                                                       in.input_init_mode_sin);
    CHKERRQ(r.g, r.h);
    if (in.input_imarker != 1 && al == 1) pic1dp_host_kiss64_jump(rng.s.data(), 2 * n);
    rng.iseed = iseed;
    rng.has_spare = filled != 0;
    rng.spare = spare;
    return;
  }
  r.v.resize(n);
  r.x.resize(n);
  if (in.input_imarker == 1)
    rng.gaussian_array(r.v.data(), n);  // :174  markers loaded like the physical Maxwellian
  else
    rng.real_array(r.v.data(), n);  // :180  (the whole local array is drawn, used or not)
  rng.real_array(r.x.data(), n);  // :222
  if (in.input_imarker == 1)
    r.g.global_ierr = pic1dp_gpu_load_markers_maxwellian(r.h, 0, r.particle_np, ninit, r.v.data(), r.x.data(),
                                                         in.input_init_nmode, in.input_init_mode,
                                                         in.input_init_mode_cos, in.input_init_mode_sin);
  else
    r.g.global_ierr = pic1dp_gpu_load_markers(r.h, 0, r.particle_np, ninit, r.v.data(), r.x.data(), in.input_v_max,
                                              in.input_init_nmode, in.input_init_mode, in.input_init_mode_cos,
                                              in.input_init_mode_sin);
  CHKERRQ(r.g, r.h);
  r.v.clear();
  r.x.clear();
}

static void particle_compute_shape_x(Rank &r) {  // :275-350
  r.g.global_ierr = pic1dp_gpu_compute_shape_x(r.h);
  CHKERRQ(r.g, r.h);
}
// RNG call-backs handed through the C ABI (the generator is this rank's module state)
static double cb_real64(void *ctx) { return static_cast<multirand::Generator *>(ctx)->real64(); }
static void cb_gaussian_array(void *ctx, double *a, int32_t n) { static_cast<multirand::Generator *>(ctx)->gaussian_array(a, n); }

static void particle_compute_dist_pertb_abs_v(Rank &r) {  // :356-403, reduced on the device
  r.g.global_ierr = pic1dp_gpu_compute_dist_pertb_abs_v(r.h, r.in->input_nv, r.in->input_v_max, nullptr);
  CHKERRQ(r.g, r.h);
}
static void particle_merge(Rank &r, double thsh_frac_dist_pertb_abs_v) {  // :411-522
  r.g.global_ierr = pic1dp_gpu_particle_merge(r.h, thsh_frac_dist_pertb_abs_v, &r.particle_np);
  CHKERRQ(r.g, r.h);
}
static void particle_remove(Rank &r, double thsh_frac_dist_pertb_abs_v) {  // :530-627
  r.g.global_ierr = pic1dp_gpu_particle_remove(r.h, thsh_frac_dist_pertb_abs_v, r.in->input_typeremove,
                                               r.in->input_remove_frac, cb_real64, &r.rng, &r.particle_np);
  CHKERRQ(r.g, r.h);
}
static void particle_split(Rank &r, double thsh_frac_dist_pertb_abs_v) {  // :635-746
  r.g.global_ierr = pic1dp_gpu_particle_split(r.h, thsh_frac_dist_pertb_abs_v, r.in->input_split_ngroup,
                                              r.in->input_split_dv_sig_frac, cb_gaussian_array, &r.rng, &r.particle_np);
  CHKERRQ(r.g, r.h);
}
// particle_optimize (:752-813): manages the calling of merge / remove / split
static void particle_optimize(Rank &r, bool &flag_optimized) {
  const pic1dp_input::Input &in = *r.in;
  flag_optimized = false;
  if (in.input_deltaf == 0) return;  // "now only support optimization for delta f"
  if (r.particle_imerge > 0 && r.particle_imerge <= in.input_nmerge) {
    if (r.g.global_time + in.input_dt >= in.input_tmerge(r.particle_imerge) && r.g.global_irk == 2) {
      particle_compute_dist_pertb_abs_v(r);
      particle_merge(r, in.input_thshmerge(r.particle_imerge));
      r.particle_imerge++;
      flag_optimized = true;
    }
  }
  if (r.particle_iremove > 0 && r.particle_iremove <= in.input_nremove) {
    if (r.g.global_time + in.input_dt >= in.input_tremove(r.particle_iremove) && r.g.global_irk == 2) {
      particle_compute_dist_pertb_abs_v(r);
      particle_remove(r, in.input_thshremove(r.particle_iremove));
      r.particle_iremove++;
      flag_optimized = true;
    }
  }
  if (r.particle_isplit > 0 && r.particle_isplit <= in.input_nsplit) {
    if (r.g.global_time + in.input_dt >= in.input_tsplit(r.particle_isplit) && r.g.global_irk == 2) {
      particle_compute_dist_pertb_abs_v(r);
      particle_split(r, in.input_thshsplit(r.particle_isplit));
      r.particle_isplit++;
      flag_optimized = true;
    }
  }
}

static void particle_final(Rank &r) {  // :819-858 (+ field_final)
  r.g.global_ierr = pic1dp_gpu_destroy(r.h);
  r.h = nullptr;
}
}  // namespace pic1dp_particle

namespace pic1dp_field {
static void field_solve_electric(Rank &r) {  // src/pic1dp_field.F90:218-270
  r.g.global_ierr = pic1dp_gpu_solve_field(r.h);
  CHKERRQ(r.g, r.h);
}
}  // namespace pic1dp_field

namespace pic1dp_interaction {
static void interaction_collect_charge(Rank &r) {  // src/pic1dp_interaction.F90:33-155
  r.g.global_ierr = pic1dp_gpu_collect_charge(r.h);
  CHKERRQ(r.g, r.h);
}
static void interaction_push_particle(Rank &r) {  // :161-370, implicit input global_irk
  r.g.global_ierr = pic1dp_gpu_push(r.h, r.g.global_irk);
  CHKERRQ(r.g, r.h);
}
}  // namespace pic1dp_interaction

namespace pic1dp_output {
// big-endian writers of the PETSc binary viewer (PetscViewerBinaryWriteInt / WriteReal / VecView)
static void put_i32(FILE *f, int32_t v) {
  unsigned char b[4] = {(unsigned char)(v >> 24), (unsigned char)(v >> 16), (unsigned char)(v >> 8), (unsigned char)v};
  fwrite(b, 1, 4, f);
}
static void put_f64(FILE *f, double d) {
  uint64_t u;
  memcpy(&u, &d, 8);
  unsigned char b[8];
  for (int i = 0; i < 8; i++) b[i] = (unsigned char)(u >> (56 - 8 * i));
  fwrite(b, 1, 8, f);
}
static void put_vec(FILE *f, const std::vector<double> &v) {  // VecView: VEC_FILE_CLASSID, n, values
  put_i32(f, 1211214);
  put_i32(f, (int32_t)v.size());
  for (double d : v) put_f64(f, d);
}
// output_init header (src/pic1dp_output.F90:74-92)
static void output_init(const pic1dp_input::Input &in, FILE *f) {
  put_i32(f, in.input_nspecies);
  put_i32(f, in.input_nmode);
  put_i32(f, in.input_nx);
  put_i32(f, in.input_nv);
  put_i32(f, in.input_nx_opd);
  put_i32(f, in.input_nv_opd);
  for (int m = 0; m < in.input_nmode; m++) put_i32(f, in.input_modes[m]);
  put_f64(f, in.input_lx);
  put_f64(f, in.input_v_max);
}
// output_all = output_field + output_ptcldist (src/pic1dp_output.F90:100-189, :196-477) from device-side reductions
static void output_all(Rank &r, FILE *f) {
  const pic1dp_input::Input &in = *r.in;
  double sc[1 + 3 * PIC1DP_MAX_SPECIES];
  r.g.global_ierr = pic1dp_gpu_output_field(r.h, sc);
  CHKERRQ(r.g, r.h);
  r.g.global_ierr = pic1dp_gpu_get_field(r.h, r.field_electric.data(), r.field_chargeden.data(), r.field_mode_re.data(),
                                         r.field_mode_im.data());
  CHKERRQ(r.g, r.h);
  const int nc = in.input_nx_opd * in.input_nv_opd;
  std::vector<double> mxv(nc), txv(nc), pxv(nc), mv(in.input_nv_opd), tv(in.input_nv_opd), pv(in.input_nv_opd);
  r.g.global_ierr = pic1dp_gpu_output_ptcldist(r.h, 0, in.input_nx_opd, in.input_nv_opd, in.input_v_max, mxv.data(),
                                               txv.data(), pxv.data(), mv.data(), tv.data(), pv.data());
  CHKERRQ(r.g, r.h);
  if (!f || r.g.global_mype != 0) return;  // only the root process writes (:457-474)
  put_f64(f, r.g.global_time);
  for (int i = 0; i < 1 + 3 * in.input_nspecies; i++) put_f64(f, sc[i]);
  put_vec(f, r.field_mode_re);
  put_vec(f, r.field_mode_im);
  put_vec(f, r.field_electric);
  put_vec(f, r.field_chargeden);
  for (auto *a : {&mxv, &txv, &pxv, &mv, &tv, &pv})
    for (double d : *a) put_f64(f, d);
  fflush(f);
}

// scalar part of output_field (src/pic1dp_output.F90:117-124, :178-181): t, int E^2 dx, mode_re, mode_im
static void output_field(Rank &r, FILE *f) {
  double energy = 0.0;
  r.g.global_ierr = pic1dp_gpu_field_energy(r.h, &energy);
  CHKERRQ(r.g, r.h);
  r.g.global_ierr = pic1dp_gpu_get_field(r.h, r.field_electric.data(), r.field_chargeden.data(), r.field_mode_re.data(),
                                         r.field_mode_im.data());
  CHKERRQ(r.g, r.h);
  if (f && r.g.global_mype == 0)
    fprintf(f, "%.17g %.17g %.17g %.17g\n", r.g.global_time, energy, r.field_mode_re[0], r.field_mode_im[0]);
}
}  // namespace pic1dp_output

// ===================================================================================================== driver
static int check_termination(const Rank &r) {  // src/pic1dp.F90:133-148
  return (r.g.global_itime >= r.in->input_ntime_max ||
          r.g.global_time + pic1dp_global::PETSC_SQRT_MACHINE_EPSILON >= r.in->input_time_max)
             ? 1
             : 0;
}

static void run_rank(const pic1dp_input::Input *in, int mype, int npe, const uint8_t *uid, double *steps_per_s) {
  Rank r;
  r.in = in;
  r.g.global_mype = mype;
  r.g.global_npe = npe;
  FILE *f = (mype == 0) ? fopen(in->out.c_str(), "w") : nullptr;
  FILE *fb = (mype == 0 && !in->petsc_out.empty()) ? fopen(in->petsc_out.c_str(), "wb") : nullptr;
  const bool binary = !in->petsc_out.empty();
  if (fb) pic1dp_output::output_init(*in, fb);
  pic1dp_input::input_init(*in);
  pic1dp_particle::particle_init(r, uid);  // + field_init
  pic1dp_particle::particle_load(r);
  if (in->input_iptclshape < 4) pic1dp_particle::particle_compute_shape_x(r);  // src/pic1dp.F90:65
  r.g.global_itime = 0;
  r.g.global_time = 0.0;
  pic1dp_interaction::interaction_collect_charge(r);  // :71
  pic1dp_field::field_solve_electric(r);              // :72
  pic1dp_output::output_field(r, f);                  // :74
  if (binary) pic1dp_output::output_all(r, fb);
  pic1dp_gpu_timer_start(r.h);
  int itermination = check_termination(r);
  while (itermination == 0) {  // :78-109
    for (r.g.global_irk = 1; r.g.global_irk <= 2; r.g.global_irk++) {
      pic1dp_interaction::interaction_push_particle(r);
      bool flag_optimized;
      pic1dp_particle::particle_optimize(r, flag_optimized);  // src/pic1dp.F90:82 (off in the default input)
      if (flag_optimized && mype == 0)                        // output_progress(2), :83
        printf("t=%g: marker optimisation, %lld markers on rank 0\n", r.g.global_time + in->input_dt, (long long)r.particle_np);
      if (in->input_iptclshape < 4) pic1dp_particle::particle_compute_shape_x(r);
      pic1dp_interaction::interaction_collect_charge(r);
      pic1dp_field::field_solve_electric(r);
    }
    r.g.global_itime++;
    r.g.global_time += in->input_dt;
    r.marker_steps += (double)r.particle_np;
    itermination = check_termination(r);
    const double eps = pic1dp_global::PETSC_SQRT_MACHINE_EPSILON;
    if (fmod(r.g.global_time + eps, in->input_output_interval) <
            fmod(r.g.global_time + eps - in->input_dt, in->input_output_interval) ||
        itermination == 1) {
      pic1dp_output::output_field(r, f);  // :98-108
      if (binary) pic1dp_output::output_all(r, fb);
    }
  }
  float ms = 0.f;
  pic1dp_gpu_timer_stop(r.h, &ms);
  if (steps_per_s) *steps_per_s = r.marker_steps / (ms * 1e-3);
  pic1dp_counters c;
  pic1dp_gpu_get_counters(r.h, &c);
  if (mype == 0)
    printf("steps=%d markers/rank=%lld kernels=%lld nccl=%lld oob=%lld deposit_mode=%d  %.3e particle-steps/s/rank (wall incl. outputs)\n",
           r.g.global_itime, (long long)r.particle_np, (long long)c.kernel_launches, (long long)c.nccl_calls,
           (long long)c.oob_markers, c.deposit_mode, r.marker_steps / (ms * 1e-3));
  if (mype == 0 && !in->markers_out.empty()) {  // final marker arrays of rank 0: int64 np, then x, v, p, w
    std::vector<double> buf((size_t)r.particle_np * 4);
    int64_t n = 0;
    double *b = buf.data();
    r.g.global_ierr = pic1dp_gpu_get_markers(r.h, 0, b, b + r.particle_np, b + 2 * r.particle_np, b + 3 * r.particle_np, &n);
    CHKERRQ(r.g, r.h);
    if (FILE *fm = fopen(in->markers_out.c_str(), "wb")) {
      fwrite(&n, 8, 1, fm);
      fwrite(b, 8, (size_t)n * 4, fm);
      fclose(fm);
    }
  }
  pic1dp_particle::particle_final(r);
  if (f) fclose(f);
  if (fb) fclose(fb);
}

// `pic1dp_host multirand_selftest`: prints the head of every engine after the default seeds (the reference's known-answer
// values, src/multirand.F90:396-425) and, after the rank-dependent constant-seed initialisation, uniform and Gaussian
// draws -- no GPU needed, so the product-side RNG can be checked on any machine (tests/test_capi_cpu.py).
static int multirand_selftest_dump() {
  for (int al = 1; al <= 3; al++) {
    multirand::Generator g;  // fresh module state per engine (like the reference, init does not clear the Gaussian buffer)
    g.default_seeds(al);
    printf("default %d", al);
    for (int i = 0; i < 10; i++) printf(" %lld", (long long)g.int64());
    printf("\n");
    g.init(al, 1, 2, 5);
    printf("real64 %d", al);
    for (int i = 0; i < 5; i++) printf(" %a", g.real64());
    printf("\n");
    double a[7], b[4];
    g.gaussian_array(a, 7);  // odd count: the second value of the last pair stays buffered ...
    g.gaussian_array(b, 4);  // ... and is consumed first by the next call
    printf("gauss %d", al);
    for (double t : a) printf(" %a", t);
    for (double t : b) printf(" %a", t);
    printf("\n");
  }
  return 0;
}

int main(int argc, char **argv) {
  if (argc == 2 && std::string(argv[1]) == "multirand_selftest") return multirand_selftest_dump();
  pic1dp_input::Input in;
  if (!pic1dp_input::parse(in, argc, argv)) {
    fprintf(stderr, "usage: %s [key=value ...]  (keys: nparticle_max nx time_max dt ngpus seed_type out ...)\n", argv[0]);
    return 2;
  }
  printf("PIC1D hot path on B200 (libpic1dp_b200, ABI %d): %lld markers, nx=%d, dt=%g, t_max=%g, %d GPU(s)\n",
         pic1dp_gpu_abi_version(), (long long)in.input_nparticle_max, in.input_nx, in.input_dt, in.input_time_max, in.ngpus);
  uint8_t uid[PIC1DP_UNIQUE_ID_BYTES] = {0};
  if (in.ngpus > 1) {
    int rc = pic1dp_gpu_comm_unique_id(uid);
    if (rc) {
      fprintf(stderr, "comm_unique_id: %s: %s\n", pic1dp_gpu_strerror(rc), pic1dp_gpu_last_error(nullptr));
      return 1;
    }
  }
  std::vector<std::thread> th;
  std::vector<double> rate(in.ngpus, 0.0);
  for (int r = 0; r < in.ngpus; r++) th.emplace_back(run_rank, &in, r, in.ngpus, uid, &rate[r]);
  for (auto &t : th) t.join();
  return 0;
}
