// drsim_device.cuh -- __host__ __device__ building blocks of the demand-response step.
//
// Everything here is shared by the fused tile kernel, the general 3-kernel path and (for the
// env-level scalars) the host-side debug entry points of the C ABI, so the CPU test-suite can
// exercise the same code that runs on the device.  Reference citations are relative to
// /root/reference/server/app.
#pragma once

#include <cstdint>
#include <cmath>

#include "../../include/drsim.h"

#if defined(__CUDACC__)
#define DRSIM_HD __host__ __device__ __forceinline__
#define DRSIM_D __device__ __forceinline__
#else
#define DRSIM_HD inline
#define DRSIM_D inline
#endif

namespace drsim {

// ------------------------------------------------------------------------------------------
// calendar: naive seconds since 1970-01-01 -> civil fields (the reference carries a naive
// datetime.datetime, environment.py:87; we carry its integer second count)
// ------------------------------------------------------------------------------------------
struct Civil {
  int year, month, day, hour, minute, second, yday;
};

DRSIM_HD int64_t days_from_civil(int y, int m, int d) {
  y -= m <= 2;
  const int64_t era = (y >= 0 ? y : y - 399) / 400;
  const int yoe = (int)(y - era * 400);
  const int doy = (153 * (m + (m > 2 ? -3 : 9)) + 2) / 5 + d - 1;
  const int doe = yoe * 365 + yoe / 4 - yoe / 100 + doy;
  return era * 146097 + (int64_t)doe - 719468;
}

DRSIM_HD Civil civil_from_epoch(int64_t s) {
  int64_t days = s / 86400;
  int64_t rem = s - days * 86400;
  if (rem < 0) { rem += 86400; days -= 1; }
  Civil c;
  c.hour = (int)(rem / 3600);
  c.minute = (int)((rem % 3600) / 60);
  c.second = (int)(rem % 60);
  const int64_t z = days + 719468;
  const int64_t era = (z >= 0 ? z : z - 146096) / 146097;
  const int doe = (int)(z - era * 146097);
  const int yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
  int y = (int)(yoe + era * 400);
  const int doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
  const int mp = (5 * doy + 2) / 153;
  c.day = doy - (153 * mp + 2) / 5 + 1;
  c.month = mp < 10 ? mp + 3 : mp - 9;
  y += (c.month <= 2);
  c.year = y;
  c.yday = (int)(days - days_from_civil(y, 1, 1)) + 1;  // datetime.timetuple().tm_yday
  return c;
}

// ------------------------------------------------------------------------------------------
// utils/utils.py:42-117 -- solar cooling load polynomial (same term order as the reference)
// ------------------------------------------------------------------------------------------
DRSIM_HD double solar_gain(const Civil &t, double window_area, double shading_coeff) {
  const double x = t.hour + t.minute / 60.0 - 7.5;
  double scl = 0.0;
  if (!(x < 0 || x > 10)) {
    const double y = t.month + t.day / 30.0 - 1;
    const double x2 = x * x, x3 = x2 * x, x4 = x3 * x;
    const double y2 = y * y, y3 = y2 * y, y4 = y3 * y;
    scl = 4.36579418e01 + x * 1.58055357e02 + y * 8.76635241e01 + x2 * -4.55944821e01 +
          x2 * y * 3.24275366e00 + x2 * y2 * -4.56096472e-01 + y2 * -1.47795612e01 +
          x * y2 * 4.68950855e00 + x * y * -3.73313090e01 + x3 * 5.78827663e00 +
          y3 * 1.04354810e00 + x3 * y * 2.12969604e-02 + x3 * y2 * 2.58881400e-03 +
          x3 * y3 * -5.11397219e-04 + x2 * y3 * 1.56398008e-02 + x * y3 * -1.18302764e-01 +
          x4 * -2.71446436e-01 + y4 * -3.97855577e-02;
  }
  return window_area * shading_coeff * scl;
}

// environment.py:132-159
DRSIM_HD double od_temp_model(const Civil &t, double day_temp, double night_temp, double phase,
                              double noise) {
  const double amplitude = (day_temp - night_temp) / 2.0;
  const double bias = (day_temp + night_temp) / 2.0;
  const double delay = -6.0 + phase;
  const double time_day = t.hour + t.minute / 60.0;
  const double two_pi = 2 * 3.141592653589793;
  double temperature = amplitude * sin(two_pi * (time_day + delay) / 24.0) + bias;
  temperature += noise;
  return temperature;
}

// utils/utils.py:4-23
template <typename real>
DRSIM_HD real deadband_l2(real target, real deadband, real value) {
  const real hi = target + deadband / 2;
  const real lo = target - deadband / 2;
  if (hi < value) return (value - hi) * (value - hi);
  if (lo > value) return (lo - value) * (lo - value);
  return (real)0;
}

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11), counter-based: block(key, counter) -> 4 x u32
// ------------------------------------------------------------------------------------------
struct U4 {
  uint32_t x, y, z, w;
};

DRSIM_HD void mulhilo32(uint32_t a, uint32_t b, uint32_t &hi, uint32_t &lo) {
  const uint64_t p = (uint64_t)a * (uint64_t)b;
  hi = (uint32_t)(p >> 32);
  lo = (uint32_t)p;
}

DRSIM_HD U4 philox4x32_10(uint64_t key, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
  uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    mulhilo32(0xD2511F53u, c0, hi0, lo0);
    mulhilo32(0xCD9E8D57u, c2, hi1, lo1);
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return U4{c0, c1, c2, c3};
}

enum : uint32_t { PURPOSE_OD = 1, PURPOSE_PERLIN = 2, PURPOSE_INTERP = 3, PURPOSE_RESET = 4, PURPOSE_RESET_ENV = 5 };
// (6 = PURPOSE_POLICY, drsim_actor.cuh)
constexpr uint32_t PURPOSE_NEIGHBOUR = 7;

// `random_sample` neighbours (cluster.py:96-99: random.sample(ids without n, c) per agent per step): a uniformly
// random ordered c-tuple of distinct houses other than `house`, as a sparse partial Fisher-Yates shuffle of the
// M = n_global - 1 other ids.  Step j draws r_j = j + mulhi(u_j, M - j) (Lemire's map without rejection: each value
// has probability within (M - j) / 2^32 <= M / 2^32 of uniform), swaps positions j and r_j of the virtual identity
// array and outputs the value now at position j, mapped past the house itself (v + (v >= house)).  Only the swaps are
// recorded: the value at a position p >= j is `held` of the last earlier step whose r_i was p, else p.  The words u_j
// are philox4x32_10(seed, rep, house, draw, PURPOSE_NEIGHBOUR | (j / 4) << 8), four per block.  next() yields
// outputs 0, 1, ... in turn; pick(k) advances to output k (both halves of a row split over two lanes).
struct CommSampler {
  uint64_t seed;
  uint32_t rep, house, draw, M;
  int j;
  U4 blk;
  int32_t pos[DRSIM_MAX_SAMPLE_COMM], held[DRSIM_MAX_SAMPLE_COMM];
  DRSIM_HD CommSampler(uint64_t seed_, uint32_t rep_, uint32_t house_, uint32_t draw_, uint32_t n_global)
      : seed(seed_), rep(rep_), house(house_), draw(draw_), M(n_global - 1u), j(0), blk{0, 0, 0, 0} {}
  DRSIM_HD int next() {
    const int w = j & 3;
    if (w == 0) blk = philox4x32_10(seed, rep, house, draw, PURPOSE_NEIGHBOUR | ((uint32_t)(j >> 2) << 8));
    const uint32_t u = w == 0 ? blk.x : w == 1 ? blk.y : w == 2 ? blk.z : blk.w;
    uint32_t hi, lo;
    mulhilo32(u, M - (uint32_t)j, hi, lo);
    const int r = j + (int)hi;
    int v = r, hj = j;
    for (int i = 0; i < j; ++i) {   // ascending: the last swap that wrote a position wins
      v = pos[i] == r ? held[i] : v;
      hj = pos[i] == j ? held[i] : hj;
    }
    pos[j] = r;
    held[j] = hj;
    ++j;
    return v + (v >= (int)house ? 1 : 0);
  }
  DRSIM_HD int pick(int k) {
    while (j < k) next();
    return next();
  }
};

DRSIM_HD double u01_open_closed(uint32_t x) { return ((double)x + 1.0) * 2.3283064365386963e-10; }  // (0,1]

// standard normal from one Philox block (Box-Muller on the first two words)
DRSIM_HD double philox_normal(uint64_t key, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
  const U4 r = philox4x32_10(key, c0, c1, c2, c3);
  const double u1 = u01_open_closed(r.x), u2 = u01_open_closed(r.y);
  return sqrt(-2.0 * log(u1)) * cos(2 * 3.141592653589793 * u2);
}

// random.triangular(low, high, mode) by inversion of the CDF
DRSIM_HD double triangular_from_u(double u, double lo, double hi, double mode) {
  const double fc = (mode - lo) / (hi - lo);
  if (u < fc) return lo + sqrt(u * (hi - lo) * (mode - lo));
  return hi - sqrt((1.0 - u) * (hi - lo) * (hi - mode));
}
DRSIM_HD double u01_half_open(uint32_t x) { return (double)x * 2.3283064365386963e-10; }  // [0,1)

// 1-D gradient ("Perlin") noise with +-1 lattice gradients drawn from Philox, octave weights of
// perlin.py:41-56 (note the last weight 1/(2^n - 1), quirk Q7).  Values are OUR definition: the
// reference uses the third-party `perlin_noise` package whose values are parity-unpinned.
DRSIM_HD double philox_perlin(uint64_t key, uint32_t env, double x_over_period, int nb_octaves,
                              int octaves_step) {
  double noise = 0.0;
  for (int j = 0; j < nb_octaves; ++j) {
    const double octaves = (double)((1 << j) * octaves_step);
    const double xs = x_over_period * octaves;
    const double fl = floor(xs);
    const double f = xs - fl;
    const uint32_t i0 = (uint32_t)(int64_t)fl;
    const U4 a = philox4x32_10(key, env, i0, (uint32_t)j, PURPOSE_PERLIN);
    const U4 b = philox4x32_10(key, env, i0 + 1u, (uint32_t)j, PURPOSE_PERLIN);
    const double g0 = (a.x & 1u) ? 1.0 : -1.0, g1 = (b.x & 1u) ? 1.0 : -1.0;
    const double fade = f * f * f * (f * (f * 6.0 - 15.0) + 10.0);
    const double v = g0 * f + fade * (g1 * (f - 1.0) - g0 * f);
    const double w = (j < nb_octaves - 1) ? 1.0 / (double)(1 << j) : 1.0 / (double)((1 << nb_octaves) - 1);
    noise += v * w;
  }
  return noise;
}

// ------------------------------------------------------------------------------------------
// flattened, kernel-side view of drsim_config (doubles; converted to `real` where used)
// ------------------------------------------------------------------------------------------
// exact unsigned division by a launch-invariant divisor (Granlund & Montgomery, PLDI'94):
// q = (t + ((n - t) >> s1)) >> s2 with t = mulhi(m, n)
struct FastDiv {
  uint32_t m, s1, s2, d;
};
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f;
  uint32_t l = 0;
  while ((1ull << l) < d) ++l;
  f.m = (uint32_t)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
  f.s1 = l < 1 ? l : 1;
  f.s2 = l > 1 ? l - 1 : 0;
  f.d = d;
  return f;
}
DRSIM_HD uint32_t fast_div(uint32_t n, const FastDiv &f) {
#if defined(__CUDA_ARCH__)
  const uint32_t t = __umulhi(f.m, n);
#else
  const uint32_t t = (uint32_t)(((uint64_t)f.m * n) >> 32);
#endif
  return (t + ((n - t) >> f.s1)) >> f.s2;
}

// fp32 hot-path constants, filled on the host so the kernels read them straight from the constant
// bank (no per-thread fp64 -> fp32 conversions, no divisions)
struct HotF {
  float db, half_db, inv_cop, inv_nrs, inv_n, neg_inv_opl, rew_scale, deadband;
};

struct SimParams {
  int R, N, Ns;  // replicas, houses, house stride (N rounded up to 4)
  HotF hf;
  FastDiv fd_dur, fd_ns;  // seconds_since_off / lockout_duration ; slot / Ns
  double inv_cop, inv_nrs, inv_norm_temp, inv_n_global, inv_norm_sig;  // reciprocals (fp32 build, fast epilogue)
  int dt;
  int64_t house_offset, n_global, rep_offset;
  double deadband, cop, latent, window_area, shading;
  int lockout_duration, solar_on;
  double default_target, dUa, dCa, dCm, dHm, dcap;
  double day_temp, night_temp, temp_std, phase;
  double alpha_temp, alpha_sig, nrs, norm_temp, norm_sig;
  int penalty_mode;
  double a_ind, a_cl2, a_cmax;
  int base_mode, interp_period, interp_k, signal_mode, n_terms, nb_octaves, octaves_step, period;
  double avg_power, amp_per_hvac;
  double amp[DRSIM_MAX_SIGNAL_TERMS], periods[DRSIM_MAX_SIGNAL_TERMS];
  int obs_layout, nb_comm, comm_mode, comm_per_rep;
  int st_solar, st_thermal, st_hvac, msg_thermal, msg_hvac;
  int own_dim, msg_dim, obs_dim;
  int noise_mode, policy;
  uint64_t seed;
};

// Same signal from pre-generated time-dependent parts (k_schedule): `aux` = sum_k ratio_k sin(2 pi t/T_k)
// (sinusoidals) or the noise value (perlin); t_sec = seconds since midnight.
DRSIM_HD double grid_signal_sched(const SimParams &p, double base, int t_sec, double aux,
                                  double artificial_ratio, double max_power) {
  double v = base;
  if (p.signal_mode == DRSIM_SIG_SINUSOIDALS) {
    v = base + base * aux;
  } else if (p.signal_mode == DRSIM_SIG_REGULAR_STEPS) {
    const double amplitude = p.amp_per_hvac * (double)p.n_global;
    const double ratio = base / amplitude;
    const double arg = (double)(t_sec % p.period) - (1 - ratio) * p.period;
    v = amplitude * (arg < 0 ? 0.0 : 1.0);
  } else if (p.signal_mode == DRSIM_SIG_PERLIN) {
    v = base + (base * p.amp[0] * aux);
    v = v > 0 ? v : 0.0;
  }
  v = v * artificial_ratio;
  return v < max_power ? v : max_power;
}

// signal_calculator.py:33-129 + power_grid.py:97-100
DRSIM_HD double grid_signal(const SimParams &p, double base, const Civil &t, double perlin,
                            double artificial_ratio, double max_power) {
  const double two_pi = 2 * 3.141592653589793;
  const int t_sec = t.hour * 3600 + t.minute * 60 + t.second;
  double v = base;
  if (p.signal_mode == DRSIM_SIG_SINUSOIDALS) {
    for (int k = 0; k < p.n_terms; ++k) v += (base * p.amp[k]) * sin(two_pi * t_sec / p.periods[k]);
  } else if (p.signal_mode == DRSIM_SIG_REGULAR_STEPS) {
    const double amplitude = p.amp_per_hvac * (double)p.n_global;
    const double ratio = base / amplitude;
    const double arg = (double)(t_sec % p.period) - (1 - ratio) * p.period;
    v = amplitude * (arg < 0 ? 0.0 : 1.0);  // np.heaviside(arg, 1)
  } else if (p.signal_mode == DRSIM_SIG_PERLIN) {
    v = base + (base * p.amp[0] * perlin);
    v = v > 0 ? v : 0.0;
  }
  v = v * artificial_ratio;
  return v < max_power ? v : max_power;
}

// ------------------------------------------------------------------------------------------
// hvac.py:43-64 -- lock-out state machine (integer, bit-exact)
// flags: bit0 turned_on, bit1 lockout
// ------------------------------------------------------------------------------------------
DRSIM_HD void hvac_fsm(uint32_t &flags, int &sso, bool action, int dt, int dur) {
  bool on = flags & 1u;
  if (!on) sso += dt;
  bool lock = !(on || sso >= dur);
  if (lock) {
    on = false;
  } else {
    on = action;
    if (on) sso = 0;
    else if (sso + dt < dur) lock = true;
  }
  flags = (on ? 1u : 0u) | (lock ? 2u : 0u);
}

// controllers/bangbang_controllers.py:18-89 (pre-step observation -> action)
template <typename real>
DRSIM_HD bool policy_action(int policy, real t_air, real target, real deadband, bool on, bool ext) {
  switch (policy) {
    case DRSIM_POLICY_DEADBAND_BANGBANG:
      if (t_air < target - deadband / 2) return false;
      if (t_air > target + deadband / 2) return true;
      return on;
    case DRSIM_POLICY_BANGBANG: return t_air > target;
    case DRSIM_POLICY_ALWAYS_ON: return true;
    default: return ext;
  }
}

// ------------------------------------------------------------------------------------------
// building.py:141-222 -- second-order ETP thermal update
// ------------------------------------------------------------------------------------------
// fp32 production path: the update is exactly affine with unit row sums, so it is applied in
// difference form with six per-house coefficients precomputed in fp64 (thermal_coefs below):
//   Ta' = Ta + [c0 (Tm - Ta) + c1 (Tod - Ta) + c2 Qa] ;  Tm' = Tm + [c3 (Ta - Tm) + c4 (Tod - Tm) + c5 Qa]
// Unit row sums make the map shift-invariant, so the fp32 planes carry the deviations
// xa = Ta - target, xm = Tm - target (|x| ~ 1 => ulp ~ 1e-7 instead of 2e-6 at 20 degC) and
// `od` is Tod - target.  The small increment is formed first and added once (one rounding).
DRSIM_HD void thermal_step_f32(float &xa, float &xm, const float c[6], float od, float Qa) {
  const float ia = fmaf(c[2], Qa, fmaf(c[1], od - xa, c[0] * (xm - xa)));
  const float im = fmaf(c[5], Qa, fmaf(c[4], od - xm, c[3] * (xa - xm)));
  xa += ia;
  xm += im;
}

#if defined(__CUDA_ARCH__)
#define DR_MUL(a, b) __dmul_rn((a), (b))
#define DR_ADD(a, b) __dadd_rn((a), (b))
#define DR_SUB(a, b) __dsub_rn((a), (b))
#define DR_DIV(a, b) __ddiv_rn((a), (b))
#else
#define DR_MUL(a, b) ((a) * (b))
#define DR_ADD(a, b) ((a) + (b))
#define DR_SUB(a, b) ((a) - (b))
#define DR_DIV(a, b) ((a) / (b))
#endif

// fp64 parity path: the reference's literal operation order with the per-house constants
// k = {Ua, Ca, Hm, r1, r2, A3, A4, e1, e2}; no FMA contraction (explicit _rn intrinsics).
DRSIM_HD void thermal_step_f64(double &ta, double &tm, const double k[9], double od, double Qa) {
  const double Ua = k[0], Ca = k[1], Hm = k[2], r1 = k[3], r2 = k[4], A3 = k[5], A4 = k[6],
               e1 = k[7], e2 = k[8];
  const double od_K = DR_ADD(od, 273.0), ta_K = DR_ADD(ta, 273.0), tm_K = DR_ADD(tm, 273.0);
  const double d = DR_ADD(Qa, DR_MUL(Ua, od_K));  // Qm + Qa + Ua*od_K with Qm = 0
  const double UaHm = DR_ADD(Ua, Hm);
  double dT = DR_SUB(DR_DIV(DR_MUL(Hm, tm_K), Ca), DR_DIV(DR_MUL(UaHm, ta_K), Ca));
  dT = DR_ADD(dT, DR_DIV(DR_MUL(Ua, od_K), Ca));
  dT = DR_ADD(dT, DR_DIV(Qa, Ca));
  const double doc = DR_DIV(d, Ua);
  const double num = DR_SUB(DR_SUB(DR_MUL(r2, ta_K), dT), DR_DIV(DR_MUL(r2, d), Ua));
  const double A1 = DR_DIV(num, DR_SUB(r2, r1));
  const double A2 = DR_SUB(DR_SUB(ta_K, doc), A1);
  const double na = DR_ADD(DR_ADD(DR_MUL(A1, e1), DR_MUL(A2, e2)), doc);
  const double nm = DR_ADD(DR_ADD(DR_ADD(DR_MUL(DR_MUL(A1, A3), e1), DR_MUL(DR_MUL(A2, A4), e2)), 0.0), doc);
  ta = DR_SUB(na, 273.0);
  tm = DR_SUB(nm, 273.0);
}

// derivation of both coefficient sets (fp64); host (set_state) and device (k_reset)
DRSIM_HD void thermal_coefs(double Ua, double Ca, double Cm, double Hm, int dt, double out12[12]) {
  const double a = Cm * Ca / Hm;
  const double b = Cm * (Ua + Hm) / Hm + Ca;
  const double c = Ua;
  const double root = sqrt(b * b - 4 * a * c);
  const double r1 = (-b + root) / (2 * a);
  const double r2 = (-b - root) / (2 * a);
  const double A3 = r1 * Ca / Hm + (Ua + Hm) / Hm;
  const double A4 = r2 * Ca / Hm + (Ua + Hm) / Hm;
  const double e1 = exp(r1 * dt), e2 = exp(r2 * dt);
  // linear map (Ta, Tm, Tod, Qa) -> (Ta', Tm') evaluated on the four basis vectors (temperatures in
  // kelvin enter linearly, so no offsets are needed)
  const double basis[4][4] = {{0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}, {1, 0, 0, 0}};
  double na[4], nm[4];
  for (int i = 0; i < 4; ++i) {
    const double ta = basis[i][0], tm = basis[i][1], od = basis[i][2], Qa = basis[i][3];
    const double d = Qa + Ua * od;
    const double dT = Hm * tm / Ca - (Ua + Hm) * ta / Ca + Ua * od / Ca + Qa / Ca;
    const double A1 = (r2 * ta - dT - r2 * d / c) / (r2 - r1);
    const double A2 = ta - d / c - A1;
    na[i] = A1 * e1 + A2 * e2 + d / c;
    nm[i] = A1 * A3 * e1 + A2 * A4 * e2 + d / c;
  }
  out12[0] = na[0];  // d Ta'/d Tm
  out12[1] = na[1];  // d Ta'/d Tod
  out12[2] = na[2];  // d Ta'/d Qa
  out12[3] = nm[3];  // d Tm'/d Ta
  out12[4] = nm[1];  // d Tm'/d Tod
  out12[5] = nm[2];  // d Tm'/d Qa
  out12[6] = r1; out12[7] = r2; out12[8] = A3; out12[9] = A4; out12[10] = e1; out12[11] = e2;
}

}  // namespace drsim
