// drsim_kernels.cuh -- sm_100a kernels of the demand-response environment step.
//
// Two execution paths over the same device functions (drsim_device.cuh):
//
//  * k_fused   one persistent kernel per step.  A CTA owns a *tile* of E whole clusters that
//              are contiguous in every SoA plane; house state is read with 128-bit loads, kept in
//              registers across the per-cluster power reduction (segmented warp shuffles + one
//              shared-memory pass), the env-level epilogue (time, outdoor temperature, signal) runs
//              on E threads, then rewards are written from registers and the observation rows are
//              assembled in shared memory and leave through TMA bulk stores
//              (cp.async.bulk.global.shared::cta).  Algorithmic bytes = every plane touched once.
//  * k_house / k_reduce / k_env / k_obs   general path for clusters larger than a tile, for the
//              steps on which the interpolated base power is re-evaluated, and for a single
//              cluster split across GPUs (the all-gather of the per-rank partial sums sits between
//              k_reduce and k_env).
//
// Reference citations are relative to /root/reference/server/app.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "drsim_device.cuh"

namespace drsim {

constexpr int kThreads = 256;       // CTA size of the house kernels
constexpr int kHousesPerThread = 4; // one 128-bit access per fp32 plane
constexpr int kTileSlots = kThreads * kHousesPerThread;
constexpr int kRed = 5;             // reduced per cluster: P, sum pen/N, max pen, sum dT, sum dT^2
constexpr int kObsChunk = 128;      // houses per k_obs CTA (general path)
constexpr int kHaloFields = 8;      // halo record of one edge house: dT/5, sso/dur, P/nrs, Pmax/nrs, 4 thermal ratios

template <typename real>
struct Planes {
  // per-house state [R][Ns]
  real *t_air, *t_mass;
  int32_t *sso;
  uint8_t *flags;
  // per-house static [R][Ns]
  const real *target, *cap;
  const real *coef[9];       // fp32: c0..c5 ; fp64: Ua, Ca, Hm, r1, r2, A3, A4, e1, e2
  const real *ratio[4];      // Ua, Ca, Cm, Hm over the defaults (only if an obs flag needs them)
  const uint8_t *interp_sub; // nearest-neighbour cell of the interpolation table
  const int32_t *dur;        // per-HVAC lock-out duration [R][Ns], or NULL: SimParams::lockout_duration for all
  // per-house outputs
  real *reward;
  void *obs;                 // [R][Ns][D] rows of element type `real`, or __nv_bfloat16 (drsim_config.obs_dtype)
  uint8_t *actions;
  // per-env [R]
  int64_t *epoch;
  double *od_temp, *solar_next, *solar_cur, *signal, *base_power, *power, *artificial_ratio, *max_power;
  double *pen_sum, *pen_max, *rew_sig;
  int32_t *t_since_interp;
  double *metrics;   // [R][DRSIM_N_METRICS]
  double *partials;  // [R][chunks][kRed]  (general path)
  double *acc;       // [R][kRed + 1]      (general path: reduced values + interpolated sum)
  const int32_t *comm_table;
  const real *interp_table;  // [162][9][5][8][12][6]
  double *halo_out;          // [R][nb_comm][kHaloFields]: message records of this shard's edge houses, or NULL

  template <typename O>
  DRSIM_HD O *rows() const { return static_cast<O *>(obs); }
};

// Observation-row element type O: `real`, or __nv_bfloat16 on an fp32 handle built with DRSIM_OBS_BF16.  A row value is
// computed in `real` as always and rounded to nearest-even where it is stored (the implicit float -> __nv_bfloat16
// conversion is __float2bfloat16_rn).  put2 stores columns 2 k, 2 k + 1 of a row with one 8- / 4-byte store.
DRSIM_D void put2(float *row, int k, float a, float b) { reinterpret_cast<float2 *>(row)[k] = make_float2(a, b); }
DRSIM_D void put2(__nv_bfloat16 *row, int k, float a, float b) {
  reinterpret_cast<__nv_bfloat162 *>(row)[k] = __floats2bfloat162_rn(a, b);
}

// One packed record per (scheduled step, replica): every env-level value of that step that does NOT
// depend on the step's cluster power, pre-computed by k_schedule_pack with the very expressions of
// env_pre_compute / env_fast_store.  The fused fp32 kernels fetch it with a few 16-byte cp.async
// copies one tile ahead, so the per-tile env thread has no global round trip and no fp64 chain on
// the path every other warp waits for at the tile barrier.
struct alignas(16) SchedRec {
  double signal, signal_prev;    // this step's signal; the one before it (reward pairs new power with old signal, Q6)
  double od, solar_next;         // -> pl.od_temp, pl.solar_next after the step
  double solar_cur, base_power;  // gain used by this step's house update; base power
  long long epoch;               // epoch after the step
  float od_prev_f, solar_f;      // house-update inputs: previous outdoor temperature, this step's gain (fp32)
  float signal_n, solar_n, od_n; // normalised observation columns (norm.py:113-114,132-135,164-165)
  int tsi;                       // t_since_interp after the step
};
static_assert(sizeof(SchedRec) == 80, "SchedRec is copied in five 16-byte pieces");

struct StepIn {
  const SchedRec *sched_rec;  // this step's records [R], or NULL (inline evaluation)
  double *host_env;           // drsim_step_host: mapped pinned [R][4] (power, signal, od_temp, mean reward) written by the kernel, or NULL
  // house-sharded ring cluster: message records of the L houses before / the H houses after this
  // shard, element (r, j) at base + (r * nb_comm + j) * kHaloFields (see k_reduce / k_obs)
  const double *halo_left, *halo_right;
  const uint8_t *actions;
  // drsim_step_host, copy-engine mode: `actions` is a device staging plane that ONE linear DMA is filling
  // while the kernel runs.  Consumed words are re-poisoned with 0xFFFFFFFF, so a word still holding the
  // poison has not arrived yet and is polled (bounded; *act_poll_err is set on a time-out).  NULL otherwise.
  int *act_poll_err;
  const double *od_noise;
  const double *perlin;
  const int32_t *interp_ids;
  // pre-generated env-level time series for this step (k_schedule), or NULL: inline evaluation
  const double *sched_od, *sched_solar, *sched_aux;
  const int32_t *sched_tsec;
  int64_t step;
  // house-sharded exchange: sequence number of this step's exchange on the handle -- starts at 1, grows by
  // one per sharded step and is NEVER reset (drsim_reset / drsim_set_state keep it), so a flag left by an
  // earlier episode can never equal the value a later step waits for; its low bit selects the inbox parity
  int64_t xseq;
  int do_interp;
  int advance;  // 1 = real step, 0 = refresh (recompute signal / obs without advancing time)
  // in-kernel step loop (drsim_run_tape: an action tape or an on-device policy on k_fused_tma, k_fused_rows, k_small):
  // this launch advances stream_steps consecutive steps.  Every byte a CTA reads of step k + 1 was written by the
  // same thread of the same CTA in step k (state planes, running metrics) or is an input of the call (tape, schedule
  // records), so no step boundary exists between CTAs: no launch ramp and tail, no grid-wide dependency.  k_fused_tma
  // runs each of its tiles through all the steps before the next tile (tile-major), k_fused_rows takes (step 0: its
  // tiles), (step 1: its tiles) ...  Step k reads the records sched_rec + k * R and the action plane
  // `actions + ((tape_first + k) % tape_planes) * tape_stride` (tape_planes 0: no rotation).  0 / 1 = one step.
  int stream_steps, tape_planes, tape_first;
  size_t tape_stride;
};

// Peer-memory exchange of the per-rank partial sums of ONE house-sharded cluster (SURVEY 8e): every
// rank owns an "inbox" [2 parities][world][R][kRed + 1] in its own slab plus step-stamped flags; the
// tail of k_reduce stores this rank's row straight into every peer's inbox over NVLink (st + release
// fence + flag store, system scope) and k_env spins on its own flags (acquire, bounded) before
// combining the rows in rank order -- compute, reduction and collective in the same two kernels, no
// NCCL call on the step path.
struct PeerCtx {
  int world, rank;
  double *const *inbox;               // [world] base of each rank's inbox (peer-mapped)
  unsigned long long *const *flags;   // [world] base of each rank's flags [2][world][R]
  double *const *halo;                // [world] base of each rank's halo inbox [2][R][nb_comm][kHaloFields]
  unsigned long long *const *pinbox;  // [world] base of each rank's EARLY cluster-power inbox [2][world][R][4] (PowerLL words)
  // [world] base of each rank's row inbox as self-validating words [2][world][R][16], or NULL: rows travel as plain
  // doubles + release flag (needed when halo records travel with them: those announce house state)
  unsigned long long *const *rowll;
  int *err;                           // local: set when a wait timed out
};

// a rank's reduced row (kRed + 1 doubles) as one 128-byte line of self-validating words, system scope
DRSIM_D void rowll_store(unsigned long long *dst, uint32_t tag32, const double *v) {
#if defined(__CUDA_ARCH__)
  const unsigned long long tag = (unsigned long long)tag32 << 32;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const unsigned long long bits = k <= kRed ? (unsigned long long)__double_as_longlong(v[k]) : 0ull;
    asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(dst + 2 * k), "l"(tag | (bits & 0xffffffffull)),
                 "l"(tag | (bits >> 32))
                 : "memory");
  }
#endif
}
// one poll of a row: true (and v filled) when all its words carry this step's tag
DRSIM_D bool rowll_try(const unsigned long long *src, uint32_t tag32, double v[kRed + 1]) {
  bool ok = true;
#if defined(__CUDA_ARCH__)
  unsigned long long w[2 * (kRed + 1)];
#pragma unroll
  for (int k = 0; k <= kRed; ++k)
    asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w[2 * k]), "=l"(w[2 * k + 1]) : "l"(src + 2 * k) : "memory");
#pragma unroll
  for (int k = 0; k < 2 * (kRed + 1); ++k) ok = ok && (uint32_t)(w[k] >> 32) == tag32;
#pragma unroll
  for (int k = 0; k <= kRed; ++k) v[k] = __longlong_as_double((long long)((w[2 * k + 1] << 32) | (w[2 * k] & 0xffffffffull)));
#endif
  return ok;
}

// One double as a self-validating 32-byte record: words 0 / 1 = (tag << 32 | low / high half), words 2 / 3 = tag
// only (the whole sector is written, so no reader makes the L2 complete a partial sector from HBM).
DRSIM_D void powll_store(unsigned long long *rec, uint32_t tag32, double v, bool sys) {
#if defined(__CUDA_ARCH__)
  const unsigned long long tag = (unsigned long long)tag32 << 32;
  const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
  if (sys) {
    asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(rec), "l"(tag | (bits & 0xffffffffull)), "l"(tag | (bits >> 32)) : "memory");
    asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(rec + 2), "l"(tag), "l"(tag) : "memory");
  } else {
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(rec), "l"(tag | (bits & 0xffffffffull)), "l"(tag | (bits >> 32)) : "memory");
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(rec + 2), "l"(tag), "l"(tag) : "memory");
  }
#endif
}
DRSIM_D void powll_issue(const unsigned long long *rec, unsigned long long w[2]) {
#if defined(__CUDA_ARCH__)
  asm volatile("ld.relaxed.sys.global.v2.u64 {%0, %1}, [%2];" : "=l"(w[0]), "=l"(w[1]) : "l"(rec) : "memory");
#endif
}
DRSIM_D bool powll_check(const unsigned long long w[2], uint32_t tag32, double &v) {
#if defined(__CUDA_ARCH__)
  v = __longlong_as_double((long long)((w[1] << 32) | (w[0] & 0xffffffffull)));
#endif
  return (uint32_t)(w[0] >> 32) == tag32 && (uint32_t)(w[1] >> 32) == tag32;
}

// a house-sharded cluster whose observation rows carry ring-neighbour messages exchanges the message
// records of the shard's edge houses every step (SURVEY 8e: "halo")
DRSIM_HD bool needs_halo(const SimParams &p) {
  return p.N != (int)p.n_global && p.obs_layout == DRSIM_OBS_HAND_ENGINEERED && p.nb_comm > 0;
}

// Launch-invariant constants in registers.  The fp32 build multiplies by reciprocals (<= 1 ulp
// from the true quotient, far inside the 1e-5 budget); the fp64 build divides like the reference.
template <typename real>
struct KC {
  real cop, nrs, db, one_plus_latent, norm_temp, n_glob;
  real inv_cop, inv_nrs, inv_norm_temp, inv_n, neg_inv_opl;
  DRSIM_D explicit KC(const SimParams &p) {
    cop = (real)p.cop; nrs = (real)p.nrs; db = (real)p.deadband; one_plus_latent = (real)(1.0 + p.latent);
    norm_temp = (real)p.norm_temp; n_glob = (real)p.n_global;
    inv_cop = (real)p.inv_cop; inv_nrs = (real)p.inv_nrs; inv_norm_temp = (real)p.inv_norm_temp;
    inv_n = (real)p.inv_n_global;
    neg_inv_opl = (real)p.hf.neg_inv_opl;
  }
};
DRSIM_D float qdiv(float x, float, float inv) { return x * inv; }
DRSIM_D double qdiv(double x, double d, double) { return x / d; }
DRSIM_D float div5(float x) { return x * 0.2f; }
DRSIM_D double div5(double x) { return x / 5.0; }

// ------------------------------------------------------------------------------------------
// vector access helpers: 4 consecutive houses per thread
// ------------------------------------------------------------------------------------------
DRSIM_D void load4(const float *p, float v[4]) {
  const float4 t = *reinterpret_cast<const float4 *>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
DRSIM_D void load4(const double *p, double v[4]) {
  const double2 a = reinterpret_cast<const double2 *>(p)[0];
  const double2 b = reinterpret_cast<const double2 *>(p)[1];
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
DRSIM_D void load4_ro(const float *p, float v[4]) {
  const float4 t = __ldg(reinterpret_cast<const float4 *>(p));
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
DRSIM_D void load4_ro(const double *p, double v[4]) {
  const double2 a = __ldg(reinterpret_cast<const double2 *>(p));
  const double2 b = __ldg(reinterpret_cast<const double2 *>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
DRSIM_D void store4(float *p, const float v[4]) {
  *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
}
DRSIM_D void store4(double *p, const double v[4]) {
  reinterpret_cast<double2 *>(p)[0] = make_double2(v[0], v[1]);
  reinterpret_cast<double2 *>(p)[1] = make_double2(v[2], v[3]);
}
DRSIM_D void load4i(const int32_t *p, int v[4]) {
  const int4 t = *reinterpret_cast<const int4 *>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
DRSIM_D void store4i(int32_t *p, const int v[4]) {
  *reinterpret_cast<int4 *>(p) = make_int4(v[0], v[1], v[2], v[3]);
}
DRSIM_D uint32_t load4b(const uint8_t *p) { return *reinterpret_cast<const uint32_t *>(p); }
DRSIM_D void store4b(uint8_t *p, uint32_t v) { *reinterpret_cast<uint32_t *>(p) = v; }

// Programmatic dependent launch (PDL): the fused step kernels are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so step t+1's CTAs become resident while step
// t's last CTAs drain.  pdl_trigger lets the next kernel in the stream start launching; pdl_wait
// blocks until every kernel before this one in the stream has completed and flushed its writes --
// nothing written by an earlier kernel (state planes, actions, schedule records) is touched before
// it, only the launch-invariant static planes.  Both are no-ops in a normal launch.
DRSIM_D void pdl_trigger() {
#if defined(__CUDA_ARCH__)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
}
DRSIM_D void pdl_wait() {
#if defined(__CUDA_ARCH__)
  asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}

// L2 eviction-priority policies (PTX createpolicy): the per-step working set is state + static planes
// (~45 B/house, re-read every step) plus the streamed outputs (observation rows, rewards).  Marking the
// former evict_last and the latter evict_first lets the 126 MB L2 keep the planes that the next step
// reads again instead of the rows nobody on the device reads back.
DRSIM_D uint64_t l2_policy_evict_first() {
  uint64_t pol = 0;
#if defined(__CUDA_ARCH__)
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
#endif
  return pol;
}
DRSIM_D uint64_t l2_policy_evict_last() {
  uint64_t pol = 0;
#if defined(__CUDA_ARCH__)
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
#endif
  return pol;
}
DRSIM_D void bulk_store_s2g_hint(void *gdst, const void *ssrc, uint32_t bytes, uint64_t pol) {
#if defined(__CUDA_ARCH__)
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(gdst), "r"(s),
               "r"(bytes), "l"(pol)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
#endif
}
DRSIM_D void st4_hint(float *p, const float v[4], uint64_t pol) {
#if defined(__CUDA_ARCH__)
  asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]),
               "f"(v[3]), "l"(pol)
               : "memory");
#endif
}
DRSIM_D void st4i_hint(int32_t *p, const int v[4], uint64_t pol) {
#if defined(__CUDA_ARCH__)
  asm volatile("st.global.L2::cache_hint.v4.s32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]),
               "r"(v[3]), "l"(pol)
               : "memory");
#endif
}
DRSIM_D void st1u_hint(uint8_t *p, uint32_t v, uint64_t pol) {
#if defined(__CUDA_ARCH__)
  asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
#endif
}
template <typename real> struct NCoef;
template <> struct NCoef<float> { static constexpr int n = 6; };
template <> struct NCoef<double> { static constexpr int n = 9; };

DRSIM_D void thermal_step(float &ta, float &tm, const float *c, float od, float Qa) {
  thermal_step_f32(ta, tm, c, od, Qa);
}
DRSIM_D void thermal_step(double &ta, double &tm, const double *c, double od, double Qa) {
  thermal_step_f64(ta, tm, c, od, Qa);
}
// fp32: every kernel multiplies by the same host-rounded -1/(1+latent), so all paths are bit-identical
DRSIM_D float hvac_heat(float cap, float, float neg_inv_opl) { return cap * neg_inv_opl; }
DRSIM_D double hvac_heat(double cap, double one_plus_latent, double) { return DR_DIV(DR_MUL(-1.0, cap), one_plus_latent); }

// Temperature representation of the t_air / t_mass planes (see drsim_ptrs.temp_is_deviation):
// fp32 stores the deviation from the set-point, fp64 the absolute temperature (literal replay).
template <typename real> struct Rep;
template <> struct Rep<float> {
  static DRSIM_D float dev(float x, float) { return x; }                                // Ta - target
  static DRSIM_D float minus20(float x, float target) { return x + (target - 20.f); }   // Ta - 20
  static DRSIM_D float od_in(float od, float target) { return od - target; }
  static DRSIM_D float pen(float target, float db, float x) { return deadband_l2<float>(0.f, db, x); }
  static DRSIM_D bool act(int policy, float x, float, float db, bool on, bool ext) {
    return policy_action<float>(policy, x, 0.f, db, on, ext);
  }
};
template <> struct Rep<double> {
  static DRSIM_D double dev(double t, double target) { return t - target; }
  static DRSIM_D double minus20(double t, double) { return t - 20.0; }
  static DRSIM_D double od_in(double od, double) { return od; }
  static DRSIM_D double pen(double target, double db, double t) { return deadband_l2<double>(target, db, t); }
  static DRSIM_D bool act(int policy, double t, double target, double db, bool on, bool ext) {
    return policy_action<double>(policy, t, target, db, on, ext);
  }
};

// ------------------------------------------------------------------------------------------
// the per-thread house work: 4 houses, loaded with vector accesses, updated in registers
// ------------------------------------------------------------------------------------------
template <typename real>
struct House4 {
  real ta[4], tm[4], target[4], cap[4];
  int sso[4];
  uint32_t flags;  // 4 x u8
  int valid;       // number of real houses among the 4 slots
};

// Loads state + static planes of 4 houses at plane offset `off`, applies the policy / action,
// hvac.py:43-64, building.py:141-222, writes the state back and returns the per-thread partial
// sums in red[kRed].
template <typename real, bool ALWAYS_ADVANCE = false>
DRSIM_D void house4_step(const Planes<real> &pl, const SimParams &p, const KC<real> &kc, const StepIn &in,
                         size_t off, int valid, real od_prev, real solar, House4<real> &h, real red[kRed]) {
  const bool advance = ALWAYS_ADVANCE || in.advance;
  constexpr int NC = NCoef<real>::n;
  real coef[NC][4];
  load4(pl.t_air + off, h.ta);
  load4(pl.t_mass + off, h.tm);
  load4i(pl.sso + off, h.sso);
  h.flags = load4b(pl.flags + off);
  load4_ro(pl.target + off, h.target);
  load4_ro(pl.cap + off, h.cap);
#pragma unroll
  for (int k = 0; k < NC; ++k) load4_ro(pl.coef[k] + off, coef[k]);
  uint32_t act = 0;
  if (p.policy == DRSIM_POLICY_EXTERNAL || p.policy == DRSIM_POLICY_GREEDY_MYOPIC)
    act = load4b((in.actions ? in.actions : pl.actions) + off);
  h.valid = valid;
  const real db = kc.db;
  real P = 0, ps = 0, pm = 0, ds = 0, d2 = 0;
  uint32_t nf = h.flags;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (j < valid) {
      uint32_t f = (h.flags >> (8 * j)) & 0xffu;
      const bool ext = (act >> (8 * j)) & 0xffu;
      const bool a = Rep<real>::act(p.policy, h.ta[j], h.target[j], db, f & 1u, ext);
      if (advance) {
        hvac_fsm(f, h.sso[j], a, p.dt, pl.dur ? __ldg(pl.dur + off + j) : p.lockout_duration);
        const real q = (f & 1u) ? hvac_heat(h.cap[j], kc.one_plus_latent, kc.neg_inv_opl) : (real)0;
        real c[NC];
#pragma unroll
        for (int k = 0; k < NC; ++k) c[k] = coef[k][j];
        thermal_step(h.ta[j], h.tm[j], c, Rep<real>::od_in(od_prev, h.target[j]), q + solar);
      }
      nf = (nf & ~(0xffu << (8 * j))) | (f << (8 * j));
      if (f & 1u) P += qdiv(h.cap[j], kc.cop, kc.inv_cop);
      const real pen = Rep<real>::pen(h.target[j], db, h.ta[j]);
      ps += qdiv(pen, kc.n_glob, kc.inv_n);
      pm = pen > pm ? pen : pm;
      const real dT = Rep<real>::dev(h.ta[j], h.target[j]);
      ds += dT;
      d2 += dT * dT;
    }
  }
  h.flags = nf;
  if (advance) {
    store4(pl.t_air + off, h.ta);
    store4(pl.t_mass + off, h.tm);
    store4i(pl.sso + off, h.sso);
    store4b(pl.flags + off, h.flags);
  }
  red[0] = P; red[1] = ps; red[2] = pm; red[3] = ds; red[4] = d2;
}

// Lean fp32 specialisation of house4_step for the fused production kernel: branch-free lock-out
// FSM (hvac.py:43-64), deviation-form thermal update, constants straight from the constant bank.
// Padding slots (N % 4 != 0) carry zero state / zero coefficients and are masked out of the sums.
DRSIM_D void house4_step_f32(const Planes<float> &pl, const SimParams &p, const StepIn &in, size_t off, int valid,
                             float od_prev, float solar, House4<float> &h, float red[kRed]) {
  float c[6][4];
  load4(pl.t_air + off, h.ta);
  load4(pl.t_mass + off, h.tm);
  load4i(pl.sso + off, h.sso);
  h.flags = load4b(pl.flags + off);
  load4_ro(pl.target + off, h.target);
  load4_ro(pl.cap + off, h.cap);
#pragma unroll
  for (int k = 0; k < 6; ++k) load4_ro(pl.coef[k] + off, c[k]);
  uint32_t act = 0;
  const int policy = p.policy;
  if (policy == DRSIM_POLICY_EXTERNAL || policy == DRSIM_POLICY_GREEDY_MYOPIC)
    act = load4b((in.actions ? in.actions : pl.actions) + off);
  h.valid = valid;
  const int dt = p.dt, dur = p.lockout_duration;
  const float half_db = p.hf.half_db;
  float P = 0, ps = 0, pm = 0, ds = 0, d2 = 0;
  uint32_t nf = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint32_t f0 = (h.flags >> (8 * j)) & 0xffu;
    const bool on = f0 & 1u;
    bool a = (act >> (8 * j)) & 0xffu;
    if (policy == DRSIM_POLICY_DEADBAND_BANGBANG) a = h.ta[j] < -half_db ? false : (h.ta[j] > half_db ? true : on);
    else if (policy == DRSIM_POLICY_BANGBANG) a = h.ta[j] > 0.f;
    else if (policy == DRSIM_POLICY_ALWAYS_ON) a = true;
    int sso = h.sso[j] + (on ? 0 : dt);
    bool lock = !on && sso < dur;
    const bool on_n = !lock && a;
    sso = on_n ? 0 : sso;
    lock = lock || (!on_n && sso + dt < dur);
    h.sso[j] = sso;
    nf |= ((on_n ? 1u : 0u) | (lock ? 2u : 0u)) << (8 * j);
    const float Qa = (on_n ? h.cap[j] * p.hf.neg_inv_opl : 0.f) + solar;
    const float odr = od_prev - h.target[j];
    const float xa = h.ta[j], xm = h.tm[j];
    const float ia = fmaf(c[2][j], Qa, fmaf(c[1][j], odr - xa, c[0][j] * (xm - xa)));
    const float im = fmaf(c[5][j], Qa, fmaf(c[4][j], odr - xm, c[3][j] * (xa - xm)));
    h.ta[j] = xa + ia;
    h.tm[j] = xm + im;
    const float m = j < valid ? 1.f : 0.f;
    P = fmaf(on_n ? m : 0.f, h.cap[j] * p.hf.inv_cop, P);
    const float d = fmaxf(fabsf(h.ta[j]) - half_db, 0.f);
    const float pen = d * d * m;
    ps = fmaf(pen, p.hf.inv_n, ps);
    pm = fmaxf(pm, pen);
    ds = fmaf(m, h.ta[j], ds);
    d2 = fmaf(h.ta[j] * m, h.ta[j], d2);
  }
  h.flags = nf;
  store4(pl.t_air + off, h.ta);
  store4(pl.t_mass + off, h.tm);
  store4i(pl.sso + off, h.sso);
  store4b(pl.flags + off, h.flags);
  red[0] = P; red[1] = ps; red[2] = pm; red[3] = ds; red[4] = d2;
}

template <bool ALWAYS_ADVANCE>
DRSIM_D void house4_dispatch(const Planes<float> &pl, const SimParams &p, const KC<float> &, const StepIn &in,
                             size_t off, int valid, float od_prev, float solar, House4<float> &h, float red[kRed]) {
  static_assert(ALWAYS_ADVANCE, "lean path is only used by the fused kernel");
  house4_step_f32(pl, p, in, off, valid, od_prev, solar, h, red);
}
template <bool ALWAYS_ADVANCE>
DRSIM_D void house4_dispatch(const Planes<double> &pl, const SimParams &p, const KC<double> &kc, const StepIn &in,
                             size_t off, int valid, double od_prev, double solar, House4<double> &h, double red[kRed]) {
  house4_step<double, ALWAYS_ADVANCE>(pl, p, kc, in, off, valid, od_prev, solar, h, red);
}


// Inputs of 4 houses as the fused fp32 kernel receives them (from shared memory / registers)
struct Raw4f {
  float ta[4], tm[4], target[4], cap[4], c[6][4];
  int sso[4];
  uint32_t flags, act;
  float od, solar;
};

// COMPUTE half of the lean fp32 house step (see house4_step_f32): consumes a Raw4f.
template <bool EXT_ONLY>
DRSIM_D void house4_compute_f32(const Planes<float> &pl, const SimParams &p, const Raw4f &w, size_t off, int valid,
                                House4<float> &h, float red[kRed], uint64_t keep_policy = 0) {
  const int policy = EXT_ONLY ? (int)DRSIM_POLICY_EXTERNAL : p.policy;
  h.valid = valid;
  const int dt = p.dt, dur = p.lockout_duration;
  const float half_db = p.hf.half_db;
  float P = 0, ps = 0, pm = 0, ds = 0, d2 = 0;
  uint32_t nf = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint32_t f0 = (w.flags >> (8 * j)) & 0xffu;
    const bool on = f0 & 1u;
    bool a = (w.act >> (8 * j)) & 0xffu;
    if (policy == DRSIM_POLICY_DEADBAND_BANGBANG) a = w.ta[j] < -half_db ? false : (w.ta[j] > half_db ? true : on);
    else if (policy == DRSIM_POLICY_BANGBANG) a = w.ta[j] > 0.f;
    else if (policy == DRSIM_POLICY_ALWAYS_ON) a = true;
    int sso = w.sso[j] + (on ? 0 : dt);
    bool lock = !on && sso < dur;
    const bool on_n = !lock && a;
    sso = on_n ? 0 : sso;
    lock = lock || (!on_n && sso + dt < dur);
    h.sso[j] = sso;
    nf |= ((on_n ? 1u : 0u) | (lock ? 2u : 0u)) << (8 * j);
    const float cap = w.cap[j], tg = w.target[j];
    h.cap[j] = cap;
    h.target[j] = tg;
    const float Qa = (on_n ? cap * p.hf.neg_inv_opl : 0.f) + w.solar;
    const float odr = w.od - tg;
    const float xa = w.ta[j], xm = w.tm[j];
    const float ia = fmaf(w.c[2][j], Qa, fmaf(w.c[1][j], odr - xa, w.c[0][j] * (xm - xa)));
    const float im = fmaf(w.c[5][j], Qa, fmaf(w.c[4][j], odr - xm, w.c[3][j] * (xa - xm)));
    h.ta[j] = xa + ia;
    h.tm[j] = xm + im;
    const float m = j < valid ? 1.f : 0.f;
    P = fmaf(on_n ? m : 0.f, cap * p.hf.inv_cop, P);
    const float d = fmaxf(fabsf(h.ta[j]) - half_db, 0.f);
    const float pen = d * d * m;
    ps = fmaf(pen, p.hf.inv_n, ps);
    pm = fmaxf(pm, pen);
    ds = fmaf(m, h.ta[j], ds);
    d2 = fmaf(h.ta[j] * m, h.ta[j], d2);
  }
  h.flags = nf;
  if (keep_policy) {  // state planes are re-read by the next step: keep them in L2
    st4_hint(pl.t_air + off, h.ta, keep_policy);
    st4_hint(pl.t_mass + off, h.tm, keep_policy);
    st4i_hint(pl.sso + off, h.sso, keep_policy);
    st1u_hint(pl.flags + off, h.flags, keep_policy);
  } else {
    store4(pl.t_air + off, h.ta);
    store4(pl.t_mass + off, h.tm);
    store4i(pl.sso + off, h.sso);
    store4b(pl.flags + off, h.flags);
  }
  red[0] = P; red[1] = ps; red[2] = pm; red[3] = ds; red[4] = d2;
}

template <typename T, typename U>
DRSIM_D void red_combine(T a[kRed], const U b[kRed]) {
  a[0] += (T)b[0]; a[1] += (T)b[1]; a[2] = a[2] > (T)b[2] ? a[2] : (T)b[2]; a[3] += (T)b[3]; a[4] += (T)b[4];
}

// ------------------------------------------------------------------------------------------
// env-level epilogue (one thread per cluster): environment.py:87-106
// ------------------------------------------------------------------------------------------
struct EnvRegs {
  int64_t epoch;
  double od_temp, solar_next, signal, base_power, artificial_ratio, max_power;
  int t_since_interp;
  // this step's pre-generated values (k_schedule), valid when StepIn::sched_od != NULL
  double s_od, s_solar, s_aux;
  int s_tsec;
  double m[DRSIM_N_METRICS];  // running metrics, prefetched for the fast path
};

template <typename real>
DRSIM_D EnvRegs env_load(const Planes<real> &pl, const StepIn &in, int r) {
  EnvRegs e;
  e.epoch = pl.epoch[r];
  e.od_temp = pl.od_temp[r];
  e.solar_next = pl.solar_next[r];
  e.signal = pl.signal[r];
  e.base_power = pl.base_power[r];
  e.artificial_ratio = pl.artificial_ratio[r];
  e.max_power = pl.max_power[r];
  e.t_since_interp = pl.t_since_interp[r];
  if (in.sched_od) {
    e.s_od = in.sched_od[r]; e.s_solar = in.sched_solar[r]; e.s_aux = in.sched_aux[r]; e.s_tsec = in.sched_tsec[r];
    const double *m = pl.metrics + (size_t)r * DRSIM_N_METRICS;
#pragma unroll
    for (int k = 0; k < DRSIM_N_METRICS; ++k) e.m[k] = m[k];
  }
  return e;
}

// values the house/obs phases need from the env epilogue
template <typename real>
struct EnvBroadcast {
  real power_n, signal_n, solar_n, od_n, rew_sig, pen_common, pen_max;
};

// mean over the cluster of the per-agent reward (rewards_calculator.py:174-179), from the reduced
// penalties: mean individual penalty == the common_L2 value
DRSIM_D double mean_reward(const SimParams &p, double pen_mean, double pen_max, double rew_sig) {
  double pen = pen_mean;
  if (p.penalty_mode == DRSIM_PEN_COMMON_MAX) pen = pen_max;
  else if (p.penalty_mode == DRSIM_PEN_MIXTURE)
    pen = (p.a_ind * pen_mean + p.a_cl2 * pen_mean + p.a_cmax * pen_max) / (p.a_ind + p.a_cl2 + p.a_cmax);
  return -(p.alpha_temp * pen / p.norm_temp + rew_sig);
}

// alpha_sig * ((P - S_old) / N)^2 / norm (rewards_calculator.py:198, :177), reciprocal form shared by
// every kernel path so that they agree bit for bit
DRSIM_D double signal_penalty(const SimParams &p, double P, double s_old) {
  const double dev = (P - s_old) * p.inv_n_global;
  return p.alpha_sig * (dev * dev) * p.inv_norm_sig;
}

// what env_epilogue leaves in the env planes: computed first (env_epilogue_compute), stored afterwards
// (env_epilogue_store), so that a caller with consumers waiting for the broadcast values (k_shard) can
// publish them before paying for the stores
struct EnvOut {
  EnvRegs e;
  double solar_cur, P, rew_sig, pen_sum, pen_max;
  double mean_rew, abs_dt, sq_dt, p_minus_s;   // terms of the running-metric updates (valid when advance)
};

template <typename real>
DRSIM_D EnvBroadcast<real> env_epilogue_compute(const Planes<real> &pl, const SimParams &p, const StepIn &in,
                                                int r, EnvRegs e, const double red[kRed], double interp_sum, EnvOut &o) {
  const uint32_t env_global = (uint32_t)(p.rep_offset + r);
  double solar_cur, rew_sig = 0.0, P;
  const bool sched = in.advance && in.sched_od != nullptr;
  if (in.advance) {
    e.epoch += p.dt;                                               // environment.py:87
    solar_cur = e.solar_next;                                      // gain used by this step's update
    P = red[0];
    rew_sig = signal_penalty(p, P, e.signal);                      // old signal (quirk Q6)
    // running rollout metrics (metrics_service.py:108-157 restated as per-cluster sums)
    o.mean_rew = mean_reward(p, red[1], red[2], rew_sig);
    o.abs_dt = fabs(red[3]);
    o.sq_dt = red[4];
    o.p_minus_s = P - e.signal;
  } else {
    solar_cur = pl.solar_cur[r];
    // a refresh keeps the injected cluster power: the reference's reset observation carries the
    // power cached BEFORE the property noise was applied (cluster.py:61-65 vs environment.py:58)
    P = pl.power[r];
  }
  const bool grid = in.advance || in.do_interp >= 0;
  if (grid) {                                                      // power_grid.py:130-161
    if (p.base_mode == DRSIM_BASE_CONSTANT) {
      e.base_power = p.avg_power * (double)p.n_global;
    } else if (in.do_interp > 0) {
      const double factor = p.n_global <= p.interp_k ? 1.0 : (double)p.n_global / (double)p.interp_k;
      e.base_power = interp_sum * factor;
      e.t_since_interp = 0;
    } else {
      // every power-grid step adds dt (power_grid.py:150), also a refresh that recomputes the signal without
      // firing: the plane stays equal to the host counter interp_decision advanced
      e.t_since_interp += p.dt;
    }
  }
  if (sched) {
    // fast path: every time-dependent scalar of this step was pre-generated by k_schedule
    e.solar_next = e.s_solar;
    e.od_temp = e.s_od;
    e.signal = grid_signal_sched(p, e.base_power, e.s_tsec, e.s_aux, e.artificial_ratio, e.max_power);
  } else {
    const Civil now = civil_from_epoch(e.epoch);
    if (in.advance) {
      e.solar_next = p.solar_on ? solar_gain(civil_from_epoch(e.epoch + p.dt), p.window_area, p.shading) : 0.0;
      double noise = 0.0;                                          // environment.py:158
      if (in.od_noise) noise = in.od_noise[r];
      else if (p.noise_mode == DRSIM_NOISE_PHILOX)
        noise = p.temp_std * philox_normal(p.seed, env_global, 0u, (uint32_t)in.step, PURPOSE_OD);
      e.od_temp = od_temp_model(now, p.day_temp, p.night_temp, p.phase, noise);
    }
    if (grid) {
      double perlin = 0.0;
      if (p.signal_mode == DRSIM_SIG_PERLIN) {
        if (in.perlin) perlin = in.perlin[r];
        else if (p.noise_mode == DRSIM_NOISE_PHILOX) {
          const double x = (double)(now.hour * 3600 + now.minute * 60 + now.second);
          perlin = philox_perlin(p.seed, env_global, x / (double)p.period, p.nb_octaves, p.octaves_step);
        }
      }
      e.signal = grid_signal(p, e.base_power, now, perlin, e.artificial_ratio, e.max_power);
    }
  }
  o.e = e; o.solar_cur = solar_cur; o.P = P; o.rew_sig = rew_sig; o.pen_sum = red[1]; o.pen_max = red[2];
  EnvBroadcast<real> b;
  b.power_n = (real)(P * p.inv_nrs);                               // norm.py:144-146
  b.signal_n = (real)(e.signal * p.inv_nrs * p.inv_n_global);      // norm.py:132-135
  b.solar_n = (real)(solar_cur * 1e-3);                            // norm.py:113-114
  b.od_n = (real)((e.od_temp - 20.0) * 0.2);                       // norm.py:164-165
  b.rew_sig = (real)rew_sig;
  b.pen_common = (real)red[1];
  b.pen_max = (real)red[2];
  return b;
}

template <typename real>
DRSIM_D void env_epilogue_store(const Planes<real> &pl, const SimParams &p, const StepIn &in, int r, const EnvOut &o) {
  if (in.advance) {
    // (multiply-adds as in env_stage_store: the contraction into FMAs is part of the result)
    double *m = pl.metrics + (size_t)r * DRSIM_N_METRICS;
    m[0] += 1.0;
    m[1] += o.mean_rew;
    m[2] += o.abs_dt * p.inv_n_global;
    m[3] += o.sq_dt * p.inv_n_global;
    m[4] += fabs(o.p_minus_s);
    m[5] += o.p_minus_s * o.p_minus_s;
  }
  pl.epoch[r] = o.e.epoch;
  pl.od_temp[r] = o.e.od_temp;
  pl.solar_next[r] = o.e.solar_next;
  pl.solar_cur[r] = o.solar_cur;
  pl.signal[r] = o.e.signal;
  pl.base_power[r] = o.e.base_power;
  if (in.advance) pl.power[r] = o.P;
  pl.pen_sum[r] = o.pen_sum;
  pl.pen_max[r] = o.pen_max;
  pl.rew_sig[r] = o.rew_sig;
  pl.t_since_interp[r] = o.e.t_since_interp;
}

template <typename real>
DRSIM_D EnvBroadcast<real> env_epilogue(const Planes<real> &pl, const SimParams &p, const StepIn &in,
                                        int r, EnvRegs e, const double red[kRed], double interp_sum) {
  EnvOut o;
  const EnvBroadcast<real> b = env_epilogue_compute<real>(pl, p, in, r, e, red, interp_sum, o);
  env_epilogue_store<real>(pl, p, in, r, o);
  return b;
}

// Fast epilogue of the fused kernel (schedule available, real step, no interpolator firing):
// env_fast_compute is the short critical section between the two CTA barriers (only what the house
// threads wait for); env_fast_store writes the env planes and metrics after the barrier is released.
struct EnvFast {
  double P, rew_sig, signal, solar_cur;
};

// The part of the fast epilogue that does not depend on this step's cluster power: available
// BEFORE the tile barrier.  The power-dependent scalars (power_n, rew_sig) are folded in afterwards
// by every house thread on its own (env_fold_power), so the tile has no serial section at all.
template <typename real>
DRSIM_D EnvBroadcast<real> env_pre_compute(const SimParams &p, EnvRegs &e, EnvFast &f) {
  f.solar_cur = e.solar_next;
  if (p.base_mode == DRSIM_BASE_CONSTANT) e.base_power = p.avg_power * (double)p.n_global;
  f.signal = grid_signal_sched(p, e.base_power, e.s_tsec, e.s_aux, e.artificial_ratio, e.max_power);
  EnvBroadcast<real> b;
  b.power_n = (real)0;
  b.signal_n = (real)(f.signal * p.inv_nrs * p.inv_n_global);
  b.solar_n = (real)(f.solar_cur * 1e-3);
  b.od_n = (real)((e.s_od - 20.0) * 0.2);
  b.rew_sig = (real)0;
  b.pen_common = (real)0;
  b.pen_max = (real)0;
  return b;
}

template <typename real>
DRSIM_D EnvBroadcast<real> env_fast_compute(const SimParams &p, EnvRegs &e, const double red[kRed], EnvFast &f) {
  f.P = red[0];
  f.rew_sig = signal_penalty(p, f.P, e.signal);
  f.solar_cur = e.solar_next;
  if (p.base_mode == DRSIM_BASE_CONSTANT) e.base_power = p.avg_power * (double)p.n_global;
  f.signal = grid_signal_sched(p, e.base_power, e.s_tsec, e.s_aux, e.artificial_ratio, e.max_power);
  EnvBroadcast<real> b;
  b.power_n = (real)(f.P * p.inv_nrs);
  b.signal_n = (real)(f.signal * p.inv_nrs * p.inv_n_global);
  b.solar_n = (real)(f.solar_cur * 1e-3);
  b.od_n = (real)((e.s_od - 20.0) * 0.2);
  b.rew_sig = (real)f.rew_sig;
  b.pen_common = (real)red[1];
  b.pen_max = (real)red[2];
  return b;
}

template <typename real>
DRSIM_D void env_fast_store(const Planes<real> &pl, const SimParams &p, int r, const EnvRegs &e, const EnvFast &f,
                            const double red[kRed]) {
  pl.epoch[r] = e.epoch + p.dt;
  pl.od_temp[r] = e.s_od;
  pl.solar_next[r] = e.s_solar;
  pl.solar_cur[r] = f.solar_cur;
  pl.signal[r] = f.signal;
  pl.base_power[r] = e.base_power;
  pl.power[r] = f.P;
  pl.pen_sum[r] = red[1];
  pl.pen_max[r] = red[2];
  pl.rew_sig[r] = f.rew_sig;
  if (p.base_mode != DRSIM_BASE_CONSTANT) pl.t_since_interp[r] = e.t_since_interp + p.dt;
  double *m = pl.metrics + (size_t)r * DRSIM_N_METRICS;
  const double d = f.P - e.signal;
  m[0] = e.m[0] + 1.0;
  m[1] = e.m[1] + mean_reward(p, red[1], red[2], f.rew_sig);
  m[2] = e.m[2] + fabs(red[3]) * p.inv_n_global;
  m[3] = e.m[3] + red[4] * p.inv_n_global;
  m[4] = e.m[4] + fabs(d);
  m[5] = e.m[5] + d * d;
}

// Pre-generation of the env-level time series: thread (k, r) evaluates, for step `step0 + k` of
// replica r, the outdoor temperature (environment.py:132-159 with the Philox gauss draw), the
// solar gain of the following step (utils.py:42-117), seconds since midnight and the
// time-dependent factor of the signal (signal_calculator.py:46-115).  Counter-based noise makes
// this exact: the values are the ones the inline epilogue would compute.
template <typename real>
__global__ void k_schedule(Planes<real> pl, SimParams p, int64_t step0, int K, double *od, double *solar,
                           double *aux, int32_t *tsec) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K * p.R) return;
  const int k = i / p.R, r = i - k * p.R;
  const uint32_t env_global = (uint32_t)(p.rep_offset + r);
  const int64_t epoch = pl.epoch[r] + (int64_t)(k + 1) * p.dt;
  const Civil now = civil_from_epoch(epoch);
  double noise = 0.0;
  if (p.noise_mode == DRSIM_NOISE_PHILOX)
    noise = p.temp_std * philox_normal(p.seed, env_global, 0u, (uint32_t)(step0 + k), PURPOSE_OD);
  od[i] = od_temp_model(now, p.day_temp, p.night_temp, p.phase, noise);
  solar[i] = p.solar_on ? solar_gain(civil_from_epoch(epoch + p.dt), p.window_area, p.shading) : 0.0;
  const int t_sec = now.hour * 3600 + now.minute * 60 + now.second;
  tsec[i] = t_sec;
  double a = 0.0;
  if (p.signal_mode == DRSIM_SIG_SINUSOIDALS) {
    for (int t = 0; t < p.n_terms; ++t) a += p.amp[t] * sin(2 * 3.141592653589793 * t_sec / p.periods[t]);
  } else if (p.signal_mode == DRSIM_SIG_PERLIN && p.noise_mode == DRSIM_NOISE_PHILOX) {
    a = philox_perlin(p.seed, env_global, (double)t_sec / (double)p.period, p.nb_octaves, p.octaves_step);
  }
  aux[i] = a;
}

// Second pass of the schedule: packs step k of replica r into its SchedRec from the time series of
// k_schedule and the env planes as they are at schedule time (k = 0 takes its "previous" values from
// the planes, k > 0 from step k - 1 of the series).
template <typename real>
__global__ void k_schedule_pack(Planes<real> pl, SimParams p, int K, const double *od, const double *solar,
                                const double *aux, const int32_t *tsec, SchedRec *rec) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K * p.R) return;
  const int k = i / p.R, r = i - k * p.R;
  const double base = p.base_mode == DRSIM_BASE_CONSTANT ? p.avg_power * (double)p.n_global : pl.base_power[r];
  const double ratio = pl.artificial_ratio[r], maxp = pl.max_power[r];
  SchedRec c;
  c.signal = grid_signal_sched(p, base, tsec[i], aux[i], ratio, maxp);
  c.signal_prev = k == 0 ? pl.signal[r] : grid_signal_sched(p, base, tsec[i - p.R], aux[i - p.R], ratio, maxp);
  c.od = od[i];
  c.solar_next = solar[i];
  c.solar_cur = k == 0 ? pl.solar_next[r] : solar[i - p.R];
  c.base_power = base;
  c.epoch = pl.epoch[r] + (long long)(k + 1) * p.dt;
  c.od_prev_f = (float)(k == 0 ? pl.od_temp[r] : od[i - p.R]);
  c.solar_f = (float)c.solar_cur;
  c.signal_n = (float)(c.signal * p.inv_nrs * p.inv_n_global);
  c.solar_n = (float)(c.solar_cur * 1e-3);
  c.od_n = (float)((c.od - 20.0) * 0.2);
  c.tsi = pl.t_since_interp[r] + (k + 1) * p.dt;
  rec[i] = c;
}

// rewards_calculator.py:174-179 for one house, fp32 individual_L2 fast form
DRSIM_D float reward_f32_individual(const SimParams &p, float xa, float rew_sig) {
  const float d = fmaxf(fabsf(xa) - p.hf.half_db, 0.f);
  return -fmaf(p.hf.rew_scale, d * d, rew_sig);
}

// rewards_calculator.py:135-181 for one house
template <typename real>
DRSIM_D real house_reward(const SimParams &p, const KC<real> &kc, real ta, real target, const EnvBroadcast<real> &e) {
  if constexpr (sizeof(real) == 4) {
    if (p.penalty_mode == DRSIM_PEN_INDIVIDUAL_L2) return reward_f32_individual(p, ta, e.rew_sig);
  }
  const real ind = Rep<real>::pen(target, kc.db, ta);
  real pen;
  switch (p.penalty_mode) {
    case DRSIM_PEN_COMMON_L2: pen = e.pen_common; break;
    case DRSIM_PEN_COMMON_MAX: pen = e.pen_max; break;
    case DRSIM_PEN_MIXTURE:
      pen = ((real)p.a_ind * ind + (real)p.a_cl2 * e.pen_common + (real)p.a_cmax * e.pen_max) /
            (real)(p.a_ind + p.a_cl2 + p.a_cmax);
      break;
    default: pen = ind;
  }
  return (real)-1 * (qdiv((real)p.alpha_temp * pen, kc.norm_temp, kc.inv_norm_temp) + e.rew_sig);
}

// neighbour k of house n: ring (agent_communication_builder.py:63-85) or explicit table
DRSIM_D int neighbour_of(const SimParams &p, const int32_t *table, int r, int n, int k) {
  if (p.comm_mode == DRSIM_COMM_RING) {
    const int N = (int)p.n_global, lo = p.nb_comm / 2;
    // nb_comm <= N - 1, so v lies in (-N, 2N): one conditional wrap is the exact `mod N`
    int v = k < lo ? n - lo + k : n + 1 + (k - lo);
    v = v < 0 ? v + N : v;
    return v >= N ? v - N : v;
  }
  const size_t base = p.comm_per_rep ? (size_t)r * p.N * p.nb_comm : 0;
  return __ldg(table + base + (size_t)n * p.nb_comm + k);
}

// Draw index of the rows a kernel writes (DRSIM_COMM_SAMPLE): the handle's step count as the rows see it -- in.step + 1
// after step 0 of the launch, + k + 1 after step k of an in-kernel block, in.step for a refresh (advance = 0)
DRSIM_D uint32_t rows_draw(const StepIn &in, int k = 0) { return (uint32_t)(in.step + (in.advance ? k + 1 : 0)); }

// Neighbours of one row.  SMP = false: neighbour_of, unchanged.  SMP = true (DRSIM_COMM_SAMPLE): the row's draw,
// computed once as the row's message loop asks for k = 0, 1, ... (a later k runs the draw up to it).
template <bool SMP>
struct RowNbrs {
  DRSIM_D RowNbrs(const SimParams &, int, int, uint32_t) {}
  DRSIM_D int operator()(const SimParams &p, const int32_t *table, int r, int n, int k) { return neighbour_of(p, table, r, n, k); }
};
template <>
struct RowNbrs<true> {
  CommSampler s;
  DRSIM_D RowNbrs(const SimParams &p, int r, int n, uint32_t draw)
      : s(p.seed, (uint32_t)(p.rep_offset + r), (uint32_t)(p.house_offset + n), draw, (uint32_t)p.n_global) {}
  DRSIM_D int operator()(const SimParams &, const int32_t *, int, int, int k) { return s.pick(k); }
};

// neighbour table of one draw, [R][N][nb_comm] (drsim_comm_sample)
__global__ void k_comm_sample(SimParams p, uint32_t draw, int32_t *out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)p.R * p.N) return;
  const int r = (int)(i / p.N), n = (int)(i - (int64_t)r * p.N);
  RowNbrs<true> nb(p, r, n, draw);
  for (int k = 0; k < p.nb_comm; ++k) out[i * p.nb_comm + k] = nb(p, nullptr, r, n, k);
}

// int(seconds_since_off / lockout_duration) of the house's OWN hvac (norm.py:79-82); messages use the default
// duration (norm.py:40-43) and keep fast_div
template <typename real>
DRSIM_D real own_sso_norm(const Planes<real> &pl, const SimParams &p, size_t o, int sso) {
  if (pl.dur) return (real)(sso / max(1, __ldg(pl.dur + o)));
  return (real)fast_div((uint32_t)sso, p.fd_dur);
}

// own-state part of the observation row (utils/norm.py:71-146).  `what` selects the columns
// written: bit0 = those that depend on the house only, bit1 = those that need the env epilogue
// (cluster power, signal, solar gain, outdoor temperature).
template <typename real, typename O>
DRSIM_D int obs_own(O *row, const SimParams &p, uint32_t f, real sso_n, real ta20, real tm20, real tg20,
                    const EnvBroadcast<real> &e, const real ratio[4], int what = 3) {
  int i = 0;
  const bool hs = what & 1, ev = what & 2;
  if (hs) { row[i] = (real)(f & 1u); row[i + 1] = (real)((f >> 1) & 1u); row[i + 2] = sso_n; row[i + 3] = (real)1; }
  i += 4;
  if (p.st_hvac) { if (hs) { row[i] = (real)1; row[i + 1] = (real)1; } i += 2; }
  if (ev) { row[i] = e.power_n; row[i + 1] = e.signal_n; }
  i += 2;
  if (hs) { row[i] = (real)p.deadband; row[i + 1] = div5(ta20); row[i + 2] = div5(tm20); row[i + 3] = div5(tg20); }
  i += 4;
  if (p.st_solar) { if (ev) row[i] = e.solar_n; i += 1; }
  if (p.st_thermal) {
    if (hs) { row[i] = ratio[0]; row[i + 1] = ratio[1]; row[i + 2] = ratio[2]; row[i + 3] = ratio[3]; }
    if (ev) row[i + 4] = e.od_n;
    i += 5;
  }
  return i;
}

// deterministic reduction of per-thread partials over a CTA: warp shuffles, then a fixed-order
// pass over the warp partials by thread 0
template <typename real, int WARPS>
DRSIM_D void block_reduce(real red[kRed], double out[kRed], double (*wp)[kRed]) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    real t[kRed];
#pragma unroll
    for (int k = 0; k < kRed; ++k) t[k] = __shfl_down_sync(0xffffffffu, red[k], o);
    red_combine(red, t);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0)
    for (int k = 0; k < kRed; ++k) wp[w][k] = (double)red[k];
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 0; k < kRed; ++k) out[k] = 0.0;
    for (int i = 0; i < WARPS; ++i) red_combine(out, wp[i]);
  }
}

// ------------------------------------------------------------------------------------------
// General path, kernel 1: house update + per-CTA partial sums.  grid = R * chunks CTAs.
// ------------------------------------------------------------------------------------------
template <typename real>
__global__ void __launch_bounds__(kThreads) k_house(Planes<real> pl, SimParams p, StepIn in, int chunks) {
  pdl_wait();      // general path: plain stream order, but the launch latencies of the four kernels overlap
  pdl_trigger();
  const int r = blockIdx.x / chunks, c = blockIdx.x % chunks;
  const int n0 = (c * kThreads + threadIdx.x) * kHousesPerThread;
  const KC<real> kc(p);
  real red[kRed] = {0, 0, 0, 0, 0};
  if (n0 < p.N) {
    House4<real> h;
    const int valid = min(4, p.N - n0);
    house4_step<real>(pl, p, kc, in, (size_t)r * p.Ns + n0, valid, (real)pl.od_temp[r], (real)pl.solar_next[r], h, red);
  }
  __shared__ double wp[kThreads / 32][kRed];
  double out[kRed];
  block_reduce<real, kThreads / 32>(red, out, wp);
  if (threadIdx.x == 0) {
    double *dst = pl.partials + ((size_t)r * chunks + c) * kRed;
    for (int k = 0; k < kRed; ++k) dst[k] = out[k];
  }
}

// 5-D multilinear of scipy.interpolate.interpn as used by interpolation.py:137-178
template <typename real>
DRSIM_D real interp5(const real *sub, const real x[5]) {
  const real g_air[9] = {-4, -2, -1, (real)-0.3, 0, (real)0.3, 1, 2, 4};
  const real g_mass[5] = {-4, -2, 0, 2, 4};
  const real g_od[8] = {1, 3, 5, 7, 9, 11, 13, 15};
  const real g_hour[12] = {0, 10800, 21600, 25200, 27000, 39600, 46800, 57600, 61200, 63000, 75600, 86399};
  const real g_date[6] = {0, 79, 171, 263, 354, 364};
  const real *grids[5] = {g_air, g_mass, g_od, g_hour, g_date};
  const int len[5] = {9, 5, 8, 12, 6};
  const int stride[5] = {5 * 8 * 12 * 6, 8 * 12 * 6, 12 * 6, 6, 1};
  int idx[5];
  real y[5];
#pragma unroll
  for (int d = 0; d < 5; ++d) {
    const real *g = grids[d];
    real v = x[d];
    v = v > g[len[d] - 1] ? g[len[d] - 1] : (v < g[0] ? g[0] : v);  // interpolation.py:245-264
    int i = 0;
    for (int k = 1; k < len[d] - 1; ++k) i += (g[k] <= v) ? 1 : 0;  // g[i] <= v < g[i+1], clipped to [0, n-2]
    idx[d] = i;
    y[d] = (v - g[i]) / (g[i + 1] - g[i]);
  }
  real value = 0;
  for (int corner = 0; corner < 32; ++corner) {  // last dimension fastest (itertools.product order)
    real w = 1;
    int o = 0;
#pragma unroll
    for (int d = 0; d < 5; ++d) {
      const int up = (corner >> (4 - d)) & 1;
      w = w * (up ? y[d] : ((real)1 - y[d]));
      o += (idx[d] + up) * stride[d];
    }
    value = value + __ldg(sub + o) * w;
  }
  return value;
}

// ------------------------------------------------------------------------------------------
// General path, kernel 2: per-cluster reduction of the CTA partials (+ the interpolated base
// power of the sampled houses this handle owns).  One CTA per cluster.
// ------------------------------------------------------------------------------------------
// loads that must observe what OTHER CTAs of the same launch wrote (k_shard): L2, never a stale L1 line
template <typename T>
DRSIM_D T ld_cg(const T *p) {
#if defined(__CUDA_ARCH__)
  return __ldcg(p);
#else
  return *p;
#endif
}
DRSIM_D uint8_t ld_cg(const uint8_t *p) {
#if defined(__CUDA_ARCH__)
  return (uint8_t)__ldcg(reinterpret_cast<const unsigned char *>(p));
#else
  return *p;
#endif
}

constexpr int kReduceThreads = 128;  // threads that take part in reduce_cluster (fixes the combine order)
constexpr int kReduceBatch = 2;      // tile partials a thread has in flight (register budget of the callers)

// Tile partials as self-validating words (k_shard): [tile][16] u64, word 2k / 2k+1 = (tag << 32 | low / high half
// of double k), k < kRed.  The producer needs no fence and no flag, the consumer has the value the moment the
// tags match (the "LL" idea of NCCL's low-latency protocol, here inside one GPU).
struct PartLL {
  unsigned long long *words;   // NULL: the partials are plain doubles in Planes::partials
  uint32_t tag;
  int *err;
  double *stage;               // shared memory: the reducer collects the partials here, [cap][kRed]
  int cap;                     // tiles per collection pass, a multiple of kReduceThreads
  unsigned long long *dbg;     // diagnostics: globaltimer stamps of thread 0 (slots 8..), or NULL
};

DRSIM_D void partll_store(const PartLL &ll, int tile, const double v[kRed]) {
#if defined(__CUDA_ARCH__)
  unsigned long long *dst = ll.words + (size_t)tile * 16;
  const unsigned long long tag = (unsigned long long)ll.tag << 32;
#pragma unroll
  for (int k = 0; k < kRed; ++k) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v[k]);
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(dst + 2 * k), "l"(tag | (bits & 0xffffffffull)),
                 "l"(tag | (bits >> 32))
                 : "memory");
  }
  // the record is one 128-byte line and ALL of it is written: a reader of a partially written 32-byte sector
  // would make the L2 fetch the rest of the sector from HBM first (microseconds while the step is streaming)
#pragma unroll
  for (int k = kRed; k < 8; ++k)
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(dst + 2 * k), "l"(tag), "l"(tag) : "memory");
#endif
}

// the words of one tile's partial, requested (partll_issue) and examined (partll_check) separately so that a
// thread can have the requests of several tiles in flight at once
struct PartWords {
  unsigned long long w[2 * kRed];
};
DRSIM_D void partll_issue(const PartLL &ll, int tile, PartWords &x) {
#if defined(__CUDA_ARCH__)
  const unsigned long long *src = ll.words + (size_t)tile * 16;
#pragma unroll
  for (int k = 0; k < kRed; ++k)
    asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(x.w[2 * k]), "=l"(x.w[2 * k + 1]) : "l"(src + 2 * k) : "memory");
#endif
}
// true (and v filled) when every word carries this step's tag
DRSIM_D bool partll_check(const PartLL &ll, const PartWords &x, double v[kRed]) {
  bool ok = true;
#if defined(__CUDA_ARCH__)
#pragma unroll
  for (int k = 0; k < 2 * kRed; ++k) ok = ok && (uint32_t)(x.w[k] >> 32) == ll.tag;
#pragma unroll
  for (int k = 0; k < kRed; ++k) v[k] = __longlong_as_double((long long)((x.w[2 * k + 1] << 32) | (x.w[2 * k] & 0xffffffffull)));
#endif
  return ok;
}

// Reduction of cluster r: called by EVERY thread of the CTA (it contains CTA barriers); the first
// kReduceThreads threads do the work, in an order that depends on nothing but `chunks`.
// Returns this rank's reduced row [kRed + 1] in shared memory (meaningful on thread 0 only).
template <typename real>
DRSIM_D const double *reduce_cluster(const Planes<real> &pl, const SimParams &p, const StepIn &in, int chunks, const PeerCtx &peer, int r,
                                     const PartLL ll = PartLL{nullptr, 0u, nullptr, nullptr, 0, nullptr}) {
  const bool worker = threadIdx.x < kReduceThreads;
  double red[kRed] = {0, 0, 0, 0, 0};
  // fixed assignment + fixed combine order => deterministic
  if (ll.words) {
    // Collection is decoupled from the fold: EVERY thread of the CTA polls the tiles it owns (a late tile does
    // not hold up the ones behind it -- after the last producer only that tile is outstanding) and parks the
    // values in shared memory; the workers then fold them in the fixed ascending order.
    for (int base = 0; base < chunks; base += ll.cap) {
      const int nb = min(ll.cap, chunks - base);
      const int n_own = (int)threadIdx.x < nb ? (nb - (int)threadIdx.x + (int)blockDim.x - 1) / (int)blockDim.x : 0;   // <= 32
      unsigned pending = n_own >= 32 ? 0xffffffffu : ((1u << n_own) - 1u);
      const long long t0 = clock64();
      if (ll.dbg && threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); ll.dbg[11] = t; ll.dbg[12] = 0; }
      while (pending) {
        if (ll.dbg && threadIdx.x == 0) ll.dbg[12] += 1;
        // the requests of two outstanding tiles fly together (four would spill: 80 registers of words)
        for (int j0 = 0; j0 < n_own; j0 += 2) {
          if (!((pending >> j0) & 0x3u)) continue;
          PartWords x[2];
#pragma unroll
          for (int u = 0; u < 2; ++u)
            if ((pending >> (j0 + u)) & 1u) partll_issue(ll, r * chunks + base + (int)threadIdx.x + (j0 + u) * (int)blockDim.x, x[u]);
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            if (!((pending >> (j0 + u)) & 1u)) continue;
            const int c = (int)threadIdx.x + (j0 + u) * (int)blockDim.x;
            double t[kRed];
            if (partll_check(ll, x[u], t)) {
#pragma unroll
              for (int k = 0; k < kRed; ++k) ll.stage[(size_t)c * kRed + k] = t[k];
              pending &= ~(1u << (j0 + u));
            }
          }
          if (ll.dbg && threadIdx.x == 0 && j0 == 0 && ll.dbg[12] == 1) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); ll.dbg[13] = t; }
        }
#if defined(__CUDA_ARCH__)
        if (pending) __nanosleep(200);   // the pollers share their SM (issue slots, LSU) with CTAs that still compute
#endif
        if (pending && clock64() - t0 > 4000000000ll) {   // ~2 s: give up, flag the error
          *ll.err = 1;
          for (int j = 0; j < n_own; ++j)
            if ((pending >> j) & 1u)
              for (int k = 0; k < kRed; ++k) ll.stage[(size_t)((int)threadIdx.x + j * (int)blockDim.x) * kRed + k] = 0.0;
          pending = 0;
        }
      }
      if (ll.dbg && threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); ll.dbg[8] = t; }
      __syncthreads();
      if (ll.dbg && threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); ll.dbg[9] = t; }
      if (worker)
        for (int c = threadIdx.x; c < nb; c += kReduceThreads) red_combine(red, ll.stage + (size_t)c * kRed);   // base % kReduceThreads == 0
      __syncthreads();
      if (ll.dbg && threadIdx.x == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); ll.dbg[10] = t; }
    }
    // the interpolator / halo parts below read house state written by other CTAs before they stored their partial
    if (in.do_interp > 0 || needs_halo(p)) __threadfence();
  } else if (worker)
    for (int c0 = threadIdx.x; c0 < chunks; c0 += kReduceBatch * kReduceThreads) {
      // kReduceBatch tile partials in flight per thread; they are folded in ascending order (the order is part of the result)
      double t[kReduceBatch][kRed];
#pragma unroll
      for (int u = 0; u < kReduceBatch; ++u) {
        const int c = c0 + u * kReduceThreads;
        if (c < chunks) {
          const double *src = pl.partials + ((size_t)r * chunks + c) * kRed;
#pragma unroll
          for (int k = 0; k < kRed; ++k) t[u][k] = ld_cg(src + k);
        }
      }
#pragma unroll
      for (int u = 0; u < kReduceBatch; ++u)
        if (c0 + u * kReduceThreads < chunks) red_combine(red, t[u]);
    }
  double isum = 0.0;
  if (in.do_interp > 0 && worker) {
    const int k_all = p.n_global <= p.interp_k ? (int)p.n_global : p.interp_k;
    // the interpolator sees the NEW outdoor temperature and datetime (environment.py:94,104-106);
    // both are re-derived here exactly as the epilogue will derive them
    const int64_t epoch_new = pl.epoch[r] + (in.advance ? p.dt : 0);
    const Civil now = civil_from_epoch(epoch_new);
    double od_new = pl.od_temp[r];
    if (in.advance) {
      if (in.sched_od) od_new = in.sched_od[r];
      else {
        double noise = 0.0;
        if (in.od_noise) noise = in.od_noise[r];
        else if (p.noise_mode == DRSIM_NOISE_PHILOX)
          noise = p.temp_std * philox_normal(p.seed, (uint32_t)(p.rep_offset + r), 0u, (uint32_t)in.step, PURPOSE_OD);
        od_new = od_temp_model(now, p.day_temp, p.night_temp, p.phase, noise);
      }
    }
    for (int k = threadIdx.x; k < k_all; k += kReduceThreads) {
      int64_t id;
      if (p.n_global <= p.interp_k) id = k;                       // interpolation.py:220-222
      else if (in.interp_ids) id = in.interp_ids[(size_t)r * p.interp_k + k];
      else {                                                       // random.choices, :223
        const U4 u = philox4x32_10(p.seed, (uint32_t)(p.rep_offset + r), (uint32_t)k, (uint32_t)in.step, PURPOSE_INTERP);
        id = (int64_t)(((uint64_t)u.x * (uint64_t)p.n_global) >> 32);
      }
      id -= p.house_offset;
      if (id < 0 || id >= p.N) continue;                           // owned by another rank
      const size_t o = (size_t)r * p.Ns + id;
      const real tgt = pl.target[o];
      real x[5];
      x[0] = Rep<real>::dev(ld_cg(pl.t_air + o), tgt);
      x[1] = Rep<real>::dev(ld_cg(pl.t_mass + o), tgt);
      x[2] = (real)od_new - tgt;
      if (p.solar_on) {
        x[3] = (real)(now.hour * 3600 + now.minute * 60 + now.second);
        x[4] = (real)now.yday;                                     // quirk Q12
      } else {
        x[3] = 0; x[4] = 0;
      }
      isum += (double)interp5<real>(pl.interp_table + (size_t)pl.interp_sub[o] * DRSIM_INTERP_SUBTABLE_LEN, x);
    }
  }
  __shared__ double wp[kReduceThreads / 32][kRed + 1];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double t[kRed];
#pragma unroll
    for (int k = 0; k < kRed; ++k) t[k] = __shfl_down_sync(0xffffffffu, red[k], o);
    red_combine(red, t);
    isum += __shfl_down_sync(0xffffffffu, isum, o);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0 && worker) {
    for (int k = 0; k < kRed; ++k) wp[w][k] = red[k];
    wp[w][kRed] = isum;
  }
  if (needs_halo(p) && in.advance && (int)threadIdx.x < p.nb_comm) {
    // halo records of the shard's edge houses (post-update state): entries [0, H) = my FIRST H houses
    // (the "after" neighbours of the previous shard's last houses), entries [H, H + L) = my LAST L
    // houses (the "before" neighbours of the next shard's first houses); L = c / 2, H = c - L
    const int c = p.nb_comm, L = c / 2, H = c - L, t = threadIdx.x;
    const int n = t < H ? t : p.N - L + (t - H);
    const size_t o = (size_t)r * p.Ns + n;
    const KC<real> kc(p);
    const real pmax = qdiv(pl.cap[o], kc.cop, kc.inv_cop);
    double rec[kHaloFields];
    rec[0] = (double)div5(Rep<real>::dev(ld_cg(pl.t_air + o), pl.target[o]));  // norm.py:39
    rec[1] = (double)(real)fast_div((uint32_t)ld_cg(pl.sso + o), p.fd_dur);    // norm.py:40-43
    rec[2] = (double)qdiv((ld_cg(pl.flags + o) & 1u) ? pmax : (real)0, kc.nrs, kc.inv_nrs);
    rec[3] = (double)qdiv(pmax, kc.nrs, kc.inv_nrs);
    for (int m = 0; m < 4; ++m) rec[4 + m] = p.msg_thermal ? (double)pl.ratio[m][o] : 0.0;
    double *mine = pl.halo_out + ((size_t)r * c + t) * kHaloFields;
    for (int m = 0; m < kHaloFields; ++m) mine[m] = rec[m];
    if (peer.world > 1) {
      // my first houses are the RIGHT halo of the previous rank, my last houses the LEFT halo of the next
      const int parity = (int)(in.xseq & 1);
      const int dst_rank = t < H ? (peer.rank + peer.world - 1) % peer.world : (peer.rank + 1) % peer.world;
      const int slot = t < H ? L + t : t - H;
      double *dst = peer.halo[dst_rank] + (((size_t)parity * p.R + r) * c + slot) * kHaloFields;
      for (int m = 0; m < kHaloFields; ++m) dst[m] = rec[m];
      __threadfence_system();   // each writer orders its own stores before the flag thread 0 releases below
    }
  }
  __syncthreads();
  __shared__ double s_row[kRed + 1];
  if (threadIdx.x == 0) {
    double a[kRed] = {0, 0, 0, 0, 0};
    double s = 0;
    for (int i = 0; i < kReduceThreads / 32; ++i) { red_combine(a, wp[i]); s += wp[i][kRed]; }
    double *dst = pl.acc + (size_t)r * (kRed + 1);
    for (int k = 0; k < kRed; ++k) { dst[k] = a[k]; s_row[k] = a[k]; }
    dst[kRed] = s;
    s_row[kRed] = s;
  }
  if (peer.world > 1) {
    // the collective: this rank's row goes into slot [parity][rank][r] of EVERY rank's inbox -- one thread
    // per destination, so the NVLink stores, their system-scope fences and the flag releases of the
    // `world` peers overlap instead of queueing behind one thread
    __syncthreads();
    const int q = threadIdx.x;
    if (q < peer.world && peer.rowll) {
      const size_t row = (((size_t)(in.xseq & 1) * peer.world + peer.rank) * p.R + r);
      rowll_store(peer.rowll[q] + row * 16, (uint32_t)in.xseq, s_row);   // no fence, no flag: the words validate themselves
    } else if (q < peer.world) {
      const int parity = (int)(in.xseq & 1);
      const size_t row = (((size_t)parity * peer.world + peer.rank) * p.R + r);
      double *ib = peer.inbox[q] + row * (kRed + 1);
      for (int k = 0; k <= kRed; ++k) ib[k] = s_row[k];
      __threadfence_system();
      unsigned long long *f = peer.flags[q] + row;
#if defined(__CUDA_ARCH__)
      asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f), "l"((unsigned long long)in.xseq) : "memory");
#endif
    }
  }
  return s_row;
}

template <typename real>
__global__ void __launch_bounds__(kReduceThreads) k_reduce(Planes<real> pl, SimParams p, StepIn in, int chunks, PeerCtx peer) {
  pdl_wait();
  pdl_trigger();
  reduce_cluster<real>(pl, p, in, chunks, peer, blockIdx.x);
}

// General path, kernel 3: env epilogue, one thread per cluster.  `acc` holds `n_parts` per-rank
// partial results [n_parts][R][kRed + 1] (n_parts = 1: this handle's own); they are combined here in
// rank order (sums; column 2 is a max), so every rank derives bit-identical cluster totals.
// `defer` != NULL: the env planes are NOT stored here; the caller runs env_epilogue_store(pl, in, r, *defer) later
template <typename real>
DRSIM_D EnvBroadcast<real> env_cluster(const Planes<real> &pl, const SimParams &p, const StepIn &in, const double *acc, int n_parts,
                                       const PeerCtx &peer, int r, EnvOut *defer = nullptr, const EnvRegs *pre = nullptr,
                                       const double *own_row = nullptr) {
  double red[kRed] = {0, 0, 0, 0, 0};
  double isum = 0.0;
  if (peer.world > 1 && peer.rowll) {
    // rows as self-validating words: poll each rank's line (bounded), fold in rank order
    const long long t0 = clock64();
    for (int q = 0; q < peer.world; ++q) {
      const unsigned long long *src = peer.rowll[peer.rank] + ((((size_t)(in.xseq & 1) * peer.world + q) * p.R + r) * 16);
      double t[kRed + 1];
      while (!rowll_try(src, (uint32_t)in.xseq, t)) {
        if (clock64() - t0 > 4000000000ll) {   // ~2 s: give up, flag the error
          *peer.err = 1;
          for (int k = 0; k <= kRed; ++k) t[k] = 0.0;
          break;
        }
      }
      red_combine(red, t);
      isum += t[kRed];
    }
    n_parts = 0;
    own_row = nullptr;
  } else if (peer.world > 1) {
    // wait (bounded) until every rank's row for this step has landed in the local inbox
    const int parity = (int)(in.xseq & 1);
    const unsigned long long want = (unsigned long long)in.xseq;
    const long long t0 = clock64();
    for (int q = 0; q < peer.world; ++q) {
      const unsigned long long *f = peer.flags[peer.rank] + (((size_t)parity * peer.world + q) * p.R + r);
      unsigned long long v = 0;
      do {
#if defined(__CUDA_ARCH__)
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
#endif
        if (v != want && clock64() - t0 > 4000000000ll) { *peer.err = 1; break; }  // ~2 s: give up, flag the error
      } while (v != want);
    }
    acc = peer.inbox[peer.rank] + (size_t)parity * peer.world * p.R * (kRed + 1);
    n_parts = peer.world;
  }
  if (own_row && peer.world <= 1) {   // this rank's row straight from the reducer's shared memory (one part)
    red_combine(red, own_row);
    isum += own_row[kRed];
    n_parts = 0;
  }
  for (int q = 0; q < n_parts; ++q) {
    const double *a = acc + ((size_t)q * p.R + r) * (kRed + 1);
    double t[kRed + 1];
#pragma unroll
    for (int k = 0; k <= kRed; ++k) t[k] = ld_cg(a + k);
    red_combine(red, t);
    isum += t[kRed];
  }
  if (defer) return env_epilogue_compute<real>(pl, p, in, r, pre ? *pre : env_load(pl, in, r), red, isum, *defer);
  return env_epilogue<real>(pl, p, in, r, env_load(pl, in, r), red, isum);
}

template <typename real>
__global__ void k_env(Planes<real> pl, SimParams p, StepIn in, const double *acc, int n_parts, PeerCtx peer) {
  pdl_wait();
  pdl_trigger();
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= p.R) return;
  env_cluster<real>(pl, p, in, acc, n_parts, peer, r);
}

// General path, kernel 4: rewards + observation rows for a chunk of kObsChunk houses.
// Neighbour messages are gathered from global memory (any table); rows are assembled in shared
// memory and written back with coalesced 128-bit stores (2-byte stores where bf16 rows leave a chunk unaligned).
template <typename real, typename O = real, bool SMP = false>
__global__ void __launch_bounds__(kObsChunk) k_obs(Planes<real> pl, SimParams p, StepIn in, int chunks) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  O *tile = reinterpret_cast<O *>(smem_raw);
  pdl_wait();
  pdl_trigger();
  const int r = blockIdx.x / chunks, c = blockIdx.x % chunks;
  const int n = c * kObsChunk + threadIdx.x;
  const int D = p.obs_dim;
  const KC<real> kc(p);
  EnvBroadcast<real> e;
  e.power_n = (real)(pl.power[r] * p.inv_nrs);
  e.signal_n = (real)(pl.signal[r] * p.inv_nrs * p.inv_n_global);
  e.solar_n = (real)(pl.solar_cur[r] * 1e-3);
  e.od_n = (real)((pl.od_temp[r] - 20.0) * 0.2);
  e.rew_sig = (real)pl.rew_sig[r];
  e.pen_common = (real)pl.pen_sum[r];
  e.pen_max = (real)pl.pen_max[r];
  const size_t rb = (size_t)r * p.Ns;
  if (n < p.Ns) {
    O *row = tile + (size_t)threadIdx.x * D;
    if (n < p.N) {
      const size_t o = rb + n;
      const real ta = pl.t_air[o], tm = pl.t_mass[o], tgt = pl.target[o];
      if (in.advance) pl.reward[o] = house_reward<real>(p, kc, ta, tgt, e);
      if (D > 0) {
        real ratio[4] = {0, 0, 0, 0};
        if (p.st_thermal)
          for (int k = 0; k < 4; ++k) ratio[k] = pl.ratio[k][o];
        const uint32_t f = pl.flags[o];
        int i = obs_own<real>(row, p, f, own_sso_norm<real>(pl, p, o, pl.sso[o]), Rep<real>::minus20(ta, tgt),
                              Rep<real>::minus20(tm, tgt), tgt - (real)20, e, ratio);
        if (p.obs_layout == DRSIM_OBS_HAND_ENGINEERED) {
          const bool halo = needs_halo(p);
          RowNbrs<SMP> nbr(p, r, n, rows_draw(in));
          for (int k = 0; k < p.nb_comm; ++k) {
            int nb = nbr(p, pl.comm_table, r, n + (halo ? (int)p.house_offset : 0), k);
            if (halo) {
              // ring neighbour by GLOBAL index; outside this shard it comes from the exchanged halo
              nb -= (int)p.house_offset;
              if (nb < 0 || nb >= p.N) {
                const int L = p.nb_comm / 2;
                int d = nb < 0 ? nb + (int)p.n_global : nb;   // offset from the shard start, wrapped into [0, n_global)
                d = d >= (int)p.n_global ? d - (int)p.n_global : d;
                const bool left = d >= (int)p.n_global - L;
                const double *rec = left ? in.halo_left + ((size_t)r * p.nb_comm + (d - ((int)p.n_global - L))) * kHaloFields
                                         : in.halo_right + ((size_t)r * p.nb_comm + (d - p.N)) * kHaloFields;
                for (int m = 0; m < 4; ++m) row[i++] = (real)rec[m];
                if (p.msg_thermal)
                  for (int m = 0; m < 4; ++m) row[i++] = (real)rec[4 + m];
                if (p.msg_hvac) { row[i++] = (real)p.cop; row[i++] = (real)p.latent; row[i++] = (real)p.dcap; }
                continue;
              }
            }
            const size_t q = rb + nb;
            const real pmax = qdiv(pl.cap[q], kc.cop, kc.inv_cop);
            row[i++] = div5(Rep<real>::dev(pl.t_air[q], pl.target[q]));        // norm.py:39
            row[i++] = (real)fast_div((uint32_t)pl.sso[q], p.fd_dur);          // norm.py:40-43
            row[i++] = qdiv((pl.flags[q] & 1u) ? pmax : (real)0, kc.nrs, kc.inv_nrs);
            row[i++] = qdiv(pmax, kc.nrs, kc.inv_nrs);
            if (p.msg_thermal)
              for (int m = 0; m < 4; ++m) row[i++] = (real)pl.ratio[m][q];
            if (p.msg_hvac) {                                                  // constants, quirk Q11
              row[i++] = (real)p.cop; row[i++] = (real)p.latent; row[i++] = (real)p.dcap;
            }
          }
        }
      }
    } else {
      for (int i = 0; i < D; ++i) row[i] = (real)0;  // padding slot
    }
  }
  if (D == 0) return;
  __syncthreads();
  const int rows = min(kObsChunk, p.Ns - c * kObsChunk);
  const size_t bytes = (size_t)rows * D * sizeof(O);  // rows % 4 == 0 -> multiple of 16 for 4- and 8-byte elements
  O *gdst = pl.template rows<O>() + (rb + (size_t)c * kObsChunk) * D;
  if (sizeof(O) == 2 && ((bytes | reinterpret_cast<uintptr_t>(gdst)) & 15)) {   // bf16 rows of odd D
    const unsigned short *src = reinterpret_cast<const unsigned short *>(tile);
    unsigned short *dst = reinterpret_cast<unsigned short *>(gdst);
    for (size_t i = threadIdx.x; i < bytes / 2; i += blockDim.x) dst[i] = src[i];
    return;
  }
  const uint4 *src = reinterpret_cast<const uint4 *>(tile);
  uint4 *dst = reinterpret_cast<uint4 *>(gdst);
  for (size_t i = threadIdx.x; i < bytes / 16; i += blockDim.x) dst[i] = src[i];
}

// ------------------------------------------------------------------------------------------
// TMA bulk store helpers (shared::cta -> global), PTX ISA cp.async.bulk
// ------------------------------------------------------------------------------------------
DRSIM_D void bulk_store_s2g(void *gdst, const void *ssrc, uint32_t bytes) {
#if defined(__CUDA_ARCH__)
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(ssrc);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(s), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
#endif
}
DRSIM_D void bulk_store_wait_read() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
#endif
}
// ... and for the global writes of those stores too: two bulk stores to the same address are not ordered
DRSIM_D void bulk_store_wait_all() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
#endif
}
DRSIM_D void fence_proxy_async_smem() {
#if defined(__CUDA_ARCH__)
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#endif
}

// geometry of the fused tile kernel, computed on the host
struct FusedGeom {
  int envs_per_tile;   // E: whole clusters per tile (E * Ns <= kTileSlots)
  int n_tiles;         // ceil(R / E)
  int chunk_rows;      // observation rows staged per TMA store (multiple of 4); == E * Ns: "direct"
  int max_segs;        // max clusters overlapping one warp (+1)
  int need_msg;        // neighbour messages are gathered (hand-engineered layout with nb_comm > 0)
  // dynamic shared memory offsets (bytes)
  int off_msg, off_own, off_env, off_wp, off_sold, off_tile, off_in, off_bar, off_stage, smem_bytes;
  int in_stride;       // k_fused_rows: floats per staged input plane (= tile slots)
  int use_tma;         // fp32 direct tiles: inputs staged by TMA bulk loads (k_fused_tma)
  int use_rows;        // fp32 wide rows: per-warp 32-row staging (k_fused_rows)
};

template <typename real>
struct alignas(16) Msg4 {
  real dT, sso_n, p_n, pmax_n;
};
template <typename real>
struct alignas(16) Own4 {
  real ta, tm, target, flags;
};

// resident CTAs per SM the fp32 fused kernel is compiled for.  Measured on B200 (C4 workload):
// 2 (128 registers, no spills) 51.9 us/step; 3 (80 registers) 60.0 us; 4 (64 registers) 66.6 us.
#ifndef DRSIM_FUSED_MINCTAS
#define DRSIM_FUSED_MINCTAS 2
#endif
template <typename real> struct FusedOcc { static constexpr int min_ctas = 1; };
template <> struct FusedOcc<float> { static constexpr int min_ctas = DRSIM_FUSED_MINCTAS; };

// ------------------------------------------------------------------------------------------
// Fused path, chunked variant: one persistent kernel per step (always a real step: refreshes use the
// general path) for tiles whose observation rows do not fit the staging buffer at once.  Phase 1 parks
// every house's message and own-column record in shared memory; phase 3 assembles the rows from them
// g.chunk_rows at a time, one TMA bulk store per chunk.
// ------------------------------------------------------------------------------------------
template <typename real, typename O = real, bool SMP = false>
__global__ void __launch_bounds__(kThreads, FusedOcc<real>::min_ctas)
k_fused(Planes<real> pl, SimParams p, StepIn in, FusedGeom g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Msg4<real> *s_msg = reinterpret_cast<Msg4<real> *>(smem_raw + g.off_msg);
  Own4<real> *s_own = reinterpret_cast<Own4<real> *>(smem_raw + g.off_own);
  EnvBroadcast<real> *s_env = reinterpret_cast<EnvBroadcast<real> *>(smem_raw + g.off_env);
  double *s_wp = reinterpret_cast<double *>(smem_raw + g.off_wp);  // [warps][max_segs][kRed]
  O *s_tile = reinterpret_cast<O *>(smem_raw + g.off_tile);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Ns = p.Ns, D = p.obs_dim;
  const KC<real> kc(p);
  bool store_pending = false;

  for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x) {
    const int r0 = tile * g.envs_per_tile;
    const int E = min(g.envs_per_tile, p.R - r0);
    const int slots = E * Ns;
    const size_t base = (size_t)r0 * Ns;

    // env state of the tile's clusters is fetched early by the threads that will run the epilogue
    EnvRegs er;
    if (threadIdx.x < E) er = env_load(pl, in, r0 + threadIdx.x);

    // ---- phase 1: house update in registers --------------------------------------------
    const int s0 = threadIdx.x * kHousesPerThread;
    const bool active = s0 < slots;
    const int e_loc = active ? (int)fast_div((uint32_t)s0, p.fd_ns) : -1 - warp;  // inactive: never a segment
    House4<real> h;
    real red[kRed] = {0, 0, 0, 0, 0};
    if (active) {
      const int r = r0 + e_loc;
      const int n0 = s0 - e_loc * Ns;
      house4_step<real, true>(pl, p, kc, in, base + s0, min(4, p.N - n0), (real)pl.od_temp[r], (real)pl.solar_next[r], h, red);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t f = (h.flags >> (8 * j)) & 0xffu;
        const real pmax = qdiv(h.cap[j], kc.cop, kc.inv_cop);
        Msg4<real> m;
        m.dT = div5(Rep<real>::dev(h.ta[j], h.target[j]));                  // norm.py:39
        m.sso_n = (real)fast_div((uint32_t)h.sso[j], p.fd_dur);             // norm.py:40-43
        m.p_n = qdiv((f & 1u) ? pmax : (real)0, kc.nrs, kc.inv_nrs);
        m.pmax_n = qdiv(pmax, kc.nrs, kc.inv_nrs);
        if (j >= h.valid) { m.dT = m.sso_n = m.p_n = m.pmax_n = 0; }
        s_msg[s0 + j] = m;
        Own4<real> o;
        o.ta = h.ta[j]; o.tm = h.tm[j]; o.target = h.target[j]; o.flags = (real)f;
        if (j >= h.valid) { o.ta = o.tm = o.target = o.flags = 0; }
        s_own[s0 + j] = o;
      }
    }
    // segmented warp reduction over clusters (lanes of one cluster are contiguous)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      real t[kRed];
#pragma unroll
      for (int k = 0; k < kRed; ++k) t[k] = __shfl_down_sync(0xffffffffu, red[k], o);
      const int eo = __shfl_down_sync(0xffffffffu, e_loc, o);
      if (lane + o < 32 && eo == e_loc) red_combine(red, t);
    }
    const int e_prev = __shfl_up_sync(0xffffffffu, e_loc, 1);
    const bool head = (lane == 0) || (e_prev != e_loc);
    const int e_first = __shfl_sync(0xffffffffu, e_loc, 0);
    if (head && e_loc >= 0) {
      double *dst = s_wp + ((size_t)warp * g.max_segs + (e_loc - e_first)) * kRed;
#pragma unroll
      for (int k = 0; k < kRed; ++k) dst[k] = (double)red[k];
    }
    // the previous tile's bulk store must have finished READING the staging tile before any
    // thread overwrites it in phase 3 of this tile
    if (store_pending && threadIdx.x == 0) bulk_store_wait_read();
    __syncthreads();

    // ---- phase 2: env epilogue on E threads ---------------------------------------------
    if (threadIdx.x < E) {
      const int e = threadIdx.x;
      const int w_lo = (e * Ns) / 128, w_hi = ((e + 1) * Ns - 1) / 128;
      double a[kRed] = {0, 0, 0, 0, 0};
      for (int w = w_lo; w <= w_hi; ++w) {
        const int ef = (w * 128) / Ns;  // first cluster seen by warp w
        red_combine(a, s_wp + ((size_t)w * g.max_segs + (e - ef)) * kRed);
      }
      s_env[e] = env_epilogue<real>(pl, p, in, r0 + e, er, a, 0.0);
    }
    __syncthreads();

    // ---- phase 3: rewards from registers, observation rows through shared memory --------
    if (active) {
      const EnvBroadcast<real> e = s_env[e_loc];
      real rw[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) rw[j] = j < h.valid ? house_reward<real>(p, kc, h.ta[j], h.target[j], e) : (real)0;
      store4(pl.reward + base + s0, rw);
    }
    if (D > 0) {
      for (int cb = 0; cb < slots; cb += g.chunk_rows) {
        const int rows = min(g.chunk_rows, slots - cb);
        if (cb > 0) {
          if (threadIdx.x == 0) bulk_store_wait_read();
          __syncthreads();
        }
        for (int i = threadIdx.x; i < rows; i += kThreads) {
          const int s = cb + i;
          const int e = (int)fast_div((uint32_t)s, p.fd_ns), n = s - e * Ns;
          O *row = s_tile + (size_t)i * D;
          if (n < p.N) {
            const Own4<real> o = s_own[s];
            const Msg4<real> m = s_msg[s];
            real ratio[4] = {0, 0, 0, 0};
            if (p.st_thermal)
              for (int k = 0; k < 4; ++k) ratio[k] = pl.ratio[k][base + s];
            int q = obs_own<real>(row, p, (uint32_t)o.flags, m.sso_n, Rep<real>::minus20(o.ta, o.target),
                                  Rep<real>::minus20(o.tm, o.target), o.target - (real)20, s_env[e], ratio);
            if (g.need_msg) {
              RowNbrs<SMP> nbr(p, r0 + e, n, rows_draw(in));
              for (int k = 0; k < p.nb_comm; ++k) {
                const int nb = nbr(p, pl.comm_table, r0 + e, n, k);
                const Msg4<real> mk = s_msg[e * Ns + nb];
                row[q++] = mk.dT; row[q++] = mk.sso_n; row[q++] = mk.p_n; row[q++] = mk.pmax_n;
                if (p.msg_thermal)
                  for (int t = 0; t < 4; ++t) row[q++] = (real)pl.ratio[t][base + e * Ns + nb];
                if (p.msg_hvac) { row[q++] = (real)p.cop; row[q++] = (real)p.latent; row[q++] = (real)p.dcap; }
              }
            }
          } else {
            for (int q = 0; q < D; ++q) row[q] = (real)0;
          }
        }
        fence_proxy_async_smem();
        __syncthreads();
        if (threadIdx.x == 0) {
          bulk_store_s2g(pl.template rows<O>() + (base + cb) * D, s_tile, (uint32_t)((size_t)rows * D * sizeof(O)));
          store_pending = true;
        }
      }
    }
    // s_msg / s_own / s_env / s_wp are rewritten by the next tile's phase 1: all readers are done
    // after this barrier (the staging tile itself is protected by wait_group.read above)
    __syncthreads();
  }
  if (threadIdx.x == 0 && store_pending) {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
#endif
  }
}

// ------------------------------------------------------------------------------------------
// Fused path, "direct" variant -- the production kernel.
//
// The whole tile's observation rows fit the staging buffer, so every thread writes the rows of its
// own 4 houses straight from registers.  Per tile there are exactly two CTA barriers, bracketing a
// ~100-instruction critical section on E threads (combine the warp partials, signal penalty,
// regulation signal); everything else the epilogue does (env plane stores, metrics) happens after
// the barrier is released.  Row columns that depend on the house only are written before the first
// barrier; the two env-dependent columns, the neighbour messages and the rewards after the second.
// Each warp ships its own 128 rows with one TMA bulk store (no CTA barrier in front of it).
// ------------------------------------------------------------------------------------------
template <typename real, typename O = real, bool SMP = false>
__global__ void __launch_bounds__(kThreads, FusedOcc<real>::min_ctas)
k_fused_direct(Planes<real> pl, SimParams p, StepIn in, FusedGeom g) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Msg4<real> *s_msg_base = reinterpret_cast<Msg4<real> *>(smem_raw + g.off_msg);  // [2][slots] if need_msg
  EnvBroadcast<real> *s_env = reinterpret_cast<EnvBroadcast<real> *>(smem_raw + g.off_env);
  double *s_wp = reinterpret_cast<double *>(smem_raw + g.off_wp);  // [warps][max_segs][kRed]
  O *s_tile = reinterpret_cast<O *>(smem_raw + g.off_tile);

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Ns = p.Ns, D = p.obs_dim;
  const int tile_slots = g.envs_per_tile * Ns;
  const KC<real> kc(p);
  const bool fast = in.sched_od != nullptr;
  // lean row layout: fp32, no optional state/message columns, 4-float messages
  const bool plain = sizeof(real) == 4 && p.own_dim == 10 && p.msg_dim == 4 && (D % 2) == 0;
  bool store_pending = false;  // meaningful on lane 0 of each warp
  int parity = 0;

  for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, parity ^= 1) {
    const int r0 = tile * g.envs_per_tile;
    const int E = min(g.envs_per_tile, p.R - r0);
    const int slots = E * Ns;
    const size_t base = (size_t)r0 * Ns;
    Msg4<real> *s_msg = s_msg_base + (size_t)parity * tile_slots;

    EnvRegs er;
    if (threadIdx.x < E) er = env_load(pl, in, r0 + threadIdx.x);

    // ---- phase 1: house update in registers, house-only row columns ----------------------
    const int s0 = threadIdx.x * kHousesPerThread;
    const bool active = s0 < slots;
    const int e_loc = active ? (int)fast_div((uint32_t)s0, p.fd_ns) : -1 - warp;
    const int n0 = s0 - e_loc * Ns;
    House4<real> h;
    real red[kRed] = {0, 0, 0, 0, 0};
    // the warp's previous TMA store must have finished reading its rows before they are rewritten
    if (lane == 0 && store_pending) bulk_store_wait_read();
    __syncwarp();
    if (active) {
      const int r = r0 + e_loc;
      house4_dispatch<true>(pl, p, kc, in, base + s0, min(4, p.N - n0), (real)pl.od_temp[r], (real)pl.solar_next[r], h, red);
      EnvBroadcast<real> none{};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t f = (h.flags >> (8 * j)) & 0xffu;
        const real sso_n = (real)fast_div((uint32_t)h.sso[j], p.fd_dur);            // norm.py:40-43, :79-82
        if (g.need_msg) {
          const real pmax_n = qdiv(qdiv(h.cap[j], kc.cop, kc.inv_cop), kc.nrs, kc.inv_nrs);
          Msg4<real> m;
          m.dT = div5(Rep<real>::dev(h.ta[j], h.target[j]));                        // norm.py:39
          m.sso_n = sso_n;
          m.p_n = (f & 1u) ? pmax_n : (real)0;
          m.pmax_n = pmax_n;
          if (j >= h.valid) { m.dT = m.sso_n = m.p_n = m.pmax_n = 0; }
          s_msg[s0 + j] = m;
        }
        if (D > 0) {
          O *row = s_tile + (size_t)(s0 + j) * D;
          if (plain) {
            // own_dim == 10, even D: rows are 8-byte aligned -> 64-bit shared stores
            if constexpr (sizeof(real) == 4) {
              const float tg = h.target[j] - 20.f;
              const bool ok = j < h.valid;
              put2(row, 0, ok ? (float)(f & 1u) : 0.f, ok ? (float)((f >> 1) & 1u) : 0.f);
              put2(row, 1, ok ? sso_n : 0.f, ok ? 1.f : 0.f);
              put2(row, 3, ok ? p.hf.deadband : 0.f, ok ? (h.ta[j] + tg) * 0.2f : 0.f);
              put2(row, 4, ok ? (h.tm[j] + tg) * 0.2f : 0.f, ok ? tg * 0.2f : 0.f);
              if (!ok) {
                put2(row, 2, 0.f, 0.f);
                for (int q = 5; q < D / 2; ++q) put2(row, q, 0.f, 0.f);
              }
            }
          } else if (j < h.valid) {
            real ratio[4] = {0, 0, 0, 0};
            if (p.st_thermal)
              for (int k = 0; k < 4; ++k) ratio[k] = pl.ratio[k][base + s0 + j];
            obs_own<real>(row, p, f, sso_n, Rep<real>::minus20(h.ta[j], h.target[j]),
                          Rep<real>::minus20(h.tm[j], h.target[j]), h.target[j] - (real)20, none, ratio, 1);
          } else {
            for (int q = 0; q < D; ++q) row[q] = (real)0;
          }
        }
      }
    }
    // segmented warp reduction over clusters (lanes of one cluster are contiguous)
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      real t[kRed];
#pragma unroll
      for (int k = 0; k < kRed; ++k) t[k] = __shfl_down_sync(0xffffffffu, red[k], o);
      const int eo = __shfl_down_sync(0xffffffffu, e_loc, o);
      if (lane + o < 32 && eo == e_loc) red_combine(red, t);
    }
    const int e_prev = __shfl_up_sync(0xffffffffu, e_loc, 1);
    const bool head = (lane == 0) || (e_prev != e_loc);
    const int e_first = __shfl_sync(0xffffffffu, e_loc, 0);
    if (head && e_loc >= 0) {
      double *dst = s_wp + ((size_t)warp * g.max_segs + (e_loc - e_first)) * kRed;
#pragma unroll
      for (int k = 0; k < kRed; ++k) dst[k] = (double)red[k];
    }
    __syncthreads();

    // ---- phase 2: the short critical section on E threads ---------------------------------
    double a[kRed] = {0, 0, 0, 0, 0};
    EnvFast ef;
    if (threadIdx.x < E) {
      const int e = threadIdx.x;
      const int w_lo = (e * Ns) / 128, w_hi = ((e + 1) * Ns - 1) / 128;
      for (int w = w_lo; w <= w_hi; ++w) {
        const int efst = (w * 128) / Ns;  // first cluster seen by warp w
        red_combine(a, s_wp + ((size_t)w * g.max_segs + (e - efst)) * kRed);
      }
      if (fast) s_env[e] = env_fast_compute<real>(p, er, a, ef);
      else s_env[e] = env_epilogue<real>(pl, p, in, r0 + e, er, a, 0.0);  // injected noise: full inline path
    }
    __syncthreads();

    // ---- phase 3: env-dependent columns, neighbour messages, rewards ----------------------
    if (active) {
      const EnvBroadcast<real> e = s_env[e_loc];
      real rw[4];
      bool lean_reward = false;
      if constexpr (sizeof(real) == 4) lean_reward = p.penalty_mode == DRSIM_PEN_INDIVIDUAL_L2;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if constexpr (sizeof(real) == 4) {
          rw[j] = lean_reward ? reward_f32_individual(p, h.ta[j], e.rew_sig) : house_reward<real>(p, kc, h.ta[j], h.target[j], e);
          if (j >= h.valid) rw[j] = 0.f;
        } else {
          rw[j] = j < h.valid ? house_reward<real>(p, kc, h.ta[j], h.target[j], e) : (real)0;
        }
      }
      store4(pl.reward + base + s0, rw);
      if (D > 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j < h.valid) {
            O *row = s_tile + (size_t)(s0 + j) * D;
            if (plain) {
              if constexpr (sizeof(real) == 4) {
                put2(row, 2, e.power_n, e.signal_n);
                if (g.need_msg) {
                  RowNbrs<SMP> nbr(p, r0 + e_loc, n0 + j, rows_draw(in));
                  for (int k = 0; k < p.nb_comm; ++k) {
                    const int nb = nbr(p, pl.comm_table, r0 + e_loc, n0 + j, k);
                    const float4 mk = *reinterpret_cast<const float4 *>(&s_msg[e_loc * Ns + nb]);
                    put2(row, 5 + 2 * k, mk.x, mk.y);
                    put2(row, 6 + 2 * k, mk.z, mk.w);
                  }
                }
              }
              continue;
            }
            int q = obs_own<real>(row, p, 0u, (real)0, (real)0, (real)0, (real)0, e, nullptr, 2);
            if (g.need_msg) {
              RowNbrs<SMP> nbr(p, r0 + e_loc, n0 + j, rows_draw(in));
              for (int k = 0; k < p.nb_comm; ++k) {
                const int nb = nbr(p, pl.comm_table, r0 + e_loc, n0 + j, k);
                const Msg4<real> mk = s_msg[e_loc * Ns + nb];
                row[q++] = mk.dT; row[q++] = mk.sso_n; row[q++] = mk.p_n; row[q++] = mk.pmax_n;
                if (p.msg_thermal)
                  for (int t = 0; t < 4; ++t) row[q++] = (real)pl.ratio[t][base + e_loc * Ns + nb];
                if (p.msg_hvac) { row[q++] = (real)p.cop; row[q++] = (real)p.latent; row[q++] = (real)p.dcap; }
              }
            }
          }
        }
      }
    }
    if (D > 0) {
      // every lane's generic-proxy writes to the warp's rows become visible to the async proxy,
      // then lane 0 ships the warp's rows [128 w, 128 w + 128) with one bulk store
      fence_proxy_async_smem();
      __syncwarp();
      const int w0 = warp * 128;
      if (lane == 0 && w0 < slots) {
        const int nrows = min(128, slots - w0);
        bulk_store_s2g(pl.template rows<O>() + (base + w0) * D, s_tile + (size_t)w0 * D, (uint32_t)((size_t)nrows * D * sizeof(O)));
        store_pending = true;
      }
    }
    // off the critical path: env planes + running metrics
    if (threadIdx.x < E && fast) env_fast_store<real>(pl, p, r0 + threadIdx.x, er, ef, a);
  }
  if (lane == 0 && store_pending) {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
#endif
  }
}

// ------------------------------------------------------------------------------------------
// mbarrier + TMA bulk LOAD helpers (global -> shared::cta, completion on an mbarrier)
// ------------------------------------------------------------------------------------------
DRSIM_D void mbar_init(uint64_t *bar, uint32_t count) {
#if defined(__CUDA_ARCH__)
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
#endif
}
DRSIM_D void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
#if defined(__CUDA_ARCH__)
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)),
               "r"(bytes)
               : "memory");
#endif
}
DRSIM_D void mbar_wait(uint64_t *bar, uint32_t parity) {
#if defined(__CUDA_ARCH__)
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra.uni WAIT_DONE;\n"
      "bra.uni WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(a),
      "r"(parity)
      : "memory");
#endif
}
DRSIM_D void bulk_load_g2s(void *sdst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(sdst)),
               "l"(gsrc), "r"(bytes), "r"((uint32_t)__cvta_generic_to_shared(bar))
               : "memory");
#endif
}

DRSIM_D void bulk_load_g2s_hint(void *sdst, const void *gsrc, uint32_t bytes, uint64_t *bar, uint64_t pol) {
#if defined(__CUDA_ARCH__)
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          (uint32_t)__cvta_generic_to_shared(sdst)),
      "l"(gsrc), "r"(bytes), "r"((uint32_t)__cvta_generic_to_shared(bar)), "l"(pol)
      : "memory");
#endif
}

// 16-byte asynchronous copies global -> shared (LDGSTS), used for the per-cluster schedule record
DRSIM_D void cp_async16(void *sdst, const void *gsrc) {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(sdst)), "l"(gsrc)
               : "memory");
#endif
}
DRSIM_D void cp_async_wait_all() {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.wait_all;" ::: "memory");
#endif
}

// per-cluster record staged in shared memory by the fused fp32 kernels: the step's SchedRec followed
// by the running metrics of the cluster (read-modify-write at the end of the tile)
struct alignas(16) EnvStage {
  SchedRec rec;
  double m[DRSIM_N_METRICS];
};
static_assert(sizeof(EnvStage) == 128 && DRSIM_N_METRICS == 6, "EnvStage: 5 + 3 cp.async pieces");

// issued by thread e < E for cluster r: 8 copies, no registers held while they fly
DRSIM_D void env_stage_fetch(EnvStage *dst, const SchedRec *rec, const double *metrics, int r) {
  const char *src = reinterpret_cast<const char *>(rec + r);
  char *d = reinterpret_cast<char *>(dst);
#pragma unroll
  for (int k = 0; k < 5; ++k) cp_async16(d + 16 * k, src + 16 * k);
  const char *ms = reinterpret_cast<const char *>(metrics + (size_t)r * DRSIM_N_METRICS);
#pragma unroll
  for (int k = 0; k < 3; ++k) cp_async16(d + 80 + 16 * k, ms + 16 * k);
}

// env_fast_store from a staged record: env planes + running metrics of cluster r after the step
template <typename real>
DRSIM_D void env_stage_store(const Planes<real> &pl, const SimParams &p, int r, const EnvStage &st, const double red[kRed],
                             double *host_env = nullptr, double *m_next = nullptr) {
  const SchedRec &c = st.rec;
  const double P = red[0];
  const double rew_sig = signal_penalty(p, P, c.signal_prev);
  pl.epoch[r] = c.epoch;
  pl.od_temp[r] = c.od;
  pl.solar_next[r] = c.solar_next;
  pl.solar_cur[r] = c.solar_cur;
  pl.signal[r] = c.signal;
  pl.base_power[r] = c.base_power;
  pl.power[r] = P;
  pl.pen_sum[r] = red[1];
  pl.pen_max[r] = red[2];
  pl.rew_sig[r] = rew_sig;
  if (p.base_mode != DRSIM_BASE_CONSTANT) pl.t_since_interp[r] = c.tsi;
  double *m = pl.metrics + (size_t)r * DRSIM_N_METRICS;
  const double d = P - c.signal_prev;
  const double mr = mean_reward(p, red[1], red[2], rew_sig);
  const double nm[DRSIM_N_METRICS] = {st.m[0] + 1.0, st.m[1] + mr, st.m[2] + fabs(red[3]) * p.inv_n_global,
                                      st.m[3] + red[4] * p.inv_n_global, st.m[4] + fabs(d), st.m[5] + d * d};
#pragma unroll
  for (int q = 0; q < DRSIM_N_METRICS; ++q) m[q] = nm[q];
  if (m_next) {  // in-kernel episode: the next step's staged record takes its running metrics from here
#pragma unroll
    for (int q = 0; q < DRSIM_N_METRICS; ++q) m_next[q] = nm[q];
  }
  if (host_env) {  // drsim_step_host: the per-cluster results go straight to host memory (posted PCIe writes, no D2H copy)
    double *o = host_env + (size_t)r * 4;
    o[0] = P; o[1] = c.signal; o[2] = c.od; o[3] = mr;
  }
}

constexpr int kInPlanes = 12;  // fp32 planes staged by TMA: Ta, Tm, sso, target, cap, 6 coefficients (+1 spare)

// Phase counters of the k_fused_tma step loop (build with -DDRSIM_TILE_DBG, read by drsim_debug_tile_phases and
// profiles/tools/tile_phases.py): every warp accumulates the clock() cycles of each phase of a tile-step over the
// launch, and lane 0 adds them to g_tile_dbg[cta][warp][phase].  In the default build the marks compile to nothing.
enum TilePhase { kPhHouse, kPhRows, kPhBarrier, kPhFold, kPhStore, kPhEpilogue, kPhSteps, kTilePhases = 8 };
#ifdef DRSIM_TILE_DBG
constexpr int kTileDbgCtas = 1024;
__device__ unsigned long long g_tile_dbg[kTileDbgCtas][kThreads / 32][kTilePhases];
struct TileClock {   // 32-bit counters (a launch is a few million cycles per warp): few registers in the debug build
  unsigned t, acc[kTilePhases];
  DRSIM_D TileClock() : t((unsigned)clock()) {
#pragma unroll
    for (int k = 0; k < kTilePhases; ++k) acc[k] = 0;
  }
  DRSIM_D void mark(int k) { const unsigned n = (unsigned)clock(); acc[k] += n - t; t = n; }
  DRSIM_D void step() { ++acc[kPhSteps]; }
  DRSIM_D void flush() {
    if ((threadIdx.x & 31) == 0 && blockIdx.x < kTileDbgCtas)
#pragma unroll
      for (int k = 0; k < kTilePhases; ++k) atomicAdd(&g_tile_dbg[blockIdx.x][threadIdx.x >> 5][k], (unsigned long long)acc[k]);
  }
};
#else
struct TileClock {
  DRSIM_D void mark(int) {}
  DRSIM_D void step() {}
  DRSIM_D void flush() {}
};
#endif

// ------------------------------------------------------------------------------------------
// Fused path, fp32 production kernel with TMA-staged inputs.
//
// Same tile structure as k_fused_direct, but the eleven 32-bit input planes of a tile never go
// through registers on their way in: each warp owns the 128 house slots it processes, prefetches
// them for the NEXT tile with eleven TMA bulk loads (cp.async.bulk.shared.global, completion on the
// warp's own mbarrier) as soon as it has consumed the current ones, and reads them back with
// conflict-free 128-bit shared loads.  HBM therefore stays busy while the CTA sits in its two
// barriers and assembles observation rows; the load path needs only warp-level synchronisation.
// The two byte planes (flags, actions) are 8-byte aligned at odd replica indices, which the bulk
// copy engine cannot address, so they are prefetched through two registers instead.
// ------------------------------------------------------------------------------------------
// MODE selects a compile-time specialisation so the hot instantiations carry no runtime layout /
// policy branches: 0 = generic (everything decided at run time), 1 = one cluster per tile, plain
// 10-column rows without neighbour messages, external actions, individual_L2, scheduled noise
// (BASELINE config 4), 2 = several clusters per tile, plain rows WITH 4-float neighbour messages,
// external actions, individual_L2, scheduled noise (config 3).
// thread-private staging copies (LDGSTS): 16 / 8 / 4 bytes global -> shared with an L2 eviction hint
DRSIM_D void cp_async16_hint(void *sdst, const void *gsrc, uint64_t pol) {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(sdst)),
               "l"(gsrc), "l"(pol)
               : "memory");
#endif
}
DRSIM_D void cp_async8(void *sdst, const void *gsrc) {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(sdst)), "l"(gsrc)
               : "memory");
#endif
}
DRSIM_D void cp_async4(void *sdst, const void *gsrc) {
#if defined(__CUDA_ARCH__)
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(sdst)), "l"(gsrc)
               : "memory");
#endif
}



// Action word of a thread's four houses on the copy-engine path of drsim_step_host (see StepIn::act_poll_err)
DRSIM_D uint32_t act_word_polled(const uint8_t *actions, size_t off, uint32_t staged, int *err) {
  uint32_t v = staged;
#if defined(__CUDA_ARCH__)
  uint32_t *ga = reinterpret_cast<uint32_t *>(const_cast<uint8_t *>(actions + off));
  if (v == 0xFFFFFFFFu) {
    for (int spin = 0;; ++spin) {
      asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(ga) : "memory");
      if (v != 0xFFFFFFFFu) break;
      if (spin > (1 << 21)) { *err = 1; v = 0; break; }   // ~2 s: the copy never came
      __nanosleep(100);
    }
  }
  *ga = 0xFFFFFFFFu;   // poison for the next step's copy
#endif
  return v;
}

// Observation rows of MODE 1 of k_fused_tma (plain 10-column rows, no messages).  A thread's four rows are contiguous in
// the tile's staging rows: 160 bytes in fp32, 80 in bf16.  Before the tile barrier the thread writes all of them with
// 16-byte stores, the power / signal columns (4, 5) as zeros; after the fold own_rows10_patch puts those two columns
// into the valid rows.  fp32: at a 160-byte lane stride lanes t and t + 4 of a quarter-warp would hit the same banks, so
// lanes with bit 2 set assemble their houses in the order 2, 3, 0, 1: their k-th store lands 80 bytes (20 banks) away
// from that of lane t and each 16-byte store takes one wavefront per quarter-warp.  bf16 needs no swap: an 80-byte
// lane stride already puts the eight lanes of a quarter-warp on distinct banks.
template <typename O>
DRSIM_D void own_rows10(O *rows, const House4<float> &h, const SimParams &p, int lane) {
  const int sw = (sizeof(O) == 4 && (lane & 4)) ? 2 : 0;
  float v[40];
#pragma unroll
  for (int jv = 0; jv < 4; ++jv) {   // row jv of the thread's store order holds house jv ^ sw
    const int j = jv ^ sw;
    const float ta = sw ? h.ta[jv ^ 2] : h.ta[jv];
    const float tm = sw ? h.tm[jv ^ 2] : h.tm[jv];
    const float target = sw ? h.target[jv ^ 2] : h.target[jv];
    const int sso = sw ? h.sso[jv ^ 2] : h.sso[jv];
    const uint32_t f = (h.flags >> (8 * j)) & 0xffu;
    const float sso_n = (float)fast_div((uint32_t)sso, p.fd_dur);            // norm.py:40-43, :79-82
    const bool ok = j < h.valid;
    const float tg = target - 20.f;
    float *r = v + 10 * jv;
    r[0] = ok ? (float)(f & 1u) : 0.f;
    r[1] = ok ? (float)((f >> 1) & 1u) : 0.f;
    r[2] = ok ? sso_n : 0.f;
    r[3] = ok ? 1.f : 0.f;
    r[4] = 0.f;
    r[5] = 0.f;
    r[6] = ok ? p.hf.deadband : 0.f;
    r[7] = ok ? (ta + tg) * 0.2f : 0.f;
    r[8] = ok ? (tm + tg) * 0.2f : 0.f;
    r[9] = ok ? tg * 0.2f : 0.f;
  }
  if constexpr (sizeof(O) == 4) {
    float4 *dst = reinterpret_cast<float4 *>(rows);
#pragma unroll
    for (int k = 0; k < 10; ++k)
      dst[k < 5 ? k + 5 * (sw >> 1) : k - 5 * (sw >> 1)] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
  } else {
    auto pk = [&](int i) {
      const __nv_bfloat162 b = __floats2bfloat162_rn(v[i], v[i + 1]);
      return *reinterpret_cast<const uint32_t *>(&b);
    };
    uint4 *dst = reinterpret_cast<uint4 *>(rows);
#pragma unroll
    for (int k = 0; k < 5; ++k) dst[k] = make_uint4(pk(8 * k), pk(8 * k + 2), pk(8 * k + 4), pk(8 * k + 6));
  }
}

// columns 4, 5 of the thread's valid rows.  The k-th store goes to row (k + lane / 4) % 4 (fp32: 8-byte stores, taken by
// half-warps) or (k + lane / 8) % 4 (bf16: 4-byte stores), which spreads each store over all 32 banks.
template <typename O>
DRSIM_D void own_rows10_patch(O *rows, int valid, int lane, float power_n, float signal_n) {
  const int rot = sizeof(O) == 4 ? lane >> 2 : lane >> 3;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int j = (k + rot) & 3;
    if (j < valid) put2(rows + 10 * j, 2, power_n, signal_n);
  }
}

// POLL = copy-engine mode of drsim_step_host (StepIn::act_poll_err): a separate instantiation, so the
// device-resident step does not carry the branch (measured: 0.6 us of 39 on C4)
template <int MODE, bool POLL = false, typename O = float, bool SMP = false>
__global__ void __launch_bounds__(kThreads, DRSIM_FUSED_MINCTAS)
k_fused_tma(Planes<float> pl, SimParams p, StepIn in, FusedGeom g) {
  typedef float real;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Msg4<real> *s_msg_base = reinterpret_cast<Msg4<real> *>(smem_raw + g.off_msg);
  // s_env / s_wp / s_sold are double-buffered by tile parity: a warp may run ahead into the next
  // tile's phase 1 while slower warps still read this tile's values (one CTA barrier per tile)
  EnvBroadcast<real> *s_env_base = reinterpret_cast<EnvBroadcast<real> *>(smem_raw + g.off_env);
  double *s_wp_base = reinterpret_cast<double *>(smem_raw + g.off_wp);
  double *s_sold_base = reinterpret_cast<double *>(smem_raw + g.off_sold);  // [2][E] previous signal
  EnvStage *s_stage_base = reinterpret_cast<EnvStage *>(smem_raw + g.off_stage);  // [2][E] schedule record + metrics
  O *s_tile = reinterpret_cast<O *>(smem_raw + g.off_tile);
  float *s_in = reinterpret_cast<float *>(smem_raw + g.off_in);        // [kInPlanes][kTileSlots]

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Ns = p.Ns, D = MODE == 1 ? 10 : p.obs_dim;   // MODE 1 runs on 10-column rows only (tile_route)
  const int tile_slots = g.envs_per_tile * Ns;
  const KC<real> kc(p);
  const bool fast = MODE ? true : in.sched_od != nullptr;
  const bool plain = MODE ? true : (p.own_dim == 10 && p.msg_dim == 4 && (D % 2) == 0);
  const bool ext = MODE ? true : (p.policy == DRSIM_POLICY_EXTERNAL || p.policy == DRSIM_POLICY_GREEDY_MYOPIC);
  const bool need_msg = MODE == 1 ? false : (MODE == 2 ? true : g.need_msg != 0);
  const bool one_env = MODE == 1 ? true : (MODE == 2 ? false : g.envs_per_tile == 1);
  const bool individual = MODE ? true : p.penalty_mode == DRSIM_PEN_INDIVIDUAL_L2;
  const uint8_t *actions = in.actions ? in.actions : pl.actions;
  const uint64_t pol_keep = l2_policy_evict_last(), pol_stream = l2_policy_evict_first();
  bool store_pending = false;
  int parity = 0;
  const int s0 = threadIdx.x * kHousesPerThread;
  const int w0 = warp * 128;

  // the spare staging plane holds the thread-private small inputs: flags word, action word, (od, solar)
  uint32_t *s_flags = reinterpret_cast<uint32_t *>(s_in + (size_t)11 * kTileSlots);
  uint32_t *s_act = s_flags + kThreads;
  float2 *s_os = reinterpret_cast<float2 *>(s_act + kThreads);

  // prefetch of tile `t`.  Every thread copies the 16 bytes it will consume of each of the eleven
  // 32-bit planes (plus its flags / action words and the cluster's two fp32 scalars) straight into its
  // own staging slots with cp.async: no registers are held while the copies fly, nobody else reads the
  // slots, so completion is one cp.async.wait_all of the thread itself -- no barrier, no mbarrier, and
  // none of the per-copy issue latency of 512-byte TMA bulk loads (measured: 20 % of the stall samples)
  float nx_od = 0.f, nx_solar = 0.f;
  const int n_steps = in.stream_steps > 1 ? in.stream_steps : 1;   // in-kernel step loop (StepIn::stream_steps)
  auto step_actions = [&](int st) -> const uint8_t * {
    if (n_steps == 1 || !in.actions) return actions;
    const int j = in.tape_first + st;
    return in.actions + (size_t)(in.tape_planes > 0 ? j % in.tape_planes : j) * in.tape_stride;
  };
  // every tile starts at step 0 of the launch.  `part`: 1 = launch-invariant static planes only (may run
  // before pdl_wait), 2 = the rest, 3 = both
  auto prefetch = [&](int t, int part) {
    constexpr int st = 0;
    const int tr0 = t * g.envs_per_tile;
    const int tslots = min(g.envs_per_tile, p.R - tr0) * Ns;
    const size_t tbase = (size_t)tr0 * Ns;
    if (s0 < tslots) {
      const int r = tr0 + (one_env ? 0 : (int)fast_div((uint32_t)s0, p.fd_ns));
      const size_t o = tbase + s0;
      float *d = s_in + s0;
      if (part & 1) {
        cp_async16_hint(d + 3 * kTileSlots, pl.target + o, pol_keep);
        cp_async16_hint(d + 4 * kTileSlots, pl.cap + o, pol_keep);
#pragma unroll
        for (int c = 0; c < 6; ++c) cp_async16_hint(d + (5 + c) * kTileSlots, pl.coef[c] + o, pol_keep);
      }
      if (part & 2) {
        cp_async16_hint(d, pl.t_air + o, pol_keep);
        cp_async16_hint(d + kTileSlots, pl.t_mass + o, pol_keep);
        cp_async16_hint(d + 2 * kTileSlots, pl.sso + o, pol_keep);
        cp_async4(s_flags + threadIdx.x, pl.flags + o);
        if (ext) cp_async4(s_act + threadIdx.x, step_actions(st) + o);
        if (fast) cp_async8(s_os + threadIdx.x, &in.sched_rec[(size_t)st * p.R + r].od_prev_f);
      }
      if (!fast && (part & 2)) {
        nx_od = (float)pl.od_temp[r];
        nx_solar = (float)pl.solar_next[r];
      }
    }
  };
  // schedule record + running metrics of tile t's clusters at step 0 -> shared memory (threads e < E, cp.async)
  auto fetch_env = [&](int t, int par) {
    const int tr0 = t * g.envs_per_tile;
    if ((int)threadIdx.x < min(g.envs_per_tile, p.R - tr0))
      env_stage_fetch(s_stage_base + (size_t)par * g.envs_per_tile + threadIdx.x, in.sched_rec, pl.metrics, tr0 + threadIdx.x);
  };
  pdl_trigger();
  if ((int)blockIdx.x < g.n_tiles) prefetch(blockIdx.x, 1);
  pdl_wait();
  if ((int)blockIdx.x < g.n_tiles) {
    prefetch(blockIdx.x, 2);
    if (fast) fetch_env(blockIdx.x, 0);
  }

  TileClock clk;
  // Tile-major step loop: a tile runs through all n_steps steps before the CTA moves to its next tile.
  // Between two steps of a tile the thread's updated state goes back into its own staging slots, the static
  // planes stay there, the next step's action word, (od, solar) pair and schedule record are fetched while
  // this step computes, and the running metrics travel through the staged record: the tile's planes come
  // from global memory once per launch.  Every step still stores everything a single step stores.
  for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x)
  for (int st = 0; st < n_steps; ++st, parity ^= 1) {
    const bool more = st + 1 < n_steps;   // the item after this one is this tile's next step
    const int nt = tile + gridDim.x;      // ... otherwise the CTA's next tile, from step 0
    const int r0 = tile * g.envs_per_tile;
    const int E = min(g.envs_per_tile, p.R - r0);
    const int slots = E * Ns;
    const size_t base = (size_t)r0 * Ns;
    Msg4<real> *s_msg = s_msg_base + (size_t)parity * tile_slots;
    EnvBroadcast<real> *s_env = s_env_base + (size_t)parity * g.envs_per_tile;
    double *s_wp = s_wp_base + (size_t)parity * (kThreads / 32) * g.max_segs * kRed;
    double *s_sold = s_sold_base + (size_t)parity * g.envs_per_tile;

    const EnvStage *s_stage = s_stage_base + (size_t)parity * g.envs_per_tile;
    EnvRegs er;
    if constexpr (MODE == 0) {
      if (!fast && threadIdx.x < E) er = env_load(pl, in, r0 + threadIdx.x);
    }

    // ---- phase 1 -----------------------------------------------------------------------
    const bool active = s0 < slots;
    const int e_loc = active ? (one_env ? 0 : (int)fast_div((uint32_t)s0, p.fd_ns)) : -1 - warp;
    const int n0 = s0 - e_loc * Ns;
    House4<real> h;
    real red[kRed] = {0, 0, 0, 0, 0};
    cp_async_wait_all();   // the thread's own staging copies of this tile have landed
    Raw4f w;
    if (active) {
      const float4 *in4 = reinterpret_cast<const float4 *>(s_in) + threadIdx.x;
      auto ld = [&](int k, float v[4]) {
        const float4 t = in4[(size_t)k * (kTileSlots / 4)];
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      };
      ld(0, w.ta); ld(1, w.tm);
      {
        const int4 t = reinterpret_cast<const int4 *>(s_in)[(size_t)2 * (kTileSlots / 4) + threadIdx.x];
        w.sso[0] = t.x; w.sso[1] = t.y; w.sso[2] = t.z; w.sso[3] = t.w;
      }
      ld(3, w.target); ld(4, w.cap);
#pragma unroll
      for (int k = 0; k < 6; ++k) ld(5 + k, w.c[k]);
      w.flags = s_flags[threadIdx.x];
      w.act = ext ? s_act[threadIdx.x] : 0u;
      if constexpr (POLL) {
        if (ext) w.act = act_word_polled(actions, base + s0, w.act, in.act_poll_err);
      }
      if (fast) { const float2 v = s_os[threadIdx.x]; w.od = v.x; w.solar = v.y; }
      else { w.od = nx_od; w.solar = nx_solar; }
    }
    // the thread holds its inputs in registers: on the tile's last step its staging slots are free, the next
    // tile's copies are issued now and have the whole tile to land
    if (!more && nt < g.n_tiles) prefetch(nt, 3);
    if (active) house4_compute_f32<MODE != 0>(pl, p, w, base + s0, min(4, p.N - n0), h, red, pol_keep);
    if (more && active) {   // the next step reads its state from the thread's own staging slots, its small inputs come now
      if (ext) cp_async4(s_act + threadIdx.x, step_actions(st + 1) + base + s0);
      if (fast) cp_async8(s_os + threadIdx.x, &in.sched_rec[(size_t)(st + 1) * p.R + r0 + e_loc].od_prev_f);
      float4 *o4 = reinterpret_cast<float4 *>(s_in) + threadIdx.x;
      o4[0] = make_float4(h.ta[0], h.ta[1], h.ta[2], h.ta[3]);
      o4[kTileSlots / 4] = make_float4(h.tm[0], h.tm[1], h.tm[2], h.tm[3]);
      reinterpret_cast<int4 *>(s_in)[(size_t)2 * (kTileSlots / 4) + threadIdx.x] = make_int4(h.sso[0], h.sso[1], h.sso[2], h.sso[3]);
      s_flags[threadIdx.x] = h.flags;
    }
    clk.mark(kPhHouse);
    // the previous tile's row store must have drained the warp's staging rows before they are rewritten
    // (waited for here, after the house update, not at the top of the tile)
    if (lane == 0 && store_pending) bulk_store_wait_read();
    __syncwarp();
    clk.mark(kPhStore);
    if (MODE == 1 && active) {
      own_rows10(s_tile + (size_t)s0 * 10, h, p, lane);
    } else if (active) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t f = (h.flags >> (8 * j)) & 0xffu;
        const real sso_n = (real)fast_div((uint32_t)h.sso[j], p.fd_dur);            // norm.py:40-43, :79-82
        const bool ok = j < h.valid;
        if (need_msg) {
          const real pmax_n = h.cap[j] * p.hf.inv_cop * p.hf.inv_nrs;
          Msg4<real> m;
          m.dT = ok ? h.ta[j] * 0.2f : 0.f;                                         // norm.py:39
          m.sso_n = ok ? sso_n : 0.f;
          m.p_n = (ok && (f & 1u)) ? pmax_n : 0.f;
          m.pmax_n = ok ? pmax_n : 0.f;
          s_msg[s0 + j] = m;
        }
        if (D > 0) {
          O *row = s_tile + (size_t)(s0 + j) * D;
          if (plain) {
            const float tg = h.target[j] - 20.f;
            put2(row, 0, ok ? (float)(f & 1u) : 0.f, ok ? (float)((f >> 1) & 1u) : 0.f);
            put2(row, 1, ok ? sso_n : 0.f, ok ? 1.f : 0.f);
            put2(row, 3, ok ? p.hf.deadband : 0.f, ok ? (h.ta[j] + tg) * 0.2f : 0.f);
            put2(row, 4, ok ? (h.tm[j] + tg) * 0.2f : 0.f, ok ? tg * 0.2f : 0.f);
            if (!ok) {
              put2(row, 2, 0.f, 0.f);
              for (int q = 5; q < D / 2; ++q) put2(row, q, 0.f, 0.f);
            }
          } else if (ok) {
            EnvBroadcast<real> none{};
            real ratio[4] = {0, 0, 0, 0};
            if (p.st_thermal)
              for (int k = 0; k < 4; ++k) ratio[k] = pl.ratio[k][base + s0 + j];
            obs_own<real>(row, p, f, sso_n, h.ta[j] + (h.target[j] - 20.f), h.tm[j] + (h.target[j] - 20.f),
                          h.target[j] - 20.f, none, ratio, 1);
          } else {
            for (int q = 0; q < D; ++q) row[q] = 0.f;
          }
        }
      }
    }
    if (one_env) {
      // one cluster per tile: plain butterfly, every warp stores one partial
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        real t[kRed];
#pragma unroll
        for (int k = 0; k < kRed; ++k) t[k] = __shfl_xor_sync(0xffffffffu, red[k], o);
        red_combine(red, t);
      }
      if (lane == 0) {
        double *dst = s_wp + (size_t)warp * g.max_segs * kRed;
#pragma unroll
        for (int k = 0; k < kRed; ++k) dst[k] = (double)red[k];
      }
    } else {
      // segmented warp reduction over clusters (lanes of one cluster are contiguous)
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        real t[kRed];
#pragma unroll
        for (int k = 0; k < kRed; ++k) t[k] = __shfl_down_sync(0xffffffffu, red[k], o);
        const int eo = __shfl_down_sync(0xffffffffu, e_loc, o);
        if (lane + o < 32 && eo == e_loc) red_combine(red, t);
      }
      const int e_prev = __shfl_up_sync(0xffffffffu, e_loc, 1);
      const bool head = (lane == 0) || (e_prev != e_loc);
      const int e_first = __shfl_sync(0xffffffffu, e_loc, 0);
      if (head && e_loc >= 0) {
        double *dst = s_wp + ((size_t)warp * g.max_segs + (e_loc - e_first)) * kRed;
#pragma unroll
        for (int k = 0; k < kRed; ++k) dst[k] = (double)red[k];
      }
    }
    clk.mark(kPhRows);
    if (fast && threadIdx.x < E) cp_async_wait_all();  // this tile's records (issued a whole tile ago) are in s_stage
    __syncthreads();
    clk.mark(kPhBarrier);
    // every warp is past the previous tile's phase 3: the other parity of s_stage is free again
    if (fast) {
      if (more) {
        if ((int)threadIdx.x < E) {   // record of the next step; its metrics part is filled by env_stage_store
          const char *src = reinterpret_cast<const char *>(in.sched_rec + (size_t)(st + 1) * p.R + r0 + threadIdx.x);
          char *d = reinterpret_cast<char *>(s_stage_base + (size_t)(parity ^ 1) * g.envs_per_tile + threadIdx.x);
#pragma unroll
          for (int q = 0; q < 5; ++q) cp_async16(d + 16 * q, src + 16 * q);
        }
      } else if (nt < g.n_tiles) {
        fetch_env(nt, parity ^ 1);
      }
    }

    // ---- phase 2 -------------------------------------------------------------------------
    // combine the warp partials of cluster e in warp order (deterministic, identical everywhere)
    auto combine = [&](int e, double a[kRed], bool all) {
      const int w_lo = (e * Ns) >> 7, w_hi = ((e + 1) * Ns - 1) >> 7;
      for (int w = w_lo; w <= w_hi; ++w) {
        const int efst = (int)fast_div((uint32_t)(w << 7), p.fd_ns);  // first cluster seen by warp w
        const double *src = s_wp + ((size_t)w * g.max_segs + (e - efst)) * kRed;
        if (all) red_combine(a, src);
        else a[0] += src[0];
      }
    };
    EnvBroadcast<real> eb{};
    if (fast) {
      // no serial section: every house thread folds the cluster power into the pre-computed
      // broadcast values by itself
      if (one_env) {
        // one cluster per tile: lanes 0..7 fetch one warp partial each, a 3-level butterfly in
        // fixed order gives every lane of every warp the same totals
        double a[3] = {0, 0, 0};
        if (lane < kThreads / 32 && lane * 128 < slots) {
          const double *src = s_wp + (size_t)lane * g.max_segs * kRed;
          a[0] = src[0]; a[1] = src[1]; a[2] = src[2];
        }
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
          a[0] += __shfl_xor_sync(0xffffffffu, a[0], o);
          a[1] += __shfl_xor_sync(0xffffffffu, a[1], o);
          a[2] = fmax(a[2], __shfl_xor_sync(0xffffffffu, a[2], o));
        }
        a[0] = __shfl_sync(0xffffffffu, a[0], 0);
        a[1] = __shfl_sync(0xffffffffu, a[1], 0);
        a[2] = __shfl_sync(0xffffffffu, a[2], 0);
        const SchedRec &c = s_stage[0].rec;
        eb.signal_n = c.signal_n; eb.solar_n = c.solar_n; eb.od_n = c.od_n;
        eb.power_n = (real)(a[0] * p.inv_nrs);
        eb.rew_sig = (real)signal_penalty(p, a[0], c.signal_prev);
        eb.pen_common = (real)a[1];
        eb.pen_max = (real)a[2];
      } else if (active) {
        double a[kRed] = {0, 0, 0, 0, 0};
        combine(e_loc, a, !individual);
        const SchedRec &c = s_stage[e_loc].rec;
        eb.signal_n = c.signal_n; eb.solar_n = c.solar_n; eb.od_n = c.od_n;
        eb.power_n = (real)(a[0] * p.inv_nrs);
        eb.rew_sig = (real)signal_penalty(p, a[0], c.signal_prev);
        eb.pen_common = (real)a[1];
        eb.pen_max = (real)a[2];
      }
    } else if constexpr (MODE == 0) {
      if (threadIdx.x < E) {
        double a[kRed] = {0, 0, 0, 0, 0};
        combine(threadIdx.x, a, true);
        s_env[threadIdx.x] = env_epilogue<real>(pl, p, in, r0 + threadIdx.x, er, a, 0.0);  // injected noise: inline
      }
      __syncthreads();
      if (active) eb = s_env[e_loc];
    }

    // ---- phase 3 -----------------------------------------------------------------------
    if (active) {
      const EnvBroadcast<real> e = eb;
      real rw[4];
      const bool lean_reward = individual;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        rw[j] = lean_reward ? reward_f32_individual(p, h.ta[j], e.rew_sig) : house_reward<real>(p, kc, h.ta[j], h.target[j], e);
        if (j >= h.valid) rw[j] = 0.f;
      }
      st4_hint(pl.reward + base + s0, rw, pol_stream);
      clk.mark(kPhFold);
      if (MODE == 1) {
        own_rows10_patch(s_tile + (size_t)s0 * 10, h.valid, lane, e.power_n, e.signal_n);
      } else if (D > 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j < h.valid) {
            O *row = s_tile + (size_t)(s0 + j) * D;
            if (plain) {
              put2(row, 2, e.power_n, e.signal_n);
              if (need_msg) {
                RowNbrs<SMP> nbr(p, r0 + e_loc, n0 + j, rows_draw(in, st));
                for (int k = 0; k < p.nb_comm; ++k) {
                  const int nb = nbr(p, pl.comm_table, r0 + e_loc, n0 + j, k);
                  const float4 mk = *reinterpret_cast<const float4 *>(&s_msg[e_loc * Ns + nb]);
                  put2(row, 5 + 2 * k, mk.x, mk.y);
                  put2(row, 6 + 2 * k, mk.z, mk.w);
                }
              }
              continue;
            }
            int q = obs_own<real>(row, p, 0u, 0.f, 0.f, 0.f, 0.f, e, nullptr, 2);
            if (need_msg) {
              RowNbrs<SMP> nbr(p, r0 + e_loc, n0 + j, rows_draw(in, st));
              for (int k = 0; k < p.nb_comm; ++k) {
                const int nb = nbr(p, pl.comm_table, r0 + e_loc, n0 + j, k);
                const Msg4<real> mk = s_msg[e_loc * Ns + nb];
                row[q++] = mk.dT; row[q++] = mk.sso_n; row[q++] = mk.p_n; row[q++] = mk.pmax_n;
                if (p.msg_thermal)
                  for (int t = 0; t < 4; ++t) row[q++] = (real)pl.ratio[t][base + e_loc * Ns + nb];
                if (p.msg_hvac) { row[q++] = (real)p.cop; row[q++] = (real)p.latent; row[q++] = (real)p.dcap; }
              }
            }
          }
        }
      }
    }
    if (D > 0) {
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0 && w0 < slots) {
        const int nrows = min(128, slots - w0);
        // the tile's previous step stored the same rows: its global writes must have landed, or they could
        // overwrite this step's (waited for here, a whole step after that store was issued)
        if (st > 0) bulk_store_wait_all();
        bulk_store_s2g_hint(pl.template rows<O>() + (base + w0) * D, s_tile + (size_t)w0 * D, (uint32_t)((size_t)nrows * D * sizeof(O)),
                            pol_stream);
        store_pending = true;
      }
    }
    clk.mark(kPhStore);
    // off the critical path: env planes + running metrics of cluster threadIdx.x
    if (threadIdx.x < E && fast) {
      double a[kRed] = {0, 0, 0, 0, 0};
      combine(threadIdx.x, a, true);
      double *m_next = more ? (s_stage_base + (size_t)(parity ^ 1) * g.envs_per_tile + threadIdx.x)->m : nullptr;
      env_stage_store<real>(pl, p, r0 + threadIdx.x, s_stage[threadIdx.x], a, in.host_env, m_next);
    }
    clk.mark(kPhEpilogue);
    clk.step();
  }
  // shared memory must outlive the reads of the last row store; its global writes complete with the grid
  if (lane == 0 && store_pending) bulk_store_wait_read();
  clk.flush();
}

// ------------------------------------------------------------------------------------------
// Fused path, fp32, wide rows (hand-engineered layout with neighbour messages, D = 10 + 4 c):
// the tile's rows (1000 x 200 B for BASELINE config 3) do not fit a staging buffer, so each warp
// assembles the rows of its own 128 slots 32 at a time -- lane l builds row 128 w + 32 g + l from
// the own-state / message records in shared memory -- and ships every 32-row group (6.4 KB
// contiguous) with one TMA bulk store.  Inputs come through 128-bit global loads.  Two CTA barriers
// per tile (message records are read across warps; the power fold-in runs on E threads).
// Conditions (checked by the host): plain columns, external actions, individual_L2, schedule.
// ------------------------------------------------------------------------------------------
DRSIM_D void raw_load_f32(const Planes<float> &pl, const StepIn &in, size_t off, int r, Raw4f &w) {
  load4(pl.t_air + off, w.ta);
  load4(pl.t_mass + off, w.tm);
  load4i(pl.sso + off, w.sso);
  w.flags = load4b(pl.flags + off);
  load4_ro(pl.target + off, w.target);
  load4_ro(pl.cap + off, w.cap);
#pragma unroll
  for (int k = 0; k < 6; ++k) load4_ro(pl.coef[k] + off, w.c[k]);
  w.act = load4b((in.actions ? in.actions : pl.actions) + off);
  // fp32 house-update inputs straight from the step's record (no fp64 conversion)
  const float2 v = *reinterpret_cast<const float2 *>(&in.sched_rec[r].od_prev_f);
  w.od = v.x; w.solar = v.y;
}

constexpr int kRowGroup = 16;  // rows per warp-level TMA store in k_fused_rows (two lanes assemble one row)

// STAGED = inputs prefetched one tile ahead into thread-private shared-memory slots (needs 44 B of
// shared memory per house slot); false = 128-bit register loads at the top of the tile (large clusters)
template <bool STAGED, bool POLL = false, typename O = float, bool SMP = false>
__global__ void __launch_bounds__(kThreads, 2)
k_fused_rows(Planes<float> pl, SimParams p, StepIn in, FusedGeom g) {
  typedef float real;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float4 *s_msg_base = reinterpret_cast<float4 *>(smem_raw + g.off_msg);   // [2][slots] (dT, sso_n, p_n, pmax_n)
  // own records are double-buffered like the messages: any warp assembles any row group, so a warp
  // already in the next tile's phase 1 must not overwrite records a slower warp still reads
  float4 *s_own_base = reinterpret_cast<float4 *>(smem_raw + g.off_own);   // [2][slots] (ta_n, tm_n, tg_n, flags)
  EnvBroadcast<real> *s_env_base = reinterpret_cast<EnvBroadcast<real> *>(smem_raw + g.off_env);
  double *s_wp_base = reinterpret_cast<double *>(smem_raw + g.off_wp);
  double *s_sold_base = reinterpret_cast<double *>(smem_raw + g.off_sold);
  O *s_stage = reinterpret_cast<O *>(smem_raw + g.off_tile);         // [warps][kRowGroup][D]
  EnvStage *s_rec_base = reinterpret_cast<EnvStage *>(smem_raw + g.off_stage);  // [2][E] schedule record + metrics

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Ns = p.Ns, D = p.obs_dim, nbc = p.nb_comm;
  const int tile_slots = g.envs_per_tile * Ns;
  const int s0 = threadIdx.x * kHousesPerThread;
  const int w0 = warp * 128;
  O *stage = s_stage + (size_t)warp * kRowGroup * D;
  bool store_pending = false;
  int parity = 0;

  // schedule record + running metrics of tile t's clusters -> shared memory (threads e < E, cp.async)
  auto fetch_env = [&](int t, int st, int par) {
    const int tr0 = t * g.envs_per_tile;
    if ((int)threadIdx.x < min(g.envs_per_tile, p.R - tr0))
      env_stage_fetch(s_rec_base + (size_t)par * g.envs_per_tile + threadIdx.x, in.sched_rec + (size_t)st * p.R, pl.metrics,
                      tr0 + threadIdx.x);
  };
  // thread-private input staging (see k_fused_tma): the 16 bytes a thread consumes of each of the
  // eleven 32-bit planes, its flags / action words and its cluster's two fp32 scalars are copied into
  // the thread's own slots with cp.async one tile ahead; `part` 1 = static planes (before pdl_wait)
  float *s_in = reinterpret_cast<float *>(smem_raw + g.off_in);   // [11][in_stride] + small inputs
  const int in_stride = g.in_stride;
  uint32_t *s_flags = reinterpret_cast<uint32_t *>(s_in + (size_t)11 * in_stride);
  uint32_t *s_act = s_flags + kThreads;
  float2 *s_os = reinterpret_cast<float2 *>(s_act + kThreads);
  const uint8_t *actions = in.actions ? in.actions : pl.actions;
  // (plain cp.async here: with a run-time plane stride, ptxas 12.9 encodes the L2::cache_hint form of
  // LDGSTS with a uniform-register shared offset that the B200 rejects as an illegal instruction)
  // in-kernel step loop over an action tape (StepIn::stream_steps, see k_fused_tma; STAGED only)
  const int n_stream = (STAGED && in.stream_steps > 1) ? in.stream_steps : 1;
  auto step_actions = [&](int st) -> const uint8_t * {
    if (n_stream == 1 || !in.actions) return actions;
    const int j = in.tape_first + st;
    return in.actions + (size_t)(in.tape_planes > 0 ? j % in.tape_planes : j) * in.tape_stride;
  };
  auto prefetch = [&](int t, int st, int part) {
    if constexpr (!STAGED) return;
    const int tr0 = t * g.envs_per_tile;
    const int tslots = min(g.envs_per_tile, p.R - tr0) * Ns;
    if (s0 >= tslots) return;
    const size_t o = (size_t)tr0 * Ns + s0;
    float *d = s_in + s0;
    if (part & 1) {
      cp_async16(d + 3 * in_stride, pl.target + o);
      cp_async16(d + 4 * in_stride, pl.cap + o);
#pragma unroll
      for (int c = 0; c < 6; ++c) cp_async16(d + (5 + c) * in_stride, pl.coef[c] + o);
    }
    if (part & 2) {
      cp_async16(d, pl.t_air + o);
      cp_async16(d + in_stride, pl.t_mass + o);
      cp_async16(d + 2 * in_stride, pl.sso + o);
      cp_async4(s_flags + threadIdx.x, pl.flags + o);
      cp_async4(s_act + threadIdx.x, step_actions(st) + o);
      cp_async8(s_os + threadIdx.x, &in.sched_rec[(size_t)st * p.R + tr0 + (int)fast_div((uint32_t)s0, p.fd_ns)].od_prev_f);
    }
  };
  pdl_trigger();
  if ((int)blockIdx.x < g.n_tiles) prefetch(blockIdx.x, 0, 1);
  pdl_wait();
  if ((int)blockIdx.x < g.n_tiles) {
    prefetch(blockIdx.x, 0, 2);
    fetch_env(blockIdx.x, 0, 0);
  }

  for (int st = 0; st < n_stream; ++st)
  for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, parity ^= 1) {
    // the item after this one: the CTA's next tile of this step, or its first tile of the next step of the stream
    int nt = tile + gridDim.x, nst = st;
    if (nt >= g.n_tiles && st + 1 < n_stream) { nt = blockIdx.x; nst = st + 1; }
    const int r0 = tile * g.envs_per_tile;
    const int E = min(g.envs_per_tile, p.R - r0);
    const int slots = E * Ns;
    const size_t base = (size_t)r0 * Ns;
    float4 *s_msg = s_msg_base + (size_t)parity * tile_slots;
    float4 *s_own = s_own_base + (size_t)parity * tile_slots;
    EnvBroadcast<real> *s_env = s_env_base + (size_t)parity * g.envs_per_tile;
    double *s_wp = s_wp_base + (size_t)parity * (kThreads / 32) * g.max_segs * kRed;
    double *s_sold = s_sold_base + (size_t)parity * g.envs_per_tile;

    const EnvStage *s_rec = s_rec_base + (size_t)parity * g.envs_per_tile;

    // ---- phase 1: house update, own / message records ------------------------------------
    const bool active = s0 < slots;
    const int e_loc = active ? (int)fast_div((uint32_t)s0, p.fd_ns) : -1 - warp;
    const int n0 = s0 - e_loc * Ns;
    House4<real> h;
    real red[kRed] = {0, 0, 0, 0, 0};
    real pen_r[4] = {0, 0, 0, 0};
    cp_async_wait_all();   // the thread's own staging copies of this tile have landed
    Raw4f w;
    if constexpr (!STAGED) {
      if (active) raw_load_f32(pl, in, base + s0, r0 + e_loc, w);
    } else if (active) {
      const float4 *in4 = reinterpret_cast<const float4 *>(s_in + s0);
      auto ld = [&](int q, float v[4]) {
        const float4 t = in4[(size_t)q * (in_stride / 4)];
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      };
      ld(0, w.ta); ld(1, w.tm);
      {
        const int4 t = reinterpret_cast<const int4 *>(s_in + s0)[(size_t)2 * (in_stride / 4)];
        w.sso[0] = t.x; w.sso[1] = t.y; w.sso[2] = t.z; w.sso[3] = t.w;
      }
      ld(3, w.target); ld(4, w.cap);
#pragma unroll
      for (int q = 0; q < 6; ++q) ld(5 + q, w.c[q]);
      w.flags = s_flags[threadIdx.x];
      w.act = s_act[threadIdx.x];
      if constexpr (POLL) w.act = act_word_polled(actions, base + s0, w.act, in.act_poll_err);
      const float2 v = s_os[threadIdx.x];
      w.od = v.x; w.solar = v.y;
    }
    // the thread holds its inputs in registers: the next tile's copies fly during this tile
    if (nt < g.n_tiles) prefetch(nt, nst, 3);
    if (active) {
      house4_compute_f32<true>(pl, p, w, base + s0, min(4, p.N - n0), h, red);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t f = (h.flags >> (8 * j)) & 0xffu;
        const bool ok = j < h.valid;
        const real sso_n = (real)fast_div((uint32_t)h.sso[j], p.fd_dur);
        const real pmax_n = h.cap[j] * p.hf.inv_cop * p.hf.inv_nrs;
        const float tg = h.target[j] - 20.f;
        s_msg[s0 + j] = ok ? make_float4(h.ta[j] * 0.2f, sso_n, (f & 1u) ? pmax_n : 0.f, pmax_n) : make_float4(0, 0, 0, 0);
        s_own[s0 + j] = make_float4((h.ta[j] + tg) * 0.2f, (h.tm[j] + tg) * 0.2f, tg * 0.2f, (float)f);
        const float d = fmaxf(fabsf(h.ta[j]) - p.hf.half_db, 0.f);
        pen_r[j] = ok ? p.hf.rew_scale * d * d : 0.f;
      }
    }
    // segmented warp reduction over clusters
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      real t[kRed];
#pragma unroll
      for (int k = 0; k < kRed; ++k) t[k] = __shfl_down_sync(0xffffffffu, red[k], o);
      const int eo = __shfl_down_sync(0xffffffffu, e_loc, o);
      if (lane + o < 32 && eo == e_loc) red_combine(red, t);
    }
    const int e_prev = __shfl_up_sync(0xffffffffu, e_loc, 1);
    const bool head = (lane == 0) || (e_prev != e_loc);
    const int e_first = __shfl_sync(0xffffffffu, e_loc, 0);
    if (head && e_loc >= 0) {
      double *dst = s_wp + ((size_t)warp * g.max_segs + (e_loc - e_first)) * kRed;
#pragma unroll
      for (int k = 0; k < kRed; ++k) dst[k] = (double)red[k];
    }
    if (threadIdx.x < E) cp_async_wait_all();  // this tile's records (issued a whole tile ago) are in s_rec
    __syncthreads();
    // every warp is past the previous tile: the other parity of s_rec is free again
    if (nt < g.n_tiles) fetch_env(nt, nst, parity ^ 1);

    // ---- phase 2: fold the cluster power in (E threads, a few dozen instructions) ----------
    double a[kRed] = {0, 0, 0, 0, 0};
    if (threadIdx.x < E) {
      const int e = threadIdx.x;
      const int w_lo = (e * Ns) >> 7, w_hi = ((e + 1) * Ns - 1) >> 7;
      for (int w = w_lo; w <= w_hi; ++w) {
        const int efst = (int)fast_div((uint32_t)(w << 7), p.fd_ns);
        red_combine(a, s_wp + ((size_t)w * g.max_segs + (e - efst)) * kRed);
      }
      const SchedRec &c = s_rec[e].rec;
      s_env[e].signal_n = c.signal_n;
      s_env[e].power_n = (real)(a[0] * p.inv_nrs);
      s_env[e].rew_sig = (real)signal_penalty(p, a[0], c.signal_prev);
    }
    __syncthreads();

    // ---- phase 3: rewards, then the warp's rows 32 at a time -------------------------------
    if (active) {
      const real rs = s_env[e_loc].rew_sig;
      real rw[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) rw[j] = j < h.valid ? -(pen_r[j] + rs) : 0.f;
      store4(pl.reward + base + s0, rw);
    }
    // the tile's 32-row groups are dealt round-robin to ALL warps (own / message records of every slot
    // are in shared memory), so warps whose house slots lie beyond the tile's end assemble rows too
    const int n_groups = (slots + kRowGroup - 1) / kRowGroup;
    const bool ring = p.comm_mode == DRSIM_COMM_RING;
    const int nb_lo = nbc / 2, nb_hi = nbc - nb_lo;
    for (int gidx = warp; gidx < n_groups; gidx += kThreads / 32) {
      const int gs = gidx * kRowGroup;  // first slot of the group
      if (lane == 0 && store_pending) bulk_store_wait_read();
      __syncwarp();
      const int row = lane >> 1, half = lane & 1;   // two lanes per row: own part + first run | second run
      const int s = gs + row;
      if (s < slots) {
        const int e = (int)fast_div((uint32_t)s, p.fd_ns), n = s - e * Ns;
        O *orow = stage + (size_t)row * D;
        if (n < p.N) {
          if (half == 0) {
            const float4 o = s_own[s];
            const float4 m = s_msg[s];
            const EnvBroadcast<real> ev = s_env[e];
            const uint32_t f = (uint32_t)o.w;
            put2(orow, 0, (float)(f & 1u), (float)((f >> 1) & 1u));
            put2(orow, 1, m.y, 1.f);
            put2(orow, 2, ev.power_n, ev.signal_n);
            put2(orow, 3, p.hf.deadband, o.x);
            put2(orow, 4, o.y, o.z);
          }
          const float4 *mb = s_msg + e * Ns;
          const int k0 = half ? nb_lo : 0, k1 = half ? nbc : nb_lo;
          if (ring && n >= nb_lo && n + nb_hi < p.N) {
            // ring neighbours that do not wrap are two contiguous runs of message records
            // (agent_communication_builder.py:74-84): n - lo .. n - 1 and n + 1 .. n + hi
            const float4 *src = mb + (half ? n + 1 - nb_lo : n - nb_lo);
            for (int q = k0; q < k1; ++q) {
              const float4 mk = src[q];
              put2(orow, 5 + 2 * q, mk.x, mk.y);
              put2(orow, 6 + 2 * q, mk.z, mk.w);
            }
          } else {
            RowNbrs<SMP> nbr(p, r0 + e, n, rows_draw(in, st));   // (the second half runs the draw through the first)
            for (int q = k0; q < k1; ++q) {
              const float4 mk = mb[nbr(p, pl.comm_table, r0 + e, n, q)];
              put2(orow, 5 + 2 * q, mk.x, mk.y);
              put2(orow, 6 + 2 * q, mk.z, mk.w);
            }
          }
        } else {
          for (int q = half; q < D / 2; q += 2) put2(orow, q, 0.f, 0.f);
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        const int nrows = min(kRowGroup, slots - gs);
        bulk_store_s2g(pl.template rows<O>() + (base + gs) * D, stage, (uint32_t)((size_t)nrows * D * sizeof(O)));
        store_pending = true;
      }
    }
    if (threadIdx.x < E) env_stage_store<real>(pl, p, r0 + threadIdx.x, s_rec[threadIdx.x], a, in.host_env);
  }
  if (lane == 0 && store_pending) bulk_store_wait_read();
}

// ------------------------------------------------------------------------------------------
// Small clusters, latency-oriented (BASELINE config 1: the default 10-house cluster).  The tile
// kernels give every thread four houses, so a 10-house cluster runs on three threads and one step
// is a ~2,000-instruction dependent chain (8 us).  Here a WARP owns a cluster of at most 32 houses,
// one house per lane: the lock-out state machine and the thermal update of house4_compute_f32 per
// lane, the five cluster sums by shuffle butterflies, the power fold-in / reward / row of every
// house by its own lane, neighbour messages by shuffles instead of shared memory.  The state lives
// in registers across the steps of one launch (StepIn::stream_steps: on-device policy or action
// tape) and goes back to the planes after every step like everything else the
// step produces.  Conditions (checked by the host): fp32, scheduled env path, plain columns.
// ------------------------------------------------------------------------------------------
constexpr int kSmallWarps = 4;   // clusters per CTA

template <typename O = float, bool SMP = false>
__global__ void __launch_bounds__(kSmallWarps * 32) k_small(Planes<float> pl, SimParams p, StepIn in) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int r = (int)blockIdx.x * kSmallWarps + warp;
  pdl_trigger();
  if (r >= p.R) return;
  const int Ns = p.Ns, N = p.N, D = p.obs_dim, nbc = p.nb_comm;
  const KC<float> kc(p);
  const bool slot = lane < Ns, ok = lane < N;          // plane slot / real house
  const size_t o = (size_t)r * Ns + (slot ? lane : 0);
  const int policy = p.policy;
  const bool ext = policy == DRSIM_POLICY_EXTERNAL || policy == DRSIM_POLICY_GREEDY_MYOPIC;
  const bool individual = p.penalty_mode == DRSIM_PEN_INDIVIDUAL_L2;
  const bool need_msg = p.obs_layout == DRSIM_OBS_HAND_ENGINEERED && nbc > 0;
  const int dt = p.dt, dur = p.lockout_duration;
  const float half_db = p.hf.half_db;
  // launch-invariant planes before the dependency wait, what the step before wrote after it
  // (padding slots of the plane stride are stepped like houses with zero planes, exactly as the tile kernels do)
  float tg = 0.f, cap = 0.f, c[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (slot) {
    tg = __ldg(pl.target + o);
    cap = __ldg(pl.cap + o);
#pragma unroll
    for (int k = 0; k < 6; ++k) c[k] = __ldg(pl.coef[k] + o);
  }
  pdl_wait();
  float ta = 0.f, tm = 0.f;
  int sso = 0;
  uint32_t f = 0;
  if (slot) { ta = pl.t_air[o]; tm = pl.t_mass[o]; sso = pl.sso[o]; f = pl.flags[o]; }
  double m[DRSIM_N_METRICS];
#pragma unroll
  for (int q = 0; q < DRSIM_N_METRICS; ++q) m[q] = pl.metrics[(size_t)r * DRSIM_N_METRICS + q];
  const int n_steps = max(1, in.stream_steps);
  const float pmax_n = cap * p.hf.inv_cop * p.hf.inv_nrs;
  const float tg20 = tg - 20.f;

  for (int k = 0; k < n_steps; ++k) {
    const SchedRec *rec = in.sched_rec + (size_t)k * p.R + r;
    const float od = __ldg(&rec->od_prev_f), solar = __ldg(&rec->solar_f);
    // ---- house update: the expressions of house4_compute_f32 for one house ----
    const bool on = f & 1u;
    bool a = false;
    if (ext) {
      const uint8_t *acts = in.actions ? in.actions : pl.actions;
      if (in.actions && in.stream_steps > 1) {
        const int j = in.tape_first + k;
        acts = in.actions + (size_t)(in.tape_planes > 0 ? j % in.tape_planes : j) * in.tape_stride;
      }
      a = slot && acts[o] != 0;
    } else if (policy == DRSIM_POLICY_DEADBAND_BANGBANG) a = ta < -half_db ? false : (ta > half_db ? true : on);
    else if (policy == DRSIM_POLICY_BANGBANG) a = ta > 0.f;
    else if (policy == DRSIM_POLICY_ALWAYS_ON) a = true;
    sso = sso + (on ? 0 : dt);
    bool lock = !on && sso < dur;
    const bool on_n = !lock && a;
    sso = on_n ? 0 : sso;
    lock = lock || (!on_n && sso + dt < dur);
    f = (on_n ? 1u : 0u) | (lock ? 2u : 0u);
    const float Qa = (on_n ? cap * p.hf.neg_inv_opl : 0.f) + solar;
    const float odr = od - tg;
    const float ia = fmaf(c[2], Qa, fmaf(c[1], odr - ta, c[0] * (tm - ta)));
    const float im = fmaf(c[5], Qa, fmaf(c[4], odr - tm, c[3] * (ta - tm)));
    ta = ta + ia;
    tm = tm + im;
    const float mk = ok ? 1.f : 0.f;
    const float dd = fmaxf(fabsf(ta) - half_db, 0.f);
    const float pen = dd * dd * mk;
    float red[kRed] = {fmaf(on_n ? mk : 0.f, cap * p.hf.inv_cop, 0.f), fmaf(pen, p.hf.inv_n, 0.f), pen, mk * ta, (ta * mk) * ta};
    // ---- the five cluster sums: every lane ends up with the totals ----
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
      float t[kRed];
#pragma unroll
      for (int q = 0; q < kRed; ++q) t[q] = __shfl_xor_sync(0xffffffffu, red[q], s);
      red_combine(red, t);
    }
    double rd[kRed];
#pragma unroll
    for (int q = 0; q < kRed; ++q) rd[q] = (double)red[q];
    // ---- env values every house needs (the fold-in of the fused kernels) ----
    EnvBroadcast<float> e;
    e.signal_n = __ldg(&rec->signal_n); e.solar_n = __ldg(&rec->solar_n); e.od_n = __ldg(&rec->od_n);
    e.power_n = (float)(rd[0] * p.inv_nrs);
    e.rew_sig = (float)signal_penalty(p, rd[0], __ldg(&rec->signal_prev));
    e.pen_common = (float)rd[1];
    e.pen_max = (float)rd[2];
    // ---- outputs of the step: state, reward, observation row ----
    if (slot) {
      pl.t_air[o] = ta; pl.t_mass[o] = tm; pl.sso[o] = sso; pl.flags[o] = (uint8_t)f;
      pl.reward[o] = ok ? (individual ? reward_f32_individual(p, ta, e.rew_sig) : house_reward<float>(p, kc, ta, tg, e)) : 0.f;
    }
    const float sso_n = (float)fast_div((uint32_t)sso, p.fd_dur);                     // norm.py:40-43, :79-82
    // this house's message record (building.py:102-139 through norm.py:31-60), read by its neighbours through shuffles
    const float m0 = ok ? ta * 0.2f : 0.f, m1 = ok ? sso_n : 0.f, m2 = (ok && (f & 1u)) ? pmax_n : 0.f, m3 = ok ? pmax_n : 0.f;
    if (D > 0) {
      O *row = pl.template rows<O>() + o * D;
      if (slot) {
        put2(row, 0, ok ? (float)(f & 1u) : 0.f, ok ? (float)((f >> 1) & 1u) : 0.f);
        put2(row, 1, ok ? sso_n : 0.f, ok ? 1.f : 0.f);
        put2(row, 2, ok ? e.power_n : 0.f, ok ? e.signal_n : 0.f);
        put2(row, 3, ok ? p.hf.deadband : 0.f, ok ? (ta + tg20) * 0.2f : 0.f);
        put2(row, 4, ok ? (tm + tg20) * 0.2f : 0.f, ok ? tg20 * 0.2f : 0.f);
      }
      if (need_msg) {
        RowNbrs<SMP> nbr(p, r, lane, rows_draw(in, k));
        for (int q = 0; q < nbc; ++q) {      // (every lane takes part in the shuffles)
          const int nb = ok ? nbr(p, pl.comm_table, r, lane, q) : 0;
          const float v0 = __shfl_sync(0xffffffffu, m0, nb), v1 = __shfl_sync(0xffffffffu, m1, nb),
                      v2 = __shfl_sync(0xffffffffu, m2, nb), v3 = __shfl_sync(0xffffffffu, m3, nb);
          if (slot) {
            put2(row, 5 + 2 * q, ok ? v0 : 0.f, ok ? v1 : 0.f);
            put2(row, 6 + 2 * q, ok ? v2 : 0.f, ok ? v3 : 0.f);
          }
        }
      } else if (slot && !ok) {
        for (int q = 5; q < D / 2; ++q) put2(row, q, 0.f, 0.f);
      }
    }
    // ---- env planes + running metrics (one lane; the staged record of the fused kernels, built in registers) ----
    if (lane == 0) {
      EnvStage st;
      st.rec = *rec;
#pragma unroll
      for (int q = 0; q < DRSIM_N_METRICS; ++q) st.m[q] = m[q];
      env_stage_store<float>(pl, p, r, st, rd, in.host_env, m);
    }
  }
}

// host snapshot of the dict API (drsim_snapshot): dense [R][N] arrays + [R][kSnapEnv] env scalars in mapped pinned memory
struct SnapPtrs {
  double *t_air, *t_mass, *reward;   // [R][N]
  int32_t *sso;                      // [R][N]
  uint8_t *on, *lockout;             // [R][N]
  double *env;                       // [R][kSnapEnv]
};
constexpr int kSnapEnv = 8;   // od_temp, signal, power, solar, base_power, epoch, t_since_interp, max_power

// The same mapping for the steps k_small does not take: the fp64 build (the drop-in `Environment` replays the
// reference's kelvin formula in fp64 and injects its noise per step) with every observation / message option --
// one house per lane through the helpers of house4_step (hvac.py:43-64, building.py:141-222), butterfly sums in
// `real`, the scheduled or the inline env epilogue on lane 0 (environment.py:87-106), rows written by their own
// lane with obs_own (utils/norm.py:71-218).  One step per launch.  A 10-house cluster took 35 us on the fp64
// tile kernel (three active threads, a serial fp64 epilogue between two CTA barriers).
// `snap` / `snap_obs` (optional, mapped pinned host memory): the host snapshot of drsim_step_host_snapshot is written
// by the same lanes -- no second kernel and no D2H copy behind the step, one synchronisation for the whole call.
template <typename real, bool SMP = false>
__global__ void __launch_bounds__(kSmallWarps * 32) k_small_gen(Planes<real> pl, SimParams p, StepIn in, SnapPtrs snap, real *snap_obs) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int r = (int)blockIdx.x * kSmallWarps + warp;
  pdl_trigger();
  if (r >= p.R) return;
  constexpr int NC = NCoef<real>::n;
  const int Ns = p.Ns, N = p.N, D = p.obs_dim, nbc = p.nb_comm;
  const KC<real> kc(p);
  const bool slot = lane < Ns, ok = lane < N;
  const size_t rb = (size_t)r * Ns, o = rb + (slot ? lane : 0);
  const bool ext = p.policy == DRSIM_POLICY_EXTERNAL || p.policy == DRSIM_POLICY_GREEDY_MYOPIC;
  const bool need_msg = p.obs_layout == DRSIM_OBS_HAND_ENGINEERED && nbc > 0;
  real tg = 0, cap = 0, c[NC];
#pragma unroll
  for (int k = 0; k < NC; ++k) c[k] = 0;
  if (ok) {
    tg = __ldg(pl.target + o);
    cap = __ldg(pl.cap + o);
#pragma unroll
    for (int k = 0; k < NC; ++k) c[k] = __ldg(pl.coef[k] + o);
  }
  pdl_wait();
  EnvRegs er{};
  if (lane == 0) er = env_load(pl, in, r);
  const real od_prev = (real)pl.od_temp[r], solar = (real)pl.solar_next[r];
  real ta = 0, tm = 0;
  int sso = 0;
  uint32_t f = 0;
  real red[kRed] = {0, 0, 0, 0, 0};
  if (ok) {   // one house of house4_step (padding slots are not stepped on this path)
    ta = pl.t_air[o]; tm = pl.t_mass[o]; sso = pl.sso[o]; f = pl.flags[o];
    const bool extv = ext && (in.actions ? in.actions : pl.actions)[o] != 0;
    const bool a = Rep<real>::act(p.policy, ta, tg, kc.db, f & 1u, extv);
    hvac_fsm(f, sso, a, p.dt, p.lockout_duration);
    const real q = (f & 1u) ? hvac_heat(cap, kc.one_plus_latent, kc.neg_inv_opl) : (real)0;
    thermal_step(ta, tm, c, Rep<real>::od_in(od_prev, tg), q + solar);
    if (f & 1u) red[0] = qdiv(cap, kc.cop, kc.inv_cop);
    const real pen = Rep<real>::pen(tg, kc.db, ta);
    red[1] = qdiv(pen, kc.n_glob, kc.inv_n);
    red[2] = pen;
    const real dT = Rep<real>::dev(ta, tg);
    red[3] = dT;
    red[4] = dT * dT;
    pl.t_air[o] = ta; pl.t_mass[o] = tm; pl.sso[o] = sso; pl.flags[o] = (uint8_t)f;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    real t[kRed];
#pragma unroll
    for (int q = 0; q < kRed; ++q) t[q] = __shfl_xor_sync(0xffffffffu, red[q], s);
    red_combine(red, t);
  }
  double a[kRed];
#pragma unroll
  for (int q = 0; q < kRed; ++q) a[q] = (double)red[q];
  // env epilogue on lane 0, its broadcast values to every lane
  EnvBroadcast<real> e{};
  EnvFast ef{};
  const bool fast = in.sched_od != nullptr;
  if (lane == 0) e = fast ? env_fast_compute<real>(p, er, a, ef) : env_epilogue<real>(pl, p, in, r, er, a, 0.0);
  e.power_n = __shfl_sync(0xffffffffu, e.power_n, 0); e.signal_n = __shfl_sync(0xffffffffu, e.signal_n, 0);
  e.solar_n = __shfl_sync(0xffffffffu, e.solar_n, 0); e.od_n = __shfl_sync(0xffffffffu, e.od_n, 0);
  e.rew_sig = __shfl_sync(0xffffffffu, e.rew_sig, 0); e.pen_common = __shfl_sync(0xffffffffu, e.pen_common, 0);
  e.pen_max = __shfl_sync(0xffffffffu, e.pen_max, 0);
  if (slot) pl.reward[o] = ok ? house_reward<real>(p, kc, ta, tg, e) : (real)0;
  if (D > 0) {
    const real sso_n = (real)fast_div((uint32_t)sso, p.fd_dur);                     // norm.py:40-43, :79-82
    const real pmax_n = qdiv(qdiv(cap, kc.cop, kc.inv_cop), kc.nrs, kc.inv_nrs);
    // this house's message record (building.py:102-139 through norm.py:31-60): its neighbours read it through shuffles
    const real m0 = ok ? div5(Rep<real>::dev(ta, tg)) : (real)0, m1 = ok ? sso_n : (real)0,
               m2 = (ok && (f & 1u)) ? pmax_n : (real)0, m3 = ok ? pmax_n : (real)0;
    real *row = pl.template rows<real>() + o * D;
    int q = 0;
    if (ok) {
      real ratio[4] = {0, 0, 0, 0};
      if (p.st_thermal)
        for (int k = 0; k < 4; ++k) ratio[k] = pl.ratio[k][o];
      q = obs_own<real>(row, p, f, sso_n, Rep<real>::minus20(ta, tg), Rep<real>::minus20(tm, tg), tg - (real)20, e, ratio, 3);
    } else if (slot) {
      for (int k = 0; k < D; ++k) row[k] = (real)0;
    }
    if (need_msg) {
      RowNbrs<SMP> nbr(p, r, lane, rows_draw(in));
      for (int k = 0; k < nbc; ++k) {      // (every lane takes part in the shuffles)
        const int nb = ok ? nbr(p, pl.comm_table, r, lane, k) : 0;
        const real v0 = __shfl_sync(0xffffffffu, m0, nb), v1 = __shfl_sync(0xffffffffu, m1, nb),
                   v2 = __shfl_sync(0xffffffffu, m2, nb), v3 = __shfl_sync(0xffffffffu, m3, nb);
        if (ok) {
          row[q++] = v0; row[q++] = v1; row[q++] = v2; row[q++] = v3;
          if (p.msg_thermal)
            for (int t = 0; t < 4; ++t) row[q++] = (real)pl.ratio[t][rb + nb];
          if (p.msg_hvac) { row[q++] = (real)p.cop; row[q++] = (real)p.latent; row[q++] = (real)p.dcap; }
        }
      }
    }
  }
  if (lane == 0 && fast) env_fast_store<real>(pl, p, r, er, ef, a);   // env planes + running metrics, off the other lanes' path
  if (snap.t_air) {   // the arrays of k_snapshot, from registers (fp32 planes hold deviations from the set-point)
    if (ok) {
      const size_t i = (size_t)r * N + lane;
      const double shift = sizeof(real) == 4 ? (double)tg : 0.0;
      snap.t_air[i] = (double)ta + shift;
      snap.t_mass[i] = (double)tm + shift;
      snap.reward[i] = (double)pl.reward[o];
      snap.sso[i] = sso;
      snap.on[i] = (uint8_t)(f & 1u);
      snap.lockout[i] = (uint8_t)((f >> 1) & 1u);
      if (snap_obs && D > 0) {
        const real *src = pl.template rows<real>() + o * D;
        real *dst = snap_obs + i * D;
        for (int k = 0; k < D; ++k) dst[k] = src[k];
      }
    }
    if (lane == 0) {   // (the env planes were just written by this lane)
      double *ev = snap.env + (size_t)r * kSnapEnv;
      ev[0] = pl.od_temp[r]; ev[1] = pl.signal[r]; ev[2] = pl.power[r]; ev[3] = pl.solar_cur[r];
      ev[4] = pl.base_power[r]; ev[5] = (double)pl.epoch[r]; ev[6] = (double)pl.t_since_interp[r]; ev[7] = pl.max_power[r];
    }
  }
}

// ------------------------------------------------------------------------------------------
// Reset on the device (SURVEY 8a-15): property noise + initial state from Philox streams keyed by
// (global replica, global house, draw) and (global replica, draw); the update coefficients are
// derived in fp64 right here.  One thread per house; thread n == 0 of a replica also writes the env
// scalars.  Distributions follow building.py:224-267 / hvac.py:36-41,66-70 / environment.py:176-194.
// ------------------------------------------------------------------------------------------
struct ResetArgs {
  uint64_t seed;
  int mode, randomize_date, quirk_ua, n_caps;
  int64_t start_epoch;
  double init_air, init_mass, std_target, f_lo, f_hi;
  double caps[8];
};

template <typename real>
__global__ void k_reset(Planes<real> pl, SimParams p, ResetArgs a, real *coef_w[9], real *ratio_w[4]) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)p.R * p.Ns) return;
  const int r = (int)(i / p.Ns), n = (int)(i - (int64_t)r * p.Ns);
  const uint32_t env = (uint32_t)(p.rep_offset + r), house = (uint32_t)(p.house_offset + n);
  real *t_air = const_cast<real *>(pl.t_air), *t_mass = const_cast<real *>(pl.t_mass);
  real *target_w = const_cast<real *>(pl.target), *cap_w = const_cast<real *>(pl.cap);
  if (n >= p.N) {  // padding slot: neutral zeros
    t_air[i] = 0; t_mass[i] = 0; pl.sso[i] = 0; pl.flags[i] = 0; target_w[i] = 0; cap_w[i] = 0;
    for (int k = 0; k < NCoef<real>::n; ++k) coef_w[k][i] = 0;
    return;
  }
  const U4 u0 = philox4x32_10(a.seed, env, house, 0u, PURPOSE_RESET);
  const U4 u1 = philox4x32_10(a.seed, env, house, 1u, PURPOSE_RESET);
  const U4 u2 = philox4x32_10(a.seed, env, house, 2u, PURPOSE_RESET);
  // target_temp += |gauss(0, std_target)|  (building.py:236-238)
  const double g = sqrt(-2.0 * log(u01_open_closed(u0.x))) * cos(2 * 3.141592653589793 * u01_open_closed(u0.y));
  const double target = p.default_target + fabs(a.std_target * g);
  const double fu = triangular_from_u(u01_half_open(u0.z), a.f_lo, a.f_hi, 1.0);
  const double fcm = triangular_from_u(u01_half_open(u0.w), a.f_lo, a.f_hi, 1.0);
  const double fca = triangular_from_u(u01_half_open(u1.x), a.f_lo, a.f_hi, 1.0);
  const double fhm = triangular_from_u(u01_half_open(u1.y), a.f_lo, a.f_hi, 1.0);
  const double Ua = a.quirk_ua ? fu : p.dUa * fu;          // '=' instead of '*=' (quirk Q1, building.py:245)
  const double Cm = p.dCm * fcm, Ca = p.dCa * fca, Hm = p.dHm * fhm;
  const int ci = min(a.n_caps - 1, (int)(((uint64_t)u1.z * (uint64_t)a.n_caps) >> 32));
  const double cap = a.caps[ci];                           // random.choices(cooling_capacity_list), hvac.py:68
  double ta, tm;
  uint32_t flags;
  int sso;
  if (a.mode == 0) {  // Building.reset ran before the noise: un-noised temps, HVAC on (quirks Q2, Q3)
    ta = a.init_air; tm = a.init_mass; flags = 1u; sso = 0;
  } else {
    ta = target + (-2.0 + 6.0 * u01_half_open(u1.w));
    tm = target + (-2.0 + 6.0 * u01_half_open(u2.x));
    const bool on = u2.y & 1u;
    sso = on ? 0 : p.dt * (int)(u2.z & 15u);
    flags = (on ? 1u : 0u) | ((!on && sso < p.lockout_duration) ? 2u : 0u);
  }
  double co[12];
  thermal_coefs(Ua, Ca, Cm, Hm, p.dt, co);
  if (sizeof(real) == 4) {
    t_air[i] = (real)(ta - target); t_mass[i] = (real)(tm - target);
    for (int k = 0; k < 6; ++k) coef_w[k][i] = (real)co[k];
  } else {
    t_air[i] = (real)ta; t_mass[i] = (real)tm;
    coef_w[0][i] = (real)Ua; coef_w[1][i] = (real)Ca; coef_w[2][i] = (real)Hm;
    for (int k = 0; k < 6; ++k) coef_w[3 + k][i] = (real)co[6 + k];
  }
  pl.sso[i] = sso;
  pl.flags[i] = (uint8_t)flags;
  target_w[i] = (real)target;
  cap_w[i] = (real)cap;
  if (ratio_w[0]) {
    ratio_w[0][i] = (real)(Ua / p.dUa); ratio_w[1][i] = (real)(Ca / p.dCa);
    ratio_w[2][i] = (real)(Cm / p.dCm); ratio_w[3][i] = (real)(Hm / p.dHm);
  }
  if (pl.interp_sub) {
    auto near3 = [](double v) {
      v = fmin(1.1, fmax(0.9, v));
      const double d0 = fabs(0.9 - v), d1 = fabs(1.0 - v), d2 = fabs(1.1 - v);
      return d1 < d0 ? (d2 < d1 ? 2 : 1) : (d2 < d0 ? 2 : 0);
    };
    const double cc = fmin(15000.0, fmax(10000.0, cap));
    const int ihv = fabs(10000.0 - cc) <= fabs(15000.0 - cc) ? 0 : 1;
    const_cast<uint8_t *>(pl.interp_sub)[i] =
        (uint8_t)((((near3(Ua / p.dUa) * 3 + near3(Cm / p.dCm)) * 3 + near3(Ca / p.dCa)) * 3 + near3(Hm / p.dHm)) * 2 + ihv);
  }
  if (n == 0) {
    const U4 e0 = philox4x32_10(a.seed, env, 0u, 0u, PURPOSE_RESET_ENV);
    int64_t epoch = a.start_epoch;
    if (a.randomize_date)  // environment.py:189-194: randrange(364) days + randrange(86400) seconds
      epoch += (int64_t)(((uint64_t)e0.x * 364ull) >> 32) * 86400 + (int64_t)(((uint64_t)e0.y * 86400ull) >> 32);
    const double noise = p.temp_std * sqrt(-2.0 * log(u01_open_closed(e0.z))) * cos(2 * 3.141592653589793 * u01_open_closed(e0.w));
    pl.epoch[r] = epoch;
    pl.od_temp[r] = od_temp_model(civil_from_epoch(epoch), p.day_temp, p.night_temp, p.phase, noise);
    pl.solar_next[r] = p.solar_on ? solar_gain(civil_from_epoch(epoch + p.dt), p.window_area, p.shading) : 0.0;
    pl.solar_cur[r] = 0.0;
    pl.signal[r] = 0.0;
    pl.base_power[r] = 0.0;
    const double pmax0 = p.dcap / p.cop;
    pl.max_power[r] = (double)p.n_global * pmax0;           // cached from the un-noised props (quirk Q2)
    pl.power[r] = a.mode == 0 ? (double)p.n_global * pmax0 : 0.0;
    pl.t_since_interp[r] = p.interp_period + 1;
    for (int k = 0; k < DRSIM_N_METRICS; ++k) pl.metrics[(size_t)r * DRSIM_N_METRICS + k] = 0.0;
  }
}

// ------------------------------------------------------------------------------------------
// Greedy-myopic controller on device (greedy_myopic_controller.py:67-104): one CTA per cluster,
// bitonic sort of (key, id) in shared memory, then the inherently sequential knapsack scan.
// ------------------------------------------------------------------------------------------
template <typename real>
__global__ void __launch_bounds__(1024) k_greedy(Planes<real> pl, SimParams p, int n_pow2) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  double *key = reinterpret_cast<double *>(smem_raw);
  int *idx = reinterpret_cast<int *>(key + n_pow2);
  const int r = blockIdx.x;
  const size_t rb = (size_t)r * p.Ns;
  // programmatic dependent launch on both sides: this grid becomes resident under the tail of the step before it, and
  // the step kernel behind it sets itself up (static planes) while the sort runs -- it waits for this grid's completion
  // before it reads the actions
  pdl_wait();
  pdl_trigger();
  if (n_pow2 <= (int)blockDim.x) {
    // one element per thread: compare-exchange distances below 32 go through warp shuffles (no shared
    // memory, no barrier), only the 15 of 55 stages with a distance >= 32 (n = 1024) cross warps
    const int i = threadIdx.x;
    double ki = INFINITY;
    int ii = 0x7fffffff;
    if (i < p.N) {
      ki = -(double)Rep<real>::dev(pl.t_air[rb + i], pl.target[rb + i]);
      ii = i;
    }
    for (int k = 2; k <= n_pow2; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        double kl;
        int il;
        if (j >= 32) {
          if (i < n_pow2) { key[i] = ki; idx[i] = ii; }
          __syncthreads();
          kl = i < n_pow2 ? key[i ^ j] : ki;
          il = i < n_pow2 ? idx[i ^ j] : ii;
          __syncthreads();
        } else {
          kl = __shfl_xor_sync(0xffffffffu, ki, j);
          il = __shfl_xor_sync(0xffffffffu, ii, j);
        }
        const bool lower = (i & j) == 0, up = (i & k) == 0;
        const bool gt = (ki > kl) || (ki == kl && ii > il);   // (key, id) order == stable sort
        // the lower index of an ascending pair keeps the smaller element, and so on
        if (gt == (lower == up)) { ki = kl; ii = il; }
      }
    }
    if (i < n_pow2) { key[i] = ki; idx[i] = ii; }
    __syncthreads();
  } else {
  for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
    if (i < p.N) {
      key[i] = -(double)Rep<real>::dev(pl.t_air[rb + i], pl.target[rb + i]);
      idx[i] = i;
    } else {
      key[i] = INFINITY;
      idx[i] = 0x7fffffff;
    }
  }
  __syncthreads();
  for (int k = 2; k <= n_pow2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
        const int l = i ^ j;
        if (l > i) {
          const bool up = (i & k) == 0;
          const double ki = key[i], kl = key[l];
          const int ii = idx[i], il = idx[l];
          const bool gt = (ki > kl) || (ki == kl && ii > il);  // (key, id) order == stable sort
          if (gt == up) { key[i] = kl; key[l] = ki; idx[i] = il; idx[l] = ii; }
        }
      }
      __syncthreads();
    }
  }
  }
  // gather the scan's inputs in sorted order, in parallel: the keys are dead, their slots take the
  // per-house power cap / cop (greedy_myopic_controller.py:93); lock-out bit and verdict share a byte
  uint8_t *mark = reinterpret_cast<uint8_t *>(idx + n_pow2);
  double *pre = reinterpret_cast<double *>(smem_raw + (size_t)n_pow2 * 16);   // inclusive prefix sums (exact path)
  __shared__ double s_warp[32];
  __shared__ int s_first;
  bool nonneg = true, quant = true;
  for (int i = threadIdx.x; i < p.N; i += blockDim.x) {
    const int hh = idx[i];
    const double pw = (double)pl.cap[rb + hh] / p.cop;
    key[i] = pw;
    mark[i] = (pl.flags[rb + hh] >> 1) & 1u;
    nonneg = nonneg && pw >= 0.0;
    const double q = pw * 4096.0;                           // multiples of 2^-12 W below 2^20 W: every partial sum of
    quant = quant && q == floor(q) && fabs(q) < 4294967296.0;  // <= 2^16 of them is exact in fp64, in ANY order
  }
  for (int i = p.N + threadIdx.x; i < p.Ns; i += blockDim.x) pl.actions[rb + i] = 0;   // padding slots
  if (threadIdx.x == 0) s_first = p.N;
  const bool all_nonneg = __syncthreads_and(nonneg);
  const bool exact = __syncthreads_and(quant) && all_nonneg && p.N <= 65536;
  const double target = pl.signal[r];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int pos = 0;          // first house the sequential scan still has to look at
  double total = 0.0;   // accepted power before `pos`
  if (exact) {
    // The scan (:95-102) accepts every house while `pw + total < target`; up to the first refusal `total`
    // is the running sum of the sorted powers.  With exactly representable sums that prefix is the same
    // in any association, so it is computed by a block-wide parallel scan and the sequential part starts
    // at the first refusal instead of at house 0.
    const int per = (n_pow2 + blockDim.x - 1) / blockDim.x, i0 = threadIdx.x * per;
    double run = 0.0;
    for (int i = i0; i < i0 + per && i < p.N; ++i) { run += key[i]; pre[i] = run; }
    double inc = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    double off = inc - run;                                  // exclusive offset inside the warp
    for (int w = 0; w < warp; ++w) off += s_warp[w];
    int first = p.N;
    for (int i = i0; i < i0 + per && i < p.N; ++i) {
      const double v = pre[i] + off;
      pre[i] = v;
      if (v >= target && first == p.N) first = i;            // first-clause refusal (given all before accepted)
    }
    if (first < p.N) atomicMin(&s_first, first);
    __syncthreads();
    pos = s_first;
    total = pos > 0 ? pre[pos - 1] : 0.0;
    for (int i = threadIdx.x; i < pos; i += blockDim.x) mark[i] = 1;
    __syncthreads();
  }
  if (threadIdx.x < 32) {
    // The rest is sequential in `total`; one warp runs it 32 houses at a time: every lane fetches one
    // house, the values reach all lanes through shuffles, and all lanes replay the same fp64 chain
    // (DADD -> compare -> select), so `total` stays warp-uniform.  pw + total == total + pw bit for bit.
    for (int base = pos; base < p.N; base += 32) {
      const int i = base + lane;
      // powers >= 0: once the total has reached the target neither clause can accept any more
      if (all_nonneg && total >= target) {
        if (i < p.N) mark[i] = 0;
        continue;
      }
      const double my_pw = i < p.N ? key[i] : 0.0;
      const int my_lock = i < p.N ? (int)(mark[i] & 1u) : 1;
      const int cnt = min(32, p.N - base);
      bool my_take = false;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const double pw = __shfl_sync(0xffffffffu, my_pw, j);
        const int lock = __shfl_sync(0xffffffffu, my_lock, j);
        if (j < cnt) {
          const double t1 = pw + total;
          const bool take = t1 < target || (fabs(t1 - target) < fabs(total - target) && !lock);
          total = take ? t1 : total;
          if (j == lane) my_take = take;
        }
      }
      if (i < p.N) mark[i] = my_take ? 1 : 0;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < p.N; i += blockDim.x) pl.actions[rb + idx[i]] = mark[i];
}

// ------------------------------------------------------------------------------------------
// Per-cluster summary for the UI feed (client_manager_service.py:64-118 description values, :178-197
// graph series): one CTA per replica, fp64 sums in a fixed order (thread-strided partials, butterfly
// inside the warp, warps combined in index order) => run-to-run identical.
//   out[r] = { locked HVACs, sum Ta, sum (Ta - target), sum |Ta - target|, sum Tm, sum target, running HVACs, N }
// ------------------------------------------------------------------------------------------
constexpr int kSummaryFields = 8;

template <typename real>
__global__ void __launch_bounds__(256) k_summary(Planes<real> pl, SimParams p, double *out) {
  const int r = blockIdx.x;
  const size_t rb = (size_t)r * p.Ns;
  double s[7] = {0, 0, 0, 0, 0, 0, 0};
  for (int i = threadIdx.x; i < p.N; i += blockDim.x) {
    const double tgt = (double)pl.target[rb + i];
    const double d = (double)Rep<real>::dev(pl.t_air[rb + i], pl.target[rb + i]);
    const double dm = (double)Rep<real>::dev(pl.t_mass[rb + i], pl.target[rb + i]);
    const uint32_t f = pl.flags[rb + i];
    s[0] += (double)((f >> 1) & 1u);
    s[1] += d + tgt;
    s[2] += d;
    s[3] += fabs(d);
    s[4] += dm + tgt;
    s[5] += tgt;
    s[6] += (double)(f & 1u);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
#pragma unroll
    for (int k = 0; k < 7; ++k) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
  __shared__ double wp[8][7];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0)
    for (int k = 0; k < 7; ++k) wp[w][k] = s[k];
  __syncthreads();
  if (threadIdx.x < 7) {
    double t = 0.0;
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) t += wp[q][threadIdx.x];
    out[(size_t)r * kSummaryFields + threadIdx.x] = t;
  }
  if (threadIdx.x == 7) out[(size_t)r * kSummaryFields + 7] = (double)p.N;
}

// ------------------------------------------------------------------------------------------
// The reference's running metrics, LITERALLY (server/app/services/metrics_service.py:108-157, SURVEY 8f-3):
// one launch after a step accumulates, per cluster, the twelve cumulative fields of `Metrics.update` with its
// own expressions -- `temp_error = indoor_temp - target_temp / nb_agents` (:131-134: the division binds to the
// set-point only), `signal_error = (reg_signal - cluster_hvac_power) / nb_agents**2` added once per agent
// (:143-148) -- so that the logged values of a rollout on the device are the reference's, slips included.
//   acc[r] = { cumul_avg_reward, cumul_temp_offset, cumul_temp_error, max_temp_error, cumul_signal_offset,
//              cumul_signal_error, cumul_squared_error_temp, cumul_OD_temp, cumul_signal, cumul_cons,
//              cumul_squared_error_sig, cumul_squared_max_error_temp }
//   prev[r] = { reg_signal, OD_temp, cluster_hvac_power } of the observation BEFORE the step (obs_dict)
// Fixed-order fp64 sums (strided per thread, butterfly inside the warp, warps in index order).
// ------------------------------------------------------------------------------------------
constexpr int kRefMetricFields = 12;

template <typename real>
__global__ void __launch_bounds__(256) k_metrics_ref(Planes<real> pl, SimParams p, const double *prev, double *acc, int collect_sq) {
  const int r = blockIdx.x;
  const size_t rb = (size_t)r * p.Ns;
  const double n = (double)p.N;
  double s[4] = {0, 0, 0, 0};   // sum temp_error, sum |temp_error|, sum temp_error^2, sum reward / n
  double mx = acc[(size_t)r * kRefMetricFields + 3];
  for (int i = threadIdx.x; i < p.N; i += blockDim.x) {
    const double tgt = (double)pl.target[rb + i];
    const double ta = (double)Rep<real>::dev(pl.t_air[rb + i], pl.target[rb + i]) + tgt;
    const double te = ta - tgt / n;
    s[0] += te;
    s[1] += fabs(te);
    s[2] += te * te;
    s[3] += (double)pl.reward[rb + i] / n;
    mx = fmax(mx, te);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int k = 0; k < 4; ++k) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  __shared__ double wp[8][5];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    for (int k = 0; k < 4; ++k) wp[w][k] = s[k];
    wp[w][4] = mx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double t[4] = {0, 0, 0, 0};
    double m = wp[0][4];
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) {
      for (int k = 0; k < 4; ++k) t[k] += wp[q][k];
      m = fmax(m, wp[q][4]);
    }
    double *a = acc + (size_t)r * kRefMetricFields;
    const double sig_old = prev[(size_t)r * 3], od_old = prev[(size_t)r * 3 + 1], p_old = prev[(size_t)r * 3 + 2];
    const double se = (sig_old - pl.power[r]) / (n * n);
    a[0] += t[3];
    a[1] += t[0];
    a[2] += t[1];
    a[3] = m;
    a[4] += n * se;
    a[5] += n * fabs(se);
    if (collect_sq) a[6] += t[2];
    a[7] += od_old;
    a[8] += sig_old;
    a[9] += p_old;
    if (collect_sq) { a[10] += sig_old * sig_old; a[11] = m * m; }
  }
}

// ------------------------------------------------------------------------------------------
// Snapshot for the dict API (Environment.get_obs, environment.py:110-130): everything the per-agent observation
// dicts are built from, written by ONE launch straight into mapped pinned host memory -- absolute temperatures
// as fp64 (the fp32 build keeps deviations), rewards as fp64, seconds_since_off, the two flags, the env scalars.
// The observation rows follow by one copy-engine transfer; the caller synchronises once.
// ------------------------------------------------------------------------------------------

template <typename real>
__global__ void k_snapshot(Planes<real> pl, SimParams p, SnapPtrs o) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (long long)p.R * p.N) {
    const int r = (int)(i / p.N), n = (int)(i - (long long)r * p.N);
    const size_t s = (size_t)r * p.Ns + n;
    const double tgt = (double)pl.target[s];
    const bool dev = sizeof(real) == 4;
    o.t_air[i] = (double)pl.t_air[s] + (dev ? tgt : 0.0);
    o.t_mass[i] = (double)pl.t_mass[s] + (dev ? tgt : 0.0);
    o.reward[i] = (double)pl.reward[s];
    o.sso[i] = pl.sso[s];
    const uint32_t f = pl.flags[s];
    o.on[i] = (uint8_t)(f & 1u);
    o.lockout[i] = (uint8_t)((f >> 1) & 1u);
  }
  if (i < p.R) {
    double *e = o.env + (size_t)i * kSnapEnv;
    e[0] = pl.od_temp[i]; e[1] = pl.signal[i]; e[2] = pl.power[i]; e[3] = pl.solar_cur[i];
    e[4] = pl.base_power[i]; e[5] = (double)pl.epoch[i]; e[6] = (double)pl.t_since_interp[i]; e[7] = pl.max_power[i];
  }
}

}  // namespace drsim
