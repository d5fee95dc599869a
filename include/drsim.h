/*
 * drsim.h -- C ABI of the B200-native demand-response environment step (libdrsim.so).
 *
 * The reference (ALLabMTL/marl-demandresponse) is pure Python and has no FFI for this path:
 * callers construct `Environment(env_props)` directly and call `reset()` / `step(action_dict)`
 * (server/app/core/environment/environment.py:39,49,72; call sites
 * server/app/services/controller_manager.py:109,172 and training_manager.py:161,231).  This
 * header is therefore the boundary a maintainer would bind with `ctypes` from a replacement
 * `Environment` class (see INTEGRATION.md); every entry point names the reference code it
 * replaces.
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success or a negative DRSIM_E_* code,
 *     the message is available from drsim_last_error() (thread-local);
 *   - the library owns all device buffers of a handle (one cudaMalloc slab); callers own the
 *     action / injected-noise buffers they pass in;
 *   - one handle is bound to one CUDA device; calls on a handle are not re-entrant and are
 *     ordered by the `stream` argument (a cudaStream_t passed as void*, NULL = default stream);
 *   - there is NO CPU fallback: drsim_create fails unless the device is compute capability 10.x.
 *
 * Layout: per-house planes are structure-of-arrays [n_rep][house_stride] with
 * house_stride = n_house rounded up to a multiple of 4 (16-byte vector accesses); per-replica
 * ("env") scalars are [n_rep] doubles.
 */
#ifndef DRSIM_H_
#define DRSIM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRSIM_ABI_VERSION 4
#define DRSIM_MAX_SIGNAL_TERMS 8
#define DRSIM_INTERP_SUBTABLES 162      /* 3*3*3*3*2 nearest-neighbour cells            */
#define DRSIM_INTERP_SUBTABLE_LEN 25920 /* 9*5*8*12*6 values of the 5-D multilinear part */

enum { DRSIM_OK = 0, DRSIM_E_ARG = -1, DRSIM_E_CUDA = -2, DRSIM_E_DEVICE = -3, DRSIM_E_STATE = -4 };

enum { DRSIM_F32 = 0, DRSIM_F64 = 1 };
/* rewards_calculator.py:46-133 */
enum { DRSIM_PEN_INDIVIDUAL_L2 = 0, DRSIM_PEN_COMMON_L2 = 1, DRSIM_PEN_COMMON_MAX = 2, DRSIM_PEN_MIXTURE = 3 };
/* power_grid.py:144-161 */
enum { DRSIM_BASE_CONSTANT = 0, DRSIM_BASE_INTERPOLATION = 1 };
/* signal_calculator.py:33-115 */
enum { DRSIM_SIG_FLAT = 0, DRSIM_SIG_SINUSOIDALS = 1, DRSIM_SIG_REGULAR_STEPS = 2, DRSIM_SIG_PERLIN = 3 };
/* observation layouts: none, utils/norm.py:178-218 (hand-engineered, with neighbour messages),
 * "TarMAC" = own-state features only + static neighbour index tensor (SURVEY 8a-12) */
enum { DRSIM_OBS_NONE = 0, DRSIM_OBS_HAND_ENGINEERED = 1, DRSIM_OBS_TARMAC = 2 };
/* element type of the observation rows: the build's `real`, or bfloat16 (fp32 build only).  A bf16 row element is
 * the fp32 element the kernels compute, rounded to nearest-even where it is stored; nothing else changes. */
enum { DRSIM_OBS_F32 = 0, DRSIM_OBS_BF16 = 1 };
/* neighbour source: arithmetic ring (agent_communication_builder.py:63-85), explicit table, or a fresh uniform
 * sample per step (`random_sample`, cluster.py:96-99): neighbour k of house n in the rows written after the handle's
 * d-th step (d = drsim_step_count; rows of drsim_reset / drsim_refresh use the current count) is output k of a
 * sparse partial Fisher-Yates shuffle of the other houses driven by Philox4x32-10 keyed (seed, global replica,
 * global house, d, purpose 7 | block << 8) -- see drsim_comm_sample and DESIGN.md.  Replicas only: a house-sharded
 * handle rejects it.  nb_comm <= DRSIM_MAX_SAMPLE_COMM in this mode (the swap record is per-thread). */
enum { DRSIM_COMM_RING = 0, DRSIM_COMM_TABLE = 1, DRSIM_COMM_SAMPLE = 2 };
#define DRSIM_MAX_SAMPLE_COMM 32
/* where per-step noise comes from when the matching pointer of drsim_step_args is NULL */
enum { DRSIM_NOISE_ZERO = 0, DRSIM_NOISE_PHILOX = 1 };
/* action source: caller-provided, or restated controllers
 * (controllers/bangbang_controllers.py:18-89, greedy_myopic_controller.py:67-104).  Greedy-myopic sorts the whole
 * cluster in shared memory: replicas only (a house-sharded handle rejects it) and n_house <= 8192. */
enum {
  DRSIM_POLICY_EXTERNAL = 0,
  DRSIM_POLICY_DEADBAND_BANGBANG = 1,
  DRSIM_POLICY_BANGBANG = 2,
  DRSIM_POLICY_ALWAYS_ON = 3,
  DRSIM_POLICY_GREEDY_MYOPIC = 4
};
/* kernel path: auto, force the fused single-kernel tile path, force the general 3-kernel path */
enum { DRSIM_PATH_AUTO = 0, DRSIM_PATH_FUSED = 1, DRSIM_PATH_SPLIT = 2 };

/* Flattened EnvironmentProperties (environment_properties.py:339-371 and the classes it nests). */
typedef struct drsim_config {
  int32_t abi_version; /* must be DRSIM_ABI_VERSION */
  int32_t n_rep;       /* R independent replicas of the cluster                           */
  int32_t n_house;     /* N = cluster_prop.nb_agents (houses owned by THIS handle)        */
  int32_t precision;   /* DRSIM_F32 | DRSIM_F64                                           */
  int32_t dt;          /* time_step.seconds (hvac.py:46)                                  */
  int32_t path;        /* DRSIM_PATH_*                                                    */

  /* single very large cluster split across devices (SURVEY 8e): this handle owns houses
   * [house_offset, house_offset + n_house) of a cluster of n_house_global houses; 0/0 = whole */
  int64_t house_offset;
  int64_t n_house_global;
  int64_t rep_offset; /* global index of local replica 0 (keys the Philox streams)          */

  /* BuildingProperties / HvacProperties defaults (environment_properties.py:70-205) */
  double deadband;
  double cop;
  double latent_cooling_fraction;
  int32_t lockout_duration;
  int32_t solar_gain; /* bool */
  double window_area;
  double shading_coeff;
  double default_target_temp;
  double default_Ua, default_Ca, default_Cm, default_Hm;
  double default_cooling_capacity;

  /* TemperatureProperties (cluster_properties.py:9-28) */
  double day_temp, night_temp, temp_std, phase;

  /* RewardProperties (environment_properties.py:221-258) */
  double alpha_temp, alpha_sig, norm_reg_sig;
  int32_t penalty_mode;
  int32_t obs_dtype; /* DRSIM_OBS_F32 | DRSIM_OBS_BF16 (needs precision DRSIM_F32 and an observation layout) */
  double alpha_ind_l2, alpha_common_l2, alpha_common_max;

  /* PowerGridProperties (power_grid_properties.py:6-70) */
  int32_t base_power_mode;
  int32_t interp_update_period;
  int32_t interp_nb_agents;
  int32_t signal_mode;
  double avg_power_per_hvac;
  int32_t n_signal_terms; /* len(amplitude_ratios) == len(periods) for sinusoidals */
  int32_t nb_octaves;
  double amplitude_ratios[DRSIM_MAX_SIGNAL_TERMS];
  double periods[DRSIM_MAX_SIGNAL_TERMS];
  double amplitude_per_hvac;
  int32_t octaves_step;
  int32_t period;

  /* observation layout (utils/norm.py, StateProperties / MessageProperties) */
  int32_t obs_layout;
  int32_t nb_comm;   /* min(max_nb_agents_communication, N-1), agent_communication_builder.py:49-52 */
  int32_t comm_mode; /* DRSIM_COMM_* */
  int32_t state_solar_gain, state_thermal, state_hvac;
  int32_t message_thermal, message_hvac;

  int32_t noise_mode; /* DRSIM_NOISE_* */
  int32_t policy;     /* DRSIM_POLICY_* */
  uint64_t seed;      /* Philox key */
} drsim_config;

/* Host-side full state, fp64, row-major [n_rep][n_house] / [n_rep]; NULL members are skipped by
 * drsim_set_state and left untouched by drsim_get_state.  The four thermal parameters are turned
 * into the per-house update coefficients inside drsim_set_state (building.py:160-201). */
typedef struct drsim_host_state {
  double *t_air, *t_mass;          /* Building.indoor_temp / current_mass_temp            */
  double *target;                  /* init_props.target_temp                              */
  double *Ua, *Ca, *Cm, *Hm;       /* init_props thermal parameters                       */
  double *cap;                     /* hvac.init_props.cooling_capacity                    */
  uint8_t *on, *lockout;           /* HVAC.turned_on / lockout                            */
  int32_t *sso;                    /* HVAC.seconds_since_off                              */
  int64_t *epoch;                  /* Environment.date_time as naive seconds since 1970   */
  double *od_temp;                 /* Environment.current_od_temp                         */
  double *signal;                  /* PowerGrid.current_signal                            */
  double *base_power;              /* PowerGrid.base_power                                */
  double *power;                   /* Cluster.current_power_consumption                   */
  double *solar;                   /* Building.current_solar_gain (cluster-wide)          */
  double *artificial_ratio;        /* PowerGridProperties.artificial_ratio (post-draw)    */
  double *max_power;               /* Cluster.max_power                                   */
  int32_t *t_since_interp;         /* PowerGrid.time_since_last_interp                    */
  /* optional [n_rep][n_house][12]: precomputed output of drsim_host_thermal_coefs for each house
   * (set_state only).  When NULL the library derives it from Ua, Ca, Cm, Hm with libm; a caller
   * that wants the constants of building.py:196-206 bit-identical to NumPy's passes its own. */
  double *thermal_coefs;
  /* optional [n_rep][n_house]: per-HVAC lock-out duration in seconds (the legacy env draws
   * lockout_duration + randint(-lockout_noise, lockout_noise) per HVAC, v0/env/MA_DemandResponse.py:397-403).
   * NULL = the handle's common drsim_config.lockout_duration.  A handle that has been given durations differing
   * from the common one steps on the general path (the fused tile kernels share one duration) until drsim_reset. */
  int32_t *lockout_duration;
} drsim_host_state;

/* Device pointers of a handle (zero-copy views for torch / cupy).  `real` planes are float
 * (DRSIM_F32) or double (DRSIM_F64); `row` elements are obs_bytes wide: real, or bfloat16 (DRSIM_OBS_BF16). */
typedef struct drsim_ptrs {
  int32_t n_rep, n_house, house_stride, obs_dim, real_bytes, nb_comm;
  /* 1 (DRSIM_F32): the t_air / t_mass planes hold the DEVIATION from the house set-point,
   * Ta - target and Tm - target (what reward, messages, controllers and the interpolator consume;
   * it also keeps fp32 rounding at the 1e-7 degC level); 0 (DRSIM_F64): absolute degC. */
  int32_t temp_is_deviation;
  int32_t obs_bytes;           /* size of one observation-row element: 8, 4 or 2 (bfloat16) */
  void *t_air, *t_mass;        /* real  [R][stride] */
  int32_t *sso;                /* i32   [R][stride] */
  uint8_t *flags;              /* u8    [R][stride]  bit0 = turned_on, bit1 = lockout */
  void *target, *cap;          /* real  [R][stride] */
  void *reward;                /* real  [R][stride] */
  void *obs;                   /* row   [R][stride][obs_dim] */
  uint8_t *actions;            /* u8    [R][stride]  internal action plane (policies / host API) */
  int64_t *epoch;              /* i64   [R] */
  double *od_temp, *signal, *base_power, *power, *solar, *pen_sum, *pen_max; /* f64 [R] */
  int32_t *comm_table;         /* i32   [N][nb_comm] (or [R][N][nb_comm] if per-replica) or NULL */
  double *metrics;             /* f64   [R][DRSIM_N_METRICS] running rollout accumulators */
  double *acc;                 /* f64   [R][DRSIM_N_ACC] per-rank partial sums of drsim_step_begin */
  double *rew_sig;             /* f64   [R] alpha_sig * signal penalty / norm of the last step */
  /* House-sharded ring cluster with neighbour messages: [R][nb_comm][DRSIM_HALO_FIELDS] message records
   * of this shard's edge houses after drsim_step_begin -- entries [0, H) = its FIRST H houses, entries
   * [H, H + L) = its LAST L houses, L = nb_comm / 2, H = nb_comm - L
   * (agent_communication_builder.py:74-84); NULL when no halo is exchanged. */
  double *halo_out;
} drsim_ptrs;

#define DRSIM_HALO_FIELDS 8 /* (Ta-target)/5, sso/dur, P/nrs, Pmax/nrs (norm.py:31-48), 4 thermal ratios (:50-57) */

#define DRSIM_N_ACC 6 /* P, sum pen/N, max pen, sum dT, sum dT^2, interpolated base-power sum */

#define DRSIM_N_METRICS 6 /* steps, sum reward/N, sum |Ta-target|/N, sum (Ta-target)^2/N, sum |P-S|, sum (P-S)^2 */

/* Per-step inputs, all DEVICE pointers; NULL selects the handle's own source. */
typedef struct drsim_step_args {
  const uint8_t *actions;     /* u8 [R][house_stride]; NULL = internal plane / on-device policy      */
  const double *od_noise;     /* [R]  the random.gauss(0, temp_std) draw of environment.py:158       */
  const double *perlin;       /* [R]  value of Perlin.calculate_noise (perlin.py:41-56)              */
  const int32_t *interp_ids;  /* [R][interp_nb_agents] ids of random.choices (interpolation.py:223)  */
} drsim_step_args;

typedef struct drsim_handle drsim_t;

/* Environment.__init__ (environment.py:39-47): allocate a simulator for R x N houses on `device`. */
int drsim_create(const drsim_config *cfg, int device, drsim_t **out);
int drsim_destroy(drsim_t *h);
/* copy.deepcopy(env) (training_manager.py:269): clone all device state into a new handle. */
int drsim_clone(const drsim_t *h, drsim_t **out);
int drsim_buffers(drsim_t *h, drsim_ptrs *out);

/* State injection / extraction (replaces poking Building/HVAC attributes, building.py:49-61,
 * hvac.py:36-41).  Synchronous with respect to `stream`. */
int drsim_set_state(drsim_t *h, const drsim_host_state *st, void *stream);
int drsim_get_state(drsim_t *h, drsim_host_state *st, void *stream);

/* Environment.reset / apply_noise on the device (environment.py:49-70,161-194; building.py:224-267;
 * hvac.py:36-41,66-70; SURVEY 8a-15): draws every house property from counter-based Philox streams
 * keyed by (seed, global replica, global house, draw) instead of Python's Mersenne Twister -- the
 * DISTRIBUTIONS are the reference's, the stream is ours.  mode 0 = reference reset (target +=
 * |N(0, std_target)|, Ua = tri(lo, hi, 1) if quirk_ua else Ua * tri, Cm/Ca/Hm *= tri, capacity uniform
 * in caps[], initial temperatures un-noised, HVAC on, quirks Q1-Q3); mode 1 = the synthetic benchmark
 * state of SURVEY 8d (Ta, Tm = target + U(-2, 4), on ~ Bernoulli(1/2), sso = 0 | dt * U{0..15}).
 * Also initialises the env scalars (start datetime + U{0..363} d + U{0..86399} s when randomize_date,
 * outdoor temperature, max_power).  Follow with drsim_refresh(h, NULL, 1, stream). */
typedef struct drsim_reset_args {
  uint64_t seed;
  int32_t mode;
  int32_t randomize_date;
  int64_t start_epoch;
  double init_air_temp, init_mass_temp;
  double std_target_temp;
  double factor_low, factor_high;
  int32_t quirk_ua;
  int32_t n_caps;
  double caps[8];
} drsim_reset_args;
int drsim_reset(drsim_t *h, const drsim_reset_args *args, void *stream);

/* Cluster.agent_communicators (cluster.py:66-70): explicit neighbour table, host int32
 * [n_house][nb_comm] (per_replica = 0) or [n_rep][n_house][nb_comm] (per_replica = 1). */
int drsim_set_comm_table(drsim_t *h, const int32_t *table, int per_replica, void *stream);

/* DRSIM_COMM_SAMPLE handle: writes the neighbour table of draw `draw` -- device int32 [n_rep][n_house][nb_comm],
 * global house ids -- on `stream`.  draw < 0: the draw behind the current observation rows (= drsim_step_count).
 * This is what a TarMAC policy attends over.  DRSIM_E_STATE on a handle of another mode. */
int drsim_comm_sample(drsim_t *h, int64_t draw, int32_t *d_out, void *stream);

/* steps taken since creation or the last drsim_reset (drsim_step, drsim_run, step_host, rollout, sharded steps);
 * drsim_clone copies it */
int64_t drsim_step_count(const drsim_t *h);

/* PowerInterpolator.values (interpolation.py:88-90) re-ordered to
 * [162][9][5][8][12][6] (see DESIGN.md), host fp64. */
int drsim_set_interp_table(drsim_t *h, const double *sub_tables, void *stream);

/* Environment.step (environment.py:72-108): one step of every replica on `stream`. */
int drsim_step(drsim_t *h, const drsim_step_args *args, void *stream);

/* `n_steps` consecutive Environment.step calls (environment.py:72-108) in one C call: a rollout under an
 * on-device policy (args->actions NULL) or the replay of an action tape -- step k reads its actions at
 * args->actions + k * action_stride bytes (stride 0: the same plane every step).  Injected noise and
 * sampled ids are per-step inputs and are rejected when n_steps > 1.  Results are those of n_steps
 * drsim_step calls. */
int drsim_run(drsim_t *h, const drsim_step_args *args, int n_steps, size_t action_stride, void *stream);
/* The same with a ROTATING action tape of `tape_planes` planes: step k reads plane k % tape_planes
 * (tape_planes = 0: no wrap, drsim_run).  Also accepts a house-sharded handle (every step is then a
 * drsim_step_sharded: all ranks must run the same number of steps), so that a rollout of one cluster split
 * across GPUs is enqueued by one C call per rank instead of one host-language call per step.
 * On the staged fused kernels (fp32, replicas on one GPU, constant base power, at least two tiles per CTA) the
 * steps of a block of schedule records run INSIDE one launch: a CTA's inputs of step k + 1 are its own outputs of
 * step k plus the tape, so consecutive steps have no boundary between CTAs (DESIGN.md section 4; bit-identical to
 * one launch per step, which DRSIM_NO_STREAM=1 in the environment restores).  The action planes of the whole block
 * must therefore stay untouched until the call's work on `stream` has completed -- as for any asynchronous call. */
int drsim_run_tape(drsim_t *h, const drsim_step_args *args, int n_steps, size_t action_stride, int tape_planes,
                   void *stream);

/* PowerGrid.step at reset + get_obs (environment.py:66-70): recompute signal (optional) and the
 * observation / message gather from the current state without advancing time. */
int drsim_refresh(drsim_t *h, const drsim_step_args *args, int recompute_signal, void *stream);

/* Environment.step for ONE cluster whose houses are split across several handles / GPUs
 * (SURVEY 8e): drsim_step_begin updates the local houses and leaves this rank's partial sums in
 * drsim_ptrs.acc ([R][DRSIM_N_ACC]: cluster power cluster.py:88, penalty sums, interpolated base
 * power).  The caller all-gathers them across ranks (NCCL over NVLink: 48 bytes per rank) and hands
 * the gathered device array [n_parts][R][DRSIM_N_ACC] (rank order) to drsim_step_finish, which
 * combines it in rank order (deterministic, identical on every rank) and runs the env epilogue,
 * rewards and observations.  acc_gathered = NULL uses the handle's own partials. */
int drsim_step_begin(drsim_t *h, const drsim_step_args *args, void *stream);
int drsim_step_finish(drsim_t *h, const drsim_step_args *args, const double *acc_gathered, int n_parts,
                      void *stream);
/* drsim_step_begin + drsim_step_finish(h, args, NULL, -1 or 1, stream) in one call, for the peer-memory
 * exchange (after drsim_ipc_attach / drsim_peer_attach_local) or a single rank: nothing is needed from the
 * host in between.  Runs as ONE persistent kernel (house update, reduction, NVLink push of the partial sums
 * and halo records, bounded wait, env epilogue, rewards, observations); results are bit-identical to the
 * begin / finish pair.  Fails with DRSIM_E_STATE once an exchange wait has timed out on an earlier step. */
int drsim_step_sharded(drsim_t *h, const drsim_step_args *args, void *stream);

/* Same, for a sharded cluster whose observation rows carry ring-neighbour messages (cluster.py:91-111):
 * halo_gathered = the drsim_ptrs.halo_out blocks of all ranks, all-gathered in rank order
 * ([n_parts][R][nb_comm][DRSIM_HALO_FIELDS]); `rank` = this handle's position in that order.  The
 * neighbours that fall outside the shard are read from the adjacent ranks' blocks. */
int drsim_step_finish_gathered(drsim_t *h, const double *acc_gathered, const double *halo_gathered, int n_parts,
                               int rank, void *stream);

/* Peer-memory variant of the same exchange (no NCCL on the step path): every rank exports an IPC
 * handle of its slab + the offsets of its "inbox" (96 bytes), the handles of all ranks are attached,
 * and from then on drsim_step_begin pushes this rank's partial sums straight into every rank's inbox
 * over NVLink from the tail of the reduction kernel, and drsim_step_finish(h, args, NULL, -1, stream)
 * waits (bounded, ~2 s) for all rows inside the epilogue kernel.  drsim_peer_status reports a timeout. */
int drsim_ipc_export(drsim_t *h, void *out96);
int drsim_ipc_attach(drsim_t *h, int rank, int world, const void *handles96, void *stream);
int drsim_peer_status(drsim_t *h, void *stream);
/* The same attachment for `world` handles of ONE process, in rank order (raw device pointers instead of
 * IPC handles): several shards on one GPU -- their steps must then be issued on different streams, the
 * kernels of the shards wait for one another -- or several GPUs driven by one process (peer access is
 * enabled here).  Replaces nothing in the reference (cluster.py:73-89 is one Python loop). */
int drsim_peer_attach_local(drsim_t *const *handles, int world, void *stream);

/* Same step with HOST buffers (pinned or pageable): actions u8 [R][N] in, per-env results out
 * ([R][4] doubles: power, signal, od_temp, mean reward); transfers are inside the call and ordered on
 * `stream`; the call returns after the results have landed (stream synchronised).  When the step runs on
 * one of the staged fused kernels and `actions` is pinned (device-mapped) memory with N % 4 == 0, the
 * transfer overlaps the kernel: planes under 256 KB are read in place over PCIe by the kernel, one tile
 * ahead of their use; larger ones travel as one linear copy-engine transfer (on a stream of the handle)
 * into a staging plane the kernel consumes as it lands -- on that path an action byte must be 0 or 1
 * (four 0xFF bytes in one aligned word mark "not arrived yet"; a word that never arrives ends in DRSIM_E_STATE
 * after ~2 s, the step having been committed with those houses off: the handle then refuses every further step
 * until drsim_set_state / drsim_reset re-injects a state).  The kernel
 * writes the [R][4] results itself -- straight into `env_out` when that is pinned memory too, else into a
 * mapped buffer of the handle; otherwise explicit copies are used.  The environment variable
 * DRSIM_HOST_ACTIONS = zerocopy | dma (read by drsim_create) forces one transfer mode. */
int drsim_step_host(drsim_t *h, const uint8_t *actions, const double *od_noise, const double *perlin,
                    const int32_t *interp_ids, double *env_out, void *stream);

/* Environment.step with HOST buffers and the reference's full return value (environment.py:108: per-agent
 * observations and rewards): drsim_step_host, then reward_out[R][N] (`real` = float or double as the handle was built)
 * and obs_out[R][N][obs_dim] (float, double or bfloat16 as drsim_ptrs.obs_bytes says; row-major, no padding; either may
 * be NULL) are copied back behind the kernel,
 * ahead of the call's one stream synchronisation.  On BASELINE config 4 that is 90 MB per step: PCIe-bound. */
int drsim_step_host_full(drsim_t *h, const uint8_t *actions, const double *od_noise, const double *perlin,
                         const int32_t *interp_ids, double *env_out, void *reward_out, void *obs_out, void *stream);

/* What Environment.get_obs (environment.py:110-130, cluster.py:113-121, building.py:79-100, hvac.py:72-83) builds
 * its 21-key per-agent dicts from, in ONE call: a kernel writes the house state (absolute temperatures and rewards
 * as fp64, seconds_since_off, the two flags) and the env scalars straight into pinned host memory of the handle,
 * the observation rows follow by one copy, the stream is synchronised once.  The pointers stay valid until the
 * next snapshot of the handle (copy what must outlive it).
 * env[r] = { OD_temp, reg_signal, cluster_hvac_power, solar_gain, base_power, epoch, time_since_last_interp, max_power }. */
typedef struct drsim_snapshot_view {
  int32_t n_rep, n_house, obs_dim, real_bytes;
  const double *t_air, *t_mass, *reward; /* [R][N] */
  const int32_t *sso;                    /* [R][N] */
  const uint8_t *on, *lockout;           /* [R][N] */
  const double *env;                     /* [R][8] */
  const void *obs;                       /* [R][N][obs_dim] float | double | bfloat16 as the handle was built, or NULL */
} drsim_snapshot_view;
int drsim_snapshot(drsim_t *h, drsim_snapshot_view *out, void *stream);
/* Environment.step for the dict API: drsim_step_host (host action / noise buffers in) followed by the snapshot,
 * with ONE stream synchronisation for both. */
int drsim_step_host_snapshot(drsim_t *h, const uint8_t *actions, const double *od_noise, const double *perlin,
                             const int32_t *interp_ids, drsim_snapshot_view *out, void *stream);

/* MA-PPO actor of the reference (agents/trainables/network.py:14-35: Linear(obs_dim, h1) - ReLU -
 * Linear(h1, h2) - ReLU - Linear(h2, 2) - softmax), all DEVICE pointers in torch.nn.Linear layout
 * (weight [out][in], row-major fp32). */
typedef struct drsim_actor_net {
  const float *w1, *b1; /* [h1][obs_dim], [h1] */
  const float *w2, *b2; /* [h2][h1], [h2] */
  const float *w3, *b3; /* [2][h2], [2] */
  int32_t h1, h2;       /* 1 .. 111 each */
  /* 0 = one TF32 pass per product (|dp| <= 5e-3 against an fp32 forward), 1 = "3xTF32": every operand split into
   * hi + lo TF32 halves, three tensor-core passes per product, fp32-grade probabilities (|dp| ~ 1e-6).
   * On a handle with bfloat16 rows (DRSIM_OBS_BF16) only 1 is accepted: the 3xTF32 actor widens the rows as it loads
   * them, with results bit-identical to the same actor on the widened fp32 rows; 0 fails with DRSIM_E_ARG. */
  int32_t precision;
  int32_t pad_;
} drsim_actor_net;

/* MAPPO.select_actions (mappo.py:83-97) for every house of every replica, on the device (SURVEY 8f-2):
 * the actor runs on the handle's observation rows (fp32 build, obs_dim <= 64) as two tcgen05 TF32 GEMMs
 * per 128-row tile, the categorical draw uses a Philox uniform keyed (seed, replica, house, step), the
 * chosen actions go into the handle's action plane (so the next drsim_step with args->actions == NULL
 * consumes them) and, when the pointers are not NULL, prob_drawn[R][stride] receives the probability of
 * the drawn action (the PPO ratio's denominator) and prob_on[R][stride] the probability of action 1. */
int drsim_policy_step(drsim_t *h, const drsim_actor_net *net, uint64_t seed, float *prob_drawn, float *prob_on,
                      void *stream);

/* One transition of an MA-PPO rollout ENTIRELY on the device, stored where the caller wants it (SURVEY 8f-2):
 * MAPPO.select_actions (mappo.py:83-97) on state_t, Environment.step (environment.py:72-108) on the drawn actions and
 * MAPPO.store_transition (mappo.py:105-127; training_manager.py:224-240) in one call.  All DEVICE pointers, plane
 * layout of the handle (row stride = house_stride); obs / reward / next_obs 16-byte aligned, actions / prob 4-byte
 * aligned; the step kernels write the slot directly:
 *   obs      [R][stride][obs_dim] row  state_t the actor reads (NULL: the handle's own rows = the last step's result)
 *   actions  [R][stride] u8            a_t drawn by the actor, consumed by the step            (Transition.action)
 *   prob     [R][stride] f32           probability of a_t under the actor (mappo.py:95)        (Transition.a_log_prob)
 *   reward   [R][stride] f32           r_t                                                       (Transition.reward)
 *   next_obs [R][stride][obs_dim] row  state_{t+1}: pass it as `obs` of the next transition     (Transition.next_state)
 * (`row` = f32, or bf16 on a handle built with DRSIM_OBS_BF16)
 * Transition.others_actions is the `actions` plane without the agent's own entry; `done` is the caller's
 * (training_manager.py:233: end of the episode).  The reference does not evaluate its critic during the rollout
 * (mappo.py:99-103 is commented out): Critic(cat(state, others_actions)) runs in update() on these buffers. */
typedef struct drsim_rollout_slot {
  const void *obs;
  uint8_t *actions;
  float *prob;
  void *reward;
  void *next_obs;
} drsim_rollout_slot;
int drsim_rollout_transition(drsim_t *h, const drsim_actor_net *net, uint64_t seed, const drsim_rollout_slot *slot,
                             void *stream);

/* number of kernels launched by this handle since creation (bench.py "gpu_launches") */
int64_t drsim_launch_count(const drsim_t *h);

/* Geometry of the fused step kernel chosen for this handle (diagnostics and tests):
 * out[0] = variant (0 none: general path only, 1 chunked rows, 2 register-direct, 3 staged inputs +
 * whole-tile rows, 4 staged inputs + per-warp row groups), out[1] = clusters per tile,
 * out[2] = tiles, out[3] = grid (CTAs), out[4] = dynamic shared memory per CTA (bytes),
 * out[5] = resident CTAs per SM.  The environment variable DRSIM_TILE_ENVS (read by drsim_create)
 * caps the clusters per tile instead of the built-in round-count heuristic. */
int drsim_fused_info(const drsim_t *h, int32_t out[6]);

/* Route of the last step launched on this handle (diagnostics and tests), -1 before the first step (a refresh counts):
 * which kernels ran it.  A handle's steps take different routes: refreshes, interpolator firings, injected noise,
 * polled actions or per-HVAC lock-out durations move a step off the tile kernel that drsim_fused_info reports. */
#define DRSIM_ROUTE_FOUR_KERNEL 0          /* k_house + k_reduce + k_env + k_obs */
#define DRSIM_ROUTE_SHARD 1                /* k_shard */
#define DRSIM_ROUTE_FUSED 2                /* k_fused (rows staged in CTA-wide chunks) */
#define DRSIM_ROUTE_FUSED_DIRECT 3         /* k_fused_direct */
#define DRSIM_ROUTE_FUSED_TMA0 4           /* k_fused_tma<0> */
#define DRSIM_ROUTE_FUSED_TMA1 5           /* k_fused_tma<1> */
#define DRSIM_ROUTE_FUSED_TMA2 6           /* k_fused_tma<2> */
#define DRSIM_ROUTE_FUSED_ROWS_STAGED 7    /* k_fused_rows<staged> */
#define DRSIM_ROUTE_FUSED_ROWS_UNSTAGED 8  /* k_fused_rows<unstaged> */
#define DRSIM_ROUTE_SMALL 9                /* k_small */
#define DRSIM_ROUTE_SMALL_GEN 10           /* k_small_gen<double> */
int drsim_step_route(const drsim_t *h);

/* Per-cluster summary behind the reference's UI feed (ClientManagerService.update_data,
 * server/app/services/client_manager_service.py:147-197; description values :64-118): one launch,
 * d_out = device [R][DRSIM_SUMMARY_FIELDS] fp64 =
 * { locked HVACs, sum Ta, sum (Ta - target), sum |Ta - target|, sum Tm, sum target, running HVACs, N }.
 * Sums are taken in a fixed order (run-to-run identical). */
#define DRSIM_SUMMARY_FIELDS 8
int drsim_cluster_summary(drsim_t *h, double *d_out, void *stream);

/* Metrics.update (server/app/services/metrics_service.py:108-157) LITERALLY, for every cluster, after a step:
 * d_acc = device [R][DRSIM_REF_METRIC_FIELDS] fp64 running values =
 * { cumul_avg_reward, cumul_temp_offset, cumul_temp_error, max_temp_error, cumul_signal_offset, cumul_signal_error,
 *   cumul_squared_error_temp, cumul_OD_temp, cumul_signal, cumul_cons, cumul_squared_error_sig,
 *   cumul_squared_max_error_temp } (zero them = Metrics.initialize, :70-107); d_prev = device [R][3] fp64 =
 * { reg_signal, OD_temp, cluster_hvac_power } of the observation BEFORE the step (what the reference reads from
 * obs_dict, :150-152; the caller snapshots them); collect_squares = (time_step >= start_stats_from), :139,:154.
 * The reference's own expressions are kept, precedence slips included (temp_error = indoor_temp - target_temp /
 * nb_agents; signal error / nb_agents**2 once per agent), so the logged values are the reference's. */
#define DRSIM_REF_METRIC_FIELDS 12
int drsim_metrics_update(drsim_t *h, const double *d_prev, double *d_acc, int collect_squares, void *stream);

/* Host-side restatements of the env-level scalars, exported for CPU tests of the shared
 * __host__ __device__ code (utils/utils.py:42-117, environment.py:132-159). */
double drsim_host_solar_gain(int64_t epoch, double window_area, double shading_coeff);
double drsim_host_od_temp(int64_t epoch, double day_temp, double night_temp, double phase, double noise);
void drsim_host_civil(int64_t epoch, int32_t out7[7]); /* year, month, day, hour, minute, second, yday */
/* per-house update coefficients from (Ua, Ca, Cm, Hm, dt): out[0..5] = difference-form f32-path
 * coefficients (fp64), out[6..11] = r1, r2, A3, A4, e1, e2 of building.py:196-206 */
void drsim_host_thermal_coefs(double Ua, double Ca, double Cm, double Hm, int32_t dt, double out12[12]);
/* Philox4x32-10 block, for cross-checking the NumPy restatement */
void drsim_host_philox(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out4[4]);
/* the DRSIM_COMM_SAMPLE draw of one house: out[0..c) = its c sampled neighbours (global ids), the device's code.
 * Requires 1 <= c <= min(n_global - 1, DRSIM_MAX_SAMPLE_COMM); otherwise out is left untouched. */
void drsim_host_comm_sample(uint64_t seed, int64_t rep, int64_t house, int64_t draw, int64_t n_global, int c, int32_t *out);

const char *drsim_last_error(void);
int drsim_abi_version(void);
/* sizeof(drsim_config / drsim_host_state / drsim_ptrs / drsim_step_args / drsim_reset_args) */
int drsim_sizeof(int which);

#ifdef __cplusplus
}
#endif
#endif /* DRSIM_H_ */
