// drsim_api.cu -- C ABI of libdrsim.so (see include/drsim.h).  Host-side orchestration only:
// buffer carving, state injection / extraction, per-step path selection and kernel launches.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <type_traits>
#include <vector>

#include "drsim_kernels.cuh"
#include "drsim_shard.cuh"
#include "drsim_actor.cuh"

using namespace drsim;

static thread_local std::string g_err;

static int fail(int code, const std::string &msg) {
  g_err = msg;
  return code;
}

#define CU_TRY(expr)                                                                              \
  do {                                                                                            \
    cudaError_t e_ = (expr);                                                                      \
    if (e_ != cudaSuccess)                                                                        \
      return fail(DRSIM_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));              \
  } while (0)

namespace {

constexpr size_t kAlign = 256;

struct Carver {
  size_t off = 0;
  size_t take(size_t bytes) {
    const size_t o = off;
    off += (bytes + kAlign - 1) / kAlign * kAlign;
    return o;
  }
};

}  // namespace

struct drsim_handle {
  drsim_config cfg;
  SimParams p;
  int device = 0;
  int sm_count = 148;
  int real_bytes = 4;
  int obs_bytes = 4;   // observation-row element: real_bytes, or 2 (DRSIM_OBS_BF16)
  unsigned char *slab = nullptr;
  size_t slab_bytes = 0;
  // offsets inside the slab
  size_t o_t_air, o_t_mass, o_sso, o_flags, o_target, o_cap, o_coef[9], o_ratio[4], o_sub, o_reward, o_obs,
      o_actions, o_epoch, o_od, o_solar_next, o_solar_cur, o_signal, o_base, o_power, o_art, o_maxp, o_pen_sum,
      o_pen_max, o_rew_sig, o_tsi, o_metrics, o_partials, o_acc, o_comm, o_interp, o_in_od, o_in_perlin, o_in_ids,
      o_sched_od, o_sched_solar, o_sched_aux, o_sched_tsec, o_sched_rec, o_ptrpack, o_halo_out, o_halo_in;
  double cfg_artificial_ratio = 1.0;
  int fused_per_sm = 1;  // resident CTAs per SM of the fused kernel in use
  static constexpr int kSched = 64;  // steps pre-generated per k_schedule launch
  bool sched_valid = false;
  int64_t sched_base = 0;
  bool has_ratio = false, has_interp = false, has_comm = false;
  bool has_dur = false;   // per-HVAC lock-out durations were injected (plane o_dur is live): general path only
  size_t o_dur = 0;
  int chunks = 1;       // CTAs per cluster in the general path
  int obs_chunks = 1;   // k_obs CTAs per cluster
  bool fused_ok = false;   // plan_fused found a tile kernel for this shape (taken while fused_ready)
  bool fused_direct = false;   // ... whose tile's rows fit the staging buffer at once (k_fused_direct, not k_fused)
  FusedGeom geom{};
  int fused_grid = 0;
  int64_t step = 0;
  int t_since_interp = 0;  // host mirror of PowerGrid.time_since_last_interp (common to all replicas)
  int64_t launches = 0;
  // peer-memory exchange (house-sharded cluster over several GPUs)
  int peer_world = 1, peer_rank = 0;
  size_t o_inbox = 0, o_pflags = 0, o_peer_tab = 0, o_peer_err = 0;
  std::vector<void *> peer_mapped;  // cudaIpcOpenMemHandle results to close
  // sequence number of the house-sharded exchange (StepIn::xseq): +1 per sharded step, never reset
  int64_t xseq = 0;
  // single-kernel step of clusters larger than a tile / house-sharded clusters (drsim_shard.cuh)
  ShardGeom shard{};
  int shard_grid = 0, shard_capacity = 0;
  bool shard_ok = false;
  size_t o_sh_partll = 0, o_sh_envll = 0, o_sh_pearly = 0, o_pinbox = 0, o_rowll = 0;
  // drsim_rollout_transition: the step writes rewards / observation rows into the caller's transition slot
  void *obs_override = nullptr, *reward_override = nullptr;
  // small host inputs of drsim_step_host (actions / noise / ids of a small cluster) are staged in pinned mapped
  // memory and READ IN PLACE by the kernel: no copy-engine call for a handful of bytes
  unsigned char *h_in = nullptr, *h_in_dev = nullptr;
  // pinned + mapped snapshot for the dict API (drsim_snapshot)
  unsigned char *h_snap = nullptr, *h_snap_dev = nullptr;
  size_t snap_bytes = 0, snap_obs_off = 0;
  bool snap_next = false, snap_fused = false;   // transient: the next small-cluster step writes the host snapshot itself
  unsigned long long *actor_dbg = nullptr;   // DRSIM_ACTOR_DBG: phase stamps of CTA 0 of the last k_actor3 launch
  unsigned long long *shard_dbg = nullptr;   // DRSIM_SHARD_DBG: per-CTA time stamps of the last k_shard launch
  int *h_peer_err = nullptr, *h_peer_err_dev = nullptr;   // mapped: set by a kernel whose exchange wait timed out
  int *h_actor_err = nullptr, *h_actor_err_dev = nullptr; // mapped: set by k_actor3<SplitF16x3> when an operand overflows fp16
  int pending_interp = 0;  // decision of drsim_step_begin, consumed by drsim_step_finish
  StepIn pending_in{};
  // pinned staging for drsim_step_host; h_env_dev = the same memory as the device sees it (mapped)
  double *h_env = nullptr;
  double *h_env_dev = nullptr;
  // copy-engine mode of drsim_step_host: poisoned device staging plane for the actions, its own
  // non-blocking stream, and a mapped int the kernel sets when a poll times out
  size_t o_act_stage = 0;
  cudaStream_t copy_stream = nullptr;
  int *h_poll_err = nullptr, *h_poll_err_dev = nullptr;
  int host_actions_mode = 0;       // 0 auto, 1 always read in place (zero-copy), 2 always copy engine
  bool act_poll_next = false;      // the next fused step polls its action words (see StepIn::act_poll_err)
  double *mirror_next = nullptr;   // the next fused step writes its per-cluster results [R][4] straight to this mapped host buffer
  unsigned char *actor_image = nullptr;   // packed weight operands of drsim_policy_step (k_actor_pack)
  bool broken = false;             // a step was committed with missing inputs: refuse to step until state is re-injected
  int last_route = -1;             // StepRoute of the last step launched (drsim_step_route)

  template <typename T>
  T *at(size_t off) const {
    return reinterpret_cast<T *>(slab + off);
  }
};


template <typename real>
static Planes<real> make_planes(const drsim_handle *h) {
  Planes<real> pl{};
  pl.t_air = h->at<real>(h->o_t_air);
  pl.t_mass = h->at<real>(h->o_t_mass);
  pl.sso = h->at<int32_t>(h->o_sso);
  pl.flags = h->at<uint8_t>(h->o_flags);
  pl.target = h->at<real>(h->o_target);
  pl.cap = h->at<real>(h->o_cap);
  for (int k = 0; k < NCoef<real>::n; ++k) pl.coef[k] = h->at<real>(h->o_coef[k]);
  for (int k = 0; k < 4; ++k) pl.ratio[k] = h->has_ratio ? h->at<real>(h->o_ratio[k]) : nullptr;
  pl.interp_sub = h->has_interp ? h->at<uint8_t>(h->o_sub) : nullptr;
  pl.dur = h->has_dur ? h->at<int32_t>(h->o_dur) : nullptr;
  pl.reward = h->reward_override ? static_cast<real *>(h->reward_override) : h->at<real>(h->o_reward);
  pl.obs = !h->p.obs_dim ? nullptr : (h->obs_override ? h->obs_override : static_cast<void *>(h->slab + h->o_obs));
  pl.actions = h->at<uint8_t>(h->o_actions);
  pl.epoch = h->at<int64_t>(h->o_epoch);
  pl.od_temp = h->at<double>(h->o_od);
  pl.solar_next = h->at<double>(h->o_solar_next);
  pl.solar_cur = h->at<double>(h->o_solar_cur);
  pl.signal = h->at<double>(h->o_signal);
  pl.base_power = h->at<double>(h->o_base);
  pl.power = h->at<double>(h->o_power);
  pl.artificial_ratio = h->at<double>(h->o_art);
  pl.max_power = h->at<double>(h->o_maxp);
  pl.pen_sum = h->at<double>(h->o_pen_sum);
  pl.pen_max = h->at<double>(h->o_pen_max);
  pl.rew_sig = h->at<double>(h->o_rew_sig);
  pl.t_since_interp = h->at<int32_t>(h->o_tsi);
  pl.metrics = h->at<double>(h->o_metrics);
  pl.partials = h->at<double>(h->o_partials);
  pl.acc = h->at<double>(h->o_acc);
  pl.comm_table = h->has_comm ? h->at<int32_t>(h->o_comm) : nullptr;
  pl.interp_table = h->has_interp ? h->at<real>(h->o_interp) : nullptr;
  pl.halo_out = needs_halo(h->p) ? h->at<double>(h->o_halo_out) : nullptr;
  return pl;
}

static int fill_params(const drsim_config &c, SimParams &p, std::string &why) {
  if (c.abi_version != DRSIM_ABI_VERSION) { why = "abi_version mismatch"; return -1; }
  if (c.n_rep < 1 || c.n_house < 1) { why = "n_rep and n_house must be >= 1"; return -1; }
  if (c.precision != DRSIM_F32 && c.precision != DRSIM_F64) { why = "precision"; return -1; }
  if (c.dt < 1) { why = "dt must be >= 1 s"; return -1; }
  if (c.cop <= 0 || c.lockout_duration < 0) { why = "hvac properties"; return -1; }
  if (c.n_signal_terms < 0 || c.n_signal_terms > DRSIM_MAX_SIGNAL_TERMS) { why = "n_signal_terms"; return -1; }
  if (c.signal_mode == DRSIM_SIG_PERLIN && c.n_signal_terms < 1) { why = "perlin needs amplitude_ratios[0]"; return -1; }
  if (c.signal_mode == DRSIM_SIG_REGULAR_STEPS && c.period < 1) { why = "regular_steps needs period"; return -1; }
  if (c.nb_comm < 0) { why = "nb_comm"; return -1; }
  memset(&p, 0, sizeof(p));
  p.R = c.n_rep;
  p.N = c.n_house;
  p.Ns = (c.n_house + 3) / 4 * 4;
  p.dt = c.dt;
  p.house_offset = c.house_offset;
  p.n_global = c.n_house_global > 0 ? c.n_house_global : c.n_house;
  p.rep_offset = c.rep_offset;
  if (p.house_offset < 0 || p.house_offset + p.N > p.n_global) { why = "house_offset / n_house_global"; return -1; }
  p.deadband = c.deadband; p.cop = c.cop; p.latent = c.latent_cooling_fraction;
  p.window_area = c.window_area; p.shading = c.shading_coeff;
  p.lockout_duration = c.lockout_duration; p.solar_on = c.solar_gain;
  p.default_target = c.default_target_temp;
  p.dUa = c.default_Ua; p.dCa = c.default_Ca; p.dCm = c.default_Cm; p.dHm = c.default_Hm;
  p.dcap = c.default_cooling_capacity;
  p.day_temp = c.day_temp; p.night_temp = c.night_temp; p.temp_std = c.temp_std; p.phase = c.phase;
  p.alpha_temp = c.alpha_temp; p.alpha_sig = c.alpha_sig; p.nrs = c.norm_reg_sig;
  {  // rewards_calculator.py:155-165 via utils.py:4-23
    const double t0 = c.default_target_temp;
    const double v = t0 + 1, hi = t0 + 0.0 / 2;
    p.norm_temp = (v - hi) * (v - hi);
    const double lo = c.norm_reg_sig - 0.0 / 2, vs = 0.75 * c.norm_reg_sig;
    p.norm_sig = (lo - vs) * (lo - vs);
  }
  p.penalty_mode = c.penalty_mode;
  p.a_ind = c.alpha_ind_l2; p.a_cl2 = c.alpha_common_l2; p.a_cmax = c.alpha_common_max;
  p.base_mode = c.base_power_mode; p.interp_period = c.interp_update_period; p.interp_k = c.interp_nb_agents;
  p.signal_mode = c.signal_mode; p.n_terms = c.n_signal_terms; p.nb_octaves = c.nb_octaves;
  p.octaves_step = c.octaves_step; p.period = c.period;
  p.avg_power = c.avg_power_per_hvac; p.amp_per_hvac = c.amplitude_per_hvac;
  for (int k = 0; k < DRSIM_MAX_SIGNAL_TERMS; ++k) { p.amp[k] = c.amplitude_ratios[k]; p.periods[k] = c.periods[k]; }
  p.obs_layout = c.obs_layout; p.nb_comm = c.nb_comm; p.comm_mode = c.comm_mode; p.comm_per_rep = 0;
  p.st_solar = c.state_solar_gain; p.st_thermal = c.state_thermal; p.st_hvac = c.state_hvac;
  p.msg_thermal = c.message_thermal; p.msg_hvac = c.message_hvac;
  p.own_dim = 10 + (p.st_hvac ? 2 : 0) + (p.st_solar ? 1 : 0) + (p.st_thermal ? 5 : 0);
  p.msg_dim = 4 + (p.msg_thermal ? 4 : 0) + (p.msg_hvac ? 3 : 0);
  if (p.obs_layout == DRSIM_OBS_NONE) p.obs_dim = 0;
  else if (p.obs_layout == DRSIM_OBS_TARMAC) p.obs_dim = p.own_dim;
  else if (p.obs_layout == DRSIM_OBS_HAND_ENGINEERED) p.obs_dim = p.own_dim + p.nb_comm * p.msg_dim;
  else { why = "obs_layout"; return -1; }
  if (c.obs_dtype != DRSIM_OBS_F32 && c.obs_dtype != DRSIM_OBS_BF16) { why = "obs_dtype"; return -1; }
  if (c.obs_dtype == DRSIM_OBS_BF16 && c.precision != DRSIM_F32) {
    why = "obs_dtype = DRSIM_OBS_BF16 needs precision = DRSIM_F32 (the fp64 build keeps fp64 rows)";
    return -1;
  }
  if (c.obs_dtype == DRSIM_OBS_BF16 && p.obs_layout == DRSIM_OBS_NONE) {
    why = "obs_dtype = DRSIM_OBS_BF16 needs an observation layout (obs_layout = none writes no rows)";
    return -1;
  }
  if (c.comm_mode != DRSIM_COMM_RING && c.comm_mode != DRSIM_COMM_TABLE && c.comm_mode != DRSIM_COMM_SAMPLE) {
    why = "comm_mode";
    return -1;
  }
  if (p.obs_layout == DRSIM_OBS_HAND_ENGINEERED && p.nb_comm > 0 && p.N != p.n_global &&
      (p.comm_mode != DRSIM_COMM_RING || p.N < p.nb_comm)) {
    why = "house-sharded cluster with neighbour messages: only the ring (`neighbours`) mode is exchanged as a halo (table "
          "modes and `random_sample` are replicas only), and every shard must hold at least nb_comm houses";
    return -1;
  }
  if (c.policy == DRSIM_POLICY_GREEDY_MYOPIC && p.N != p.n_global) {
    why = "policy = DRSIM_POLICY_GREEDY_MYOPIC on a house-sharded cluster: the greedy scan sorts the whole cluster "
          "against its signal, so it runs on replicas only (n_house_local == n_house_global)";
    return -1;
  }
  if (p.comm_mode == DRSIM_COMM_SAMPLE && (p.nb_comm > DRSIM_MAX_SAMPLE_COMM || p.nb_comm > p.n_global - 1)) {
    why = "comm_mode = DRSIM_COMM_SAMPLE (`random_sample`) needs nb_comm <= min(n_house - 1, DRSIM_MAX_SAMPLE_COMM = " +
          std::to_string(DRSIM_MAX_SAMPLE_COMM) + "), got " + std::to_string(p.nb_comm);
    return -1;
  }
  if (p.base_mode == DRSIM_BASE_INTERPOLATION && (p.interp_k < 1 || p.interp_period < 1)) { why = "interp props"; return -1; }
  p.noise_mode = c.noise_mode; p.policy = c.policy; p.seed = c.seed;
  p.fd_dur = make_fastdiv((uint32_t)std::max(1, c.lockout_duration));
  p.fd_ns = make_fastdiv((uint32_t)p.Ns);
  p.inv_cop = 1.0 / p.cop; p.inv_nrs = 1.0 / p.nrs; p.inv_norm_temp = 1.0 / p.norm_temp;
  p.inv_n_global = 1.0 / (double)p.n_global; p.inv_norm_sig = 1.0 / p.norm_sig;
  p.hf.db = (float)p.deadband; p.hf.half_db = (float)(p.deadband / 2); p.hf.deadband = (float)p.deadband;
  p.hf.inv_cop = (float)p.inv_cop; p.hf.inv_nrs = (float)p.inv_nrs; p.hf.inv_n = (float)p.inv_n_global;
  p.hf.neg_inv_opl = (float)(-1.0 / (1.0 + p.latent)); p.hf.rew_scale = (float)(p.alpha_temp / p.norm_temp);
  if (c.lockout_duration < 1) { why = "lockout_duration must be >= 1 s"; return -1; }
  return 0;
}

// Template arguments of a handle's step kernels: real = the build (fp32 / fp64); O = observation-row element (real, or
// __nv_bfloat16 on an fp32 handle with DRSIM_OBS_BF16); S = the rows carry `random_sample` neighbours, drawn in the
// kernel (a compile-time flag, so the table / ring instantiations are the code they were; planning and routing ignore it)
template <typename Real, typename Obs, bool Sampled>
struct KernelTypes {
  using real = Real;
  using O = Obs;
  static constexpr bool S = Sampled;
};

// calls f(KernelTypes<...>{}) with the handle's template arguments: the one place they are derived from the handle
template <typename F>
static int with_kernel_types(const drsim_handle *h, F &&f) {
  const SimParams &p = h->p;
  const bool s = p.comm_mode == DRSIM_COMM_SAMPLE && p.obs_layout == DRSIM_OBS_HAND_ENGINEERED && p.nb_comm > 0;
  if (h->real_bytes == 8) return s ? f(KernelTypes<double, double, true>{}) : f(KernelTypes<double, double, false>{});
  if (h->obs_bytes == 2)
    return s ? f(KernelTypes<float, __nv_bfloat16, true>{}) : f(KernelTypes<float, __nv_bfloat16, false>{});
  return s ? f(KernelTypes<float, float, true>{}) : f(KernelTypes<float, float, false>{});
}

static void plan_fused(drsim_handle *h, int e_cap = 1 << 30) {
  const SimParams &p = h->p;
  h->fused_ok = false;
  if (h->cfg.path == DRSIM_PATH_SPLIT) return;
  if (p.Ns > kTileSlots || p.N != p.n_global) return;
  FusedGeom g{};
  g.envs_per_tile = std::max(1, std::min(std::min(p.R, kTileSlots / p.Ns), e_cap));
  g.n_tiles = (p.R + g.envs_per_tile - 1) / g.envs_per_tile;
  g.max_segs = p.Ns >= 128 ? 2 : (128 + p.Ns - 1) / p.Ns + 1;
  // bf16 rows of odd width: a 4-row group is 8 D bytes, not a multiple of the 16 a bulk store moves -- general path
  if (h->obs_bytes == 2 && (p.obs_dim & 1)) return;
  g.need_msg = (p.obs_layout == DRSIM_OBS_HAND_ENGINEERED && p.nb_comm > 0) ? 1 : 0;
  const int rb = h->real_bytes;
  const int slots = g.envs_per_tile * p.Ns;
  // staging is planned for rows of `real` whatever the row dtype: a bf16 handle then takes the kernel variant and tile
  // of the fp32 handle (its rows fill half of each staging slot), so its rows are the fp32 handle's rows, rounded
  const size_t row = (size_t)p.obs_dim * rb;
  auto layout = [&](bool direct, int chunk, bool allow_tma = true) {
    size_t off = 0;
    auto take = [&](size_t b) { size_t o = off; off += (b + 127) / 128 * 128; return (int)o; };
    g.off_msg = take((g.need_msg || !direct) ? (size_t)slots * 4 * rb * (direct ? 2 : 1) : 0);
    g.off_own = take(!direct ? (size_t)slots * 4 * rb : 0);
    g.off_env = take((size_t)g.envs_per_tile * 8 * rb * 2);
    g.off_wp = take((size_t)(kThreads / 32) * g.max_segs * kRed * sizeof(double) * 2);
    g.off_sold = take((size_t)g.envs_per_tile * sizeof(double) * 2);
    g.off_tile = (int)off;
    g.chunk_rows = chunk;
    off += ((size_t)chunk * row + 127) / 128 * 128;
    g.use_tma = (direct && rb == 4 && allow_tma) ? 1 : 0;
    if (g.use_tma) {
      g.off_in = take((size_t)kInPlanes * kTileSlots * 4);
      g.off_bar = take((size_t)(kThreads / 32) * 8 + 16 * 8);  // mbarriers + plane base pointers
      g.off_stage = take((size_t)g.envs_per_tile * sizeof(EnvStage) * 2);
    }
    g.smem_bytes = (int)off;
    return off;
  };
  // direct: the whole tile's rows staged at once (one TMA store per warp, rows from registers)
  layout(true, row ? slots : 0);
  // many tiny clusters per tile: the per-cluster schedule records of the TMA variant may not fit
  if (g.smem_bytes > 112 * 1024) layout(true, row ? slots : 0, false);
  if (g.smem_bytes > 112 * 1024) {
    // chunked staging; aim for >= 2 resident CTAs per SM, fall back to one big CTA
    if (row == 0) return;  // nothing to chunk: general path
    const size_t fixed = layout(false, 0) - 0;
    int chunk = 0;
    const size_t budgets[2] = {110 * 1024, 220 * 1024};
    for (size_t b : budgets) {
      if (fixed + 32 * row > b) continue;
      chunk = (int)std::min<size_t>((b - fixed - 256) / row, (size_t)slots) / 4 * 4;
      if (chunk >= 32) break;
    }
    if (chunk < 4) return;  // does not fit: general path
    layout(false, chunk);
  }
  // fp32 wide rows (hand-engineered layout that does not fit the direct staging): per-warp staging
  if (g.chunk_rows != (row ? slots : 0) && rb == 4 && g.need_msg && p.own_dim == 10 && p.msg_dim == 4 &&
      (p.obs_dim % 2) == 0 && slots % 4 == 0) {
    for (int staged = 1; staged >= 0; --staged) {
      FusedGeom w = g;
      size_t off = 0;
      auto take = [&](size_t b) { size_t o = off; off += (b + 127) / 128 * 128; return (int)o; };
      w.off_msg = take((size_t)slots * 16 * 2);
      w.off_own = take((size_t)slots * 16 * 2);
      w.off_env = take((size_t)g.envs_per_tile * 32 * 2);
      w.off_wp = take((size_t)(kThreads / 32) * g.max_segs * kRed * sizeof(double) * 2);
      w.off_sold = take((size_t)g.envs_per_tile * sizeof(double) * 2);
      w.off_tile = take((size_t)(kThreads / 32) * kRowGroup * row);
      w.off_stage = take((size_t)g.envs_per_tile * sizeof(EnvStage) * 2);
      w.in_stride = staged ? slots : 0;   // 0: inputs through registers (k_fused_rows<false>)
      w.off_in = staged ? take((size_t)11 * slots * 4 + (size_t)kThreads * 16) : 0;
      w.smem_bytes = (int)off;
      w.use_rows = 1;
      w.use_tma = 0;
      if (off <= 113 * 1024) { g = w; break; }
    }
  }
  h->geom = g;
  h->fused_direct = g.chunk_rows == g.envs_per_tile * p.Ns || p.obs_dim == 0;
  h->fused_ok = true;
}

static int plan_shard(drsim_handle *h);

// k_greedy sorts a cluster in shared memory: its width rounded up to a power of two, 24 bytes an entry
static int greedy_n2(const SimParams &p) {
  int n2 = 1;
  while (n2 < p.N) n2 <<= 1;
  return n2;
}

// shared-memory attributes of the tile kernel plan_fused chose (and its resident CTAs per SM), k_obs and k_greedy
template <typename K>
static int configure_step_kernels(drsim_handle *h, int &per_sm) {
  using real = typename K::real;
  using O = typename K::O;
  constexpr bool S = K::S;
  const FusedGeom &g = h->geom;
  if constexpr (sizeof(real) == 4) {
    if (h->fused_ok && g.use_rows) {
      auto kern = g.in_stride ? k_fused_rows<true, false, O, S> : k_fused_rows<false, false, O, S>;
      CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
      if (g.in_stride)
        CU_TRY(cudaFuncSetAttribute(k_fused_rows<true, true, O, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
      CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, g.smem_bytes));
    } else if (h->fused_ok && g.use_tma) {
      // (MODE 1 writes no messages: it is never launched with S)
      CU_TRY(cudaFuncSetAttribute(k_fused_tma<0, false, O, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
      CU_TRY(cudaFuncSetAttribute(k_fused_tma<1, false, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
      CU_TRY(cudaFuncSetAttribute(k_fused_tma<2, false, O, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
      CU_TRY(cudaFuncSetAttribute(k_fused_tma<0, true, O, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
      CU_TRY(cudaFuncSetAttribute(k_fused_tma<1, true, O>, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
      CU_TRY(cudaFuncSetAttribute(k_fused_tma<2, true, O, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
      CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fused_tma<0, false, O, S>, kThreads, g.smem_bytes));
    }
  }
  if (h->fused_ok && !g.use_rows && !g.use_tma) {
    auto kern = h->fused_direct ? k_fused_direct<real, O, S> : k_fused<real, O, S>;
    CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, g.smem_bytes));
  }
  const size_t obs_smem = (size_t)kObsChunk * h->p.obs_dim * sizeof(O);
  if (obs_smem > 48 * 1024)
    CU_TRY(cudaFuncSetAttribute(k_obs<real, O, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)obs_smem));
  if (h->p.policy == DRSIM_POLICY_GREEDY_MYOPIC) {
    constexpr int kGreedySmem = 200 * 1024;
    const size_t sm = (size_t)greedy_n2(h->p) * 24;
    if (sm > kGreedySmem) return fail(DRSIM_E_ARG, "greedy-myopic: cluster too large for the shared-memory sort");
    // the cap, whatever this handle's size: the attribute belongs to the kernel, so a smaller handle created later must
    // not lower it under a larger one's launch; and the kernel's static shared memory counts against the 48 KB default
    // too (2048 slots = exactly 48 KB of dynamic memory does not launch without the attribute)
    CU_TRY(cudaFuncSetAttribute(k_greedy<real>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGreedySmem));
  }
  return 0;
}

static int configure_kernels(drsim_handle *h) {
  int per_sm = 0;
  if (int rc = with_kernel_types(h, [&](auto k) { return configure_step_kernels<decltype(k)>(h, per_sm); })) return rc;
  if (h->fused_ok) {
    if (per_sm < 1) { h->fused_ok = false; }
    else { h->fused_grid = std::min(h->geom.n_tiles, per_sm * h->sm_count); h->fused_per_sm = per_sm; }
  }
  return 0;
}

extern "C" int drsim_create(const drsim_config *cfg, int device, drsim_t **out) {
  if (!cfg || !out) return fail(DRSIM_E_ARG, "null argument");
  *out = nullptr;
  SimParams p;
  std::string why;
  if (fill_params(*cfg, p, why)) return fail(DRSIM_E_ARG, "drsim_create: " + why);
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(DRSIM_E_DEVICE, std::string("drsim requires an sm_100 (B200) device, found ") + prop.name +
                                    " (cc " + std::to_string(prop.major) + "." + std::to_string(prop.minor) +
                                    "); there is no CPU or other-arch fallback");
  CU_TRY(cudaSetDevice(device));
  auto *h = new drsim_handle();
  h->cfg = *cfg;
  h->p = p;
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  h->real_bytes = cfg->precision == DRSIM_F64 ? 8 : 4;
  h->obs_bytes = cfg->obs_dtype == DRSIM_OBS_BF16 ? 2 : h->real_bytes;
  const int rb = h->real_bytes;
  h->has_ratio = p.st_thermal || p.msg_thermal;
  h->has_interp = p.base_mode == DRSIM_BASE_INTERPOLATION;
  h->has_comm = p.comm_mode == DRSIM_COMM_TABLE && p.nb_comm > 0;
  h->chunks = (p.Ns / 4 + kThreads - 1) / kThreads;
  h->obs_chunks = (p.Ns + kObsChunk - 1) / kObsChunk;
  h->t_since_interp = p.interp_period + 1;  // power_grid.py:64-66

  Carver cv;
  const size_t HP = (size_t)p.R * p.Ns;
  h->o_t_air = cv.take(HP * rb); h->o_t_mass = cv.take(HP * rb);
  h->o_sso = cv.take(HP * 4); h->o_flags = cv.take(HP);
  h->o_target = cv.take(HP * rb); h->o_cap = cv.take(HP * rb);
  const int nc = cfg->precision == DRSIM_F64 ? 9 : 6;
  for (int k = 0; k < nc; ++k) h->o_coef[k] = cv.take(HP * rb);
  if (h->has_ratio) for (int k = 0; k < 4; ++k) h->o_ratio[k] = cv.take(HP * rb);
  if (h->has_interp) { h->o_sub = cv.take(HP); h->o_interp = cv.take((size_t)DRSIM_INTERP_SUBTABLES * DRSIM_INTERP_SUBTABLE_LEN * rb); }
  h->o_reward = cv.take(HP * rb);
  h->o_dur = cv.take(HP * 4);
  h->o_obs = cv.take(HP * p.obs_dim * h->obs_bytes + 16);
  h->o_actions = cv.take(HP);
  h->o_act_stage = cv.take(HP);
  const size_t E8 = (size_t)p.R * 8;
  h->o_epoch = cv.take(E8);
  // contiguous env-output block (one D2H copy in drsim_step_host): power, signal, od, pen_sum, pen_max, rew_sig
  const size_t blk = cv.take(E8 * 6);
  h->o_power = blk; h->o_signal = blk + E8; h->o_od = blk + 2 * E8;
  h->o_pen_sum = blk + 3 * E8; h->o_pen_max = blk + 4 * E8; h->o_rew_sig = blk + 5 * E8;
  h->o_solar_next = cv.take(E8); h->o_solar_cur = cv.take(E8); h->o_base = cv.take(E8);
  h->o_art = cv.take(E8); h->o_maxp = cv.take(E8); h->o_tsi = cv.take((size_t)p.R * 4);
  h->o_metrics = cv.take(E8 * DRSIM_N_METRICS);
  h->o_partials = cv.take(E8 * h->chunks * kRed);
  h->o_acc = cv.take(E8 * DRSIM_N_ACC);
  if (h->has_comm) h->o_comm = cv.take((size_t)p.R * p.N * p.nb_comm * 4);  // room for per-replica tables
  h->o_in_od = cv.take(E8); h->o_in_perlin = cv.take(E8);
  h->o_in_ids = cv.take((size_t)p.R * std::max(1, p.interp_k) * 4);
  h->o_ptrpack = cv.take(256);
  {
    const int wmax = 16;  // ranks of one box
    h->o_inbox = cv.take((size_t)2 * wmax * p.R * DRSIM_N_ACC * 8);
    h->o_pflags = cv.take((size_t)2 * wmax * p.R * 8);
    h->o_peer_tab = cv.take((size_t)5 * wmax * 8);
    const size_t halo = needs_halo(p) ? (size_t)p.R * p.nb_comm * kHaloFields * 8 : 0;
    h->o_halo_out = cv.take(halo);
    h->o_halo_in = cv.take(2 * halo);
    h->o_peer_err = cv.take(8);
    h->o_sh_partll = cv.take((size_t)p.R * h->chunks * 16 * 8);
    h->o_sh_pearly = cv.take((size_t)p.R * h->chunks * 4 * 8);
    h->o_pinbox = cv.take((size_t)2 * wmax * p.R * 4 * 8);
    h->o_rowll = cv.take((size_t)2 * wmax * p.R * 16 * 8);
    h->o_sh_envll = cv.take((size_t)p.R * 16 * 8);
  }
  h->o_sched_od = cv.take(E8 * drsim_handle::kSched); h->o_sched_solar = cv.take(E8 * drsim_handle::kSched);
  h->o_sched_aux = cv.take(E8 * drsim_handle::kSched); h->o_sched_tsec = cv.take((size_t)p.R * 4 * drsim_handle::kSched);
  h->o_sched_rec = cv.take((size_t)p.R * sizeof(SchedRec) * drsim_handle::kSched);
  h->slab_bytes = cv.off;
  cudaError_t e = cudaMalloc(&h->slab, h->slab_bytes);
  if (e != cudaSuccess) {
    delete h;
    return fail(DRSIM_E_CUDA, std::string("cudaMalloc of ") + std::to_string(cv.off) + " bytes: " + cudaGetErrorString(e));
  }
  cudaMemset(h->slab, 0, h->slab_bytes);
  cudaMemset(h->slab + h->o_act_stage, 0xFF, HP);
  cudaHostAlloc(&h->h_env, E8 * 6 + 16, cudaHostAllocMapped);
  if (h->h_env && cudaHostGetDevicePointer(reinterpret_cast<void **>(&h->h_env_dev), h->h_env, 0) != cudaSuccess) {
    h->h_env_dev = nullptr;
    cudaGetLastError();
  }
  if (h->h_env && h->h_env_dev) {
    h->h_poll_err = reinterpret_cast<int *>(h->h_env + (size_t)p.R * 6);
    h->h_poll_err_dev = reinterpret_cast<int *>(h->h_env_dev + (size_t)p.R * 6);
    *h->h_poll_err = 0;
    h->h_peer_err = h->h_poll_err + 1;
    h->h_peer_err_dev = h->h_poll_err_dev + 1;
    *h->h_peer_err = 0;
    h->h_actor_err = h->h_poll_err + 2;
    h->h_actor_err_dev = h->h_poll_err_dev + 2;
    *h->h_actor_err = 0;
    if (cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
      h->copy_stream = nullptr;
      cudaGetLastError();
    }
  }
  if (const char *m = getenv("DRSIM_HOST_ACTIONS"))
    h->host_actions_mode = !strcmp(m, "zerocopy") ? 1 : (!strcmp(m, "dma") ? 2 : 0);
  plan_fused(h);
  int rc = configure_kernels(h);
  if (rc) { drsim_destroy(h); return rc; }
  const int e_max0 = p.Ns <= kTileSlots ? std::min(p.R, kTileSlots / p.Ns) : 0;
  if (e_max0 > 1 && cfg->path != DRSIM_PATH_SPLIT && p.N == p.n_global) {
    // Tile-size selection.  The grid is persistent (one wave of resident CTAs), so a step costs
    // ceil(n_tiles / resident) rounds of one tile each: with the largest tile that fits, BASELINE
    // config 3 (4096 x 100 houses) is 410 tiles on 296 CTAs = 2 rounds, the second 38 % full.  Pick the
    // clusters-per-tile count that minimises rounds x (tile slots + a fixed per-tile cost), planning
    // every candidate so that its kernel variant and shared-memory footprint are the real ones.
    const int e_max = e_max0;
    const long fixed_slots = 96;   // per-tile overhead (barriers, reductions, env records) in house-slot units
    double best_cost = -1;
    int best_e = e_max;
    for (int e = e_max; e >= 1; --e) {
      plan_fused(h, e);
      if (!h->fused_ok) continue;
      const FusedGeom &g = h->geom;
      const bool lean = g.use_rows || h->fused_direct;   // the chunked k_fused variant is markedly slower
      const int per_sm = rb == 8 ? 1 : std::max(1, std::min(2, (int)(226 * 1024 / std::max(1, g.smem_bytes))));
      const long resident = (long)per_sm * h->sm_count;
      const long rounds = (g.n_tiles + resident - 1) / resident;
      const double cost = (double)rounds * ((double)e * p.Ns + fixed_slots) * (lean ? 1.0 : 1.6);
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best_e = e; }
    }
    if (const char *force = getenv("DRSIM_TILE_ENVS")) {
      const int e = atoi(force);
      if (e >= 1) best_e = std::min(e, e_max);
    }
    plan_fused(h, best_e);
    rc = configure_kernels(h);
    if (rc) { drsim_destroy(h); return rc; }
    if (!h->fused_ok) {  // the chosen tile did not configure: back to the largest one
      plan_fused(h);
      rc = configure_kernels(h);
      if (rc) { drsim_destroy(h); return rc; }
    }
  }
  rc = plan_shard(h);
  if (rc) { drsim_destroy(h); return rc; }
  if (cfg->path == DRSIM_PATH_FUSED && !h->fused_ok) {
    drsim_destroy(h);
    return fail(DRSIM_E_ARG, "path=FUSED requested but the cluster does not fit a tile (N > 1024, sharded, or obs row too large)");
  }
  *out = h;
  return 0;
}

extern "C" int drsim_destroy(drsim_t *h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  for (void *ptr : h->peer_mapped) cudaIpcCloseMemHandle(ptr);
  if (h->slab) cudaFree(h->slab);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->h_env) cudaFreeHost(h->h_env);
  if (h->actor_image) cudaFree(h->actor_image);
  if (h->shard_dbg) cudaFree(h->shard_dbg);
  if (h->actor_dbg) cudaFree(h->actor_dbg);
  if (h->h_snap) cudaFreeHost(h->h_snap);
  if (h->h_in) cudaFreeHost(h->h_in);
  delete h;
  return 0;
}

extern "C" int drsim_clone(const drsim_t *src, drsim_t **out) {
  if (!src || !out) return fail(DRSIM_E_ARG, "null argument");
  drsim_t *h = nullptr;
  int rc = drsim_create(&src->cfg, src->device, &h);
  if (rc) return rc;
  CU_TRY(cudaMemcpy(h->slab, src->slab, src->slab_bytes, cudaMemcpyDeviceToDevice));
  h->p = src->p;
  h->step = src->step;
  h->t_since_interp = src->t_since_interp;
  h->sched_valid = src->sched_valid;
  h->sched_base = src->sched_base;
  h->xseq = src->xseq;
  h->has_dur = src->has_dur;
  h->shard = src->shard; h->shard_grid = src->shard_grid; h->shard_ok = src->shard_ok;
  *out = h;
  return 0;
}

extern "C" int drsim_buffers(drsim_t *h, drsim_ptrs *o) {
  if (!h || !o) return fail(DRSIM_E_ARG, "null argument");
  memset(o, 0, sizeof(*o));
  o->n_rep = h->p.R; o->n_house = h->p.N; o->house_stride = h->p.Ns; o->obs_dim = h->p.obs_dim;
  o->real_bytes = h->real_bytes; o->nb_comm = h->p.nb_comm;
  o->temp_is_deviation = h->real_bytes == 4 ? 1 : 0;
  o->obs_bytes = h->obs_bytes;
  o->t_air = h->slab + h->o_t_air; o->t_mass = h->slab + h->o_t_mass;
  o->sso = h->at<int32_t>(h->o_sso); o->flags = h->at<uint8_t>(h->o_flags);
  o->target = h->slab + h->o_target; o->cap = h->slab + h->o_cap;
  o->reward = h->slab + h->o_reward; o->obs = h->p.obs_dim ? h->slab + h->o_obs : nullptr;
  o->halo_out = needs_halo(h->p) ? h->at<double>(h->o_halo_out) : nullptr;
  o->actions = h->at<uint8_t>(h->o_actions);
  o->epoch = h->at<int64_t>(h->o_epoch);
  o->od_temp = h->at<double>(h->o_od); o->signal = h->at<double>(h->o_signal);
  o->base_power = h->at<double>(h->o_base); o->power = h->at<double>(h->o_power);
  o->solar = h->at<double>(h->o_solar_cur); o->pen_sum = h->at<double>(h->o_pen_sum);
  o->pen_max = h->at<double>(h->o_pen_max);
  o->comm_table = h->has_comm ? h->at<int32_t>(h->o_comm) : nullptr;
  o->metrics = h->at<double>(h->o_metrics);
  o->acc = h->at<double>(h->o_acc);
  o->rew_sig = h->at<double>(h->o_rew_sig);
  return 0;
}

// ---- state injection -----------------------------------------------------------------------
template <typename T, typename F>
static int upload_house(drsim_handle *h, size_t off, cudaStream_t s, F &&value) {
  const SimParams &p = h->p;
  std::vector<T> buf((size_t)p.R * p.Ns);
  for (int r = 0; r < p.R; ++r)
    for (int n = 0; n < p.Ns; ++n) buf[(size_t)r * p.Ns + n] = n < p.N ? (T)value((size_t)r * p.N + n) : (T)0;
  CU_TRY(cudaMemcpyAsync(h->slab + off, buf.data(), buf.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  CU_TRY(cudaStreamSynchronize(s));
  return 0;
}

template <typename T, typename SRC>
static int upload_env(drsim_handle *h, size_t off, cudaStream_t s, const SRC *src) {
  std::vector<T> buf(h->p.R);
  for (int r = 0; r < h->p.R; ++r) buf[r] = (T)src[r];
  CU_TRY(cudaMemcpyAsync(h->slab + off, buf.data(), buf.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  CU_TRY(cudaStreamSynchronize(s));
  return 0;
}

template <typename T, typename DST>
static int download_house(drsim_handle *h, size_t off, cudaStream_t s, DST *dst, int shift = 0, int mask = -1) {
  const SimParams &p = h->p;
  std::vector<T> buf((size_t)p.R * p.Ns);
  CU_TRY(cudaMemcpyAsync(buf.data(), h->slab + off, buf.size() * sizeof(T), cudaMemcpyDeviceToHost, s));
  CU_TRY(cudaStreamSynchronize(s));
  for (int r = 0; r < p.R; ++r)
    for (int n = 0; n < p.N; ++n) {
      const T v = buf[(size_t)r * p.Ns + n];
      dst[(size_t)r * p.N + n] = mask == -1 ? (DST)v : (DST)(((int)v >> shift) & mask);
    }
  return 0;
}

template <typename T, typename DST>
static int download_env(drsim_handle *h, size_t off, cudaStream_t s, DST *dst) {
  std::vector<T> buf(h->p.R);
  CU_TRY(cudaMemcpyAsync(buf.data(), h->slab + off, buf.size() * sizeof(T), cudaMemcpyDeviceToHost, s));
  CU_TRY(cudaStreamSynchronize(s));
  for (int r = 0; r < h->p.R; ++r) dst[r] = (DST)buf[r];
  return 0;
}

static int nearest3(double v) {  // grid {0.9, 1, 1.1}, np.argmin(|grid - v|) after clipping
  v = std::min(1.1, std::max(0.9, v));
  const double g[3] = {0.9, 1, 1.1};
  int best = 0;
  double bd = std::fabs(g[0] - v);
  for (int i = 1; i < 3; ++i) {
    const double d = std::fabs(g[i] - v);
    if (d < bd) { bd = d; best = i; }
  }
  return best;
}

template <typename real>
static int set_state_t(drsim_handle *h, const drsim_host_state *st, cudaStream_t s) {
  const SimParams &p = h->p;
  int rc;
#define UP_HOUSE(field, T, off)                                                           \
  if (st->field) {                                                                        \
    auto *src = st->field;                                                                \
    if ((rc = upload_house<T>(h, off, s, [src](size_t i) { return src[i]; }))) return rc; \
  }
  UP_HOUSE(target, real, h->o_target)
  if (st->t_air || st->t_mass) {
    // fp32 planes carry Ta - target / Tm - target (formed in fp64, then rounded once)
    std::vector<double> tgt;
    const double *tg = st->target;
    if (sizeof(real) == 4 && !tg) {
      tgt.resize((size_t)p.R * p.N);
      if ((rc = download_house<real>(h, h->o_target, s, tgt.data()))) return rc;
      tg = tgt.data();
    }
    const bool devi = sizeof(real) == 4;
    if (st->t_air) {
      auto *src = st->t_air;
      if ((rc = upload_house<real>(h, h->o_t_air, s, [=](size_t i) { return devi ? src[i] - tg[i] : src[i]; }))) return rc;
    }
    if (st->t_mass) {
      auto *src = st->t_mass;
      if ((rc = upload_house<real>(h, h->o_t_mass, s, [=](size_t i) { return devi ? src[i] - tg[i] : src[i]; }))) return rc;
    }
  }
  UP_HOUSE(cap, real, h->o_cap)
  UP_HOUSE(sso, int32_t, h->o_sso)
  if (st->lockout_duration) {
    // per-HVAC lock-out durations (v0/env/MA_DemandResponse.py:397-403): live only when some house differs from
    // the common duration -- the fused tile kernels and the plain k_shard variant share one duration
    bool differs = false;
    for (size_t i = 0; i < (size_t)p.R * p.N; ++i) {
      if (st->lockout_duration[i] < 1) return fail(DRSIM_E_ARG, "set_state: lockout_duration must be >= 1 s");
      differs = differs || st->lockout_duration[i] != p.lockout_duration;
    }
    UP_HOUSE(lockout_duration, int32_t, h->o_dur)
    if (differs != h->has_dur) {
      h->has_dur = differs;
      if ((rc = plan_shard(h))) return rc;   // (the plain variant is out while the plane is live)
    }
  }
#undef UP_HOUSE
  if (st->on || st->lockout) {
    if (!(st->on && st->lockout)) return fail(DRSIM_E_ARG, "set_state: on and lockout must be given together");
    auto *on = st->on;
    auto *lk = st->lockout;
    if ((rc = upload_house<uint8_t>(h, h->o_flags, s, [on, lk](size_t i) { return (on[i] ? 1 : 0) | (lk[i] ? 2 : 0); })))
      return rc;
  }
  if (st->Ua || st->Ca || st->Cm || st->Hm) {
    if (!(st->Ua && st->Ca && st->Cm && st->Hm)) return fail(DRSIM_E_ARG, "set_state: Ua, Ca, Cm, Hm must be given together");
    const size_t n = (size_t)p.R * p.N;
    std::vector<double> co_own;
    const double *co = st->thermal_coefs;
    if (!co) {
      co_own.resize(n * 12);
      for (size_t i = 0; i < n; ++i) thermal_coefs(st->Ua[i], st->Ca[i], st->Cm[i], st->Hm[i], p.dt, &co_own[i * 12]);
      co = co_own.data();
    }
    if (sizeof(real) == 4) {
      for (int k = 0; k < 6; ++k)
        if ((rc = upload_house<real>(h, h->o_coef[k], s, [co, k](size_t i) { return co[i * 12 + k]; }))) return rc;
    } else {
      const double *src[3] = {st->Ua, st->Ca, st->Hm};
      for (int k = 0; k < 3; ++k) {
        const double *a = src[k];
        if ((rc = upload_house<real>(h, h->o_coef[k], s, [a](size_t i) { return a[i]; }))) return rc;
      }
      for (int k = 0; k < 6; ++k)
        if ((rc = upload_house<real>(h, h->o_coef[3 + k], s, [co, k](size_t i) { return co[i * 12 + 6 + k]; }))) return rc;
    }
    if (h->has_ratio) {
      const double *src[4] = {st->Ua, st->Ca, st->Cm, st->Hm};
      const double dflt[4] = {p.dUa, p.dCa, p.dCm, p.dHm};
      for (int k = 0; k < 4; ++k) {
        const double *a = src[k];
        const double d = dflt[k];
        if ((rc = upload_house<real>(h, h->o_ratio[k], s, [a, d](size_t i) { return a[i] / d; }))) return rc;
      }
    }
    if (h->has_interp) {
      if (!st->cap) return fail(DRSIM_E_ARG, "set_state: interpolation needs cap together with the thermal parameters");
      auto *Ua = st->Ua; auto *Ca = st->Ca; auto *Cm = st->Cm; auto *Hm = st->Hm; auto *cap = st->cap;
      const SimParams pp = p;
      if ((rc = upload_house<uint8_t>(h, h->o_sub, s, [=](size_t i) {
             // interpolation.py:148-162, :227-235, :245-264 (key order Ua, Cm, Ca, Hm, then HVAC_power)
             const int iu = nearest3(Ua[i] / pp.dUa), icm = nearest3(Cm[i] / pp.dCm);
             const int ica = nearest3(Ca[i] / pp.dCa), ihm = nearest3(Hm[i] / pp.dHm);
             const double c = std::min(15000.0, std::max(10000.0, cap[i]));
             const int ihv = std::fabs(10000.0 - c) <= std::fabs(15000.0 - c) ? 0 : 1;
             return (((iu * 3 + icm) * 3 + ica) * 3 + ihm) * 2 + ihv;
           })))
        return rc;
    }
  }
#define UP_ENV(field, T, off) \
  if (st->field && (rc = upload_env<T>(h, off, s, st->field))) return rc;
  UP_ENV(epoch, int64_t, h->o_epoch)
  UP_ENV(od_temp, double, h->o_od)
  UP_ENV(signal, double, h->o_signal)
  UP_ENV(base_power, double, h->o_base)
  UP_ENV(power, double, h->o_power)
  UP_ENV(solar, double, h->o_solar_cur)
  UP_ENV(artificial_ratio, double, h->o_art)
  UP_ENV(max_power, double, h->o_maxp)
  UP_ENV(t_since_interp, int32_t, h->o_tsi)
#undef UP_ENV
  if (st->t_since_interp) h->t_since_interp = st->t_since_interp[0];
  if (st->epoch) {
    // solar gain of the NEXT step's datetime (building.py:176-181 uses the already-advanced time)
    std::vector<double> sn(p.R);
    for (int r = 0; r < p.R; ++r)
      sn[r] = p.solar_on ? solar_gain(civil_from_epoch(st->epoch[r] + p.dt), p.window_area, p.shading) : 0.0;
    if ((rc = upload_env<double>(h, h->o_solar_next, s, sn.data()))) return rc;
  }
  return 0;
}

extern "C" int drsim_set_state(drsim_t *h, const drsim_host_state *st, void *stream) {
  if (!h || !st) return fail(DRSIM_E_ARG, "null argument");
  // the interpolator fires for the whole handle at once (interp_decision): one counter, common to all replicas
  if (st->t_since_interp)
    for (int r = 1; r < h->p.R; ++r)
      if (st->t_since_interp[r] != st->t_since_interp[0])
        return fail(DRSIM_E_ARG, "set_state: t_since_interp must be the same on every replica (the interpolator fires "
                                 "for all replicas of a handle on the same step)");
  CU_TRY(cudaSetDevice(h->device));
  h->sched_valid = false;
  h->broken = false;
  auto s = (cudaStream_t)stream;
  return h->real_bytes == 8 ? set_state_t<double>(h, st, s) : set_state_t<float>(h, st, s);
}

// One D2H copy for the house planes and one for the env scalars (they are carved contiguously),
// then the requested members are unpacked on the host: a full snapshot costs two memcpys + one sync.
template <typename real>
static int get_state_t(drsim_handle *h, drsim_host_state *st, cudaStream_t s) {
  const SimParams &p = h->p;
  const size_t HP = (size_t)p.R * p.Ns;
  const bool want_house = st->t_air || st->t_mass || st->target || st->cap || st->sso || st->on || st->lockout;
  const bool want_env = st->epoch || st->od_temp || st->signal || st->base_power || st->power || st->solar ||
                        st->artificial_ratio || st->max_power || st->t_since_interp;
  const size_t h_lo = h->o_t_air, h_hi = h->o_cap + HP * sizeof(real);
  const size_t e_lo = h->o_epoch, e_hi = h->o_tsi + (size_t)p.R * 4;
  std::vector<unsigned char> hb, eb;
  if (want_house) {
    hb.resize(h_hi - h_lo);
    CU_TRY(cudaMemcpyAsync(hb.data(), h->slab + h_lo, hb.size(), cudaMemcpyDeviceToHost, s));
  }
  if (want_env) {
    eb.resize(e_hi - e_lo);
    CU_TRY(cudaMemcpyAsync(eb.data(), h->slab + e_lo, eb.size(), cudaMemcpyDeviceToHost, s));
  }
  CU_TRY(cudaStreamSynchronize(s));
  auto house = [&](size_t off) { return hb.data() + (off - h_lo); };
  auto env = [&](size_t off) { return eb.data() + (off - e_lo); };
  const bool devi = sizeof(real) == 4;
  const real *tgt = want_house ? reinterpret_cast<const real *>(house(h->o_target)) : nullptr;
  auto unpack_real = [&](size_t off, double *dst, bool add_target) {
    const real *src = reinterpret_cast<const real *>(house(off));
    for (int r = 0; r < p.R; ++r)
      for (int n = 0; n < p.N; ++n) {
        const size_t i = (size_t)r * p.Ns + n;
        dst[(size_t)r * p.N + n] = (double)src[i] + (add_target ? (double)tgt[i] : 0.0);
      }
  };
  if (st->t_air) unpack_real(h->o_t_air, st->t_air, devi);
  if (st->t_mass) unpack_real(h->o_t_mass, st->t_mass, devi);
  if (st->target) unpack_real(h->o_target, st->target, false);
  if (st->cap) unpack_real(h->o_cap, st->cap, false);
  if (st->sso || st->on || st->lockout) {
    const int32_t *sso = reinterpret_cast<const int32_t *>(house(h->o_sso));
    const uint8_t *fl = house(h->o_flags);
    for (int r = 0; r < p.R; ++r)
      for (int n = 0; n < p.N; ++n) {
        const size_t i = (size_t)r * p.Ns + n, o = (size_t)r * p.N + n;
        if (st->sso) st->sso[o] = sso[i];
        if (st->on) st->on[o] = fl[i] & 1u;
        if (st->lockout) st->lockout[o] = (fl[i] >> 1) & 1u;
      }
  }
  auto env_d = [&](size_t off, double *dst) {
    if (!dst) return;
    const double *src = reinterpret_cast<const double *>(env(off));
    for (int r = 0; r < p.R; ++r) dst[r] = src[r];
  };
  if (st->epoch) {
    const int64_t *src = reinterpret_cast<const int64_t *>(env(h->o_epoch));
    for (int r = 0; r < p.R; ++r) st->epoch[r] = src[r];
  }
  env_d(h->o_od, st->od_temp); env_d(h->o_signal, st->signal); env_d(h->o_base, st->base_power);
  env_d(h->o_power, st->power); env_d(h->o_solar_cur, st->solar); env_d(h->o_art, st->artificial_ratio);
  env_d(h->o_maxp, st->max_power);
  if (st->t_since_interp) {
    const int32_t *src = reinterpret_cast<const int32_t *>(env(h->o_tsi));
    for (int r = 0; r < p.R; ++r) st->t_since_interp[r] = src[r];
  }
  if (st->lockout_duration) {
    std::vector<int32_t> d(HP, p.lockout_duration);
    if (h->has_dur) {
      CU_TRY(cudaMemcpyAsync(d.data(), h->slab + h->o_dur, HP * 4, cudaMemcpyDeviceToHost, s));
      CU_TRY(cudaStreamSynchronize(s));
    }
    for (int r = 0; r < p.R; ++r)
      for (int n = 0; n < p.N; ++n) st->lockout_duration[(size_t)r * p.N + n] = d[(size_t)r * p.Ns + n];
  }
  return 0;
}

extern "C" int drsim_get_state(drsim_t *h, drsim_host_state *st, void *stream) {
  if (!h || !st) return fail(DRSIM_E_ARG, "null argument");
  CU_TRY(cudaSetDevice(h->device));
  auto s = (cudaStream_t)stream;
  return h->real_bytes == 8 ? get_state_t<double>(h, st, s) : get_state_t<float>(h, st, s);
}

extern "C" int drsim_set_comm_table(drsim_t *h, const int32_t *table, int per_replica, void *stream) {
  if (!h || !table) return fail(DRSIM_E_ARG, "null argument");
  if (!h->has_comm) return fail(DRSIM_E_STATE, "handle was not created with comm_mode = DRSIM_COMM_TABLE and nb_comm > 0");
  CU_TRY(cudaSetDevice(h->device));
  const SimParams &p = h->p;
  const size_t n = (size_t)(per_replica ? p.R : 1) * p.N * p.nb_comm;
  for (size_t i = 0; i < n; ++i)
    if (table[i] < 0 || table[i] >= p.n_global) return fail(DRSIM_E_ARG, "neighbour id out of range");
  auto s = (cudaStream_t)stream;
  CU_TRY(cudaMemcpyAsync(h->slab + h->o_comm, table, n * 4, cudaMemcpyHostToDevice, s));
  CU_TRY(cudaStreamSynchronize(s));
  h->p.comm_per_rep = per_replica ? 1 : 0;
  return 0;
}

extern "C" int drsim_set_interp_table(drsim_t *h, const double *sub, void *stream) {
  if (!h || !sub) return fail(DRSIM_E_ARG, "null argument");
  if (!h->has_interp) return fail(DRSIM_E_STATE, "handle was not created with base_power_mode = interpolation");
  CU_TRY(cudaSetDevice(h->device));
  const size_t n = (size_t)DRSIM_INTERP_SUBTABLES * DRSIM_INTERP_SUBTABLE_LEN;
  auto s = (cudaStream_t)stream;
  if (h->real_bytes == 8) {
    CU_TRY(cudaMemcpyAsync(h->slab + h->o_interp, sub, n * 8, cudaMemcpyHostToDevice, s));
    CU_TRY(cudaStreamSynchronize(s));
  } else {
    std::vector<float> f(n);
    for (size_t i = 0; i < n; ++i) f[i] = (float)sub[i];
    CU_TRY(cudaMemcpyAsync(h->slab + h->o_interp, f.data(), n * 4, cudaMemcpyHostToDevice, s));
    CU_TRY(cudaStreamSynchronize(s));
  }
  return 0;
}

// ---- stepping ------------------------------------------------------------------------------
static PeerCtx make_peer(const drsim_handle *h) {
  PeerCtx pc{};
  pc.world = h->peer_world;
  pc.rank = h->peer_rank;
  pc.inbox = reinterpret_cast<double *const *>(h->slab + h->o_peer_tab);
  pc.flags = reinterpret_cast<unsigned long long *const *>(h->slab + h->o_peer_tab + 16 * 8);
  pc.halo = reinterpret_cast<double *const *>(h->slab + h->o_peer_tab + 32 * 8);
  pc.pinbox = reinterpret_cast<unsigned long long *const *>(h->slab + h->o_peer_tab + 48 * 8);
  pc.rowll = nullptr;   // (k_shard without halo records switches the word protocol on, see launch_shard)
  pc.err = h->h_peer_err_dev ? h->h_peer_err_dev : reinterpret_cast<int *>(h->slab + h->o_peer_err);
  return pc;
}

// Launch with programmatic stream serialisation (PDL): the kernel may become resident while the
// previous kernel of the stream drains; it calls griddepcontrol.wait before it touches anything an
// earlier kernel wrote (see pdl_wait in drsim_kernels.cuh).
template <typename... KArgs, typename... Args>
static void launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- step routes ------------------------------------------------------------------------------
// The kernels a step runs on.  The values are the DRSIM_ROUTE_* of drsim.h (drsim_step_route).
enum class StepRoute : int {
  FourKernel = DRSIM_ROUTE_FOUR_KERNEL,   // k_house + k_reduce + k_env + k_obs: every step any other route cannot take
  Shard = DRSIM_ROUTE_SHARD,              // k_shard: clusters larger than a tile, house-sharded clusters, steps off the tile path
  FusedChunked = DRSIM_ROUTE_FUSED,       // k_fused: the tile's rows staged in CTA-wide chunks
  FusedDirect = DRSIM_ROUTE_FUSED_DIRECT,
  Tma0 = DRSIM_ROUTE_FUSED_TMA0,
  Tma1 = DRSIM_ROUTE_FUSED_TMA1,
  Tma2 = DRSIM_ROUTE_FUSED_TMA2,
  RowsStaged = DRSIM_ROUTE_FUSED_ROWS_STAGED,
  RowsUnstaged = DRSIM_ROUTE_FUSED_ROWS_UNSTAGED,
  Small = DRSIM_ROUTE_SMALL,
  SmallGen = DRSIM_ROUTE_SMALL_GEN,
};

// What a step is, as far as its route goes.  Known before make_in builds its StepIn: make_in sets the schedule
// pointers exactly when the step advances without injected noise.
struct StepKind {
  bool advance;    // a step of the power grid (not a refresh)
  bool interp;     // the interpolator fires on this step
  bool injected;   // outdoor-temperature or perlin noise comes from the caller (no scheduled records)
  bool poll;       // copy-engine actions, polled word by word by the kernel (drsim_step_host)
};

// the tile kernels run the handle's fused plan; per-HVAC lock-out durations take the general path while they differ
static bool fused_ready(const drsim_handle *h) { return h->fused_ok && !h->has_dur; }

static bool shard_plain(const drsim_handle *h) {
  return h->real_bytes == 4 && h->p.obs_dim == 10 && h->p.own_dim == 10 && !h->has_dur;
}

// can a step run as ONE k_shard launch?  (refreshes, the NCCL-gathered exchange and a halo without attached peers stay
// on the four-kernel path)
static bool shard_step_ok(const drsim_handle *h) {
  if (!h->shard_ok) return false;
  if (needs_halo(h->p) && h->peer_world < 2) return false;
  return true;
}

// Clusters that fit a warp (<= 32 plane slots) in a handful of replicas: the latency-oriented kernels (one house per
// lane) instead of the tile kernels (four houses per thread).  k_small (fp32) takes plain columns only; k_small_gen
// (the fp64 build: the drop-in Environment) any observation / message option.
static bool small_cluster(const drsim_handle *h) {
  const SimParams &p = h->p;
  if (getenv("DRSIM_NO_SMALL") || p.Ns > 32 || p.N != p.n_global || p.R > 256) return false;
  if (h->real_bytes == 8 || p.obs_dim == 0) return true;
  if (p.own_dim != 10 || (p.obs_dim & 1)) return false;
  const bool msgs = p.obs_layout == DRSIM_OBS_HAND_ENGINEERED && p.nb_comm > 0;
  return msgs ? (p.msg_dim == 4 && p.obs_dim == 10 + 4 * p.nb_comm) : p.obs_dim == 10;
}

// The tile kernel plan_fused chose.  k_fused_tma is specialised by the step: MODE 1 = plain 10-column rows without messages, one
// cluster per tile; MODE 2 = plain rows with messages, several clusters per tile (both for scheduled steps with external
// actions and the individual penalty); MODE 0 = everything else.
static StepRoute tile_route(const drsim_handle *h, bool scheduled) {
  const SimParams &p = h->p;
  const FusedGeom &g = h->geom;
  if (g.use_rows) return g.in_stride ? StepRoute::RowsStaged : StepRoute::RowsUnstaged;
  if (!g.use_tma) return h->fused_direct ? StepRoute::FusedDirect : StepRoute::FusedChunked;
  const bool plain = p.own_dim == 10 && p.msg_dim == 4 && (p.obs_dim % 2) == 0 && p.obs_dim > 0;
  const bool common = plain && scheduled && p.policy == DRSIM_POLICY_EXTERNAL && p.penalty_mode == DRSIM_PEN_INDIVIDUAL_L2;
  if (common && !g.need_msg && g.envs_per_tile == 1 && p.obs_dim == 10) return StepRoute::Tma1;
  if (common && g.need_msg && g.envs_per_tile > 1) return StepRoute::Tma2;
  return StepRoute::Tma0;
}

static bool is_tma(StepRoute r) { return r == StepRoute::Tma0 || r == StepRoute::Tma1 || r == StepRoute::Tma2; }

// the route of one step of this handle
static StepRoute step_route(const drsim_handle *h, const StepKind &k) {
  const SimParams &p = h->p;
  const bool scheduled = k.advance && !k.injected;
  if (fused_ready(h) && k.advance && !k.interp) {
    if ((h->real_bytes == 8 || (scheduled && !k.poll)) && small_cluster(h))
      return h->real_bytes == 8 ? StepRoute::SmallGen : StepRoute::Small;
    const StepRoute t = tile_route(h, scheduled);
    // k_fused_rows takes scheduled steps with the actions in the action plane (external, or written there by k_greedy)
    // and the individual penalty
    const bool rows_ok = scheduled && (p.policy == DRSIM_POLICY_EXTERNAL || p.policy == DRSIM_POLICY_GREEDY_MYOPIC) &&
                         p.penalty_mode == DRSIM_PEN_INDIVIDUAL_L2;
    if ((t == StepRoute::RowsStaged || t == StepRoute::RowsUnstaged) && !rows_ok) return StepRoute::FourKernel;
    return t;
  }
  if (k.advance && p.N == p.n_global && shard_step_ok(h)) return StepRoute::Shard;
  return StepRoute::FourKernel;
}

// ---- launches ---------------------------------------------------------------------------------
// greedy-myopic policy: k_greedy writes this step's actions into the action plane, ahead of the step kernels
static void launch_greedy(drsim_handle *h, const StepIn &in, cudaStream_t s) {
  const SimParams &p = h->p;
  if (p.policy != DRSIM_POLICY_GREEDY_MYOPIC || !in.advance || in.actions) return;
  const int n2 = greedy_n2(p);
  with_kernel_types(h, [&](auto k) {
    using real = typename decltype(k)::real;
    launch_pdl(k_greedy<real>, p.R, std::min(1024, std::max(32, n2)), (size_t)n2 * 24, s, make_planes<real>(h), p, n2);
    return 0;
  });
  h->launches++;
}

static int launch_house_phase(drsim_handle *h, const StepIn &in, cudaStream_t s) {
  const SimParams &p = h->p;
  with_kernel_types(h, [&](auto k) {
    using real = typename decltype(k)::real;
    const Planes<real> pl = make_planes<real>(h);
    launch_pdl(k_house<real>, p.R * h->chunks, kThreads, 0, s, pl, p, in, h->chunks);
    launch_pdl(k_reduce<real>, p.R, 128, 0, s, pl, p, in, h->chunks, make_peer(h));
    return 0;
  });
  h->launches += 2;
  CU_TRY(cudaGetLastError());
  return 0;
}

static int launch_env_phase(drsim_handle *h, const StepIn &in, const double *acc, int n_parts, cudaStream_t s) {
  const SimParams &p = h->p;
  PeerCtx pc = make_peer(h);
  if (acc || n_parts >= 0) pc.world = 1;  // explicit partials (or the handle's own): no peer wait
  with_kernel_types(h, [&](auto k) {
    using K = decltype(k);
    using real = typename K::real;
    const Planes<real> pl = make_planes<real>(h);
    launch_pdl(k_env<real>, (p.R + 127) / 128, 128, 0, s, pl, p, in, (const double *)(acc ? acc : pl.acc), acc ? n_parts : 1, pc);
    launch_pdl(k_obs<real, typename K::O, K::S>, p.R * h->obs_chunks, kObsChunk, (size_t)kObsChunk * p.obs_dim * h->obs_bytes,
               s, pl, p, in, h->obs_chunks);
    return 0;
  });
  h->launches += 2;
  CU_TRY(cudaGetLastError());
  return 0;
}

// ---- single-kernel step of the general path (drsim_shard.cuh) ---------------------------------
template <typename K>
static auto shard_kernel(const drsim_handle *h) {
  auto kern = k_shard<typename K::real, false, typename K::O, K::S>;
  if constexpr (sizeof(typename K::real) == 4) {
    if (shard_plain(h)) kern = k_shard<float, true, typename K::O>;   // (plain rows carry no messages)
  }
  return kern;
}

template <typename K>
static int plan_shard_as(drsim_handle *h) {
  using real = typename K::real;
  const SimParams &p = h->p;
  ShardGeom g{};
  h->shard_ok = false;
  if (getenv("DRSIM_NO_SHARD_KERNEL")) return 0;
  const int rb = (int)sizeof(real);
  if (h->obs_bytes == 2 && (p.obs_dim & 1)) return 0;   // bf16 rows of odd width: four-kernel path (see plan_fused)
  const bool plain = shard_plain(h);
  g.chunks = h->chunks;
  g.n_tiles = p.R * h->chunks;
  const int min_ctas = FusedOcc<real>::min_ctas;
  const size_t budget = min_ctas >= 2 ? 110 * 1024 : 200 * 1024;
  const size_t group = (size_t)kShardGroup * p.obs_dim * h->obs_bytes;
  g.nbuf = (size_t)(kThreads / 32) * 2 * group <= 48 * 1024 ? 2 : 1;
  // (also where the reducer parks the tile partials it collects: room for at least kReduceThreads of them)
  const size_t rows = plain ? (size_t)kTileSlots * 10 * 4
                            : std::max<size_t>((size_t)kReduceThreads * kRed * 8, (size_t)(kThreads / 32) * g.nbuf * group);
  g.part_cap = (int)std::min<size_t>(32 * kThreads, rows / (kRed * 8) / kReduceThreads * kReduceThreads);
  if (rows + 1024 > budget) return 0;   // rows too wide: four-kernel path
  g.tile_bytes = kTileSlots * (3 * rb + 5);
  g.off_rows = 0;
  g.off_saved = (int)((rows + 127) / 128 * 128);
  // tiles kept in shared memory between the phases: as many as a CTA owns, as long as min_ctas CTAs stay resident
  // per SM (the occupancy query knows the kernel's static shared memory and the per-CTA reservation)
  const int cap0 = std::min(g.n_tiles, min_ctas * h->sm_count);
  const int per_cta0 = (g.n_tiles + cap0 - 1) / cap0;
  g.t_smem = (int)std::min<size_t>(per_cta0, (budget - g.off_saved) / g.tile_bytes);
  if (const char *e = getenv("DRSIM_SHARD_TSMEM")) g.t_smem = std::max(0, std::min(g.t_smem, atoi(e)));
  const auto kern = shard_kernel<K>(h);
  int per_sm = 0;
  for (;; --g.t_smem) {
    g.smem_bytes = g.off_saved + g.t_smem * g.tile_bytes;
    CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, g.smem_bytes));
    if (per_sm >= min_ctas || g.t_smem == 0) break;
  }
  if (per_sm < 1) return 0;
  h->shard_capacity = per_sm * h->sm_count;
  // one cluster on the plain path: one more CTA, which owns no tile and only reduces (see `dedicated` in k_shard)
  const int extra = (plain && p.R == 1 && p.penalty_mode == DRSIM_PEN_INDIVIDUAL_L2) ? 1 : 0;
  h->shard_grid = std::min(g.n_tiles + extra, h->shard_capacity);
  h->shard = g;
  h->shard_ok = true;
  return 0;
}

static int plan_shard(drsim_handle *h) {
  return with_kernel_types(h, [&](auto k) { return plan_shard_as<decltype(k)>(h); });
}

template <typename K>
static void launch_shard(drsim_handle *h, StepIn in, cudaStream_t s) {
  const SimParams &p = h->p;
  if (needs_halo(p)) {   // the peers push their edge-house records into this rank's halo inbox (reduce_cluster)
    const int L = p.nb_comm / 2;
    const size_t per_rank = (size_t)p.R * p.nb_comm * kHaloFields;
    const double *inbox = h->at<double>(h->o_halo_in) + (size_t)(in.xseq & 1) * per_rank;
    in.halo_left = inbox;
    in.halo_right = inbox + (size_t)L * kHaloFields;
  }
  ShardCtx sc{};
  sc.partll = h->at<unsigned long long>(h->o_sh_partll);
  sc.pearly = h->at<unsigned long long>(h->o_sh_pearly);
  sc.pinbox = h->at<unsigned long long>(h->o_pinbox);
  sc.envll = h->at<unsigned long long>(h->o_sh_envll);
  sc.err = h->h_peer_err_dev ? h->h_peer_err_dev : reinterpret_cast<int *>(h->slab + h->o_peer_err);
  if (!h->shard_dbg && getenv("DRSIM_SHARD_DBG")) cudaMalloc(&h->shard_dbg, (size_t)h->shard_capacity * 16 * 8);
  sc.dbg = h->shard_dbg;
  PeerCtx pc = make_peer(h);
  if (!needs_halo(p)) pc.rowll = reinterpret_cast<unsigned long long *const *>(h->slab + h->o_peer_tab + 64 * 8);
  launch_pdl(shard_kernel<K>(h), h->shard_grid, kThreads, (size_t)h->shard.smem_bytes, s, make_planes<typename K::real>(h), p,
             in, h->shard, sc, pc);
}

static int exchange_error(const drsim_handle *h) {
  if (h->h_peer_err && *reinterpret_cast<volatile int *>(h->h_peer_err))
    return fail(DRSIM_E_STATE, "an in-kernel exchange wait timed out on an earlier step (a rank / CTA did not deliver its partial "
                               "sums within ~2 s): power, signal and rewards since then are not valid");
  return 0;
}

// the one kernel of a single-kernel route; grid = the persistent grid of the tile kernels
template <typename K>
static void launch_step_kernel(drsim_handle *h, StepRoute r, const StepIn &in, int grid, const SnapPtrs &snap,
                               unsigned char *snap_obs, cudaStream_t s) {
  using real = typename K::real;
  using O = typename K::O;
  constexpr bool S = K::S;
  const Planes<real> pl = make_planes<real>(h);
  const SimParams &p = h->p;
  const FusedGeom &g = h->geom;
  const int small_grid = (p.R + kSmallWarps - 1) / kSmallWarps;
  const bool poll = in.act_poll_err != nullptr;
  switch (r) {
    case StepRoute::Shard: launch_shard<K>(h, in, s); return;
    case StepRoute::FusedChunked: k_fused<real, O, S><<<grid, kThreads, g.smem_bytes, s>>>(pl, p, in, g); return;
    case StepRoute::FusedDirect: k_fused_direct<real, O, S><<<grid, kThreads, g.smem_bytes, s>>>(pl, p, in, g); return;
    default: break;
  }
  if constexpr (sizeof(real) == 8) {
    if (r == StepRoute::SmallGen)
      launch_pdl(k_small_gen<double, S>, small_grid, kSmallWarps * 32, 0, s, pl, p, in, snap, reinterpret_cast<double *>(snap_obs));
  } else {
    switch (r) {
      case StepRoute::Tma0:
        launch_pdl(poll ? k_fused_tma<0, true, O, S> : k_fused_tma<0, false, O, S>, grid, kThreads, g.smem_bytes, s, pl, p, in, g);
        break;
      case StepRoute::Tma1:
        launch_pdl(poll ? k_fused_tma<1, true, O> : k_fused_tma<1, false, O>, grid, kThreads, g.smem_bytes, s, pl, p, in, g);
        break;
      case StepRoute::Tma2:
        launch_pdl(poll ? k_fused_tma<2, true, O, S> : k_fused_tma<2, false, O, S>, grid, kThreads, g.smem_bytes, s, pl, p, in, g);
        break;
      case StepRoute::RowsStaged:
        launch_pdl(poll ? k_fused_rows<true, true, O, S> : k_fused_rows<true, false, O, S>, grid, kThreads, g.smem_bytes, s, pl,
                   p, in, g);
        break;
      case StepRoute::RowsUnstaged:   // (inputs through registers: never a polled step, see can_dma in step_host_impl)
        launch_pdl(k_fused_rows<false, false, O, S>, grid, kThreads, g.smem_bytes, s, pl, p, in, g);
        break;
      case StepRoute::Small: launch_pdl(k_small<O, S>, small_grid, kSmallWarps * 32, 0, s, pl, p, in); break;
      default: break;
    }
  }
}

static int snap_targets(drsim_handle *h, SnapPtrs &o, unsigned char **obs_dev);

// the launches of one step on route r
static int launch_step(drsim_handle *h, StepRoute r, const StepIn &in, int grid, cudaStream_t s) {
  h->last_route = (int)r;
  launch_greedy(h, in, s);
  if (r == StepRoute::FourKernel) {
    if (int rc = launch_house_phase(h, in, s)) return rc;
    return launch_env_phase(h, in, nullptr, 1, s);
  }
  SnapPtrs snap{};
  unsigned char *snap_obs = nullptr;
  if (r == StepRoute::SmallGen && h->snap_next) {   // k_small_gen writes the host snapshot itself
    if (int rc = snap_targets(h, snap, &snap_obs)) return rc;
    h->snap_fused = true;
  }
  with_kernel_types(h, [&](auto k) {
    launch_step_kernel<decltype(k)>(h, r, in, grid, snap, snap_obs, s);
    return 0;
  });
  h->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

template <typename real>
static void launch_schedule(drsim_handle *h, cudaStream_t s) {
  const Planes<real> pl = make_planes<real>(h);
  const int n = drsim_handle::kSched * h->p.R;
  k_schedule<real><<<(n + 127) / 128, 128, 0, s>>>(pl, h->p, h->step, drsim_handle::kSched, h->at<double>(h->o_sched_od),
                                                    h->at<double>(h->o_sched_solar), h->at<double>(h->o_sched_aux),
                                                    h->at<int32_t>(h->o_sched_tsec));
  k_schedule_pack<real><<<(n + 127) / 128, 128, 0, s>>>(pl, h->p, drsim_handle::kSched, h->at<double>(h->o_sched_od),
                                                         h->at<double>(h->o_sched_solar), h->at<double>(h->o_sched_aux),
                                                         h->at<int32_t>(h->o_sched_tsec), h->at<SchedRec>(h->o_sched_rec));
  h->launches += 2;
}

// When no noise is injected for this step the env-level time series comes from the pre-generated
// schedule (regenerated every kSched steps, off the per-step critical path).
static StepIn make_in(drsim_handle *h, const drsim_step_args *a, int advance, int do_interp, cudaStream_t s) {
  StepIn in{};
  if (a) { in.actions = a->actions; in.od_noise = a->od_noise; in.perlin = a->perlin; in.interp_ids = a->interp_ids; }
  in.host_env = h->mirror_next;
  in.act_poll_err = h->act_poll_next ? h->h_poll_err_dev : nullptr;
  in.step = h->step;
  in.xseq = h->xseq;
  in.advance = advance;
  in.do_interp = do_interp;
  if (advance && !in.od_noise && !in.perlin) {
    if (!h->sched_valid || h->step < h->sched_base || h->step >= h->sched_base + drsim_handle::kSched) {
      if (h->real_bytes == 8) launch_schedule<double>(h, s); else launch_schedule<float>(h, s);
      h->sched_base = h->step;
      h->sched_valid = true;
    }
    const size_t slot = (size_t)(h->step - h->sched_base) * h->p.R;
    in.sched_od = h->at<double>(h->o_sched_od) + slot;
    in.sched_solar = h->at<double>(h->o_sched_solar) + slot;
    in.sched_aux = h->at<double>(h->o_sched_aux) + slot;
    in.sched_tsec = h->at<int32_t>(h->o_sched_tsec) + slot;
    in.sched_rec = h->at<SchedRec>(h->o_sched_rec) + slot;
  }
  return in;
}

// decides whether the interpolator fires on this power-grid step (power_grid.py:150-161) and
// advances the host mirror of the counter
static int interp_decision(drsim_handle *h) {
  if (h->p.base_mode != DRSIM_BASE_INTERPOLATION) return 0;
  h->t_since_interp += h->p.dt;
  if (h->t_since_interp >= h->p.interp_period) { h->t_since_interp = 0; return 1; }
  return 0;
}

static int run_step(drsim_handle *h, const drsim_step_args *a, int advance, int do_interp, cudaStream_t s) {
  if (h->broken)
    return fail(DRSIM_E_STATE, "an earlier host-buffer step was committed with missing actions: re-inject the state "
                               "(drsim_set_state / drsim_reset) before stepping again");
  const StepKind kind{advance != 0, do_interp > 0, a && (a->od_noise || a->perlin), h->act_poll_next};
  const StepRoute r = step_route(h, kind);
  h->xseq++;
  const StepIn in = make_in(h, a, advance, do_interp, s);
  if (h->p.N != h->p.n_global) return fail(DRSIM_E_STATE, "house-sharded cluster: use drsim_step_begin / drsim_step_finish");
  const int rc = launch_step(h, r, in, h->fused_grid, s);
  // the packed schedule records chain each step to the one before it (previous signal / outdoor
  // temperature, base power): any step that did not follow the schedule ends their validity
  if (!(advance && in.sched_rec && do_interp <= 0)) h->sched_valid = false;
  return rc;
}

extern "C" int drsim_step(drsim_t *h, const drsim_step_args *args, void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  CU_TRY(cudaSetDevice(h->device));
  const int di = interp_decision(h);
  int rc = run_step(h, args, 1, di, (cudaStream_t)stream);
  if (!rc) h->step++;
  return rc;
}

// n_steps consecutive steps in one C call: a rollout under an on-device policy, or the replay of an
// action tape, without a host-language round trip per step (a 10-house cluster steps in ~2 us of GPU
// time; the per-call overhead of a scripting host is several times that)
extern "C" int drsim_run(drsim_t *h, const drsim_step_args *args, int n_steps, size_t action_stride, void *stream) {
  return drsim_run_tape(h, args, n_steps, action_stride, 0, stream);
}

extern "C" int drsim_run_tape(drsim_t *h, const drsim_step_args *args, int n_steps, size_t action_stride, int tape_planes,
                              void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  if (n_steps < 0) return fail(DRSIM_E_ARG, "n_steps must be >= 0");
  if (tape_planes < 0) return fail(DRSIM_E_ARG, "tape_planes must be >= 0");
  if (h->p.N != h->p.n_global) {
    // house-sharded cluster: every step is drsim_step_sharded (peer exchange inside the kernel, or one rank)
    if (h->peer_world < 2 && needs_halo(h->p))
      return fail(DRSIM_E_STATE, "house-sharded cluster with a halo: attach the peers first (drsim_ipc_attach)");
    drsim_step_args a{};
    if (args) a = *args;
    if (n_steps > 1 && (a.od_noise || a.perlin || a.interp_ids))
      return fail(DRSIM_E_ARG, "drsim_run: injected noise / sampled ids are per-step inputs (n_steps must be 1)");
    const uint8_t *tape = a.actions;
    for (int k = 0; k < n_steps; ++k) {
      a.actions = tape ? tape + (size_t)(tape_planes > 0 ? k % tape_planes : k) * action_stride : nullptr;
      const int rc = drsim_step_sharded(h, &a, stream);
      if (rc) return rc;
    }
    return 0;
  }
  drsim_step_args a{};
  if (args) a = *args;
  if (n_steps > 1 && (a.od_noise || a.perlin || a.interp_ids))
    return fail(DRSIM_E_ARG, "drsim_run: injected noise / sampled ids are per-step inputs (n_steps must be 1)");
  CU_TRY(cudaSetDevice(h->device));
  const uint8_t *tape = a.actions;
  // Action tape, or an on-device policy, on k_small / k_fused_tma / k_fused_rows: the step loop runs INSIDE the kernel
  // (StepIn::stream_steps), one launch per block of scheduled records.  Nothing a CTA reads of step k + 1 comes from
  // another CTA, so the steps of a block have no boundary between them (no launch ramp / tail, no grid-wide wait).
  // k_small keeps the state in registers and k_fused_tma runs a tile through all the steps before its next tile,
  // both on any number of tiles.  k_fused_rows takes the steps in turn over all its tiles, so a CTA needs at least two
  // (its next step's first tile must not be the tile it is still updating): it runs on min(resident CTAs, tiles / 2)
  // CTAs, and only when that costs at most a tenth of the resident grid.
  const SimParams &p = h->p;
  const StepRoute r = step_route(h, StepKind{true, false, false, false});
  const int sgrid = fused_ready(h) ? std::min(h->fused_grid, h->geom.n_tiles / 2) : 0;
  const bool loop_route = r == StepRoute::Small || is_tma(r) ||
                          (r == StepRoute::RowsStaged && tape && sgrid * 10 >= h->fused_grid * 9);
  const bool policy_ok = tape ? p.policy == DRSIM_POLICY_EXTERNAL
                              : (p.policy != DRSIM_POLICY_EXTERNAL && p.policy != DRSIM_POLICY_GREEDY_MYOPIC);
  const bool taped = n_steps > 1 && loop_route && policy_ok && p.base_mode == DRSIM_BASE_CONSTANT && !h->mirror_next &&
                     !h->act_poll_next && !h->obs_override && !h->reward_override && !h->broken && !getenv("DRSIM_NO_STREAM");
  int first = 0;
  if (taped) {
    const int grid = r == StepRoute::RowsStaged ? sgrid : h->fused_grid;
    a.actions = tape;
    while (first < n_steps) {
      h->xseq++;
      StepIn in = make_in(h, &a, 1, 0, (cudaStream_t)stream);   // (re)generates the schedule block when the step leaves it
      const int k = (int)std::min<int64_t>(n_steps - first, h->sched_base + drsim_handle::kSched - h->step);
      in.stream_steps = k;
      in.tape_planes = tape_planes;
      in.tape_first = first;
      in.tape_stride = action_stride;
      if (k == 1 && tape) in.actions = tape + (size_t)(tape_planes > 0 ? first % tape_planes : first) * action_stride;
      const int rc = launch_step(h, r, in, grid, (cudaStream_t)stream);
      if (rc) return rc;
      h->step += k;
      first += k;
    }
  }
  for (int k = first; k < n_steps; ++k) {
    a.actions = tape ? tape + (size_t)(tape_planes > 0 ? k % tape_planes : k) * action_stride : nullptr;
    const int di = interp_decision(h);
    const int rc = run_step(h, &a, 1, di, (cudaStream_t)stream);
    if (rc) return rc;
    h->step++;
  }
  return 0;
}

extern "C" int drsim_refresh(drsim_t *h, const drsim_step_args *args, int recompute_signal, void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  CU_TRY(cudaSetDevice(h->device));
  if (h->p.N != h->p.n_global)
    return fail(DRSIM_E_STATE, "drsim_refresh is not available on a house-sharded cluster");
  int di = -1;
  if (recompute_signal) di = interp_decision(h);
  return run_step(h, args, 0, di, (cudaStream_t)stream);
}

extern "C" int drsim_step_begin(drsim_t *h, const drsim_step_args *args, void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  CU_TRY(cudaSetDevice(h->device));
  h->pending_interp = interp_decision(h);
  h->xseq++;
  const StepIn in = make_in(h, args, 1, h->pending_interp, (cudaStream_t)stream);
  h->pending_in = in;
  h->last_route = (int)StepRoute::FourKernel;
  launch_greedy(h, in, (cudaStream_t)stream);
  return launch_house_phase(h, in, (cudaStream_t)stream);
}

static int step_finish_impl(drsim_handle *h, const double *acc, const double *halo, int n_parts, int rank,
                            cudaStream_t stream) {
  CU_TRY(cudaSetDevice(h->device));
  StepIn in = h->pending_in;
  if (acc && n_parts < 1) return fail(DRSIM_E_ARG, "n_parts must be >= 1");
  if (!acc && n_parts < 0 && h->peer_world < 2) return fail(DRSIM_E_STATE, "peer exchange requested but drsim_ipc_attach was not called");
  if (needs_halo(h->p)) {
    const SimParams &p = h->p;
    const int c = p.nb_comm, L = c / 2, H = c - L;
    const size_t per_rank = (size_t)p.R * c * kHaloFields;
    if (halo) {
      // gathered halo_out blocks of all ranks, rank order: the previous rank's LAST L houses are this
      // shard's left halo, the next rank's FIRST H houses its right halo
      if (n_parts < 2 || rank < 0 || rank >= n_parts) return fail(DRSIM_E_ARG, "halo_gathered needs n_parts >= 2 and a valid rank");
      in.halo_left = halo + (size_t)((rank + n_parts - 1) % n_parts) * per_rank + (size_t)H * kHaloFields;
      in.halo_right = halo + (size_t)((rank + 1) % n_parts) * per_rank;
    } else if (!acc && n_parts < 0) {
      const double *inbox = h->at<double>(h->o_halo_in) + (size_t)(in.xseq & 1) * per_rank;   // pushed by the peers
      in.halo_left = inbox;
      in.halo_right = inbox + (size_t)L * kHaloFields;
    } else {
      return fail(DRSIM_E_ARG, "this house-sharded cluster exchanges neighbour messages: pass the gathered halo records "
                               "(drsim_step_finish_gathered) or use the peer exchange");
    }
  }
  int rc = launch_env_phase(h, in, acc, n_parts, stream);
  if (!rc) h->step++;
  return rc;
}

extern "C" int drsim_step_finish(drsim_t *h, const drsim_step_args *args, const double *acc, int n_parts, void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  (void)args;
  return step_finish_impl(h, acc, nullptr, n_parts, -1, (cudaStream_t)stream);
}

// step_begin + step_finish(NULL, -1) in one call: the peer-memory exchange (or a single rank) needs nothing
// from the host between the two halves, and a house-sharded step is launch-bound (4 small kernels), so
// the second Python -> C round trip is worth saving
extern "C" int drsim_step_sharded(drsim_t *h, const drsim_step_args *args, void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  if (int rc = exchange_error(h)) return rc;
  if (shard_step_ok(h)) {
    // house update, reduction, peer push, wait, epilogue, rewards and observations in ONE launch (k_shard)
    CU_TRY(cudaSetDevice(h->device));
    const int di = interp_decision(h);
    h->xseq++;
    const StepIn in = make_in(h, args, 1, di, (cudaStream_t)stream);
    const int rc = launch_step(h, StepRoute::Shard, in, h->fused_grid, (cudaStream_t)stream);
    // the packed schedule records chain each step to the one before it: a step off the schedule ends their validity
    if (!(in.sched_rec && di <= 0)) h->sched_valid = false;
    if (!rc) h->step++;
    return rc;
  }
  int rc = drsim_step_begin(h, args, stream);
  if (rc) return rc;
  return step_finish_impl(h, nullptr, nullptr, h->peer_world > 1 ? -1 : 1, -1, (cudaStream_t)stream);
}

extern "C" int drsim_step_finish_gathered(drsim_t *h, const double *acc_gathered, const double *halo_gathered, int n_parts,
                                          int rank, void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  if (!acc_gathered) return fail(DRSIM_E_ARG, "acc_gathered is required");
  return step_finish_impl(h, acc_gathered, halo_gathered, n_parts, rank, (cudaStream_t)stream);
}

// Host-buffer step.  On the staged fused path the action transfer overlaps the kernel instead of
// preceding it: small planes (< 256 KB) are read in place from the caller's pinned (device-mapped)
// buffer by the kernel itself; larger ones travel as ONE linear copy-engine DMA, issued next to the
// kernel on the handle's own stream, into a poisoned staging plane that the kernel consumes word by
// word as it lands (measured on B200: the copy engine moves 2 MB at 51 GB/s, in-place reads from the
// SMs reach ~30 GB/s).  The per-cluster results are written by the kernel straight into the caller's
// pinned result buffer.  Pageable buffers, padded rows (N % 4 != 0) and every other step kind use
// explicit copies.
// ---- snapshot for the dict API ---------------------------------------------------------------
static size_t snap_layout(const drsim_handle *h, size_t off[8]) {
  const size_t HN = (size_t)h->p.R * h->p.N;
  size_t o = 0;
  auto take = [&](size_t b) { const size_t r = o; o += (b + 255) / 256 * 256; return r; };
  off[0] = take(HN * 8); off[1] = take(HN * 8); off[2] = take(HN * 8); off[3] = take(HN * 4); off[4] = take(HN);
  off[5] = take(HN); off[6] = take((size_t)h->p.R * kSnapEnv * 8); off[7] = take(HN * h->p.obs_dim * h->obs_bytes);
  return o;
}

// enqueues the snapshot kernel + the observation-row copy on `s`; the caller synchronises
// the mapped pinned snapshot buffer (allocated on first use) as the device sees it
static int snap_targets(drsim_handle *h, SnapPtrs &o, unsigned char **obs_dev) {
  size_t off[8];
  const size_t bytes = snap_layout(h, off);
  if (bytes > ((size_t)512 << 20)) return fail(DRSIM_E_ARG, "drsim_snapshot: more than 512 MB -- use the tensor views for clusters this large");
  if (!h->h_snap) {
    CU_TRY(cudaHostAlloc(reinterpret_cast<void **>(&h->h_snap), bytes, cudaHostAllocMapped));
    CU_TRY(cudaHostGetDevicePointer(reinterpret_cast<void **>(&h->h_snap_dev), h->h_snap, 0));
    h->snap_bytes = bytes;
  }
  unsigned char *d = h->h_snap_dev;
  o.t_air = reinterpret_cast<double *>(d + off[0]); o.t_mass = reinterpret_cast<double *>(d + off[1]);
  o.reward = reinterpret_cast<double *>(d + off[2]); o.sso = reinterpret_cast<int32_t *>(d + off[3]);
  o.on = d + off[4]; o.lockout = d + off[5]; o.env = reinterpret_cast<double *>(d + off[6]);
  if (obs_dev) *obs_dev = h->p.obs_dim ? d + off[7] : nullptr;
  return 0;
}

static int enqueue_snapshot(drsim_handle *h, cudaStream_t s) {
  size_t off[8];
  snap_layout(h, off);
  SnapPtrs o{};
  if (int rc = snap_targets(h, o, nullptr)) return rc;
  const SimParams &p = h->p;
  const long long n = std::max<long long>((long long)p.R * p.N, p.R);
  if (h->real_bytes == 8) k_snapshot<double><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(make_planes<double>(h), p, o);
  else k_snapshot<float><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(make_planes<float>(h), p, o);
  h->launches++;
  if (p.obs_dim) {
    const size_t row = (size_t)p.obs_dim * h->obs_bytes;
    if (p.Ns == p.N) CU_TRY(cudaMemcpyAsync(h->h_snap + off[7], h->slab + h->o_obs, (size_t)p.R * p.N * row, cudaMemcpyDeviceToHost, s));
    else CU_TRY(cudaMemcpy2DAsync(h->h_snap + off[7], (size_t)p.N * row, h->slab + h->o_obs, (size_t)p.Ns * row, (size_t)p.N * row, p.R,
                                  cudaMemcpyDeviceToHost, s));
  }
  CU_TRY(cudaGetLastError());
  return 0;
}

static void fill_snapshot_view(const drsim_handle *h, drsim_snapshot_view *v) {
  size_t off[8];
  snap_layout(h, off);
  const unsigned char *b = h->h_snap;
  v->n_rep = h->p.R; v->n_house = h->p.N; v->obs_dim = h->p.obs_dim; v->real_bytes = h->real_bytes;
  v->t_air = reinterpret_cast<const double *>(b + off[0]); v->t_mass = reinterpret_cast<const double *>(b + off[1]);
  v->reward = reinterpret_cast<const double *>(b + off[2]); v->sso = reinterpret_cast<const int32_t *>(b + off[3]);
  v->on = b + off[4]; v->lockout = b + off[5]; v->env = reinterpret_cast<const double *>(b + off[6]);
  v->obs = h->p.obs_dim ? b + off[7] : nullptr;
}

extern "C" int drsim_snapshot(drsim_t *h, drsim_snapshot_view *out, void *stream) {
  if (!h || !out) return fail(DRSIM_E_ARG, "null argument");
  CU_TRY(cudaSetDevice(h->device));
  if (int rc = enqueue_snapshot(h, (cudaStream_t)stream)) return rc;
  CU_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  fill_snapshot_view(h, out);
  return 0;
}

static int step_host_impl(drsim_t *h, const uint8_t *actions, const double *od_noise, const double *perlin,
                          const int32_t *interp_ids, double *env_out, void *reward_out, void *obs_out, void *stream,
                          drsim_snapshot_view *snap = nullptr) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  CU_TRY(cudaSetDevice(h->device));
  auto s = (cudaStream_t)stream;
  const SimParams &p = h->p;
  if (obs_out && !p.obs_dim) return fail(DRSIM_E_ARG, "drsim_step_host_full: obs_out given but the handle has obs_layout = none");
  drsim_step_args a{};
  const int tsi_before = h->t_since_interp;
  const int di = interp_decision(h);
  // The staged tile kernels (k_fused_tma, k_fused_rows) prefetch their inputs one tile ahead, so they can read the
  // actions in place from mapped host memory, and they mirror the per-cluster results into mapped host memory.
  // `polled` is the route of this step if its actions are polled; only k_fused_rows<unstaged> has no polling variant.
  const bool injected = od_noise || perlin;
  const StepRoute polled = step_route(h, StepKind{true, di > 0, injected, true});
  const bool staged = !injected && (is_tma(polled) || polled == StepRoute::RowsStaged || polled == StepRoute::RowsUnstaged);
  bool dma_poll = false;
  // small inputs: staged in the handle's pinned mapped page and read in place by the kernels (the call ends with a
  // stream synchronisation, so the page is free again when it returns)
  constexpr size_t kInAct = 8192, kInOd = 2048, kInIds = 4096;
  const bool small_in = (size_t)p.R * p.Ns <= kInAct && (size_t)p.R * 8 <= kInOd && (size_t)p.R * std::max(1, p.interp_k) * 4 <= kInIds;
  if (small_in && !h->h_in) {
    if (cudaHostAlloc(reinterpret_cast<void **>(&h->h_in), kInAct + 2 * kInOd + kInIds, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer(reinterpret_cast<void **>(&h->h_in_dev), h->h_in, 0) != cudaSuccess) {
      cudaGetLastError();
      if (h->h_in) cudaFreeHost(h->h_in);
      h->h_in = h->h_in_dev = nullptr;
    }
  }
  const bool in_place = small_in && h->h_in_dev;
  if (actions && in_place) {
    for (int r = 0; r < p.R; ++r) memcpy(h->h_in + (size_t)r * p.Ns, actions + (size_t)r * p.N, p.N);
    a.actions = h->h_in_dev;
  } else if (actions) {
    const uint8_t *mapped = nullptr;
    if (staged && p.Ns == p.N && (p.policy == DRSIM_POLICY_EXTERNAL)) {
      cudaPointerAttributes at{};
      if (cudaPointerGetAttributes(&at, actions) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer)
        mapped = static_cast<const uint8_t *>(at.devicePointer);
      else
        cudaGetLastError();
    }
    // Large action planes: ONE linear DMA into the poisoned staging plane on the handle's own stream,
    // launched next to the kernel, which consumes the words as they land (the copy engine moves ~50 GB/s,
    // in-place reads from the SMs ~30 GB/s).  Small ones are read in place (no copy start-up latency).
    // Needs the stream sync this call ends with (env_out), so the next copy cannot overtake this kernel.
    const size_t act_bytes = (size_t)p.R * p.N;
    const bool can_dma = mapped && h->copy_stream && h->h_poll_err_dev && env_out && h->h_env_dev &&
                         polled != StepRoute::RowsUnstaged;
    const bool want_dma = h->host_actions_mode == 2 || (h->host_actions_mode == 0 && act_bytes >= ((size_t)256 << 10));
    if (can_dma && want_dma) {
      CU_TRY(cudaMemcpyAsync(h->slab + h->o_act_stage, actions, act_bytes, cudaMemcpyHostToDevice, h->copy_stream));
      a.actions = h->at<uint8_t>(h->o_act_stage);
      dma_poll = true;
    } else if (mapped) {
      a.actions = mapped;
    } else {
      if (p.Ns == p.N)  // contiguous rows: one linear DMA instead of R row descriptors
        CU_TRY(cudaMemcpyAsync(h->slab + h->o_actions, actions, (size_t)p.R * p.N, cudaMemcpyHostToDevice, s));
      else
        CU_TRY(cudaMemcpy2DAsync(h->slab + h->o_actions, p.Ns, actions, p.N, p.N, p.R, cudaMemcpyHostToDevice, s));
      a.actions = h->at<uint8_t>(h->o_actions);
    }
  }
  if (od_noise && in_place) {
    memcpy(h->h_in + kInAct, od_noise, (size_t)p.R * 8);
    a.od_noise = reinterpret_cast<const double *>(h->h_in_dev + kInAct);
  } else if (od_noise) {
    CU_TRY(cudaMemcpyAsync(h->slab + h->o_in_od, od_noise, (size_t)p.R * 8, cudaMemcpyHostToDevice, s));
    a.od_noise = h->at<double>(h->o_in_od);
  }
  if (perlin && in_place) {
    memcpy(h->h_in + kInAct + kInOd, perlin, (size_t)p.R * 8);
    a.perlin = reinterpret_cast<const double *>(h->h_in_dev + kInAct + kInOd);
  } else if (perlin) {
    CU_TRY(cudaMemcpyAsync(h->slab + h->o_in_perlin, perlin, (size_t)p.R * 8, cudaMemcpyHostToDevice, s));
    a.perlin = h->at<double>(h->o_in_perlin);
  }
  if (interp_ids && in_place) {
    memcpy(h->h_in + kInAct + 2 * kInOd, interp_ids, (size_t)p.R * p.interp_k * 4);
    a.interp_ids = reinterpret_cast<const int32_t *>(h->h_in_dev + kInAct + 2 * kInOd);
  } else if (interp_ids) {
    CU_TRY(cudaMemcpyAsync(h->slab + h->o_in_ids, interp_ids, (size_t)p.R * p.interp_k * 4, cudaMemcpyHostToDevice, s));
    a.interp_ids = h->at<int32_t>(h->o_in_ids);
  }
  // Results: on the staged path the kernel writes [R][4] itself -- into the caller's buffer when that is
  // device-mapped pinned memory, else into the handle's mapped buffer (one small memcpy afterwards)
  double *mirror = nullptr;
  bool direct_out = false;
  if (staged && env_out) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, env_out) == cudaSuccess && at.type == cudaMemoryTypeHost && at.devicePointer) {
      mirror = static_cast<double *>(at.devicePointer);
      direct_out = true;
    } else {
      cudaGetLastError();
      mirror = h->h_env_dev;
    }
  }
  h->mirror_next = mirror;
  h->act_poll_next = dma_poll;
  h->snap_next = snap != nullptr;   // a small-cluster step (k_small_gen) writes the snapshot itself
  h->snap_fused = false;
  int rc = run_step(h, &a, 1, di, s);
  h->mirror_next = nullptr;
  h->act_poll_next = false;
  h->snap_next = false;
  if (rc) {
    if (dma_poll) {  // the kernel did not run: nothing consumed the copy, restore the poison
      cudaStreamSynchronize(h->copy_stream);
      cudaMemset(h->slab + h->o_act_stage, 0xFF, (size_t)p.R * p.Ns);
    }
    h->t_since_interp = tsi_before;
    return rc;
  }
  h->step++;
  // Environment.step returns the per-agent observations and rewards (environment.py:108): the full result goes
  // back to the caller's host buffers behind the kernel, ahead of the one stream synchronisation below
  if (reward_out) {
    if (p.Ns == p.N) CU_TRY(cudaMemcpyAsync(reward_out, h->slab + h->o_reward, (size_t)p.R * p.N * h->real_bytes, cudaMemcpyDeviceToHost, s));
    else CU_TRY(cudaMemcpy2DAsync(reward_out, (size_t)p.N * h->real_bytes, h->slab + h->o_reward, (size_t)p.Ns * h->real_bytes,
                                  (size_t)p.N * h->real_bytes, p.R, cudaMemcpyDeviceToHost, s));
  }
  if (obs_out) {
    const size_t row = (size_t)p.obs_dim * h->obs_bytes;
    if (p.Ns == p.N) CU_TRY(cudaMemcpyAsync(obs_out, h->slab + h->o_obs, (size_t)p.R * p.N * row, cudaMemcpyDeviceToHost, s));
    else CU_TRY(cudaMemcpy2DAsync(obs_out, (size_t)p.N * row, h->slab + h->o_obs, (size_t)p.Ns * row, (size_t)p.N * row, p.R,
                                  cudaMemcpyDeviceToHost, s));
  }
  if (snap && !h->snap_fused) {
    if (int rc2 = enqueue_snapshot(h, s)) return rc2;
  }
  if (env_out && mirror) {
    CU_TRY(cudaStreamSynchronize(s));
    if (dma_poll && *h->h_poll_err) {
      // the kernel substituted "off" for the words that never came: the state it committed is not the step the
      // caller asked for.  The handle is marked broken (every later step fails) until state is injected again.
      *h->h_poll_err = 0;
      cudaStreamSynchronize(h->copy_stream);
      cudaMemset(h->slab + h->o_act_stage, 0xFF, (size_t)p.R * p.Ns);
      h->broken = true;
      return fail(DRSIM_E_STATE, "drsim_step_host: the action copy did not arrive (poll timed out); the step was committed with "
                                 "missing actions -- re-inject the state (drsim_set_state / drsim_reset) before stepping again");
    }
    if (!direct_out) memcpy(env_out, h->h_env, (size_t)p.R * 4 * sizeof(double));
  } else if (env_out) {
    const size_t E8 = (size_t)p.R * 8;
    CU_TRY(cudaMemcpyAsync(h->h_env, h->slab + h->o_power, E8 * 6, cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    const double *v = h->h_env;   // six [R] planes: power, signal, od, pen_sum, pen_max, rew_sig
    const size_t sk = (size_t)p.R;
    for (int r = 0; r < p.R; ++r) {
      const double *q = v + r;
      const double ps = q[3 * sk], pm = q[4 * sk];
      double pen = ps;  // mean individual penalty == common_L2 value
      if (p.penalty_mode == DRSIM_PEN_COMMON_MAX) pen = pm;
      else if (p.penalty_mode == DRSIM_PEN_MIXTURE)
        pen = (p.a_ind * ps + p.a_cl2 * ps + p.a_cmax * pm) / (p.a_ind + p.a_cl2 + p.a_cmax);
      env_out[r * 4 + 0] = q[0];
      env_out[r * 4 + 1] = q[1 * sk];
      env_out[r * 4 + 2] = q[2 * sk];
      env_out[r * 4 + 3] = -(p.alpha_temp * pen / p.norm_temp + q[5 * sk]);
    }
  } else {
    CU_TRY(cudaStreamSynchronize(s));
  }
  if (snap) fill_snapshot_view(h, snap);
  return 0;
}

extern "C" int drsim_step_host_snapshot(drsim_t *h, const uint8_t *actions, const double *od_noise, const double *perlin,
                                        const int32_t *interp_ids, drsim_snapshot_view *out, void *stream) {
  if (!out) return fail(DRSIM_E_ARG, "null argument");
  return step_host_impl(h, actions, od_noise, perlin, interp_ids, nullptr, nullptr, nullptr, stream, out);
}

extern "C" int drsim_step_host(drsim_t *h, const uint8_t *actions, const double *od_noise, const double *perlin,
                               const int32_t *interp_ids, double *env_out, void *stream) {
  return step_host_impl(h, actions, od_noise, perlin, interp_ids, env_out, nullptr, nullptr, stream);
}

extern "C" int drsim_step_host_full(drsim_t *h, const uint8_t *actions, const double *od_noise, const double *perlin,
                                    const int32_t *interp_ids, double *env_out, void *reward_out, void *obs_out, void *stream) {
  return step_host_impl(h, actions, od_noise, perlin, interp_ids, env_out, reward_out, obs_out, stream);
}

template <typename real>
struct PtrPack {
  real *coef[9];
  real *ratio[4];
};

template <typename real>
static int reset_t(drsim_handle *h, const ResetArgs &a, cudaStream_t s) {
  const Planes<real> pl = make_planes<real>(h);
  PtrPack<real> host{};
  for (int k = 0; k < NCoef<real>::n; ++k) host.coef[k] = h->at<real>(h->o_coef[k]);
  for (int k = 0; k < 4; ++k) host.ratio[k] = h->has_ratio ? h->at<real>(h->o_ratio[k]) : nullptr;
  // the pointer tables live in the (otherwise unused at reset) injected-noise staging area
  PtrPack<real> *dev = reinterpret_cast<PtrPack<real> *>(h->slab + h->o_ptrpack);
  CU_TRY(cudaMemcpyAsync(dev, &host, sizeof(host), cudaMemcpyHostToDevice, s));
  const int64_t n = (int64_t)h->p.R * h->p.Ns;
  k_reset<real><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(pl, h->p, a, dev->coef, dev->ratio);
  h->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int drsim_reset(drsim_t *h, const drsim_reset_args *ra, void *stream) {
  if (!h || !ra) return fail(DRSIM_E_ARG, "null argument");
  if (ra->n_caps < 1 || ra->n_caps > 8) return fail(DRSIM_E_ARG, "n_caps must be in [1, 8]");
  if (!(ra->factor_low < 1.0 && 1.0 < ra->factor_high)) return fail(DRSIM_E_ARG, "need factor_low < 1 < factor_high");
  CU_TRY(cudaSetDevice(h->device));
  ResetArgs a{};
  a.seed = ra->seed; a.mode = ra->mode; a.randomize_date = ra->randomize_date; a.quirk_ua = ra->quirk_ua;
  a.n_caps = ra->n_caps; a.start_epoch = ra->start_epoch; a.init_air = ra->init_air_temp; a.init_mass = ra->init_mass_temp;
  a.std_target = ra->std_target_temp; a.f_lo = ra->factor_low; a.f_hi = ra->factor_high;
  for (int k = 0; k < 8; ++k) a.caps[k] = ra->caps[k];
  h->sched_valid = false;
  h->broken = false;
  h->step = 0;
  h->t_since_interp = h->p.interp_period + 1;
  if (h->has_dur) {   // the device reset draws no lock-out noise: back to the common duration
    h->has_dur = false;
    if (int rc = plan_shard(h)) return rc;
  }
  // artificial ratio: power_grid.py:46-49 draws ratio * range^(2u - 1); range == 1 in every shipped config
  {
    std::vector<double> ar(h->p.R, h->cfg_artificial_ratio);
    CU_TRY(cudaMemcpyAsync(h->slab + h->o_art, ar.data(), ar.size() * 8, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CU_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  }
  return h->real_bytes == 8 ? reset_t<double>(h, a, (cudaStream_t)stream) : reset_t<float>(h, a, (cudaStream_t)stream);
}

extern "C" int drsim_ipc_export(drsim_t *h, void *out96) {
  if (!h || !out96) return fail(DRSIM_E_ARG, "null argument");
  CU_TRY(cudaSetDevice(h->device));
  cudaIpcMemHandle_t mh;
  CU_TRY(cudaIpcGetMemHandle(&mh, h->slab));
  unsigned char *o = static_cast<unsigned char *>(out96);
  memcpy(o, &mh, 64);
  const uint64_t off[4] = {(uint64_t)h->o_inbox, (uint64_t)h->o_pflags, (uint64_t)h->o_halo_in, (uint64_t)h->o_pinbox};
  memcpy(o + 64, off, 32);
  return 0;
}

extern "C" int drsim_ipc_attach(drsim_t *h, int rank, int world, const void *handles96, void *stream) {
  if (!h || !handles96) return fail(DRSIM_E_ARG, "null argument");
  if (world < 1 || world > 16 || rank < 0 || rank >= world) return fail(DRSIM_E_ARG, "rank / world");
  CU_TRY(cudaSetDevice(h->device));
  const unsigned char *in = static_cast<const unsigned char *>(handles96);
  std::vector<uint64_t> tab(80, 0);
  for (int q = 0; q < world; ++q) {
    cudaIpcMemHandle_t mh;
    uint64_t off[4];
    memcpy(&mh, in + (size_t)q * 96, 64);
    memcpy(off, in + (size_t)q * 96 + 64, 32);
    unsigned char *base = nullptr;
    if (q == rank) base = h->slab;
    else {
      void *ptr = nullptr;
      CU_TRY(cudaIpcOpenMemHandle(&ptr, mh, cudaIpcMemLazyEnablePeerAccess));
      h->peer_mapped.push_back(ptr);
      base = static_cast<unsigned char *>(ptr);
    }
    tab[q] = (uint64_t)(uintptr_t)(base + off[0]);
    tab[16 + q] = (uint64_t)(uintptr_t)(base + off[1]);
    tab[32 + q] = (uint64_t)(uintptr_t)(base + off[2]);
    tab[48 + q] = (uint64_t)(uintptr_t)(base + off[3]);
    tab[64 + q] = (uint64_t)(uintptr_t)(base + off[3] + (h->o_rowll - h->o_pinbox));   // same slab layout on every rank (same R)
  }
  auto s = (cudaStream_t)stream;
  CU_TRY(cudaMemcpyAsync(h->slab + h->o_peer_tab, tab.data(), 80 * 8, cudaMemcpyHostToDevice, s));
  CU_TRY(cudaMemsetAsync(h->slab + h->o_pflags, 0, (size_t)2 * 16 * h->p.R * 8, s));
  CU_TRY(cudaMemsetAsync(h->slab + h->o_peer_err, 0, 8, s));
  CU_TRY(cudaStreamSynchronize(s));
  h->peer_world = world;
  h->peer_rank = rank;
  return 0;
}

// Same attachment for handles living in ONE process: raw device pointers instead of IPC handles (several
// shards on one GPU -- the kernels of the shards must then run concurrently, i.e. on different streams --
// or several GPUs driven by one process, peer access enabled here).
extern "C" int drsim_peer_attach_local(drsim_t *const *handles, int world, void *stream) {
  if (!handles) return fail(DRSIM_E_ARG, "null argument");
  if (world < 1 || world > 16) return fail(DRSIM_E_ARG, "world must be in [1, 16]");
  for (int q = 0; q < world; ++q)
    if (!handles[q]) return fail(DRSIM_E_ARG, "null handle");
  for (int i = 0; i < world; ++i) {
    drsim_handle *h = handles[i];
    CU_TRY(cudaSetDevice(h->device));
    std::vector<uint64_t> tab(80, 0);
    int same_device = 0;
    for (int q = 0; q < world; ++q) {
      const drsim_handle *o = handles[q];
      if (o->p.R != h->p.R) return fail(DRSIM_E_ARG, "drsim_peer_attach_local: the shards must have the same number of replicas");
      if (o->device == h->device) same_device++;
      else {
        const cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
          return fail(DRSIM_E_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
        cudaGetLastError();
      }
      tab[q] = (uint64_t)(uintptr_t)(o->slab + o->o_inbox);
      tab[16 + q] = (uint64_t)(uintptr_t)(o->slab + o->o_pflags);
      tab[32 + q] = (uint64_t)(uintptr_t)(o->slab + o->o_halo_in);
      tab[48 + q] = (uint64_t)(uintptr_t)(o->slab + o->o_pinbox);
      tab[64 + q] = (uint64_t)(uintptr_t)(o->slab + o->o_rowll);
    }
    auto s = (cudaStream_t)stream;
    CU_TRY(cudaMemcpyAsync(h->slab + h->o_peer_tab, tab.data(), 80 * 8, cudaMemcpyHostToDevice, s));
    CU_TRY(cudaMemsetAsync(h->slab + h->o_pflags, 0, (size_t)2 * 16 * h->p.R * 8, s));
    CU_TRY(cudaMemsetAsync(h->slab + h->o_peer_err, 0, 8, s));
    CU_TRY(cudaStreamSynchronize(s));
    h->peer_world = world;
    h->peer_rank = i;
    // shards that share a device share its SMs: every shard's persistent grid must be resident at once
    if (h->shard_ok) h->shard_grid = std::max(1, std::min(h->shard_grid, h->shard_capacity / same_device));
  }
  return 0;
}

extern "C" int drsim_peer_status(drsim_t *h, void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  int err = 0;
  CU_TRY(cudaMemcpyAsync(&err, h->slab + h->o_peer_err, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CU_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  if (h->h_peer_err) err |= *reinterpret_cast<volatile int *>(h->h_peer_err);
  if (err) return fail(DRSIM_E_STATE, "a peer-exchange wait timed out (a rank did not deliver its partial sums)");
  return 0;
}

static int policy_step_impl(drsim_t *h, const drsim_actor_net *net, uint64_t seed, const void *obs_in, uint8_t *actions_out,
                            float *prob_drawn, float *prob_on, void *stream);

using ActorKernel = void (*)(ActorArgs);

// the k_actor3 instantiation for PRE = pre 16-byte K chunks per producer thread: the smallest of S::kPre that holds them
template <class S, typename O>
static ActorKernel act3_kernel(int pre) {
  return pre <= S::kPre[0]   ? k_actor3<S, S::kPre[0], O>
         : pre <= S::kPre[1] ? k_actor3<S, S::kPre[1], O>
         : pre <= S::kPre[2] ? k_actor3<S, S::kPre[2], O>
                             : k_actor3<S, S::kPre[3], O>;
}

// the range flag of the f16x3 actor (k_actor3<SplitF16x3>), reported once and cleared
static int actor_range_error(drsim_t *h) {
  if (!h->h_actor_err || !*reinterpret_cast<volatile int *>(h->h_actor_err)) return 0;
  *reinterpret_cast<volatile int *>(h->h_actor_err) = 0;
  return fail(DRSIM_E_STATE, "f16x3 actor: an observation element or hidden activation of a live row was outside the fp16 range "
                             "(|x| >= 65520) in an earlier launch: its actions and probabilities are not valid; use precision = 1 (3xTF32)");
}

extern "C" int drsim_actor_status(drsim_t *h, void *stream) {
  if (!h) return fail(DRSIM_E_ARG, "null handle");
  CU_TRY(cudaSetDevice(h->device));
  CU_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return actor_range_error(h);
}

extern "C" int drsim_policy_step(drsim_t *h, const drsim_actor_net *net, uint64_t seed, float *prob_drawn, float *prob_on,
                                 void *stream) {
  return policy_step_impl(h, net, seed, nullptr, nullptr, prob_drawn, prob_on, stream);
}

// MAPPO.select_actions + Environment.step + MAPPO.store_transition (mappo.py:83-127, training_manager.py:224-240) for
// every agent of every replica, with the transition landing in the caller's device buffers: the actor reads
// state_t from slot->obs and writes a_t / p(a_t) into the slot, the step consumes a_t from there and writes r_t and
// state_{t+1} straight into the slot -- nothing is copied, nothing leaves the device.
extern "C" int drsim_rollout_transition(drsim_t *h, const drsim_actor_net *net, uint64_t seed, const drsim_rollout_slot *slot,
                                        void *stream) {
  if (!h || !net || !slot) return fail(DRSIM_E_ARG, "null argument");
  if (!slot->actions || !slot->prob || !slot->reward || !slot->next_obs)
    return fail(DRSIM_E_ARG, "drsim_rollout_transition: actions, prob, reward and next_obs are required");
  if (h->p.N != h->p.n_global) return fail(DRSIM_E_STATE, "drsim_rollout_transition: not available on a house-sharded cluster");
  auto misaligned = [](const void *q, uintptr_t a) { return (reinterpret_cast<uintptr_t>(q) & (a - 1)) != 0; };
  if (misaligned(slot->obs, 16) || misaligned(slot->reward, 16) || misaligned(slot->next_obs, 16) || misaligned(slot->actions, 4) ||
      misaligned(slot->prob, 4))
    return fail(DRSIM_E_ARG, "drsim_rollout_transition: obs / reward / next_obs must be 16-byte aligned, actions / prob 4-byte aligned");
  int rc = policy_step_impl(h, net, seed, slot->obs, slot->actions, slot->prob, nullptr, stream);
  if (rc) return rc;
  drsim_step_args a{};
  a.actions = slot->actions;
  h->obs_override = slot->next_obs;
  h->reward_override = slot->reward;
  rc = drsim_step(h, &a, stream);
  h->obs_override = nullptr;
  h->reward_override = nullptr;
  return rc;
}

static int policy_step_impl(drsim_t *h, const drsim_actor_net *net, uint64_t seed, const void *obs_in, uint8_t *actions_out,
                            float *prob_drawn, float *prob_on, void *stream) {
  if (!h || !net) return fail(DRSIM_E_ARG, "null argument");
  if (int rc = actor_range_error(h)) return rc;
  const SimParams &p = h->p;
  if (net->precision < 0 || net->precision > 2)
    return fail(DRSIM_E_ARG, "drsim_policy_step: precision must be 0 (tf32), 1 (tf32x3) or 2 (f16x3)");
  if (h->real_bytes != 4) return fail(DRSIM_E_ARG, "drsim_policy_step needs the fp32 build (observation rows are its input)");
  if (p.obs_dim < 1 || p.obs_dim > 64) return fail(DRSIM_E_ARG, "drsim_policy_step: obs_dim must be in [1, 64]");
  if (net->h1 < 1 || net->h1 > 128 || net->h2 < 1 || net->h2 > 128) return fail(DRSIM_E_ARG, "drsim_policy_step: h1, h2 in [1, 128]");
  if (!net->w1 || !net->b1 || !net->w2 || !net->b2 || !net->w3 || !net->b3) return fail(DRSIM_E_ARG, "drsim_policy_step: null weight pointer");
  const bool bf16 = h->obs_bytes == 2;
  if (bf16 && net->precision == 0)
    return fail(DRSIM_E_ARG, "drsim_policy_step: bfloat16 observation rows need precision = 1 (3xTF32) or 2 (f16x3); the "
                             "single-pass actor stages fp32 rows");
  CU_TRY(cudaSetDevice(h->device));
  ActorArgs a{};
  a.obs = obs_in ? obs_in : static_cast<const void *>(h->slab + h->o_obs);
  a.w1 = net->w1; a.b1 = net->b1; a.w2 = net->w2; a.b2 = net->b2; a.w3 = net->w3; a.b3 = net->b3;
  a.actions = actions_out ? actions_out : h->at<uint8_t>(h->o_actions);
  a.prob = prob_drawn; a.prob_on = prob_on;
  a.rows = (long long)p.R * p.Ns;
  a.Ns = p.Ns; a.N = p.N; a.D = p.obs_dim; a.h1 = net->h1; a.h2 = net->h2;
  int off = 0;
  auto take = [&](int b) { int o = off; off += (b + 127) / 128 * 128; return o; };
  auto up = [](int x, int m) { return (x + m - 1) / m * m; };
  a.seed = seed; a.step = h->step; a.rep_offset = p.rep_offset;
  const int tiles = (int)((a.rows + kActRows - 1) / kActRows);
  const cudaStream_t st = (cudaStream_t)stream;
  ActorKernel kern = k_actor2;
  int grid = std::min((tiles + 1) / 2, h->sm_count), threads = kAct2Threads;
  if (net->precision == 0) {
    // one spare K column per layer carries the bias (constant-one column in A), one spare output row regenerates the one
    a.K1 = up(a.D + 1, 8); a.N1 = up(a.h1 + 1, 16);
    a.K2 = up(a.h1 + 1, 8); a.N2 = up(a.h2 + 1, 16);
    a.K3 = up(a.h2 + 1, 8);
    if (a.N1 + a.N2 + kActN3 > 256)
      return fail(DRSIM_E_ARG, "drsim_policy_step: h1 + h2 too wide for two tile slots in tensor memory (N1 + N2 + 16 <= 256 "
                               "columns, N1 = h1 + 1 and N2 = h2 + 1 each rounded up to 16)");
    a.off_w1 = take(a.N1 * a.K1 * 4); a.off_w2 = take(a.N2 * a.K2 * 4);
    a.off_vec = take(kActN3 * a.K3 * 4);          // output-layer operand
    a.off_a1 = take(2 * kActRows * a.K1 * 4);     // two tile slots: observation operand (canonical layout)
    a.off_a2 = take(2 * ((kActRows * a.D * 4 + 127) / 128 * 128));   // two tile slots: raw row-major staging of the next tile
    a.off_bar = take(128);
    a.smem_bytes = off;
    if (a.smem_bytes > 227 * 1024) return fail(DRSIM_E_ARG, "drsim_policy_step: network / observation too wide for shared memory");
  } else {
    // k_actor3<S>: split operands (S = SplitTf32x3 for precision 1, SplitF16x3 for 2), one CTA per SM, warp-specialised; the
    // output layer runs in fp32 FMAs.  The widest f16x3 shape (D = 64, h1 = h2 = 128) takes 222,592 bytes of shared memory and
    // N1 + 2 N2 = 400 tensor-memory columns: no f16x3 width within the limits above is refused.
    auto layout = [&](auto split) -> int {
      using S = decltype(split);
      if (S::kRangeCheck && !h->h_actor_err_dev)
        return fail(DRSIM_E_CUDA, "drsim_policy_step: f16x3 needs mapped host memory for its range flag");
      a.K1 = up(a.D + 1, S::kK); a.N1 = up(a.h1 + 1, 16);
      a.K2 = up(a.h1 + 1, S::kK); a.N2 = up(a.h2, 16);
      if (S::kR1Sets * a.N1 + 2 * a.N2 > 512)
        return fail(DRSIM_E_ARG, "drsim_policy_step: h1 + h2 too wide for the split activations in tensor memory");
      a.off_w1 = take(a.N1 * a.K1 * S::kEl); a.off_w2 = take(a.N2 * a.K2 * S::kEl);
      a.w_bytes = off;                              // one weight block
      off = S::kWBlocks * a.w_bytes;
      if (S::kRangeCheck) a.off_sc = take(a.N1 * 4);   // 2^-s of the layer-1 columns
      a.off_w3 = take((2 * a.N2 + 2) * 4);          // output layer, fp32 (f16x3: carrying the layer-2 2^-s)
      a.off_a1 = off;                               // = size of the packed image
      take(2 * kActRows * a.K1 * S::kEl);           // observation operand, hi and lo (the next tile's rows wait in registers)
      a.off_bar = take(128);
      a.smem_bytes = off;
      if (a.smem_bytes > 227 * 1024)
        return fail(DRSIM_E_ARG, "drsim_policy_step: network / observation too wide for the 3xTF32 variant's shared memory "
                                 "(hi + lo weight halves); use precision = 0");
      const int pre = a.K1 / S::kK;                 // 16-byte K chunks per producer thread
      kern = bf16 ? act3_kernel<S, __nv_bfloat16>(pre) : act3_kernel<S, float>(pre);
      return 0;
    };
    if (int rc = net->precision == 1 ? layout(SplitTf32x3{}) : layout(SplitF16x3{})) return rc;
    a.range_err = h->h_actor_err_dev;
    grid = std::min(tiles, h->sm_count);
    threads = kAct3Threads;
    if (!h->actor_dbg && getenv("DRSIM_ACTOR_DBG")) {
      CU_TRY(cudaMalloc(&h->actor_dbg, 8 * 3 * 16 * 8));
      CU_TRY(cudaMemset(h->actor_dbg, 0, 8 * 3 * 16 * 8));
    }
    a.dbg = h->actor_dbg;
  }
  if (!h->actor_image) CU_TRY(cudaMalloc(&h->actor_image, 256 * 1024));
  a.image = h->actor_image;
  if (net->precision == 0) k_actor_pack<<<40, 512, 0, st>>>(a, h->actor_image);
  else if (net->precision == 1) k_actor_pack3x<<<40, 512, 0, st>>>(a, h->actor_image);
  else k_actor_pack3h<<<(a.N1 + a.N2 + 15) / 16, 512, 0, st>>>(a, h->actor_image);
  CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes));
  launch_pdl(kern, grid, threads, (size_t)a.smem_bytes, st, a);
  h->launches += 2;   // pack + actor
  CU_TRY(cudaGetLastError());
  return 0;
}

// diagnostics, not part of the documented ABI: per-CTA globaltimer stamps [grid][16] of the last k_shard launch
// (start, after the dependency wait, phase 1 done, arrival / reduction done, first broadcast values seen, end)
extern "C" int drsim_debug_shard_times(drsim_t *h, unsigned long long *host_out, int max_ctas) {
  if (!h || !h->shard_dbg || !host_out) return 0;
  const int n = std::min(max_ctas, h->shard_grid);
  cudaMemcpy(host_out, h->shard_dbg, (size_t)n * 128, cudaMemcpyDeviceToHost);
  return n;
}

// diagnostics, not part of the documented ABI: per-warp phase cycles of the k_fused_tma step loop [cta][warp][kTilePhases]
// (house update, own rows, barrier wait, fold + reward, row store, epilogue, tile-steps), summed over the launches since
// the last reset.  Returns the number of CTA slots copied; 0 unless the library was built with -DDRSIM_TILE_DBG.
extern "C" int drsim_debug_tile_phases(unsigned long long *host_out, int max_ctas, int reset) {
#ifdef DRSIM_TILE_DBG
  const int n = std::min(max_ctas, kTileDbgCtas);
  if (host_out && n > 0 && cudaMemcpyFromSymbol(host_out, g_tile_dbg, (size_t)n * sizeof(g_tile_dbg[0])) != cudaSuccess) return 0;
  void *dev = nullptr;
  if (reset && (cudaGetSymbolAddress(&dev, g_tile_dbg) != cudaSuccess || cudaMemset(dev, 0, sizeof(g_tile_dbg)) != cudaSuccess))
    return 0;
  return n;
#else
  (void)host_out; (void)max_ctas; (void)reset;
  return 0;
#endif
}

// diagnostics, not part of the documented ABI: clock64 stamps [tile < 8][producer, consumer, MMA warp][16] of CTA 0 of the
// last k_actor3 launch (DRSIM_ACTOR_DBG=1)
extern "C" int drsim_debug_actor_times(drsim_t *h, unsigned long long *host_out) {
  if (!h || !h->actor_dbg || !host_out) return 0;
  cudaMemcpy(host_out, h->actor_dbg, 8 * 3 * 16 * 8, cudaMemcpyDeviceToHost);
  return 8 * 3 * 16;
}

extern "C" int64_t drsim_launch_count(const drsim_t *h) { return h ? h->launches : 0; }

extern "C" int drsim_fused_info(const drsim_t *h, int32_t out[6]) {
  if (!h || !out) return fail(DRSIM_E_ARG, "null argument");
  const bool f = fused_ready(h);
  const StepRoute t = tile_route(h, true);
  int variant = 0;   // none, chunked, direct, staged (k_fused_tma), staged_rows (k_fused_rows)
  if (f) variant = t == StepRoute::FusedChunked ? 1 : t == StepRoute::FusedDirect ? 2 : is_tma(t) ? 3 : 4;
  out[0] = variant;
  out[1] = f ? h->geom.envs_per_tile : 0;
  out[2] = f ? h->geom.n_tiles : 0;
  out[3] = f ? h->fused_grid : 0;
  out[4] = f ? h->geom.smem_bytes : 0;
  out[5] = f ? h->fused_per_sm : 0;
  return 0;
}

extern "C" int drsim_step_route(const drsim_t *h) { return h ? h->last_route : -1; }

template <typename real>
static int summary_impl(drsim_t *h, double *d_out, cudaStream_t st) {
  const Planes<real> pl = make_planes<real>(h);
  k_summary<real><<<h->p.R, 256, 0, st>>>(pl, h->p, d_out);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int drsim_cluster_summary(drsim_t *h, double *d_out, void *stream) {
  if (!h || !d_out) return fail(DRSIM_E_ARG, "null argument");
  CU_TRY(cudaSetDevice(h->device));
  return h->real_bytes == 8 ? summary_impl<double>(h, d_out, (cudaStream_t)stream)
                            : summary_impl<float>(h, d_out, (cudaStream_t)stream);
}

template <typename real>
static int metrics_ref_impl(drsim_t *h, const double *prev, double *acc, int collect_sq, cudaStream_t st) {
  const Planes<real> pl = make_planes<real>(h);
  k_metrics_ref<real><<<h->p.R, 256, 0, st>>>(pl, h->p, prev, acc, collect_sq);
  h->launches++;
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int drsim_metrics_update(drsim_t *h, const double *d_prev, double *d_acc, int collect_squares, void *stream) {
  if (!h || !d_prev || !d_acc) return fail(DRSIM_E_ARG, "null argument");
  if (h->p.N != h->p.n_global) return fail(DRSIM_E_STATE, "drsim_metrics_update: not available on a house-sharded cluster");
  CU_TRY(cudaSetDevice(h->device));
  return h->real_bytes == 8 ? metrics_ref_impl<double>(h, d_prev, d_acc, collect_squares, (cudaStream_t)stream)
                            : metrics_ref_impl<float>(h, d_prev, d_acc, collect_squares, (cudaStream_t)stream);
}

// ---- host-side debug entry points ----------------------------------------------------------
extern "C" double drsim_host_solar_gain(int64_t epoch, double window_area, double shading_coeff) {
  return solar_gain(civil_from_epoch(epoch), window_area, shading_coeff);
}
extern "C" double drsim_host_od_temp(int64_t epoch, double day_temp, double night_temp, double phase, double noise) {
  return od_temp_model(civil_from_epoch(epoch), day_temp, night_temp, phase, noise);
}
extern "C" void drsim_host_civil(int64_t epoch, int32_t out7[7]) {
  const Civil c = civil_from_epoch(epoch);
  out7[0] = c.year; out7[1] = c.month; out7[2] = c.day; out7[3] = c.hour; out7[4] = c.minute; out7[5] = c.second;
  out7[6] = c.yday;
}
extern "C" void drsim_host_thermal_coefs(double Ua, double Ca, double Cm, double Hm, int32_t dt, double out12[12]) {
  thermal_coefs(Ua, Ca, Cm, Hm, dt, out12);
}
extern "C" int drsim_comm_sample(drsim_t *h, int64_t draw, int32_t *d_out, void *stream) {
  if (!h || !d_out) return fail(DRSIM_E_ARG, "null argument");
  const SimParams &p = h->p;
  if (p.comm_mode != DRSIM_COMM_SAMPLE || p.nb_comm < 1)
    return fail(DRSIM_E_STATE, "drsim_comm_sample: the handle was not created with comm_mode = DRSIM_COMM_SAMPLE and nb_comm > 0");
  CU_TRY(cudaSetDevice(h->device));
  const int64_t n = (int64_t)p.R * p.N;
  k_comm_sample<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p, (uint32_t)(draw < 0 ? h->step : draw), d_out);
  CU_TRY(cudaGetLastError());
  return 0;
}

extern "C" int64_t drsim_step_count(const drsim_t *h) { return h ? h->step : -1; }

extern "C" void drsim_host_comm_sample(uint64_t seed, int64_t rep, int64_t house, int64_t draw, int64_t n_global, int c,
                                       int32_t *out) {
  if (!out || c < 1 || c > DRSIM_MAX_SAMPLE_COMM || c > n_global - 1 || house < 0 || house >= n_global) return;
  CommSampler smp(seed, (uint32_t)rep, (uint32_t)house, (uint32_t)draw, (uint32_t)n_global);
  for (int k = 0; k < c; ++k) out[k] = smp.next();
}

extern "C" void drsim_host_philox(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out4[4]) {
  const U4 r = philox4x32_10(seed, c0, c1, c2, c3);
  out4[0] = r.x; out4[1] = r.y; out4[2] = r.z; out4[3] = r.w;
}

extern "C" const char *drsim_last_error(void) { return g_err.c_str(); }
extern "C" int drsim_abi_version(void) { return DRSIM_ABI_VERSION; }
extern "C" int drsim_sizeof(int which) {
  switch (which) {
    case 0: return (int)sizeof(drsim_config);
    case 1: return (int)sizeof(drsim_host_state);
    case 2: return (int)sizeof(drsim_ptrs);
    case 3: return (int)sizeof(drsim_step_args);
    case 4: return (int)sizeof(drsim_reset_args);
    default: return -1;
  }
}
