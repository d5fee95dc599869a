// drsim_shard.cuh -- ONE persistent kernel for the step of clusters that do not fit a tile: a
// cluster of more than 1024 houses, and above all ONE very large cluster split by houses across
// the GPUs of a box (BASELINE config 5, SURVEY 8e row 2).
//
// It replaces the four launches k_house -> k_reduce -> k_env -> k_obs of the general path by one
// grid of resident CTAs (grid <= resident capacity, so every CTA is on an SM from the start); a CTA
// owns a contiguous run of 1024-house tiles:
//
//   phase 1  the CTA updates its tiles (hvac.py:43-64, building.py:141-222), keeps the post-update
//            state of its first tiles in shared memory and writes each tile's partial sums; then ONE
//            fence and one atomic per cluster it touched ARRIVE its tiles at the cluster's counter;
//   reduce   the CTA whose arrival completes cluster r combines the tile partials -- same chunk
//            geometry and combine order as k_house / k_reduce, so the sums are bit-identical to the
//            four-kernel path -- and, on a house-sharded cluster, stores this rank's row (and the halo
//            records of the shard's edge houses) straight into every peer's inbox over NVLink
//            (cluster.py:73-89 is the sum being distributed);
//   env      one thread waits (bounded) for the rows of all ranks, combines them in rank order, runs
//            the env epilogue (environment.py:87-106) and PUBLISHES the cluster's broadcast values
//            under a flag stamped with the exchange sequence number;
//   phase 2  every CTA waits for the flag of its tile's cluster and writes rewards and observation
//            rows (rewards_calculator.py:135-181, utils/norm.py:71-218).  PLAIN (fp32, 10-column rows
//            without neighbour messages -- the config-5 layout): every thread finishes the 4 houses it
//            updated, rows go through a whole-tile staging buffer and leave with one TMA bulk store per
//            warp.  Otherwise: one house per lane, 32-row groups, one TMA bulk store per group.
//
// Nothing crosses a kernel boundary inside the step: reduction, collective and the consumers of the
// reduced values are one launch.  Phase 1 never waits, so every arrival / push eventually happens and
// the waits of the env threads and of phase 2 cannot deadlock; all spins are bounded (~2 s) and
// report through ShardCtx::err / PeerCtx::err.
#pragma once

#include "drsim_kernels.cuh"

namespace drsim {

constexpr int kShardGroup = 32;    // rows per warp-level TMA store of the generic phase 2 (one row per lane)
constexpr int kShardBatch = 4;     // tiles whose partials a CTA publishes together (one CTA barrier per batch)
constexpr int kShardFinish = 4;    // clusters a CTA completes at a time (reduce all, then one lane per cluster finishes)

struct ShardGeom {
  int chunks;       // 1024-house tiles per cluster: the chunk geometry of k_house (fixes the partial sums)
  int n_tiles;      // R * chunks
  int t_smem;       // tiles per CTA whose post-update state stays in shared memory between the phases
  int nbuf;         // generic phase 2: row-group staging buffers per warp (1 or 2)
  int tile_bytes;   // bytes of one saved tile
  int off_saved;    // [t_smem] saved tiles
  int off_rows;     // PLAIN: [1024][D] floats; generic: [warps][nbuf][kShardGroup][D] reals
  int part_cap;     // tile partials the row staging area can park during the reduction (multiple of kReduceThreads)
  int smem_bytes;
};

struct ShardCtx {
  unsigned long long *partll;  // [R * chunks][16] tile partials as self-validating words (PartLL)
  unsigned long long *pearly;  // [R * chunks][4] EARLY tile power (see the pre-pass in k_shard), one 32-byte record each
  unsigned long long *pinbox;  // this handle's own early cluster-power inbox [2][world][R][4] (what PeerCtx::pinbox[rank] points at)
  // [R][16] self-validating words: the 7 broadcast values of cluster r as doubles, each split into two
  // (tag << 32 | 32 data bits) words, tag = low half of StepIn::xseq.  A consumer polls the 14 words with ONE
  // coalesced load and has the values the moment all tags match -- no separate flag, no second round trip.
  unsigned long long *envll;
  int *err;                    // set when a wait timed out
  unsigned long long *dbg;     // diagnostics (DRSIM_SHARD_DBG): [grid][16] globaltimer stamps of thread 0, or NULL
};

template <typename real>
struct ShardSaved {
  real *ta, *tm, *tg;
  int *sso;
  uint8_t *flags;
  DRSIM_D ShardSaved(unsigned char *base) {
    ta = reinterpret_cast<real *>(base);
    tm = ta + kTileSlots;
    tg = tm + kTileSlots;
    sso = reinterpret_cast<int *>(tg + kTileSlots);
    flags = reinterpret_cast<uint8_t *>(sso + kTileSlots);
  }
};

// one thread: publish cluster r's broadcast values (reals are exactly representable as doubles)
template <typename real>
DRSIM_D void shard_publish(const ShardCtx &sc, const StepIn &in, int r, const EnvBroadcast<real> &e) {
  const double v[7] = {(double)e.power_n, (double)e.signal_n, (double)e.solar_n, (double)e.od_n,
                       (double)e.rew_sig, (double)e.pen_common, (double)e.pen_max};
  unsigned long long *dst = sc.envll + (size_t)r * 16;
  const unsigned long long tag = (unsigned long long)(uint32_t)in.xseq << 32;
  __threadfence();   // release: whatever the consumers read after seeing these words (other CTAs' state, halo) is ordered before them
#if defined(__CUDA_ARCH__)
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(v[k]);
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(dst + 2 * k), "l"(tag | (bits & 0xffffffffull)) : "memory");
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(dst + 2 * k + 1), "l"(tag | (bits >> 32)) : "memory");
  }
  // (whole 128-byte line written: no partially valid sector for the L2 to complete from HBM under the pollers)
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(dst + 14), "l"(tag) : "memory");
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(dst + 15), "l"(tag) : "memory");
#endif
}

// whole warp: bounded wait for cluster r's broadcast values
template <typename real>
DRSIM_D EnvBroadcast<real> shard_wait_env(const ShardCtx &sc, const StepIn &in, int r, int lane) {
  const unsigned long long *src = sc.envll + (size_t)r * 16;
  const uint32_t tag = (uint32_t)in.xseq;
  unsigned long long w = 0;
  const long long t0 = clock64();
  for (;;) {
#if defined(__CUDA_ARCH__)
    if (lane < 14) asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(src + lane) : "memory");
#endif
    if (__all_sync(0xffffffffu, lane >= 14 || (uint32_t)(w >> 32) == tag)) break;
    if (__any_sync(0xffffffffu, clock64() - t0 > 4000000000ll)) {   // ~2 s: give up, flag the error
      if (lane == 0) *sc.err = 1;
      break;
    }
#if defined(__CUDA_ARCH__)
    __nanosleep(100);
#endif
  }
  __threadfence();   // acquire side of the release in shard_publish
  const uint32_t half = (uint32_t)w;
  double v[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    const uint32_t lo = __shfl_sync(0xffffffffu, half, 2 * k), hi = __shfl_sync(0xffffffffu, half, 2 * k + 1);
    v[k] = __longlong_as_double((long long)(((unsigned long long)hi << 32) | lo));
  }
  EnvBroadcast<real> e;
  e.power_n = (real)v[0]; e.signal_n = (real)v[1]; e.solar_n = (real)v[2]; e.od_n = (real)v[3];
  e.rew_sig = (real)v[4]; e.pen_common = (real)v[5]; e.pen_max = (real)v[6];
  return e;
}

// whole warp, scheduled step with constant base power: the cluster power straight from the early inbox -- lane q
// polls rank q's record, the ranks are folded in rank order (the order of env_cluster) -- and every other
// broadcast value from the step's packed record.  No reducer-side combine / publish hop in between.
template <typename real>
DRSIM_D EnvBroadcast<real> shard_wait_power(const ShardCtx &sc, const SimParams &p, const StepIn &in, int world, int r, int lane) {
  const uint32_t tag = (uint32_t)in.xseq;
  const unsigned long long *rec = sc.pinbox + ((((size_t)(in.xseq & 1) * world + min(lane, world - 1)) * p.R + r) * 4);
  const SchedRec &c = in.sched_rec[r];
  const float sn = c.signal_n, so = c.solar_n, on = c.od_n;
  const double sprev = c.signal_prev;
  double v = 0.0;
  const long long t0 = clock64();
  for (;;) {
    unsigned long long w[2];
    powll_issue(rec, w);
    const bool ok = powll_check(w, tag, v);
    if (__all_sync(0xffffffffu, ok || lane >= world)) break;
    if (__any_sync(0xffffffffu, clock64() - t0 > 4000000000ll)) {   // ~2 s: give up, flag the error
      if (lane == 0) *sc.err = 1;
      v = 0.0;
      break;
    }
#if defined(__CUDA_ARCH__)
    __nanosleep(100);
#endif
  }
  double P = 0.0;
  for (int q = 0; q < world; ++q) P += __shfl_sync(0xffffffffu, v, q);
  EnvBroadcast<real> e;
  e.power_n = (real)(P * p.inv_nrs);
  e.signal_n = (real)sn; e.solar_n = (real)so; e.od_n = (real)on;
  e.rew_sig = (real)signal_penalty(p, P, sprev);
  e.pen_common = (real)0;   // individual_L2 (the early path's condition): not consumed
  e.pen_max = (real)0;
  return e;
}

DRSIM_D void ld4_cg(const float *p, float v[4]) {
#if defined(__CUDA_ARCH__)
  const float4 t = __ldcg(reinterpret_cast<const float4 *>(p));
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
#endif
}
DRSIM_D void ld4i_cg(const int32_t *p, int v[4]) {
#if defined(__CUDA_ARCH__)
  const int4 t = __ldcg(reinterpret_cast<const int4 *>(p));
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
#endif
}

// PLAIN = fp32 build, 10-column rows without neighbour messages (TarMAC layout / nb_comm = 0)
template <typename real, bool PLAIN, typename O = real, bool SMP = false>
__global__ void __launch_bounds__(kThreads, FusedOcc<real>::min_ctas)
k_shard(Planes<real> pl, SimParams p, StepIn in, ShardGeom g, ShardCtx sc, PeerCtx peer) {
  static_assert(!PLAIN || sizeof(real) == 4, "the plain variant is fp32 only");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double s_wp[kShardBatch][kThreads / 32][kRed];   // warp partials of the tiles of one arrival batch
  __shared__ EnvRegs s_er[kShardFinish];
  __shared__ EnvStage s_st[kShardFinish];
  __shared__ double s_rows[kShardFinish][kRed + 1];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Ns = p.Ns, D = p.obs_dim;
  const int s0 = threadIdx.x * kHousesPerThread;
  const KC<real> kc(p);
  // EARLY CLUSTER POWER.  Rewards and rows need the cluster power, and the power needs every house -- but only its
  // lock-out state machine (hvac.py:43-64), not its thermal update.  On the plain fp32 path with the individual
  // penalty a PRE-PASS over flags / sso / action / capacity (10 of the 103 bytes per house) forms the tile powers
  // with the arithmetic of the main pass, the reducer combines and publishes them while everybody runs the main
  // house update, and nobody waits between the two phases.  The other reduced quantities (penalty sums for the
  // running metrics, env planes) follow after phase 1, off the critical path.
  const bool early = PLAIN && p.penalty_mode == DRSIM_PEN_INDIVIDUAL_L2 && in.do_interp <= 0;
  // one cluster: CTA 0 owns no tile and only reduces (it polls while the others compute; the host adds it to the grid)
  const bool dedicated = early && p.R == 1 && gridDim.x > 1;
  // scheduled step with constant base power (fp32): the step's packed record (k_schedule_pack) holds every env
  // scalar that does not depend on the cluster power, exactly as the epilogue would compute it
  const bool fast_env = sizeof(real) == 4 && in.sched_rec != nullptr && p.base_mode == DRSIM_BASE_CONSTANT && in.do_interp <= 0;
  const bool direct = early && fast_env;   // the consumers take the cluster power straight from the early inbox
  const int n_work = dedicated ? (int)gridDim.x - 1 : (int)gridDim.x, wid = dedicated ? (int)blockIdx.x - 1 : (int)blockIdx.x;
  // this CTA's contiguous run of tiles (balanced: sizes differ by at most one)
  const int t_lo = wid < 0 ? 0 : (int)(((long long)wid * g.n_tiles) / n_work);
  const int t_hi = wid < 0 ? 0 : (int)(((long long)(wid + 1) * g.n_tiles) / n_work);
  // clusters this CTA completes: those whose first tile it owns (or all of them: dedicated reducer)
  const int r_lo = dedicated ? 0 : (t_lo + g.chunks - 1) / g.chunks;
  const int r_hi = dedicated ? (blockIdx.x == 0 ? p.R : 0) : (t_hi + g.chunks - 1) / g.chunks;
  pdl_trigger();
  auto stamp = [&](int k) {
#if defined(__CUDA_ARCH__)
    if (sc.dbg && threadIdx.x == 0) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      sc.dbg[(size_t)blockIdx.x * 16 + k] = t;
    }
#endif
  };
  stamp(0);
  // PLAIN: the inputs of a tile are staged one tile ahead by thread-private cp.async copies (no registers held
  // while they fly, completion = the thread's own wait_all): the state planes and the set-point go straight into
  // the tile's SAVED slots (the update then overwrites them in place), capacity / coefficients / actions into
  // the row staging area, which is idle during phase 1.  part 1 = launch-invariant planes (may run before
  // pdl_wait), 2 = what an earlier kernel wrote.
  float *s_in = reinterpret_cast<float *>(smem_raw + g.off_rows);            // [7][1024] cap, c0..c5 ; then [256] action words
  uint32_t *s_act = reinterpret_cast<uint32_t *>(s_in + 7 * kTileSlots);
  const bool ext = p.policy == DRSIM_POLICY_EXTERNAL || p.policy == DRSIM_POLICY_GREEDY_MYOPIC;
  auto prefetch = [&](int tile, int part) {
    if constexpr (PLAIN) {
      const int it = tile - t_lo;
      const int r = tile / g.chunks, c = tile - r * g.chunks;
      const int n0 = c * kTileSlots + s0;
      if (n0 >= p.N) return;
      const size_t off = (size_t)r * Ns + n0;
      const ShardSaved<float> sv(smem_raw + g.off_saved + (size_t)it * g.tile_bytes);
      if (part & 1) {
        cp_async16(sv.tg + s0, pl.target + off);
        cp_async16(s_in + s0, pl.cap + off);
#pragma unroll
        for (int k = 0; k < 6; ++k) cp_async16(s_in + (1 + k) * kTileSlots + s0, pl.coef[k] + off);
      }
      if (part & 2) {
        cp_async16(sv.ta + s0, pl.t_air + off);
        cp_async16(sv.tm + s0, pl.t_mass + off);
        cp_async16(sv.sso + s0, pl.sso + off);
        cp_async4(sv.flags + s0, pl.flags + off);
        if (ext) cp_async4(s_act + threadIdx.x, (in.actions ? in.actions : pl.actions) + off);
      }
    }
  };
  const bool staged0 = PLAIN && g.t_smem > 0 && t_hi > t_lo;
  // (a CTA that reduces early parks the tile powers in the row staging area: its first copies wait until then)
  const bool stage_late = early && r_hi > r_lo;
  if (staged0 && !stage_late) prefetch(t_lo, 1);
  pdl_wait();
  if (staged0 && !stage_late) prefetch(t_lo, 2);
  stamp(1);

  // Tiles [f_lo, f_hi) (at most kShardBatch) are done: their partials are formed from the warp partials in warp
  // order (the arithmetic of block_reduce in k_house) and published as self-validating words -- no atomic, and
  // no fence unless a consumer of the partial will also read house STATE written by this CTA (`vis`).
  // the reducer parks the collected partials in the (still unused) row staging area
  const PartLL ll{sc.partll, (uint32_t)in.xseq, sc.err, reinterpret_cast<double *>(smem_raw + g.off_rows), g.part_cap,
                  sc.dbg ? sc.dbg + (size_t)blockIdx.x * 16 : nullptr};
  const bool vis = !PLAIN || in.do_interp > 0;
  auto flush = [&](int f_lo, int f_hi) {
    if (vis) __threadfence();   // this thread's state stores are visible device-wide before the partial that announces them
    __syncthreads();
    if ((int)threadIdx.x < f_hi - f_lo) {
      double out[kRed] = {0, 0, 0, 0, 0};
      for (int i = 0; i < kThreads / 32; ++i) red_combine(out, s_wp[threadIdx.x][i]);
      partll_store(ll, f_lo + threadIdx.x, out);   // tile index == r * chunks + c
    }
    __syncthreads();   // s_wp may be rewritten
  };

  // ---- early cluster power: pre-pass + reduction + publication ----------------------------------------
  if constexpr (PLAIN) {
    if (early) {
      const uint32_t tag = (uint32_t)in.xseq;
      const int dt = p.dt, dur = p.lockout_duration;
      const float half_db = p.hf.half_db;
      const int policy = p.policy;
      const bool need_ta = policy == DRSIM_POLICY_DEADBAND_BANGBANG || policy == DRSIM_POLICY_BANGBANG;
      for (int b0 = t_lo; b0 < t_hi; b0 += kShardBatch) {
        const int b1 = min(t_hi, b0 + kShardBatch);
        for (int tile = b0; tile < b1; ++tile) {
          const int r = tile / g.chunks, c = tile - r * g.chunks;
          const int n0 = c * kTileSlots + s0;
          float P = 0.f;
          if (n0 < p.N) {
            const size_t off = (size_t)r * Ns + n0;
            const int valid = min(4, p.N - n0);
            const uint32_t flags = load4b(pl.flags + off);
            int sso[4];
            float cap[4], ta[4] = {0.f, 0.f, 0.f, 0.f};
            load4i(pl.sso + off, sso);
            load4_ro(pl.cap + off, cap);
            if (need_ta) load4(pl.t_air + off, ta);
            const uint32_t act = ext ? load4b((in.actions ? in.actions : pl.actions) + off) : 0u;
#pragma unroll
            for (int j = 0; j < 4; ++j) {   // the state machine and the power term of house4_compute_f32, nothing else
              const bool on = (flags >> (8 * j)) & 1u;
              bool a = (act >> (8 * j)) & 0xffu;
              if (policy == DRSIM_POLICY_DEADBAND_BANGBANG) a = ta[j] < -half_db ? false : (ta[j] > half_db ? true : on);
              else if (policy == DRSIM_POLICY_BANGBANG) a = ta[j] > 0.f;
              else if (policy == DRSIM_POLICY_ALWAYS_ON) a = true;
              const int s = sso[j] + (on ? 0 : dt);
              const bool on_n = !(!on && s < dur) && a;
              const float m = j < valid ? 1.f : 0.f;
              P = fmaf(on_n ? m : 0.f, cap[j] * p.hf.inv_cop, P);
            }
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) P += __shfl_down_sync(0xffffffffu, P, o);
          if (lane == 0) s_wp[tile - b0][warp][0] = (double)P;
        }
        __syncthreads();
        if ((int)threadIdx.x < b1 - b0) {
          double out = 0.0;
          for (int i = 0; i < kThreads / 32; ++i) out += s_wp[threadIdx.x][i][0];
          powll_store(sc.pearly + (size_t)(b0 + threadIdx.x) * 4, tag, out, false);
        }
        __syncthreads();
      }
      // the reducer of cluster r: collect the tile powers (all requests of a thread in flight together), fold them in
      // the order of reduce_cluster, exchange with the peers (house-sharded cluster), publish
      double *stage = reinterpret_cast<double *>(smem_raw + g.off_rows);
      for (int r = r_lo; r < r_hi; ++r) {
        if (threadIdx.x == kThreads - 32 && !direct) s_er[0] = env_load(pl, in, r);   // fetched under the poll
        double red0 = 0.0;
        for (int base = 0; base < g.chunks; base += g.part_cap) {
          const int nb = min(g.part_cap, g.chunks - base);
          const int n_own = (int)threadIdx.x < nb ? (nb - (int)threadIdx.x + kThreads - 1) / kThreads : 0;   // <= 32
          unsigned pending = n_own >= 32 ? 0xffffffffu : ((1u << n_own) - 1u);
          const long long t0 = clock64();
          while (pending) {
            for (int j0 = 0; j0 < n_own; j0 += 4) {
              if (!((pending >> j0) & 0xfu)) continue;
              unsigned long long w[4][2];
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if ((pending >> (j0 + u)) & 1u)
                  powll_issue(sc.pearly + (size_t)(r * g.chunks + base + (int)threadIdx.x + (j0 + u) * kThreads) * 4, w[u]);
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                double v;
                if (((pending >> (j0 + u)) & 1u) && powll_check(w[u], tag, v)) {
                  stage[(int)threadIdx.x + (j0 + u) * kThreads] = v;
                  pending &= ~(1u << (j0 + u));
                }
              }
            }
            if (pending) __nanosleep(200);   // the pollers share their SM (issue slots, LSU) with a CTA that computes
            if (pending && clock64() - t0 > 4000000000ll) {   // ~2 s: give up, flag the error
              *sc.err = 1;
              for (int j = 0; j < n_own; ++j)
                if ((pending >> j) & 1u) stage[(int)threadIdx.x + j * kThreads] = 0.0;
              pending = 0;
            }
          }
          __syncthreads();
          if (threadIdx.x < kReduceThreads)
            for (int c = threadIdx.x; c < nb; c += kReduceThreads) red0 += stage[c];
          __syncthreads();
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) red0 += __shfl_down_sync(0xffffffffu, red0, o);
        if (lane == 0 && threadIdx.x < kReduceThreads) s_rows[0][warp] = red0;
        __syncthreads();
        if (threadIdx.x == 0) {
          double P_rank = 0.0;
          for (int i = 0; i < kReduceThreads / 32; ++i) P_rank += s_rows[0][i];
          double P_total = 0.0;
          const int parity = (int)(in.xseq & 1);
          if (peer.world > 1) {
            for (int q = 0; q < peer.world; ++q)
              powll_store(peer.pinbox[q] + ((((size_t)parity * peer.world + peer.rank) * p.R + r) * 4), tag, P_rank, true);
          } else {
            powll_store(sc.pinbox + (((size_t)parity * p.R + r) * 4), tag, P_rank, false);
          }
          if (direct) {
            // nothing else to do here: every consumer folds the inbox itself (shard_wait_power)
          } else if (peer.world > 1) {
            const long long t0 = clock64();
            for (int q = 0; q < peer.world; ++q) {   // rank order: the order env_cluster folds the late rows in
              const unsigned long long *rec = peer.pinbox[peer.rank] + ((((size_t)parity * peer.world + q) * p.R + r) * 4);
              double v = 0.0;
              for (;;) {
                unsigned long long w[2];
                powll_issue(rec, w);
                if (powll_check(w, tag, v)) break;
                if (clock64() - t0 > 4000000000ll) { *peer.err = 1; v = 0.0; break; }
              }
              P_total += v;
            }
          } else {
            P_total += P_rank;
          }
          if (!direct) {
            const double red5[kRed] = {P_total, 0.0, 0.0, 0.0, 0.0};
            EnvOut o;
            shard_publish<real>(sc, in, r, env_epilogue_compute<real>(pl, p, in, r, s_er[0], red5, 0.0, o));
          }
        }
        __syncthreads();
      }
    }
  }
  if (staged0 && stage_late) prefetch(t_lo, 3);
  stamp(14);

  // ---- phase 1: house update of every tile of this CTA ------------------------------------------
  for (int tile = t_lo; tile < t_hi; ++tile) {
    const int it = tile - t_lo;
    const int r = tile / g.chunks, c = tile - r * g.chunks;
    const int n0 = c * kTileSlots + s0;
    real red[kRed] = {0, 0, 0, 0, 0};
    if constexpr (PLAIN) {
      // a thread with no house in this tile (cluster tail) may own houses of the next one
      if (n0 >= p.N && it + 1 < g.t_smem && tile + 1 < t_hi) { cp_async_wait_all(); prefetch(tile + 1, 3); }
    }
    if (n0 < p.N) {
      House4<real> h;
      const size_t off = (size_t)r * Ns + n0;
      if constexpr (PLAIN) {
        Raw4f w;
        if (it < g.t_smem) {   // staged one tile ago
          const ShardSaved<float> sv(smem_raw + g.off_saved + (size_t)it * g.tile_bytes);
          cp_async_wait_all();
          load4(sv.ta + s0, w.ta);
          load4(sv.tm + s0, w.tm);
          load4i(sv.sso + s0, w.sso);
          w.flags = *reinterpret_cast<const uint32_t *>(sv.flags + s0);
          load4(sv.tg + s0, w.target);
          load4(s_in + s0, w.cap);
#pragma unroll
          for (int k = 0; k < 6; ++k) load4(s_in + (1 + k) * kTileSlots + s0, w.c[k]);
          w.act = ext ? s_act[threadIdx.x] : 0u;
          // the thread holds its inputs in registers: its staging slots are free for the next tile's copies
          if (it + 1 < g.t_smem && tile + 1 < t_hi) prefetch(tile + 1, 3);
        } else {
          load4(pl.t_air + off, w.ta);
          load4(pl.t_mass + off, w.tm);
          load4i(pl.sso + off, w.sso);
          w.flags = load4b(pl.flags + off);
          load4_ro(pl.target + off, w.target);
          load4_ro(pl.cap + off, w.cap);
#pragma unroll
          for (int k = 0; k < 6; ++k) load4_ro(pl.coef[k] + off, w.c[k]);
          w.act = ext ? load4b((in.actions ? in.actions : pl.actions) + off) : 0u;
        }
        w.od = (float)pl.od_temp[r];
        w.solar = (float)pl.solar_next[r];
        house4_compute_f32<false>(pl, p, w, off, min(4, p.N - n0), h, red);
      } else {
        house4_step<real, true>(pl, p, kc, in, off, min(4, p.N - n0), (real)pl.od_temp[r], (real)pl.solar_next[r], h, red);
      }
      if (it < g.t_smem) {
        const ShardSaved<real> sv(smem_raw + g.off_saved + (size_t)it * g.tile_bytes);
        store4(sv.ta + s0, h.ta);
        store4(sv.tm + s0, h.tm);
        store4(sv.tg + s0, h.target);
        store4i(sv.sso + s0, h.sso);
        *reinterpret_cast<uint32_t *>(sv.flags + s0) = h.flags;
      }
    }
    // warp stage of block_reduce (k_house): shuffle tree in `real`, lane 0 keeps the warp partial as double
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      real t[kRed];
#pragma unroll
      for (int k = 0; k < kRed; ++k) t[k] = __shfl_down_sync(0xffffffffu, red[k], o);
      red_combine(red, t);
    }
    if (lane == 0)
      for (int k = 0; k < kRed; ++k) s_wp[it % kShardBatch][warp][k] = (double)red[k];
    if ((it + 1) % kShardBatch == 0 && tile + 1 < t_hi) flush(tile + 1 - kShardBatch, tile + 1);
  }
  stamp(2);
  if (t_hi > t_lo) flush(t_lo + (t_hi - t_lo - 1) / kShardBatch * kShardBatch, t_hi);

  // ---- reduce + env: this CTA completes the clusters whose FIRST tile it owns ---------------------
  // Only now, with nothing left to contribute: every partial / push this CTA owes anybody is out, so the polls
  // and peer waits below cannot deadlock (clusters are taken in ascending order on every rank).
  {
    // (several ranks: the late rows are combined by env_cluster, which also runs the full epilogue -- off the critical path)
    const bool fast_late = fast_env && peer.world <= 1;
    for (int rg = r_lo; rg < r_hi; rg += kShardFinish) {
      const int ng = min(kShardFinish, r_hi - rg);
      for (int k = 0; k < ng; ++k) {
        const int r = rg + k;
        // previous step's env scalars (or, on the scheduled path, this step's packed record + running metrics),
        // fetched while the partials are being collected
        if (threadIdx.x == kThreads - 32) {
          if (fast_late) {
            s_st[k].rec = in.sched_rec[r];
            for (int q = 0; q < DRSIM_N_METRICS; ++q) s_st[k].m[q] = pl.metrics[(size_t)r * DRSIM_N_METRICS + q];
          } else {
            s_er[k] = env_load(pl, in, r);
          }
        }
        const double *row = reduce_cluster<real>(pl, p, in, g.chunks, peer, r, ll);
        if (threadIdx.x == 0) {
#pragma unroll
          for (int q = 0; q <= kRed; ++q) s_rows[k][q] = row[q];
        }
        __syncthreads();
      }
      stamp(6);
      // lane 0 of warp k finishes cluster rg + k: wait for the peers' rows (house-sharded cluster), env epilogue,
      // broadcast values to the consumers first, env planes / metrics afterwards
      if (lane == 0 && warp < ng) {
        const int r = rg + warp;
        if (fast_late) {
          // every env scalar that does not depend on the cluster power is in the step's record (k_schedule_pack):
          // the consumers are two multiplications away from their values (expressions of the fused kernels)
          const SchedRec &c = s_st[warp].rec;
          const double *a = s_rows[warp];
          EnvBroadcast<real> b;
          b.power_n = (real)(a[0] * p.inv_nrs);
          b.signal_n = c.signal_n; b.solar_n = c.solar_n; b.od_n = c.od_n;
          b.rew_sig = (real)signal_penalty(p, a[0], c.signal_prev);
          b.pen_common = (real)a[1];
          b.pen_max = (real)a[2];
          if (!early) shard_publish<real>(sc, in, r, b);   // (early: the consumers have had these values since the pre-pass)
          stamp(7);
          env_stage_store<real>(pl, p, r, s_st[warp], a);
        } else {
          EnvOut o;
          const EnvBroadcast<real> b = env_cluster<real>(pl, p, in, nullptr, 0, peer, r, &o, &s_er[warp], s_rows[warp]);
          if (!early) shard_publish<real>(sc, in, r, b);
          stamp(7);
          env_epilogue_store<real>(pl, p, in, r, o);
        }
      }
      __syncthreads();
    }
  }
  stamp(3);

  // ---- phase 2: rewards + observation rows --------------------------------------------------------
  int r_have = -1;
  EnvBroadcast<real> e{};
  auto env_of = [&](int r) {   // warp-uniform: (re)fetch the broadcast values when the cluster changes
    if (r == r_have) return;
    e = direct ? shard_wait_power<real>(sc, p, in, peer.world, r, lane) : shard_wait_env<real>(sc, in, r, lane);
    r_have = r;
  };

  if constexpr (PLAIN) {
    O *s_tile = reinterpret_cast<O *>(smem_raw + g.off_rows);
    bool store_pending = false;
    const int w0 = warp * 128;
    for (int tile = t_lo; tile < t_hi; ++tile) {
      const int it = tile - t_lo;
      const int r = tile / g.chunks, c = tile - r * g.chunks;
      env_of(r);
      if (tile == t_lo) stamp(4);
      const int n0 = c * kTileSlots + s0;
      const size_t rb = (size_t)r * Ns;
      const int slots = min(kTileSlots, Ns - c * kTileSlots);   // house slots of this tile (multiple of 4)
      // the warp's previous bulk store must have finished reading its rows before they are rewritten
      if (lane == 0 && store_pending) bulk_store_wait_read();
      __syncwarp();
      if (s0 < slots) {
        const size_t off = rb + n0;
        const int valid = min(4, p.N - n0);
        float ta[4], tm[4], tg[4];
        int sso[4];
        uint32_t flags;
        if (it < g.t_smem) {
          const ShardSaved<float> sv(smem_raw + g.off_saved + (size_t)it * g.tile_bytes);
          load4(sv.ta + s0, ta); load4(sv.tm + s0, tm); load4(sv.tg + s0, tg); load4i(sv.sso + s0, sso);
          flags = *reinterpret_cast<const uint32_t *>(sv.flags + s0);
        } else {
          ld4_cg(pl.t_air + off, ta); ld4_cg(pl.t_mass + off, tm); load4_ro(pl.target + off, tg); ld4i_cg(pl.sso + off, sso);
#if defined(__CUDA_ARCH__)
          flags = __ldcg(reinterpret_cast<const uint32_t *>(pl.flags + off));
#endif
        }
        float rw[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool ok = j < valid;
          rw[j] = ok ? house_reward<float>(p, kc, ta[j], tg[j], e) : 0.f;
          const uint32_t f = (flags >> (8 * j)) & 0xffu;
          const float sso_n = (float)fast_div((uint32_t)sso[j], p.fd_dur);          // norm.py:40-43, :79-82
          const float t20 = tg[j] - 20.f;
          O *row = s_tile + (size_t)(s0 + j) * 10;
          put2(row, 0, ok ? (float)(f & 1u) : 0.f, ok ? (float)((f >> 1) & 1u) : 0.f);
          put2(row, 1, ok ? sso_n : 0.f, ok ? 1.f : 0.f);
          put2(row, 2, ok ? e.power_n : 0.f, ok ? e.signal_n : 0.f);
          put2(row, 3, ok ? p.hf.deadband : 0.f, ok ? (ta[j] + t20) * 0.2f : 0.f);
          put2(row, 4, ok ? (tm[j] + t20) * 0.2f : 0.f, ok ? t20 * 0.2f : 0.f);
        }
        store4(pl.reward + off, rw);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0 && w0 < slots) {
        const int nrows = min(128, slots - w0);
        bulk_store_s2g(pl.template rows<O>() + (rb + (size_t)c * kTileSlots + w0) * 10, s_tile + (size_t)w0 * 10,
                       (uint32_t)(nrows * 10 * sizeof(O)));
        store_pending = true;
      }
    }
    // shared memory must outlive the reads of the last row stores; their global writes complete with the grid
    if (lane == 0 && store_pending) bulk_store_wait_read();
    stamp(5);
  } else {
    O *rows_w = reinterpret_cast<O *>(smem_raw + g.off_rows) + (size_t)warp * g.nbuf * kShardGroup * D;
    const bool halo = needs_halo(p);
    int grp = 0;   // row groups this warp has shipped (selects the staging buffer)
    for (int tile = t_lo; tile < t_hi; ++tile) {
      const int it = tile - t_lo;
      const int r = tile / g.chunks, c = tile - r * g.chunks;
      env_of(r);
      const bool saved = it < g.t_smem;
      const ShardSaved<real> sv(smem_raw + g.off_saved + (size_t)(saved ? it : 0) * g.tile_bytes);
      const size_t rb = (size_t)r * Ns;
      for (int gi = 0; gi < 128 / kShardGroup; ++gi) {
        const int hs0 = warp * 128 + gi * kShardGroup;   // first house of the group inside the tile
        const int ng0 = c * kTileSlots + hs0;            // ... inside the cluster
        if (ng0 >= Ns) break;                            // warp-uniform: nothing of this group exists
        const int n = ng0 + lane, hs = hs0 + lane;
        O *row = rows_w + ((size_t)(grp % g.nbuf) * kShardGroup + lane) * D;
        if (D > 0) {
          // the bulk store that last used this staging buffer must have finished reading it
          if (lane == 0 && grp >= g.nbuf) {
#if defined(__CUDA_ARCH__)
            if (g.nbuf == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
#endif
          }
          __syncwarp();
        }
        if (n < p.N) {
          const size_t o = rb + n;
          real ta, tm, tgt;
          int sso;
          uint32_t f;
          if (saved) { ta = sv.ta[hs]; tm = sv.tm[hs]; tgt = sv.tg[hs]; sso = sv.sso[hs]; f = sv.flags[hs]; }
          else { ta = ld_cg(pl.t_air + o); tm = ld_cg(pl.t_mass + o); tgt = pl.target[o]; sso = ld_cg(pl.sso + o); f = ld_cg(pl.flags + o); }
          pl.reward[o] = house_reward<real>(p, kc, ta, tgt, e);
          if (D > 0) {
            real ratio[4] = {0, 0, 0, 0};
            if (p.st_thermal)
              for (int k = 0; k < 4; ++k) ratio[k] = pl.ratio[k][o];
            int i = obs_own<real>(row, p, f, own_sso_norm<real>(pl, p, o, sso), Rep<real>::minus20(ta, tgt),
                                  Rep<real>::minus20(tm, tgt), tgt - (real)20, e, ratio);
            if (p.obs_layout == DRSIM_OBS_HAND_ENGINEERED) {
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
                    for (int m = 0; m < 4; ++m) row[i++] = (real)ld_cg(rec + m);
                    if (p.msg_thermal)
                      for (int m = 0; m < 4; ++m) row[i++] = (real)ld_cg(rec + 4 + m);
                    if (p.msg_hvac) { row[i++] = (real)p.cop; row[i++] = (real)p.latent; row[i++] = (real)p.dcap; }
                    continue;
                  }
                }
                const size_t q = rb + nb;
                const real pmax = qdiv(pl.cap[q], kc.cop, kc.inv_cop);
                row[i++] = div5(Rep<real>::dev(ld_cg(pl.t_air + q), pl.target[q]));       // norm.py:39
                row[i++] = (real)fast_div((uint32_t)ld_cg(pl.sso + q), p.fd_dur);         // norm.py:40-43
                row[i++] = qdiv((ld_cg(pl.flags + q) & 1u) ? pmax : (real)0, kc.nrs, kc.inv_nrs);
                row[i++] = qdiv(pmax, kc.nrs, kc.inv_nrs);
                if (p.msg_thermal)
                  for (int m = 0; m < 4; ++m) row[i++] = (real)pl.ratio[m][q];
                if (p.msg_hvac) {                                                         // constants, quirk Q11
                  row[i++] = (real)p.cop; row[i++] = (real)p.latent; row[i++] = (real)p.dcap;
                }
              }
            }
          }
        } else if (n < Ns) {
          for (int i = 0; i < D; ++i) row[i] = (real)0;  // padding slot
        }
        if (D > 0) {
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            const int nrows = min(kShardGroup, Ns - ng0);   // multiple of 4: the byte count is a multiple of 16
            bulk_store_s2g(pl.template rows<O>() + (rb + ng0) * D, rows_w + (size_t)(grp % g.nbuf) * kShardGroup * D,
                           (uint32_t)((size_t)nrows * D * sizeof(O)));
          }
          ++grp;
        }
      }
    }
    if (lane == 0 && grp > 0) bulk_store_wait_read();
  }
}

}  // namespace drsim
