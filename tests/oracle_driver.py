"""The NumPy oracle (``oracle.np_oracle``) driven beside a ``BatchedEnv`` on the GPU.

The device draws its outdoor-temperature noise and its Perlin signal noise from Philox streams keyed by
(seed, global replica, step); ``od_noise`` and ``perlin`` restate them with ``oracle.philox``.  ``oracle_run`` replays
a whole trajectory from an initial state.  ``OracleDriver`` steps a handle and checks it against the oracle on a few
picked replicas (the first, the last -- in the ragged last tile -- and one in the middle of a multi-cluster tile):

* re-anchored (``step``): before every GPU step the oracle is loaded with the GPU state (``get_state``, env scalars
  included) and stepped once, so the comparison isolates the error of ONE step.  The GPU path is not touched.
* free-running (``start_free`` / ``advance_free`` / ``check_free``): the oracle starts from the GPU state at one
  point and is driven by the same actions and restated noise over many steps.

Tolerances.  Discrete state (on, lockout, seconds since off) and the epoch are compared bit for bit on ALL replicas:
with external actions they do not depend on temperatures, so the lock-out state machine restated on the whole batch
holds over any horizon.  Under an on-device controller the actions are the reference controller's on the device's own
pre-step planes, so the same bit-exact check holds (``controller_inputs`` / ``controller_actions``).  Cluster power then
follows from them (1e-6 relative: an fp32 sum of up to 1000 terms).
Outdoor temperature, signal and base power are fp64 env scalars in both builds: 1e-9 relative.  Temperatures: one
fp32 step of the difference-form update is at rounding level, 4e-6 absolute (``test_per_step_error_fp32_is_at_rounding
_level``); free-running fp32 trajectories get the 2e-4 drift allowance of the batched oracle tests; the fp64 build
replays the reference's literal arithmetic, 1e-9.  Rewards, observations and the running metrics: the BASELINE.json
north star, rtol 1e-5 of (|value| + natural scale 1) in fp32, and 1e-9 of the same in fp64.
"""
from __future__ import annotations

import numpy as np

from golden_util import _close

HOUSE_STATIC = ("Ua", "Ca", "Cm", "Hm")
KEYS = ("dt_air", "dt_mass", "t_air", "t_mass", "sso", "flags", "reward", "obs", "signal", "power", "od_temp",
        "base_power", "metrics")


def prop(n, **over):
    """Environment properties of an ``n``-house cluster; ``over`` maps ``a/b/c`` paths to values."""
    p = {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": 4.0,
         "cluster_prop": {"nb_agents": n, "house_prop": {"target_temp": 19.0}}}
    for path, v in over.items():
        d = p
        keys = path.split("/")
        for k in keys[:-1]:
            d = d.setdefault(k, {})
        d[keys[-1]] = v
    return p


# neighbours_2D: N -> (row_size, max_communication_distance); the table is 2 d (d + 1) wide
NB_2D = {12: (4, 1), 100: (10, 1), 300: (15, 1), 1000: (25, 2), 1300: (26, 2), 2500: (50, 2)}


def config(n, pen="individual_L2", sig="perlin", state="none", msg="none", nb="neighbours", c=10, start=None, dist=None,
           **extra):
    """Properties of one matrix cell.  The deadband keeps ``common_max_error`` non-zero and the lock-out FSM busy."""
    over = {"cluster_prop/house_prop/deadband": 0.4,
            "reward_prop/penalty_props/mode": pen,
            "reward_prop/penalty_props/alpha_common_max": 1.0,
            "power_grid_prop/signal_properties/mode": sig,
            "state_prop/solar_gain": state in ("solar", "all"),
            "state_prop/thermal": state == "all",
            "state_prop/hvac": state == "all",
            "cluster_prop/message_prop/thermal": msg == "th_hvac",
            "cluster_prop/message_prop/hvac": msg == "th_hvac",
            "cluster_prop/agents_comm_prop/mode": nb,
            "cluster_prop/agents_comm_prop/max_nb_agents_communication": c}
    if nb == "neighbours_2D":
        row, d = NB_2D[n]
        dist = d if dist is None else dist
        over["cluster_prop/agents_comm_prop/row_size"] = row
        over["cluster_prop/agents_comm_prop/max_communication_distance"] = dist
    if start is not None:
        over["start_datetime"] = start
    over.update(extra)
    return prop(n, **over)


# route -> (precision, R, N, layout, path, environment, expected)
#   expected: route = last_route after a step; variant = fused_info()["variant"]; e = clusters per tile;
#   launches = kernel launches per step
ROUTES = {
    "k_fused_tma<1>": ("f32", 12, 1000, "tarmac", "auto", {}, dict(route="k_fused_tma<1>", variant="staged", e=1, launches=1)),
    "k_fused_tma<2>": ("f32", 30, 100, "hand_engineered", "auto", {"DRSIM_TILE_ENVS": 3},
                       dict(route="k_fused_tma<2>", variant="staged", e=3, launches=1)),
    "k_fused_tma<0>/1-per-tile": ("f32", 9, 300, "hand_engineered", "auto", {"DRSIM_TILE_ENVS": 1},
                                  dict(route="k_fused_tma<0>", variant="staged", e=1, launches=1)),
    "k_fused_tma<0>/3-per-tile": ("f32", 30, 100, "hand_engineered", "auto", {"DRSIM_TILE_ENVS": 3},
                                  dict(route="k_fused_tma<0>", variant="staged", e=3, launches=1)),
    "k_fused_rows<staged>": ("f32", 60, 100, "hand_engineered", "auto", {"DRSIM_TILE_ENVS": 7},
                             dict(route="k_fused_rows<staged>", variant="staged_rows", e=7, launches=1)),
    "k_fused_rows<unstaged>": ("f32", 6, 1000, "hand_engineered", "auto", {},
                               dict(route="k_fused_rows<unstaged>", variant="staged_rows", e=1, launches=1)),
    "general/rows-fallback": ("f32", 60, 100, "hand_engineered", "auto", {"DRSIM_TILE_ENVS": 7},
                              dict(route="four-kernel", variant="staged_rows", e=7, launches=4)),
    "k_fused/chunked": ("f32", 3, 1000, "hand_engineered", "auto", {}, dict(route="k_fused", variant="chunked", e=1, launches=1)),
    # 85 clusters per tile: their schedule records do not fit next to the TMA planes (rows of at most 16 columns)
    "k_fused_direct": ("f32", 300, 10, "hand_engineered", "auto", {"DRSIM_TILE_ENVS": 85},
                       dict(route="k_fused_direct", variant="direct", e=85, launches=1)),
    "k_small": ("f32", 7, 10, "hand_engineered", "auto", {}, dict(route="k_small", launches=1)),
    "k_shard": ("f32", 2, 2500, "hand_engineered", "auto", {}, dict(route="k_shard", variant="none", launches=1)),
    "four-kernel": ("f32", 24, 100, "hand_engineered", "split", {"DRSIM_NO_SHARD_KERNEL": 1},
                    dict(route="four-kernel", variant="none", launches=4)),
    "k_fused_direct<double>": ("f64", 24, 100, "hand_engineered", "auto", {"DRSIM_TILE_ENVS": 2},
                               dict(route="k_fused_direct", variant="direct", e=2, launches=1)),
    "k_fused<double>/chunked": ("f64", 3, 1000, "hand_engineered", "auto", {},
                                dict(route="k_fused", variant="chunked", e=1, launches=1)),
    "k_small_gen<double>": ("f64", 7, 10, "hand_engineered", "auto", {}, dict(route="k_small_gen", launches=1)),
    "k_shard<double>": ("f64", 3, 1300, "hand_engineered", "auto", {}, dict(route="k_shard", variant="none", launches=1)),
}


def loop_launches(first_step, T, block_base):
    """Launches of ``drsim_run_tape`` on a loop route: one step kernel per 64-step schedule block, plus the two schedule
    kernels when the run enters a block that has not been generated (``block_base`` = start of the current block)."""
    n, s, base = 0, first_step, block_base
    while s < first_step + T:
        if base is None or not base <= s < base + 64:
            base, n = s, n + 2
        k = min(first_step + T - s, base + 64 - s)
        n, s = n + 1, s + k
    return n


# ---- on-device controllers -------------------------------------------------------------------
def controller_inputs(env):
    """What a controller reads before a step, as the device reads it: the temperature ``x`` against ``target`` (fp32:
    the deviation plane against 0; fp64: the absolute temperature against the set-point), capacities, the on and
    lock-out bits of ``flags`` and the cluster's ``signal`` (the observation's ``reg_signal``).  fp64 ``[R, N]`` /
    ``[R]``."""
    import torch

    torch.cuda.synchronize()
    v = env.state
    f64 = lambda t: t.double().cpu().numpy()   # noqa: E731
    x = f64(v["dt_air"]) if v["temp_is_deviation"] else f64(v["t_air"])
    target = np.zeros_like(x) if v["temp_is_deviation"] else f64(v["target"])
    flags = v["flags"].cpu().numpy()
    return dict(x=x, target=target, cap=f64(v["cap"]), on=(flags & 1).astype(bool),
                lockout=((flags >> 1) & 1).astype(bool), signal=f64(v["signal"]))


def controller_actions(policy, deadband, cop, x, target, cap, on, lockout, signal):
    """The reference controllers of ``oracle.np_oracle`` on ``[R, N]`` inputs.  Greedy-myopic keys are ``-(x -
    target)`` and powers ``cap / cop``, the fp64 arithmetic ``k_greedy`` does in the same order; ties go by index.

    The bang-bang family in the fp32 build decides on the deviation against ``float(deadband / 2)``: the same decision
    as the reference's on ``target + deviation`` when half the deadband is exact in fp32 (0.5, 1.0).  A deadband whose
    half is not (0.4) may decide differently on a deviation of exactly ``float(deadband / 2)``."""
    from oracle.np_oracle import bangbang, deadband_bangbang, greedy_myopic

    if policy == "deadband_bangbang":
        return deadband_bangbang(x, target, deadband, on)
    if policy == "bangbang":
        return bangbang(x, target)
    if policy == "always_on":
        return np.ones(x.shape, dtype=bool)
    assert policy == "greedy_myopic", policy
    return np.stack([greedy_myopic(x[r], target[r], cap[r], cop, lockout[r], signal[r]) for r in range(x.shape[0])])


def policy_name(env):
    from marl_demandresponse_b200 import _lib

    return {v: k for k, v in _lib.POLICY.items()}[int(env.sim.cfg.policy)]


def check_greedy_plane(env, want, what):
    """The action plane ``k_greedy`` wrote: ``want`` on every house of every replica, 0 in the padding slots."""
    import torch

    torch.cuda.synchronize()
    got = env.state["actions_padded"].cpu().numpy()
    N = want.shape[1]
    bad = np.argwhere(got[:, :N] != want.astype(np.uint8))
    assert bad.size == 0, f"{what}: greedy action differs at (replica, house) {bad[:6].tolist()}"
    assert not got[:, N:].any(), f"{what}: padding slots of the action plane are not 0"


def od_noise(seed, reps, steps, temp_std=1.0):
    """``[len(steps), len(reps)]``: the outdoor-temperature noise of global replicas ``reps`` at Philox steps ``steps``."""
    from oracle import philox

    return np.array([[philox.od_noise(seed, r, t, temp_std) for r in reps] for t in steps])


def perlin(seed, reps, epochs, signal_prop=None):
    """``[T, len(reps)]``: the Perlin signal noise of global replicas ``reps`` at the epochs ``[T]`` or ``[T, len(reps)]``."""
    from oracle import philox

    sp = signal_prop or {"nb_octaves": 5, "octaves_step": 5, "period": 300}
    ep = np.broadcast_to(np.asarray(epochs, dtype=np.int64).reshape(len(epochs), -1), (len(epochs), len(reps)))
    return np.array([[philox.perlin(seed, r, (int(e) % 86400) / sp["period"], sp["nb_octaves"], sp["octaves_step"])
                      for r, e in zip(reps, row)] for row in ep])


def oracle_run(env_prop, st, actions, od, pe):
    """The oracle from state ``st``: the reset's power-grid step with ``pe[0]``, then step t with ``actions[t]``,
    ``od[t]`` and ``pe[t + 1]``.  Returns the oracle and the rewards ``[T, R, N]``."""
    from oracle.np_oracle import NpOracle, from_epoch

    orc = NpOracle(env_prop, st["t_air"].shape[0])
    orc.set_state(st)
    orc.power_grid_step([from_epoch(e) for e in orc.state["epoch"]], None if pe is None else pe[0])
    rew = [orc.step(actions[t], od[t], None if pe is None else pe[t + 1]) for t in range(actions.shape[0])]
    return orc, np.array(rew)


def pick_replicas(R, envs_per_tile):
    """First replica, last replica (ragged last tile) and one in the middle of a multi-cluster tile."""
    e = max(1, envs_per_tile)
    mid_tile = ((R + e - 1) // e) // 2
    mid = min(R - 1, mid_tile * e + e // 2)
    return sorted({0, mid, R - 1})


def tolerances(precision, anchored):
    if precision == "f64":
        return {"temp": 1e-9, "rel": 1e-9}
    return {"temp": 4e-6 if anchored else 2e-4, "rel": 1e-5}


class OracleDriver:
    """Steps ``env`` with external actions, or under its on-device controller, and compares it with the oracle (see
    the module docstring)."""

    def __init__(self, env, env_prop, st0, step_index=0, picks=None):
        from oracle.config import normalize_env_prop

        self.env, self.env_prop = env, env_prop
        self.p = normalize_env_prop(env_prop)
        self.R, self.N = env.n_replicas, env.n_houses
        self.precision = "f64" if env.sim.real == np.float64 else "f32"
        self.picks = pick_replicas(self.R, env.sim.fused_info()["envs_per_tile"]) if picks is None else list(picks)
        self.static = {k: np.broadcast_to(np.asarray(st0[k], dtype=np.float64), (self.R, self.N))[self.picks]
                       for k in HOUSE_STATIC}
        self.step_index = step_index          # the handle's step counter: the Philox step of the next step
        self.sp = self.p["power_grid_prop"]["signal_properties"]
        self.temp_std = self.p["temp_prop"]["temp_std"]
        self.dur = self.p["cluster_prop"]["house_prop"]["hvac_prop"]["lockout_duration"]
        self.cop = self.p["cluster_prop"]["house_prop"]["hvac_prop"]["cop"]
        self.deadband = self.p["cluster_prop"]["house_prop"]["deadband"]
        self.policy = policy_name(env)
        s = env.get_state()
        self.disc = {k: s[k].astype(np.int64) for k in ("on", "lockout", "sso")}
        self.epoch = s["epoch"].astype(np.int64)
        self.metrics0 = env.metrics.double().cpu().numpy().copy()
        self.rew_sum = np.zeros(len(self.picks))
        self.n_steps = 0
        self.free = None

    # ---- noise and state -------------------------------------------------------------------
    def _noise(self, step, epochs):
        reps = [self.env.rep_offset + r for r in self.picks]
        od = od_noise(self.env.seed, reps, [step], self.temp_std)[0]
        pe = perlin(self.env.seed, reps, [epochs], self.sp)[0] if self.sp["mode"] == "perlin" else None
        return od, pe

    def _oracle(self, gpu_state):
        from oracle.np_oracle import NpOracle

        st = {k: (v[self.picks] if np.ndim(v) >= 1 and np.shape(v)[0] == self.R else v) for k, v in gpu_state.items()}
        st.update(self.static)
        orc = NpOracle(self.env_prop, len(self.picks))
        orc.set_state(st)
        return orc

    def _table(self):
        """The handle's own neighbour table; without one the oracle's ring table, or none at all when the rows carry no
        messages (a table mode on the TarMAC layout)."""
        if self.env._table is not None:
            return self.env._table
        if self.p["cluster_prop"]["agents_comm_prop"]["mode"] == "neighbours":
            return None
        return np.zeros((self.N, 0), dtype=np.int32)

    def _advance_discrete(self, acts):
        from oracle.np_oracle import hvac_fsm

        on, lock, sso = hvac_fsm(self.disc["on"], self.disc["lockout"], self.disc["sso"], acts,
                                 int(self.p["time_step"]), self.dur)
        self.disc = {"on": on.astype(np.int64), "lockout": lock.astype(np.int64), "sso": sso.astype(np.int64)}
        self.epoch = self.epoch + int(self.p["time_step"])

    # ---- comparisons -----------------------------------------------------------------------
    def _check_all_replicas(self, got, what):
        for k in ("on", "lockout", "sso"):
            bad = np.argwhere(got[k].astype(np.int64) != self.disc[k])
            assert bad.size == 0, f"{what}: {k} differs at (replica, house) {bad[:6].tolist()}"
        assert np.array_equal(got["epoch"].astype(np.int64), self.epoch), f"{what}: epoch"
        p_sum = (got["on"].astype(np.float64) * got["cap"] / self.cop).sum(axis=1)
        _close(got["power"], p_sum, 1e-6, 0.0, f"{what}: power (sum over houses)")

    def _check_picked(self, got, orc, rew, rew_ref, obs, anchored, what):
        tol = tolerances(self.precision, anchored)
        s, pk = orc.state, self.picks
        for k in ("on", "lockout", "sso"):
            assert np.array_equal(got[k][pk].astype(np.int64), s[k].astype(np.int64)), f"{what}: {k} (oracle)"
        assert np.array_equal(got["epoch"][pk], s["epoch"]), f"{what}: epoch (oracle)"
        for k in ("od_temp", "signal", "base_power"):
            _close(got[k][pk], s[k], 1e-9, 0.0, f"{what}: {k}")
        _close(got["power"][pk], s["power"], 1e-6, 0.0, f"{what}: power")
        for k in ("t_air", "t_mass"):
            _close(got[k][pk], s[k], 0.0, tol["temp"], f"{what}: {k}")
        _close(rew, rew_ref, tol["rel"], tol["rel"], f"{what}: rewards")
        if obs is not None:
            want = orc.obs_vectors(self._table())[..., :obs.shape[-1]]
            assert want.shape == obs.shape, (want.shape, obs.shape)
            _close(obs, want, tol["rel"], tol["rel"], f"{what}: observations")

    def _gpu(self):
        import torch

        torch.cuda.synchronize()
        got = self.env.get_state()
        rew = self.env.reward[self.picks].double().cpu().numpy()
        obs = self.env.obs[self.picks].double().cpu().numpy() if self.env.obs is not None else None
        return got, rew, obs

    # ---- stepping ----------------------------------------------------------------------------
    def _controller(self, inputs):
        return controller_actions(self.policy, self.deadband, self.cop, **inputs)

    def _free_actions(self):
        """The restated controller on the free-running oracle's own state (picked replicas)."""
        s = self.free.state
        return self._controller(dict(x=s["t_air"], target=s["target"], cap=s["cap"], on=s["on"], lockout=s["lockout"],
                                     signal=s["signal"]))

    def step(self, acts=None, check=True):
        """One GPU step on ``acts`` (numpy ``[R, N]``), checked against one oracle step from the GPU state before it.
        ``acts`` None: the handle's on-device controller chooses, and the actions are the reference controller's on
        the pre-step planes (``controller_inputs``); greedy-myopic's action plane is checked against them on every
        replica, and the discrete state checks every policy's.  A free-running oracle is then driven by the restated
        controller on its own state.  Returns the number of kernel launches the step made."""
        import torch

        before = self.env.get_state() if check else None
        on_device = acts is None
        if on_device:
            acts = self._controller(controller_inputs(self.env))
        free_acts = (self._free_actions() if on_device else acts[self.picks]) if self.free is not None else None
        l0 = self.env.sim.launch_count
        self.env.step(None if on_device else torch.as_tensor(acts, device="cuda"))
        launches = self.env.sim.launch_count - l0
        what = f"step {self.n_steps}"
        if on_device and self.policy == "greedy_myopic":
            check_greedy_plane(self.env, acts, what)
        self._advance_discrete(acts)
        if self.free is not None:
            self._advance_free_one(free_acts)
        if check:
            got, rew, obs = self._gpu()
            self._check_all_replicas(got, what)
            orc = self._oracle(before)
            od, pe = self._noise(self.step_index, self.epoch[self.picks])
            rew_ref = orc.step(acts[self.picks], od, pe)
            self._check_picked(got, orc, rew, rew_ref, obs, True, what)
            self.rew_sum += rew_ref.mean(axis=1)
            self._rew_scale = getattr(self, "_rew_scale", 0.0) + np.abs(rew_ref).mean(axis=1) + 1.0
        self.step_index += 1
        self.n_steps += 1
        return launches

    def check_metrics(self):
        """Running metrics since the driver started: the step count exactly (all replicas), the sum of the mean
        rewards on the picked replicas (the per-step reward tolerance, summed)."""
        m = self.env.metrics.double().cpu().numpy() - self.metrics0
        assert np.all(m[:, 0] == self.n_steps), m[:, 0]
        rel = tolerances(self.precision, True)["rel"]
        err = np.abs(m[self.picks, 1] - self.rew_sum)
        assert np.all(err <= rel * self._rew_scale), (m[self.picks, 1], self.rew_sum)

    # ---- free-running -------------------------------------------------------------------------
    def start_free(self):
        """Start a free-running oracle from the GPU state now."""
        self.free = self._oracle(self.env.get_state())
        self.free_metrics0 = self.env.metrics.double().cpu().numpy().copy()
        self.free_rew = None
        self.free_rew_sum = np.zeros(len(self.picks))
        self.free_rew_scale = np.zeros(len(self.picks))
        self.free_steps = 0

    def _advance_free_one(self, acts_picked):
        od, pe = self._noise(self.step_index, self.epoch[self.picks])
        self.free_rew = self.free.step(acts_picked, od, pe)
        self.free_rew_sum += self.free_rew.mean(axis=1)
        self.free_rew_scale += np.abs(self.free_rew).mean(axis=1) + 1.0
        self.free_steps += 1

    def advance_free(self, acts):
        """Account for a step the GPU took outside :meth:`step` (e.g. inside ``run``): discrete state and free oracle."""
        self._advance_discrete(acts)
        self._advance_free_one(acts[self.picks])
        self.step_index += 1
        self.n_steps += 1

    def check_free(self, what="free-running"):
        got, rew, obs = self._gpu()
        self._check_all_replicas(got, what)
        self._check_picked(got, self.free, rew, self.free_rew, obs, False, what)
        m = self.env.metrics.double().cpu().numpy() - self.free_metrics0
        assert np.all(m[:, 0] == self.free_steps), m[:, 0]
        rel = tolerances(self.precision, False)["rel"]
        err = np.abs(m[self.picks, 1] - self.free_rew_sum)
        assert np.all(err <= rel * self.free_rew_scale), (what, m[self.picks, 1], self.free_rew_sum)


def same_state(a, b):
    """Every plane of two handles bit for bit (the keys a handle has)."""
    import torch

    for k in KEYS:
        if k in a.state and a.state[k] is not None:
            assert torch.equal(a.state[k], b.state[k]), k
