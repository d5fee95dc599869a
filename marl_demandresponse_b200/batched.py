"""``BatchedEnv``: thousands of independent cluster replicas stepped by one kernel launch.

The torch tensors handed out by :attr:`BatchedEnv.state`, ``obs`` and ``reward`` alias the
library's device buffers (zero-copy); nothing is copied per step.  ``step`` is ordered on the
caller's current CUDA stream.
"""
from __future__ import annotations

import datetime as _dt
from typing import Any, Dict, Optional

import numpy as np

from .core import DrSim, comm_width, flatten_config, to_epoch
from .properties import EnvironmentProperties, as_props


def ring_table(n: int, c: int) -> np.ndarray:
    """``neighbours`` mode table (agent_communication_builder.py:63-85), [N, c] int32."""
    i = np.arange(n)[:, None]
    lo, hi = c // 2, (c + 1) // 2
    before = (i - lo + np.arange(lo)[None, :]) % n
    after = (i + 1 + np.arange(hi)[None, :]) % n
    return np.concatenate([before, after], axis=1).astype(np.int32)


def synthetic_state(props: Any, n_rep: int, seed: int = 1234, rep_offset: int = 0,
                    start: Optional[_dt.datetime] = None, quirk_ua: bool = False) -> Dict[str, np.ndarray]:
    """Seeded synthetic cluster state (SURVEY.md section 8d): identical for a given global replica
    index whatever the placement (each replica draws from ``default_rng([seed, replica])``).

    per house: ``target = t0 + |N(0,1)|``, ``Ta, Tm = target + U(-2, 4)``, thermal parameters =
    defaults x triangular(0.9, 1.1, 1) (``quirk_ua``: Ua = the bare factor, quirk Q1), capacity
    uniform in the configured list, ``on`` ~ Bernoulli(0.5), ``sso`` = 0 if on else 4 U{0..15}.
    """
    p = as_props(props)
    hp, hv = p.cluster_prop.house_prop, p.cluster_prop.house_prop.hvac_prop
    N, R = p.cluster_prop.nb_agents, int(n_rep)
    dur, dt = hv.lockout_duration, int(p.time_step.seconds)
    caps = np.asarray(hv.noise_prop.cooling_capacity_list, dtype=np.float64)
    lo, hi = hp.noise_prop.factor_thermo_low, hp.noise_prop.factor_thermo_high
    st = {k: np.empty((R, N)) for k in ("t_air", "t_mass", "target", "Ua", "Ca", "Cm", "Hm", "cap")}
    st["on"] = np.empty((R, N), dtype=np.uint8)
    st["lockout"] = np.empty((R, N), dtype=np.uint8)
    st["sso"] = np.empty((R, N), dtype=np.int32)
    for r in range(R):
        g = np.random.default_rng([seed, rep_offset + r])
        tgt = hp.target_temp + np.abs(g.normal(0.0, hp.noise_prop.std_target_temp, N))
        st["target"][r] = tgt
        st["t_air"][r] = tgt + g.uniform(-2.0, 4.0, N)
        st["t_mass"][r] = tgt + g.uniform(-2.0, 4.0, N)
        f = g.triangular(lo, 1.0, hi, (4, N))
        st["Ua"][r] = f[0] if quirk_ua else hp.Ua * f[0]
        st["Cm"][r], st["Ca"][r], st["Hm"][r] = hp.Cm * f[1], hp.Ca * f[2], hp.Hm * f[3]
        st["cap"][r] = caps[g.integers(0, len(caps), N)]
        on = g.random(N) < 0.5
        sso = np.where(on, 0, dt * g.integers(0, 16, N))
        st["on"][r], st["sso"][r] = on, sso
        st["lockout"][r] = (~on) & (sso < dur)
    when = start or _dt.datetime(2021, 6, 15, 12, 0, 0)
    tp = p.temp_prop
    t_day = when.hour + when.minute / 60.0
    od = (tp.day_temp - tp.night_temp) / 2.0 * np.sin(2 * np.pi * (t_day - 6.0 + tp.phase) / 24.0) \
        + (tp.day_temp + tp.night_temp) / 2.0
    st["epoch"] = np.full(R, to_epoch(when), dtype=np.int64)
    st["od_temp"] = np.full(R, od)
    st["signal"] = np.zeros(R)
    st["base_power"] = np.zeros(R)
    st["artificial_ratio"] = np.full(R, p.power_grid_prop.artificial_ratio)
    st["max_power"] = np.full(R, N * hv.cooling_capacity / hv.cop)
    st["power"] = np.where(st["on"] > 0, st["cap"] / hv.cop, 0.0).sum(axis=1)
    st["solar"] = np.zeros(R)
    return st


def reset_counter(props: Any, state: Dict[str, np.ndarray], n_rep: int) -> Dict[str, np.ndarray]:
    """``state`` with the interpolator's counter of a new episode: the reference builds a new ``PowerGrid`` at every
    reset, whose counter starts at ``interp_update_period + 1`` (power_grid.py:64-66), so the interpolator fires at
    the reset.  A state that carries ``t_since_interp`` keeps its own."""
    if "t_since_interp" in state:
        return state
    period = as_props(props).power_grid_prop.base_power_props.interp_update_period
    return {**state, "t_since_interp": np.full(n_rep, period + 1, dtype=np.int32)}


class BatchedEnv:
    """R independent replicas of the reference's cluster environment on one GPU.

    Parameters mirror ``Environment`` plus: ``n_replicas``; ``obs_layout`` in
    {"hand_engineered", "tarmac", "none"}; ``policy`` ("external" actions or an on-device
    controller); ``noise`` ("philox": counter-based streams keyed by (replica, step); "zero");
    ``rep_offset`` = global index of the first local replica (sharding across GPUs); ``obs_dtype`` =
    "float32" or "bfloat16" (fp32 build: the rows are written, stored and handed out in bf16, each element the
    fp32 value rounded to nearest-even).
    """

    def __init__(self, env_props: Any = None, n_replicas: int = 1, device: int = 0, precision: str = "f32",
                 obs_layout: str = "hand_engineered", policy: str = "external", noise: str = "philox",
                 seed: int = 0, path: str = "auto", rep_offset: int = 0, interp_table: Optional[np.ndarray] = None,
                 obs_dtype: str = "float32"):
        self.props: EnvironmentProperties = as_props(env_props)
        self.init_props = self.props
        self.n_replicas = int(n_replicas)
        self.n_houses = int(self.props.cluster_prop.nb_agents)
        self.rep_offset = int(rep_offset)
        self.seed = int(seed)
        cfg = flatten_config(self.props, n_replicas, precision, obs_layout, policy, noise, seed, path,
                             rep_offset=rep_offset, obs_dtype=obs_dtype)
        self.sim = DrSim(cfg, device)
        self.device = device
        self.comm_mode = self.props.cluster_prop.agents_comm_prop.mode
        self.comm_width = comm_width(self.props)
        # a table mode's static table is drawn once: here when the rows carry messages, else at the first
        # neighbour_index(); `random_sample` draws on the device every step instead (no table)
        self._table: Optional[np.ndarray] = None
        if self._table_mode() and obs_layout == "hand_engineered":
            self._table = self._static_table()
            self.sim.set_comm_table(self._table)
        if interp_table is not None:
            self.sim.set_interp_table(interp_table)
        self._v = self.sim.views()

    # ---- neighbour index tensor (TarMAC attention mask / message routing) -----------------
    def _table_mode(self) -> bool:
        return self.comm_mode not in ("neighbours", "random_sample") and self.comm_width > 0

    def _static_table(self) -> np.ndarray:
        from .environment import build_comm_table

        return build_comm_table(self.props)

    def neighbour_index(self, draw: Optional[int] = None):
        """int32 neighbour tensor on the device.  ``random_sample``: ``[R, N, c]``, the neighbours behind the current
        observation rows, or those of draw ``draw`` (the draw index is the step count the rows were written at, see
        ``DrSim.step_count``).  Other modes: the mode's static ``[N, c]`` table."""
        import torch

        if self.comm_mode == "random_sample":
            return self.sim.comm_sample(draw)
        if self._table is None and self._table_mode():
            self._table = self._static_table()
        t = self._table if self._table is not None else ring_table(self.n_houses, self.comm_width)
        return torch.as_tensor(t, device=f"cuda:{self.device}")

    # ---- reset / state --------------------------------------------------------------------
    def reset(self, state: Optional[Dict[str, np.ndarray]] = None, seed: Optional[int] = None,
              device_mode: Optional[str] = None, quirk_ua: bool = True):
        """Inject ``state`` (default: the seeded synthetic state), compute the first regulation
        signal (``PowerGrid.step`` at reset, environment.py:66-68) and return the observations.
        ``device_mode`` = "reference" | "synthetic" draws the state on the GPU instead
        (``drsim_reset``: the reference's reset distributions from Philox streams).  Either way a new episode
        begins: the running metrics (``metrics``) start again from zero, and an interpolated base power is
        computed afresh (the counter starts at ``interp_update_period + 1`` unless ``state`` carries
        ``t_since_interp``)."""
        if device_mode is not None:
            self.sim.reset_device(self.props, self.seed if seed is None else seed, device_mode, quirk_ua)
            self.sim.refresh(True)
            return self.obs
        if state is None:
            state = synthetic_state(self.props, self.n_replicas, self.seed if seed is None else seed, self.rep_offset)
        self.sim.set_state(reset_counter(self.props, state, self.n_replicas))
        self._v["metrics"].zero_()   # on the current stream, like drsim_reset
        self.sim.refresh(True)
        return self.obs

    def set_state(self, state: Dict[str, np.ndarray]) -> None:
        """Overwrite the given planes (restoring a state mid-episode): the running metrics keep counting."""
        self.sim.set_state(state)

    def get_state(self, keys=None) -> Dict[str, np.ndarray]:
        return self.sim.get_state(keys)

    @property
    def state(self) -> Dict[str, Any]:
        """Zero-copy torch views: ``dt_air, dt_mass`` (fp32: Ta/Tm minus set-point) or
        ``t_air, t_mass`` (fp64), ``sso`` i32, ``flags`` u8 (bit0 on, bit1 lockout), ``target``,
        ``cap`` -- all ``[R, N]``; per-replica ``epoch, od_temp, signal, base_power, power`` ``[R]``."""
        return self._v

    @property
    def obs(self):
        return self._v["obs"]

    @property
    def reward(self):
        return self._v["reward"]

    @property
    def power(self):
        return self._v["power"]

    @property
    def signal(self):
        return self._v["signal"]

    @property
    def od_temp(self):
        return self._v["od_temp"]

    @property
    def metrics(self):
        return self._v["metrics"]

    # ---- stepping -------------------------------------------------------------------------
    def step(self, actions=None, od_noise=None, perlin=None, interp_ids=None):
        """One environment step of every replica.  ``actions``: CUDA uint8/bool tensor ``[R, N]``
        (ignored by on-device policies).  Returns ``(obs [R,N,D], reward [R,N])`` views."""
        sim = self.sim
        a = None
        if actions is not None:
            if actions.dtype != self._v["actions"].dtype:
                actions = actions.to(self._v["actions"].dtype)
            if sim.N == sim.Ns and actions.is_contiguous() and tuple(actions.shape) == (sim.R, sim.N):
                a = actions  # read in place, no copy
            else:
                self._v["actions"].copy_(actions)
        sim.step(a, od_noise, perlin, interp_ids)
        return self._v["obs"], self._v["reward"]

    def run(self, n_steps: int, action_tape=None, rotate: bool = False):
        """``n_steps`` steps in one C call (``drsim_run``): a rollout under an on-device policy
        (``action_tape`` None) or the replay of recorded actions, ``action_tape`` u8 CUDA ``[n_steps, R, N]``
        (or ``[R, N]``: the same actions every step; ``rotate=True``: ``[T, R, N]``, step k replays plane
        ``k % T``).  Same results as ``n_steps`` calls of :meth:`step`."""
        sim = self.sim
        if action_tape is not None:
            if action_tape.dtype != self._v["actions"].dtype:
                action_tape = action_tape.to(self._v["actions"].dtype)
            if sim.N != sim.Ns:   # pad the house axis to the plane stride
                import torch

                padded = torch.zeros(tuple(action_tape.shape[:-1]) + (sim.Ns,), dtype=action_tape.dtype, device=action_tape.device)
                padded[..., :sim.N] = action_tape
                action_tape = padded
            action_tape = action_tape.contiguous()
        sim.run(n_steps, action_tape, rotate=rotate)
        return self._v["obs"], self._v["reward"]

    # ---- on-device MA-PPO actor (SURVEY 8f-2) ----------------------------------------------
    @staticmethod
    def actor_weights(actor) -> tuple:
        """``(w1, b1, w2, b2, w3, b3)`` fp32 CUDA tensors of a reference-style ``Actor`` module
        (``network.py:14-35``: ``actor.fc`` = three ``nn.Linear``) or of any sequence of three
        ``(weight, bias)`` pairs."""
        import torch

        layers = list(actor.fc) if hasattr(actor, "fc") else list(actor)
        if len(layers) != 3:
            raise ValueError("the on-device actor is the reference's two-hidden-layer MLP (three Linear layers)")
        out = []
        for lin in layers:
            w, b = (lin.weight, lin.bias) if hasattr(lin, "weight") else lin
            out += [w.detach().to(device="cuda", dtype=torch.float32).contiguous(),
                    b.detach().to(device="cuda", dtype=torch.float32).contiguous()]
        return tuple(out)

    def policy_step(self, weights, seed: Optional[int] = None, want_prob: bool = True, precision: str = "tf32x3"):
        """``MAPPO.select_actions`` (mappo.py:83-97) for all ``R * N`` agents in one kernel: actor
        forward on the current observation rows (tcgen05 TF32 GEMMs), softmax, categorical draw from a
        Philox uniform keyed (seed, replica, house, step).  The drawn actions land in the action plane
        (``state["actions"]``); returns ``(actions u8 [R,N], prob_of_drawn_action f32 [R,N] | None)``.
        ``precision``: "tf32x3" (default), "f16x3" or "tf32", see :meth:`DrSim.policy_step`."""
        import torch

        sim = self.sim
        prob = None
        if want_prob:
            if getattr(self, "_prob", None) is None:
                self._prob = torch.zeros((sim.R, sim.Ns), dtype=torch.float32, device=f"cuda:{self.device}")
            prob = self._prob
        sim.policy_step(weights, self.seed if seed is None else seed, prob_drawn=prob, precision=precision)
        return self._v["actions"], (prob[:, :sim.N] if prob is not None else None)

    def rollout_step(self, weights, seed: Optional[int] = None, precision: str = "tf32x3"):
        """One transition of a rollout entirely on the device: actor + draw, then the environment
        step on the drawn actions.  Returns ``(obs', reward, actions, prob_of_drawn_action)``.  ``precision`` as for
        :meth:`policy_step`."""
        actions, prob = self.policy_step(weights, seed, precision=precision)
        self.sim.step(None)
        return self._v["obs"], self._v["reward"], actions, prob

    def collect(self, weights, buf, n_steps=None, seed: Optional[int] = None, done_last: bool = False,
                precision: str = "tf32x3"):
        """A rollout segment entirely on the device, stored in a :class:`~.rollout.RolloutBuffer` (SURVEY 8f-2:
        ``select_actions`` + ``env.step`` + ``store_transition`` of mappo.py:83-127 per transition, one C call).
        ``precision`` as for :meth:`policy_step`; with "f16x3" the segment ends with ``actor_status``, which raises if an
        operand left the fp16 range during the segment."""
        from .rollout import collect

        return collect(self, weights, buf, n_steps, seed, done_last, precision=precision)

    def step_host(self, actions_host, env_out=None, reward_out=None, obs_out=None):
        """End-to-end step with HOST buffers: ``actions_host`` uint8 / bool ``[R, N]`` (pinned torch CPU
        tensor or numpy, values 0 / 1) is copied in, the per-replica results ``[R, 4]`` = (power, signal,
        outdoor temperature, mean reward) are copied back.  With ``reward_out [R, N]`` / ``obs_out [R, N, D]``
        (host buffers of the build's dtype) the reference's full ``step`` result -- per-agent observations
        and rewards, environment.py:108 -- comes back too (``drsim_step_host_full``)."""
        return self.sim.step_host(actions_host, env_out=env_out, reward_out=reward_out, obs_out=obs_out)

    def clone(self) -> "BatchedEnv":
        other = object.__new__(BatchedEnv)
        other.__dict__.update(self.__dict__)
        other.sim = self.sim.clone()
        other._v = other.sim.views()
        return other

    __deepcopy__ = lambda self, memo: self.clone()  # noqa: E731
