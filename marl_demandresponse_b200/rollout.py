"""Device-resident MA-PPO rollout storage (SURVEY.md section 8f-2).

The reference collects its rollout with three Python loops per step -- ``select_actions`` (one batch-1 actor forward
per agent, mappo.py:83-97), ``env.step``, ``store_transition`` (one ``Transition`` namedtuple per agent holding the
state vector, the action, the OTHER agents' actions, the action probability, the reward and the next state,
mappo.py:105-127; driven by training_manager.py:224-240) -- and turns the list into tensors again in ``update``
(mappo.py:129-152).  Here the transitions are written where ``update`` wants them, by the kernels themselves:

    buf = RolloutBuffer(env, horizon)          # torch CUDA tensors, plane layout of the simulator
    env.collect(weights, buf)                  # horizon x drsim_rollout_transition, nothing leaves the GPU
    buf.state(t), buf.action(t), buf.prob(t), buf.reward(t), buf.next_state(t), buf.others_actions(t)
    buf.returns(gamma)                         # Gt of mappo.py:147-152

``obs[t]`` is ``state_t`` and ``obs[t + 1]`` is ``next_state_t``: the rows are stored once.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

from . import _lib


class RolloutBuffer:
    def __init__(self, env, horizon: int):
        import torch

        sim = env.sim
        self._env = env
        if sim.real is not __import__("numpy").float32 or not sim.D:
            raise ValueError("the on-device rollout needs the fp32 build with an observation layout")
        self.sim, self.T = sim, int(horizon)
        R, N, Ns, D = sim.R, sim.N, sim.Ns, sim.D
        self.R, self.N, self.Ns, self.D = R, N, Ns, D
        dev = f"cuda:{sim.device}"
        # obs[t] is one contiguous plane; the transition needs each plane on a 16-byte boundary, which a bf16 plane of
        # odd width (R Ns D 2 bytes) does not keep by itself: planes are spaced by a stride padded to 16 bytes
        dtype, per16 = (torch.bfloat16, 8) if sim.obs_bf16 else (torch.float32, 4)
        stride = (R * Ns * D + per16 - 1) // per16 * per16
        flat = torch.zeros((self.T + 1) * stride, dtype=dtype, device=dev)
        self.obs = flat.as_strided((self.T + 1, R, Ns, D), (stride, Ns * D, D, 1))
        self.actions = torch.zeros((self.T, R, Ns), dtype=torch.uint8, device=dev)
        self.probs = torch.zeros((self.T, R, Ns), dtype=torch.float32, device=dev)
        self.rewards = torch.zeros((self.T, R, Ns), dtype=torch.float32, device=dev)
        self.done = torch.zeros((self.T,), dtype=torch.bool, device=dev)
        self.filled = 0
        self.draw0 = 0   # step count of the handle when obs[0] was written (`random_sample` draw index of obs[0])

    # ---- Transition fields (mappo.py:23-35), [R, N, ...] views of step t ---------------------
    def state(self, t: int):
        return self.obs[t, :, :self.N]

    def next_state(self, t: int):
        return self.obs[t + 1, :, :self.N]

    def action(self, t: int):
        return self.actions[t, :, :self.N]

    def prob(self, t: int):
        return self.probs[t, :, :self.N]

    def reward(self, t: int):
        return self.rewards[t, :, :self.N]

    def neighbour_index(self, t: int):
        """``random_sample`` handle: the ``[R, N, c]`` neighbour table behind ``obs[t]`` (its draw is
        ``draw0 + t``); other modes: the handle's static table."""
        if self._env.comm_mode == "random_sample":
            return self.sim.comm_sample(self.draw0 + int(t))
        return self._env.neighbour_index()

    def others_actions(self, t: int):
        """``[R, N, N - 1]``: for every agent the actions of all OTHER agents of its cluster in id order
        (``action_k.pop(observation_id)``, mappo.py:113-116) -- a gather of the action plane, built on demand."""
        import torch

        a = self.action(t)                                            # [R, N]
        n = self.N
        idx = torch.arange(n, device=a.device)
        cols = torch.arange(n - 1, device=a.device)[None, :] + (torch.arange(n - 1, device=a.device)[None, :] >= idx[:, None]).long()
        return a[:, cols]                                             # [R, N, N - 1]

    def returns(self, gamma: float):
        """``Gt`` of mappo.py:147-152 per agent, ``[T, R, N]``: ``R = reward + gamma * R``, reset where ``done``."""
        import torch

        out = torch.empty((self.filled, self.R, self.N), dtype=torch.float32, device=self.rewards.device)
        run = torch.zeros((self.R, self.N), dtype=torch.float32, device=self.rewards.device)
        for t in reversed(range(self.filled)):
            if bool(self.done[t]):
                run = torch.zeros_like(run)
            run = self.reward(t) + gamma * run
            out[t] = run
        return out


def collect(env, weights, buf: RolloutBuffer, n_steps: Optional[int] = None, seed: Optional[int] = None,
            done_last: bool = False, stream=None, precision: str = "tf32x3") -> RolloutBuffer:
    """``n_steps`` (default: the buffer's horizon) rollout transitions on the device, stored in ``buf``:
    per transition ONE C call (``drsim_rollout_transition``: actor + categorical draw, then the environment step
    writing reward and next observation rows straight into the buffer).  ``precision``: the actor's, see
    ``DrSim.policy_step``; "f16x3" ends the segment with ``DrSim.actor_status`` (a synchronisation), which raises if an
    operand left the fp16 range: the segment's actions and probabilities are then not valid."""
    sim = env.sim
    T = buf.T if n_steps is None else int(n_steps)
    if T > buf.T:
        raise ValueError("n_steps exceeds the buffer's horizon")
    net = sim.actor_net(weights, precision)
    buf.obs[0].copy_(sim.views()["obs_padded"])     # state_0 = the rows of the last step / reset (one copy per segment)
    buf.draw0 = sim.step_count
    seed = env.seed if seed is None else int(seed)
    st = sim._stream(stream)
    slot = _lib.RolloutSlot()
    for t in range(T):
        slot.obs, slot.next_obs = buf.obs[t].data_ptr(), buf.obs[t + 1].data_ptr()
        slot.actions, slot.prob, slot.reward = buf.actions[t].data_ptr(), buf.probs[t].data_ptr(), buf.rewards[t].data_ptr()
        _lib.check(sim._L.drsim_rollout_transition(sim._h, C.byref(net), seed & (2 ** 64 - 1), C.byref(slot), st))
    if T:   # the simulator's own planes show the last step's result again (one copy per segment, not per step)
        v = sim.views()
        v["obs_padded"].copy_(buf.obs[T])
        v["reward"].copy_(buf.rewards[T - 1, :, :sim.N])
    buf.done.zero_()
    if done_last and T:
        buf.done[T - 1] = True
    buf.filled = T
    if precision == "f16x3":
        sim.actor_status(stream)
    return buf
