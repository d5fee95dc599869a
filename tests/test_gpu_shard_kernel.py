"""The single persistent kernel of the general path (``k_shard``, csrc/drsim_shard.cuh): clusters larger
than a tile and ONE cluster split by houses across several handles (BASELINE config 5, SURVEY 8e row 2;
reference: cluster.py:73-89, environment.py:72-108).

* bit-identity with the four-kernel path it replaces (k_house -> k_reduce -> k_env -> k_obs);
* the PEER exchange (partial sums + halo records stored into the peers' inboxes from inside the kernel,
  bounded in-kernel wait) driven on ONE GPU: three handles attached with raw device pointers
  (``drsim_peer_attach_local``), each stepped on its own stream, against the unsharded cluster.
"""
import copy
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

KEYS_STATE = ("sso", "flags", "reward", "obs", "signal", "power", "od_temp", "base_power", "metrics", "pen_sum", "pen_max",
              "rew_sig", "epoch")


def _prop(n, **over):
    p = {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": 4.0,
         "cluster_prop": {"nb_agents": n, "house_prop": {"target_temp": 19.0}}}
    for path, v in over.items():
        d = p
        keys = path.split("/")
        for k in keys[:-1]:
            d = d.setdefault(k, {})
        d[keys[-1]] = v
    return p


class _env_var:
    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        for k, v in self.kv.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = str(v)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _temps(state):
    return ("dt_air", "dt_mass") if state["temp_is_deviation"] else ("t_air", "t_mass")


CASES = [
    # n, R, layout, precision, overrides, steps, tsmem (None = planned)
    (3000, 2, "tarmac", "f32", {}, 12, None),
    (3000, 2, "tarmac", "f32", {}, 12, 0),            # post-update state re-read from L2 instead of shared memory
    (5000, 3, "tarmac", "f32", {}, 6, 1),             # mixed: first tile of a CTA saved, the rest re-read
    (2500, 2, "hand_engineered", "f32", {}, 10, None),
    (1300, 3, "hand_engineered", "f64", {"reward_prop/penalty_props/mode": "mixture"}, 8, None),
    (1027, 2, "tarmac", "f64", {"reward_prop/penalty_props/mode": "common_max_error"}, 8, None),
    (2200, 2, "hand_engineered", "f32", {"cluster_prop/agents_comm_prop/mode": "closed_groups"}, 8, None),
    (130, 5, "hand_engineered", "f32", {"power_grid_prop/base_power_props/mode": "interpolation",
                                        "power_grid_prop/base_power_props/interp_update_period": 12}, 14, None),
    (2600, 2, "tarmac", "f32", {"power_grid_prop/base_power_props/mode": "interpolation",
                                "power_grid_prop/base_power_props/interp_update_period": 12,
                                "power_grid_prop/signal_properties/mode": "sinusoidals"}, 10, None),
]


@pytest.mark.parametrize("n,R,layout,precision,over,T,tsmem", CASES)
def test_single_kernel_step_is_bit_identical_to_the_four_kernel_path(n, R, layout, precision, over, T, tsmem):
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.config import synthetic_table

    prop = _prop(n, **over)
    interp = "interpolation" in str(over)
    table = synthetic_table(7) if interp else None
    st = synthetic_state(prop, R, seed=3)
    with _env_var(DRSIM_NO_SHARD_KERNEL=None, DRSIM_SHARD_TSMEM=tsmem):
        one = BatchedEnv(prop, R, precision=precision, obs_layout=layout, noise="philox", seed=9, path="split", interp_table=table)
    with _env_var(DRSIM_NO_SHARD_KERNEL=1):
        four = BatchedEnv(prop, R, precision=precision, obs_layout=layout, noise="philox", seed=9, path="split", interp_table=table)
    one.reset(copy.deepcopy(st))
    four.reset(copy.deepcopy(st))
    acts = (np.random.default_rng(2).random((T, R, n)) < 0.5).astype(np.uint8)
    l0, l1 = one.sim.launch_count, four.sim.launch_count
    for t in range(T):
        a = torch.as_tensor(acts[t], device="cuda")
        one.step(a)
        four.step(a)
    torch.cuda.synchronize()
    one.sim.peer_status()
    # one launch per step (+ the schedule kernels after an interpolator firing) against four
    assert one.sim.launch_count - l0 <= (four.sim.launch_count - l1) - 3 * T
    for k in KEYS_STATE + _temps(one.state):
        assert torch.equal(one.state[k], four.state[k]), k


def _sharded_vs_whole(layout, base_mode, W, n, R, T, no_shard_kernel=False, resets=0):
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.core import DrSim
    from marl_demandresponse_b200.sharded import ShardedClusterEnv
    from oracle.config import synthetic_table

    table = synthetic_table(7)
    prop = _prop(n, **{"power_grid_prop/base_power_props/mode": base_mode,
                       "power_grid_prop/base_power_props/interp_update_period": 20,
                       "power_grid_prop/signal_properties/mode": "sinusoidals"})
    with _env_var(DRSIM_NO_SHARD_KERNEL=1 if no_shard_kernel else None):
        whole = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=9, path="split",
                           interp_table=table if base_mode == "interpolation" else None)
        parts = [ShardedClusterEnv(prop, R, rank=r, world=W, obs_layout=layout, noise="philox", seed=9) for r in range(W)]
    DrSim.peer_attach_local([p_.sim for p_ in parts])
    for p_ in parts:
        p_.exchange, p_.world = "peer", W    # (constructed rank by rank without a process group)
    streams = [torch.cuda.Stream() for _ in parts]
    rng = np.random.default_rng(2)
    for episode in range(resets + 1):
        st = synthetic_state(prop, R, seed=3 + episode)
        whole.reset(copy.deepcopy(st))
        for p_ in parts:
            if base_mode == "interpolation":
                p_.sim.set_interp_table(table)
            p_.reset(copy.deepcopy(st))
            # the signal computed at reset by the unsharded env is an input of the sharded ones
            p_.sim.set_state({k: whole.get_state([k])[k] for k in ("signal", "base_power", "t_since_interp")})
        torch.cuda.synchronize()
        acts = (rng.random((T, R, n)) < 0.5).astype(np.uint8)
        for t in range(T):
            a = torch.as_tensor(acts[t], device="cuda")
            whole.step(a)
            torch.cuda.synchronize()
            # every shard on its own stream: the kernels of the shards wait for one another's stores
            for p_, s in zip(parts, streams):
                with torch.cuda.stream(s):
                    p_.state["actions"].copy_(a[:, p_.lo:p_.hi])
                    p_.step(None)
        torch.cuda.synchronize()
        for p_ in parts:
            p_.sim.peer_status()
        ws = whole.state
        wm = ws["metrics"].cpu().numpy()
        # every reset starts the running metrics from zero: one episode's steps, whole-cluster sums on every shard
        # (folded in another order: fp32 tolerance of the summed values, the reward sum also of 1 per step)
        assert np.all(wm[:, 0] == T), (episode, wm[:, 0])
        mtol = 1e-5 * np.abs(wm)
        mtol[:, 1] += 1e-5 * T
        for p_ in parts:
            ps = p_.state
            pm = ps["metrics"].cpu().numpy()
            assert np.array_equal(pm[:, 0], wm[:, 0]), (layout, base_mode, episode, p_.rank)
            assert np.all(np.abs(pm - wm) <= mtol), (layout, base_mode, episode, p_.rank, pm, wm)
            for k in ("sso", "flags", "dt_air", "dt_mass"):
                assert torch.equal(ws[k][:, p_.lo:p_.hi], ps[k]), (layout, base_mode, episode, k)
            for k in ("power", "signal", "od_temp", "base_power"):
                torch.testing.assert_close(ws[k], ps[k], rtol=1e-12, atol=0)
            torch.testing.assert_close(ws["reward"][:, p_.lo:p_.hi], ps["reward"], rtol=1e-6, atol=1e-7)
            torch.testing.assert_close(ws["obs"][:, p_.lo:p_.hi], ps["obs"], rtol=1e-6, atol=1e-7)
    return parts


@pytest.mark.parametrize("layout,base_mode", [("tarmac", "constant"), ("hand_engineered", "constant"), ("tarmac", "interpolation")])
def test_peer_exchange_between_three_handles_on_one_gpu(layout, base_mode):
    """The in-kernel peer exchange (partial sums pushed into every peer's inbox, halo records into the two
    adjacent ones, bounded acquire-wait) needs no second GPU to be exercised: three shards of one cluster live
    on this GPU and are stepped on three streams."""
    parts = _sharded_vs_whole(layout, base_mode, W=3, n=7000, R=2, T=45 if base_mode == "interpolation" else 12)
    assert all(p_.sim.launch_count > 0 for p_ in parts)


def test_peer_exchange_four_kernel_variant_on_one_gpu():
    """Same exchange through the begin / finish pair (k_reduce pushes, k_env waits): the path a rollback to the
    four-kernel step would take."""
    _sharded_vs_whole("hand_engineered", "constant", W=2, n=4100, R=2, T=8, no_shard_kernel=True)


def test_peer_exchange_survives_short_episodes_and_resets():
    """Exchange flags are stamped with a sequence number that never restarts: after a 3-step episode and a
    re-injected state the next episode must not find `its` flag already set by the previous one (a stale row
    would be combined instead of the peers' new partial sums)."""
    _sharded_vs_whole("hand_engineered", "constant", W=3, n=6000, R=1, T=3, resets=3)


def test_exchange_timeout_is_reported_not_silent():
    """A shard whose peers never step gives up after its bounded wait, flags the error, and every later step on
    the handle fails loudly (DRSIM_E_STATE) instead of combining whatever the inbox holds."""
    import torch

    from marl_demandresponse_b200._lib import DrsimError
    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.core import DrSim
    from marl_demandresponse_b200.sharded import ShardedClusterEnv

    prop = _prop(4000)
    parts = [ShardedClusterEnv(prop, 1, rank=r, world=2, obs_layout="tarmac", noise="philox", seed=9) for r in range(2)]
    DrSim.peer_attach_local([p_.sim for p_ in parts])
    st = synthetic_state(prop, 1, seed=3)
    for p_ in parts:
        p_.exchange, p_.world = "peer", 2
        p_.reset(copy.deepcopy(st))
    parts[0].step(None)            # rank 1 never steps: rank 0 waits ~2 s in the kernel, then gives up
    torch.cuda.synchronize()
    with pytest.raises(DrsimError, match="timed out"):
        parts[0].sim.peer_status()
    with pytest.raises(DrsimError, match="timed out"):
        parts[0].step(None)
