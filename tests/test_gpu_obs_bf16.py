"""Observation rows in bfloat16 (``obs_dtype="bfloat16"`` on the fp32 build).

Every case steps an fp32 handle and a bf16 handle from the same state on the same inputs and checks, after every step,
that each bf16 row element is the fp32 element rounded to nearest-even (bit for bit, zero padding rows included) and
that everything else -- state planes, rewards, env scalars, running metrics -- is bit-identical.  The two handles must
run the same kernels: where the tile planner could pick a different tile size for the narrower rows, DRSIM_TILE_ENVS
pins the fp32 handle's choice on both."""
import copy
import ctypes as C
import os
from contextlib import contextmanager

import numpy as np
import pytest

KEYS = ("dt_air", "dt_mass", "sso", "flags", "reward", "epoch", "od_temp", "signal", "base_power", "power", "solar",
        "pen_sum", "pen_max", "rew_sig", "metrics")


def _prop(n, **over):
    p = {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": 4.0,
         "cluster_prop": {"nb_agents": n, "house_prop": {"target_temp": 19.0},
                          "agents_comm_prop": {"max_nb_agents_communication": 10}},
         "power_grid_prop": {"signal_properties": {"mode": "sinusoidals"}}}
    for path, v in over.items():
        d = p
        keys = path.split("/")
        for k in keys[:-1]:
            d = d.setdefault(k, {})
        d[keys[-1]] = v
    return p


@contextmanager
def _env_var(**kv):
    old = {k: os.environ.get(k) for k in kv}
    for k, v in kv.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _rows_match(f32, b16):
    """Row contract over the padded planes: bf16 element == round-to-nearest-even of the fp32 element."""
    import torch

    assert b16.dtype == torch.bfloat16 and f32.dtype == torch.float32 and b16.shape == f32.shape
    return torch.equal(b16.view(torch.int16), f32.to(torch.bfloat16).view(torch.int16))


def _check(a, b, what=""):
    import torch

    torch.cuda.synchronize()
    assert _rows_match(a.state["obs_padded"], b.state["obs_padded"]), ("rows", what)
    for k in KEYS:
        if a.state.get(k) is not None:
            assert torch.equal(a.state[k], b.state[k]), (k, what)


def _pair(prop, R, tile_envs=None, env=None, **kw):
    """fp32 and bf16 BatchedEnv on the same kernels (same fused variant and tile size; the grid may differ where the
    narrower rows let more CTAs share an SM -- tiles are independent of one another)."""
    from marl_demandresponse_b200 import BatchedEnv

    with _env_var(**(env or {})):
        with _env_var(DRSIM_TILE_ENVS=tile_envs):
            probe = BatchedEnv(prop, R, **kw)
            e = probe.sim.fused_info()["envs_per_tile"]
        del probe
        with _env_var(DRSIM_TILE_ENVS=e if e > 0 else tile_envs):
            a = BatchedEnv(prop, R, **kw)
            b = BatchedEnv(prop, R, obs_dtype="bfloat16", **kw)
    if a._table is not None:   # random neighbour modes draw their table per environment: give both the same one
        b._table = a._table
        b.sim.set_comm_table(a._table)
    ia, ib = a.sim.fused_info(), b.sim.fused_info()
    assert all(ia[k] == ib[k] for k in ("variant", "envs_per_tile", "tiles")), (ia, ib)
    return a, b


def _drive(a, b, T, seed=8, check_every=True):
    import torch

    R, N = a.n_replicas, a.n_houses
    acts = (np.random.default_rng(seed).random((T, R, N)) < 0.5).astype(np.uint8)
    for t in range(T):
        x = torch.as_tensor(acts[t], device="cuda")
        a.step(x)
        b.step(x)
        if check_every:
            _check(a, b, t)
    _check(a, b, T)


def _reset_both(a, b, prop, R, seed=13):
    from marl_demandresponse_b200.batched import synthetic_state

    st = synthetic_state(prop, R, seed=seed)
    a.reset(copy.deepcopy(st))
    b.reset(copy.deepcopy(st))
    _check(a, b, "reset")


# ---- 1. every kernel that writes rows -----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("R,n,layout,tile_envs,variant", [
    (60, 100, "hand_engineered", 7, "staged_rows"),
    (60, 100, "hand_engineered", 10, None),
    (4096, 100, "hand_engineered", None, "staged_rows"),
    (60, 100, "tarmac", 10, "staged"),
    (6000, 100, "tarmac", 10, "staged"),
    (6000, 100, "hand_engineered", 5, None),
    (700, 40, "hand_engineered", None, None),
    (900, 1000, "tarmac", None, "staged"),
    (600, 1000, "hand_engineered", None, "staged_rows"),
])
def test_fused_variants(R, n, layout, tile_envs, variant):
    prop = _prop(n)
    a, b = _pair(prop, R, tile_envs, obs_layout=layout, noise="philox", seed=21)
    if variant is not None:
        assert b.sim.fused_info()["variant"] == variant
    _reset_both(a, b, prop, R)
    _drive(a, b, 4)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [10, 22, 32])
def test_small_clusters(n):
    import torch

    prop = _prop(n)
    a, b = _pair(prop, 50, obs_layout="hand_engineered", noise="philox", seed=3)
    _reset_both(a, b, prop, 50)
    _drive(a, b, 2)
    l0 = b.sim.launch_count
    x = torch.ones((50, n), dtype=torch.uint8, device="cuda")
    a.step(x)
    b.step(x)
    assert b.sim.launch_count - l0 == 1   # one k_small launch per step
    _check(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("n,R,layout,path,four,launches", [
    (100, 50, "hand_engineered", "split", True, 4),   # k_house / k_reduce / k_env / k_obs
    (100, 50, "hand_engineered", "split", False, 1),  # k_shard, generic rows with messages
    (1500, 3, "tarmac", "auto", False, 1),            # k_shard, plain 10-column rows
    (2500, 2, "hand_engineered", "auto", False, 1),   # k_shard, generic rows with messages
    (1, 40, "hand_engineered", "auto", False, None),
    (5, 40, "tarmac", "auto", False, None),
    (37, 300, "hand_engineered", "auto", False, None),
    (1023, 20, "hand_engineered", "auto", False, None),
    (1025, 3, "tarmac", "auto", False, 1),
])
def test_general_shard_and_ragged(n, R, layout, path, four, launches):
    import torch

    prop = _prop(n)
    a, b = _pair(prop, R, env={"DRSIM_NO_SHARD_KERNEL": 1 if four else None}, obs_layout=layout, noise="philox", seed=5,
                 path=path)
    _reset_both(a, b, prop, R)
    _drive(a, b, 3)
    l0 = b.sim.launch_count
    x = torch.zeros((R, n), dtype=torch.uint8, device="cuda")
    a.step(x)
    b.step(x)
    if launches is not None:
        assert b.sim.launch_count - l0 == launches
    _check(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["neighbours", "random_fixed"])
@pytest.mark.parametrize("flags", ["none", "solar", "all"])
@pytest.mark.parametrize("layout", ["tarmac", "hand_engineered"])
def test_layouts_modes_and_flags(mode, flags, layout):
    over = {"cluster_prop/agents_comm_prop/mode": mode, "cluster_prop/agents_comm_prop/max_nb_agents_communication": 3}
    if flags == "solar":
        over["state_prop"] = {"solar_gain": True}
    if flags == "all":
        over.update({"state_prop": {"solar_gain": True, "thermal": True, "hvac": True},
                     "cluster_prop/message_prop": {"thermal": True, "hvac": True}})
    prop = _prop(60, **over)
    # bf16 rows of odd width leave 4-row groups off the 16-byte grid of the bulk stores: such a handle steps on the
    # four-kernel path, so the fp32 handle is put there too
    from marl_demandresponse_b200 import BatchedEnv

    D = BatchedEnv(prop, 2, obs_layout=layout).sim.D
    odd = D % 2 == 1
    a, b = _pair(prop, 40, env={"DRSIM_NO_SHARD_KERNEL": 1 if odd else None}, obs_layout=layout, noise="philox", seed=9,
                 path="split" if odd else "auto")
    assert (b.sim.fused_info()["variant"] == "none") == odd
    _reset_both(a, b, prop, 40)
    _drive(a, b, 3)


# ---- 2. the in-kernel step loop -------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("n,R,layout,policy,T,pre", [
    (1000, 400, "tarmac", "external", 70, 0),
    (1000, 640, "tarmac", "external", 100, 5),          # starts mid-block, crosses the 64-step boundary
    (1000, 100, "tarmac", "deadband_bangbang", 70, 0),  # on-device policy
    (10, 64, "hand_engineered", "bangbang", 40, 3),     # k_small
])
def test_in_kernel_loop_equals_per_step_launches(n, R, layout, policy, T, pre):
    import torch

    from marl_demandresponse_b200 import BatchedEnv

    a = BatchedEnv(_prop(n), R, policy=policy, noise="philox", seed=7, obs_layout=layout, obs_dtype="bfloat16")
    a.reset()
    ref = BatchedEnv(_prop(n), R, policy=policy, noise="philox", seed=7, obs_layout=layout)
    ref.reset()
    planes = 3
    tape = None
    if policy == "external":
        tape = (torch.rand((planes, R, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(3)) < 0.5).to(torch.uint8)
    for t in range(pre):
        a.step(None if tape is None else tape[t % planes])
        ref.step(None if tape is None else tape[t % planes])
    b = copy.deepcopy(a)
    l0 = a.sim.launch_count
    a.run(T, tape, rotate=True)
    ref.run(T, tape, rotate=True)
    torch.cuda.synchronize()
    assert a.sim.launch_count - l0 <= 3 * ((pre + T + 63) // 64 - pre // 64)   # one step kernel per schedule block
    with _env_var(DRSIM_NO_STREAM=1):
        b.run(T, tape, rotate=True)
    torch.cuda.synchronize()
    assert torch.equal(a.state["obs_padded"].view(torch.int16), b.state["obs_padded"].view(torch.int16))
    for k in KEYS:
        assert torch.equal(a.state[k], b.state[k]), k
    _check(ref, a)


# ---- 3. reset / refresh and interpolation ---------------------------------------------------------------------------

@pytest.mark.gpu
def test_reset_paths():
    prop = _prop(100)
    a, b = _pair(prop, 30, obs_layout="hand_engineered", noise="philox", seed=4)
    _reset_both(a, b, prop, 30)
    a.reset(device_mode="reference")
    b.reset(device_mode="reference")
    _check(a, b, "device reset")
    _drive(a, b, 2)


@pytest.mark.gpu
def test_interpolation_steps():
    from oracle.config import synthetic_table

    table = synthetic_table(7)
    prop = _prop(1000, **{"power_grid_prop/base_power_props/mode": "interpolation",
                          "power_grid_prop/base_power_props/interp_update_period": 12})
    a, b = _pair(prop, 2, obs_layout="hand_engineered", noise="philox", seed=11, interp_table=table)
    _reset_both(a, b, prop, 2)
    _drive(a, b, 8)   # the interpolator fires at reset, after 3 steps and after 6


# ---- 4. host-buffer steps and the snapshot --------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["dma", "zerocopy"])
@pytest.mark.parametrize("n,R,layout", [(1000, 300, "tarmac"), (100, 600, "hand_engineered")])
def test_step_host(mode, n, R, layout):
    import torch

    prop = _prop(n)
    with _env_var(DRSIM_HOST_ACTIONS=mode):
        a, b = _pair(prop, R, obs_layout=layout, noise="philox", seed=2)
    _reset_both(a, b, prop, R)
    rng = np.random.default_rng(1)
    for t in range(3):
        acts = torch.from_numpy((rng.random((R, n)) < 0.5).astype(np.uint8)).pin_memory()
        ea, eb = a.step_host(acts), b.step_host(acts)
        assert np.array_equal(ea, eb)
        _check(a, b, t)
    acts = torch.from_numpy((rng.random((R, n)) < 0.5).astype(np.uint8)).pin_memory()
    of = torch.empty((R, n, a.sim.D), dtype=torch.float32).pin_memory()
    ob = torch.empty((R, n, a.sim.D), dtype=torch.bfloat16).pin_memory()
    a.step_host(acts, obs_out=of)
    b.step_host(acts, obs_out=ob)
    _check(a, b, "full")
    assert torch.equal(ob.view(torch.int16), b.state["obs"].cpu().view(torch.int16))
    raw = np.empty((R, n, a.sim.D), dtype=np.uint16)
    b.step_host(acts.numpy(), obs_out=raw)
    a.step_host(acts.numpy(), obs_out=of)
    _check(a, b, "full numpy")
    assert np.array_equal(raw, b.state["obs"].cpu().view(torch.int16).numpy().view(np.uint16))
    snap = b.sim.snapshot()
    assert snap["obs"].dtype == np.uint16 and np.array_equal(snap["obs"], raw)


# ---- 5. actor and rollout -------------------------------------------------------------------------------------------

def _actor(D, h1=32, h2=24):
    import torch

    g = torch.Generator().manual_seed(5)
    ws = []
    for fi, fo in ((D, h1), (h1, h2), (h2, 2)):
        ws += [(torch.randn((fo, fi), generator=g) / fi ** 0.5).cuda(), (0.1 * torch.randn((fo,), generator=g)).cuda()]
    return tuple(w.contiguous() for w in ws)


@pytest.mark.gpu
def test_rollout_equals_fp32_on_rounded_rows():
    import torch

    from marl_demandresponse_b200 import _lib
    from marl_demandresponse_b200.rollout import RolloutBuffer

    n, R, T = 100, 64, 8
    prop = _prop(n, **{"cluster_prop/agents_comm_prop/max_nb_agents_communication": 4})
    a, b = _pair(prop, R, obs_layout="hand_engineered", noise="philox", seed=6)
    _reset_both(a, b, prop, R)
    w = _actor(a.sim.D)
    bb = RolloutBuffer(b, T)
    assert bb.obs.dtype == torch.bfloat16
    b.collect(w, bb, seed=17)
    # fp32 reference: one transition at a time, the rows it reads rounded to bf16 first
    ba = RolloutBuffer(a, T)
    ba.obs[0].copy_(a.state["obs_padded"].to(torch.bfloat16).float())
    net = a.sim.actor_net(w, "tf32x3")
    slot = _lib.RolloutSlot()
    for t in range(T):
        slot.obs, slot.next_obs = ba.obs[t].data_ptr(), ba.obs[t + 1].data_ptr()
        slot.actions, slot.prob, slot.reward = ba.actions[t].data_ptr(), ba.probs[t].data_ptr(), ba.rewards[t].data_ptr()
        _lib.check(a.sim._L.drsim_rollout_transition(a.sim._h, C.byref(net), 17, C.byref(slot), a.sim._stream()))
        torch.cuda.synchronize()
        assert _rows_match(ba.obs[t + 1], bb.obs[t + 1]), t
        ba.obs[t + 1].copy_(ba.obs[t + 1].to(torch.bfloat16).float())
    torch.cuda.synchronize()
    assert torch.equal(ba.actions, bb.actions)
    assert torch.equal(ba.probs, bb.probs)
    assert torch.equal(ba.rewards, bb.rewards)
    for k in ("dt_air", "dt_mass", "sso", "flags", "power", "signal", "metrics"):
        assert torch.equal(a.state[k], b.state[k]), k
    with pytest.raises(Exception, match="3xTF32"):
        b.policy_step(w, precision="tf32")


# ---- 6. a sharded cluster -------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_sharded_ring_messages():
    import torch

    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.core import DrSim
    from marl_demandresponse_b200.sharded import ShardedClusterEnv

    n, R, W, T = 7000, 2, 3, 6
    prop = _prop(n)
    shards = {}
    for dtype in ("float32", "bfloat16"):
        parts = [ShardedClusterEnv(prop, R, rank=r, world=W, obs_layout="hand_engineered", noise="philox", seed=9,
                                   obs_dtype=dtype) for r in range(W)]
        DrSim.peer_attach_local([p_.sim for p_ in parts])
        for p_ in parts:
            p_.exchange, p_.world = "peer", W
            p_.reset(copy.deepcopy(synthetic_state(prop, R, seed=3)))
        shards[dtype] = parts
    streams = [torch.cuda.Stream() for _ in range(W)]
    acts = (np.random.default_rng(2).random((T, R, n)) < 0.5).astype(np.uint8)
    for t in range(T):
        x = torch.as_tensor(acts[t], device="cuda")
        torch.cuda.synchronize()
        for parts in shards.values():
            for p_, s in zip(parts, streams):
                with torch.cuda.stream(s):
                    p_.state["actions"].copy_(x[:, p_.lo:p_.hi])
                    p_.step(None)
            torch.cuda.synchronize()
        for pa, pb in zip(shards["float32"], shards["bfloat16"]):
            pb.sim.peer_status()
            assert _rows_match(pa.state["obs_padded"], pb.state["obs_padded"]), t
            for k in ("dt_air", "dt_mass", "sso", "flags", "reward", "power", "signal"):
                assert torch.equal(pa.state[k], pb.state[k]), (t, k)


# ---- 7. rejections and the ABI ---------------------------------------------------------------------------------------

def test_obs_dtype_in_abi():
    from marl_demandresponse_b200 import _lib

    L = _lib.lib()
    assert L.drsim_abi_version() == _lib.ABI_VERSION == 4
    for which, st in enumerate((_lib.Config, _lib.HostState, _lib.Ptrs, _lib.StepArgs, _lib.ResetArgs)):
        assert L.drsim_sizeof(which) == C.sizeof(st)
    assert _lib.Config.obs_dtype.offset == _lib.Config.penalty_mode.offset + 4
    assert _lib.Ptrs.obs_bytes.offset == _lib.Ptrs.temp_is_deviation.offset + 4


@pytest.mark.parametrize("kw,msg", [({"precision": "f64"}, b"precision"), ({"obs_layout": "none"}, b"observation layout")])
def test_bf16_rejected_without_fp32_rows(kw, msg):
    from marl_demandresponse_b200 import _lib, flatten_config

    args = {"precision": "f32", "obs_layout": "tarmac", **kw}
    cfg = flatten_config(_prop(20), 1, args["precision"], args["obs_layout"], obs_dtype="bfloat16")
    L = _lib.lib()
    h = C.c_void_p()
    assert L.drsim_create(C.byref(cfg), 0, C.byref(h)) == -1 and not h.value
    assert msg in L.drsim_last_error()


def test_unknown_obs_dtype_rejected():
    from marl_demandresponse_b200 import flatten_config

    with pytest.raises(ValueError, match="obs_dtype"):
        flatten_config(_prop(20), 1, obs_dtype="float16")
