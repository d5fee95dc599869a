"""BatchedEnv / Philox / drop-in Environment on the GPU, against the NumPy oracle."""
import copy
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


from oracle_driver import OracleDriver, od_noise as _od_noise, oracle_run as _oracle_run, perlin as _perlin
from oracle_driver import prop as _prop


@pytest.mark.parametrize("n,R,layout,path", [(100, 24, "hand_engineered", "auto"), (1000, 6, "tarmac", "auto"),
                                             (1000, 3, "hand_engineered", "auto"), (2500, 2, "hand_engineered", "auto"),
                                             (100, 24, "hand_engineered", "split"), (37, 9, "hand_engineered", "auto"),
                                             # clusters that fit a warp: the one-house-per-lane kernel (k_small)
                                             (10, 7, "hand_engineered", "auto"), (22, 5, "tarmac", "auto"),
                                             (32, 3, "hand_engineered", "auto"), (9, 130, "hand_engineered", "auto")])
def test_batched_env_philox_matches_oracle(n, R, layout, path):
    """Device Philox streams (od noise, perlin-like signal noise) == their NumPy restatement, and the
    whole batched step == the oracle driven by those values."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    T, seed, off = 12, 77, 1000
    prop = _prop(n)
    env = BatchedEnv(prop, R, precision="f32", obs_layout=layout, noise="philox", seed=seed, path=path, rep_offset=off)
    st = synthetic_state(prop, R, seed=5, rep_offset=off)
    env.reset(copy.deepcopy(st))
    rng = np.random.default_rng(3)
    acts = (rng.random((T, R, n)) < 0.5).astype(np.uint8)
    # the values the device streams must produce
    epoch0 = int(st["epoch"][0])
    reps = [off + r for r in range(R)]
    od_noise = _od_noise(seed, reps, range(T))
    perlin = _perlin(seed, reps, [epoch0 + 4 * t for t in range(T + 1)])
    rewards = []
    for t in range(T):
        obs, rew = env.step(torch.as_tensor(acts[t], device="cuda"))
        rewards.append(rew.double().cpu().numpy())
    got = env.get_state()
    orc, rew_ref = _oracle_run(prop, copy.deepcopy(st), acts, od_noise, perlin)
    s = orc.state
    for k in ("on", "lockout", "sso"):
        assert np.array_equal(got[k].astype(np.int64), s[k].astype(np.int64)), k
    assert np.array_equal(got["epoch"], s["epoch"])
    np.testing.assert_allclose(got["od_temp"], s["od_temp"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(got["signal"], s["signal"], rtol=1e-9)
    np.testing.assert_allclose(got["power"], s["power"], rtol=1e-6)
    np.testing.assert_allclose(got["t_air"], s["t_air"], rtol=0, atol=2e-4)
    np.testing.assert_allclose(got["t_mass"], s["t_mass"], rtol=0, atol=2e-4)
    np.testing.assert_allclose(np.array(rewards), rew_ref, rtol=1e-5, atol=1e-5)
    want = orc.obs_vectors()
    if layout == "tarmac":
        want = want[:, :, :10]
    np.testing.assert_allclose(env.obs.double().cpu().numpy(), want, rtol=1e-5, atol=1e-5)
    # rollout metrics: steps and mean reward
    m = env.metrics.cpu().numpy()
    assert np.all(m[:, 0] == T)
    np.testing.assert_allclose(m[:, 1], rew_ref.mean(axis=2).sum(axis=0), rtol=1e-4, atol=1e-4)


def test_fused_and_general_paths_agree_and_are_deterministic():
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    prop = _prop(200)
    R, T = 40, 15
    st = synthetic_state(prop, R, seed=9)
    acts = (np.random.default_rng(1).random((T, R, 200)) < 0.5).astype(np.uint8)
    out = []
    for path in ("fused", "split", "fused"):
        env = BatchedEnv(prop, R, precision="f32", noise="philox", seed=4, path=path)
        env.reset(copy.deepcopy(st))
        for t in range(T):
            env.step(torch.as_tensor(acts[t], device="cuda"))
        torch.cuda.synchronize()
        v = env.state
        out.append({k: v[k].clone().cpu().numpy() for k in ("dt_air", "dt_mass", "sso", "flags", "reward", "obs")})
    for k in out[0]:
        assert np.array_equal(out[0][k], out[2][k]), f"run-to-run difference in {k}"
        if k in ("sso", "flags"):
            assert np.array_equal(out[0][k], out[1][k]), k
        else:
            np.testing.assert_allclose(out[0][k], out[1][k], rtol=2e-6, atol=2e-6)


def test_schedule_records_follow_mixed_step_kinds():
    """The packed schedule records chain every step to the one before it.  A rollout that mixes
    scheduled steps, steps with injected outdoor noise, interpolator firings (every 5th step) and a
    refresh must give the same trajectory on the fused kernels (records) as on the general path
    (inline env epilogue): env scalars identical to the last bit, discrete state bit-exact."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.config import synthetic_table

    table = synthetic_table(7)
    for n, layout, sig in ((96, "hand_engineered", "sinusoidals"), (1000, "tarmac", "perlin")):
        R, T = 7, 70
        prop = _prop(n, **{"power_grid_prop/base_power_props/mode": "interpolation",
                           "power_grid_prop/base_power_props/interp_update_period": 20,
                           "power_grid_prop/signal_properties/mode": sig})
        st = synthetic_state(prop, R, seed=3)
        acts = (np.random.default_rng(2).random((T, R, n)) < 0.5).astype(np.uint8)
        inj = torch.as_tensor(np.random.default_rng(4).normal(size=(T, R)), device="cuda")
        out = {}
        for path in ("fused", "split"):
            env = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=9, path=path, interp_table=table)
            env.reset(copy.deepcopy(st))
            snaps = []
            for t in range(T):
                od = inj[t].contiguous() if t % 11 == 3 else None     # a step that leaves the schedule
                env.step(torch.as_tensor(acts[t], device="cuda"), od_noise=od)
                if t == 40:
                    env.sim.refresh(True)
                if t % 9 == 0 or t == T - 1:
                    torch.cuda.synchronize()
                    snaps.append({k: env.state[k].clone() for k in
                                  ("signal", "od_temp", "base_power", "power", "epoch", "sso", "flags", "dt_air", "reward", "obs",
                                   "metrics")})
            out[path] = snaps
        for a, b in zip(out["fused"], out["split"]):
            for k in ("signal", "od_temp", "base_power", "epoch", "sso", "flags"):
                assert torch.equal(a[k], b[k]), (n, k)
            for k in ("power", "dt_air", "reward", "obs", "metrics"):
                torch.testing.assert_close(a[k], b[k], rtol=2e-6, atol=2e-6)


@pytest.mark.parametrize("R,n,layout,tile_envs,variant", [
    (60, 100, "hand_engineered", 7, "staged_rows"),     # several clusters per tile, per-warp row groups
    (60, 100, "hand_engineered", 10, None),            # largest tile
    (4096, 100, "hand_engineered", None, "staged_rows"),  # BASELINE config 3: 586 tiles on 296 CTAs (2 tiles per CTA)
    (60, 100, "tarmac", 10, "staged"),                 # several clusters per tile, whole-tile rows
    (6000, 100, "tarmac", 10, "staged"),               # ... and two tiles per CTA
    (6000, 100, "hand_engineered", 5, None),           # five clusters per tile, four tiles per CTA
    (700, 40, "hand_engineered", None, None),          # whatever the round-count heuristic picks
    (900, 1000, "tarmac", None, "staged"),             # BASELINE config 4 layout, 3+ tiles per CTA
    (600, 1000, "hand_engineered", None, "staged_rows"),  # 1000-house clusters with D = 50: row groups, inputs through registers
])
def test_fused_kernel_variants_match_general_path(R, n, layout, tile_envs, variant, monkeypatch):
    """Every fused-kernel variant / tile size (forced through DRSIM_TILE_ENVS where the heuristic would
    not pick it at a test-sized R) against the general path on the same inputs: discrete state and env
    scalars bit-exact, continuous values to fp32 rounding; plus the oracle on three replicas."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    if tile_envs is not None:
        monkeypatch.setenv("DRSIM_TILE_ENVS", str(tile_envs))
    prop = _prop(n)
    T = 9
    st = synthetic_state(prop, R, seed=13)
    acts = (np.random.default_rng(8).random((T, R, n)) < 0.5).astype(np.uint8)
    out = {}
    for path in ("fused", "split"):
        env = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=21, path=path)
        if path == "fused":
            info = env.sim.fused_info()
            if variant is not None:
                assert info["variant"] == variant, info
            if tile_envs is not None:
                assert info["envs_per_tile"] == min(tile_envs, 1024 // env.sim.Ns), info
        env.reset(copy.deepcopy(st))
        if path == "fused":   # every step re-anchored on the oracle on three replicas (first, last, mid-tile)
            drv = OracleDriver(env, prop, st)
            assert len(drv.picks) == 3, drv.picks
            for t in range(T):
                drv.step(acts[t])
            drv.check_metrics()
        else:
            for t in range(T):
                env.step(torch.as_tensor(acts[t], device="cuda"))
        torch.cuda.synchronize()
        out[path] = {k: env.state[k].clone() for k in
                     ("signal", "od_temp", "epoch", "sso", "flags", "power", "dt_air", "dt_mass", "reward", "obs", "metrics")}
    a, b = out["fused"], out["split"]
    for k in ("signal", "od_temp", "epoch", "sso", "flags"):
        assert torch.equal(a[k], b[k]), k
    for k in ("power", "dt_air", "dt_mass", "reward", "obs", "metrics"):
        torch.testing.assert_close(a[k], b[k], rtol=2e-6, atol=2e-6)


@pytest.mark.parametrize("n,R,layout,base_mode", [(1000, 300, "tarmac", "constant"), (100, 2500, "hand_engineered", "constant"),
                                                 (100, 64, "tarmac", "interpolation"), (37, 9, "hand_engineered", "constant")])
@pytest.mark.parametrize("host_actions", ["zerocopy", "dma"])
def test_step_host_zero_copy_equals_device_step(n, R, layout, base_mode, host_actions, monkeypatch):
    """drsim_step_host with PINNED host buffers (``zerocopy``: actions read in place over PCIe by the staged
    fused kernel; ``dma``: one linear copy-engine transfer into the poisoned staging plane, consumed by the
    kernel as it lands; results mirrored into mapped memory either way), with pageable buffers
    (explicit copies) and the device-resident step: identical state, identical per-replica results,
    including the steps on which the interpolator fires (general path) and padded rows (N % 4 != 0)."""
    import torch

    monkeypatch.setenv("DRSIM_HOST_ACTIONS", host_actions)   # read by drsim_create

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.config import synthetic_table

    over = {"power_grid_prop/base_power_props/mode": base_mode}
    if base_mode == "interpolation":
        over["power_grid_prop/base_power_props/interp_update_period"] = 20
    prop = _prop(n, **over)
    T = 14
    st = synthetic_state(prop, R, seed=5)
    acts = (np.random.default_rng(6).random((T, R, n)) < 0.5).astype(np.uint8)
    table = synthetic_table(7) if base_mode == "interpolation" else None
    envs = [BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=3, interp_table=table) for _ in range(3)]
    for e in envs:
        e.reset(copy.deepcopy(st))
    out_pin = torch.zeros((R, 4), dtype=torch.float64).pin_memory()
    for t in range(T):
        envs[0].step(torch.as_tensor(acts[t], device="cuda"))
        a_pin = torch.as_tensor(acts[t]).pin_memory()
        envs[1].step_host(a_pin, out_pin)
        out_page = envs[2].step_host(acts[t])
        torch.cuda.synchronize()
        ref = envs[0].state
        mean_rew = ref["reward"].double().mean(dim=1).cpu().numpy()
        for out in (out_pin.numpy(), out_page):
            assert np.array_equal(out[:, 0], ref["power"].cpu().numpy()), t
            assert np.array_equal(out[:, 1], ref["signal"].cpu().numpy()), t
            assert np.array_equal(out[:, 2], ref["od_temp"].cpu().numpy()), t
            np.testing.assert_allclose(out[:, 3], mean_rew, rtol=1e-5, atol=1e-6)
    for e in envs[1:]:
        for k in ("sso", "flags", "dt_air", "dt_mass", "reward", "obs", "signal", "power", "metrics"):
            assert torch.equal(envs[0].state[k], e.state[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("n,R,layout", [(100, 9, "hand_engineered"), (1000, 3, "tarmac"), (10, 5, "hand_engineered")])
def test_step_host_full_returns_obs_and_reward(n, R, layout):
    """drsim_step_host_full: what Environment.step returns (environment.py:108) -- per-agent observations and
    rewards -- lands in the caller's host buffers (pinned and pageable), identical to the device tensors of a
    device-resident step; N = 10 exercises the padded rows (house stride 12)."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    prop = _prop(n)
    st = synthetic_state(prop, R, seed=5)
    acts = (np.random.default_rng(6).random((6, R, n)) < 0.5).astype(np.uint8)
    envs = [BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=3) for _ in range(3)]
    for e in envs:
        e.reset(copy.deepcopy(st))
    D = envs[0].sim.D
    env_pin = torch.zeros((R, 4), dtype=torch.float64).pin_memory()
    rew_pin = torch.zeros((R, n), dtype=torch.float32).pin_memory()
    obs_pin = torch.zeros((R, n, D), dtype=torch.float32).pin_memory()
    rew_np, obs_np = np.zeros((R, n), np.float32), np.zeros((R, n, D), np.float32)
    for t in range(6):
        obs_d, rew_d = envs[0].step(torch.as_tensor(acts[t], device="cuda"))
        envs[1].step_host(torch.as_tensor(acts[t]).pin_memory(), env_pin, reward_out=rew_pin, obs_out=obs_pin)
        envs[2].step_host(acts[t].astype(bool), None, reward_out=rew_np, obs_out=obs_np)
        torch.cuda.synchronize()
        for rew, obs in ((rew_pin.numpy(), obs_pin.numpy()), (rew_np, obs_np)):
            assert np.array_equal(rew, rew_d.cpu().numpy()), t
            assert np.array_equal(obs, obs_d.cpu().numpy()), t
        assert np.array_equal(env_pin.numpy()[:, 0], envs[0].state["power"].cpu().numpy())
    with pytest.raises(ValueError):
        envs[1].step_host(torch.zeros((R, n), dtype=torch.int32), env_pin)      # a 4-byte dtype is not reinterpreted as bytes
    with pytest.raises(ValueError):
        envs[1].step_host(torch.zeros((R, n + 1), dtype=torch.uint8), env_pin)   # wrong shape


def _forward64(fc, x):
    """The same network evaluated in fp64 (the yardstick both fp32 evaluations are measured against)."""
    import torch

    x = x.double()
    x = torch.relu(x @ fc[0].weight.double().T + fc[0].bias.double())
    x = torch.relu(x @ fc[1].weight.double().T + fc[1].bias.double())
    return x @ fc[2].weight.double().T + fc[2].bias.double()


def _torch_actor(D, h1, h2, seed):
    """The reference's Actor (network.py:14-35) restated in plain PyTorch fp32."""
    import torch

    torch.manual_seed(seed)
    fc = torch.nn.ModuleList([torch.nn.Linear(D, h1), torch.nn.Linear(h1, h2), torch.nn.Linear(h2, 2)]).cuda()

    def forward(x):
        x = torch.relu(fc[0](x))
        x = torch.relu(fc[1](x))
        return torch.softmax(fc[2](x), dim=1)

    return fc, forward


@pytest.mark.parametrize("R,n,layout,h1,h2,nb_comm", [
    (300, 100, "hand_engineered", 100, 100, 10), (7, 1000, "tarmac", 100, 100, 10), (33, 37, "hand_engineered", 64, 48, 10),
    (5, 9, "tarmac", 111, 96, 10),                      # wide layers: 240 of the 256 TMEM columns of a k_actor2 tile slot
    (520, 100, "hand_engineered", 100, 100, 10),        # three tiles per CTA: every pipeline slot is recycled
    (1100, 100, "tarmac", 32, 16, 10),                  # narrow layers: a single chunk, nothing through the spare columns
    (40, 100, "hand_engineered", 100, 100, 3),          # D = 22: the 4-chunk instantiation of the row handling
    (40, 100, "hand_engineered", 80, 100, 12)])         # D = 58: the 9-chunk instantiation; 16 in-place columns
def test_on_device_actor_matches_torch_fp32(R, n, layout, h1, h2, nb_comm):
    """SURVEY 8f-2: the tcgen05 actor + categorical draw against a plain PyTorch fp32 forward of the same
    weights.  Probabilities: TF32 operands (10-bit mantissa, rounded to nearest), fp32 accumulation -> |dp| <= 5e-3
    on logits three times wider than the default initialisation gives.  The draw
    must be the inverse-CDF rule on the Philox uniform of (seed, replica, house, step), recomputed here
    with the NumPy restatement of the generator; the drawn actions must then drive the next env step."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle import philox

    prop = _prop(n, **{"cluster_prop/agents_comm_prop/max_nb_agents_communication": nb_comm})
    env = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=17, rep_offset=40)
    env.reset(synthetic_state(prop, R, seed=4, rep_offset=40))
    D = env.sim.D
    fc, forward = _torch_actor(D, h1, h2, seed=3)
    with torch.no_grad():
        for lin in fc:                       # wider logits than the default init: probabilities away from 1/2
            lin.weight.mul_(3.0)
    weights = BatchedEnv.actor_weights(fc)
    a0 = (torch.rand((R, n), device="cuda") < 0.5).to(torch.uint8)
    env.step(a0)                             # step 0 -> observations of step 1
    obs = env.obs.clone()
    with torch.no_grad():
        p_ref = forward(obs.reshape(-1, D)).reshape(R, n, 2)
    prob_on = torch.zeros((R, env.sim.Ns), dtype=torch.float32, device="cuda")
    prob = torch.zeros_like(prob_on)
    # "tf32x3" (default): operands split into hi + lo TF32 halves, three passes per product -> fp32-grade
    env.sim.policy_step(weights, seed=99, prob_drawn=prob, prob_on=prob_on, precision="tf32x3")
    torch.cuda.synchronize()
    with torch.no_grad():
        p_ref64 = torch.softmax(_forward64(fc, obs.reshape(-1, D)), dim=1).reshape(R, n, 2)
    err3 = float((prob_on[:, :n].double() - p_ref64[..., 1]).abs().max())
    ref_err = float((p_ref.double() - p_ref64).abs().max())     # what a plain fp32 forward is off by itself
    assert err3 <= 2e-6 + 2 * ref_err, (err3, ref_err)
    # its draw and the probability it reports for the drawn action (same rule as below, on its own probabilities)
    act3, p_on3 = env.state["actions"][:, :n].clone(), prob_on[:, :n].clone()
    torch.testing.assert_close(prob[:, :n], torch.where(act3.bool(), p_on3, 1.0 - p_on3), rtol=0, atol=1e-6)
    u3 = np.stack([(np.asarray(philox.philox4x32_10(99, 40 + r, np.arange(n), 1, 6)[0], dtype=np.uint64) >> np.uint64(8))
                   .astype(np.float64) * 2.0 ** -24 for r in range(R)])
    p03 = (1.0 - p_on3).double().cpu().numpy()
    clear3 = np.abs(u3 - p03) > 1e-6
    assert np.array_equal(act3.cpu().numpy()[clear3], (u3 >= p03).astype(np.uint8)[clear3])
    assert clear3.mean() > 0.999
    assert int(env.state["actions"][:, n:].sum()) == 0           # padding slots get action 0
    # "tf32": one pass, 10-bit operands
    env.sim.policy_step(weights, seed=99, prob_drawn=prob, prob_on=prob_on, precision="tf32")
    torch.cuda.synchronize()
    act = env.state["actions"][:, :n].clone()
    p_on = prob_on[:, :n]
    assert float((p_on - p_ref[..., 1]).abs().max()) <= 5e-3
    # probability reported for the drawn action
    want = torch.where(act.bool(), p_on, 1.0 - p_on)
    torch.testing.assert_close(prob[:, :n], want, rtol=0, atol=1e-6)
    # the draw: u < p0 -> action 0, with u from the 24 top bits of Philox word 0 of (replica, house, step, purpose 6)
    step = 1
    u = np.empty((R, n))
    for r in range(R):
        x = philox.philox4x32_10(99, 40 + r, np.arange(n), step, 6)[0]
        u[r] = (np.asarray(x, dtype=np.uint64) >> np.uint64(8)).astype(np.float64) * 2.0 ** -24
    p0 = (1.0 - p_on).double().cpu().numpy()
    expect = (u >= p0).astype(np.uint8)
    clear = np.abs(u - p0) > 1e-6            # away from the threshold the rule is unambiguous
    assert np.array_equal(act.cpu().numpy()[clear], expect[clear])
    assert clear.mean() > 0.999
    # the drawn actions are what the next step consumes
    ref = env.clone()
    env.sim.step(None)
    ref.step(act.contiguous())
    torch.cuda.synchronize()
    for k in ("sso", "flags", "dt_air", "reward", "obs"):
        assert torch.equal(env.state[k], ref.state[k]), k


def test_replica_placement_invariance():
    """Shard [4, 8) of a 12-replica job == replicas 4..7 of the whole job (Philox keyed by the
    global replica index, synthetic state keyed by it too): the basis of the multi-GPU sharding."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv

    prop = _prop(64)
    whole = BatchedEnv(prop, 12, noise="philox", seed=11)
    part = BatchedEnv(prop, 4, noise="philox", seed=11, rep_offset=4)
    whole.reset()
    part.reset()
    a = (torch.rand((12, 64), device="cuda", generator=torch.Generator(device="cuda").manual_seed(5)) < 0.5).to(torch.uint8)
    for t in range(10):
        whole.step(a)
        part.step(a[4:8].contiguous())
    torch.cuda.synchronize()
    for k in ("dt_air", "dt_mass", "sso", "flags", "reward", "obs", "signal", "od_temp"):
        assert torch.equal(whole.state[k][4:8], part.state[k]), k


def test_on_device_policies_match_oracle_controllers():
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from oracle.np_oracle import NpOracle, deadband_bangbang, from_epoch, greedy_myopic

    # greedy-myopic: cop 2.5 gives exactly representable powers (parallel-prefix path of k_greedy), cop 2.3
    # does not (fully sequential scan); 1000 houses = 32 chunks of the warp-cooperative scan
    for policy, n, cop in (("deadband_bangbang", 90, 2.5), ("greedy_myopic", 300, 2.5), ("greedy_myopic", 1000, 2.5),
                           ("greedy_myopic", 300, 2.3), ("greedy_myopic", 37, 2.3)):
        prop = _prop(n, **{"cluster_prop/house_prop/deadband": 0.5, "power_grid_prop/signal_properties/mode": "sinusoidals",
                           "cluster_prop/house_prop/hvac_prop/cop": cop})
        R, T = 3, 25
        st = synthetic_state(prop, R, seed=21)
        env = BatchedEnv(prop, R, precision="f64", policy=policy, noise="zero", path="auto")
        env.reset(copy.deepcopy(st))
        orc = NpOracle(prop, R)
        orc.set_state(copy.deepcopy(st))
        orc.power_grid_step([from_epoch(e) for e in orc.state["epoch"]], None)
        for t in range(T):
            s = orc.state
            if policy == "deadband_bangbang":
                a = deadband_bangbang(s["t_air"], s["target"], 0.5, s["on"])
            else:
                a = np.stack([greedy_myopic(s["t_air"][r], s["target"][r], s["cap"][r], cop, s["lockout"][r], s["signal"][r])
                              for r in range(R)])
            orc.step(a, np.zeros(R), None)
            env.step(None)
        got = env.get_state()
        for k in ("on", "lockout", "sso"):
            assert np.array_equal(got[k].astype(np.int64), orc.state[k].astype(np.int64)), (policy, n, cop, k)
        np.testing.assert_allclose(got["t_air"], orc.state["t_air"], rtol=0, atol=1e-9)


@pytest.mark.parametrize("n,R,policy,base_mode,layout", [
    (10, 5, "deadband_bangbang", "constant", "hand_engineered"),   # in-kernel episode, one tile
    (1000, 7, "bangbang", "constant", "tarmac"),                   # in-kernel episode, one cluster per tile
    (37, 300, "deadband_bangbang", "constant", "hand_engineered"), # in-kernel episode, 12 tiles of 25 clusters, padded rows
    (100, 40, "deadband_bangbang", "interpolation", "tarmac"),     # interpolated base power: per-step loop
    (130, 5, "external", "interpolation", "hand_engineered"), (1000, 5, "greedy_myopic", "constant", "hand_engineered"),
    (37, 5, "external", "constant", "hand_engineered")])
def test_run_equals_repeated_steps(n, R, policy, base_mode, layout):
    """``drsim_run`` (n steps in one C call: in-kernel step loop under an on-device policy, per-step launches
    otherwise, optionally replaying an action tape) == n ``drsim_step`` calls, bit for bit."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv

    prop = _prop(n, **{"power_grid_prop/base_power_props/mode": base_mode, "cluster_prop/house_prop/deadband": 0.4,
                       "power_grid_prop/signal_properties/mode": "sinusoidals"})
    table = np.random.default_rng(3).uniform(0, 6000, 3 * 3 * 3 * 3 * 9 * 5 * 8 * 2 * 12 * 6) if base_mode == "interpolation" else None
    T = 90   # 90 steps: crosses a 64-step schedule block and (interpolation) the 75-step update
    a = BatchedEnv(prop, R, policy=policy, noise="philox", seed=13, obs_layout=layout, interp_table=table)
    a.reset()
    b = copy.deepcopy(a)
    tape = None
    if policy == "external":
        tape = (torch.rand((T, R, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)) < 0.5).to(torch.uint8)
    for t in range(T):
        a.step(None if tape is None else tape[t])
    b.run(40, None if tape is None else tape[:40])
    b.run(T - 40, None if tape is None else tape[40:])
    torch.cuda.synchronize()
    for k in ("dt_air", "dt_mass", "sso", "flags", "reward", "obs", "signal", "power", "od_temp", "base_power", "metrics"):
        assert torch.equal(a.state[k], b.state[k]), k
    with pytest.raises(Exception):   # injected noise is a per-step input: rejected for n_steps > 1
        _run_with_noise(b, R)


@pytest.mark.parametrize("n,R,layout,rotate,policy,nb_comm,tile_envs", [
    (1000, 640, "tarmac", True, "external", 10, None),             # one cluster per tile (k_fused_tma<1>), 2.2 tiles per CTA
    (1000, 2048, "tarmac", True, "external", 10, None),            # BASELINE config 4 at full size: 7 tiles per CTA
    (100, 6100, "tarmac", False, "external", 10, None),            # ten clusters per tile (generic instantiation)
    (37, 16000, "tarmac", True, "external", 10, None),             # padded rows, ragged last tile
    (100, 4096, "hand_engineered", True, "external", 10, None),    # BASELINE config 3: wide rows (k_fused_rows), 586 tiles on 293 CTAs
    (100, 1800, "hand_engineered", True, "external", 2, 3),        # messages in whole-tile rows (k_fused_tma<2>): 18 columns, 3 clusters per tile
    (100, 6100, "tarmac", True, "deadband_bangbang", 10, None)])   # on-device policy, no tape
def test_tape_stream_equals_per_step_launches(n, R, layout, rotate, policy, nb_comm, tile_envs, monkeypatch):
    """``drsim_run_tape`` on the staged fused kernel with at least two tiles per CTA runs the step loop INSIDE the
    kernel (StepIn::stream_steps: no boundary between the steps of a schedule block).  Same bits as one launch per
    step (``DRSIM_NO_STREAM=1``), over a schedule-block boundary, with a rotating and a linear tape."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv

    if tile_envs is not None:
        monkeypatch.setenv("DRSIM_TILE_ENVS", str(tile_envs))
    prop = _prop(n, **{"power_grid_prop/signal_properties/mode": "sinusoidals",
                       "cluster_prop/agents_comm_prop/max_nb_agents_communication": nb_comm})
    T = 70 if rotate else 9
    planes = 3 if rotate else T
    a = BatchedEnv(prop, R, policy=policy, noise="philox", seed=5, obs_layout=layout)
    a.reset()
    info = a.sim.fused_info()
    assert info["variant"] in ("staged", "staged_rows") and (info["tiles"] // 2) * 10 >= info["grid"] * 9, info          # otherwise the stream is not taken and the test is vacuous
    b = copy.deepcopy(a)
    tape = (torch.rand((planes, R, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) < 0.5).to(torch.uint8)
    if policy != "external":
        tape = None
    launches0 = a.sim.launch_count
    a.run(T, tape, rotate=rotate)
    torch.cuda.synchronize()
    assert a.sim.launch_count - launches0 <= 2 * 3 + 2     # two schedule blocks (+ their two generator kernels each), not T launches
    os.environ["DRSIM_NO_STREAM"] = "1"
    try:
        b.run(T, tape, rotate=rotate)
    finally:
        del os.environ["DRSIM_NO_STREAM"]
    torch.cuda.synchronize()
    for k in ("dt_air", "dt_mass", "sso", "flags", "reward", "obs", "signal", "power", "od_temp", "metrics"):
        assert torch.equal(a.state[k], b.state[k]), k
    # and the stream leaves the handle in a state ordinary steps continue from
    a.step(None if tape is None else tape[0]); b.step(None if tape is None else tape[0])
    torch.cuda.synchronize()
    for k in ("dt_air", "sso", "flags", "reward", "obs", "metrics"):
        assert torch.equal(a.state[k], b.state[k]), k


@pytest.mark.parametrize("n,R,layout,policy,nb_comm", [(10, 5, "hand_engineered", "external", 9), (10, 1, "hand_engineered", "deadband_bangbang", 9),
                                                    (31, 200, "tarmac", "external", 10), (12, 9, "hand_engineered", "bangbang", 4),
                                                    (5, 3, "none", "external", 2)])
def test_small_cluster_kernel_matches_tile_kernels(n, R, layout, policy, nb_comm):
    """Clusters of at most 32 houses in a handful of replicas step on ``k_small`` (one house per lane, the state in
    registers across the steps of a launch).  Against the tile kernels (``DRSIM_NO_SMALL=1``): discrete state and env
    scalars bit-exact, continuous values to fp32 rounding (the cluster sums are associated differently); the in-kernel
    step loop (on-device policy / action tape) == one launch per step, bit for bit."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv

    prop = _prop(n, **{"power_grid_prop/signal_properties/mode": "sinusoidals", "cluster_prop/house_prop/deadband": 0.4,
                       "cluster_prop/agents_comm_prop/max_nb_agents_communication": nb_comm})
    T = 70
    tape = None
    if policy == "external":
        tape = (torch.rand((T, R, n), device="cuda", generator=torch.Generator(device="cuda").manual_seed(4)) < 0.5).to(torch.uint8)
    a = BatchedEnv(prop, R, policy=policy, noise="philox", seed=9, obs_layout=layout)
    a.reset()
    b, c = copy.deepcopy(a), copy.deepcopy(a)
    l0 = a.sim.launch_count
    a.run(T, tape)                                       # k_small, steps inside the kernel
    assert a.sim.launch_count - l0 <= 2 * 3
    for t in range(T):                                   # k_small, one launch per step
        b.step(None if tape is None else tape[t])
    os.environ["DRSIM_NO_SMALL"] = "1"
    try:
        for t in range(T):                               # tile kernels
            c.step(None if tape is None else tape[t])
    finally:
        del os.environ["DRSIM_NO_SMALL"]
    torch.cuda.synchronize()
    keys = [k for k in ("dt_air", "dt_mass", "sso", "flags", "reward", "obs", "signal", "power", "od_temp", "metrics")
            if a.state[k] is not None]                   # (obs_layout "none": no observation plane)
    for k in keys:
        assert torch.equal(a.state[k], b.state[k]), k
    for k in ("sso", "flags", "signal", "od_temp"):
        assert torch.equal(a.state[k], c.state[k]), k
    for k in ("dt_air", "dt_mass", "reward", "obs", "power", "metrics"):
        if k in keys:
            torch.testing.assert_close(a.state[k], c.state[k], rtol=3e-6, atol=3e-6)


def _run_with_noise(env, R):
    import ctypes as C

    import torch

    from marl_demandresponse_b200 import _lib

    args = env.sim._args(None, torch.zeros(R, dtype=torch.float64, device="cuda"))
    _lib.check(env.sim._L.drsim_run(env.sim._h, C.byref(args), 2, 0, None))


def test_clone_is_a_deep_copy():
    import torch

    from marl_demandresponse_b200 import BatchedEnv

    env = BatchedEnv(_prop(50), 8, noise="philox", seed=2)
    env.reset()
    a = torch.ones((8, 50), dtype=torch.uint8, device="cuda")
    for _ in range(5):
        env.step(a)
    twin = copy.deepcopy(env)
    for _ in range(7):
        env.step(a)
        twin.step(a)
    torch.cuda.synchronize()
    for k in ("dt_air", "sso", "flags", "obs", "reward", "signal"):
        assert torch.equal(env.state[k], twin.state[k]), k
    snap = twin.state["dt_air"].clone()
    env.step(a)
    torch.cuda.synchronize()
    assert torch.equal(twin.state["dt_air"], snap), "stepping the original must not touch the clone"


def test_house_sharded_cluster_equals_unsharded():
    """One cluster split over 3 handles (the per-rank partials gathered by hand, as the NCCL
    all-gather would) == the same cluster on one handle: discrete state bit-exact, power / signal /
    rewards identical, for the constant and the interpolated base power; with the hand-engineered
    layout the observation rows (ring-neighbour messages across the shard edges, exchanged as a halo)
    must be identical too."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.sharded import ShardedClusterEnv
    from oracle.config import synthetic_table

    table = synthetic_table(7)
    for base_mode, layout in (("constant", "tarmac"), ("interpolation", "tarmac"), ("constant", "hand_engineered")):
        n, R, W, T = 3000, 2, 3, 80 if base_mode == "interpolation" else 10
        prop = _prop(n, **{"power_grid_prop/base_power_props/mode": base_mode,
                           "power_grid_prop/signal_properties/mode": "sinusoidals"})
        st = synthetic_state(prop, R, seed=3)
        whole = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=9, path="split",
                           interp_table=table if base_mode == "interpolation" else None)
        whole.reset(copy.deepcopy(st))
        parts = [ShardedClusterEnv(prop, R, rank=r, world=W, obs_layout=layout, noise="philox", seed=9) for r in range(W)]
        for p_ in parts:
            if base_mode == "interpolation":
                p_.sim.set_interp_table(table)
            p_.reset(copy.deepcopy(st))
            # the signal computed at reset by the unsharded env is an input of the sharded ones
            p_.sim.set_state({"signal": whole.get_state(["signal"])["signal"],
                              "base_power": whole.get_state(["base_power"])["base_power"],
                              "t_since_interp": whole.get_state(["t_since_interp"])["t_since_interp"]})
        acts = (np.random.default_rng(2).random((T, R, n)) < 0.5).astype(np.uint8)
        for t in range(T):
            a = torch.as_tensor(acts[t], device="cuda")
            whole.step(a)
            for p_ in parts:
                p_.sim.views()["actions"].copy_(a[:, p_.lo:p_.hi])
                p_.sim.step_begin(None)
            gathered = torch.stack([p_.state["acc"] for p_ in parts]).contiguous()
            if layout == "hand_engineered":   # ring-neighbour messages cross the shard edges: halo records too
                halo = torch.stack([p_.state["halo_out"] for p_ in parts]).contiguous()
                for i, p_ in enumerate(parts):
                    p_.sim.step_finish_gathered(gathered, halo, W, i)
                continue
            for p_ in parts:
                p_.sim.step_finish(gathered, W)
        torch.cuda.synchronize()
        ws = whole.state
        for p_ in parts:
            ps = p_.state
            for k in ("sso", "flags", "dt_air", "dt_mass"):
                assert torch.equal(ws[k][:, p_.lo:p_.hi], ps[k]), (base_mode, k)
            for k in ("power", "signal", "od_temp", "base_power"):
                torch.testing.assert_close(ws[k], ps[k], rtol=1e-12, atol=0)
            torch.testing.assert_close(ws["reward"][:, p_.lo:p_.hi], ps["reward"], rtol=1e-6, atol=1e-7)
            torch.testing.assert_close(ws["obs"][:, p_.lo:p_.hi], ps["obs"], rtol=1e-6, atol=1e-7)


def test_full_size_c4_spot_check_against_oracle():
    """BASELINE config 4 at its full single-GPU size (2048 replicas x 1000 houses, TarMAC layout):
    three replicas are re-simulated by the oracle from the same state / Philox noise; cluster power
    must also equal the sum of the per-house powers implied by the discrete state everywhere."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    n, R, T, seed = 1000, 2048, 8, 1234
    prop = _prop(n)
    env = BatchedEnv(prop, R, precision="f32", obs_layout="tarmac", noise="philox", seed=seed)
    st = synthetic_state(prop, R, seed=seed)
    env.reset(st)
    g = torch.Generator(device="cuda").manual_seed(7)
    acts = [(torch.rand((R, n), device="cuda", generator=g) < 0.5).to(torch.uint8) for _ in range(T)]
    for t in range(T):
        env.step(acts[t])
    torch.cuda.synchronize()
    got = env.get_state()
    # size-independent property: aggregate power == sum over houses of on * cap / cop
    p_sum = (got["on"].astype(np.float64) * got["cap"] / 2.5).sum(axis=1)
    np.testing.assert_allclose(got["power"], p_sum, rtol=1e-6)
    assert np.all(got["sso"][got["on"] == 1] == 0)
    assert np.all(got["epoch"] == st["epoch"] + 4 * T)
    pick = [0, 777, 2047]
    sub = {k: (v[pick] if np.asarray(v).shape[:1] == (R,) else v) for k, v in st.items()}
    epoch0 = int(st["epoch"][0])
    od_noise = _od_noise(seed, pick, range(T))
    perlin = _perlin(seed, pick, [epoch0 + 4 * t for t in range(T + 1)])
    a_np = np.stack([a[pick].cpu().numpy() for a in acts])
    orc, _ = _oracle_run(prop, sub, a_np, od_noise, perlin)
    for k in ("on", "lockout", "sso"):
        assert np.array_equal(got[k][pick].astype(np.int64), orc.state[k].astype(np.int64)), k
    np.testing.assert_allclose(got["t_air"][pick], orc.state["t_air"], rtol=0, atol=2e-4)
    np.testing.assert_allclose(got["signal"][pick], orc.state["signal"], rtol=1e-9)
    np.testing.assert_allclose(env.obs[pick].double().cpu().numpy(), orc.obs_vectors()[:, :, :10], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("n,R", [(1, 5), (2, 3), (5, 300), (1023, 2), (1024, 2), (1025, 2)])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_edge_sizes_match_oracle(n, R, precision):
    """Ragged / degenerate cluster sizes: a single house (no neighbours, D = 10), sizes that are not
    multiples of the 4-house vector width, the tile capacity and one past it (general path)."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state

    T, seed = 6, 3
    prop = _prop(n, **{"reward_prop/penalty_props/mode": "mixture", "cluster_prop/house_prop/deadband": 0.4})
    env = BatchedEnv(prop, R, precision=precision, noise="philox", seed=seed)
    st = synthetic_state(prop, R, seed=8)
    env.reset(copy.deepcopy(st))
    acts = (np.random.default_rng(4).random((T, R, n)) < 0.5).astype(np.uint8)
    epoch0 = int(st["epoch"][0])
    od_noise = _od_noise(seed, range(R), range(T))
    perlin = _perlin(seed, range(R), [epoch0 + 4 * t for t in range(T + 1)])
    rew = []
    for t in range(T):
        _, r_ = env.step(torch.as_tensor(acts[t], device="cuda"))
        rew.append(r_.double().cpu().numpy())
    orc, rew_ref = _oracle_run(prop, copy.deepcopy(st), acts, od_noise, perlin)
    got = env.get_state()
    for k in ("on", "lockout", "sso"):
        assert np.array_equal(got[k].astype(np.int64), orc.state[k].astype(np.int64)), k
    tol = 2e-4 if precision == "f32" else 1e-9
    np.testing.assert_allclose(got["t_air"], orc.state["t_air"], rtol=0, atol=tol)
    np.testing.assert_allclose(np.array(rew), rew_ref, rtol=1e-5 if precision == "f32" else 1e-9, atol=tol)
    assert env.obs.shape == (R, n, 10 + 4 * min(10, n - 1))
    np.testing.assert_allclose(env.obs.double().cpu().numpy(), orc.obs_vectors(), rtol=1e-5, atol=1e-5 if precision == "f32" else 1e-9)


def test_maximum_size_single_cluster_of_one_million_houses():
    """BASELINE config 5 on one GPU: one 1,000,000-house cluster (general path, 977 CTAs per
    cluster) against the oracle: discrete state bit-exact, aggregate power to fp32 accuracy."""
    import torch

    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.sharded import ShardedClusterEnv

    n, T, seed = 1_000_000, 3, 5
    prop = _prop(n)
    st = synthetic_state(prop, 1, seed=2)
    env = ShardedClusterEnv(prop, 1, rank=0, world=1, noise="philox", seed=seed)
    env.reset(copy.deepcopy(st))
    env.sim.refresh(True)
    acts = (np.random.default_rng(6).random((T, 1, n)) < 0.5).astype(np.uint8)
    epoch0 = int(st["epoch"][0])
    od_noise = _od_noise(seed, [0], range(T))
    perlin = _perlin(seed, [0], [epoch0 + 4 * t for t in range(T + 1)])
    for t in range(T):
        env.step(torch.as_tensor(acts[t], device="cuda"))
    orc, rew_ref = _oracle_run(prop, copy.deepcopy(st), acts, od_noise, perlin)
    got = env.sim.get_state()
    for k in ("on", "lockout", "sso"):
        assert np.array_equal(got[k].astype(np.int64), orc.state[k].astype(np.int64)), k
    np.testing.assert_allclose(got["power"], orc.state["power"], rtol=1e-6)
    np.testing.assert_allclose(got["signal"], orc.state["signal"], rtol=1e-9)
    np.testing.assert_allclose(got["t_air"], orc.state["t_air"], rtol=0, atol=2e-4)
    np.testing.assert_allclose(env.state["reward"].double().cpu().numpy(), rew_ref[-1], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("mode", ["reference", "synthetic"])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_device_reset_matches_numpy_restatement(mode, precision):
    """drsim_reset (Environment.reset distributions on Philox streams, SURVEY 8a-15) == its NumPy
    restatement, then a few steps from that state == the oracle from the restated state."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from oracle import philox

    n, R, seed, off, T = 150, 7, 99, 40, 5
    prop = _prop(n, **{"start_datetime_mode": "random"})
    env = BatchedEnv(prop, R, precision=precision, noise="philox", seed=seed, rep_offset=off)
    env.reset(device_mode=mode)
    got = env.get_state()
    want = philox.reset_state(seed, R, prop, mode, True, off)
    for k in ("on", "lockout", "sso", "epoch"):
        assert np.array_equal(np.asarray(got[k]).astype(np.int64), np.asarray(want[k]).astype(np.int64)), k
    tol = 1e-5 if precision == "f32" else 1e-12
    for k in ("target", "cap", "t_air", "t_mass", "od_temp", "max_power"):
        np.testing.assert_allclose(got[k], want[k], rtol=tol, atol=tol, err_msg=k)
    # property-noise statistics are the reference's: target >= default, factors in [0.9, 1.1], caps in the list
    assert np.all(got["target"] >= 19.0) and set(np.unique(got["cap"])) <= {12500.0, 15000.0, 17500.0}
    if mode == "reference":
        assert np.all(got["on"] == 1) and np.allclose(got["t_air"], 20.0, rtol=0, atol=1e-5)
    # continue from the device-drawn state and compare with the oracle started from the restated one
    acts = (np.random.default_rng(0).random((T, R, n)) < 0.5).astype(np.uint8)
    reps = [off + r for r in range(R)]
    od_noise = _od_noise(seed, reps, range(T))
    perlin = _perlin(seed, reps, [np.asarray(want["epoch"]) + 4 * t for t in range(T + 1)])
    for t in range(T):
        env.step(torch.as_tensor(acts[t], device="cuda"))
    if mode == "reference":
        want["power"] = np.full(R, n * 6000.0)
    orc, _ = _oracle_run(prop, want, acts, od_noise, perlin)
    got = env.get_state()
    for k in ("on", "lockout", "sso"):
        assert np.array_equal(got[k].astype(np.int64), orc.state[k].astype(np.int64)), k
    np.testing.assert_allclose(got["t_air"], orc.state["t_air"], rtol=0, atol=2e-4 if precision == "f32" else 1e-8)
    np.testing.assert_allclose(got["signal"], orc.state["signal"], rtol=1e-9)


def test_monte_carlo_table_generator_matches_oracle():
    """SURVEY 8f-1: the GPU generator of the interpolation table (4,199,040 single-house bang-bang
    simulations x 75 steps) against the oracle restatement of monteCarlo.py on a random sample of
    grid points (fp64 build: exact closed loop), plus shape / range checks on a larger fp32 run."""
    from marl_demandresponse_b200 import montecarlo as mc
    from oracle.montecarlo import table_entries

    rng = np.random.default_rng(0)
    idx = np.sort(rng.choice(4_199_040, size=3000, replace=False))
    got = mc.generate_table(idx, precision="f64")
    prop = mc.env_prop_for_table()
    pts = mc.grid_points(idx)
    want = table_entries(prop, mc.initial_state(pts, prop), pts["OD_temp"])
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-6)
    # physical sanity: between 0 and the HVAC electrical power, hotter start -> not less consumption on average
    assert np.all(got >= 0) and np.all(got <= pts["HVAC_power"] / 2.5 + 1e-6)
    got32 = mc.generate_table(idx, precision="f32")
    # fp32 closed loop may flip a bang-bang decision on a tie; the table average is robust to it
    close = np.isclose(got32, want, rtol=1e-4, atol=0.5)
    assert close.mean() > 0.995, close.mean()
    assert abs(got32.mean() - want.mean()) < 1e-3 * want.mean()
