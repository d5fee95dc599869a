"""The device-resident MA-PPO rollout (SURVEY 8f-2): ``BatchedEnv.collect`` stores, per transition, what the
reference's ``MAPPO.store_transition`` stores (mappo.py:105-127; loop of training_manager.py:224-240) -- state,
action, the other agents' actions, the action's probability, reward, next state -- in device buffers the kernels
write directly.  Checked against the step-by-step path (``policy_step`` + ``step``) bit for bit, and against the
reference's own bookkeeping restated on the host."""
import copy

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _prop(n):
    return {"start_datetime": "2021-06-15T11:58:20", "start_datetime_mode": "fixed", "time_step": 4.0,
            "cluster_prop": {"nb_agents": n, "house_prop": {"target_temp": 19.0}}}


def _actor(D, seed=3):
    import torch

    torch.manual_seed(seed)
    fc = torch.nn.ModuleList([torch.nn.Linear(D, 100), torch.nn.Linear(100, 100), torch.nn.Linear(100, 2)]).cuda()
    with torch.no_grad():
        for lin in fc:
            lin.weight.mul_(3.0)
    return fc


@pytest.mark.parametrize("R,n,layout,state_prop,obs_dtype", [
    pytest.param(64, 100, "hand_engineered", {}, "float32", id="64-100-hand_engineered"),
    pytest.param(5, 1000, "tarmac", {}, "float32", id="5-1000-tarmac"),
    pytest.param(9, 37, "hand_engineered", {}, "float32", id="9-37-hand_engineered"),
    pytest.param(3, 2500, "tarmac", {}, "float32", id="3-2500-tarmac"),
    # bf16 rows of odd width (D = 11): one plane is 6600 bytes, off the 16-byte grid the transition needs
    pytest.param(3, 100, "tarmac", {"solar_gain": True}, "bfloat16", id="3-100-tarmac-solar-bfloat16")])
def test_collect_equals_policy_step_plus_step(R, n, layout, state_prop, obs_dtype):
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.rollout import RolloutBuffer

    T = 7
    prop = {**_prop(n), "state_prop": state_prop}
    st = synthetic_state(prop, R, seed=4)
    a = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=17, obs_dtype=obs_dtype)
    b = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=17, obs_dtype=obs_dtype)
    a.reset(copy.deepcopy(st))
    b.reset(copy.deepcopy(st))
    weights = BatchedEnv.actor_weights(_actor(a.sim.D))
    buf = RolloutBuffer(a, T)
    a.collect(weights, buf, done_last=True)
    assert all(buf.obs[t].is_contiguous() and buf.obs[t].data_ptr() % 16 == 0 for t in range(T + 1))
    states, actions, probs, rewards = [], [], [], []
    for t in range(T):
        states.append(b.obs.clone())
        act, prob = b.policy_step(weights)
        actions.append(act.clone())
        probs.append(prob.clone())
        b.sim.step(None)
        rewards.append(b.reward.clone())
    torch.cuda.synchronize()
    a.sim.peer_status()
    for t in range(T):
        assert torch.equal(buf.state(t), states[t]), ("state", t)
        assert torch.equal(buf.action(t), actions[t]), ("action", t)
        assert torch.equal(buf.prob(t), probs[t]), ("prob", t)
        assert torch.equal(buf.reward(t), rewards[t]), ("reward", t)
    assert torch.equal(buf.next_state(T - 1), b.obs)
    # the simulator itself went through the same T steps
    for k in ("dt_air", "dt_mass", "sso", "flags", "signal", "power", "metrics"):
        assert torch.equal(a.state[k], b.state[k]), k
    # a second segment continues from the handle's state, reading state_0 from the last next_state
    a.collect(weights, buf, n_steps=3)
    for t in range(3):
        s = b.obs.clone()
        act, prob = b.policy_step(weights)
        act = act.clone()
        b.sim.step(None)
        assert torch.equal(buf.state(t), s) and torch.equal(buf.action(t), act) and torch.equal(buf.reward(t), b.reward)


def test_buffer_fields_are_the_reference_transition_fields():
    """others_actions / Gt as mappo.py builds them (:113-116, :147-152), from the device buffers."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.rollout import RolloutBuffer

    R, n, T, gamma = 3, 12, 6, 0.9
    env = BatchedEnv(_prop(n), R, noise="philox", seed=2)
    env.reset()
    buf = RolloutBuffer(env, T)
    env.collect(BatchedEnv.actor_weights(_actor(env.sim.D)), buf, done_last=True)
    torch.cuda.synchronize()
    act = buf.actions[:, :, :n].cpu().numpy()
    rew = buf.rewards[:, :, :n].double().cpu().numpy()
    oth = buf.others_actions(2).cpu().numpy()
    for r in range(R):
        last_actions = {i: int(act[2, r, i]) for i in range(n)}
        for i in range(n):
            action_k = copy.deepcopy(last_actions)          # mappo.py:113-116
            action_k.pop(i)
            assert oth[r, i].tolist() == list(action_k.values())
    done = [False] * (T - 1) + [True]
    Gt = buf.returns(gamma).double().cpu().numpy()
    for r in range(R):
        for i in range(n):
            run, want = 0.0, []
            for t in reversed(range(T)):                     # mappo.py:147-152
                if done[t]:
                    run = 0.0
                run = rew[t, r, i] + gamma * run
                want.insert(0, run)
            np.testing.assert_allclose(Gt[:, r, i], want, rtol=1e-5, atol=1e-5)
