"""The "f16x3" actor (``k_actor3<SplitF16x3, PRE, O>``: three passes on fp16 halves with per-neuron power-of-two weight scales)
against its operand-exact reference ``actor_ref_f16x3``: every compared row's ``prob_on`` lies within the
first-principles bound AND within the fp32-grade tolerance of the plain fp64 forward, and the max |dp| against that
forward is printed next to the 3xTF32 actor's on the same rows.

The set-up is that of ``test_gpu_actor.py`` (synthetic rows written into the observation plane of a handle that has
stepped, replicas at a non-zero global index, a two-word seed, huge values in the padding slots).  After every launch
``actor_status`` must report nothing: padding slots never set the range flag.  Covered: every instantiation (PRE = 1, 2,
4, 5) with fp32 and bf16 rows of even and odd width; hidden widths up to h1 = h2 = 128 at D = 64 (fp16 operands fit where
3xTF32 refuses); row counts; output pointers; the refusals one step past each limit; the fp16 range (rows and hidden
activations at and above 65504, tiny and huge weights): exact results or the reported refusal, never a silent wrong
probability; the rollout (``collect`` equals ``policy_step`` + ``step`` bit for bit) and real environment rows of the C3
and C4 shapes against the 3xTF32 actor."""
import copy

import numpy as np
import pytest

import actor_ref_f16x3 as hr
from oracle import actor_ref as ar
from test_gpu_actor import PAD_VALUE, SEED, STEPS, _env, _refused, _run, _sample, _uniform, _weights, _write_rows

pytestmark = pytest.mark.gpu

K = "f16x3"


def _tf32x3_fits(d, h1, h2):
    from test_gpu_actor import actor_layout

    return actor_layout(d, h1, h2, "tf32x3")[2]


def _check(env, stored, net, out, idx, what, tf32x3=None):
    sim = env.sim
    sim.actor_status()                                  # no operand left the fp16 range (padding slots included)
    act, prob, prob_on = out
    live = np.arange(sim.R * sim.Ns) % sim.Ns < sim.N
    assert not act[~live].any() and not prob[~live].any() and not prob_on[~live].any(), (what, "padding slots")
    assert set(np.unique(act)) <= {0, 1}
    p_ref, bound, info = hr.forward(stored[idx], *net)
    assert info["in_range"].all(), what
    got = prob_on[idx].astype(np.float64)
    err = np.abs(got - p_ref)
    worst = int(np.argmax(err / bound))
    assert np.all(err <= bound), (what, "row", int(idx[worst]), got[worst], p_ref[worst], bound[worst])
    assert bound.max() <= 1e-3, (what, bound.max())
    tol = hr.fp32_grade_tolerance(stored[idx], *net)
    p64 = ar.forward64(stored[idx], *net)
    err64 = np.abs(got - p64)
    assert err64.max() <= tol, (what, "fp32 grade", int(idx[np.argmax(err64)]), float(err64.max()), tol)
    line = (f"actor {what} f16x3: rows {len(idx)}, max |dp|/bound {float((err / bound).max()):.3g}, max |dp64| "
            f"{float(err64.max()):.3g} of {tol:.3g}")
    if tf32x3 is not None:
        line += f"; tf32x3 max |dp64| {float(np.abs(tf32x3[2][idx] - p64).max()):.3g}"
    print(line)
    u, p0 = _uniform(idx, sim.Ns, STEPS), 1.0 - p_ref
    clear = np.abs(u - p0) > bound + 2.0 ** -22
    assert (~clear).sum() <= max(2, 0.001 * len(idx)), (what, clear.mean())
    assert np.array_equal(act[idx][clear], (u >= p0)[clear].astype(np.uint8)), (what, "draw")
    on = act[idx] == 1
    assert np.array_equal(prob[idx][on], prob_on[idx][on])
    assert np.all(np.abs(prob[idx][~on].astype(np.float64) - (1.0 - got[~on])) <= 2.0 ** -22)


def _case(env, d, h1, h2, seed, what, padding_check=False, net=None, rows=None, compare=True):
    rng = np.random.default_rng(seed)
    sim = env.sim
    net = ar.sample_net(rng, d, h1, h2) if net is None else net
    rows = ar.sample_rows(rng, sim.R * sim.Ns, d, net) if rows is None else rows
    idx = _sample(sim, rng)
    w = _weights(net)
    stored = _write_rows(env, rows, PAD_VALUE)
    out = _run(env, w, K)
    other = _run(env, w, "tf32x3") if compare and _tf32x3_fits(d, h1, h2) else None
    _check(env, stored, net, out, idx, what, other)
    if padding_check:   # huge padding values change nothing else, bit for bit
        _write_rows(env, rows, 0.0)
        again = _run(env, w, K)
        live = np.arange(sim.R * sim.Ns) % sim.Ns < sim.N
        for a, b in zip(out, again):
            assert np.array_equal(a[live].view(np.uint8), b[live].view(np.uint8)), (what, "padding leaks")


# ---- every instantiation, fp32 and bf16 rows, even and odd widths ---------------------------------------------------

@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("d", [10, 11, 22, 23, 50, 47, 58, 59, 64])
def test_instantiations(d, dtype):
    # D <= 15: PRE 1, <= 31: 2, <= 63: 4, 64: 5.  900 rows = 7 * 128 + 4; house 99 of every replica is a padding slot
    env = _env(d, 99, 9, dtype)
    _case(env, d, 100, 100, seed=d, what=f"D={d} {dtype}", padding_check=True)


# ---- hidden widths: everything up to h1 = h2 = 128 at D = 64 fits -----------------------------------------------------

@pytest.mark.parametrize("d,h1,h2", [(23, 1, 1), (23, 1, 128), (23, 128, 1), (23, 128, 128), (64, 128, 128),
                                     (47, 120, 127), (64, 100, 100), (23, 127, 113)])
def test_network_widths(d, h1, h2):
    env = _env(d, 99, 13)
    _case(env, d, h1, h2, seed=h1 * 1000 + h2 + d, what=f"{h1}x{h2} D={d}")


# ---- row counts ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("r,n", [(3, 37), (9, 99), (1600, 99)])
def test_row_counts(r, n, dtype):
    env = _env(11, n, r, dtype)
    _case(env, 11, 100, 100, seed=r, what=f"R={r} N={n} {dtype}", padding_check=True)


# ---- output pointers -------------------------------------------------------------------------------------------------

def test_output_pointer_combinations():
    env = _env(22, 99, 9)
    rng = np.random.default_rng(11)
    net = ar.sample_net(rng, 22, 64, 48)
    _write_rows(env, ar.sample_rows(rng, 900, 22, net), PAD_VALUE)
    w = _weights(net)
    full = _run(env, w, K)
    for want in ((False, False), (True, False), (False, True)):
        out = _run(env, w, K, want)
        assert np.array_equal(out[0], full[0]), want
        for k, flag in enumerate(want):
            if flag:
                assert np.array_equal(out[1 + k], full[1 + k]), want
            else:
                assert np.all(out[1 + k] == np.float32(-7.0)), want
    env.sim.actor_status()


# ---- refusals, one step past each accepted limit ----------------------------------------------------------------------

def test_refusals():
    import ctypes as C

    from marl_demandresponse_b200 import _lib

    rng = np.random.default_rng(3)
    env = _env(23, 99, 9)
    for h1, h2 in ((129, 8), (8, 129), (0, 8)):
        w = _weights(ar.sample_net(rng, 23, h1, h2))
        _refused(env, lambda: env.sim.policy_step(w, seed=SEED, precision=K), "h1, h2 in")
    e65 = _env(65, 20, 2)
    w = _weights(ar.sample_net(rng, 65, 16, 16))
    _refused(e65, lambda: e65.sim.policy_step(w, seed=SEED, precision=K), r"obs_dim must be in \[1, 64\]")
    # precision values other than 0, 1, 2
    sim = env.sim
    w = _weights(ar.sample_net(rng, 23, 32, 32))
    for bad in (3, -1, 100):
        net = sim.actor_net(w, K)
        net.precision = bad
        _refused(env, lambda: _lib.check(sim._L.drsim_policy_step(sim._h, C.byref(net), SEED, None, None, sim._stream())),
                 "precision must be 0")


# ---- the fp16 range: exact, or reported -------------------------------------------------------------------------------

def _flagged(env, fn):
    """Runs ``fn`` (one f16x3 launch) and returns whether ``actor_status`` reported the range flag."""
    from marl_demandresponse_b200 import _lib

    fn()
    try:
        env.sim.actor_status()
    except _lib.DrsimError as e:
        assert "f16x3" in str(e) and "65520" in str(e), str(e)
        return True
    return False


def test_range_rows_and_activations():
    from marl_demandresponse_b200 import _lib

    env = _env(11, 99, 9)
    sim = env.sim
    rng = np.random.default_rng(21)
    net = ar.sample_net(rng, 11, 100, 100)
    net = (net[0] * np.where(np.arange(11) < 4, 1.0, 0.25).astype(np.float32),) + net[1:]   # 65504 x w1 stays below 65520
    w = _weights(net)
    base = ar.sample_rows(rng, 900, 11, net)
    idx = _sample(sim, rng)
    live_rows = np.flatnonzero(np.arange(900) % sim.Ns < sim.N)

    # the largest fp16 value in live rows: in range, exact
    rows = base.copy()
    rows[live_rows[::7], 4] = 65504.0
    rows[live_rows[3::7], 5] = -65504.0
    stored = _write_rows(env, rows, PAD_VALUE)
    out = _run(env, w, K)
    _check(env, stored, net, out, idx, "rows at 65504")

    # beyond it: an observation element of one live row, then hidden activations of one live row (the row itself in range)
    for what, value, col in (("row element 7e4", 70000.0, 2), ("row element -1e30", -1e30, 0), ("hidden 1e5", 60000.0, None)):
        # (the hidden case: every element in range, |w1| ~ 0.3 makes activations of ~1e5)
        rows = base.copy()
        r = live_rows[len(live_rows) // 2]
        if col is None:
            rows[r, :] = value
        else:
            rows[r, col] = value
        stored = _write_rows(env, rows, PAD_VALUE)
        _, _, info = hr.forward(stored[[r]], *net)
        assert info["out_of_range"][0], what
        assert _flagged(env, lambda: _run(env, w, K)), what
        # the flag is reported once: the handle works again, and rows back in range are exact
        _write_rows(env, base, PAD_VALUE)
        assert not _flagged(env, lambda: _run(env, w, K)), what

    # a flagged launch also fails the NEXT actor call of the handle (nothing launched)
    rows = base.copy()
    rows[live_rows[0], 1] = 1e6
    _write_rows(env, rows, PAD_VALUE)
    _run(env, w, K)
    import torch

    torch.cuda.synchronize()
    _refused(env, lambda: sim.policy_step(w, seed=SEED, precision=K), "f16x3")
    sim.actor_status()                                  # reported once


@pytest.mark.parametrize("scale", [1e-4, 1e-30, 300.0])
def test_range_tiny_and_huge_weights(scale):
    """Weights far below the fp16 normal range (the per-neuron scale lifts them) and large ones (hidden activations stay
    in range for these rows): exact."""
    env = _env(23, 99, 9)
    rng = np.random.default_rng(int(abs(np.log10(scale))) + 5)
    net = list(ar.sample_net(rng, 23, 100, 100))
    net[0] = (net[0] * np.float32(scale)).astype(np.float32)
    net[1] = (net[1] * np.float32(scale)).astype(np.float32)
    net[2] = (net[2] / np.float32(scale) if scale > 1 else net[2]).astype(np.float32)
    rows = ar.sample_rows(rng, 900, 23)
    _case(env, 23, 100, 100, seed=7, what=f"weights x {scale:g}", net=tuple(net), rows=rows)


# ---- the rollout ---------------------------------------------------------------------------------------------------------

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
    pytest.param(3, 100, "tarmac", {"solar_gain": True}, "bfloat16", id="3-100-tarmac-solar-bfloat16")])
def test_collect_equals_policy_step_plus_step(R, n, layout, state_prop, obs_dtype):
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from marl_demandresponse_b200.batched import synthetic_state
    from marl_demandresponse_b200.rollout import RolloutBuffer
    from oracle_driver import prop as _prop

    T = 7
    prop = {**_prop(n), "state_prop": state_prop}
    st = synthetic_state(prop, R, seed=4)
    a = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=17, obs_dtype=obs_dtype)
    b = BatchedEnv(prop, R, obs_layout=layout, noise="philox", seed=17, obs_dtype=obs_dtype)
    a.reset(copy.deepcopy(st))
    b.reset(copy.deepcopy(st))
    weights = BatchedEnv.actor_weights(_actor(a.sim.D))
    buf = RolloutBuffer(a, T)
    a.collect(weights, buf, done_last=True, precision=K)
    states, actions, probs, rewards = [], [], [], []
    for t in range(T):
        states.append(b.obs.clone())
        act, prob = b.policy_step(weights, precision=K)
        actions.append(act.clone())
        probs.append(prob.clone())
        b.sim.step(None)
        rewards.append(b.reward.clone())
    torch.cuda.synchronize()
    b.sim.actor_status()
    for t in range(T):
        assert torch.equal(buf.state(t), states[t]), ("state", t)
        assert torch.equal(buf.action(t), actions[t]), ("action", t)
        assert torch.equal(buf.prob(t), probs[t]), ("prob", t)
        assert torch.equal(buf.reward(t), rewards[t]), ("reward", t)
    assert torch.equal(buf.next_state(T - 1), b.obs)
    for k in ("dt_air", "dt_mass", "sso", "flags", "signal", "power", "metrics"):
        assert torch.equal(a.state[k], b.state[k]), k


@pytest.mark.parametrize("shape", ["c4", "c3"])
def test_real_rows_agree_with_tf32x3(shape):
    """The environment's own rows at the benchmark's C4 (2048 x 1000, tarmac, D = 10) and C3 (4096 x 100,
    hand-engineered, D = 50) shapes with a 100 x 100 actor: on every row the two fp32-grade actors agree within the sum
    of their tolerances, and each is within its tolerance of the fp64 forward on a sample."""
    import torch

    from marl_demandresponse_b200 import BatchedEnv
    from oracle_driver import prop as _prop

    R, n, layout = (2048, 1000, "tarmac") if shape == "c4" else (4096, 100, "hand_engineered")
    env = BatchedEnv(_prop(n), R, obs_layout=layout, noise="philox", seed=1)
    env.reset()
    sim = env.sim
    w = BatchedEnv.actor_weights(_actor(sim.D, seed=0))
    zeros = torch.zeros((R, n), dtype=torch.uint8, device="cuda")
    for _ in range(3):
        env.step(zeros)
    outs = {}
    for k in ("tf32x3", K):
        p_on = torch.zeros((R, sim.Ns), dtype=torch.float32, device="cuda")
        sim.policy_step(w, seed=SEED, prob_on=p_on, precision=k)
        outs[k] = (sim.views()["actions_padded"].cpu().numpy().reshape(-1).copy(), p_on.cpu().numpy().reshape(-1).astype(np.float64))
    sim.actor_status()
    rows = sim.views()["obs_padded"].float().cpu().numpy().reshape(-1, sim.D)
    net = tuple(t.cpu().numpy() for t in w)
    live = np.flatnonzero(np.arange(R * sim.Ns) % sim.Ns < n)
    rng = np.random.default_rng(0)
    pick = np.sort(rng.choice(live, 20000, replace=False))
    tol = hr.fp32_grade_tolerance(rows[pick], *net)
    p64 = ar.forward64(rows[pick], *net)
    e = {k: float(np.abs(outs[k][1][pick] - p64).max()) for k in outs}
    print(f"actor real rows {shape}: max |dp64| f16x3 {e[K]:.3g}, tf32x3 {e['tf32x3']:.3g}, tolerance {tol:.3g}")
    assert e[K] <= tol and e["tf32x3"] <= tol
    diff = np.abs(outs[K][1][live] - outs["tf32x3"][1][live])
    print(f"actor real rows {shape}: max |p_f16x3 - p_tf32x3| over {len(live)} rows {float(diff.max()):.3g}")
    assert diff.max() <= 2 * tol
