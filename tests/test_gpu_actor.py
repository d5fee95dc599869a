"""The tcgen05 actor kernels (``k_actor2`` = "tf32", ``k_actor3<SplitTf32x3, PRE, O>`` = "tf32x3") against the operand-exact
reference ``oracle.actor_ref``: every row's ``prob_on`` must lie within the reference's first-principles error bound.

The rows are synthetic (``actor_ref.sample_rows``: four decades of magnitudes, exact zeros, values on TF32 ties, a few
saturating rows) and are written straight into the handle's observation plane, so the actor is tested apart from the
step.  The handle has stepped a few times first (the draw is keyed by a step index > 1), its replicas start at a
non-zero global index and the seed uses both key words of the Philox draw.  Padding slots (house >= N) hold huge finite
values: they must still get action 0 and probability 0, and leave every other row bit-identical.

Covered: every ``k_actor3<SplitTf32x3>`` instantiation (PRE = 2, 4, 7, 9) with fp32 and bf16 rows of even and odd width, and
``k_actor2`` on the fp32 rows; hidden widths from 1 to 128 up to each kernel's tensor- and shared-memory limits; row
counts below one tile, one row into a tile, and many tiles per CTA; all output-pointer combinations; the refusals."""
import ctypes as C

import numpy as np
import pytest

from oracle import actor_ref as ar
from oracle_driver import prop as _prop

pytestmark = pytest.mark.gpu

SEED = 0x123456789ABCDEF0     # both 32-bit words of the Philox key matter
REP_OFFSET = 1000
STEPS = 3                     # steps taken before the actor runs: the draw's step index is 3
PURPOSE_POLICY = 6
SMEM_MAX = 227 * 1024
# largest per-row bound accepted in any case: keeps a vacuous bound from passing the comparison.  The bound charges
# every fp32 accumulation its worst case (K 2^-23 sum |a w|), which for "tf32x3" is about as wide as the error of a
# single TF32 pass; that kernel is also held to fp32-grade probabilities (actor_ref.fp32_grade_tolerance, ~2e-6)
MAX_BOUND = {"tf32": 2e-3, "tf32x3": 1e-3}
PAD_VALUE = 1e30

# observation widths reachable by configuration: D -> (layout, property overrides)
_SOLAR = {"state_prop/solar_gain": True}


def _comm(c, **over):
    return {"cluster_prop/agents_comm_prop/max_nb_agents_communication": c, **over}


WIDTHS = {
    10: ("tarmac", {}),                                          # k_actor3<SplitTf32x3, 2>
    11: ("tarmac", _SOLAR),
    22: ("hand_engineered", _comm(3)),                           # <4>
    23: ("hand_engineered", _comm(3, **_SOLAR)),
    50: ("hand_engineered", _comm(10)),                          # <7>
    47: ("hand_engineered", _comm(9, **_SOLAR)),
    58: ("hand_engineered", _comm(12)),                          # <9>
    59: ("hand_engineered", _comm(12, **_SOLAR)),
    64: ("hand_engineered", _comm(13, **{"state_prop/hvac": True})),   # 12 own columns + 13 four-column messages
    65: ("hand_engineered", _comm(13, **{"state_prop/hvac": True}, **_SOLAR)),   # one past the actor's limit
}


def _r(x, m):
    return (x + m - 1) // m * m


def actor_layout(d, h1, h2, kernel):
    """The host's layout rules of ``policy_step_impl`` (drsim_api.cu): (TMEM columns, dynamic shared memory bytes)
    and whether the launch is accepted."""
    k1, n1, k2 = _r(d + 1, 8), _r(h1 + 1, 16), _r(h1 + 1, 8)
    if kernel == "tf32x3":
        n2 = _r(h2, 16)
        tmem = 2 * (n1 + n2)                                          # R1 | L1 | R2[0] | R2[1]
        w = _r(n1 * k1 * 4, 128) + _r(n2 * k2 * 4, 128)
        smem = 2 * w + _r((2 * n2 + 2) * 4, 128) + _r(2 * 128 * k1 * 4, 128) + 128
    else:
        n2, k3 = _r(h2 + 1, 16), _r(h2 + 1, 8)
        tmem = 2 * (n1 + n2 + 16)                                     # two tile slots of 256 columns
        smem = (_r(n1 * k1 * 4, 128) + _r(n2 * k2 * 4, 128) + _r(16 * k3 * 4, 128) + _r(2 * 128 * k1 * 4, 128)
                + _r(2 * _r(128 * d * 4, 128), 128) + 128)
    ok = 1 <= d <= 64 and 1 <= h1 <= 128 and 1 <= h2 <= 128 and tmem <= 512 and smem <= SMEM_MAX
    return tmem, smem, ok


def _env(d, n, r, dtype="float32"):
    import torch

    from marl_demandresponse_b200 import BatchedEnv

    layout, over = WIDTHS[d]
    env = BatchedEnv(_prop(n, **over), r, obs_layout=layout, noise="philox", seed=7, rep_offset=REP_OFFSET,
                     obs_dtype=dtype)
    assert env.sim.D == d
    env.reset(device_mode="synthetic")
    zeros = torch.zeros((r, n), dtype=torch.uint8, device="cuda")
    for _ in range(STEPS):
        env.step(zeros)
    assert env.sim.step_count == STEPS
    return env


def _write_rows(env, rows, pad):
    """Rows ``[R * Ns, D]`` (fp32) into the observation plane; padding slots get ``pad``.  Returns the values stored
    (bf16 handles: the rows rounded to bf16)."""
    import torch

    sim = env.sim
    x = rows.reshape(sim.R, sim.Ns, sim.D).copy()
    x[:, sim.N:, :] = pad * np.where(np.arange(sim.D) % 2 == 0, 1.0, -1.0).astype(np.float32)
    plane = sim.views()["obs_padded"]
    plane.copy_(torch.from_numpy(x).to(plane.dtype))
    torch.cuda.synchronize()
    stored = plane.float().cpu().numpy().reshape(-1, sim.D)
    if sim.obs_bf16:
        assert np.array_equal(stored, ar.bf16(x.reshape(-1, sim.D)))
    return stored


def _run(env, weights, kernel, want=(True, True), sentinel=-7.0):
    import torch

    sim = env.sim
    bufs = [torch.full((sim.R, sim.Ns), sentinel, dtype=torch.float32, device="cuda") for _ in range(2)]
    prob, prob_on = (b if w else None for b, w in zip(bufs, want))
    sim.policy_step(weights, seed=SEED, prob_drawn=prob, prob_on=prob_on, precision=kernel)
    torch.cuda.synchronize()
    out = [sim.views()["actions_padded"].cpu().numpy().reshape(-1)]
    return out + [b.cpu().numpy().reshape(-1) for b in bufs]


def _uniform(rows_idx, ns, step):
    from oracle import philox

    x = philox.philox4x32_10(SEED, REP_OFFSET + rows_idx // ns, rows_idx % ns, step, PURPOSE_POLICY)[0]
    return (x.astype(np.uint64) >> np.uint64(8)).astype(np.float64) * 2.0 ** -24


def _sample(sim, rng, n_sample=4000):
    """Rows compared against the reference: all rows of the first and the last tile, a seeded sample of the rest;
    live rows (house < N) only."""
    m = sim.R * sim.Ns
    idx = np.arange(m)
    if m > 2 * 128 + n_sample:
        mid = idx[128:(m - 1) // 128 * 128]
        idx = np.concatenate([idx[:128], np.sort(rng.choice(mid, n_sample, replace=False)), idx[(m - 1) // 128 * 128:]])
    return idx[idx % sim.Ns < sim.N]


def _check(sim, stored, net, kernel, out, idx, what):
    act, prob, prob_on = out
    live = np.arange(sim.R * sim.Ns) % sim.Ns < sim.N
    assert not act[~live].any() and not prob[~live].any() and not prob_on[~live].any(), (what, "padding slots")
    assert set(np.unique(act)) <= {0, 1}
    p_ref, bound, _ = ar.forward(stored[idx], *net, kernel=kernel)
    got = prob_on[idx].astype(np.float64)
    err = np.abs(got - p_ref)
    worst = int(np.argmax(err / bound))
    assert np.all(err <= bound), (what, kernel, "row", int(idx[worst]), got[worst], p_ref[worst], bound[worst])
    assert bound.max() <= MAX_BOUND[kernel], (what, kernel, bound.max())
    line = (f"actor {what} {kernel}: rows {len(idx)}, max |dp|/bound {float((err / bound).max()):.3g}, "
            f"max bound {float(bound.max()):.3g}")
    if kernel == "tf32x3":   # fp32-grade: the bound above cannot tell three TF32 passes from one, this can
        tol = ar.fp32_grade_tolerance(stored[idx], *net)
        err64 = np.abs(got - ar.forward64(stored[idx], *net))
        assert err64.max() <= tol, (what, "fp32 grade", int(idx[np.argmax(err64)]), float(err64.max()), tol)
        line += f", max |dp64| {float(err64.max()):.3g} of {tol:.3g}"
    print(line)
    # the draw: u < p0 -> action 0, u from the top 24 bits of Philox word 0 of (seed; replica, house, step, purpose)
    u, p0 = _uniform(idx, sim.Ns, STEPS), 1.0 - p_ref
    clear = np.abs(u - p0) > bound + 2.0 ** -22
    assert (~clear).sum() <= max(2, 0.001 * len(idx)), (what, clear.mean())   # 99.9 %, or two rows of a small case
    assert np.array_equal(act[idx][clear], (u >= p0)[clear].astype(np.uint8)), (what, kernel, "draw")
    # prob = the probability of the action that was drawn
    on = act[idx] == 1
    assert np.array_equal(prob[idx][on], prob_on[idx][on])
    assert np.all(np.abs(prob[idx][~on].astype(np.float64) - (1.0 - got[~on])) <= 2.0 ** -22)


def _weights(net):
    import torch

    return tuple(torch.from_numpy(w).cuda() for w in net)


def _case(env, d, h1, h2, kernels, seed, what, padding_check=False):
    rng = np.random.default_rng(seed)
    sim = env.sim
    net = ar.sample_net(rng, d, h1, h2)
    rows = ar.sample_rows(rng, sim.R * sim.Ns, d, net)
    idx = _sample(sim, rng)
    for kernel in kernels:
        assert actor_layout(d, h1, h2, kernel)[2], (d, h1, h2, kernel)
    w = _weights(net)
    stored = _write_rows(env, rows, PAD_VALUE)
    outs = {k: _run(env, w, k) for k in kernels}
    for k in kernels:
        _check(sim, stored, net, k, outs[k], idx, what)
    if padding_check:   # huge padding values change nothing else, bit for bit
        _write_rows(env, rows, 0.0)
        for k in kernels:
            again = _run(env, w, k)
            live = np.arange(sim.R * sim.Ns) % sim.Ns < sim.N
            for a, b in zip(outs[k], again):
                assert np.array_equal(a[live].view(np.uint8), b[live].view(np.uint8)), (what, k, "padding leaks")


# ---- every instantiation of the row handling, fp32 and bf16 rows, even and odd widths -------------------------------

@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("d", [10, 11, 22, 23, 50, 47, 58, 59, 64])
def test_instantiations(d, dtype):
    # R * Ns = 900 = 7 * 128 + 4: the last tile holds four rows; house 99 of every replica is a padding slot
    env = _env(d, 99, 9, dtype)
    h2 = 96 if d == 64 else 100            # 100 x 100 at D = 64 exceeds the 3xTF32 shared memory (refusal test)
    kernels = ("tf32x3",) if dtype == "bfloat16" else ("tf32x3", "tf32")
    _case(env, d, 100, h2, kernels, seed=d, what=f"D={d} {dtype}", padding_check=True)


# ---- hidden widths up to each kernel's limits -----------------------------------------------------------------------

# tf32: N1 + N2 + 16 = 256 columns fill a k_actor2 tile slot; tf32x3: 2 (N1 + N2) = 512 fill the tensor memory,
# h1 = 128 (K2 = 136) is the only width with a fifth 32-column chunk of the layer-2 operand
WIDTH_CASES = [
    (23, 1, 1, "tf32"), (23, 1, 1, "tf32x3"), (23, 1, 128, "tf32"), (23, 1, 128, "tf32x3"),
    (23, 100, 100, "tf32"), (23, 100, 100, "tf32x3"),
    (23, 128, 95, "tf32"), (23, 127, 111, "tf32"), (23, 111, 127, "tf32"),
    (23, 128, 112, "tf32x3"), (23, 127, 128, "tf32x3"),
    (47, 120, 127, "tf32x3"),     # 1792 bytes under 227 KB of shared memory: the closest any reachable width gets
]


@pytest.mark.parametrize("d,h1,h2,kernel", WIDTH_CASES)
def test_network_widths(d, h1, h2, kernel):
    tmem, smem, ok = actor_layout(d, h1, h2, kernel)
    assert ok
    if (h1, h2) in ((128, 95), (127, 111), (111, 127), (128, 112), (127, 128)):
        assert tmem == 512        # k_actor2: both 256-column slots full; k_actor3 (tf32x3): R1 | L1 | R2[0] | R2[1] fill 512
    if (d, h1, h2) == (47, 120, 127):
        assert SMEM_MAX - 2048 < smem <= SMEM_MAX
    env = _env(d, 99, 13)
    _case(env, d, h1, h2, (kernel,), seed=h1 * 1000 + h2, what=f"{h1}x{h2} D={d}")


# ---- row counts: one partial tile, a four-row last tile, many tiles per CTA -----------------------------------------

@pytest.mark.parametrize("dtype,kernels", [("float32", ("tf32x3", "tf32")), ("bfloat16", ("tf32x3",))])
@pytest.mark.parametrize("r,n", [(3, 37), (9, 99), (1600, 99)])
def test_row_counts(r, n, dtype, kernels):
    # 120 rows; 900 = 7 * 128 + 4; 160000 rows = 1250 tiles: each of 148 CTAs takes about 8.4 tiles (k_actor3: both
    # R2 slots recycled four times) or 4.2 per tile slot (k_actor2)
    env = _env(11, n, r, dtype)
    _case(env, 11, 100, 100, kernels, seed=r, what=f"R={r} N={n} {dtype}", padding_check=True)


# ---- output pointers -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kernel", ["tf32", "tf32x3"])
def test_output_pointer_combinations(kernel):
    env = _env(22, 99, 9)
    rng = np.random.default_rng(11)
    net = ar.sample_net(rng, 22, 64, 48)
    _write_rows(env, ar.sample_rows(rng, 900, 22, net), PAD_VALUE)
    w = _weights(net)
    full = _run(env, w, kernel)
    sentinel = np.float32(-7.0)
    for want in ((False, False), (True, False), (False, True)):
        out = _run(env, w, kernel, want)
        assert np.array_equal(out[0], full[0]), want                        # the draw does not depend on the outputs
        for k, flag in enumerate(want):
            if flag:
                assert np.array_equal(out[1 + k], full[1 + k]), want
            else:
                assert np.all(out[1 + k] == sentinel), want                  # a null output is not written


# ---- refusals --------------------------------------------------------------------------------------------------------

def _refused(env, fn, match):
    import torch

    from marl_demandresponse_b200 import _lib

    sim = env.sim
    plane = sim.views()["actions_padded"]
    plane.fill_(1)
    before, l0 = plane.clone(), sim.launch_count
    with pytest.raises(_lib.DrsimError, match=match):
        fn()
    torch.cuda.synchronize()
    assert sim.launch_count == l0 and torch.equal(plane, before)


def test_refusals():
    from marl_demandresponse_b200 import _lib
    from marl_demandresponse_b200.rollout import RolloutBuffer

    rng = np.random.default_rng(3)
    env = _env(23, 99, 9)
    for h1, h2, kernel, match in [(129, 8, "tf32x3", "h1, h2 in"), (8, 0, "tf32", "h1, h2 in"),
                                  (128, 96, "tf32", "two tile slots in tensor memory"),
                                  (128, 113, "tf32x3", "split activations in tensor memory")]:
        assert not actor_layout(23, h1, h2, kernel)[2]
        w = _weights(ar.sample_net(rng, 23, h1, h2))
        _refused(env, lambda: env.sim.policy_step(w, seed=SEED, precision=kernel), match)
    # the first refused shapes are one step past the accepted ones of test_network_widths
    assert actor_layout(23, 128, 95, "tf32")[2] and actor_layout(23, 128, 112, "tf32x3")[2]

    e64 = _env(64, 20, 2)
    assert actor_layout(64, 100, 100, "tf32")[2] and not actor_layout(64, 100, 100, "tf32x3")[2]
    w = _weights(ar.sample_net(rng, 64, 100, 100))
    _refused(e64, lambda: e64.sim.policy_step(w, seed=SEED, precision="tf32x3"), "precision = 0")

    e65 = _env(65, 20, 2)
    w = _weights(ar.sample_net(rng, 65, 16, 16))
    for kernel in ("tf32", "tf32x3"):
        _refused(e65, lambda: e65.sim.policy_step(w, seed=SEED, precision=kernel), r"obs_dim must be in \[1, 64\]")

    # rollout slots: obs / reward / next_obs on 16 bytes, actions / prob on 4
    buf = RolloutBuffer(env, 2)
    sim = env.sim
    w = _weights(ar.sample_net(rng, 23, 32, 32))   # kept alive: the net below holds raw device pointers into it
    net = sim.actor_net(w, "tf32x3")
    good = dict(obs=buf.obs[0].data_ptr(), next_obs=buf.obs[1].data_ptr(), actions=buf.actions[0].data_ptr(),
                prob=buf.probs[0].data_ptr(), reward=buf.rewards[0].data_ptr())
    for field, off in (("obs", 4), ("next_obs", 8), ("reward", 4), ("actions", 1), ("prob", 2)):
        slot = _lib.RolloutSlot(**{**good, field: good[field] + off})
        _refused(env, lambda: _lib.check(sim._L.drsim_rollout_transition(sim._h, C.byref(net), SEED, C.byref(slot),
                                                                         sim._stream())), "aligned")
