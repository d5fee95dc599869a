"""``random_sample`` neighbours drawn on the device (DRSIM_COMM_SAMPLE), host side.

The device draws neighbour k of house n after the handle's d-th step with one ``__host__ __device__`` sampler
(``CommSampler``, drsim_device.cuh); ``drsim_host_comm_sample`` runs that code on the host and ``comm_sample_np``
restates it in NumPy.  These tests pin the two to each other bit for bit, check that the restatement has the
distribution of ``random.sample(ids without n, c)`` (a uniformly random ordered c-tuple of distinct other houses), and
check the configuration mapping.  Every sample comes from fixed seeds, so the statistical tests are deterministic.
"""
import ctypes as C
import itertools

import numpy as np
import pytest
from scipy import stats

import comm_sample_np

P_MIN = 1e-4   # fixed seeds: each p-value below is a constant; a correct sampler sits far above this


def _host(seed, rep, house, draw, n, c):
    from marl_demandresponse_b200 import _lib

    out = (C.c_int32 * c)()
    _lib.lib().drsim_host_comm_sample(seed, rep, house, draw, n, c, C.cast(out, C.c_void_p))
    return list(out)


def test_host_sampler_equals_numpy_restatement():
    rng = np.random.default_rng(7)
    cases = [(2, 1), (3, 2), (4, 3), (10, 9), (10, 1), (33, 32), (100, 10), (1000, 10), (10 ** 6, 32), (10 ** 6, 1),
             (10 ** 6, 5), (2 ** 31 - 1, 7)]
    for _ in range(3000):
        n = int(rng.choice([2, 3, 5, 9, 10, 17, 100, 1000, 10 ** 6]))
        c = int(rng.integers(1, min(n - 1, 32) + 1))
        cases.append((n, c))
    for i, (n, c) in enumerate(cases):
        seed = int(rng.integers(0, 2 ** 63)) if i % 2 else int(rng.integers(0, 2 ** 20))
        rep, house, draw = int(rng.integers(0, 2 ** 32)), int(rng.integers(0, min(n, 2 ** 31))), int(rng.integers(0, 2 ** 32))
        want = comm_sample_np.comm_sample(seed, rep, house, draw, n, c)
        got = _host(seed, rep, house, draw, n, c)
        assert got == want.tolist(), (seed, rep, house, draw, n, c, got, want)


def test_vectorised_table_matches_per_house_draws():
    t = comm_sample_np.comm_sample_table(11, 3, 12, 5, 11, rep_offset=40)
    assert t.shape == (3, 12, 11)
    for r in range(3):
        for n in range(12):
            assert t[r, n].tolist() == _host(11, 40 + r, n, 5, 12, 11)


def _rows(n, c, reps=200, draws=60, seed=3):
    """[reps * draws * n, c] draws of every house (different replicas and draw indices)."""
    out = [comm_sample_np.comm_sample_table(seed, reps, n, d, c) for d in range(draws)]
    return np.concatenate(out).reshape(-1, n, c)


@pytest.mark.parametrize("n,c", [(4, 3), (6, 2)])
def test_every_ordered_tuple_is_equally_likely(n, c):
    rows = _rows(n, c)                                  # [S, n, c]
    for house in range(n):
        others = [i for i in range(n) if i != house]
        tuples = {t: k for k, t in enumerate(itertools.permutations(others, c))}
        idx = np.array([tuples[tuple(r)] for r in rows[:, house].tolist()])
        counts = np.bincount(idx, minlength=len(tuples))
        assert stats.chisquare(counts).pvalue > P_MIN, (house, counts)


@pytest.mark.parametrize("n,c,reps,draws", [(10, 9, 200, 60), (1000, 10, 40, 4)])
def test_positions_and_pairs_are_uniform(n, c, reps, draws):
    rows = _rows(n, c, reps, draws)                     # [S, n, c]
    # offset of a neighbour past the house itself: uniform over 0 .. n - 2 at every position
    off = (rows - np.arange(n)[None, :, None]) % n - 1
    for k in range(c):
        counts = np.bincount(off[:, :, k].ravel(), minlength=n - 1)
        assert stats.chisquare(counts).pvalue > P_MIN, ("position", k)
    # pairs of positions (0, 1) and (0, c - 1): uniform over the ordered pairs of distinct offsets, counted in
    # b x b bins of offsets (b = 9: every pair; b = 10 deciles for n = 1000, each bin weighted by its pairs)
    b = min(n - 1, 10)
    q = (n - 1 + b - 1) // b
    size = np.bincount(np.arange(n - 1) // q, minlength=b).astype(np.float64)
    want = np.outer(size, size) - np.diag(size)        # distinct ordered pairs per bin pair
    for k in (1, c - 1):
        x, y = off[:, :, 0].ravel(), off[:, :, k].ravel()
        assert not np.any(x == y)
        got = np.bincount((x // q) * b + y // q, minlength=b * b).astype(np.float64)
        keep = want.ravel() > 0
        exp = want.ravel()[keep] / want.sum() * got.sum()
        assert stats.chisquare(got[keep], exp).pvalue > P_MIN, ("pair", k)


@pytest.mark.parametrize("n,c", [(2, 1), (5, 4), (10, 9), (33, 32), (1000, 10)])
def test_no_self_reference_and_no_repeat(n, c):
    t = np.concatenate([comm_sample_np.comm_sample_table(9, 16, n, d, c) for d in range(4)])
    assert t.min() >= 0 and t.max() < n
    assert not np.any(t == np.arange(n)[None, :, None])
    s = np.sort(t, axis=-1)
    assert not np.any(s[..., 1:] == s[..., :-1])


def test_consecutive_draws_of_a_house_are_independent():
    n, c = 10, 3
    a = np.concatenate([comm_sample_np.comm_sample_table(5, 400, n, d, c) for d in range(0, 40, 2)])
    b = np.concatenate([comm_sample_np.comm_sample_table(5, 400, n, d + 1, c) for d in range(0, 40, 2)])
    off = lambda t: (t - np.arange(n)[None, :, None]) % n - 1  # noqa: E731
    x, y = off(a)[..., 0].ravel(), off(b)[..., 0].ravel()
    table = np.bincount(x * (n - 1) + y, minlength=(n - 1) ** 2).reshape(n - 1, n - 1)
    assert stats.chi2_contingency(table).pvalue > P_MIN
    assert np.mean(a == b) < 0.2   # a repeated draw would match everywhere


def test_flatten_config_maps_random_sample_to_the_device_draw():
    from marl_demandresponse_b200 import _lib
    from marl_demandresponse_b200.core import flatten_config

    def props(mode):
        return {"cluster_prop": {"nb_agents": 12, "agents_comm_prop": {"mode": mode, "max_nb_agents_communication": 5}}}

    assert flatten_config(props("random_sample")).comm_mode == _lib.COMM_SAMPLE
    assert flatten_config(props("random_sample"), comm_table=True).comm_mode == _lib.COMM_TABLE
    assert flatten_config(props("random_fixed")).comm_mode == _lib.COMM_TABLE
    assert flatten_config(props("neighbours")).comm_mode == _lib.COMM_RING
    assert _lib.lib().drsim_step_count(None) == -1


def _create_error(cfg):
    from marl_demandresponse_b200 import _lib

    L = _lib.lib()
    h = C.c_void_p()
    rc = L.drsim_create(C.byref(cfg), 0, C.byref(h))
    return rc, L.drsim_last_error().decode()


def test_house_sharded_random_sample_is_refused():
    from marl_demandresponse_b200 import _lib
    from marl_demandresponse_b200.core import flatten_config
    from marl_demandresponse_b200.sharded import ShardedClusterEnv

    p = {"cluster_prop": {"nb_agents": 64, "agents_comm_prop": {"mode": "random_sample", "max_nb_agents_communication": 4}}}
    with pytest.raises(ValueError, match="random_sample"):
        ShardedClusterEnv(p, 2, rank=0, world=2, obs_layout="hand_engineered")
    # the C ABI refuses the configuration before it looks for a device
    cfg = flatten_config(p, 2, "f32", "hand_engineered", path="split", house_offset=0, n_house_local=32)
    assert cfg.comm_mode == _lib.COMM_SAMPLE
    rc, msg = _create_error(cfg)
    assert rc == -1 and "random_sample" in msg, (rc, msg)


def test_sampled_neighbour_count_is_bounded():
    from marl_demandresponse_b200 import _lib
    from marl_demandresponse_b200.core import flatten_config

    p = {"cluster_prop": {"nb_agents": 64, "agents_comm_prop": {"mode": "random_sample", "max_nb_agents_communication": 33}}}
    cfg = flatten_config(p, 2)
    assert cfg.nb_comm == 33 > _lib.MAX_SAMPLE_COMM
    rc, msg = _create_error(cfg)
    assert rc == -1 and "DRSIM_MAX_SAMPLE_COMM" in msg, (rc, msg)
    cfg.comm_mode = 3
    assert _create_error(cfg) == (-1, "drsim_create: comm_mode")
