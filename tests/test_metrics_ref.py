"""The literal ``Metrics.update`` (metrics_service.py:108-157, precedence slips included) -- SURVEY 8f-3:
the NumPy restatement against values recorded from the REAL reference class (CPU), and the device kernel
``drsim_metrics_update`` against the same values (GPU)."""
import glob
import json
import os

import numpy as np
import pytest

from golden_util import GOLDEN_DIR, GoldenCase

FILES = sorted(glob.glob(os.path.join(GOLDEN_DIR, "metrics_*.json")))


def _before(case, t):
    """(t_air, signal, power, od_temp) of the observation BEFORE step t."""
    z, s0 = case.z, case.state0
    if t == 0:
        return np.asarray(s0["t_air"])[0], float(np.asarray(s0["signal"])[0]), float(np.asarray(s0["power"])[0]), \
            float(np.asarray(s0["od_temp"])[0])
    return z["t_air"][t - 1], float(z["signal"][t - 1]), float(z["power"][t - 1]), float(z["od_temp"][t - 1])


@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f)[8:-5] for f in FILES])
def test_restatement_matches_the_real_metrics_class(path):
    from oracle.metrics_ref import FIELDS, RefMetrics

    g = json.load(open(path))
    assert g["fields"] == FIELDS
    case = GoldenCase(g["case"])
    m = RefMetrics(case.N, g["start_stats_from"])
    tg = np.asarray(case.state0["target"])[0]
    for t in range(case.T):
        _, sig, p_old, od = _before(case, t)
        m.update(case.z["t_air"][t], tg, case.z["rewards"][t], sig, float(case.z["power"][t]), od, p_old, t)
        np.testing.assert_allclose(m.row(), g["per_step"][t], rtol=1e-13, atol=1e-12)
    rms = m.rms(case.T)
    for k, v in g["rms"].items():
        assert abs(rms[k] - v) <= 1e-12 * max(1.0, abs(v)), k


def test_batched_restatement_matches_the_per_house_loop():
    """``BatchedRefMetrics`` (the ``[R, N]`` form the device metrics are checked against) against ``RefMetrics``
    cluster by cluster: random states, several clusters, squared sums collected from step 5 on, ``Metrics.reset``
    half-way through."""
    from oracle.metrics_ref import FIELDS, RESET_FIELDS, BatchedRefMetrics, RefMetrics

    rng = np.random.default_rng(11)
    R, N, T, start = 5, 37, 14, 5
    bm = BatchedRefMetrics(R, N, start)
    refs = [RefMetrics(N, start) for _ in range(R)]
    for t in range(T):
        if t == 8:
            bm.reset()
            for m in refs:
                for f in RESET_FIELDS:
                    m.v[f] = 0.0
        target = 19.0 + np.abs(rng.normal(0.0, 0.5, (R, N)))
        t_air = target + rng.uniform(-2.0, 4.0, (R, N))
        rew = -rng.uniform(0.0, 2.0, (R, N))
        sig, p_new, p_old = (rng.uniform(0.5, 1.5, R) * 6000.0 * N for _ in range(3))
        od = rng.uniform(25.0, 35.0, R)
        bm.update(t_air, target, rew, sig, p_new, od, p_old, t)
        for r, m in enumerate(refs):
            m.update(t_air[r], target[r], rew[r], sig[r], p_new[r], od[r], p_old[r], t)
        want = np.array([m.row() for m in refs])
        # offsets may cancel across steps: their scale is the matching sum of absolute values
        scale = np.abs(want)
        for signed, absolute in (("cumul_temp_offset", "cumul_temp_error"), ("cumul_signal_offset", "cumul_signal_error")):
            scale[:, FIELDS.index(signed)] = want[:, FIELDS.index(absolute)]
        err = np.abs(bm.values - want)
        assert np.all(err <= 1e-13 * (1.0 + scale)), (t, np.argwhere(err > 1e-13 * (1.0 + scale)).tolist())
    rms = bm.rms(T)
    for r, m in enumerate(refs):
        for k, v in m.rms(T).items():
            assert abs(rms[k][r] - v) <= 1e-13 * max(1.0, abs(v)), (r, k)


@pytest.mark.gpu
@pytest.mark.parametrize("path", FILES, ids=[os.path.basename(f)[8:-5] for f in FILES])
def test_device_metrics_match_the_real_metrics_class(path):
    """The same trajectories replayed through the CUDA step (fp64 build); after every step the device accumulators
    of ``ReferenceMetrics`` (one launch of k_metrics_ref over the state planes) against the recorded values."""
    import torch

    from cuda_stepper import CudaStepper
    from marl_demandresponse_b200.metrics import ReferenceMetrics

    g = json.load(open(path))
    case = GoldenCase(g["case"])
    st = CudaStepper(case.env_prop, 1, "f64", "auto", table=case.table())
    st.set_state(case.state0)
    st.obs_vectors(case.comm(0))
    m = ReferenceMetrics(st.sim, start_stats_from=g["start_stats_from"])
    z = case.z
    uses_perlin = case.env_prop["power_grid_prop"]["signal_properties"]["mode"] == "perlin"
    for t in range(case.T):
        m.begin_step()
        ids = z["interp_ids"][t][None] if z["interp_ids"][t][0] >= 0 else None
        st.step(z["actions"][t][None], [z["od_noise"][t]], [z["perlin"][t]] if uses_perlin else None, ids)
        m.end_step(t)
        got = m.values()[0]
        want = np.asarray(g["per_step"][t])
        err, tol = np.abs(got - want), 1e-9 * np.maximum(1.0, np.abs(want))
        assert np.all(err <= tol), (t, [(f, float(a), float(b)) for f, a, b, e, l in zip(g["fields"], got, want, err, tol) if e > l])
    rms = m.rms(case.T)
    for k, v in g["rms"].items():
        assert abs(float(rms[k][0]) - v) <= 1e-9 * max(1.0, abs(v)), k
    torch.cuda.synchronize()
