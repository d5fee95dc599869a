"""The interpolated base power on the CPU: the oracle's interpolator pinned to ``scipy.interpolate.interpn``, and the
fp32 error bound of the kernel's ``interp5<float>`` (``interp_ref``) checked on a float32 emulation of the kernel --
inside the bound as written, outside it with each planted mistake."""
import numpy as np
import pytest

import interp_ref as ir
from oracle.config import DEFAULT_ENV_PROP, synthetic_table
from oracle.np_oracle import interp_point, interp_static_index, interp_sub_tables

TABLE = synthetic_table(7)
SCALE = float(np.abs(TABLE).max())
HOUSE = DEFAULT_ENV_PROP["cluster_prop"]["house_prop"]
DEFAULTS = np.array([HOUSE["Ua"], HOUSE["Cm"], HOUSE["Ca"], HOUSE["Hm"]])


@pytest.fixture(scope="module")
def pts():
    p = ir.point_set(np.random.default_rng(11))
    p["cells"] = ir.cells(p["ratios"], p["cap"])
    p["ref"] = ir.ref_values(TABLE, p["cells"], p["x"])
    return p


def test_point_set_covers_the_edges(pts):
    x = pts["x"]
    for d, g in enumerate(ir.GRIDS):
        assert np.isin(g, x[:, d]).all(), d                        # every node
        assert (x[:, d] < g[0]).any() and (x[:, d] > g[-1]).any(), d
    assert {0.0, 86399.0} <= set(x[:, 3]) and {1.0, 364.0, 365.0, 366.0} <= set(x[:, 4])
    assert (pts["cap"] == 12500.0).any()
    for mid in (0.95, 1.05):
        assert (pts["ratios"] == mid).any()


def test_reference_ties_and_clipping():
    """The reference's own nearest-node rule: first minimum on ties (12500 W goes to 10000 W), clipping at the ends."""
    assert ir.nearest("HVAC_power", np.array([12500.0, 12500.0 + 1e-6, 5000.0, 20000.0])).tolist() == [0, 1, 0, 1]
    assert ir.nearest("Ua_ratio", np.array([0.5, 0.95 - 1e-9, 0.95 + 1e-9, 1.05 - 1e-9, 1.05 + 1e-9, 2.0])).tolist() == \
        [0, 0, 1, 1, 2, 2]
    # date 365 / 366 clip to the last node: the same value as 364
    sub = np.arange(ir.SUB_LEN, dtype=np.float64).reshape(ir.SUB_SHAPE)
    x = np.array([[0.1, 0.2, 4.0, 3600.0, d] for d in (364.0, 365.0, 366.0)])
    v = ir.interpn(ir.GRIDS, sub, ir.clip_points(x), method="linear")
    assert v[0] == v[1] == v[2]


def test_oracle_static_index_matches_reference(pts):
    ratios, cap = pts["ratios"], pts["cap"]
    Ua, Cm, Ca, Hm = (ratios[i] * DEFAULTS[i] for i in range(4))
    got = interp_static_index(Ua, Cm, Ca, Hm, cap, HOUSE)
    want = ir.cells((Ua / DEFAULTS[0], Cm / DEFAULTS[1], Ca / DEFAULTS[2], Hm / DEFAULTS[3]), cap)
    assert np.array_equal(got, ir.flat_cell(want))


def test_oracle_sub_tables_match_reference():
    t10 = TABLE.reshape(ir.INTERP_SHAPE)
    sub = interp_sub_tables(TABLE)
    rng = np.random.default_rng(3)
    for _ in range(40):
        c = np.array([rng.integers(3), rng.integers(3), rng.integers(3), rng.integers(3), rng.integers(2)])
        assert np.array_equal(sub[ir.flat_cell(c)], ir.cell_table(t10, c))


def test_oracle_interp_point_matches_scipy(pts):
    got = interp_point(interp_sub_tables(TABLE), ir.flat_cell(pts["cells"]), *pts["x"].T)
    err = np.abs(got - pts["ref"])
    assert err.max() <= 1e-12 * SCALE, err.max()


def _emulated(pts, mistake=None):
    sub32 = ir.sub_tables_f32(TABLE)
    x32 = pts["x"].astype(np.float32)
    e_in = np.abs(x32.astype(np.float64) - pts["x"])
    got = ir.interp5_f32(sub32, pts["cells"], x32, mistake).astype(np.float64)
    return got, ir.f32_bound(TABLE, pts["cells"], pts["x"], e_in)


def test_fp32_emulation_within_the_bound(pts):
    got, bound = _emulated(pts)
    err = np.abs(got - pts["ref"])
    assert np.all(err <= bound), (err / bound).max()
    # the bound is a few dozen fp32 roundings of the table scale, not a blanket allowance
    assert bound.max() < 200 * ir.U * SCALE, bound.max()
    print(f"fp32 emulation: max error {err.max():.3e} W, max bound {bound.max():.3e} W, max error / bound "
          f"{(err / bound).max():.3f}")


def test_fp32_sum_bound_holds_for_a_sampled_cluster(pts):
    """Base power of a cluster: the houses' fp32 values summed in fp64 and scaled by N / k, inside ``sum_bound``."""
    got, bound = _emulated(pts)
    rng = np.random.default_rng(5)
    for n, k in ((100, 100), (1000, 100), (7, 3)):
        ids = rng.integers(0, len(got), size=min(n, k))
        factor = 1.0 if n <= k else n / k
        dev = float(np.sum(got[ids].astype(np.float64))) * factor
        want = float(np.sum(pts["ref"][ids])) * factor
        assert abs(dev - want) <= ir.sum_bound(pts["ref"][ids], bound[ids], n, k)


@pytest.mark.parametrize("mistake", ["swap", "low", "flip"])
def test_planted_mistakes_land_outside_the_bound(pts, mistake):
    got, bound = _emulated(pts, mistake)
    err = np.abs(got - pts["ref"])
    x = ir.clip_points(pts["x"])
    if mistake == "low":   # only a point on an interior node of some axis has an interval one too low
        live = np.zeros(len(err), dtype=bool)
        for d, g in enumerate(ir.GRIDS):
            live |= np.isin(x[:, d], g[1:-1].astype(np.float32).astype(np.float64))
    elif mistake == "swap":
        live = x[:, 0] != x[:, 1]
    else:
        live = np.ones(len(err), dtype=bool)
    assert live.sum() > 50
    outside = err[live] > bound[live]
    assert outside.mean() > 0.9, (mistake, outside.mean())
