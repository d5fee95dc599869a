"""The interpolated base power (interpolation.py:137-243) restated for the tests, independently of ``oracle.np_oracle``.

* ``ref_values``: the reference itself.  The 10-D table reshaped to ``INTERP_SHAPE``; the nearest index on the four
  thermal ratios and ``HVAC_power`` by a plain argmin after clipping (first minimum on ties); then
  ``scipy.interpolate.interpn(..., method="linear")`` on the five linear axes after clipping.
* ``interp5_f32``: a float32 emulation of the kernel's ``interp5<float>`` in its operation order (clip, interval by
  counting nodes ``<= v``, ``y = (v - g[i]) / (g[i+1] - g[i])``, 32 corners with the last axis fastest, the weight
  multiplied in axis order, terms accumulated in corner order), on the fp32 copy of the table.  ``mistake`` plants
  the errors the bound must catch.
* ``f32_bound``: a first-principles bound on ``|interp5<float> - reference|`` for one house, and ``sum_bound`` the
  bound of the base power, the sum over the sampled houses scaled by ``N / k``.

The bound of one house, with ``u = 2^-24``, ``gamma_n = n u / (1 - n u)``:

* inputs: the kernel interpolates at ``v`` instead of the exact ``x``; ``|v - x|`` per axis is the caller's
  ``e_in`` (the fp32 rounding of ``Ta - target``, ``Tm - target``, ``(float)od - target``), plus the rounding of the
  grid nodes to fp32 (``+-0.3`` on the air axis: interpolating on shifted nodes is interpolating at a shifted point,
  by at most the node shift).  Linear interpolation is continuous across nodes, so whichever interval the kernel
  picks at a node, the value moves by at most ``L_d |v_d - x_d|`` per axis, ``L_d`` the largest slope along axis
  ``d`` over the cells around ``x`` (one interval either side on every axis);
* weights: ``y`` takes three roundings (``|y^ - y| <= gamma_3 y``) and ``1 - y`` one more; the five factors of a
  weight are multiplied with four roundings.  Summed over the 32 corners, the weights are off by at most
  ``omega - 1``, ``omega = (1 + u)^4 (1 + 2 gamma_3 + u (1 + gamma_3))^5``;
* the table rounded to fp32 (``u |T|``) and the 32-term accumulation (``gamma_32`` of the sum of |terms|).

With ``T`` the largest ``|table|`` around ``x``: ``E = sum_d L_d e_d + T ((omega - 1) + u omega + gamma_32 (1 + u)
omega)``.  The kernel adds the houses' fp32 values in fp64 and scales by ``N / k``: ``gamma_{k+3}`` (fp64) of the sum
of |values| on top.
"""
from __future__ import annotations

import datetime as _dt

import numpy as np
from scipy.interpolate import interpn

from oracle.config import INTERP_GRIDS, INTERP_SHAPE

LIN = ("air_temp", "mass_temp", "OD_temp", "hour", "date")
NEAR = ("Ua_ratio", "Cm_ratio", "Ca_ratio", "Hm_ratio", "HVAC_power")
GRIDS = tuple(np.asarray(INTERP_GRIDS[k], dtype=np.float64) for k in LIN)
SUB_SHAPE = tuple(len(g) for g in GRIDS)                    # (9, 5, 8, 12, 6)
SUB_LEN = int(np.prod(SUB_SHAPE))
STRIDE = tuple(int(np.prod(SUB_SHAPE[d + 1:])) for d in range(5))
U = 2.0 ** -24
U64 = 2.0 ** -53


def gamma(n, u=U):
    return n * u / (1 - n * u)


OMEGA = (1 + U) ** 4 * (1 + 2 * gamma(3) + U * (1 + gamma(3))) ** 5
# the rounding of the fp32 grid nodes, per axis
NODE_SHIFT = np.array([np.abs(g - g.astype(np.float32).astype(np.float64)).max() for g in GRIDS])


# ---- the reference ----------------------------------------------------------------------------
def nearest(key, v):
    """Index of the nearest node of ``key``'s grid after clipping; the first on ties."""
    g = np.asarray(INTERP_GRIDS[key], dtype=np.float64)
    v = np.clip(np.asarray(v, dtype=np.float64), g.min(), g.max())
    return np.argmin(np.abs(g[None, :] - v.reshape(-1, 1)), axis=1).reshape(np.shape(v))


def cells(ratios, cap):
    """``[M, 5]`` nearest indices (Ua, Cm, Ca, Hm ratio, HVAC_power) of ``ratios`` = (Ua, Cm, Ca, Hm) / defaults."""
    return np.stack([nearest(k, r) for k, r in zip(NEAR[:4], ratios)] + [nearest("HVAC_power", cap)], axis=-1)


def cell_table(t10, c):
    """The 5-D (air, mass, OD, hour, date) table of nearest cell ``c`` (5 indices) of the 10-D table."""
    return t10[c[0], c[1], c[2], c[3], :, :, :, c[4]]


def clip_points(x):
    return np.stack([np.clip(np.asarray(x, dtype=np.float64)[..., d], g[0], g[-1]) for d, g in enumerate(GRIDS)], axis=-1)


def ref_values(table, cell_idx, x):
    """``[M]`` reference values at points ``x [M, 5]`` (air, mass, OD, hour, date) in cells ``cell_idx [M, 5]``."""
    t10 = np.asarray(table, dtype=np.float64).reshape(INTERP_SHAPE)
    xc = clip_points(x)
    out = np.empty(xc.shape[0])
    keys = [tuple(c) for c in np.asarray(cell_idx)]
    for c in set(keys):
        sel = np.array([k == c for k in keys])
        out[sel] = interpn(GRIDS, cell_table(t10, c), xc[sel], method="linear")
    return out


# ---- the device's fp32 arithmetic -------------------------------------------------------------
def sub_tables_f32(table):
    """The fp32 copy of the table as the device holds it: ``[162 * SUB_LEN]``, cell (Ua, Cm, Ca, Hm, HVAC) major."""
    t10 = np.asarray(table, dtype=np.float64).reshape(INTERP_SHAPE)
    return np.ascontiguousarray(np.moveaxis(t10, 7, 4)).reshape(-1).astype(np.float32)


def flat_cell(cell_idx):
    c = np.asarray(cell_idx)
    return (((c[..., 0] * 3 + c[..., 1]) * 3 + c[..., 2]) * 3 + c[..., 3]) * 2 + c[..., 4]


def interp5_f32(sub32, cell_idx, x32, mistake=None):
    """``interp5<float>`` on fp32 inputs ``x32 [M, 5]``.  ``mistake``: "swap" (air and mass inputs exchanged),
    "low" (the corners of the interval one too low when the point sits on an interior node, the weights unchanged),
    "flip" (each axis' weights taken from the wrong side)."""
    x32 = np.asarray(x32, dtype=np.float32)
    if mistake == "swap":
        x32 = x32[:, [1, 0, 2, 3, 4]]
    M = x32.shape[0]
    one = np.float32(1)
    idx, ys = [], []
    for d, g in enumerate(GRIDS):
        g32 = g.astype(np.float32)
        v = x32[:, d]
        v = np.where(v > g32[-1], g32[-1], np.where(v < g32[0], g32[0], v))
        i = np.zeros(M, dtype=np.int64)
        for k in range(1, len(g) - 1):
            i += (g32[k] <= v)
        y = ((v - g32[i]) / (g32[i + 1] - g32[i])).astype(np.float32)
        if mistake == "low":
            i = np.where((v == g32[i]) & (i > 0), i - 1, i)
        idx.append(i)
        ys.append(y)
    base = flat_cell(cell_idx).astype(np.int64) * SUB_LEN
    value = np.zeros(M, dtype=np.float32)
    for corner in range(32):
        w = np.ones(M, dtype=np.float32)
        o = base.copy()
        for d in range(5):
            up = (corner >> (4 - d)) & 1
            if mistake == "flip":
                up_w = 1 - up
            else:
                up_w = up
            w = w * (ys[d] if up_w else one - ys[d])
            o = o + (idx[d] + up) * STRIDE[d]
        value = value + sub32[o] * w
    return value


def f32_bound(table, cell_idx, x, e_in):
    """``[M]`` bound on ``|interp5<float> - ref_values|`` for one house (see the module docstring): ``x [M, 5]`` the
    exact inputs, ``e_in [M, 5]`` the distance of the kernel's fp32 inputs from them."""
    t10 = np.asarray(table, dtype=np.float64).reshape(INTERP_SHAPE)
    xc = clip_points(x)
    e = np.asarray(e_in, dtype=np.float64) + NODE_SHIFT[None, :]
    out = np.empty(xc.shape[0])
    arith = (OMEGA - 1) + U * OMEGA + gamma(32) * (1 + U) * OMEGA
    for m in range(xc.shape[0]):
        sub = cell_table(t10, cell_idx[m])
        sl, gs = [], []
        for d, g in enumerate(GRIDS):
            i = int(np.clip(np.searchsorted(g, xc[m, d], side="right") - 1, 0, len(g) - 2))
            lo, hi = max(i - 1, 0), min(i + 2, len(g) - 1)
            sl.append(slice(lo, hi + 1))
            gs.append(g[lo:hi + 1])
        block = sub[tuple(sl)]
        slope = 0.0
        for d in range(5):
            shape = [1] * 5
            shape[d] = -1
            s = np.abs(np.diff(block, axis=d)) / np.diff(gs[d]).reshape(shape)
            slope += s.max() * e[m, d]
        out[m] = slope + np.abs(block).max() * arith
    return out


def sum_bound(values, bounds, n, k):
    """Bound of the base power ``(N / k) * sum`` over the sampled houses (with repeats): the houses' bounds, plus the
    fp64 sum and scaling."""
    factor = 1.0 if n <= k else n / k
    terms = np.abs(values) + bounds
    return factor * (np.sum(bounds) + gamma(len(values) + 3, U64) * np.sum(terms))


def od_input_error(od, target32):
    """``|(float)od - target - (od - target)|``: the fp32 outdoor-temperature input of the kernel against the exact one."""
    od = np.asarray(od, dtype=np.float64)
    t32 = np.asarray(target32, dtype=np.float32)
    x32 = (np.asarray(od, dtype=np.float32) - t32).astype(np.float64)
    return np.abs(x32 - (od - t32.astype(np.float64)))


def when_inputs(epoch, solar):
    """(hour, date) inputs of the interpolator at ``epoch`` (naive seconds since 1970): seconds of the day and the
    1-based day of the year (quirk Q12) with solar gain, both 0 without."""
    if not solar:
        return 0.0, 0.0
    w = _dt.datetime(1970, 1, 1) + _dt.timedelta(seconds=int(epoch))
    return float(w.hour * 3600 + w.minute * 60 + w.second), float(w.timetuple().tm_yday)


def ref_base_power(table, house, h, ids, od, epoch, solar, n, k, fp32):
    """Reference base power of one cluster and its tolerance: ``house`` = the cluster's ``[N]`` planes (``t_air,
    t_mass, target, cap, Ua, Cm, Ca, Hm`` and the default thermal parameters ``dUa, dCm, dCa, dHm`` as scalars), ``ids``
    the sampled houses (with repeats), ``od`` / ``epoch`` what the interpolator sees.  The inputs are the device's own
    planes (fp32 build: the fp32 deviations, exact in fp64), so the tolerance is the fp32 bound of ``sum_bound``, or
    1e-12 relative in fp64."""
    ids = np.asarray(ids, dtype=np.int64)
    g = {key: np.asarray(house[key], dtype=np.float64)[ids] for key in ("t_air", "t_mass", "target", "cap", "Ua", "Cm", "Ca", "Hm")}
    c = cells((g["Ua"] / h["dUa"], g["Cm"] / h["dCm"], g["Ca"] / h["dCa"], g["Hm"] / h["dHm"]), g["cap"])
    hour, date = when_inputs(epoch, solar)
    x = np.stack([g["t_air"] - g["target"], g["t_mass"] - g["target"], float(od) - g["target"],
                  np.full(len(ids), hour), np.full(len(ids), date)], axis=1)
    vals = ref_values(table, c, x)
    factor = 1.0 if n <= k else n / k
    total = 0.0
    for v in vals:
        total += v
    base = total * factor
    if not fp32:
        return base, 1e-12 * max(abs(base), 1.0)
    e_in = np.zeros_like(x)
    e_in[:, 0] = np.abs(x[:, 0].astype(np.float32).astype(np.float64) - x[:, 0])
    e_in[:, 1] = np.abs(x[:, 1].astype(np.float32).astype(np.float64) - x[:, 1])
    e_in[:, 2] = od_input_error(np.full(len(ids), float(od)), g["target"])
    return base, sum_bound(vals, f32_bound(table, c, x, e_in), n, k)


# ---- points ------------------------------------------------------------------------------------
def point_set(rng, m_random=400):
    """Inputs that exercise every branch: dict of ``ratios`` (4, M), ``cap`` (M) and ``x`` (M, 5).

    Random interior points; every node of every axis; points beyond each end of each axis; ratios on either side of
    the 0.95 / 1.05 midpoints and on them; ``HVAC_power`` 12500 (an exact tie); hour 0 and 86399; date 1, 364, 365
    and 366 (1-based, clipped at 364)."""
    pts = []

    def add(x, ratios=None, cap=None):
        pts.append((np.asarray(x, dtype=np.float64),
                    np.asarray(ratios if ratios is not None else rng.uniform(0.85, 1.15, 4)),
                    float(cap if cap is not None else rng.choice([9000.0, 10000.0, 12500.0, 15000.0, 16000.0]))))

    def rand_x():
        return np.array([rng.uniform(g[0], g[-1]) for g in GRIDS])

    for _ in range(m_random):
        add(rand_x())
    for d, g in enumerate(GRIDS):
        for v in g:
            for _ in range(3):
                x = rand_x()
                x[d] = v
                add(x)
        span = g[-1] - g[0]
        for v in (g[0] - 0.3 * span, g[0] - 1e-3, g[-1] + 1e-3, g[-1] + 0.3 * span):
            x = rand_x()
            x[d] = v
            add(x)
    nodes = [rng.choice(g) for g in GRIDS]
    add(np.array(nodes, dtype=np.float64))
    for mid in (0.95, 1.05):
        for r in (mid - 1e-9, mid, mid + 1e-9):
            for k in range(4):
                ratios = rng.uniform(0.85, 1.15, 4)
                ratios[k] = r
                add(rand_x(), ratios)
    for cap in (12500.0, 12500.0 - 1e-6, 12500.0 + 1e-6, 10000.0, 15000.0, 5000.0, 20000.0):
        add(rand_x(), cap=cap)
    for hour in (0.0, 86399.0):
        for date in (1.0, 364.0, 365.0, 366.0):
            x = rand_x()
            x[3], x[4] = hour, date
            add(x)
    x = np.stack([p[0] for p in pts])
    ratios = np.stack([p[1] for p in pts], axis=1)
    cap = np.array([p[2] for p in pts])
    return {"x": x, "ratios": ratios, "cap": cap}
