"""CPU checks of the "f16x3" actor reference (``actor_ref_f16x3``): the fp16 rounding is IEEE's, a NumPy emulation of the
kernel's arithmetic stays inside the first-principles bound and inside the fp32-grade tolerance, and that tolerance tells
the three fp16 passes from fewer (a truncating split stays fp32-grade: the rounding itself is pinned bit for bit)."""
import numpy as np
import pytest

import actor_ref_f16x3 as hr
from oracle import actor_ref as ar


def _bits16(*b):
    return np.array(b, dtype=np.uint16).view(np.float16).astype(np.float64)


def test_fp16_is_numpy_float16_on_ties_subnormals_and_the_overflow_edge():
    rng = np.random.default_rng(0)
    # every fp16 value and every midpoint between neighbours (ties: even wins), as fp32 inputs
    allh = np.arange(0, 0x7C00, dtype=np.uint16).view(np.float16).astype(np.float64)
    mids = (allh[:-1] + allh[1:]) / 2
    x = np.concatenate([allh, mids, np.nextafter(mids, 0), np.nextafter(mids, np.inf)]).astype(np.float32)
    x = np.concatenate([x, -x, rng.standard_normal(100_000).astype(np.float32) * 10.0 ** rng.uniform(-9, 5, 100_000)])
    # around the largest finite value and the overflow threshold
    x = np.concatenate([x, np.float32([65504, 65519, 65519.996, 65520, 65536, 1e30, 6e-8, 5.96e-8, 2.98e-8, 2.99e-8, 1e-12])])
    x = x.astype(np.float32)
    with np.errstate(over="ignore"):
        want = x.astype(np.float16).astype(np.float64)
    got = hr.fp16(x)
    assert np.array_equal(got.astype(np.float16).view(np.uint16), want.astype(np.float16).view(np.uint16))
    assert np.array_equal(np.signbit(got), np.signbit(want))
    assert hr.fp16(np.float32(65519.99))[()] == 65504.0 and np.isinf(hr.fp16(np.float32(65520.0)))
    assert hr.fp16(2.0 ** -25) == 0.0 and hr.fp16(2.0 ** -25 * 1.5) == 2.0 ** -24   # halfway to the smallest subnormal: even (0)
    assert np.array_equal(hr.fp16(_bits16(0x0001, 0x03FF, 0x0400, 0x7BFF)), _bits16(0x0001, 0x03FF, 0x0400, 0x7BFF))


def test_split_recovers_22_bits_and_the_scales_keep_weights_normal():
    rng = np.random.default_rng(1)
    x = (rng.standard_normal(200_000) * 10.0 ** rng.uniform(-4, 4.5, 200_000)).astype(np.float32).astype(np.float64)
    x = x[np.abs(x) < hr.F16_MAX]
    hi, lo = hr.split(x)
    err = np.abs(hi + lo * 2.0 ** -11 - x)
    assert np.all(err <= 2.0 ** -22 * np.abs(x) + 2.0 ** -36)
    for scale in (1e-30, 1e-3, 1.0, 1e3, 1e30):
        w = (rng.standard_normal((50, 33)) * scale).astype(np.float32)
        w_hi, w_d, w_lo, s = hr.split_weights(w)
        m = np.abs(np.ldexp(w.astype(np.float64), s[:, None])).max(1)
        assert np.all((m >= 2.0 ** 13) & (m < 2.0 ** 14)), scale
        big = np.abs(w_hi) >= 2.0 ** 3                      # W_hi 2^-11 normal from |W_hi| >= 2^-3; the top entries are
        assert np.all(w_d[big] == w_hi[big] * 2.0 ** -11)   # exact
        wp = np.ldexp(w.astype(np.float64), s[:, None])
        assert np.all(np.abs(w_hi + w_lo - wp) <= 2.0 ** -22 * np.abs(wp) + 2.0 ** -25)


def _trunc16(x):
    """Round toward zero to fp16 (the slip the rounding must not make)."""
    x = np.asarray(x, dtype=np.float64)
    r = hr.fp16(x)
    return np.where(np.abs(r) > np.abs(x), np.nextafter(r.astype(np.float16), np.float16(0)).astype(np.float64), r)


def emulate(rows, net, rnd=hr.fp16, passes=("hh", "ld", "hl")):
    """The kernel in NumPy fp32 (BLAS accumulation order): scaled fp16 weight halves, fp16 operand halves, the passes
    ``hh`` = A_hi W_hi, ``ld`` = A_lo W_d, ``hl`` = A_hi W_lo; ``rnd`` for every fp16 rounding."""
    w1, b1, w2, b2, w3, b3 = (np.asarray(t, np.float32) for t in net)
    f = np.float32
    a = np.asarray(rows, np.float32)
    for w, b in ((w1, b1), (w2, b2)):
        w_aug = np.concatenate([w, b[:, None]], axis=1)
        s = hr.row_scales(w_aug)
        wp = np.ldexp(w_aug, s[:, None].astype(np.int32)).astype(np.float32)
        w_hi = rnd(wp).astype(f)
        w_d, w_lo = rnd(w_hi * f(2.0 ** -11)).astype(f), rnd(wp - w_hi).astype(f)
        x = np.concatenate([a, np.ones((a.shape[0], 1), f)], axis=1)
        a_hi = rnd(x).astype(f)
        a_lo = rnd((x - a_hi) * f(2048.0)).astype(f)
        z = np.zeros((x.shape[0], w.shape[0]), f)
        for name, (p, q) in (("hh", (a_hi, w_hi)), ("ld", (a_lo, w_d)), ("hl", (a_hi, w_lo))):
            if name in passes:
                z = z + p @ q.T
        a = np.maximum(z * np.ldexp(f(1.0), -s.astype(np.int32)).astype(f)[None, :], f(0))
    l = a @ w3.T + b3
    e = np.exp(l - l.max(1, keepdims=True))
    return (e[:, 1] / (e[:, 0] + e[:, 1])).astype(np.float64)


SHAPES = [(10, 100, 100), (11, 100, 100), (23, 128, 112), (50, 100, 100), (64, 128, 128), (23, 1, 128), (10, 1, 1)]


@pytest.mark.parametrize("d,h1,h2", SHAPES)
def test_bound_and_fp32_grade_hold_for_the_emulation(d, h1, h2):
    rng = np.random.default_rng(d * 1000 + h1 + h2)
    net = ar.sample_net(rng, d, h1, h2)
    rows = ar.sample_rows(rng, 2048, d, net)
    for rows_k in (rows, ar.bf16(rows)):
        p, bound, info = hr.forward(rows_k, *net)
        assert info["in_range"].all() and not info["out_of_range"].any()
        got = emulate(rows_k, net)
        assert np.all(np.abs(got - p) <= bound)
        assert bound.max() <= 1e-3
        tol = hr.fp32_grade_tolerance(rows_k, *net)
        assert np.abs(got - ar.forward64(rows_k, *net)).max() <= 0.25 * tol


@pytest.mark.parametrize("d,h1,h2", [(11, 100, 100), (23, 128, 112), (50, 100, 100), (64, 128, 128)])
def test_fp32_grade_tolerance_separates_three_passes_from_fewer(d, h1, h2):
    rng = np.random.default_rng(d * 7 + h1)
    net = ar.sample_net(rng, d, h1, h2)
    rows = ar.sample_rows(rng, 900, d, net)
    tol = hr.fp32_grade_tolerance(rows, *net)
    p64 = ar.forward64(rows, *net)
    err = lambda **kw: float(np.abs(emulate(rows, net, **kw) - p64).max())   # noqa: E731
    assert err() <= 0.25 * tol
    for passes in (("hh",), ("hh", "ld"), ("hh", "hl")):
        assert err(passes=passes) > 4 * tol, passes
    # truncating instead of rounding is NOT visible here: the lo half absorbs the larger hi error (x - A_hi stays exact)
    # and the product still carries ~21 bits.  The rounding is pinned bit for bit by the helper test above instead.
    assert err(rnd=_trunc16) <= tol
    assert not np.array_equal(_trunc16(rows), hr.fp16(rows))


def _study_case(weight_scale, row_scale):
    """The CPU study's network (D = 50, 100 x 100, weights x 3) and rows, optionally rescaled."""
    rng = np.random.default_rng(0)
    net = list(ar.sample_net(rng, 50, 100, 100))
    net = [(t * np.float32(3.0 * weight_scale)).astype(np.float32) if i % 2 == 0 else t for i, t in enumerate(net)]
    x = rng.normal(0, 1, (4000, 50)).astype(np.float32) * np.array([1, 1, 4, 1, 3, 3, .5, 1, 1, 1] * 5, dtype=np.float32)
    return (x * np.float32(row_scale)).astype(np.float32), net


@pytest.mark.parametrize("weight_scale,row_scale", [(1.0, 1.0), (0.1, 10.0), (1e-4, 1.0), (30.0, 1.0)])
def test_small_and_large_weights(weight_scale, row_scale):
    """Ten times smaller weights with ten times larger rows (the study's subnormal case), tiny weights (1e-4: the
    unscaled W_hi 2^-11 would lie far below the fp16 normal range) and large ones: still fp32-grade."""
    rows, net = _study_case(weight_scale, row_scale)
    p, bound, info = hr.forward(rows, *net)
    assert info["in_range"].all()
    got = emulate(rows, net)
    assert np.all(np.abs(got - p) <= bound)
    tol = hr.fp32_grade_tolerance(rows, *net)
    assert np.abs(got - ar.forward64(rows, *net)).max() <= tol


def test_range_classification():
    rng = np.random.default_rng(9)
    net = ar.sample_net(rng, 11, 32, 32)
    rows = ar.sample_rows(rng, 6, 11).astype(np.float32)
    rows[1, 3] = 65504.0             # the largest fp16 value: in range
    rows[2, 0] = -70000.0            # an observation element beyond it
    rows[3, :] = 60000.0             # in range itself, but hidden activations of ~1e5 (w1 ~ N(0, 1 / 11))
    _, _, info = hr.forward(rows, *net)
    assert info["in_range"][[0, 1, 4, 5]].all() and not info["out_of_range"][[0, 1, 4, 5]].any()
    assert info["out_of_range"][2] and info["out_of_range"][3]
