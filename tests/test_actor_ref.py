"""The operand-exact actor reference (``oracle.actor_ref``) on its own, without a GPU: the TF32 bit rule, the 3xTF32
split, and its error bound against fp32 emulations of the two kernels -- which must stay inside the bound when they
round like the kernels and leave it when they truncate -- and the fp32-grade tolerance of the 3xTF32 kernel, which an
emulation with fewer than three passes per product must leave."""
import numpy as np
import pytest

from oracle import actor_ref as ar


def _bits(*words):
    return np.array(words, dtype=np.uint32).view(np.float32)


def test_tf32_edge_bit_patterns():
    cases = {
        0x3F800000: 0x3F800000,   # 1.0: already TF32
        0x3F800FFF: 0x3F800000,   # just below the tie: down
        0x3F801000: 0x3F802000,   # exactly on the tie: away from zero
        0x3F803000: 0x3F804000,   # tie above an odd mantissa: still away from zero (not to even)
        0xBF801000: 0xBF802000,   # negative tie: away from zero (magnitude up)
        0xBF800FFF: 0xBF800000,
        0x00000000: 0x00000000,   # +0
        0x80000000: 0x80000000,   # -0 keeps its sign
        0x3FFFF000: 0x40000000,   # the carry runs into the exponent: 2 - 2^-11 rounds to 2
        0x7F7FE000: 0x7F7FE000,   # largest finite TF32
        0x7F7FEFFF: 0x7F7FE000,   # the largest fp32 values that round to it
        0x7F7FF000: 0x7F800000,   # from here on the rule overflows to infinity (the kernels see finite operands)
    }
    got = ar.tf32(_bits(*cases)).view(np.uint32)
    assert [hex(int(g)) for g in got] == [hex(v) for v in cases.values()]
    assert ar.tf32(_bits(0x3F801000)).dtype == np.float32


def test_tf32_fp64_rule_equals_fp32_rule_on_fp32_values():
    rng = np.random.default_rng(0)
    bits = rng.integers(0, 2 ** 32, 200_000, dtype=np.uint64).astype(np.uint32)
    bits = bits[(bits & 0x7F800000) != 0x7F800000]                          # finite
    bits = bits[((bits & 0x7F800000) != 0) | ((bits & 0x7FFFFF) == 0)]        # no subnormals
    bits = bits[(bits & 0x7FFFFFFF) < 0x7F7FF000]                            # no overflow to infinity
    x = bits.view(np.float32)
    assert np.array_equal(ar.tf32(x).astype(np.float64), ar.tf32(x.astype(np.float64)))


def test_split_recovers_21_bits():
    """hi.hi + lo.hi + hi.lo of the split operands is within 2^-20 of the exact product (the dropped lo.lo term and the
    two lo roundings are 2^-22 each); one TF32 pass is ~2^-11 off."""
    rng = np.random.default_rng(1)
    a = (rng.standard_normal(100_000) * 10.0 ** rng.uniform(-3, 3, 100_000)).astype(np.float32)
    w = (rng.standard_normal(100_000) * 10.0 ** rng.uniform(-3, 3, 100_000)).astype(np.float32)
    exact = a.astype(np.float64) * w.astype(np.float64)
    rel3 = np.abs(ar.emulate_split_product(a, w) - exact) / np.abs(exact)
    rel1 = np.abs(ar.tf32(a).astype(np.float64) * ar.tf32(w).astype(np.float64) - exact) / np.abs(exact)
    assert rel3.max() <= 2.0 ** -20
    assert np.median(rel3) > 2.0 ** -30      # not exact: the lo halves carry real bits
    assert rel1.max() > 2.0 ** -12 and rel1.max() <= 2.0 ** -10


def test_bf16_is_round_to_nearest_even():
    x = _bits(0x3F808000, 0x3F818000, 0x3F808001, 0xBF817FFF, 0x00000000)
    assert [hex(int(v)) for v in ar.bf16(x).view(np.uint32)] == ["0x3f800000", "0x3f820000", "0x3f810000", "0xbf810000", "0x0"]
    assert np.array_equal(ar.tf32(ar.bf16(x)), ar.bf16(x))     # exact in TF32: the lo half of a bf16 row is zero


def _trunc(x):
    return (np.asarray(x, dtype=np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def _emulate(rows, net, kernel, rnd=ar.tf32, passes=("hh", "lh", "hl")):
    """The kernel in NumPy fp32 (BLAS accumulation order, ``rnd`` for every TF32 rounding); ``passes``: the split
    products ``k_actor3<SplitTf32x3>`` accumulates (hi.hi, lo.hi, hi.lo)."""
    w1, b1, w2, b2, w3, b3 = net
    if kernel == "tf32":
        a = rnd(rows)
        for w, b in ((w1, b1), (w2, b2)):
            a = rnd(np.maximum(a @ rnd(w).T + rnd(b), np.float32(0)))
        l = a @ rnd(w3).T + rnd(b3)
        e = np.exp(l - l.max(1, keepdims=True))
        return (np.float32(1) - e[:, 0] / (e[:, 0] + e[:, 1])).astype(np.float64)

    def split(x):
        hi = rnd(x)
        return hi, rnd(x - hi)

    a = rows
    for w, b in ((w1, b1), (w2, b2)):
        (ah, al), (wh, wl), (bh, bl) = split(a), split(w), split(b)
        z = bh + bl if "hl" in passes else bh                  # the bias column: A = 1, hi 1, lo 0
        for name, (x, y) in (("hh", (ah, wh)), ("lh", (al, wh)), ("hl", (ah, wl))):
            if name in passes:
                z = z + x @ y.T
        a = np.maximum(z, np.float32(0))
    l = a @ w3.T + b3
    e = np.exp(l - l.max(1, keepdims=True))
    return (e[:, 1] / (e[:, 0] + e[:, 1])).astype(np.float64)


@pytest.mark.parametrize("d,h1,h2", [(11, 100, 100), (64, 128, 112), (23, 1, 128), (10, 1, 1), (59, 128, 95)])
def test_bound_holds_for_fp32_emulation_and_catches_truncation(d, h1, h2):
    rng = np.random.default_rng(d * 1000 + h1 + h2)
    net = ar.sample_net(rng, d, h1, h2)
    rows = ar.sample_rows(rng, 4096, d, net)
    for rows_k in (rows, ar.bf16(rows)):
        for kernel in ar.KERNELS:
            p, bound, _ = ar.forward(rows_k, *net, kernel=kernel)
            assert np.all(np.abs(_emulate(rows_k, net, kernel) - p) <= bound), kernel
    # TF32 truncation instead of rounding (a one-character slip in ``to_tf32``) leaves the single-pass bound
    p, bound, _ = ar.forward(rows, *net, kernel="tf32")
    assert np.sum(np.abs(_emulate(rows, net, "tf32", _trunc) - p) > bound) >= 10


def test_sample_net_spreads_probabilities_and_saturates_some_rows():
    rng = np.random.default_rng(5)
    net = ar.sample_net(rng, 22, 100, 100)
    rows = ar.sample_rows(rng, 20_000, 22, net)
    p, bound, info = ar.forward(rows, *net)
    d = np.abs(info["logits"][:, 1] - info["logits"][:, 0])
    assert ((p > 0.01) & (p < 0.99)).mean() > 0.9
    assert 20 <= (d > 30).sum() <= 0.03 * len(d)
    assert (rows == 0).mean() > 0.05 and ((rows.view(np.uint32) & 0x1FFF) == 0x1000).mean() > 0.05


@pytest.mark.parametrize("d,h1,h2", [(11, 100, 100), (23, 128, 112), (47, 120, 127), (64, 100, 96), (23, 1, 128),
                                     (23, 127, 128), (59, 100, 100)])
def test_fp32_grade_tolerance_separates_three_passes_from_fewer(d, h1, h2):
    """The 3xTF32 kernel's second check: its emulation stays well inside ``fp32_grade_tolerance``; dropping both lo
    passes (a single TF32 pass) or either one of them leaves it, on fp32 and on bf16 rows."""
    rng = np.random.default_rng(d * 7 + h1)
    net = ar.sample_net(rng, d, h1, h2)
    rows = ar.sample_rows(rng, 900, d, net)
    for rows_k in (rows, ar.bf16(rows)):
        tol = ar.fp32_grade_tolerance(rows_k, *net)
        assert tol < 5e-6
        p64 = ar.forward64(rows_k, *net)
        err = lambda passes: float(np.abs(_emulate(rows_k, net, "tf32x3", passes=passes) - p64).max())   # noqa: E731
        assert err(("hh", "lh", "hl")) <= 0.25 * tol
        for passes in (("hh",), ("hh", "lh"), ("hh", "hl")):
            assert err(passes) > 4 * tol, passes
