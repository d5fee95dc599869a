"""Operand-exact reference of the "f16x3" actor (``k_actor3<SplitF16x3>`` of ``csrc/drsim_actor.cuh``) -- test infrastructure, in the
manner of ``oracle/actor_ref.py`` (whose ``KERNELS`` / ``forward`` cover "tf32" and "tf32x3"; the rules below extend its
radius rules to the fp16 split).

The kernel, operand for operand (layers 1 and 2; ``[a | 1]`` and ``[W | b]`` are the operands with the bias column):

* per output neuron n a power-of-two scale ``2^s_n``: ``m_n = max_k |W[n, k]|`` (bias included), ``m_n = f 2^e`` with
  ``f`` in [0.5, 1), ``s_n = min(14 - e, 126)`` (``s_n = 0`` for an all-zero row); ``W' = fp32(W 2^s_n)``;
* ``W_hi = fp16(W')``, ``W_d = fp16(W_hi 2^-11)``, ``W_lo = fp16(W' - W_hi)``; ``A_hi = fp16(x)``,
  ``A_lo = fp16((x - A_hi) 2^11)`` (fp16: round to nearest even, subnormals, overflow to infinity from 65520 on);
* ``D' = A_hi W_hi + A_lo W_d + A_hi W_lo`` accumulated in fp32; layer 1: ``a1 = relu(D' 2^-s)`` (producers); layer 2:
  ``relu(D')`` times ``fp32(w3 2^-s)`` (consumers) -- the same fp32 product as ``relu(D' 2^-s) w3``;
* output layer in fp32 FMAs, softmax with ``expf``, ``p1 = e1 / (e0 + e1)`` (as ``k_actor3<SplitTf32x3>``);
* range: a live row whose observation elements or hidden activations reach ``|x| >= 65520`` sets the handle's flag.

Radius rules beyond ``oracle/actor_ref.py``: with ``u = 2^-11`` and normal fp16 halves, ``x = A_hi + A_lo u + e_a`` with
``|e_a| <= u^2 |x|``, ``W' = W_hi + W_lo + e_w`` with ``|e_w| <= u^2 |W'|``, ``W_d = W_hi u + d_w``.  The split product
differs from ``x W'`` by ``-x e_w - (x - A_hi) W_lo - e_a W_hi + A_lo d_w``: at most ``3 u^2 |x W'|`` (plus ``2^-44``
terms), and where fp16 subnormals enter, ``|d_w| <= 2^-25`` and ``|A_lo| <= |x|`` add ``2^-25 |x|``, ``e_w`` and ``e_a``
at most ``2^-25`` resp. ``2^-36`` absolute.  In unscaled units (divide by ``2^s``) one product is off by at most
``|x| (3 u^2 |w| + 2^-24 2^-s) + 2^-35 |w|``; the kernel's operand (off by ``r``) and the reference's both carry that
error, so a product with an inexact operand moves by at most ``r |w| + (2 |x| + r) (3 u^2 |w| + 2^-24 2^-s) + 2^-34 |w|``.
"""
from __future__ import annotations

import numpy as np

from oracle import actor_ref as ar

F16_MAX = 65504.0
F16_OVERFLOW = 65520.0   # |x| from which round-to-nearest-even gives infinity


def fp16(x):
    """Round to IEEE fp16, nearest even, with subnormals and overflow to +-inf; fp64 result.  One rounding of the exact
    input value (fp32 or fp64)."""
    x = np.asarray(x, dtype=np.float64)
    ax = np.abs(x)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        e = np.floor(np.log2(np.where(ax > 0, ax, 1.0)))
        # log2 can be off by one next to a power of two: correct e so that 2^e <= ax < 2^(e + 1)
        e = np.where(np.ldexp(1.0, e.astype(np.int64)) > ax, e - 1, e)
        e = np.where(np.ldexp(1.0, (e + 1).astype(np.int64)) <= ax, e + 1, e)
        q = np.ldexp(1.0, (np.maximum(e, -14) - 10).astype(np.int64))   # fp16 spacing at ax (subnormal: 2^-24)
        r = np.rint(ax / q) * q                                        # np.rint: ties to even; ax / q is exact
    r = np.where(ax >= F16_OVERFLOW, np.inf, np.where(ax > 0, r, 0.0))
    return np.copysign(r, x)


def split(x):
    """``(A_hi, A_lo)`` of the kernel: ``hi = fp16(x)``, ``lo = fp16((x - hi) 2^11)`` (the difference is exact)."""
    hi = fp16(x)
    with np.errstate(invalid="ignore"):
        return hi, fp16((np.asarray(x, dtype=np.float64) - hi) * 2048.0)


def row_scales(w_aug):
    """``s_n`` per row of the augmented fp32 weights ``[W | b]`` (bias column included)."""
    m = np.abs(np.asarray(w_aug, dtype=np.float64)).max(axis=1)
    e = np.frexp(m)[1]
    return np.where(m > 0, np.minimum(14 - e, 126), 0).astype(np.int64)


def split_weights(w_aug):
    """``(W_hi, W_d, W_lo, s)`` of the kernel's image for the augmented fp32 weights ``[n_out, K]``."""
    w_aug = np.asarray(w_aug, dtype=np.float32)
    s = row_scales(w_aug)
    wp = np.ldexp(w_aug, s[:, None].astype(np.int32)).astype(np.float64)   # fp32 product by 2^s, rounded as on the device
    wp = wp.astype(np.float32).astype(np.float64)
    hi = fp16(wp)
    return hi, fp16(hi * 2.0 ** -11), fp16(wp - hi), s


def _layer(a, ra, w, b):
    """One tensor-core layer of ``k_actor3<SplitF16x3>``: value (unscaled, before ReLU) and radius.  ``a`` fp64 ``[M, K]`` with
    radius ``ra``; ``w``, ``b`` fp32."""
    w_aug = np.concatenate([np.asarray(w, np.float32), np.asarray(b, np.float32)[:, None]], axis=1)
    w_hi, w_d, w_lo, s = split_weights(w_aug)
    down = np.ldexp(1.0, -s)
    a_aug = np.concatenate([a, np.ones((a.shape[0], 1))], axis=1)
    ra_aug = np.concatenate([ra, np.zeros((a.shape[0], 1))], axis=1)
    a_hi, a_lo = split(a_aug)
    with np.errstate(invalid="ignore", over="ignore"):
        v = (a_hi @ w_hi.T + a_lo @ w_d.T + a_hi @ w_lo.T) * down[None, :]
    aw = np.abs(w_aug.astype(np.float64))
    inexact = ra_aug > 0
    t = np.where(inexact, 2.0 * np.abs(a_aug) + ra_aug, 0.0)
    rho = (ra_aug @ aw.T + (3.0 * 2.0 ** -22) * (t @ aw.T) + 2.0 ** -24 * t.sum(1)[:, None] * down[None, :]
           + 2.0 ** -34 * (inexact.astype(np.float64) @ aw.T))
    # fp32 accumulation of 3 K products: each split product is at most |a w| (1 + 2^-9) + |a| 2^-24 2^-s (+ 2^-35 |w|)
    mag = (((np.abs(a_aug) + ra_aug) @ aw.T) * (1 + 2.0 ** -9) + 2.0 ** -24 * (np.abs(a_aug) + ra_aug).sum(1)[:, None]
           * down[None, :] + 2.0 ** -35 * aw.sum(1)[None, :])
    n_terms = 3 * a_aug.shape[1]
    return v, rho + n_terms * (ar.EPS32 + ar.EPS64) * mag + mag * 2.0 ** -40


def forward(rows, w1, b1, w2, b2, w3, b3):
    """``(p_on, bound, info)`` as ``oracle.actor_ref.forward`` for "f16x3", plus in ``info``: ``in_range`` (every
    operand of the row surely below 65520 in the kernel: the row's result is valid and within ``bound``) and
    ``out_of_range`` (some operand surely at or above it: the kernel sets the flag)."""
    f32 = lambda t: np.asarray(t, dtype=np.float32)   # noqa: E731
    x = f32(rows).astype(np.float64)
    w1, b1, w2, b2, w3, b3 = (f32(t) for t in (w1, b1, w2, b2, w3, b3))
    h2 = w2.shape[0]
    amax_lo = np.abs(x).max(axis=1)
    amax_hi = amax_lo.copy()
    a, ra = x, np.zeros(x.shape)
    for w, b in ((w1, b1), (w2, b2)):
        v, r = _layer(a, ra, w, b)
        a, ra = ar._relu(v, r)
        if w is w1:   # the hidden activations of layer 1 are layer 2's operand
            amax_lo = np.fmax(amax_lo, np.fmax.reduce(np.maximum(a - ra, 0.0), axis=1))
            amax_hi = np.fmax(amax_hi, np.max(a + ra, axis=1))
    l, rl = ar._dot(a, ra, w3.astype(np.float64), b3.astype(np.float64), h2 + 2)
    d, rd = l[:, 1] - l[:, 0], rl[:, 0] + rl[:, 1]
    with np.errstate(invalid="ignore"):
        p = ar._sigmoid(d)
        move = np.maximum(ar._sigmoid(d + rd) - p, p - ar._sigmoid(d - rd))
        dn = np.sign(d) * np.maximum(np.abs(d) - rd, 0.0)
        pn = ar._sigmoid(dn)
        softmax = 2.0 ** -21 + pn * (1.0 - pn) * (1.25 * (np.abs(d) + rd) + 8.0) * ar.EPS32
    info = {"logits": l, "logit_radius": rl, "in_range": amax_hi < F16_OVERFLOW, "out_of_range": amax_lo >= F16_OVERFLOW}
    return p, move + softmax, info


def fp32_grade_tolerance(rows, *net):
    """The fp32-grade promise of "f16x3", the same as that of "tf32x3" (``oracle.actor_ref.fp32_grade_tolerance``)."""
    return ar.fp32_grade_tolerance(rows, *net)
