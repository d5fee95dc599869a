"""Operand-exact reference of the tcgen05 actor kernels -- TEST INFRASTRUCTURE (see oracle/__init__.py).

``forward`` evaluates the MA-PPO actor (Linear-ReLU-Linear-ReLU-Linear-softmax) in fp64 NumPy the way each kernel of
``csrc/drsim_actor.cuh`` does it, operand roundings included, and carries beside every value a radius: a bound, derived
from first principles below, on how far the kernel's fp32 value can lie from the reference value.  The result is the
probability of action 1 per row and a per-row bound on ``|p_kernel - p_ref|``.

``k_actor2`` ("tf32", one pass): rows, weights and biases are rounded to TF32 (the biases ride in the GEMM as an extra K
column); after each ReLU the activation is rounded to TF32 in tensor memory; the output layer is a TF32 GEMM too;
softmax with ``__expf`` and ``p1 = 1 - p0``.

``k_actor3x`` ("tf32x3"): every GEMM operand is split as ``hi = tf32(x)``, ``lo = tf32(x - hi)`` and the products are
accumulated as ``A_hi W_hi + A_lo W_hi + A_hi W_lo`` (layers 1 and 2, bias again in the GEMM); ReLU on fp32 activations;
the output layer in fp32 FMAs on plain fp32 ``w3``, ``b3``; softmax with ``expf`` and ``p1 = e1 / (e0 + e1)``.

bfloat16 rows are the fp32 build's rows rounded to bf16 (``bf16``): such a value is exact in TF32, its lo half is zero.

Radius rules (``r`` bounds ``|kernel - reference|`` of one element):

* a product of two TF32 values (11 significant bits each) is exact in fp32 and in fp64;
* accumulating K products (any order, any fp32 rounding or truncation: at most one fp32 ulp = ``2^-23`` of the running
  magnitude per add) adds at most ``K * 2^-23 * sum |a w|`` -- the tensor core's accumulation is not documented, so
  nothing tighter is assumed; the fp64 sums of the reference add ``K * 2^-52 * sum |a w|``;
* an operand off by ``r`` moves a dot product by at most ``r |w|``;
* ReLU does not grow the radius (it is 1-Lipschitz);
* rounding to TF32: where the interval ``[v - r, v + r]`` holds no rounding boundary, kernel and reference round to the
  same TF32 value (rounding is monotone) and the radius drops to 0; where it holds one, it grows by one TF32 ulp;
* the hi / lo split: with ``x = hi + lo + e``, ``|e| <= 2^-22 |x|`` and ``|lo| <= 2^-11 |x|`` (same for ``w``), the split
  product ``A_hi W_hi + A_lo W_hi + A_hi W_lo`` differs from ``x w`` by ``lo_x lo_w + (hi_x + lo_x) e_w + e_x w``, at most
  ``3 * 2^-22 |x w|`` (plus a 2^-44 term); kernel (operand off by ``r``) and reference both carry that error, so one
  split product moves by at most ``|w| (r (1 + 2^-20) + 1.5 * 2^-20 (|v| + r))``, charged as
  ``|w| (r (1 + 2^-19) + 2^-19 |v|)``;
* softmax: the logit difference ``d = l1 - l0`` off by ``r0 + r1`` moves ``sigmoid(d)`` by at most its change over that
  interval; evaluating it in fp32 adds ``2^-21 + p (1 - p) (1.25 |d| + 8) 2^-23`` (``__expf`` is accurate to
  ``2 + 1.17 |x|`` ulp, ``expf`` to 2 ulp, the division and ``1 - p0`` round once each).
"""
from __future__ import annotations

import numpy as np

EPS32 = 2.0 ** -23      # one fp32 ulp relative to the magnitude it is taken at (upper bound)
EPS64 = 2.0 ** -52
KERNELS = ("tf32", "tf32x3")


def tf32(x):
    """The kernels' ``to_tf32``: round to the 10-bit TF32 mantissa, ties away from zero, ``(bits + 0x1000) & 0xffffe000``
    on the fp32 pattern.  fp32 input -> fp32 result (bit-exact with the device).  fp64 input -> fp64 result by the same
    rule at fp64 width (``(bits + 2^41) & ~(2^42 - 1)``), which equals the fp32 rule on every finite fp32 value and
    rounds the reference's fp64 intermediates without a detour through fp32."""
    x = np.asarray(x)
    if x.dtype == np.float32:
        b = x.view(np.uint32)
        return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)
    x = np.asarray(x, dtype=np.float64)
    b = x.view(np.uint64)
    return ((b + np.uint64(1 << 41)) & np.uint64(~((1 << 42) - 1) & 0xFFFFFFFFFFFFFFFF)).view(np.float64)


def split(x):
    """``hi = tf32(x)``, ``lo = tf32(x - hi)`` (the subtraction is exact in the input's precision)."""
    hi = tf32(x)
    return hi, tf32(x - hi)


def bf16(x):
    """fp32 -> bfloat16, round to nearest even (what the fp32 build stores in bf16 rows), returned as fp32."""
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    r = (b + np.uint32(0x7FFF) + ((b >> np.uint32(16)) & np.uint32(1))) & np.uint32(0xFFFF0000)
    return r.view(np.float32)


def _tf32_ulp(m):
    """One TF32 ulp at magnitude ``m`` (> 0): 2^(floor(log2 m) - 10)."""
    return np.ldexp(1.0, np.frexp(m)[1] - 11)


def _round_tf32(v, r):
    """TF32 rounding of an fp32 value known to lie in ``[v - r, v + r]`` (v >= 0 after ReLU): reference value and
    radius of the rounded value."""
    rv = tf32(v)
    lo, hi = np.maximum(v - r, 0.0), v + r
    crosses = tf32(lo) != tf32(hi)
    return rv, np.where(crosses, r + _tf32_ulp(np.maximum(hi, 1e-300)), 0.0)


def _dot(a, ra, w, b, n_terms):
    """``a @ w.T + b`` with operand radius ``ra`` (per element of ``a``; ``w``, ``b`` exact): value and radius after
    accumulating ``n_terms`` products per output in fp32."""
    aw = np.abs(w)
    v = a @ w.T + b
    mag = (np.abs(a) + ra) @ aw.T + np.abs(b)
    return v, ra @ aw.T + n_terms * (EPS32 + EPS64) * mag


def _dot3x(a, ra, w, b):
    """Layer of ``k_actor3x``: ``A_hi W_hi + A_lo W_hi + A_hi W_lo`` with the bias as the K column of a constant one."""
    a_hi, a_lo = split(a)
    w_hi, w_lo = split(w)
    b_hi, b_lo = split(b)
    v = a_hi @ w_hi.T + a_lo @ w_hi.T + a_hi @ w_lo.T + (b_hi + b_lo)
    rho = np.where(ra > 0, ra * (1 + 2.0 ** -19) + 2.0 ** -19 * np.abs(a), 0.0)   # split-product deviation per |w|
    aw = np.abs(w)
    n_terms = 3 * (a.shape[1] + 1)
    mag = ((np.abs(a) + ra + rho) @ aw.T + np.abs(b)) * (1 + 2.0 ** -9)
    return v, rho @ aw.T + n_terms * (EPS32 + EPS64) * mag


def _relu(v, r):
    return np.maximum(v, 0.0), np.where(v + r < 0, 0.0, r)


def _sigmoid(d):
    return 0.5 * (1.0 + np.tanh(0.5 * d))


def forward(rows, w1, b1, w2, b2, w3, b3, kernel: str = "tf32x3"):
    """Probability of action 1 (``prob_on``) per row and the bound on ``|p_kernel - p_ref|``, both fp64 ``[M]``.

    ``rows`` ``[M, D]``: the values the kernel reads (bf16 rows: their exact values, see ``bf16``); weights in
    ``torch.nn.Linear`` layout, any float dtype holding fp32 values.  Returns ``(p_on, bound, info)``; ``info`` holds the
    logits and their radii."""
    if kernel not in KERNELS:
        raise ValueError(f"kernel must be one of {KERNELS}")
    f32 = lambda t: np.asarray(t, dtype=np.float32)   # noqa: E731
    x = f32(rows)
    w1, b1, w2, b2, w3, b3 = (f32(t) for t in (w1, b1, w2, b2, w3, b3))
    h2 = w2.shape[0]
    if kernel == "tf32":
        t = lambda q: tf32(q).astype(np.float64)   # noqa: E731
        a, ra = t(x), np.zeros(x.shape)
        v, r = _dot(a, ra, t(w1), t(b1), x.shape[1] + 1)
        a, ra = _round_tf32(*_relu(v, r))
        v, r = _dot(a, ra, t(w2), t(b2), w1.shape[0] + 1)
        a, ra = _round_tf32(*_relu(v, r))
        l, rl = _dot(a, ra, t(w3), t(b3), h2 + 1)
    else:
        a, ra = x.astype(np.float64), np.zeros(x.shape)
        v, r = _dot3x(a, ra, w1.astype(np.float64), b1.astype(np.float64))
        a, ra = _relu(v, r)
        v, r = _dot3x(a, ra, w2.astype(np.float64), b2.astype(np.float64))
        a, ra = _relu(v, r)
        # fp32 FMA chains (two per logit) and one add: h2 + 1 roundings
        l, rl = _dot(a, ra, w3.astype(np.float64), b3.astype(np.float64), h2 + 2)
    d, rd = l[:, 1] - l[:, 0], rl[:, 0] + rl[:, 1]
    p = _sigmoid(d)
    move = np.maximum(_sigmoid(d + rd) - p, p - _sigmoid(d - rd))
    dn = np.sign(d) * np.maximum(np.abs(d) - rd, 0.0)      # the point of the interval nearest 0: largest p (1 - p)
    pn = _sigmoid(dn)
    softmax = 2.0 ** -21 + pn * (1.0 - pn) * (1.25 * (np.abs(d) + rd) + 8.0) * EPS32
    return p, move + softmax, {"logits": l, "logit_radius": rl}


def forward64(rows, w1, b1, w2, b2, w3, b3):
    """Probability of action 1 of a plain fp64 forward on the fp32 values of rows and weights (no TF32 anywhere)."""
    x, w1, b1, w2, b2, w3, b3 = (np.asarray(t, dtype=np.float32).astype(np.float64) for t in (rows, w1, b1, w2, b2, w3, b3))
    a = np.maximum(x @ w1.T + b1, 0.0)
    a = np.maximum(a @ w2.T + b2, 0.0)
    l = a @ w3.T + b3
    return _sigmoid(l[:, 1] - l[:, 0])


def forward32(rows, w1, b1, w2, b2, w3, b3):
    """The same forward in plain fp32 (NumPy / BLAS accumulation, fp32 softmax)."""
    x, w1, b1, w2, b2, w3, b3 = (np.asarray(t, dtype=np.float32) for t in (rows, w1, b1, w2, b2, w3, b3))
    a = np.maximum(x @ w1.T + b1, np.float32(0))
    a = np.maximum(a @ w2.T + b2, np.float32(0))
    l = a @ w3.T + b3
    e = np.exp(l - l.max(1, keepdims=True))
    return (e[:, 1] / (e[:, 0] + e[:, 1])).astype(np.float64)


def fp32_grade_tolerance(rows, *net):
    """What ``k_actor3x`` promises beyond the operand-exact bound: fp32-grade probabilities, within
    ``2e-6 + 2 max |p_fp32 - p_fp64|`` of the plain fp64 forward on the same rows (the rule of the torch comparison in
    test_gpu_batched).  The first-principles bound of ``forward`` charges every accumulation its worst case and is too
    wide to tell three TF32 passes from one; this tolerance is not, since a single pass is ~2^-11 off per product."""
    return 2e-6 + 2.0 * float(np.abs(forward32(rows, *net) - forward64(rows, *net)).max())


def sample_rows(rng, m: int, d: int, net=None):
    """fp32 rows ``[m, d]`` that probe the operand handling: magnitudes spread over four decades with both signs, about
    10 % exact zeros and 10 % values exactly on a TF32 rounding tie (low 13 mantissa bits = 0x1000).  With ``net``
    (``sample_net``), up to 3 % of the rows are scaled by 2^8 (ties stay ties): those whose probabilities this
    saturates (``|l1 - l0| > 30``)."""
    x = (np.where(rng.random((m, d)) < 0.5, -1.0, 1.0) * 10.0 ** rng.uniform(-4.0, 0.0, (m, d))).astype(np.float32)
    x[rng.random((m, d)) < 0.1] = 0.0
    bits = x.view(np.uint32)
    tie = (rng.random((m, d)) < 0.1) & (x != 0)
    bits[tie] = (bits[tie] & np.uint32(0xFFFFE000)) | np.uint32(0x1000)
    if net is not None:
        pick = np.flatnonzero(rng.random(m) < 0.03)
        big = x[pick] * np.float32(256.0)
        logits = forward(big, *net)[2]["logits"]
        keep = np.abs(logits[:, 1] - logits[:, 0]) > 30
        x[pick[keep]] = big[keep]
    return x


def sample_net(rng, d: int, h1: int, h2: int, out_scale: float = 1.0):
    """fp32 weights ``(w1, b1, w2, b2, w3, b3)`` in ``torch.nn.Linear`` layout, scaled so that on ``sample_rows`` most
    probabilities fall in (0.01, 0.99) and a few rows saturate (``|l1 - l0| > 30``)."""
    def lin(fan_in, fan_out, gain):
        w = rng.standard_normal((fan_out, fan_in)) * gain / np.sqrt(fan_in)
        return w.astype(np.float32), (0.1 * rng.standard_normal(fan_out)).astype(np.float32)

    w1, b1 = lin(d, h1, 1.0)
    w2, b2 = lin(h1, h2, np.sqrt(2.0))
    w3, b3 = lin(h2, 2, out_scale)
    return w1, b1, w2, b2, w3, b3


def emulate_split_product(a, w):
    """``a * w`` the way ``k_actor3x`` forms one product from fp32 operands (hi.hi + lo.hi + hi.lo, exact products),
    in fp64: for the reference's own tests."""
    a_hi, a_lo = split(np.asarray(a, dtype=np.float32))
    w_hi, w_lo = split(np.asarray(w, dtype=np.float32))
    f = lambda q: q.astype(np.float64)   # noqa: E731
    return f(a_hi) * f(w_hi) + f(a_lo) * f(w_hi) + f(a_hi) * f(w_lo)
