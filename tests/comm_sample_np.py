"""NumPy restatement of the device's ``random_sample`` neighbour draw (TEST INFRASTRUCTURE).

``CommSampler`` (``drsim_device.cuh``, DRSIM_COMM_SAMPLE) is OUR definition: the reference draws ``random.sample``
from Python's Mersenne Twister.  This module restates it independently, on top of the Philox restatement of
``oracle.philox``, so the device and ``drsim_host_comm_sample`` can be checked bit for bit.

Purpose 7 (``PURPOSE_NEIGHBOUR``): counter (global replica, global house, draw, 7 | block << 8), four 32-bit words per
Philox block, block = step // 4.
"""
from __future__ import annotations

import numpy as np

from oracle.philox import philox4x32_10

PURPOSE_NEIGHBOUR = 7


def comm_sample(key: int, rep, house, draw: int, n_global: int, c: int):
    """``random.sample(ids without house, c)`` replacement of the device: a sparse partial Fisher-Yates shuffle of the
    ``M = n_global - 1`` other ids.  Step j draws ``r_j = j + mulhi(u_j, M - j)`` (Lemire's map without rejection,
    bias <= M / 2^32), swaps positions j and r_j of the identity array and outputs the value now at position j,
    mapped past the house itself.  ``rep`` / ``house`` broadcast (e.g. ``[R, 1]`` and ``[1, N]``); returns int64
    ``[..., c]`` global house ids."""
    rep, house = np.broadcast_arrays(np.asarray(rep, dtype=np.int64), np.asarray(house, dtype=np.int64))
    M = np.uint64(n_global - 1)
    pos = np.zeros(rep.shape + (c,), dtype=np.int64)
    held = np.zeros(rep.shape + (c,), dtype=np.int64)
    out = np.zeros(rep.shape + (c,), dtype=np.int64)
    words = None
    for j in range(c):
        if j % 4 == 0:
            words = philox4x32_10(key, rep, house, int(draw) & 0xFFFFFFFF, PURPOSE_NEIGHBOUR | ((j // 4) << 8))
        u = words[j % 4].astype(np.uint64)
        r = j + ((u * (M - np.uint64(j))) >> np.uint64(32)).astype(np.int64)
        v, hj = r.copy(), np.full(rep.shape, j, dtype=np.int64)
        for i in range(j):   # ascending: the last swap that wrote a position wins
            v = np.where(pos[..., i] == r, held[..., i], v)
            hj = np.where(pos[..., i] == j, held[..., i], hj)
        pos[..., j], held[..., j] = r, hj
        out[..., j] = v + (v >= house)
    return out


def comm_sample_table(key: int, n_rep: int, n_house: int, draw: int, c: int, rep_offset: int = 0):
    """The ``[R, N, c]`` table of one draw (``drsim_comm_sample``) for replicas ``rep_offset ..``."""
    return comm_sample(key, (rep_offset + np.arange(n_rep))[:, None], np.arange(n_house)[None, :], draw, n_house, c)
