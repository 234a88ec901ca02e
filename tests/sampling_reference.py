"""Reference of the policy sampling rule of fi_learner_infer_sample / fi_op_policy_sample (include/fi_learner.h): the
Philox4x32-10 generator in numpy, the greedy rule, and the inverse-CDF pick in float64, for the tests of that call.

For row r: S = legal[r] & 0xFFFF, z = the row's 16 logits. The greedy action g is numpy's argmax over S (NaN counts as largest,
ties go to the lowest index). With greedy, or when z_g is not finite, the action is g. Otherwise u = (x0 >> 8) * 2^-24, x0 =
word 0 of Philox4x32-10 at counter (r, 0, 0, 0) with key (seed low, seed high), and the action is the smallest j in S whose
cumulative weight exceeds u times the total. The kernel does that last step in fp32; `sample` does it in float64 and reports
how close u came to a cumulative boundary, so a test can accept either neighbour where fp32 rounding may decide.
"""
from __future__ import annotations

import numpy as np

A = 16
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(counter, key):
    """Random123's Philox4x32-10. counter [..., 4], key [..., 2] (uint32, broadcast) -> [..., 4] uint32."""
    c = np.asarray(counter, np.uint64)
    k = np.asarray(key, np.uint64)
    c0, c1, c2, c3 = (c[..., i] for i in range(4))
    k0, k1 = k[..., 0], k[..., 1]
    for rnd in range(10):
        if rnd:
            k0 = (k0 + _W0) & _MASK
            k1 = (k1 + _W1) & _MASK
        p0, p1 = _M0 * c0, _M1 * c2     # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
    return np.stack([c0, c1, c2, c3], -1).astype(np.uint32)


def uniforms(rows, seed):
    """u for counters rows (int array): (word 0 >> 8) * 2^-24, exactly representable in fp32 and float64."""
    r = np.asarray(rows, np.uint64)
    ctr = np.zeros(r.shape + (4,), np.uint64)
    ctr[..., 0] = r
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], np.uint64)
    x0 = philox4x32_10(ctr, key)[..., 0]
    return (x0 >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


def supports(legal, rows):
    """[rows, 16] bool from the legal words (None = every action legal); bits 16..31 are ignored."""
    if legal is None:
        return np.ones((rows, A), bool)
    w = np.asarray(legal, np.uint32).astype(np.uint64)
    return ((w[:, None] >> np.arange(A, dtype=np.uint64)) & 1) == 1


def greedy_actions(z, sup):
    """idx[argmax(z[idx])] with idx = flatnonzero(S), per row (NaN largest, ties to the lowest index); -1 for an empty S."""
    z = np.asarray(z, np.float64)
    nan_in = sup & np.isnan(z)
    with np.errstate(invalid="ignore"):
        zm = np.where(sup & ~np.isnan(z), z, -np.inf)
        top = sup & (zm == zm.max(1, keepdims=True))
    g = np.where(nan_in.any(1), np.argmax(nan_in, 1), np.argmax(top, 1))
    return np.where(sup.any(1), g, -1)


def sample(z, legal=None, seed=0, greedy=False, rows=None):
    """The float64 statement of the rule. z [n, 16] logits (fp32 values), legal [n] words or None, rows [n] the RNG counters
    (default 0..n-1). Returns (actions [n] int64, alt [n] int64, gap [n] float64): alt is the other action in S that a u
    within rounding of a cumulative boundary could give (the next action of positive weight across the nearest boundary, -1
    if none), gap the distance of u from that boundary as a fraction of the total weight (inf where no draw is made)."""
    z = np.asarray(z, np.float32).astype(np.float64)
    n = len(z)
    sup = supports(legal, n)
    g = greedy_actions(z, sup)
    act, alt, gap = g.copy(), np.full(n, -1, np.int64), np.full(n, np.inf)
    if greedy:
        return act, alt, gap
    zg = np.take_along_axis(z, np.maximum(g, 0)[:, None], 1)[:, 0]
    draw = (g >= 0) & np.isfinite(zg)
    u = uniforms(np.arange(n) if rows is None else rows, seed)
    with np.errstate(invalid="ignore", over="ignore"):
        w = np.where(sup & draw[:, None], np.exp(np.where(sup, z, 0.0) - zg[:, None]), 0.0)
    tot = w.sum(1)
    tot[~draw] = 1.0
    c = np.cumsum(w, 1) / tot[:, None]
    pos = w > 0
    j = np.arange(A)
    above = (c > u[:, None]) & pos
    last = A - 1 - np.argmax(pos[:, ::-1], 1)
    k = np.where(above.any(1), np.argmax(above, 1), last)         # the smallest j in S with P_j > u W
    hi = np.take_along_axis(c, k[:, None], 1)[:, 0]
    lo = hi - np.take_along_axis(w, k[:, None], 1)[:, 0] / tot
    below_nb = pos & (j < k[:, None])
    above_nb = pos & (j > k[:, None])
    nb_lo = np.where(below_nb.any(1), A - 1 - np.argmax(below_nb[:, ::-1], 1), -1)
    nb_hi = np.where(above_nb.any(1), np.argmax(above_nb, 1), -1)
    near_lo = u - lo <= hi - u
    act = np.where(draw, k, act)
    alt = np.where(draw, np.where(near_lo, nb_lo, nb_hi), -1)
    gap = np.where(draw, np.where(near_lo, u - lo, hi - u), np.inf)
    return act, alt, gap


def masked_softmax(z, sup):
    """float64 softmax of one row over its support (0 outside)."""
    z = np.where(sup, np.asarray(z, np.float64), -np.inf)
    e = np.exp(z - z.max())
    return e / e.sum()
