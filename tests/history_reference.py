"""Float64 statement of the FarmerLstm step on variable-length move histories (fi_learner_config.history_length, record word
183, include/fi_learner.h), for the tests of that option.

Slot b of an [m, T] batch is one sample whose history is its first L_b = (W == 0 || W > T) ? T : W records, W being word 183
of its record 0. Its value is the reference model on z[b, :L_b]: the LSTM over those steps, h_{L_b-1} ‖ x -> dense stack -> y.
The loss is the usual mean over the m samples, so the step is the C oracle's loss_grad run on each group of samples with equal
L, cut to T = L, with loss_denom = m, summed. orc_farmer_loss_grad zeroes its gradient on every call, so the sum is taken
here. Nothing past L_b is read: z is sliced before any arithmetic.

tests/test_history_length.py holds this module to torch float64 autograd of nn.LSTM on pack_padded_sequence.
"""
from __future__ import annotations

import numpy as np

import _util as U
import length_reference as LR
from oracle import pyoracle as po

WORD = LR.WORD
lengths_of = LR.lengths_of
X_RECS = 8   # x[484] spans words 192..255 of records 0..7


def loss_grad_history(o, z, x, target, lengths, loss_denom=None):
    """(loss, grads) of the OracleFarmer `o` at its current parameters on histories z[b, :lengths[b]]; loss_denom defaults
    to m (the mean over the whole batch)."""
    z, x, target = np.asarray(z, np.float32), np.asarray(x, np.float32), np.asarray(target, np.float32)
    m, t = z.shape[0], z.shape[1]
    L = np.asarray(lengths, np.int64)
    assert L.shape == (m,) and np.all((L >= 1) & (L <= t))
    denom = loss_denom or m
    total, grads = 0.0, None
    for n in np.unique(L):
        idx = np.flatnonzero(L == n)
        total += o.loss_grad(np.ascontiguousarray(z[idx, :n]), np.ascontiguousarray(x[idx]), np.ascontiguousarray(target[idx]),
                             loss_denom=denom)
        g = o.grads()
        grads = g if grads is None else grads + g
    return total, grads


def dense_preactivations(params, z, x, lengths):
    """The five hidden pre-activations [5, m, 512] in float64 at `params` with each history cut to its length (the ReLU
    decisions the float64 step makes)."""
    p, off, T = np.asarray(params, np.float64), 0, []
    for shp in U.FARMER_SHAPES:
        n = int(np.prod(shp))
        T.append(p[off:off + n].reshape(shp))
        off += n
    sig = lambda v: 1.0 / (1.0 + np.exp(-v))   # noqa: E731
    m, t = z.shape[0], z.shape[1]
    L = np.asarray(lengths)
    h, c, last = np.zeros((m, 128)), np.zeros((m, 128)), np.zeros((m, 128))
    for s in range(int(L.max())):
        g = z[:, s].astype(np.float64) @ T[0].T + T[2] + h @ T[1].T + T[3]
        c = sig(g[:, 128:256]) * c + sig(g[:, :128]) * np.tanh(g[:, 256:384])
        h = sig(g[:, 384:]) * np.tanh(c)
        last[L == s + 1] = h[L == s + 1]
    a, pre = np.concatenate([last, x.astype(np.float64)], axis=1), []
    for layer in range(5):
        pre.append(a @ T[4 + 2 * layer].T + T[5 + 2 * layer])
        a = np.maximum(pre[-1], 0.0)
    return np.stack(pre)


def pack_history_slots(z, x, target, words, pad=None) -> np.ndarray:
    """pyoracle.pack_farmer_slots with length words `words` [m] (uint32) in word 183 of record 0. pad: None leaves the region a
    history learner must not read as the packer wrote it (z of every record); "zeros" zeroes it; "garbage" fills it with NaN,
    +-inf, 1e30 and random bit patterns. That region is words 0..161 of records L..T-1 and every word of records
    max(L, 8)..T-1."""
    z = np.asarray(z, np.float32)
    m, t = z.shape[0], z.shape[1]
    L = lengths_of(words, t)
    slots = po.pack_farmer_slots(z, x, target)
    w = slots.view(np.uint32).reshape(m, t, po.REC_WORDS)
    if pad is not None:
        rec = np.arange(t)[None, :]
        z_past = rec >= L[:, None]                               # [m, t]: z words of these records
        all_past = rec >= np.maximum(L, X_RECS)[:, None]          # [m, t]: every word of these records
        mask = np.zeros(w.shape, bool)
        mask[..., :po.Z_DIM] = z_past[..., None]
        mask |= all_past[..., None]
        if pad == "zeros":
            w[mask] = 0
        elif pad == "garbage":
            n = int(mask.sum())
            rng = np.random.default_rng(n)
            g = rng.integers(0, 1 << 32, size=n, dtype=np.uint64).astype(np.uint32)
            special = np.array([np.nan, np.inf, -np.inf, 1e30, -1e30], np.float32).view(np.uint32)
            pick = rng.integers(0, 6, size=n)
            w[mask] = np.where(pick < 5, special[np.minimum(pick, 4)], g)
        else:
            raise ValueError(pad)
    w[:, 0, WORD] = np.asarray(words, np.uint32)
    return slots
