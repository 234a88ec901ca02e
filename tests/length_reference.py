"""Float64 reference of the V-trace loss and actor-critic step on variable-length trajectories (fi_learner_config.variable_length,
record word 183, include/fi_learner.h), for the tests of that option.

Trajectory b of a [m, t] batch holds L_b = (W == 0 || W > t) ? t : W valid steps, W being word 183 of its record 0. The step
is the step on the trajectories cut to their first L_b records: the bootstrap is word 181 of record L_b - 1, the losses sum
over valid steps only, and the rows past L_b have zero observations (they still run through the network) and a zero
d(head). Nothing past L_b is read here either: the functions slice it away before any arithmetic.

The loss of each trajectory is the C oracle's own (orc_vtrace_losses) on its first L_b steps, or, with legal-action words,
tests/legal_reference.py's masked loss on them; the actor-critic forward / backward around it is float64 numpy, as in
legal_reference.ac_loss_grad_legal. tests/test_variable_length.py holds this module to torch float64 autograd and to the
C oracle run on the truncated trajectories.
"""
from __future__ import annotations

import numpy as np

import legal_reference as LR
from oracle import pyoracle as po

A = po.NUM_ACTIONS
HID, ZD = LR.HID, LR.ZD
WORD = 183


def lengths_of(words, t):
    """[m] valid steps per trajectory from the length words W (uint32): W when 1 <= W <= t, else t."""
    w = np.asarray(words, np.uint32).astype(np.int64)
    return np.where((w == 0) | (w > t), t, w)


def valid_rows(lengths, t):
    """[m, t] bool: step s of trajectory b is valid (s < L_b)."""
    return np.arange(t)[None, :] < np.asarray(lengths)[:, None]


def vtrace_losses_length(oracle, logits, value, mu_logits, action, reward, discount, bootstrap, legal, lengths, **cfg):
    """Oracle.vtrace_losses (legal None) or legal_reference.vtrace_losses_legal per trajectory on its first L_b steps;
    bootstrap [m] is the value in word 181 of record L_b - 1. Losses sum over the trajectories in order; dlogits, dvalue, vs
    and pg_adv are [m, t(, A)] with exact zeros past L_b."""
    m, t = np.asarray(action).shape
    L = np.asarray(lengths, np.int64)
    assert L.shape == (m,) and np.all((L >= 1) & (L <= t))
    out = dict(losses=np.zeros(4), dlogits=np.zeros((m, t, A)), dvalue=np.zeros((m, t)), vs=np.zeros((m, t)),
               pg_adv=np.zeros((m, t)))
    for b in range(m):
        n = int(L[b])
        cut = lambda x: np.ascontiguousarray(np.asarray(x)[b:b + 1, :n])   # noqa: E731
        args = (cut(logits), cut(value), cut(mu_logits), cut(action), cut(reward), cut(discount),
                np.asarray(bootstrap)[b:b + 1])
        r = (oracle.vtrace_losses(*args, **cfg) if legal is None else
             LR.vtrace_losses_legal(oracle, *args, cut(legal), **cfg))
        out["losses"] += r["losses"]
        for k in ("dlogits", "dvalue", "vs", "pg_adv"):
            out[k][b, :n] = r[k][0]
    return out


def ac_loss_grad_length(oracle, params, obs, mu, act, rew, disc, boot, legal, lengths, relu_mask=None, **cfg):
    """The actor-critic step's loss and gradient over the flat parameter arena at `params`, in float64, with per-trajectory
    lengths: legal_reference.ac_loss_grad_legal with zero observations past L_b and vtrace_losses_length as the loss (legal
    None = every action legal, the oracle's own loss). relu_mask ([5, rows*512] uint8, the CUDA run's decisions over every
    row, padding included) pins the ReLU units. Returns (losses[4], grads[AC_PARAMS], units overridden, largest |z|/rms
    among them)."""
    m, t = np.asarray(act).shape
    rows = m * t
    W = LR._tensors(np.asarray(params, np.float64))
    keep = valid_rows(lengths, t).reshape(rows, 1)
    x = np.where(keep, np.asarray(obs, np.float32).reshape(rows, ZD).astype(np.float64), 0.0)
    ins, gates = [x], []
    n_over, max_over = 0, 0.0
    for li in range(5):
        z = ins[-1] @ W[2 * li].T + W[2 * li + 1]
        on = z > 0.0
        if relu_mask is not None:
            want = np.asarray(relu_mask).reshape(5, rows, HID)[li] != 0
            diff = want != on
            if diff.any():
                rms = np.sqrt((z * z).mean()) + 1e-300
                n_over += int(diff.sum())
                max_over = max(max_over, float(np.abs(z[diff]).max() / rms))
            on = want
        gates.append(on)
        ins.append(np.where(on, z, 0.0))
    head = ins[-1] @ W[10].T + W[11]
    r = vtrace_losses_length(oracle, head[:, :A].reshape(m, t, A), head[:, A].reshape(m, t), mu, act, rew, disc, boot, legal,
                             lengths, **cfg)
    dh = np.concatenate([r["dlogits"].reshape(rows, A), r["dvalue"].reshape(rows, 1)], 1)
    g = [None] * 12
    g[10], g[11] = dh.T @ ins[5], dh.sum(0)
    da = (dh @ W[10]) * gates[4]
    for li in range(4, -1, -1):
        g[2 * li], g[2 * li + 1] = da.T @ ins[li], da.sum(0)
        if li > 0:
            da = (da @ W[2 * li]) * gates[li - 1]
    return r["losses"], np.concatenate([a.ravel() for a in g]), n_over, max_over


def pack_length_slots(obs, mu_logits, action, reward, discount, bootstrap, words, legal=None, pad=None) -> np.ndarray:
    """Records of [m, t] trajectories with length words `words` [m] (uint32) in word 183 of record 0 and bootstrap[b] in
    word 181 of record L_b - 1 (the last record when L_b = t, as pyoracle.pack_vtrace_slots puts it). legal: words for
    record word 182. pad: None leaves the records past L_b as the packer wrote them; "zeros" zeroes them; "garbage" fills
    every word of them with NaN, +-inf, 1e30 and random bit patterns."""
    m, t = np.asarray(action).shape
    L = lengths_of(words, t)
    slots = (po.pack_vtrace_slots(obs, mu_logits, action, reward, discount, bootstrap) if legal is None else
             LR.pack_vtrace_slots_legal(obs, mu_logits, action, reward, discount, bootstrap, legal))
    w = slots.view(np.uint32).reshape(m, t, po.REC_WORDS)
    f = slots.view(np.float32).reshape(m, t, po.REC_WORDS)
    f[:, t - 1, 181] = 0.0
    f[np.arange(m), L - 1, 181] = np.asarray(bootstrap, np.float32)
    past = ~valid_rows(L, t)
    if pad == "zeros":
        w[past] = 0
    elif pad == "garbage":
        n = int(past.sum())
        rng = np.random.default_rng(n)
        g = rng.integers(0, 1 << 32, size=(n, po.REC_WORDS), dtype=np.uint64).astype(np.uint32)
        special = np.array([np.nan, np.inf, -np.inf, 1e30, -1e30], np.float32).view(np.uint32)
        pick = rng.integers(0, 6, size=g.shape)
        g = np.where(pick < 5, special[np.minimum(pick, 4)], g)
        w[past] = g
    w[:, 0, WORD] = np.asarray(words, np.uint32)
    return slots
