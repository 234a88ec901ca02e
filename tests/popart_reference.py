"""Float64 reference of PopArt value normalisation in the actor-critic V-trace step (fi_learner_config.popart_beta,
include/fi_learner.h), for the tests of that option.

Step s runs with statistics mu_s, nu_s and sigma_s = sigma(mu_s, nu_s). Head column 16 is the normalised value n_t and
V_t = sigma_s n_t + mu_s is what V-trace sees (the bootstrap stays in reward units), so vs_t and A_t come from the C oracle's
recurrence through tests/length_reference.py (which composes legal-action words and trajectory lengths). Around it:
policy-gradient loss sum -log pi(a) A / sigma, baseline loss 1/2 sum ((vs - mu) / sigma - n)^2, the entropy unchanged, and
S1 = sum vs, S2 = sum vs^2, N = valid transitions. After the optimiser, the statistics move by beta towards the batch's moments
and the value row is rescaled so that sigma n + mu is unchanged; the published model carries sigma w and sigma b + mu in that row.
"""
from __future__ import annotations

import numpy as np

import legal_reference as LR
import length_reference as LenR
from oracle import pyoracle as po

A = po.NUM_ACTIONS
HID, ZD = LR.HID, LR.ZD
W_OFF = po.AC_PARAMS - 17 - 17 * HID + 16 * HID   # head.w row 16
B_OFF = po.AC_PARAMS - 1                           # head.b[16]


def sigma(mu, nu):
    """clamp(sqrt(max(nu - mu^2, 0)), 1e-4, 1e6), each operation rounded once as the library does."""
    var = float(nu) - float(mu) * float(mu)
    return min(max(np.sqrt(var) if var > 0.0 else 0.0, 1e-4), 1e6)


def vtrace_losses_popart(oracle, logits, nvalue, mu_logits, action, reward, discount, bootstrap, mu, sig, legal=None,
                         lengths=None, **cfg):
    """The PopArt loss head at statistics (mu, sig): losses {total, pg, baseline, entropy} in normalised units, dlogits,
    dvalue (d/dn), vs and pg_adv in reward units (zero past each trajectory's length) and sums {S1, S2, N}."""
    c = {**po.DEFAULT_VTRACE, **cfg}
    m, t = np.asarray(action).shape
    L = np.full(m, t, np.int64) if lengths is None else np.asarray(lengths, np.int64)
    n = np.asarray(nvalue, np.float64)
    V = sig * n + mu
    r = LenR.vtrace_losses_length(oracle, logits, V, mu_logits, action, reward, discount, bootstrap, legal, L, **cfg)
    vs, adv = r["vs"], r["pg_adv"]
    valid = LenR.valid_rows(L, t)
    act = np.asarray(action, np.int64)
    sup = LR.support(np.full((m, t), 0xFFFF, np.uint32) if legal is None else legal, act)
    logp = LR.masked_log_softmax(np.asarray(logits, np.float64), sup)
    p = np.where(sup, np.exp(logp), 0.0)
    plogp = (p * logp).sum(-1)
    take = np.take_along_axis(logp, act[..., None], -1)[..., 0]
    adv_n = adv / sig
    verr = (vs - mu) / sig - n
    onehot = np.arange(A) == act[..., None]
    dlogits = np.where(sup, adv_n[..., None] * (p - onehot) + c["entropy_cost"] * p * (logp - plogp[..., None]), 0.0)
    dlogits = np.where(valid[..., None], dlogits, 0.0)
    pg = -(take * adv_n)[valid].sum()
    bl = 0.5 * (verr ** 2)[valid].sum()
    ent = plogp[valid].sum()
    losses = np.array([pg + c["baseline_cost"] * bl + c["entropy_cost"] * ent, pg, bl, ent])
    dvalue = np.where(valid, -c["baseline_cost"] * verr, 0.0)
    sums = np.array([vs[valid].sum(), (vs[valid] ** 2).sum(), float(valid.sum())])
    return dict(losses=losses, dlogits=dlogits, dvalue=dvalue, vs=np.where(valid, vs, 0.0), pg_adv=np.where(valid, adv, 0.0),
                sums=sums)


def update_stats(mu, nu, sums, beta):
    """(mu', nu') = (1 - beta) (mu, nu) + beta (S1 / N, S2 / N)."""
    s1, s2, n = sums
    return (1.0 - beta) * mu + beta * (s1 / n), (1.0 - beta) * nu + beta * (s2 / n)


def rescale(params, mu0, nu0, mu1, nu1):
    """The value row rescaled so that sigma n + mu is unchanged, in double, rounded to fp32 once (a new fp32 array)."""
    s0, s1 = sigma(mu0, nu0), sigma(mu1, nu1)
    out = np.array(params, np.float32, copy=True)
    w = out[W_OFF:W_OFF + HID].astype(np.float64)
    out[W_OFF:W_OFF + HID] = (w * s0 / s1).astype(np.float32)
    out[B_OFF] = np.float32((s0 * float(out[B_OFF]) + mu0 - mu1) / s1)
    return out


def publish(params, mu, nu):
    """The published (reward-unit) model of an arena: value row w -> sigma w, b -> sigma b + mu, rounded once."""
    s = sigma(mu, nu)
    out = np.array(params, np.float32, copy=True)
    out[W_OFF:W_OFF + HID] = (s * out[W_OFF:W_OFF + HID].astype(np.float64)).astype(np.float32)
    out[B_OFF] = np.float32(s * float(out[B_OFF]) + mu)
    return out


def ac_loss_grad_popart(oracle, params, obs, mu_l, act, rew, disc, boot, mu, sig, legal=None, lengths=None, relu_mask=None, **cfg):
    """The PopArt actor-critic step's loss, gradient over the flat arena and sums at `params`, in float64 (the forward and
    backward of length_reference.ac_loss_grad_length). Returns (losses[4], grads, sums[3], units overridden, largest |z|/rms)."""
    m, t = np.asarray(act).shape
    rows = m * t
    L = np.full(m, t, np.int64) if lengths is None else np.asarray(lengths, np.int64)
    W = LR._tensors(np.asarray(params, np.float64))
    keep = LenR.valid_rows(L, t).reshape(rows, 1)
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
    r = vtrace_losses_popart(oracle, head[:, :A].reshape(m, t, A), head[:, A].reshape(m, t), mu_l, act, rew, disc, boot, mu, sig,
                             legal, L, **cfg)
    dh = np.concatenate([r["dlogits"].reshape(rows, A), r["dvalue"].reshape(rows, 1)], 1)
    g = [None] * 12
    g[10], g[11] = dh.T @ ins[5], dh.sum(0)
    da = (dh @ W[10]) * gates[4]
    for li in range(4, -1, -1):
        g[2 * li], g[2 * li + 1] = da.T @ ins[li], da.sum(0)
        if li > 0:
            da = (da @ W[2 * li]) * gates[li - 1]
    return r["losses"], np.concatenate([a.ravel() for a in g]), r["sums"], n_over, max_over


class PopArtAC:
    """A float64 PopArt actor-critic learner with libtorch's Adam: params, moments, statistics. step() applies the optimiser
    to the given gradient, then the statistics update from the given sums and the value-row rescale."""

    def __init__(self, params, beta, lr=5e-4):
        self.p = np.asarray(params, np.float64).copy()
        self.m, self.v = np.zeros_like(self.p), np.zeros_like(self.p)
        self.k, self.beta, self.lr = 0, beta, lr
        self.mu, self.nu = 0.0, 1.0

    def stats32(self):
        """mu and sigma as the kernels use them (fp32 copies)."""
        return float(np.float32(self.mu)), float(np.float32(sigma(self.mu, self.nu)))

    def step(self, grads, sums):
        b1, b2, eps = 0.9, 0.999, 1e-8
        self.k += 1
        g = np.asarray(grads, np.float64)
        self.m = b1 * self.m + (1 - b1) * g
        self.v = b2 * self.v + (1 - b2) * g * g
        denom = np.sqrt(self.v) / np.sqrt(1 - b2 ** self.k) + eps
        self.p -= self.lr / (1 - b1 ** self.k) * self.m / denom
        mu1, nu1 = update_stats(self.mu, self.nu, sums, self.beta)
        s0, s1 = sigma(self.mu, self.nu), sigma(mu1, nu1)
        self.p[W_OFF:W_OFF + HID] *= s0 / s1
        self.p[B_OFF] = (s0 * self.p[B_OFF] + self.mu - mu1) / s1
        self.mu, self.nu = mu1, nu1
