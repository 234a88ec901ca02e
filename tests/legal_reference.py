"""Float64 reference of the legal-action-masked V-trace loss and actor-critic step (fi_learner_config.legal_action_mask,
record word 182, include/fi_learner.h), for the tests of that option.

For transition i the support is legal[i] | (1 << action[i]) (bits 16..31 ignored). pi and mu are softmaxes over it, the
entropy sums over it, and d(loss)/d(logit j) is 0 outside it; logits outside it never enter the arithmetic.

The V-trace recurrence is the C oracle's own (orc_vtrace); the masked softmaxes, losses and the actor-critic
forward / backward around them are float64 numpy here. tests/test_oracle_legal_actions.py holds this module to torch float64
autograd of the masked loss and, with every action legal, to the C oracle's unmasked loss and step.
"""
from __future__ import annotations

import numpy as np

from oracle import pyoracle as po

A = po.NUM_ACTIONS
HID, ZD, NHEAD = 512, po.Z_DIM, A + 1


def support(legal, act):
    """[m,t,A] bool: bit j of the legal word, or j is the action taken."""
    legal = np.asarray(legal, np.uint32)
    bits = (legal[..., None].astype(np.uint64) >> np.arange(A, dtype=np.uint64)) & 1
    return (bits == 1) | (np.arange(A) == np.asarray(act)[..., None])


def masked_log_softmax(z, sup):
    """log-softmax over the support; 0 (never used) outside it. Entries outside the support are not read into the sums."""
    zm = np.where(sup, z, -np.inf)
    mx = zm.max(-1, keepdims=True)
    e = np.where(sup, np.exp(np.where(sup, z, mx) - mx), 0.0)
    return np.where(sup, z - (mx + np.log(e.sum(-1, keepdims=True))), 0.0)


def vtrace_losses_legal(oracle, logits, value, mu_logits, action, reward, discount, bootstrap, legal, **cfg):
    """Masked counterpart of Oracle.vtrace_losses: same arguments and result dict (losses = {total, pg, baseline, entropy})."""
    c = {**po.DEFAULT_VTRACE, **cfg}
    logits, value = np.asarray(logits, np.float64), np.asarray(value, np.float64)
    act = np.asarray(action, np.int64)
    sup = support(legal, act)
    logp = masked_log_softmax(logits, sup)
    log_mu = masked_log_softmax(np.asarray(mu_logits, np.float32).astype(np.float64), sup)
    take = lambda x: np.take_along_axis(x, act[..., None], -1)[..., 0]   # noqa: E731
    log_rho = take(logp) - take(log_mu)
    f64 = lambda x: np.asarray(x, np.float32).astype(np.float64)         # noqa: E731  (records hold fp32)
    vs, adv = oracle.vtrace(log_rho, f64(discount), f64(reward), value, f64(bootstrap), c["rho_bar"], c["c_bar"],
                            c["pg_rho_bar"], c["lambda_"])
    p = np.where(sup, np.exp(logp), 0.0)
    plogp = (p * logp).sum(-1)
    pg, bl, ent = -(take(logp) * adv).sum(), 0.5 * ((vs - value) ** 2).sum(), plogp.sum()
    onehot = np.arange(A) == act[..., None]
    dlogits = np.where(sup, adv[..., None] * (p - onehot) + c["entropy_cost"] * p * (logp - plogp[..., None]), 0.0)
    losses = np.array([pg + c["baseline_cost"] * bl + c["entropy_cost"] * ent, pg, bl, ent])
    return dict(losses=losses, dlogits=dlogits, dvalue=-c["baseline_cost"] * (vs - value), vs=vs, pg_adv=adv)


def _tensors(params):
    off, out = 0, []
    for shp in ((HID, ZD), (HID,), (HID, HID), (HID,), (HID, HID), (HID,), (HID, HID), (HID,), (HID, HID), (HID,),
                (NHEAD, HID), (NHEAD,)):
        n = int(np.prod(shp))
        out.append(params[off:off + n].reshape(shp))
        off += n
    assert off == po.AC_PARAMS
    return out


def ac_loss_grad_legal(oracle, params, obs, mu, act, rew, disc, boot, legal, relu_mask=None, **cfg):
    """The actor-critic step's masked loss and its gradient over the flat parameter arena (parameters() order) at `params`,
    in float64. relu_mask ([5, rows*512] uint8, the CUDA run's decisions) pins the ReLU units the way
    Oracle.loss_grad_masked does. Returns (losses[4], grads[AC_PARAMS], units overridden, largest |z|/rms among them)."""
    m, t = np.asarray(act).shape
    rows = m * t
    W = _tensors(np.asarray(params, np.float64))
    x = np.asarray(obs, np.float32).reshape(rows, ZD).astype(np.float64)
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
    r = vtrace_losses_legal(oracle, head[:, :A].reshape(m, t, A), head[:, A].reshape(m, t), mu, act, rew, disc, boot, legal,
                            **cfg)
    dh = np.concatenate([r["dlogits"].reshape(rows, A), r["dvalue"].reshape(rows, 1)], 1)
    g = [None] * 12
    g[10], g[11] = dh.T @ ins[5], dh.sum(0)
    da = (dh @ W[10]) * gates[4]
    for li in range(4, -1, -1):
        g[2 * li], g[2 * li + 1] = da.T @ ins[li], da.sum(0)
        if li > 0:
            da = (da @ W[2 * li]) * gates[li - 1]
    return r["losses"], np.concatenate([a.ravel() for a in g]), n_over, max_over


def pack_vtrace_slots_legal(obs, mu_logits, action, reward, discount, bootstrap, legal) -> np.ndarray:
    """pyoracle.pack_vtrace_slots with the legal-action words [m,t] in record word 182."""
    slots = po.pack_vtrace_slots(obs, mu_logits, action, reward, discount, bootstrap)
    m, t = np.asarray(action).shape
    slots.view(np.uint32).reshape(m, t, po.REC_WORDS)[:, :, 182] = np.asarray(legal, np.uint32)
    return slots
