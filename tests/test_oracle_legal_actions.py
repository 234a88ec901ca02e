"""Legal-action masking of the V-trace loss, without a GPU: the float64 reference of tests/legal_reference.py against torch
float64 autograd of the masked loss and, with every action legal, against the C oracle's unmasked loss and actor-critic step;
and the C ABI of the option (struct layout, default, the configurations fi_learner_create refuses before it looks for a
device).

The masked loss (include/fi_learner.h, FI_REC_WORD_LEGAL): for transition i the support is legal[i] | (1 << action[i]);
pi and mu are softmaxes over it, the entropy sums over it, and d(loss)/d(logit j) is 0 outside it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _util as U
import legal_reference as R
from oracle import pyoracle as po

HEADER = os.path.join(U.ROOT, "include", "fi_learner.h")
A = po.NUM_ACTIONS
C1 = dict(rho_bar=2.0, c_bar=0.7, pg_rho_bar=1.5, lambda_=0.95, baseline_cost=0.25, entropy_cost=0.05)
CFGS = {"default": {}, "c1-distinct": C1}


def _vtrace_np(log_rho, disc, rew, value, boot, rho_bar, c_bar, pg_rho_bar, lambda_):
    """Paper eq. (1) with Remark 2 and section 4.2, float64, written out step by step."""
    m, t = log_rho.shape
    vs, adv = np.empty((m, t)), np.empty((m, t))
    for b in range(m):
        acc = 0.0
        for s in range(t - 1, -1, -1):
            r = np.exp(log_rho[b, s])
            v_next = boot[b] if s == t - 1 else value[b, s + 1]
            delta = min(rho_bar, r) * (rew[b, s] + disc[b, s] * v_next - value[b, s])
            acc = delta + disc[b, s] * lambda_ * min(c_bar, r) * acc
            vs[b, s] = value[b, s] + acc
        for s in range(t):
            vs_next = boot[b] if s == t - 1 else vs[b, s + 1]
            adv[b, s] = min(pg_rho_bar, np.exp(log_rho[b, s])) * (rew[b, s] + disc[b, s] * vs_next - value[b, s])
    return vs, adv


def _torch_reference(logits, value, mu, act, rew, disc, boot, legal, cfg):
    """The masked loss in torch float64 with autograd: log-softmax over the support through torch.where (entries outside
    it are never combined with -inf), vs and pg_adv as constants."""
    import torch
    c = {**po.DEFAULT_VTRACE, **cfg}
    sup = R.support(legal, act)
    S = torch.from_numpy(sup)
    z = torch.tensor(logits, dtype=torch.float64, requires_grad=True)
    v = torch.tensor(value, dtype=torch.float64, requires_grad=True)
    lse = torch.logsumexp(torch.where(S, z, torch.tensor(-np.inf, dtype=torch.float64)), -1, keepdim=True)
    logp = torch.where(S, z - lse, torch.zeros((), dtype=torch.float64))
    p = torch.where(S, torch.exp(logp), torch.zeros((), dtype=torch.float64))
    a = torch.from_numpy(act.astype(np.int64))[..., None]
    logp_a = torch.gather(logp, -1, a)[..., 0]
    mz = torch.from_numpy(mu.astype(np.float64))
    log_mu = torch.where(S, mz - torch.logsumexp(torch.where(S, mz, torch.tensor(-np.inf, dtype=torch.float64)), -1,
                                                 keepdim=True), torch.zeros((), dtype=torch.float64))
    log_rho = (logp_a.detach() - torch.gather(log_mu, -1, a)[..., 0]).numpy()
    vs, adv = _vtrace_np(log_rho, disc.astype(np.float64), rew.astype(np.float64), value, boot.astype(np.float64),
                         c["rho_bar"], c["c_bar"], c["pg_rho_bar"], c["lambda_"])
    vs_t, adv_t = torch.from_numpy(vs), torch.from_numpy(adv)
    pg = -(logp_a * adv_t).sum()
    bl = 0.5 * ((vs_t - v) ** 2).sum()
    ent = (p * logp).sum()
    total = pg + c["baseline_cost"] * bl + c["entropy_cost"] * ent
    total.backward()
    losses = np.array([total.item(), pg.item(), bl.item(), ent.item()])
    return dict(losses=losses, dlogits=z.grad.numpy(), dvalue=v.grad.numpy(), vs=vs, pg_adv=adv), sup


def _case(seed, m, t):
    """Random head outputs and records with random legal words: about one transition in six a forced move (word 0), one
    in six a word without the action's bit, some words with bits 16..31 set."""
    rng = np.random.default_rng(seed)
    logits = rng.standard_normal((m, t, A)) * 2.0
    value = rng.standard_normal((m, t))
    mu = (rng.standard_normal((m, t, A)) * 2.0).astype(np.float32)
    act = rng.integers(0, A, size=(m, t)).astype(np.int32)
    rew = rng.standard_normal((m, t)).astype(np.float32)
    disc = (0.99 * (rng.random((m, t)) >= 0.05)).astype(np.float32)
    boot = rng.standard_normal(m).astype(np.float32)
    legal = rng.integers(0, 1 << 16, size=(m, t)).astype(np.uint32) | (np.uint32(1) << act.astype(np.uint32))
    kind = rng.integers(0, 6, size=(m, t))
    legal[kind == 0] = 0
    legal[kind == 1] &= ~(np.uint32(1) << act[kind == 1].astype(np.uint32))
    legal[kind == 2] |= rng.integers(1, 1 << 16, size=int((kind == 2).sum())).astype(np.uint32) << np.uint32(16)
    return logits, value, mu, act, rew, disc, boot, legal


@pytest.mark.parametrize("name", list(CFGS))
@pytest.mark.parametrize("m,t", [(3, 7), (5, 40)])
def test_masked_reference_matches_torch_autograd(oracle, m, t, name):
    logits, value, mu, act, rew, disc, boot, legal = _case(m * t + len(name), m, t)
    assert (legal == 0).any() and ((legal >> act.astype(np.uint32)) & 1 == 0).any()
    got = R.vtrace_losses_legal(oracle, logits, value, mu, act, rew, disc, boot, legal, **CFGS[name])
    want, sup = _torch_reference(logits, value, mu, act, rew, disc, boot, legal, CFGS[name])
    for k in ("losses", "dlogits", "dvalue", "vs", "pg_adv"):
        e = U.rel_max(got[k], want[k])
        assert e <= 1e-12, (k, e)
    assert np.all(got["dlogits"][~sup] == 0.0)
    # a forced move: pi(a) = 1, so no policy gradient and no entropy gradient
    forced = sup.sum(-1) == 1
    assert forced.any() and np.all(got["dlogits"][forced] == 0.0)


def test_logits_outside_the_support_never_enter_the_arithmetic(oracle):
    """NaN, -inf and +inf in the learner's and the behaviour logits outside the support leave every output bit-identical."""
    logits, value, mu, act, rew, disc, boot, legal = _case(11, 4, 9)
    want = R.vtrace_losses_legal(oracle, logits, value, mu, act, rew, disc, boot, legal, **C1)
    out = ~R.support(legal, act)
    for fill in (np.nan, -np.inf, np.inf):
        lg, mu2 = logits.copy(), mu.copy()
        lg[out], mu2[out] = fill, fill
        got = R.vtrace_losses_legal(oracle, lg, value, mu2, act, rew, disc, boot, legal, **C1)
        for k in want:
            assert np.array_equal(got[k], want[k]), (fill, k)


def test_all_legal_mask_matches_the_unmasked_oracle(oracle):
    """Every action legal: the masked loss is the C oracle's unmasked one (orc_vtrace_losses), to 1e-12."""
    logits, value, mu, act, rew, disc, boot, _ = _case(5, 6, 33)
    a = oracle.vtrace_losses(logits, value, mu, act, rew, disc, boot, **C1)
    b = R.vtrace_losses_legal(oracle, logits, value, mu, act, rew, disc, boot, np.full(act.shape, 0xFFFF, np.uint32), **C1)
    for k in a:
        assert U.rel_max(b[k], a[k]) <= 1e-12, k


def test_all_legal_actor_critic_step_matches_the_unmasked_oracle(oracle):
    """The reference's actor-critic forward / backward with every action legal against the C oracle's step
    (orc_ac_loss_grad_masked, the same pinned ReLU decisions, some of them overridden): losses and every parameter's
    gradient to 1e-12, and the same overrides counted."""
    m, t = 3, 5
    data = U.vtrace_batch(7, m, t)
    params = U.ac_params(3)
    O = oracle.actor_critic(params, **C1)
    z_on = np.random.default_rng(2).random(5 * m * t * 512) < 0.5
    want, n_want, max_want = O.loss_grad_masked(*data, z_on.astype(np.uint8))
    got, grads, n_got, max_got = R.ac_loss_grad_legal(oracle, params, *data, np.full((m, t), 0xFFFFFFFF, np.uint32),
                                                      relu_mask=z_on.astype(np.uint8), **C1)
    assert U.rel_max(got, want) <= 1e-12 and U.rel_max(grads, O.grads()) <= 1e-12
    assert n_got == n_want > 0 and abs(max_got - max_want) <= 1e-12 * max_want
    want = O.loss_grad(*data)
    got, grads, n_got, _ = R.ac_loss_grad_legal(oracle, params, *data, np.full((m, t), 0xFFFF, np.uint32), **C1)
    assert U.rel_max(got, want) <= 1e-12 and U.rel_max(grads, O.grads()) <= 1e-12 and n_got == 0


def test_actor_critic_step_with_legal_words_uses_the_masked_loss(oracle):
    """The head gradient is 0 in illegal columns, so the head weight rows of an action that is never legal (and never taken)
    get exactly no gradient, while the unmasked loss moves them."""
    m, t = 3, 6
    obs, mu, act, rew, disc, boot = U.vtrace_batch(8, m, t)
    act = act % 8                                  # actions 8..15 never taken ...
    legal = np.full((m, t), 0x00FF, np.uint32)     # ... and never legal
    params = U.ac_params(4)
    _, g, _, _ = R.ac_loss_grad_legal(oracle, params, obs, mu, act, rew, disc, boot, legal)
    off, num = oracle.ac_table()
    head_w = g[off[10]:off[10] + num[10]].reshape(17, 512)
    head_b = g[off[11]:off[11] + num[11]]
    assert not head_w[8:16].any() and not head_b[8:16].any()
    assert head_w[:8].any() and head_w[16].any()
    O = oracle.actor_critic(params)
    O.loss_grad(obs, mu, act, rew, disc, boot)
    assert O.grads()[off[10]:off[10] + num[10]].reshape(17, 512)[8:16].any()


def test_packer_writes_word_182(oracle):
    m, t = 2, 3
    data = U.vtrace_batch(9, m, t)
    legal = np.arange(m * t, dtype=np.uint32).reshape(m, t) * np.uint32(0x01010101)
    slots = R.pack_vtrace_slots_legal(*data, legal)
    words = slots.view(np.uint32).reshape(m, t, po.REC_WORDS)
    assert np.array_equal(words[:, :, 182], legal)
    plain = po.pack_vtrace_slots(*data).view(np.uint32).reshape(m, t, po.REC_WORDS)
    words[:, :, 182] = 0
    assert np.array_equal(words, plain)


# ------------------------------------------------------------------------------- C ABI
def test_header_field_matches_ctypes(fi, tmp_path):
    from freeimpala_b200 import _lib
    c = tmp_path / "l.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fi_learner.h"\n'
                 'int main(void){printf("%zu %zu %zu %d\\n", sizeof(fi_learner_config), offsetof(fi_learner_config, legal_action_mask),'
                 'offsetof(fi_learner_config, rmsprop_momentum), FI_REC_WORD_LEGAL);return 0;}\n')
    exe = tmp_path / "l"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.dirname(HEADER), str(c), "-o", str(exe)], check=True)
    size, off, off_prev, word = map(int, subprocess.check_output([str(exe)]).split())
    K = _lib.FiLearnerConfig
    assert C.sizeof(K) == size and K.legal_action_mask.offset == off
    assert off > off_prev   # appended after the fields that existed before
    assert word == 182


def test_config_default_leaves_masking_off(fi):
    from freeimpala_b200 import _lib
    cfg = _lib.FiLearnerConfig()
    cfg.legal_action_mask = 7
    fi.load_library().fi_learner_config_default(C.byref(cfg))
    assert cfg.legal_action_mask == 0


@pytest.mark.parametrize("model,value", [("mlp_actor_critic", 2), ("mlp_actor_critic", -1), ("farmer_lstm", 1)])
def test_create_rejects_invalid_masking_before_the_device_check(fi, model, value):
    from freeimpala_b200 import _lib
    lib = fi.load_library()
    cfg = _lib.FiLearnerConfig()
    lib.fi_learner_config_default(C.byref(cfg))
    cfg.num_players, cfg.buffer_capacity, cfg.entry_size, cfg.batch_size = 1, 4, 8, 2
    cfg.model = _lib.MODEL[model]
    cfg.loss = _lib.LOSS["vtrace" if model == "mlp_actor_critic" else "mse"]
    cfg.legal_action_mask = value
    assert not lib.fi_learner_create(C.byref(cfg))
    msg = _lib.last_error()
    assert msg.startswith("fi_learner_create: legal_action_mask") and "no CUDA device" not in msg, msg


def test_learner_keyword_reaches_the_config(fi):
    with pytest.raises(fi.FiError, match="legal_action_mask"):
        fi.Learner(1, 4, 8, 2, model="farmer_lstm", legal_action_mask=True)
