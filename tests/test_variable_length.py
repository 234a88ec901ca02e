"""Variable-length trajectories, without a GPU: the float64 reference of tests/length_reference.py against torch float64
autograd and against the C oracle run on the truncated trajectories, the decoding of the length word, and the C ABI of the
option (struct layout, default, the configurations fi_learner_create refuses before it looks for a device).

The rule (include/fi_learner.h, FI_REC_WORD_LENGTH): trajectory b holds L_b = (W == 0 || W > t) ? t : W steps, W being word 183
of its record 0; the step is the step on the trajectories cut to their first L_b records, with the bootstrap from record
L_b - 1."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _util as U
import legal_reference as LR
import length_reference as R
from oracle import pyoracle as po

HEADER = os.path.join(U.ROOT, "include", "fi_learner.h")
A = po.NUM_ACTIONS
C1 = dict(rho_bar=2.0, c_bar=0.7, pg_rho_bar=1.5, lambda_=0.95, baseline_cost=0.25, entropy_cost=0.05)
CFGS = {"default": {}, "c1-distinct": C1}


def _case(seed, m, t):
    """Random head outputs and records, lengths 1 and t among random ones."""
    rng = np.random.default_rng(seed)
    logits = rng.standard_normal((m, t, A)) * 2.0
    value = rng.standard_normal((m, t))
    mu = (rng.standard_normal((m, t, A)) * 2.0).astype(np.float32)
    act = rng.integers(0, A, size=(m, t)).astype(np.int32)
    rew = rng.standard_normal((m, t)).astype(np.float32)
    disc = (0.99 * (rng.random((m, t)) >= 0.05)).astype(np.float32)
    boot = rng.standard_normal(m).astype(np.float32)
    L = rng.integers(1, t + 1, size=m)
    L[0], L[-1] = 1, t
    return logits, value, mu, act, rew, disc, boot, L


def _torch_reference(logits, value, mu, act, rew, disc, boot, L, cfg):
    """The loss over the valid steps in torch float64 with autograd on the whole [m, t] arrays: a step past L_b is masked out
    of every sum (torch.where, so its values never combine with anything), the V-trace targets come from a float64 loop that
    stops at L_b and bootstraps from boot[b] there; vs and pg_adv are constants."""
    import torch
    c = {**po.DEFAULT_VTRACE, **cfg}
    m, t = act.shape
    keep = torch.from_numpy(R.valid_rows(L, t))
    zero = torch.zeros((), dtype=torch.float64)
    z = torch.tensor(logits, dtype=torch.float64, requires_grad=True)
    v = torch.tensor(value, dtype=torch.float64, requires_grad=True)
    logp = torch.log_softmax(z, -1)
    a = torch.from_numpy(act.astype(np.int64))[..., None]
    logp_a = torch.gather(logp, -1, a)[..., 0]
    log_mu_a = torch.gather(torch.log_softmax(torch.from_numpy(mu.astype(np.float64)), -1), -1, a)[..., 0]
    rho = np.exp((logp_a - log_mu_a).detach().numpy())
    vs, adv = np.zeros((m, t)), np.zeros((m, t))
    g, r = disc.astype(np.float64), rew.astype(np.float64)
    for b in range(m):
        n, acc = int(L[b]), 0.0
        for s in range(n - 1, -1, -1):
            v_next = float(boot[b]) if s == n - 1 else value[b, s + 1]
            acc = (min(c["rho_bar"], rho[b, s]) * (r[b, s] + g[b, s] * v_next - value[b, s]) +
                   g[b, s] * c["lambda_"] * min(c["c_bar"], rho[b, s]) * acc)
            vs[b, s] = value[b, s] + acc
        for s in range(n):
            vs_next = float(boot[b]) if s == n - 1 else vs[b, s + 1]
            adv[b, s] = min(c["pg_rho_bar"], rho[b, s]) * (r[b, s] + g[b, s] * vs_next - value[b, s])
    vs_t, adv_t = torch.from_numpy(vs), torch.from_numpy(adv)
    pg = -torch.where(keep, logp_a * adv_t, zero).sum()
    bl = 0.5 * torch.where(keep, (vs_t - v) ** 2, zero).sum()
    ent = torch.where(keep, (torch.exp(logp) * logp).sum(-1), zero).sum()
    total = pg + c["baseline_cost"] * bl + c["entropy_cost"] * ent
    total.backward()
    losses = np.array([total.item(), pg.item(), bl.item(), ent.item()])
    return dict(losses=losses, dlogits=z.grad.numpy(), dvalue=v.grad.numpy(), vs=vs, pg_adv=adv)


@pytest.mark.parametrize("name", list(CFGS))
@pytest.mark.parametrize("m,t", [(3, 7), (6, 40)])
def test_length_reference_matches_torch_autograd(oracle, m, t, name):
    logits, value, mu, act, rew, disc, boot, L = _case(m * t + len(name), m, t)
    got = R.vtrace_losses_length(oracle, logits, value, mu, act, rew, disc, boot, None, L, **CFGS[name])
    want = _torch_reference(logits, value, mu, act, rew, disc, boot, L, CFGS[name])
    for k in ("losses", "dlogits", "dvalue", "vs", "pg_adv"):
        e = U.rel_max(got[k], want[k])
        assert e <= 1e-12, (k, e)
    past = ~R.valid_rows(L, t)
    assert past.any() and np.all(got["dlogits"][past] == 0.0) and np.all(got["dvalue"][past] == 0.0)


@pytest.mark.parametrize("legal", [False, True])
def test_reference_is_the_oracle_on_the_truncated_trajectories(oracle, legal):
    """Each trajectory's rows of the reference are bit-identical to the C oracle (or, with legal words, the masked reference)
    run on that trajectory cut to T = L_b, lengths 1 and t included; the loss is their sum."""
    m, t = 7, 33
    logits, value, mu, act, rew, disc, boot, L = _case(17, m, t)
    words = np.random.default_rng(3).integers(0, 1 << 16, size=(m, t)).astype(np.uint32) if legal else None
    got = R.vtrace_losses_length(oracle, logits, value, mu, act, rew, disc, boot, words, L, **C1)
    total = np.zeros(4)
    for b in range(m):
        n = int(L[b])
        cut = [np.ascontiguousarray(x[b:b + 1, :n]) for x in (logits, value, mu, act, rew, disc)]
        want = (oracle.vtrace_losses(*cut, boot[b:b + 1], **C1) if words is None else
                LR.vtrace_losses_legal(oracle, *cut, boot[b:b + 1], words[b:b + 1, :n], **C1))
        total += want["losses"]
        for k in ("dlogits", "dvalue", "vs", "pg_adv"):
            assert np.array_equal(got[k][b, :n], want[k][0]), (b, n, k)
            assert not got[k][b, n:].any(), (b, n, k)
    assert np.array_equal(got["losses"], total)


def test_actor_critic_step_is_the_oracle_on_the_truncated_trajectories(oracle):
    """Every trajectory 5 of 9 steps long: the reference's step is the C oracle's step (orc_ac_loss_grad) on the [m, 5]
    trajectories, losses and every parameter's gradient to 1e-12, whatever the records past step 5 hold."""
    m, t, n = 4, 9, 5
    obs, mu, act, rew, disc, boot = U.vtrace_batch(21, m, t)
    params = U.ac_params(21)
    O = oracle.actor_critic(params, **C1)
    want = O.loss_grad(*(np.ascontiguousarray(x[:, :n]) for x in (obs, mu, act, rew, disc)), boot)
    obs2 = obs.copy()
    obs2[:, n:] = np.nan
    got, grads, _, _ = R.ac_loss_grad_length(oracle, params, obs2, mu, act, rew, disc, boot, None, np.full(m, n), **C1)
    assert U.rel_max(got, want) <= 1e-12 and U.rel_max(grads, O.grads()) <= 1e-12


def test_length_word_zero_or_above_t_means_full_length(oracle):
    """W = 0 and W > t decode to L = t, and the reference then equals the oracle on the whole batch to 1e-12."""
    m, t = 4, 12
    assert list(R.lengths_of([0, t + 1, 0xFFFFFFFF, t, 1, 5], t)) == [t, t, t, t, 1, 5]
    logits, value, mu, act, rew, disc, boot, _ = _case(5, m, t)
    want = oracle.vtrace_losses(logits, value, mu, act, rew, disc, boot, **C1)
    for words in ([0] * m, [t + 1, t + 2, 1 << 31, 0xFFFFFFFF], [t] * m):
        got = R.vtrace_losses_length(oracle, logits, value, mu, act, rew, disc, boot, None, R.lengths_of(words, t), **C1)
        for k in want:
            assert U.rel_max(got[k], want[k]) <= 1e-12, (words, k)


def test_packer_writes_length_and_bootstrap(oracle):
    m, t = 3, 6
    obs, mu, act, rew, disc, boot = U.vtrace_batch(9, m, t)
    words = np.array([0, 2, 9], np.uint32)       # L = 6, 2, 6
    slots = R.pack_length_slots(obs, mu, act, rew, disc, boot, words, pad="garbage")
    w = slots.view(np.uint32).reshape(m, t, po.REC_WORDS)
    f = slots.view(np.float32).reshape(m, t, po.REC_WORDS)
    assert np.array_equal(w[:, 0, 183], words)
    assert f[1, 1, 181] == boot[1] and f[0, t - 1, 181] == boot[0] and f[2, t - 1, 181] == boot[2]
    plain = po.pack_vtrace_slots(obs, mu, act, rew, disc, boot).view(np.uint32).reshape(m, t, po.REC_WORDS)
    assert np.array_equal(w[1, :2, :181], plain[1, :2, :181])
    assert not np.isfinite(f[1, 2:]).all()        # the padding really is garbage


# ------------------------------------------------------------------------------- C ABI
def test_header_field_matches_ctypes(fi, tmp_path):
    from freeimpala_b200 import _lib
    c = tmp_path / "l.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fi_learner.h"\n'
                 'int main(void){printf("%zu %zu %zu %d\\n", sizeof(fi_learner_config), offsetof(fi_learner_config, variable_length),'
                 'offsetof(fi_learner_config, legal_action_mask), FI_REC_WORD_LENGTH);return 0;}\n')
    exe = tmp_path / "l"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.dirname(HEADER), str(c), "-o", str(exe)], check=True)
    size, off, off_prev, word = map(int, subprocess.check_output([str(exe)]).split())
    K = _lib.FiLearnerConfig
    assert C.sizeof(K) == size and K.variable_length.offset == off
    assert off > off_prev   # appended after the fields that existed before
    assert word == 183 == R.WORD


def test_config_default_leaves_lengths_off(fi):
    from freeimpala_b200 import _lib
    cfg = _lib.FiLearnerConfig()
    cfg.variable_length = 7
    fi.load_library().fi_learner_config_default(C.byref(cfg))
    assert cfg.variable_length == 0


@pytest.mark.parametrize("model,value", [("mlp_actor_critic", 2), ("mlp_actor_critic", -1), ("farmer_lstm", 1)])
def test_create_rejects_invalid_lengths_before_the_device_check(fi, model, value):
    from freeimpala_b200 import _lib
    lib = fi.load_library()
    cfg = _lib.FiLearnerConfig()
    lib.fi_learner_config_default(C.byref(cfg))
    cfg.num_players, cfg.buffer_capacity, cfg.entry_size, cfg.batch_size = 1, 4, 8, 2
    cfg.model = _lib.MODEL[model]
    cfg.loss = _lib.LOSS["vtrace" if model == "mlp_actor_critic" else "mse"]
    cfg.variable_length = value
    assert not lib.fi_learner_create(C.byref(cfg))
    msg = _lib.last_error()
    assert msg.startswith("fi_learner_create: variable_length") and "no CUDA device" not in msg, msg


def test_learner_keyword_reaches_the_config(fi):
    with pytest.raises(fi.FiError, match="variable_length"):
        fi.Learner(1, 4, 8, 2, model="farmer_lstm", variable_length=True)


def test_loss_head_operator_rejects_bad_flags(fi):
    """fi_op_vtrace_loss_head_opts checks its flags before it touches a pointer."""
    from freeimpala_b200 import _lib
    lib = fi.load_library()
    for legal, lengths in ((2, 0), (0, -1)):
        rc = lib.fi_op_vtrace_loss_head_opts(None, 1, 1, None, 17, 1.0, 1.0, 1.0, 1.0, 0.5, 0.01, legal, lengths,
                                             None, None, None, None, None)
        assert rc == _lib.FI_ERR_ARG and "legal and lengths" in _lib.last_error()
