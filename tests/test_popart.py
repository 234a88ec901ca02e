"""PopArt value normalisation (fi_learner_config.popart_beta), without a GPU: the float64 reference of tests/popart_reference.py
against the C oracle and torch float64 autograd, its statistics and rescale rules, the config field and its refusals."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _util as U
import length_reference as LenR
import popart_reference as R
from oracle import pyoracle as po

A = po.NUM_ACTIONS
CFG = dict(rho_bar=2.0, c_bar=0.7, pg_rho_bar=1.5, lambda_=0.95, baseline_cost=0.25, entropy_cost=0.05)


def _case(seed, m, t):
    obs, mu, act, rew, disc, boot = U.vtrace_batch(seed, m, t, done_p=0.05)
    rng = np.random.default_rng(seed + 1)
    logits = rng.standard_normal((m, t, A))
    n = rng.standard_normal((m, t))
    return logits, n, mu, act, rew, disc, boot


def test_reference_at_unit_statistics_is_the_oracles_loss(oracle):
    """mu = 0, sigma = 1: losses, d(head), vs and pg_adv are the C oracle's vtrace_losses (float64, 1e-12)."""
    logits, n, mu, act, rew, disc, boot = _case(3, 5, 37)
    got = R.vtrace_losses_popart(oracle, logits, n, mu, act, rew, disc, boot, 0.0, 1.0, **CFG)
    want = oracle.vtrace_losses(logits, n, mu, act, rew, disc, boot, **CFG)
    for k in ("losses", "dlogits", "dvalue", "vs", "pg_adv"):
        np.testing.assert_allclose(got[k], want[k], rtol=1e-12, atol=1e-12, err_msg=k)
    assert got["sums"][2] == 5 * 37
    np.testing.assert_allclose(got["sums"][:2], [want["vs"].sum(), (want["vs"] ** 2).sum()], rtol=1e-12)


@pytest.mark.parametrize("legal", [False, True])
@pytest.mark.parametrize("lengths", [False, True])
def test_reference_gradient_is_torch_autograd_of_the_normalised_loss(oracle, legal, lengths):
    """d(total)/d(logits) and d(total)/dn of the normalised loss, vs and A held constant, with mu != 0 and sigma != 1."""
    import torch
    m, t = 6, 33
    logits, n, mu_l, act, rew, disc, boot = _case(11, m, t)
    rew = rew * 100.0
    lw = np.random.default_rng(5).integers(0, 1 << 16, size=(m, t)).astype(np.uint32) if legal else None
    L = np.array([1, 7, 32, 33, 20, 33]) if lengths else None
    mu, sig = 3.5, 41.0
    r = R.vtrace_losses_popart(oracle, logits, n, mu_l, act, rew, disc, boot, mu, sig, lw, L, **CFG)
    tl = torch.tensor(logits, dtype=torch.float64, requires_grad=True)
    tn = torch.tensor(n, dtype=torch.float64, requires_grad=True)
    sup = torch.tensor(R.LR.support(np.full((m, t), 0xFFFF, np.uint32) if lw is None else lw, act))
    valid = torch.tensor(LenR.valid_rows(np.full(m, t) if L is None else L, t))
    z = torch.where(sup, tl, torch.tensor(-np.inf, dtype=torch.float64))
    logp = torch.where(sup, z - torch.logsumexp(z, -1, keepdim=True), torch.zeros((), dtype=torch.float64))
    p = torch.where(sup, logp.exp(), torch.zeros((), dtype=torch.float64))
    logp_a = logp.gather(-1, torch.tensor(act, dtype=torch.int64)[..., None])[..., 0]
    vs, adv = torch.tensor(r["vs"]), torch.tensor(r["pg_adv"])
    pg = -(logp_a * adv / sig)[valid].sum()
    bl = 0.5 * (((vs - mu) / sig - tn) ** 2)[valid].sum()
    ent = (p * logp).sum(-1)[valid].sum()
    total = pg + CFG["baseline_cost"] * bl + CFG["entropy_cost"] * ent
    total.backward()
    np.testing.assert_allclose(r["losses"], [total.item(), pg.item(), bl.item(), ent.item()], rtol=1e-12)
    np.testing.assert_allclose(r["dlogits"], tl.grad.numpy(), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(r["dvalue"], tn.grad.numpy(), rtol=1e-10, atol=1e-12)


def test_sigma_clamps_and_negative_variance():
    assert R.sigma(0.0, 1.0) == 1.0
    assert R.sigma(3.0, 25.0) == 4.0
    assert R.sigma(0.0, 1e-12) == 1e-4          # lower clamp
    assert R.sigma(0.0, 1e14) == 1e6            # upper clamp
    assert R.sigma(2.0, 3.0) == 1e-4            # nu < mu^2: variance taken as 0
    assert R.sigma(1e3, 1e6) == 1e-4            # nu == mu^2


def test_statistics_update():
    mu, nu = R.update_stats(0.0, 1.0, (50.0, 5000.0, 10.0), 0.25)
    assert (mu, nu) == (0.75 * 0.0 + 0.25 * 5.0, 0.75 * 1.0 + 0.25 * 500.0)
    assert R.update_stats(2.0, 7.0, (1.0, 1.0, 1.0), 0.0) == (2.0, 7.0)   # beta = 0 keeps them


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_rescale_preserves_the_unnormalised_value(seed):
    """After the statistics move, sigma' n' + mu' equals sigma n + mu on random last activations: 1e-12 in float64 (PopArtAC),
    1e-6 with the fp32 rounding of the arena (rescale)."""
    rng = np.random.default_rng(seed)
    params = U.ac_params(seed)
    h = np.abs(rng.standard_normal((64, R.HID)))
    P = R.PopArtAC(params, beta=0.3, lr=0.0)
    P.mu, P.nu = rng.standard_normal() * 10, 200.0 + rng.random() * 50
    before = R.sigma(P.mu, P.nu) * (h @ P.p[R.W_OFF:R.W_OFF + R.HID] + P.p[R.B_OFF]) + P.mu
    mu0, nu0 = P.mu, P.nu
    sums = (rng.standard_normal() * 1e3, 1e6 * (1 + rng.random()), 100.0)
    P.step(np.zeros_like(P.p), sums)                # lr = 0: only the statistics and the rescale move
    after = R.sigma(P.mu, P.nu) * (h @ P.p[R.W_OFF:R.W_OFF + R.HID] + P.p[R.B_OFF]) + P.mu
    assert (P.mu, P.nu) != (mu0, nu0)
    np.testing.assert_allclose(after, before, rtol=1e-12, atol=1e-12 * np.abs(before).max())
    q = R.rescale(params, mu0, nu0, P.mu, P.nu)
    w, b = q[R.W_OFF:R.W_OFF + R.HID].astype(np.float64), float(q[R.B_OFF])
    w0, b0 = params[R.W_OFF:R.W_OFF + R.HID].astype(np.float64), float(params[R.B_OFF])
    v0 = R.sigma(mu0, nu0) * (h @ w0 + b0) + mu0
    v1 = R.sigma(P.mu, P.nu) * (h @ w + b) + P.mu
    assert U.rel_max(v1, v0) < 1e-6
    others = np.ones(params.size, bool)
    others[R.W_OFF:R.W_OFF + R.HID] = others[R.B_OFF] = False
    assert np.array_equal(q[others], params[others])


def test_publish_transform():
    params = U.ac_params(4)
    pub = R.publish(params, 2.5, 31.25)              # sigma = 5
    assert np.array_equal(pub[R.W_OFF:R.W_OFF + R.HID], (5.0 * params[R.W_OFF:R.W_OFF + R.HID].astype(np.float64)).astype(np.float32))
    assert pub[R.B_OFF] == np.float32(5.0 * float(params[R.B_OFF]) + 2.5)
    pub[R.W_OFF:R.W_OFF + R.HID] = params[R.W_OFF:R.W_OFF + R.HID]
    pub[R.B_OFF] = params[R.B_OFF]
    assert np.array_equal(pub, params)
    assert np.array_equal(R.publish(params, 0.0, 1.0), params)   # unit statistics publish the arena


# ------------------------------------------------------------------------------- C ABI
HEADER = os.path.join(U.ROOT, "include", "fi_learner.h")


def test_config_field_offset_and_default(fi, tmp_path):
    from freeimpala_b200 import _lib
    c = tmp_path / "o.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fi_learner.h"\n'
                 'int main(void){printf("%zu %zu %zu\\n", sizeof(fi_learner_config), offsetof(fi_learner_config, popart_beta),'
                 'offsetof(fi_learner_config, history_length));return 0;}\n')
    exe = tmp_path / "o"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.dirname(HEADER), str(c), "-o", str(exe)], check=True)
    size, off, hist = map(int, subprocess.check_output([str(exe)]).split())
    K = _lib.FiLearnerConfig
    assert C.sizeof(K) == size and K.popart_beta.offset == off and off > hist
    cfg = K()
    fi.load_library().fi_learner_config_default(C.byref(cfg))
    assert cfg.popart_beta == 0.0


BAD = [dict(popart_beta=float("nan")), dict(popart_beta=-1e-9), dict(popart_beta=1.0 + 1e-9), dict(popart_beta=float("inf")),
       dict(popart_beta=-float("inf")), dict(popart_beta=3e-4, model=0, loss=0)]


@pytest.mark.parametrize("bad", BAD, ids=lambda d: "-".join(f"{k}={v}" for k, v in d.items()))
def test_create_rejects_invalid_popart_beta_before_the_device_check(fi, bad):
    from freeimpala_b200 import _lib
    lib = fi.load_library()
    cfg = _lib.FiLearnerConfig()
    lib.fi_learner_config_default(C.byref(cfg))
    cfg.num_players, cfg.buffer_capacity, cfg.entry_size, cfg.batch_size = 1, 4, 8, 2
    for k, v in bad.items():
        setattr(cfg, k, v)
    assert not lib.fi_learner_create(C.byref(cfg))
    msg = _lib.last_error()
    assert msg.startswith("fi_learner_create: ") and "no CUDA device" not in msg and "popart_beta" in msg, msg
    assert lib.fi_learner_create(C.byref(cfg)) is None and _lib.last_error() == msg


def test_learner_keyword_reaches_the_config(fi):
    with pytest.raises(fi.FiError, match="popart_beta"):
        fi.Learner(1, 4, 5, 2, popart_beta=2.0)
