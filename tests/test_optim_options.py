"""RMSProp, global-norm gradient clipping and the learning-rate schedule, without a GPU:
the float64 references of tests/optim_reference.py against torch.optim / torch.nn.utils on the CPU, the C header and its ctypes mirror, and the
configurations fi_learner_create refuses before it looks for a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _util as U
import optim_reference as R
from oracle import pyoracle as po

HEADER = os.path.join(U.ROOT, "include", "fi_learner.h")
STEPS = 5
LRS = [1e-3, 1e-3, 4e-4, 2.5e-4, 0.0]   # changed between steps, the last one 0


def _torch_run(params, grads, opt, lr_sched, max_norm, **kw):
    """STEPS updates of one flat float64 tensor with torch.optim + clip_grad_norm_: (params, optimiser state, norms)."""
    import torch
    p = torch.nn.Parameter(torch.from_numpy(params.astype(np.float64)))
    if opt == "rmsprop":
        o = torch.optim.RMSprop([p], lr=lr_sched[0], alpha=kw["alpha"], eps=kw["eps"], momentum=kw["momentum"],
                                centered=False, weight_decay=0, foreach=False)
    elif opt == "adam":
        o = torch.optim.Adam([p], lr=lr_sched[0], foreach=False)
    elif opt == "adamw":
        o = torch.optim.AdamW([p], lr=lr_sched[0], weight_decay=1e-2, foreach=False)
    else:
        o = torch.optim.SGD([p], lr=lr_sched[0], foreach=False)
    norms = []
    for s in range(STEPS):
        p.grad = torch.from_numpy(grads[s].copy())
        if max_norm > 0:
            norms.append(float(torch.nn.utils.clip_grad_norm_([p], max_norm, foreach=False)))
        for gr in o.param_groups:
            gr["lr"] = lr_sched[s]
        o.step()
    return p.detach().numpy().copy(), o.state[p], norms


@pytest.mark.parametrize("clip", ["off", "inactive", "active"])
@pytest.mark.parametrize("eps", [1e-8, 0.01])
@pytest.mark.parametrize("momentum", [0.0, 0.9])
def test_oracle_rmsprop_and_clipping_match_torch_float64(oracle, momentum, eps, clip):
    """OptOracle's optimiser step on the actor-critic oracle (clip on a copy of the gradient, then RMSProp) against torch.optim.RMSprop and
    torch.nn.utils.clip_grad_norm_ in float64, 5 steps, the learning rate changed between steps: <= 1e-12 relative."""
    rng = np.random.default_rng(int(momentum * 10) + int(eps * 1000) + len(clip))
    params = U.ac_params(2)
    grads = [rng.standard_normal(po.AC_PARAMS) * 10.0 ** (s - 2) for s in range(STEPS)]
    # ||g|| of the steps runs from ~11 to ~1e5: "active" clips every step, "inactive" none
    max_norm = {"off": 0.0, "inactive": 1e9, "active": 5.0}[clip]
    alpha = 0.99
    O = R.OptOracle.actor_critic(oracle, params, opt="rmsprop", lr=LRS[0])
    for s in range(STEPS):
        O.set_grads(grads[s])
        O.set_opt(LRS[s], max_grad_norm=max_norm, rmsprop_alpha=alpha, rmsprop_eps=eps, rmsprop_momentum=momentum)
        O.opt_step()
        assert np.array_equal(O.grads(), grads[s])       # clipping never writes the stored gradient back
    want_p, state, _ = _torch_run(params, grads, "rmsprop", LRS, max_norm, alpha=alpha, eps=eps, momentum=momentum)
    got_p = O.params()
    m, v = O.opt_state()
    assert U.rel_max(got_p, want_p) <= 1e-12 and U.rel_l2(got_p, want_p) <= 1e-12
    assert U.rel_max(v, state["square_avg"].numpy()) <= 1e-12
    if momentum > 0:
        assert U.rel_max(m, state["momentum_buffer"].numpy()) <= 1e-12
    else:
        assert not m.any()


@pytest.mark.parametrize("opt", ["adam", "adamw", "sgd"])
def test_oracle_clipping_with_the_other_optimisers_matches_torch(oracle, opt):
    rng = np.random.default_rng(5)
    params = U.farmer_params(3)
    grads = [rng.standard_normal(po.FARMER_PARAMS) * (1.0 + s) for s in range(STEPS)]
    O = R.OptOracle.farmer(oracle, params, opt=opt, lr=LRS[0])
    for s in range(STEPS):
        O.set_grads(grads[s])
        O.set_opt(LRS[s], max_grad_norm=40.0)
        O.opt_step()
    want_p, _, _ = _torch_run(params, grads, opt, LRS, 40.0)
    assert U.rel_max(O.params(), want_p) <= 1e-12


def test_oracle_clip_coefficient_is_torchs(oracle):
    import torch
    g = np.random.default_rng(1).standard_normal(10007) * 3.0
    for max_norm in (1.0, 299.0, 1e6):
        t = torch.nn.Parameter(torch.zeros(g.size, dtype=torch.float64))
        t.grad = torch.from_numpy(g.copy())
        norm = float(torch.nn.utils.clip_grad_norm_([t], max_norm, foreach=False))
        coef, got_norm = R.clip_coef(g, max_norm)
        assert abs(got_norm - norm) <= 1e-12 * norm
        np.testing.assert_allclose(g * coef, t.grad.numpy(), rtol=1e-12, atol=0)


def test_oracle_f32_rmsprop_restatement_tracks_float64(oracle):
    """The fp32 restatement (the kernel's bit-exact reference) stays within fp32 rounding of the float64 update."""
    rng = np.random.default_rng(9)
    n = 4099
    p32 = rng.standard_normal(n).astype(np.float32)
    p64 = p32.astype(np.float64)
    sa32, buf32, sa64, buf64 = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n), np.zeros(n)
    for s in range(4):
        g = rng.standard_normal(n).astype(np.float32)
        R.rmsprop_f32(1e-3, 0.99, 0.01, 0.9, p32, g, sa32, buf32)
        R.rmsprop_f64(1e-3, 0.99, 0.01, 0.9, p64, g.astype(np.float64), sa64, buf64)
    assert U.rel_l2(p32, p64) < 1e-6 and U.rel_l2(sa32, sa64) < 1e-6 and U.rel_l2(buf32, buf64) < 1e-6


# ------------------------------------------------------------------------------- C ABI
def test_header_with_the_new_options_compiles_as_c_and_matches_ctypes(fi, tmp_path):
    from freeimpala_b200 import _lib
    c = tmp_path / "o.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fi_learner.h"\n'
                 'int main(void){fi_opt_kind k = FI_OPT_RMSPROP; printf("%d %zu %zu %zu %zu %zu\\n", (int)k, sizeof(fi_learner_config),'
                 'offsetof(fi_learner_config, max_grad_norm), offsetof(fi_learner_config, rmsprop_alpha),'
                 'offsetof(fi_learner_config, rmsprop_eps), offsetof(fi_learner_config, rmsprop_momentum));return 0;}\n')
    exe = tmp_path / "o"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.dirname(HEADER), str(c), "-o", str(exe)], check=True)
    kind, size, *offs = map(int, subprocess.check_output([str(exe)]).split())
    K = _lib.FiLearnerConfig
    assert kind == _lib.OPT["rmsprop"] == 3
    assert C.sizeof(K) == size
    assert [K.max_grad_norm.offset, K.rmsprop_alpha.offset, K.rmsprop_eps.offset, K.rmsprop_momentum.offset] == offs
    assert offs[0] > K.checkpoint_location.offset   # appended after the fields that existed before


def test_config_default_sets_torchs_rmsprop_defaults_and_no_clipping(fi):
    from freeimpala_b200 import _lib
    cfg = _lib.FiLearnerConfig()
    fi.load_library().fi_learner_config_default(C.byref(cfg))
    assert (cfg.max_grad_norm, cfg.rmsprop_alpha, cfg.rmsprop_eps, cfg.rmsprop_momentum) == (0.0, 0.99, 1e-8, 0.0)
    assert cfg.optimizer == _lib.OPT["adam"]


BAD = [
    dict(optimizer=4), dict(optimizer=-1),
    dict(max_grad_norm=-1.0), dict(max_grad_norm=float("inf")), dict(max_grad_norm=float("nan")),
    dict(rmsprop_alpha=0.0), dict(rmsprop_alpha=1.0), dict(rmsprop_alpha=1.5), dict(rmsprop_alpha=float("nan")),
    dict(rmsprop_eps=0.0), dict(rmsprop_eps=-1e-8), dict(rmsprop_eps=float("nan")),
    dict(rmsprop_momentum=-0.1), dict(rmsprop_momentum=1.0), dict(rmsprop_momentum=float("nan")),
]


@pytest.mark.parametrize("bad", BAD, ids=lambda d: "-".join(f"{k}={v}" for k, v in d.items()))
def test_create_rejects_invalid_optimiser_options_before_the_device_check(fi, bad):
    """Checked before fi_learner_create looks for a CUDA device, so the refusal is the same with or without one."""
    from freeimpala_b200 import _lib
    lib = fi.load_library()
    cfg = _lib.FiLearnerConfig()
    lib.fi_learner_config_default(C.byref(cfg))
    cfg.num_players, cfg.buffer_capacity, cfg.entry_size, cfg.batch_size = 1, 4, 5, 2
    cfg.optimizer = _lib.OPT["rmsprop"]
    for k, v in bad.items():
        setattr(cfg, k, v)
    assert not lib.fi_learner_create(C.byref(cfg))
    msg = _lib.last_error()
    assert msg.startswith("fi_learner_create: ") and "no CUDA device" not in msg, msg
    assert any(w in msg for w in ("unknown optimizer", "max_grad_norm", "RMSProp options")), msg


def test_learner_keywords_reach_the_config(fi):
    """Learner(...) maps its keywords onto the appended fields (an invalid one is refused by the library)."""
    with pytest.raises(fi.FiError, match="max_grad_norm"):
        fi.Learner(1, 4, 5, 2, optimizer="rmsprop", max_grad_norm=-3.0)
    with pytest.raises(fi.FiError, match="RMSProp options"):
        fi.Learner(1, 4, 5, 2, optimizer="rmsprop", rmsprop_momentum=1.0)
