"""Legal-action masking of the actor-critic V-trace step on the GPU (fi_learner_config.legal_action_mask, record word 182,
include/fi_learner.h). Needs a B200.

  * the masked loss head alone (fi_op_vtrace_loss_head_legal) against the float64 reference, with forced moves and NaN / -inf
    in the logits outside the support;
  * a masking learner whose every word is 0xFFFF against a non-masking one: the same step, bit for bit, on the three
    launches of the loss head in ac_forward_backward (simt, tcgen05, tcgen05_f16 / auto) and through the replayed graph;
  * the masking learner step against the float64 reference of tests/legal_reference.py, teacher-forced and free-running,
    as tests/test_gpu_ac_paths.py checks the unmasked step against the oracle;
  * a non-masking learner never reads word 182.
"""
import numpy as np
import pytest

import _util as U
import legal_reference as R
import test_gpu_ac_paths as P
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
A = po.NUM_ACTIONS
MODES = ["simt", "tcgen05", "tcgen05_f16", "auto"]


def _legal_words(seed, act):
    """Random legal words: about one transition in six (and always the first) a forced move (word 0), one in six (and always
    the last) a word without the taken action's bit, one in six with bits 16..31 set; the rest random 16-bit sets that
    contain the action."""
    rng = np.random.default_rng(seed)
    a = act.astype(np.uint32)
    legal = rng.integers(0, 1 << 16, size=act.shape).astype(np.uint32) | (np.uint32(1) << a)
    kind = rng.integers(0, 6, size=act.shape)
    legal[kind == 0] = 0
    legal[kind == 1] &= ~(np.uint32(1) << a[kind == 1])
    legal[kind == 2] |= rng.integers(1, 1 << 16, size=int((kind == 2).sum())).astype(np.uint32) << np.uint32(16)
    legal.flat[0] = 0                                            # at least one forced move, even in a 6-transition batch
    legal.flat[-1] &= ~(np.uint32(1) << a.flat[-1])              # and one word without the action's bit
    return legal


# ------------------------------------------------------------------------------- A. the loss head alone
@pytest.mark.parametrize("t", [1, 32, 33, 100])
@pytest.mark.parametrize("fill", ["finite", "nan", "-inf"])
def test_masked_loss_head_vs_oracle(fi, oracle, t, fill):
    """t = 1 (every 32-step chunk is one step), 32 (one exact chunk), 33 (ends in a 1-step chunk), 100. Outside the support
    the head and behaviour logits hold `fill`: the outputs must not see it, d(head) there is exactly 0."""
    import torch
    m = 6
    rng = np.random.default_rng(t)
    obs, mu, act, rew, disc, boot = U.vtrace_batch(50 + t, m, t, done_p=0.05)
    legal = _legal_words(t, act)
    sup = R.support(legal, act)
    head = rng.standard_normal((m * t, 17)).astype(np.float32)
    cfg = {k: float(np.float32(v)) for k, v in P.C1.items()}
    want = R.vtrace_losses_legal(oracle, head[:, :16].reshape(m, t, A), head[:, 16].reshape(m, t), mu, act, rew, disc,
                                 boot, legal, **cfg)
    clean = head.copy()
    if fill != "finite":
        v = np.float32(np.nan if fill == "nan" else -np.inf)
        head[:, :16][~sup.reshape(-1, A)] = v
        mu = mu.copy()
        mu[~sup] = v
    batch = R.pack_vtrace_slots_legal(obs, mu, act, rew, disc, boot, legal)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    d_batch, d_head = dev(batch), dev(head)
    dhead = torch.full((m * t, 17), 7.0, device="cuda")
    vs, adv = torch.zeros(m * t, device="cuda"), torch.zeros(m * t, device="cuda")
    losses = torch.zeros(4, dtype=torch.float64, device="cuda")
    fi.ops.vtrace_loss_head(d_batch.data_ptr(), m, t, d_head.data_ptr(), 17, dhead.data_ptr(), losses.data_ptr(),
                            vs.data_ptr(), adv.data_ptr(), stream=torch.cuda.current_stream().cuda_stream, legal_mask=True,
                            **P.C1)
    torch.cuda.synchronize()
    got, got_losses, got_vs, got_adv = dhead.cpu().numpy(), losses.cpu().numpy(), vs.cpu().numpy(), adv.cpu().numpy()
    for name, a in (("losses", got_losses), ("dhead", got), ("vs", got_vs), ("pg_adv", got_adv)):
        assert np.all(np.isfinite(a)), name
    assert np.all(got[:, :16][~sup.reshape(-1, A)] == 0.0)
    forced = sup.reshape(-1, A).sum(-1) == 1
    assert forced.any() and np.all(got[forced, :16] == 0.0)
    # a loss is held to 1e-5 relative but never to less than 1e-7 of its summed term magnitudes (the policy-gradient sum
    # cancels; test_gpu_kernels.py test_vtrace_loss_head_vs_oracle says why)
    z = np.where(sup, clean[:, :16].reshape(m, t, A).astype(np.float64), -np.inf)
    logp = z - (z.max(-1, keepdims=True) + np.log(np.exp(z - z.max(-1, keepdims=True)).sum(-1, keepdims=True)))
    pg_abs = np.abs(np.take_along_axis(logp, act[..., None].astype(np.int64), -1)[..., 0] * want["pg_adv"]).sum()
    bl, ent = abs(want["losses"][2]), abs(want["losses"][3])    # one sign each: no cancellation
    magnitude = np.array([pg_abs + cfg["baseline_cost"] * bl + cfg["entropy_cost"] * ent, pg_abs, bl, ent])
    dl = want["dlogits"].reshape(-1, A)
    loss_tol = 1e-5 * np.maximum(np.abs(want["losses"]), magnitude / 100)
    errs = dict(vs=U.rel_max(got_vs, want["vs"]), pg_adv=U.rel_max(got_adv, want["pg_adv"]),
                dlogits=U.rel_max(got[:, :16], dl), dvalue=U.rel_max(got[:, 16], want["dvalue"].reshape(-1)))
    print(f"masked loss head m={m} t={t} fill {fill}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()) +
          f", forced moves {int(forced.sum())} of {m * t}")
    assert np.all(np.abs(got_losses - want["losses"]) <= loss_tol), (got_losses, want["losses"], loss_tol)
    assert all(e < 1e-5 for e in errs.values()), errs


# ------------------------------------------------------------------------------- B. all legal = no mask
def _pair_of_learners(fi, m, t, gemm_mode, params):
    on = P._ac(fi, m, t, gemm_mode=gemm_mode, legal_action_mask=True)
    off = P._ac(fi, m, t, gemm_mode=gemm_mode)
    on.set_params(0, params)
    off.set_params(0, params)
    return on, off


@pytest.mark.parametrize("gemm_mode", MODES)
def test_all_legal_words_give_the_unmasked_step(fi, gemm_mode):
    """Every word 0xFFFF (bits 16..31 random, they are ignored): 3 steps of forward_backward + apply_update, the masking and
    the non-masking learner bit-identical in gradients and parameters. The losses are sums of double atomics in a varying
    order, so they are held to rtol 1e-12."""
    m, t = 8, 40
    on, off = _pair_of_learners(fi, m, t, gemm_mode, U.ac_params(4040))
    try:
        for s in range(3):
            data = P._batch(700 + s, m, t)
            words = np.uint32(0xFFFF) | (np.random.default_rng(s).integers(0, 1 << 16, size=(m, t)).astype(np.uint32) << 16)
            on.forward_backward(0, on.stage_batch(0, R.pack_vtrace_slots_legal(*data, words)))
            off.forward_backward(0, off.stage_batch(0, po.pack_vtrace_slots(*data)))
            np.testing.assert_allclose(on.last_losses(0), off.last_losses(0), rtol=1e-12, atol=0)
            assert np.array_equal(on.get_grads(0), off.get_grads(0)), (gemm_mode, s)
            on.apply_update(0)
            off.apply_update(0)
            assert np.array_equal(on.get_params(0), off.get_params(0)), (gemm_mode, s)
    finally:
        on.close()
        off.close()


def test_all_legal_words_give_the_unmasked_step_in_the_replayed_graph(fi):
    """The same through fi_learner_step for 5 steps (auto): from the third step on each step is one replayed CUDA graph."""
    m, t = 16, 20
    on, off = _pair_of_learners(fi, m, t, "auto", U.ac_params(4041))
    try:
        for s in range(5):
            data = P._batch(710 + s, m, t)
            on.trainModel(0, on.stage_batch(0, R.pack_vtrace_slots_legal(*data, np.full((m, t), 0xFFFF, np.uint32))))
            off.trainModel(0, off.stage_batch(0, po.pack_vtrace_slots(*data)))
            np.testing.assert_allclose(on.last_losses(0), off.last_losses(0), rtol=1e-12, atol=0)
            assert np.array_equal(on.get_params(0), off.get_params(0)), s
    finally:
        on.close()
        off.close()


# ------------------------------------------------------------------------------- C. masked step vs the oracle
def _masked_step_and_check(oracle, L, O, F, cfg, data, legal, s, case, worst):
    """test_gpu_ac_paths.py _step_and_check with the legal words in the records and the masked float64 reference of
    tests/legal_reference.py at the parameters of the teacher-forced O (fed the CUDA run's ReLU decisions) and of the
    free-running F (whose gradient it sets for F's next update)."""
    obs, mu, act, rew, disc, boot = data
    m, t = act.shape
    want_free, g_free, _, _ = R.ac_loss_grad_legal(oracle, F.params(), *data, legal, **cfg)
    F.set_grads(g_free)
    L.forward_backward(0, L.stage_batch(0, R.pack_vtrace_slots_legal(*data, legal)))
    got = L.last_losses(0)
    assert np.all(np.isfinite(got)), (case, s, got)
    masks = L.debug_relu_masks(0, m * t)
    want, g_want, n_over, max_over = R.ac_loss_grad_legal(oracle, O.params(), *data, legal, relu_mask=masks, **cfg)
    assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (case, s, n_over, max_over)
    # the total sums terms of both signs: with forced moves and small legal sets the entropy sum grows and the total can
    # cancel ~200-fold (-1.13 out of terms of 87, 113 and 27), below what fp32 terms can give to 1e-5 of itself, so it
    # is held to 1e-6 of the summed magnitudes of its three terms
    atol = 1e-6 * max(abs(want[0]), abs(want[1]) + cfg.get("baseline_cost", 0.5) * abs(want[2]) +
                      cfg.get("entropy_cost", 0.01) * abs(want[3]))
    np.testing.assert_allclose(got, want, rtol=P.TOL, atol=atol, err_msg=f"{case} step {s}: teacher-forced reference")
    np.testing.assert_allclose(got, want_free, rtol=P.TOL if s == 0 else 1e-3, atol=atol,
                               err_msg=f"{case} step {s}: free-running reference")
    grads = L.get_grads(0)
    e = U.rel_l2(grads, g_want)
    assert e < P.TOL, (case, s, e)
    worst.loss = max(worst.loss, float(np.max(np.abs(got - want) / np.maximum(np.abs(want), atol))))
    worst.grad = max(worst.grad, e)
    worst.n_over, worst.max_over = max(worst.n_over, n_over), max(worst.max_over, max_over)
    return grads


@pytest.mark.parametrize("cfg_name", ["defaults", "c1-distinct"])
@pytest.mark.parametrize("m,t", [(4, 7), (9, 33), (64, 100)])
@pytest.mark.parametrize("gemm_mode", MODES)
def test_masked_step_vs_oracle(fi, oracle, gemm_mode, m, t, cfg_name):
    cfg = P.C1 if cfg_name == "c1-distinct" else {}
    case = f"legal {cfg_name}"
    params = U.ac_params(3000 + m * t)
    L = P._ac(fi, m, t, gemm_mode=gemm_mode, legal_action_mask=True, **cfg)
    try:
        L.set_params(0, params)
        O = oracle.actor_critic(params, lr=P.LR, **P._oracle_cfg(cfg))
        F = oracle.actor_critic(params, lr=P.LR, **P._oracle_cfg(cfg))
        parity, worst = U.AdamParity(O, F), P.Worst()
        for s in range(2):
            data = P._batch(800 + 10 * m + s, m, t)
            legal = _legal_words(900 + s, data[2])
            grads = _masked_step_and_check(oracle, L, O, F, P._oracle_cfg(cfg), data, legal, s, case, worst)
            L.apply_update(0)
            parity.step(grads)
        e_forced, e_trim, e_free = parity.check(L.get_params(0), P.TOL)
        print(f"ac [{case}] {m} x {t} [{gemm_mode}]: worst loss {worst.loss:.2e}, grads {worst.grad:.2e}, ReLU overrides "
              f"{worst.n_over} (max |z|/rms {worst.max_over:.1e}); params teacher-forced {e_forced:.2e}, free-running "
              f"{e_free:.2e} (trimmed {e_trim:.2e})")
    finally:
        L.close()


# ------------------------------------------------------------------------------- D. mask off ignores word 182
@pytest.mark.parametrize("gemm_mode", MODES)
def test_unmasked_learner_ignores_word_182(fi, gemm_mode):
    """Garbage in word 182 (random bit patterns, NaNs among them) of a non-masking learner's records changes nothing: the
    gradients are bit-identical to those of the same batch with the word 0 (losses: rtol 1e-12, double atomics)."""
    m, t = 8, 40
    L = P._ac(fi, m, t, gemm_mode=gemm_mode)
    try:
        L.set_params(0, U.ac_params(4042))
        data = P._batch(720, m, t)
        L.forward_backward(0, L.stage_batch(0, po.pack_vtrace_slots(*data)))
        losses, grads = L.last_losses(0), L.get_grads(0)
        garbage = np.random.default_rng(1).integers(0, 1 << 32, size=(m, t), dtype=np.uint64).astype(np.uint32)
        garbage[::3] = np.float32(np.nan).view(np.uint32)
        L.forward_backward(0, L.stage_batch(0, R.pack_vtrace_slots_legal(*data, garbage)))
        np.testing.assert_allclose(L.last_losses(0), losses, rtol=1e-12, atol=0)
        assert np.array_equal(L.get_grads(0), grads)
    finally:
        L.close()
