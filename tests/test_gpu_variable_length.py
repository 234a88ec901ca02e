"""Variable-length trajectories in the actor-critic V-trace step on the GPU (fi_learner_config.variable_length, record word 183,
include/fi_learner.h). Needs a B200.

  * the length-aware loss head alone (fi_op_vtrace_loss_head_opts) against the float64 reference, with NaN / +-inf / 1e30
    in the head rows and records past each trajectory's length;
  * two length learners whose batches differ only in the records past the lengths (zeros against garbage): bit-identical
    in every GEMM mode and through the replayed graph;
  * a length learner at full length against a non-length learner: bit-identical; a non-length learner never reads word 183;
  * the length learner's step against the float64 reference of tests/length_reference.py, as tests/test_gpu_legal_actions.py
    checks the masked step, and a T = 100 learner on 37-step trajectories against the oracle run at T = 37;
  * the threaded harness with --variable-length --sample-actions.
"""
import json
import os
import subprocess

import numpy as np
import pytest

import _util as U
import length_reference as R
import test_gpu_ac_paths as P
import test_gpu_legal_actions as GL
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
A = po.NUM_ACTIONS
MODES = ["simt", "tcgen05", "tcgen05_f16", "auto"]


def _random_lengths(seed, m, t):
    """Random length words: lengths 1 and t among uniform ones, some full lengths written as W = 0 or W > t."""
    rng = np.random.default_rng(seed)
    L = rng.integers(1, t + 1, size=m)
    L[0], L[-1] = 1, t
    words = L.astype(np.uint32)
    words[(L == t) & (np.arange(m) % 2 == 0)] = 0
    words[(L == t) & (np.arange(m) % 2 == 1)] = t + 1 + np.arange(m)[(L == t) & (np.arange(m) % 2 == 1)]
    return words


# ------------------------------------------------------------------------------- 1. the loss head alone
def _edge_lengths(t):
    """1, t and each side of every 32-step chunk edge below t."""
    return sorted({1, t} | {x for e in range(32, t, 32) for x in (e - 1, e, e + 1) if 1 <= x <= t})


@pytest.mark.parametrize("legal", [False, True])
@pytest.mark.parametrize("t", [1, 31, 32, 33, 100])
def test_length_loss_head_vs_reference(fi, oracle, t, legal):
    import torch
    lens = _edge_lengths(t)
    m = len(lens) + 2
    L = np.array(lens + [t, t], np.int64)
    words = L.astype(np.uint32)
    words[-2], words[-1] = 0, t + 7          # full length written both other ways
    rng = np.random.default_rng(t)
    obs, mu, act, rew, disc, boot = U.vtrace_batch(60 + t, m, t, done_p=0.05)
    lw = GL._legal_words(t, act) if legal else None
    head = rng.standard_normal((m * t, 17)).astype(np.float32)
    cfg = {k: float(np.float32(v)) for k, v in P.C1.items()}
    want = R.vtrace_losses_length(oracle, head[:, :16].reshape(m, t, A), head[:, 16].reshape(m, t), mu, act, rew, disc, boot,
                                  lw, L, **cfg)
    past = ~R.valid_rows(L, t).reshape(-1)
    fills = np.array([np.nan, np.inf, -np.inf, 1e30], np.float32)
    head[past] = fills[np.arange(int(past.sum()))[:, None] % 4 + np.zeros((1, 17), np.int64)]
    batch = R.pack_length_slots(obs, mu, act, rew, disc, boot, words, legal=lw, pad="garbage")
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    d_batch, d_head = dev(batch), dev(head)
    dhead = torch.full((m * t, 17), 7.0, device="cuda")
    vs, adv = torch.full((m * t,), 7.0, device="cuda"), torch.full((m * t,), 7.0, device="cuda")
    losses = torch.zeros(4, dtype=torch.float64, device="cuda")
    fi.ops.vtrace_loss_head(d_batch.data_ptr(), m, t, d_head.data_ptr(), 17, dhead.data_ptr(), losses.data_ptr(),
                            vs.data_ptr(), adv.data_ptr(), stream=torch.cuda.current_stream().cuda_stream, legal_mask=legal,
                            lengths=True, **P.C1)
    torch.cuda.synchronize()
    got, got_losses, got_vs, got_adv = dhead.cpu().numpy(), losses.cpu().numpy(), vs.cpu().numpy(), adv.cpu().numpy()
    for name, a in (("losses", got_losses), ("dhead", got), ("vs", got_vs), ("pg_adv", got_adv)):
        assert np.all(np.isfinite(a)), name
    assert np.all(got[past] == 0.0) and np.all(got_vs[past] == 0.0) and np.all(got_adv[past] == 0.0)
    dl = want["dlogits"].reshape(-1, A)
    errs = dict(vs=U.rel_max(got_vs, want["vs"]), pg_adv=U.rel_max(got_adv, want["pg_adv"]),
                dlogits=U.rel_max(got[:, :16], dl), dvalue=U.rel_max(got[:, 16], want["dvalue"].reshape(-1)))
    print(f"length loss head m={m} t={t} legal={legal}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    # the policy-gradient sum cancels (test_gpu_kernels.py test_vtrace_loss_head_vs_oracle): 1e-5 of the largest term sum
    atol = 1e-6 * (np.abs(want["losses"][1:]).sum() + 1.0)
    np.testing.assert_allclose(got_losses, want["losses"], rtol=1e-5, atol=atol)
    assert all(e < 1e-5 for e in errs.values()), errs


# ------------------------------------------------------------------------------- 2. independence from the padding bytes
def _pair(fi, m, t, gemm_mode, params, on_kw, off_kw):
    a = P._ac(fi, m, t, gemm_mode=gemm_mode, **on_kw)
    b = P._ac(fi, m, t, gemm_mode=gemm_mode, **off_kw)
    a.set_params(0, params)
    b.set_params(0, params)
    return a, b


def _garbage_in_word_183(slots, m, t, seed):
    """Word 183 of every record but record 0 is not read: random bits there."""
    w = slots.view(np.uint32).reshape(m, t, po.REC_WORDS)
    w[:, 1:, 183] = np.random.default_rng(seed).integers(0, 1 << 32, size=(m, t - 1), dtype=np.uint64).astype(np.uint32)
    return slots


def _assert_same_steps(a, b, batches_a, batches_b, graph, what):
    for s, (xa, xb) in enumerate(zip(batches_a, batches_b)):
        if graph:
            a.trainModel(0, a.stage_batch(0, xa))
            b.trainModel(0, b.stage_batch(0, xb))
        else:
            a.forward_backward(0, a.stage_batch(0, xa))
            b.forward_backward(0, b.stage_batch(0, xb))
            assert np.all(np.isfinite(a.last_losses(0)))
            assert np.array_equal(a.get_grads(0), b.get_grads(0)), (what, s)
            a.apply_update(0)
            b.apply_update(0)
        np.testing.assert_allclose(a.last_losses(0), b.last_losses(0), rtol=1e-12, atol=0, err_msg=f"{what} {s}")
        assert np.array_equal(a.get_params(0), b.get_params(0)), (what, s)


@pytest.mark.parametrize("gemm_mode", MODES)
def test_padding_bytes_change_nothing(fi, gemm_mode):
    """3 steps of forward_backward + apply_update: records past L zero in one batch, NaN / +-inf / 1e30 / random bits in the
    other (and random bits in word 183 of records 1..L-1): losses (rtol 1e-12, double atomics), gradients and parameters
    bit-identical."""
    m, t = 8, 40
    a, b = _pair(fi, m, t, gemm_mode, U.ac_params(5050), dict(variable_length=True), dict(variable_length=True))
    try:
        za, zb = [], []
        for s in range(3):
            data = P._batch(730 + s, m, t)
            words = _random_lengths(40 + s, m, t)
            za.append(R.pack_length_slots(*data, words, pad="zeros"))
            zb.append(_garbage_in_word_183(R.pack_length_slots(*data, words, pad="garbage"), m, t, s))
        _assert_same_steps(a, b, za, zb, False, gemm_mode)
    finally:
        a.close()
        b.close()


def test_padding_bytes_change_nothing_in_the_replayed_graph(fi):
    """The same through fi_learner_step for 5 steps (auto): from the third step on each step is one replayed CUDA graph."""
    m, t = 16, 20
    a, b = _pair(fi, m, t, "auto", U.ac_params(5051), dict(variable_length=True), dict(variable_length=True))
    try:
        za, zb = [], []
        for s in range(5):
            data = P._batch(740 + s, m, t)
            words = _random_lengths(50 + s, m, t)
            za.append(R.pack_length_slots(*data, words, pad="zeros"))
            zb.append(R.pack_length_slots(*data, words, pad="garbage"))
        _assert_same_steps(a, b, za, zb, True, "graph")
    finally:
        a.close()
        b.close()


# ------------------------------------------------------------------------------- 3. no change at full length
@pytest.mark.parametrize("gemm_mode", MODES)
def test_full_length_words_give_the_fixed_length_step(fi, gemm_mode):
    """Every W in {0, t}: the length learner and a non-length learner bit-identical over 3 steps."""
    m, t = 8, 40
    a, b = _pair(fi, m, t, gemm_mode, U.ac_params(5052), dict(variable_length=True), {})
    try:
        xa, xb = [], []
        for s in range(3):
            data = P._batch(750 + s, m, t)
            words = np.where(np.arange(m) % 2 == 0, 0, t).astype(np.uint32)
            xa.append(R.pack_length_slots(*data, words))
            xb.append(po.pack_vtrace_slots(*data))
        _assert_same_steps(a, b, xa, xb, False, gemm_mode)
    finally:
        a.close()
        b.close()


def test_full_length_words_give_the_fixed_length_step_in_the_replayed_graph(fi):
    m, t = 16, 20
    a, b = _pair(fi, m, t, "auto", U.ac_params(5053), dict(variable_length=True, legal_action_mask=True),
                 dict(legal_action_mask=True))
    try:
        xa, xb = [], []
        for s in range(5):
            data = P._batch(760 + s, m, t)
            lw = GL._legal_words(s, data[2])
            xa.append(R.pack_length_slots(*data, np.zeros(m, np.uint32), legal=lw))
            xb.append(R.LR.pack_vtrace_slots_legal(*data, lw))
        _assert_same_steps(a, b, xa, xb, True, "graph")
    finally:
        a.close()
        b.close()


@pytest.mark.parametrize("gemm_mode", MODES)
def test_fixed_length_learner_ignores_word_183(fi, gemm_mode):
    """Garbage in word 183 (random lengths among random bit patterns) of a non-length learner's records changes nothing."""
    m, t = 8, 40
    L = P._ac(fi, m, t, gemm_mode=gemm_mode)
    try:
        L.set_params(0, U.ac_params(5054))
        data = P._batch(770, m, t)
        L.forward_backward(0, L.stage_batch(0, po.pack_vtrace_slots(*data)))
        losses, grads = L.last_losses(0), L.get_grads(0)
        slots = po.pack_vtrace_slots(*data)
        w = slots.view(np.uint32).reshape(m, t, po.REC_WORDS)
        w[:, :, 183] = np.random.default_rng(2).integers(0, 1 << 32, size=(m, t), dtype=np.uint64).astype(np.uint32)
        w[:, 0, 183] = np.arange(1, m + 1)
        L.forward_backward(0, L.stage_batch(0, slots))
        np.testing.assert_allclose(L.last_losses(0), losses, rtol=1e-12, atol=0)
        assert np.array_equal(L.get_grads(0), grads)
    finally:
        L.close()


# ------------------------------------------------------------------------------- 4. the step against the reference
def _length_step_and_check(oracle, L, O, F, cfg, data, words, legal, s, case, worst):
    """test_gpu_legal_actions.py _masked_step_and_check with length words and tests/length_reference.py as the reference."""
    obs, mu, act, rew, disc, boot = data
    m, t = act.shape
    lens = R.lengths_of(words, t)
    want_free, g_free, _, _ = R.ac_loss_grad_length(oracle, F.params(), *data, legal, lens, **cfg)
    F.set_grads(g_free)
    L.forward_backward(0, L.stage_batch(0, R.pack_length_slots(*data, words, legal=legal, pad="garbage")))
    got = L.last_losses(0)
    assert np.all(np.isfinite(got)), (case, s, got)
    masks = L.debug_relu_masks(0, m * t)
    want, g_want, n_over, max_over = R.ac_loss_grad_length(oracle, O.params(), *data, legal, lens, relu_mask=masks, **cfg)
    assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (case, s, n_over, max_over)
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


def _run_vs_reference(fi, oracle, gemm_mode, m, t, case, make_words, legal=False, steps=2):
    params = U.ac_params(6000 + m * t)
    L = P._ac(fi, m, t, gemm_mode=gemm_mode, variable_length=True, legal_action_mask=legal)
    try:
        L.set_params(0, params)
        O = oracle.actor_critic(params, lr=P.LR)
        F = oracle.actor_critic(params, lr=P.LR)
        parity, worst = U.AdamParity(O, F), P.Worst()
        for s in range(steps):
            data = P._batch(900 + 10 * m + s, m, t)
            lw = GL._legal_words(950 + s, data[2]) if legal else None
            grads = _length_step_and_check(oracle, L, O, F, {}, data, make_words(s, m, t), lw, s, case, worst)
            L.apply_update(0)
            parity.step(grads)
        e_forced, e_trim, e_free = parity.check(L.get_params(0), P.TOL)
        print(f"ac [{case}] {m} x {t} [{gemm_mode}]: worst loss {worst.loss:.2e}, grads {worst.grad:.2e}, ReLU overrides "
              f"{worst.n_over} (max |z|/rms {worst.max_over:.1e}); params teacher-forced {e_forced:.2e}, free-running "
              f"{e_free:.2e} (trimmed {e_trim:.2e})")
    finally:
        L.close()


@pytest.mark.parametrize("m,t", [(4, 7), (9, 33), (64, 100)])
@pytest.mark.parametrize("gemm_mode", MODES)
def test_length_step_vs_reference(fi, oracle, gemm_mode, m, t):
    _run_vs_reference(fi, oracle, gemm_mode, m, t, "random lengths", lambda s, m, t: _random_lengths(960 + s, m, t))


@pytest.mark.parametrize("gemm_mode", MODES)
def test_length_step_all_length_one(fi, oracle, gemm_mode):
    _run_vs_reference(fi, oracle, gemm_mode, 64, 100, "all L = 1", lambda s, m, t: np.ones(m, np.uint32))


@pytest.mark.parametrize("gemm_mode", MODES)
def test_length_step_with_legal_mask(fi, oracle, gemm_mode):
    _run_vs_reference(fi, oracle, gemm_mode, 9, 33, "random lengths + legal", lambda s, m, t: _random_lengths(970 + s, m, t),
                      legal=True)


def test_length_step_at_the_split_k_shape(fi, oracle):
    """37 x 64 = 2368 rows (test_gpu_ac_paths.py rederive-rows2368): 9 split-K slabs re-derived to 8."""
    _run_vs_reference(fi, oracle, "auto", 37, 64, "rows 2368", lambda s, m, t: _random_lengths(980 + s, m, t))


# ------------------------------------------------------------------------------- 5. truncation
@pytest.mark.parametrize("gemm_mode", ["simt", "auto"])
def test_truncated_trajectories_match_the_oracle_at_their_length(fi, oracle, gemm_mode):
    """A T = 100 learner on trajectories of L = 37 (garbage past step 37) against the C oracle run on those trajectories at
    T = 37, fed the CUDA run's ReLU decisions of the valid rows: losses, gradients and parameters after 2 steps."""
    m, t, n = 8, 100, 37
    params = U.ac_params(7037)
    L = P._ac(fi, m, t, gemm_mode=gemm_mode, variable_length=True)
    try:
        L.set_params(0, params)
        O, F = oracle.actor_critic(params, lr=P.LR), oracle.actor_critic(params, lr=P.LR)
        parity, worst = U.AdamParity(O, F), P.Worst()
        for s in range(2):
            data = P._batch(990 + s, m, t)
            cut = tuple(np.ascontiguousarray(x[:, :n]) for x in data[:5]) + (data[5],)
            want_free = F.loss_grad(*cut)
            L.forward_backward(0, L.stage_batch(0, R.pack_length_slots(*data, np.full(m, n, np.uint32), pad="garbage")))
            got = L.last_losses(0)
            masks = L.debug_relu_masks(0, m * t).reshape(5, m, t, 512)[:, :, :n].reshape(5, -1)
            want, n_over, max_over = O.loss_grad_masked(*cut, masks)
            assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (s, n_over, max_over)
            atol = 1e-6 * abs(want[0])
            np.testing.assert_allclose(got, want, rtol=P.TOL, atol=atol)
            np.testing.assert_allclose(got, want_free, rtol=P.TOL if s == 0 else 1e-3, atol=atol)
            grads = L.get_grads(0)
            e = U.rel_l2(grads, O.grads())
            assert e < P.TOL, (s, e)
            L.apply_update(0)
            parity.step(grads)
        e_forced = parity.check(L.get_params(0), P.TOL)[0]
        print(f"ac [truncated 37 of 100] [{gemm_mode}]: grads {e:.2e}, params teacher-forced {e_forced:.2e}")
    finally:
        L.close()


# ------------------------------------------------------------------------------- 6. the harness
def test_harness_variable_length_with_sampled_actions(fi):
    """Each trajectory L uniform in 1..game_steps, only L records written (the slots' older tails stay): every update
    runs, no sampled action is illegal, and the sampled rows are exactly the transitions written."""
    from freeimpala_b200 import build
    args = ["-p", 2, "-B", 8, "-M", 4, "-a", 8, "-T", 3, "-S", 40, "--game-steps", 30, "--agent-time", 0,
            "--variable-length", "--sample-actions"]
    assert os.path.exists(build.HOST_BIN)
    r = subprocess.run([build.HOST_BIN, *map(str, args)], capture_output=True, text=True, timeout=300)
    line = [x for x in r.stdout.splitlines() if x.startswith("{")]
    assert r.returncode == 0 and line, r.stderr[-2000:]
    out = json.loads(line[-1])
    trajectories = 8 * 3 * 2
    assert out["learner_updates"] == out["expected_updates"] == 2 * (8 * 3 // 4)
    assert out["illegal_actions"] == 0
    assert out["valid_transitions"] == out["actor_sampled_rows"]
    assert trajectories <= out["valid_transitions"] < trajectories * 30
