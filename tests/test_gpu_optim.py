"""RMSProp, global-norm gradient clipping and the per-player learning rate on the B200. Needs a GPU.

  * the two kernels through the operator layer: RMSProp bit-exact against the oracle's fp32 restatement of the kernel, the
    norm within 1e-12 of numpy's float64 norm and its clip coefficient equal to the formula, run to run bit-identical;
  * the learner step (forward_backward + apply_update) against the float64 oracle for every optimiser with clipping off,
    inactive and active, on both models; the teacher-forced pattern of tests/_util.py AdamParity;
  * what must be bit-identical: clipping that never triggers vs none, graph-replayed vs stream-launched steps, lr = 0;
  * the learning-rate schedule, checkpoints with RMSProp state, and loading across optimiser families.
"""
import os
import tempfile

import numpy as np
import pytest

import _util as U
import optim_reference as R
from oracle import pyoracle as po
from test_gpu_farmer_paths import KINK_GRAD_TOL, KINK_REL, KINK_UNITS, _kink_signature

pytestmark = pytest.mark.gpu
TOL = 1e-5
# name -> (fi_opt_kind, learning rate, RMSProp eps, RMSProp momentum)
OPTS = {
    "adam": ("adam", 5e-4, 1e-8, 0.0),
    "adamw": ("adamw", 5e-4, 1e-8, 0.0),
    "sgd": ("sgd", 1e-2, 1e-8, 0.0),
    "rmsprop": ("rmsprop", 2e-4, 1e-8, 0.0),
    "rmsprop-mom": ("rmsprop", 2e-4, 0.01, 0.9),   # the IMPALA paper's setting: eps 0.01, here with momentum
}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _learner(fi, model, m, t, opt="adam", max_grad_norm=0.0, gemm_mode="auto", **kw):
    kind, lr, eps, mom = OPTS[opt]
    return fi.Learner(1, max(m, 2), t, m, 0, 0, kw.pop("ckpt", ""), "", 0, model=model, optimizer=kind, lr=lr,
                      max_grad_norm=max_grad_norm, rmsprop_eps=eps, rmsprop_momentum=mom, gemm_mode=gemm_mode, **kw)


def _slots(model, seed, m, t):
    if model == "farmer_lstm":
        return po.pack_farmer_slots(*U.farmer_batch(seed, m, t))
    return po.pack_vtrace_slots(*U.vtrace_batch(seed, m, t))


def _params(model, seed):
    return U.farmer_params(seed) if model == "farmer_lstm" else U.ac_params(seed)


# ------------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("coef", [None, 0.37], ids=["coef-null", "coef-0.37"])
@pytest.mark.parametrize("momentum", [0.0, 0.9])
@pytest.mark.parametrize("n", [3, 10007, 1142801, 1514497])
def test_rmsprop_kernel_bit_exact_vs_f32_restatement(fi, oracle, torch_cuda, n, momentum, coef):
    torch = torch_cuda
    rng = np.random.default_rng(n + int(10 * momentum))
    eps = 1e-8 if momentum == 0.0 else 0.01
    p = rng.standard_normal(n).astype(np.float32)
    sa, buf = np.zeros(n, np.float32), np.zeros(n, np.float32)
    dp, dsa, dbuf = _dev(torch, p), _dev(torch, sa), _dev(torch, buf)
    dcoef = _dev(torch, np.array([coef], np.float32)) if coef is not None else None
    st = torch.cuda.current_stream().cuda_stream
    for step in range(4):
        g = (rng.standard_normal(n) * 10.0 ** rng.integers(-4, 2)).astype(np.float32)
        dg = _dev(torch, g)
        fi.ops.rmsprop(1e-3, n, dp.data_ptr(), dg.data_ptr(), dsa.data_ptr(), dbuf.data_ptr() if momentum else None,
                       alpha=0.99, eps=eps, momentum=momentum, coef=dcoef.data_ptr() if dcoef is not None else None, stream=st)
        R.rmsprop_f32(1e-3, 0.99, eps, momentum, p, g, sa, buf if momentum else None, gscale=1.0 if coef is None else coef)
    torch.cuda.synchronize()
    assert np.array_equal(dp.cpu().numpy(), p)
    assert np.array_equal(dsa.cpu().numpy(), sa)
    assert np.array_equal(dbuf.cpu().numpy(), buf)    # untouched (zeros) without momentum


@pytest.mark.parametrize("mag", [1e-20, 1.0, 1e20])
@pytest.mark.parametrize("n", [3, 4099, 1142801, 1514497, 64 << 20])
def test_grad_norm_clip_kernel(fi, torch_cuda, n, mag):
    torch = torch_cuda
    rng = np.random.default_rng(n % 1000 + int(np.log10(mag)) + 20)
    g = (rng.standard_normal(n, dtype=np.float32) * np.float32(mag)).astype(np.float32)
    want = float(np.linalg.norm(g.astype(np.float64)))
    dg = _dev(torch, g)
    del g
    st = torch.cuda.current_stream().cuda_stream
    out = []
    for max_norm in (0.5 * want, 0.5 * want, 2.0 * want):   # active twice (run-to-run identity), then inactive
        dn = torch.zeros(1, dtype=torch.float64, device="cuda")
        dc = torch.zeros(1, dtype=torch.float32, device="cuda")
        fi.ops.grad_norm_clip(n, dg.data_ptr(), max_norm, dn.data_ptr(), dc.data_ptr(), stream=st)
        torch.cuda.synchronize()
        norm, coef = float(dn.item()), dc.cpu().numpy()[0]
        assert abs(norm - want) <= 1e-12 * want, (norm, want)
        assert coef == np.float32(min(1.0, max_norm / (norm + 1e-6)))
        out.append((norm, coef))
    assert out[0] == out[1]          # deterministic: the same bits again
    assert out[0][1] < 1.0
    if want > 1e-3:                  # (below that the 1e-6 of the formula keeps even 2x the norm clipping)
        assert out[2][1] == np.float32(1.0)


def test_grad_norm_clip_rejects_bad_arguments(fi, torch_cuda):
    torch = torch_cuda
    g = torch.ones(64, device="cuda")
    dn = torch.zeros(1, dtype=torch.float64, device="cuda")
    dc = torch.zeros(1, dtype=torch.float32, device="cuda")
    for max_norm in (0.0, -1.0, float("inf")):
        with pytest.raises(fi.FiError):
            fi.ops.grad_norm_clip(64, g.data_ptr(), max_norm, dn.data_ptr(), dc.data_ptr())
    with pytest.raises(fi.FiError):
        fi.ops.grad_norm_clip(63, g.data_ptr() + 4, 1.0, dn.data_ptr(), dc.data_ptr())   # not 16-byte aligned


# ------------------------------------------------------------------------------- learner step vs the float64 oracle
SHAPES = [("mlp_actor_critic", 64, 100), ("mlp_actor_critic", 9, 33), ("farmer_lstm", 64, 100)]


@pytest.mark.parametrize("clip", ["off", "inactive", "active"])
@pytest.mark.parametrize("opt", list(OPTS))
@pytest.mark.parametrize("model,m,t", SHAPES, ids=[f"{a}-{m}x{t}" for a, m, t in SHAPES])
def test_learner_step_vs_oracle(fi, oracle, model, m, t, opt, clip):
    """3 steps of forward_backward + apply_update. Losses within 1e-5 of the teacher-forced oracle (the actor-critic's takes
    the CUDA run's ReLU decisions, as in test_gpu_learner.py), gradients within 1e-5, the teacher-forced parameters within
    1e-5 after the last update; the free-running oracle's parameter error is printed. grad_norm_at equals the float64 norm
    of the gradient arena. The bound: above every step's norm (inactive) or ~0.1x the first step's norm (active)."""
    farmer = model == "farmer_lstm"
    kind, lr, eps, mom = OPTS[opt]
    params = _params(model, 7)
    mk = (lambda: R.OptOracle.farmer(oracle, params, opt=kind, lr=lr)) if farmer else \
        (lambda: R.OptOracle.actor_critic(oracle, params, opt=kind, lr=lr))
    O, F = mk(), mk()      # teacher-forced (fed the CUDA gradients), free-running
    if farmer:
        batches = [U.farmer_batch(900 + s, m, t) for s in range(3)]
    else:
        batches = [U.vtrace_batch(900 + s, m, t, done_p=0.03) for s in range(3)]
    want_free = [F.loss_grad(*batches[0])]
    norm0 = float(np.linalg.norm(F.grads()))
    max_norm = {"off": 0.0, "inactive": 1e3 * norm0, "active": 0.1 * norm0}[clip]
    for X in (O, F):
        X.set_opt(lr, max_grad_norm=max_norm, rmsprop_eps=eps, rmsprop_momentum=mom)
    L = _learner(fi, model, m, t, opt, max_norm)
    try:
        L.set_params(0, params)
        e_loss = e_grad = 0.0
        for s, b in enumerate(batches):
            if s > 0:
                want_free.append(F.loss_grad(*b))
            params_before = O.params()
            L.forward_backward(0, L.stage_batch(0, po.pack_farmer_slots(*b) if farmer else po.pack_vtrace_slots(*b)))
            got = L.last_losses(0)
            if farmer:
                want = O.loss_grad(*b)
                assert abs(got[0] - want) <= TOL * abs(want) + 1e-7, (s, got[0], want)
                e_loss = max(e_loss, abs(got[0] - want) / abs(want))
            else:
                masks = L.debug_relu_masks(0, m * t)
                want, n_over, max_over = O.loss_grad_masked(*b, masks)
                assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (n_over, max_over)
                np.testing.assert_allclose(got, want, rtol=TOL, atol=1e-6 * abs(want[0]))
                e_loss = max(e_loss, float(np.abs(got - want).max() / np.abs(want).max()))
            grads = L.get_grads(0)
            e = U.rel_l2(grads, O.grads())
            if e >= TOL and farmer:   # the farmer oracle takes no ReLU overrides: only the kink signature may explain it
                n_flip, worst = _kink_signature(L, m, params_before, *b[:2])
                print(f"[{model} {m}x{t} {opt} clip={clip}] step {s}: grads {e:.2e} with {n_flip} ReLU kinks ({worst:.1e})")
                assert 0 < n_flip <= KINK_UNITS and worst < KINK_REL and e < KINK_GRAD_TOL, (s, e, n_flip, worst)
            else:
                assert e < TOL, (s, e)
                e_grad = max(e_grad, e)
            L.apply_update(0)
            g64 = float(np.linalg.norm(grads.astype(np.float64)))
            if clip == "off":
                with pytest.raises(fi.FiError):
                    L.grad_norm_at(0, s + 1)
            else:
                assert abs(L.grad_norm_at(0, s + 1) - g64) <= 1e-6 * g64
                if s == 0:
                    assert (g64 > max_norm) == (clip == "active")
            O.set_grads(np.asarray(grads, np.float64))
            O.opt_step()
            F.opt_step()
        got_p = L.get_params(0)
        e_forced, e_free = U.rel_l2(got_p, O.params()), U.rel_l2(got_p, F.params())
        print(f"[{model} {m}x{t} {opt} clip={clip}] worst loss {e_loss:.2e}, grads {e_grad:.2e}; params teacher-forced "
              f"{e_forced:.2e}, free-running {e_free:.2e}")
        assert e_forced < TOL
        assert np.all(np.isfinite(got_p))
    finally:
        L.close()


# ------------------------------------------------------------------------------- bit-identities
@pytest.mark.parametrize("opt", ["adam", "sgd", "rmsprop-mom"])
def test_clipping_that_never_triggers_is_bit_identical_to_none(fi, opt):
    """coef = min(1, ...) = 1.0 exactly, and g * 1.0f = g: a bound above every norm changes no bit. 4 steps, graph from step 3."""
    m, t = 9, 33
    A, B = _learner(fi, "mlp_actor_critic", m, t, opt, 1e30), _learner(fi, "mlp_actor_critic", m, t, opt, 0.0)
    params = U.ac_params(12)
    for X in (A, B):
        X.set_params(0, params)
    for s in range(4):
        slots = _slots("mlp_actor_critic", 40 + s, m, t)
        for X in (A, B):
            X.trainModel(0, X.stage_batch(0, slots))
    assert np.array_equal(A.get_params(0), B.get_params(0))
    assert np.array_equal(A.get_opt_state(0)[1], B.get_opt_state(0)[1])
    assert np.isfinite(A.grad_norm_at(0, 4)) and A.grad_norm_at(0, 4) > 0
    A.close()
    B.close()


@pytest.mark.parametrize("model,partial", [
    pytest.param("mlp_actor_critic", False, id="mlp_actor_critic"),
    pytest.param("farmer_lstm", False, id="farmer_lstm"),
    pytest.param("mlp_actor_critic", True, id="mlp_actor_critic-partial"),
    pytest.param("farmer_lstm", True, id="farmer_lstm-partial"),
])
def test_graph_replayed_rmsprop_clipped_steps_equal_stream_launched_steps(fi, model, partial):
    """As test_gpu_learner.py's graph-replay test, with RMSProp (momentum 0.9) and clipping that triggers every step: the graph
    holds the norm kernel as a node of its own, so ten fi_learner_step calls (graph from the third, re-captured when the batch
    buffer or size changes) must give the bits of forward_backward + apply_update, norms included."""
    m, t = 16, 20
    A, B = (_learner(fi, model, m, t, "rmsprop-mom", 1e-4) for _ in range(2))
    params = _params(model, 3)
    for X in (A, B):
        X.set_params(0, params)
    slots = [_slots(model, 500 + s, m, t) for s in range(3)]
    ring = A.getSharedBuffers()[0]
    for s in range(10):
        n = m // 2 if partial and s in (5, 6, 9) else m
        if s % 4 == 3:
            assert ring.write_many(slots[s % 3]) == m
            A.trainModel(0, ring.readBatch(m))
        else:
            A.trainModel(0, A.stage_batch(0, slots[s % 3][:n]))
        B.forward_backward(0, B.stage_batch(0, slots[s % 3][:n]))
        B.apply_update(0)
        np.testing.assert_allclose(A.last_losses(0), B.last_losses(0), rtol=1e-6)
        assert A.grad_norm_at(0, s + 1) == B.grad_norm_at(0, s + 1) > 1e-4    # clipped every step
    assert np.array_equal(A.get_params(0), B.get_params(0))
    ma, va, sa = A.get_opt_state(0)
    mb, vb, sb = B.get_opt_state(0)
    assert np.array_equal(ma, mb) and np.array_equal(va, vb) and sa == sb == 10
    A.close()
    B.close()


@pytest.mark.parametrize("opt", ["adam", "rmsprop"])
def test_clipping_adds_exactly_its_one_launch_per_step(fi, opt):
    """Clipping off: the update is the one optimiser launch it always was; on: one more (the norm kernel), split and graph path."""
    m, t = 4, 7
    slots = _slots("mlp_actor_critic", 5, m, t)
    per_update, per_graph_step = {}, {}
    for clip in (0.0, 1.0):
        L = _learner(fi, "mlp_actor_critic", m, t, opt, clip, gemm_mode="simt")
        batch = L.stage_batch(0, slots)
        L.forward_backward(0, batch)
        n0 = fi.kernel_launch_count()
        L.apply_update(0)
        per_update[clip] = fi.kernel_launch_count() - n0
        for _ in range(3):          # steps 2-4: capture at step 3, replay at step 4
            L.trainModel(0, batch)
        n0 = fi.kernel_launch_count()
        L.trainModel(0, batch)
        per_graph_step[clip] = fi.kernel_launch_count() - n0
        L.close()
    assert per_update == {0.0: 1, 1.0: 2}
    assert per_graph_step[1.0] == per_graph_step[0.0] + 1


# ------------------------------------------------------------------------------- learning rate
def test_linear_lr_decay_over_graph_replayed_steps_matches_oracle(fi, oracle):
    """lr annealed linearly to zero over 10 fi_learner_step calls (8 of them graph replays): the teacher-forced oracle under
    the same schedule ends within 1e-5, and a constant-lr oracle does not (the schedule reached the graph's optimiser node)."""
    m, t, steps, lr0 = 16, 20, 10, 6e-4
    params = U.ac_params(17)
    L = _learner(fi, "mlp_actor_critic", m, t, "rmsprop-mom", 1.0)
    L.set_params(0, params)
    O = R.OptOracle.actor_critic(oracle, params, opt="rmsprop", lr=lr0)
    C = R.OptOracle.actor_critic(oracle, params, opt="rmsprop", lr=lr0)
    _, _, eps, mom = OPTS["rmsprop-mom"]
    for s in range(steps):
        lr = lr0 * (1.0 - s / steps)
        L.set_lr(0, lr)
        L.trainModel(0, L.stage_batch(0, _slots("mlp_actor_critic", 60 + s, m, t)))
        grads = np.asarray(L.get_grads(0), np.float64)
        for X, x_lr in ((O, lr), (C, lr0)):
            X.set_grads(grads)
            X.set_opt(x_lr, max_grad_norm=1.0, rmsprop_eps=eps, rmsprop_momentum=mom)
            X.opt_step()
    got = L.get_params(0)
    e, e_const = U.rel_l2(got, O.params()), U.rel_l2(got, C.params())
    print(f"lr schedule: params vs scheduled oracle {e:.2e}, vs constant-lr oracle {e_const:.2e}")
    assert e < TOL and e_const > 10 * TOL
    with pytest.raises(fi.FiError):
        L.set_lr(0, -1e-3)
    with pytest.raises(fi.FiError):
        L.set_lr(0, float("nan"))
    L.close()


@pytest.mark.parametrize("opt", ["adam", "rmsprop-mom"])
def test_lr_zero_freezes_parameters_while_state_advances(fi, opt):
    m, t = 8, 12
    L = _learner(fi, "mlp_actor_critic", m, t, opt, 1.0)
    L.set_params(0, U.ac_params(19))
    for s in range(2):
        L.trainModel(0, L.stage_batch(0, _slots("mlp_actor_critic", 70 + s, m, t)))
    p0 = L.get_params(0)
    m0, v0, step0 = L.get_opt_state(0)
    L.set_lr(0, 0.0)
    for s in range(3):              # graph capture and replays
        L.trainModel(0, L.stage_batch(0, _slots("mlp_actor_critic", 80 + s, m, t)))
    m1, v1, step1 = L.get_opt_state(0)
    assert np.array_equal(L.get_params(0), p0)
    assert step1 == step0 + 3 and not np.array_equal(v1, v0) and not np.array_equal(m1, m0)
    assert L.getModelManager().waitForModelUpdate(0, 5, 5000)     # every step still publishes a version
    assert L.getModelManager().getLatestVersion(0) == 6
    L.close()


# ------------------------------------------------------------------------------- checkpoints
def _magic(path, n):
    with open(path, "rb") as f:
        f.seek(8 + 4 * n)
        return f.read(8)


def test_rmsprop_checkpoint_resumes_bit_identically(fi):
    m, t = 4, 5
    slots = _slots("mlp_actor_critic", 1, m, t)
    with tempfile.TemporaryDirectory() as d:
        L = _learner(fi, "mlp_actor_critic", m, t, "rmsprop-mom", 0.05, gemm_mode="simt", ckpt=d)
        for _ in range(3):
            L.trainModel(0, L.stage_batch(0, slots))
        L.getModelManager().saveModel(0, 9, with_optimizer_state=True)
        assert _magic(os.path.join(d, "model_0_9.bin"), L.param_count) == b"FIRMS001"
        saved = L.get_opt_state(0)
        L.trainModel(0, L.stage_batch(0, slots))
        want = L.get_params(0)
        os.remove(os.path.join(d, "model_0_latest.bin"))
        R = _learner(fi, "mlp_actor_critic", m, t, "rmsprop-mom", 0.05, gemm_mode="simt", seed=99)
        assert R.getModelManager().loadModels(d) == 1
        got = R.get_opt_state(0)
        assert np.array_equal(got[0], saved[0]) and np.array_equal(got[1], saved[1]) and got[2] == saved[2] == 3
        R.trainModel(0, R.stage_batch(0, slots))
        assert np.array_equal(R.get_params(0), want)
        R.close()
        L.close()


@pytest.mark.parametrize("src,dst", [("adam", "rmsprop-mom"), ("rmsprop-mom", "adam")])
def test_optimiser_state_of_the_other_family_loads_weights_only(fi, capfd, src, dst):
    m, t = 4, 5
    slots = _slots("mlp_actor_critic", 2, m, t)
    with tempfile.TemporaryDirectory() as d:
        L = _learner(fi, "mlp_actor_critic", m, t, src, gemm_mode="simt", ckpt=d)
        for _ in range(2):
            L.trainModel(0, L.stage_batch(0, slots))
        L.getModelManager().saveModel(0, 5, with_optimizer_state=True)
        want = L.get_params(0)
        assert _magic(os.path.join(d, "model_0_5.bin"), L.param_count) == (b"FIOPT001" if src == "adam" else b"FIRMS001")
        L.close()                    # (stop() saves model_0_0.bin and latest.bin without optimiser state)
        os.remove(os.path.join(d, "model_0_latest.bin"))
        capfd.readouterr()
        R = _learner(fi, "mlp_actor_critic", m, t, dst, gemm_mode="simt", seed=42)
        assert R.getModelManager().loadModels(d) == 1
        err = capfd.readouterr().err
        assert sum("loaded the weights only" in line for line in err.splitlines()) == 1, err
        assert np.array_equal(R.get_params(0), want)
        mm, vv, step = R.get_opt_state(0)
        assert step == 0 and not mm.any() and not vv.any()
        assert R.getModelManager().getLatestVersion(0) == 3
        R.close()
