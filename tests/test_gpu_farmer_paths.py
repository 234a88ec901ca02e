"""The FarmerLstm step and inference against the float64 oracle at every shape that changes their code path. Needs a B200.

The step is not one code path: csrc/model_farmer.cu, csrc/gemm.cu and csrc/lstm_tc.cu pick kernels at run time from the GEMM
mode, the step's batch rows m and the sequence length t. Every case id below names the path it drives:

  proj*-ffma / proj*-tc   input projection and W_ih / W_hh gradients on 3xFP16 tensor cores (farmer_use_half): under AUTO
                          from 2 * m*t * 512 * 162 >= 64e6 FLOP, i.e. m*t >= 386; always under tcgen05_f16
  dense-f16x3             dense stack on 3xFP16 with fused epilogues (farmer_dense_tc): under AUTO from m >= 128
  dense-tf32l1 / -tf32    below that, launch_gemm's AUTO runs a dense product on 3xTF32 from 64 MFLOP: layer 1 (k = 612)
                          from m >= 103, layers 2-5 (k = 512) from m >= 123; dense-ffma: m <= 102, every product on FFMA
  tcgen05-*               3xTF32 for every product of the step
  tail-*                  FFMA recurrence: 8 batch rows per CTA, a tail CTA with m % 8 rows
  lstm_tc-*               tensor-core recurrence (opt-in): 64-row blocks in clusters of 8 CTAs, 64 or 128 live rows per
                          cluster (FI_LSTM_LIVE, else 64 while ceil(m / 64) * 8 <= 148 SMs, i.e. m <= 1152)
  partial-*               steps of fewer trajectories than batch_size: the path decisions use the step's m, the
                          workspaces were sized for batch_size
  mae-sgd / huber-adamw   losses whose dy enters the fp16 split with max|dy| taken in regression_loss_kernel

Each step is checked like test_gpu_learner.py's golden test: the loss within 1e-5 of a teacher-forced and of a free-running
float64 oracle (the mean over the step's own m), the gradients within rel_l2 1e-5 of the teacher-forced oracle's, and the
parameters after the last update through AdamParity (tests/_util.py). t >= 8 everywhere: x[484] spans records 0..7.
"""
import threading

import numpy as np
import pytest

import _util as U
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
TOL = 1e-5
ADAM_FAMILY = ("adam", "adamw")
# ReLU kinks. A dense unit whose pre-activation is within fp32 rounding of zero for one trajectory is legitimately decided
# differently by the fp32 step and the float64 oracle; its backward then passes (or stops) that trajectory's gradient through
# the unit, which moves the unit's weight-gradient row and, through it, every layer below by O(1/m). The dense stack sees only
# m rows per step (not m*t), so one such unit costs ~1e-3 of the gradient's relative L2. Measured on a B200 (1000 W limit):
# one step each of auto 102 x 8, 123 x 8, 127 x 8 and lstm_tc 200 x 33 had exactly one such unit, |pre-activation| / rms
# 2.3e-7, 8.7e-8, 3.8e-7 and 3.2e-8, gradients off by 1.28e-3, 7.5e-4, 4.0e-4 and 8.4e-4; every other step of this file
# stayed below 4e-6.
# The farmer oracle takes no ReLU overrides, so a step that misses TOL must show the signature: debug_relu_masks differs from
# the float64 decisions in at most KINK_UNITS units, each within KINK_REL of zero (|pre-activation| / rms of its layer);
# that step's gradients are then held to KINK_GRAD_TOL and the teacher-forced parameters still to TOL.
KINK_UNITS, KINK_REL, KINK_GRAD_TOL = 4, 1e-5, 2e-3


def _farmer(fi, m_cfg, t, **kw):
    return fi.Learner(1, max(m_cfg, 2), t, m_cfg, 0, 0, "", "", 0, model="farmer_lstm", **kw)


def _lstm_tc(monkeypatch, on, live=None):
    """Selects the recurrence for the steps that follow (forward_backward reads the switch and FI_LSTM_LIVE at every launch;
    the graph path would freeze the choice, so these tests never use it). Undo with fi_debug_set_lstm_tc(-1)."""
    from freeimpala_b200 import _lib
    if live is None:
        monkeypatch.delenv("FI_LSTM_LIVE", raising=False)
    else:
        monkeypatch.setenv("FI_LSTM_LIVE", str(live))
    _lib.load().fi_debug_set_lstm_tc(1 if on else 0)


def _lstm_tc_default():
    from freeimpala_b200 import _lib
    _lib.load().fi_debug_set_lstm_tc(-1)


def _check_steps(fi, oracle, case, t, ms, *, m_cfg=None, loss="mse", opt="adam", lr=5e-4, gemm_mode="auto", z_scale=1.0,
                 seed=0):
    """Steps of forward_backward + apply_update on one learner, batch m = ms[s] at step s, each against the oracles."""
    m_cfg = m_cfg or max(ms)
    params = U.farmer_params(1000 + seed)
    L = _farmer(fi, m_cfg, t, loss=loss, optimizer=opt, lr=lr, gemm_mode=gemm_mode)
    try:
        L.set_params(0, params)
        O = oracle.farmer(params, opt=opt, lr=lr, loss=loss)   # teacher-forced: fed the CUDA gradients
        F = oracle.farmer(params, opt=opt, lr=lr, loss=loss)   # free-running
        parity = U.AdamParity(O, F)
        e_loss = e_grad = 0.0
        n_kink = 0
        for s, m in enumerate(ms):
            z, x, tg = U.farmer_batch(2000 + 97 * seed + s, m, t)
            z = z * np.float32(z_scale)
            params_before = O.params()
            L.forward_backward(0, L.stage_batch(0, po.pack_farmer_slots(z, x, tg)))
            got = L.last_losses(0)[0]
            want = O.loss_grad(z, x, tg, loss_denom=m)
            want_free = F.loss_grad(z, x, tg, loss_denom=m)
            for w in (want, want_free):
                assert abs(got - w) <= TOL * abs(w) + 1e-7, (case, s, m, got, want, want_free)
                e_loss = max(e_loss, abs(got - w) / abs(w))
            grads = L.get_grads(0)
            e = U.rel_l2(grads, O.grads())
            if e >= TOL:   # only the ReLU-kink signature may explain it (see KINK_GRAD_TOL)
                n_flip, worst_rel = _kink_signature(L, m, params_before, z, x)
                print(f"farmer [{case}] step {s}: grads rel_l2 {e:.2e} (trimmed {U.trimmed_rel_l2(grads, O.grads()):.2e}) with "
                      f"{n_flip} ReLU units decided differently from float64, max |pre-activation| / rms {worst_rel:.2e}")
                assert 0 < n_flip <= KINK_UNITS and worst_rel < KINK_REL, (case, s, m, e, n_flip, worst_rel)
                assert e < KINK_GRAD_TOL, (case, s, m, e)
                n_kink += 1
            else:
                e_grad = max(e_grad, e)
            L.apply_update(0)
            parity.step(grads)
        e_forced, e_trim, e_free = parity.check(L.get_params(0), TOL)
        print(f"farmer [{case}] m={ms} t={t} {loss}/{opt} [{gemm_mode}]: worst loss {e_loss:.2e}, grads {e_grad:.2e} "
              f"(+{n_kink} ReLU-kink steps); params "
              f"teacher-forced {e_forced:.2e}, free-running {e_free:.2e} (trimmed {e_trim:.2e})")
    finally:
        L.close()


def _f64_dense_preactivations(params, z, x):
    """The five hidden pre-activations [5, m, 512] of the FarmerLstm forward in float64 (torch LSTM conventions: gate blocks
    i, f, g, o; h0 = c0 = 0), for the ReLU decisions the oracle makes at `params`."""
    p, off, T = np.asarray(params, np.float64), 0, []
    for shp in U.FARMER_SHAPES:
        n = int(np.prod(shp))
        T.append(p[off:off + n].reshape(shp))
        off += n
    sig = lambda v: 1.0 / (1.0 + np.exp(-v))   # noqa: E731
    m, t = z.shape[0], z.shape[1]
    h, c = np.zeros((m, 128)), np.zeros((m, 128))
    for s in range(t):
        g = z[:, s].astype(np.float64) @ T[0].T + T[2] + h @ T[1].T + T[3]
        c = sig(g[:, 128:256]) * c + sig(g[:, :128]) * np.tanh(g[:, 256:384])
        h = sig(g[:, 384:]) * np.tanh(c)
    a, pre = np.concatenate([h, x.astype(np.float64)], axis=1), []
    for layer in range(5):
        pre.append(a @ T[4 + 2 * layer].T + T[5 + 2 * layer])
        a = np.maximum(pre[-1], 0.0)
    return np.stack(pre)


def _kink_signature(L, m, params_before, z, x):
    """(units decided differently by the CUDA step and the float64 forward, the largest |pre-activation| / rms among them)."""
    pre = _f64_dense_preactivations(params_before, z, x)
    cuda_on = L.debug_relu_masks(0, m).reshape(5, m, 512).astype(bool)
    flips = cuda_on != (pre > 0)
    rel = np.abs(pre) / np.sqrt(np.mean(pre * pre, axis=(1, 2)))[:, None, None]
    return int(flips.sum()), float(rel[flips].max()) if flips.any() else 0.0


def _steps(opt):
    return 3 if opt in ADAM_FAMILY else 2


# ------------------------------------------------------------------------------- AUTO thresholds
@pytest.mark.parametrize("m,t", [
    pytest.param(5, 77, id="auto-proj385-ffma"),          # m*t = 385: projection and LSTM weight gradients on FFMA
    pytest.param(2, 193, id="auto-proj386-tc"),           # m*t = 386: the same three products on 3xFP16
    pytest.param(102, 8, id="auto-dense-ffma-m102"),      # every dense product on FFMA
    pytest.param(103, 8, id="auto-dense-tf32l1-m103"),    # layer 1 (k = 612) on 3xTF32, layers 2-5 on FFMA
    pytest.param(110, 8, id="auto-dense-tf32l1-m110"),
    pytest.param(122, 8, id="auto-dense-tf32l1-m122"),
    pytest.param(123, 8, id="auto-dense-tf32-m123"),      # layers 1-5 on 3xTF32
    pytest.param(127, 8, id="auto-dense-tf32-m127"),
    pytest.param(128, 8, id="auto-dense-f16x3-m128"),     # fused 3xFP16 dense stack, one whole 128-row tile
    pytest.param(129, 8, id="auto-dense-f16x3-m129"),     # ... and a 1-row tail tile
    pytest.param(200, 8, id="auto-dense-f16x3-m200"),
])
def test_step_at_the_auto_thresholds(fi, oracle, m, t, monkeypatch):
    _lstm_tc(monkeypatch, False)
    try:
        _check_steps(fi, oracle, f"auto m{m} t{t}", t, [m] * 3, gemm_mode="auto", seed=m)
    finally:
        _lstm_tc_default()


# ------------------------------------------------------------------------------- every GEMM mode
@pytest.mark.parametrize("m,t", [(65, 33), (129, 8)], ids=["m65t33", "m129t8"])
@pytest.mark.parametrize("gemm_mode", ["simt", "auto", "tcgen05", "tcgen05_f16"])
def test_step_in_every_gemm_mode(fi, oracle, gemm_mode, m, t, monkeypatch):
    """simt: every product on FFMA; tcgen05: every product on 3xTF32; tcgen05_f16 and auto: 3xFP16 projection (and at m = 129
    the fused dense stack). 65 x 33 has a 1-row tail CTA in the recurrence and a partial dense tile; 129 x 8 a 1-row tail tile."""
    _lstm_tc(monkeypatch, False)
    try:
        _check_steps(fi, oracle, f"{gemm_mode} m{m} t{t}", t, [m] * 3, gemm_mode=gemm_mode, seed=m + t)
    finally:
        _lstm_tc_default()


# ------------------------------------------------------------------------------- FFMA recurrence row tails
@pytest.mark.parametrize("m", [1, 7, 9, 15], ids=lambda m: f"simt-tail-m{m}")
def test_step_ffma_recurrence_row_tails(fi, oracle, m):
    """m % 8 rows in the last CTA of lstm_forward_kernel / lstm_backward_kernel (m = 1, 7: it is the only CTA)."""
    _check_steps(fi, oracle, f"simt tail m{m}", 8, [m] * 3, gemm_mode="simt", seed=m)


# ------------------------------------------------------------------------------- losses x optimisers on the tensor cores
LOSS_OPT = [("mae", "sgd", 1e-2), ("huber", "adamw", 5e-4), ("mse", "adam", 5e-4)]


@pytest.mark.parametrize("loss,opt,lr", LOSS_OPT, ids=[f"{a}-{b}" for a, b, _ in LOSS_OPT])
@pytest.mark.parametrize("gemm_mode", ["tcgen05_f16", "auto"])
def test_step_losses_and_optimisers_on_the_tensor_core_paths(fi, oracle, gemm_mode, loss, opt, lr, monkeypatch):
    """129 x 8: 3xFP16 projection and fused dense stack, whose backward starts from dy split to fp16 with the max|dy| that
    regression_loss_kernel takes for each loss."""
    _lstm_tc(monkeypatch, False)
    try:
        _check_steps(fi, oracle, f"{gemm_mode} {loss}/{opt}", 8, [129] * _steps(opt), loss=loss, opt=opt, lr=lr,
                     gemm_mode=gemm_mode, seed=7)
    finally:
        _lstm_tc_default()


# ------------------------------------------------------------------------------- large-magnitude inputs
@pytest.mark.parametrize("recurrence", ["ffma", "lstm_tc"], ids=["z8-ffma-recurrence", "z8-lstm_tc-recurrence"])
def test_step_with_saturating_inputs(fi, oracle, recurrence, monkeypatch):
    """z x 8 drives the gates into saturation (fast_exp / fast_tanh far from 0) and grows |c| over 100 steps; the fp16
    observation scale is far from 1. 64 x 100, both recurrences."""
    lstm_tc = recurrence == "lstm_tc"
    _lstm_tc(monkeypatch, lstm_tc)
    try:
        _check_steps(fi, oracle, f"z x 8, {recurrence}", 100, [64] * 3, gemm_mode="tcgen05_f16" if lstm_tc else "auto",
                     z_scale=8.0, seed=64)
    finally:
        _lstm_tc_default()


# ------------------------------------------------------------------------------- tensor-core recurrence
TC_CASES = ([pytest.param(m, t, live, "mse", "adam", 5e-4, id=f"lstm_tc-live{live}-m{m}t{t}")
             for live in (64, 128) for t in (8, 33) for m in (1, 63, 65, 127, 129, 200)] +
            [pytest.param(1152, 8, None, "mse", "adam", 5e-4, id="lstm_tc-autolive64-m1152"),    # 18 clusters x 8 CTAs <= 148
             pytest.param(1153, 8, None, "mse", "adam", 5e-4, id="lstm_tc-autolive128-m1153"),   # 19 x 8 > 148: 128 live rows
             pytest.param(129, 8, None, "mae", "sgd", 1e-2, id="lstm_tc-mae-sgd-m129"),
             pytest.param(129, 8, None, "huber", "adamw", 5e-4, id="lstm_tc-huber-adamw-m129")])


@pytest.mark.parametrize("m,t,live,loss,opt,lr", TC_CASES)
def test_step_with_the_tensor_core_recurrence(fi, oracle, m, t, live, loss, opt, lr, monkeypatch):
    """lstm_tc.cu under tcgen05_f16: clusters with padding rows (m = 1, 63, 65, 127, 129, 200 against 64 / 128 live rows),
    the automatic live-rows switch at m = 1152 / 1153, and the other losses and optimisers."""
    _lstm_tc(monkeypatch, True, live)
    try:
        _check_steps(fi, oracle, f"lstm_tc live {live or 'auto'}", t, [m] * _steps(opt), loss=loss, opt=opt, lr=lr,
                     gemm_mode="tcgen05_f16", seed=m + t)
    finally:
        _lstm_tc_default()


# ------------------------------------------------------------------------------- partial batches
@pytest.mark.parametrize("gemm_mode,lstm_tc", [("auto", False), ("tcgen05_f16", True)],
                         ids=["partial-auto", "partial-tcgen05_f16-lstm_tc"])
def test_step_with_partial_batches(fi, oracle, gemm_mode, lstm_tc, monkeypatch):
    """batch_size 200, steps of 200, 70, 1 and 200 trajectories on one learner: under AUTO, m = 70 / 1 fall back below the
    dense (m >= 128) and projection (m*t >= 386) thresholds with workspaces sized for 200; with the tensor-core recurrence
    its tensor-map cache is keyed on m. The loss is the mean over the step's own trajectories."""
    _lstm_tc(monkeypatch, lstm_tc)
    try:
        _check_steps(fi, oracle, f"partial {gemm_mode}{' lstm_tc' if lstm_tc else ''}", 8, [200, 70, 1, 200], m_cfg=200,
                     gemm_mode=gemm_mode, seed=200)
    finally:
        _lstm_tc_default()


# ------------------------------------------------------------------------------- inference
def test_inference_vs_oracle_as_its_workspaces_grow_and_shrink(fi, oracle):
    """fi_learner_infer on the farmer model: the inference workspaces grow on new rows / t (reallocation) and are reused for a
    smaller t afterwards (row stride t, not the allocated t)."""
    params = U.farmer_params(31)
    L = _farmer(fi, 2, 8, gemm_mode="auto")
    try:
        L.set_params(0, params)
        O = oracle.farmer(params)
        worst = 0.0
        for i, (rows, t) in enumerate([(1, 1), (7, 3), (9, 8), (65, 33), (300, 100), (9, 8), (65, 33), (1, 1)]):
            z, x, _ = U.farmer_batch(700 + i, rows, t)
            got, want = L.infer(0, z, x), O.forward(z, x)
            e = U.rel_max(got, want)
            worst = max(worst, e)
            print(f"farmer inference {rows} x {t}: rel_max {e:.2e}")
            np.testing.assert_allclose(got, want, rtol=2e-5, atol=2e-6, err_msg=f"{rows} x {t}")
        print(f"farmer inference, growing and shrinking workspaces: worst rel_max {worst:.2e}")
    finally:
        L.close()


def test_concurrent_inference_is_combined_and_matches_oracle(fi, oracle):
    """16 callers at once with t drawn from {3, 8, 33} and 1-5 rows each: only callers with equal t share a forward; every
    caller gets its own rows, and the workspaces grow while callers queue."""
    params = U.farmer_params(32)
    L = _farmer(fi, 2, 8, gemm_mode="auto")
    try:
        L.set_params(0, params)
        O = oracle.farmer(params)
        rng = np.random.default_rng(9)
        callers, rounds = 16, 6
        shapes = [[(int(rng.integers(1, 6)), int(rng.choice([3, 8, 33]))) for _ in range(rounds)] for _ in range(callers)]
        inputs = [[U.farmer_batch(1000 * a + r, *shapes[a][r])[:2] for r in range(rounds)] for a in range(callers)]
        got = [[None] * rounds for _ in range(callers)]
        barrier = threading.Barrier(callers)

        def caller(a):
            for r in range(rounds):
                barrier.wait()
                got[a][r] = L.infer(0, *inputs[a][r])

        ts = [threading.Thread(target=caller, args=(a,)) for a in range(callers)]
        for th in ts:
            th.start()
        for th in ts:
            th.join(timeout=300)
        assert not any(th.is_alive() for th in ts)
        worst = 0.0
        for a in range(callers):
            for r in range(rounds):
                want = O.forward(*inputs[a][r])
                worst = max(worst, U.rel_max(got[a][r], want))
                np.testing.assert_allclose(got[a][r], want, rtol=2e-5, atol=2e-6, err_msg=f"caller {a} round {r} {shapes[a][r]}")
        st = L.infer_stats(0)
        print(f"farmer concurrent inference: {st['calls']} calls served by {st['batches']} forwards, worst rel_max {worst:.2e}")
        assert st["calls"] == callers * rounds and st["rows"] == sum(s[0] for row in shapes for s in row)
        assert st["batches"] <= st["calls"] // 2    # combining: on average at least two callers per forward
    finally:
        L.close()
