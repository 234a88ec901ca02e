"""The actor-critic V-trace step and inference against the float64 oracle with every V-trace constant and at every row count
that changes their code path. Needs a B200.

The step (csrc/model_ac.cu) runs the trunk and head on one of three paths, chosen from the GEMM mode, and each path has its own
launch of the fused loss head (vtrace_loss_head_kernel, csrc/vtrace.cu) with the V-trace constants of fi_learner_config:

  simt                    plain fp32 FFMA GEMMs (gemm_simt.cu); the loss head writes plain fp32 d(head) rows
  tcgen05                 3xTF32 tensor-core GEMMs; the loss head writes the hi/lo pair of d(head) itself
  tcgen05_f16 / auto      3xFP16 tensor-core GEMMs (fp16 pairs with power-of-two HScales); the loss head writes fp32 rows and
                          their max |x|, split by launch_split_h

Within the tensor-core paths, launch_gemm_tc_split (gemm_tc.cu) picks kernels from rows = m * t:

  cta1-*                  forward / dgrad (trans 0 / 1) as single 128-row CTAs while rows < 256 (use_pair: m < 2 * kTcBM)
  pair-*                  from 256 rows, CTA pairs with 256 x 128 tiles; a last pair tile of <= 128 rows leaves the peer CTA
                          with no rows in bounds (257-384, 513-640, ...). In both, the 3xFP16 forward / dgrad products with a
                          split output run with 16 promotion warps (W16)
  splitk-*                the wgrad products (trans 2: dW of the K = 512 layers, dW1 with n = 162, the head with n = 17) are
                          split over K = rows by tc_splits: s = min(CTA units / tiles, num_kb / 4), num_kb = ceil(rows / bk)
                          with bk = 64 (3xFP16) or 32 (3xTF32). One split up to 448 rows (3xFP16) / 224 rows (3xTF32), two or
                          more from 449 / 225. At 2241-2368 rows (36-37 k-blocks of 64) every wgrad product is capped at
                          num_kb / 4 = 9 splits
  rederive-*              launch_gemm_tc_split then re-derives the split count from kb_per_split = ceil(num_kb / s): 37 k-blocks
                          (2305-2368 rows) give 9 splits of 5 k-blocks = 8 splits, so the ninth slab (sized for 9 by
                          gemm_tc_split_workspace_bytes) keeps whatever an earlier step left there
  partial-*               steps of fewer trajectories than batch_size: every decision above uses the step's rows, the
                          workspaces were sized for batch_size

The loss head walks each trajectory backwards in 32-step chunks (one lane per step): t = 32 is one exact chunk, t = 33 or 257
ends in a 1-step chunk. Inference (ac_infer, model_ac.cu) runs the plain fp32 forward below kInferTcRows = 256 rows and the
3xFP16 tensor-core forward (a per-player forward-only DenseStack, inf_dense) from 256 rows on, except under tcgen05, which never
takes it. Two players of one learner own separate DenseStacks, gradient arenas and optimiser states.

Each step is checked like test_gpu_learner.py's test_actor_critic_vtrace_step_vs_oracle: the oracle takes the CUDA run's ReLU
decisions (at most 4 + 2e-5 * size units overridden, each within 1e-5 * rms of zero), the losses within 1e-5 of the teacher-forced
oracle and, on step 0, of the free-running oracle (1e-3 on later steps, see tests/_util.py AdamParity), the gradients within
rel_l2 1e-5 of the teacher-forced oracle's, and the parameters after the last update through AdamParity. The oracles get the
learner's V-trace constants rounded to fp32, as the config struct holds them.
"""
import numpy as np
import pytest

import _util as U
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
TOL = 1e-5
LR = 5e-4
INF = float("inf")
# the constant sets of the V-trace cases (all six values of C1 differ from each other, so any swap of two shows)
C1 = dict(rho_bar=2.0, c_bar=0.7, pg_rho_bar=1.5, lambda_=0.95, baseline_cost=0.25, entropy_cost=0.05)
C2 = dict(lambda_=0.0, entropy_cost=0.0)                                           # one-step targets
C3 = dict(rho_bar=0.5, c_bar=3.0, pg_rho_bar=0.35, baseline_cost=1.0)               # c_bar > rho_bar
# (pg_rho_bar 0.35, not 0.25: 96 % of the step-0 transitions exceed 0.25, 93 % exceed 0.35; see _assert_thresholds_bite)
C4 = dict(rho_bar=INF, c_bar=INF, pg_rho_bar=INF)                                   # no clipping
VTRACE_SETS = {"c1-distinct": C1, "c2-lambda0": C2, "c3-cbar-gt-rhobar": C3, "c4-unclipped": C4}


def _ac(fi, m_cfg, t, players=1, **kw):
    return fi.Learner(players, max(m_cfg, 2), t, m_cfg, 0, 0, "", "", 0, model="mlp_actor_critic", lr=LR, **kw)


def _oracle_cfg(cfg):
    """The constants as the learner holds them (fi_learner_config stores floats)."""
    return {k: float(np.float32(v)) for k, v in cfg.items()}


def _batch(seed, m, t):
    return U.vtrace_batch(seed, m, t, done_p=0.03)


def _log_rho(O, obs, mu, act):
    """log(pi(a) / mu(a)) per transition from a float64 forward at the oracle's current parameters."""
    logits, _ = O.forward(obs)
    logits = logits.reshape(act.shape + (16,))
    mu = mu.astype(np.float64)

    def log_softmax(z):
        z = z - z.max(axis=-1, keepdims=True)
        return z - np.log(np.exp(z).sum(axis=-1, keepdims=True))

    a = act[..., None]
    return (np.take_along_axis(log_softmax(logits), a, -1) - np.take_along_axis(log_softmax(mu), a, -1))[..., 0]


class Worst:
    """Largest errors seen in a case, for the summary line."""

    def __init__(self):
        self.loss = self.grad = 0.0
        self.n_over = 0
        self.max_over = 0.0


def _step_and_check(L, player, O, F, data, s, case, worst, train=False):
    """One step of `player` on `data` against the teacher-forced O and the free-running F; returns the CUDA gradients."""
    obs, mu, act, rew, disc, boot = data
    m, t = act.shape
    want_free = F.loss_grad(*data)
    batch = L.stage_batch(player, po.pack_vtrace_slots(*data))
    if train:
        L.trainModel(player, batch)
    else:
        L.forward_backward(player, batch)
    got = L.last_losses(player)
    assert np.all(np.isfinite(got)), (case, s, got)
    masks = L.debug_relu_masks(player, m * t)
    want, n_over, max_over = O.loss_grad_masked(*data, masks)
    assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (case, s, n_over, max_over)
    atol = 1e-6 * abs(want[0])
    np.testing.assert_allclose(got, want, rtol=TOL, atol=atol, err_msg=f"{case} step {s}: teacher-forced oracle")
    np.testing.assert_allclose(got, want_free, rtol=TOL if s == 0 else 1e-3, atol=atol,
                               err_msg=f"{case} step {s}: free-running oracle")
    grads = L.get_grads(player)
    e = U.rel_l2(grads, O.grads())
    assert e < TOL, (case, s, e)
    worst.loss = max(worst.loss, float(np.max(np.abs(got - want) / np.maximum(np.abs(want), atol))))
    worst.grad = max(worst.grad, e)
    worst.n_over, worst.max_over = max(worst.n_over, n_over), max(worst.max_over, max_over)
    return grads


def _check_steps(fi, oracle, case, t, ms, *, m_cfg=None, gemm_mode="auto", cfg=None, seed=0, make=_batch, train=False,
                 on_step0=None):
    """Steps of one learner, batch m = ms[s] at step s, each against the oracles; forward_backward + apply_update, or
    fi_learner_step (train=True, the CUDA-graph path from the third step on)."""
    cfg = cfg or {}
    params = U.ac_params(1000 + seed)
    L = _ac(fi, m_cfg or max(ms), t, gemm_mode=gemm_mode, **cfg)
    try:
        L.set_params(0, params)
        O = oracle.actor_critic(params, lr=LR, **_oracle_cfg(cfg))   # teacher-forced: fed the CUDA gradients
        F = oracle.actor_critic(params, lr=LR, **_oracle_cfg(cfg))   # free-running
        parity = U.AdamParity(O, F)
        worst = Worst()
        for s, m in enumerate(ms):
            data = make(10 * seed + s, m, t)
            if s == 0 and on_step0:
                on_step0(O, data)
            grads = _step_and_check(L, 0, O, F, data, s, case, worst, train=train)
            if not train:
                L.apply_update(0)
            parity.step(grads)
            if train:      # the update ran inside the step: its parameters are there to compare after every step
                parity.check(L.get_params(0), TOL)
        e_forced, e_trim, e_free = parity.check(L.get_params(0), TOL)
        print(f"ac [{case}] m={ms} t={t} [{gemm_mode}]: worst loss {worst.loss:.2e}, grads {worst.grad:.2e}, "
              f"ReLU overrides {worst.n_over} (max |z|/rms {worst.max_over:.1e}); params teacher-forced {e_forced:.2e}, "
              f"free-running {e_free:.2e} (trimmed {e_trim:.2e})")
    finally:
        L.close()


# ------------------------------------------------------------------------------- A. V-trace constants
def _assert_thresholds_bite(cfg):
    """Every finite clipping threshold is exceeded by 5-95 % of the step-0 transitions (float64 log rho), so each constant
    provably changes the result."""
    def check(O, data):
        obs, mu, act = data[:3]
        ratio = np.exp(_log_rho(O, obs, mu, act))
        for k in ("rho_bar", "c_bar", "pg_rho_bar"):
            v = cfg.get(k, 1.0)
            if np.isfinite(v):
                frac = float(np.mean(ratio > v))
                print(f"  {k} = {v}: exceeded by {100 * frac:.0f} % of the transitions")
                assert 0.05 <= frac <= 0.95, (k, v, frac)
    return check


@pytest.mark.parametrize("name", list(VTRACE_SETS))
@pytest.mark.parametrize("gemm_mode", ["simt", "tcgen05", "tcgen05_f16"])
def test_step_with_vtrace_constants(fi, oracle, gemm_mode, name):
    """9 x 33 (a 1-step second loss-head chunk), 3 Adam steps: simt, tcgen05 and tcgen05_f16 reach the three launches of the
    loss head in ac_forward_backward."""
    cfg = VTRACE_SETS[name]
    _check_steps(fi, oracle, f"vtrace-{name}", 33, [9] * 3, gemm_mode=gemm_mode, cfg=cfg, seed=33,
                 on_step0=_assert_thresholds_bite(cfg))


def test_graph_replayed_steps_with_vtrace_constants(fi, oracle):
    """The constants of C1 through fi_learner_step at 16 x 20 for 5 steps: from the third step on the step is one replayed CUDA
    graph, so the constants are those captured in the loss-head node. Every step against the teacher-forced oracle."""
    _check_steps(fi, oracle, "graph-c1-distinct", 20, [16] * 5, gemm_mode="auto", cfg=C1, seed=16, train=True)


# ------------------------------------------------------------------------------- B. data edges
def _edge(kind):
    def make(seed, m, t):
        obs, mu, act, rew, disc, boot = _batch(seed, m, t)
        if kind == "mu-x4":                  # |log rho| up to ~15: clipping on both sides of every threshold
            mu = mu * np.float32(4)
        elif kind == "gamma-0-or-1":         # half the trajectories never bootstrap, the others are undiscounted
            disc = np.where(np.arange(m)[:, None] % 2 == 0, 0.0, 1.0).astype(np.float32) * np.ones((1, t), np.float32)
        elif kind == "rew-x1e4":
            rew = rew * np.float32(1e4)
        elif kind == "rew-x1e-4":
            rew = rew * np.float32(1e-4)
        elif kind == "obs-x37":              # not powers of two: a power-of-two factor only shifts the power-of-two HScale
            obs = obs * np.float32(37)
        elif kind == "obs-div300":
            obs = obs * np.float32(1 / 300)
        elif kind == "obs-spike-1e4":        # one element sets the observations' scale; the rest sit ~14 binades below it
            obs = obs.copy()
            obs[m // 2, t // 3, 77] = 1e4
        return obs, mu, act, rew, disc, boot
    return make


EDGES = {"mu-x4": C1, "gamma-0-or-1": {}, "rew-x1e4": {}, "rew-x1e-4": dict(entropy_cost=0.0), "obs-x37": {},
         "obs-div300": {}, "obs-spike-1e4": {}}


@pytest.mark.parametrize("kind", list(EDGES))
@pytest.mark.parametrize("gemm_mode", ["simt", "tcgen05_f16"])
def test_step_at_data_edges(fi, oracle, gemm_mode, kind):
    """8 x 40: two loss-head chunks, the second partial. Rewards x 1e4 and x 1e-4 (no entropy term) move the scale of the
    fp16 split of d(head) far from 1 in both directions; the observation cases move the input's HScale."""
    _check_steps(fi, oracle, f"edge-{kind}", 40, [8] * 2, gemm_mode=gemm_mode, cfg=EDGES[kind], seed=40, make=_edge(kind))


@pytest.mark.parametrize("gemm_mode", ["simt", "tcgen05_f16"])
def test_terminal_last_step_ignores_the_bootstrap(fi, oracle, gemm_mode):
    """gamma_{T-1} = 0 everywhere: the bootstrap values enter nothing, so replacing all of them must leave the losses equal
    (rtol 1e-12: they are sums of double atomics in a varying order) and the gradients bit-identical."""
    m, t = 8, 40
    params = U.ac_params(1040)
    L = _ac(fi, m, t, gemm_mode=gemm_mode)
    try:
        L.set_params(0, params)
        O, F = oracle.actor_critic(params, lr=LR), oracle.actor_critic(params, lr=LR)
        parity, worst = U.AdamParity(O, F), Worst()
        for s in range(2):
            obs, mu, act, rew, disc, boot = _batch(400 + s, m, t)
            disc[:, -1] = 0
            grads = _step_and_check(L, 0, O, F, (obs, mu, act, rew, disc, boot), s, "terminal-last", worst)
            losses = L.last_losses(0)
            other = (np.random.default_rng(s).standard_normal(m) * 100).astype(np.float32)
            L.forward_backward(0, L.stage_batch(0, po.pack_vtrace_slots(obs, mu, act, rew, disc, other)))
            np.testing.assert_allclose(L.last_losses(0), losses, rtol=1e-12, atol=0)
            assert np.array_equal(L.get_grads(0), grads), s
            L.apply_update(0)
            parity.step(grads)
        e_forced = parity.check(L.get_params(0), TOL)[0]
        print(f"ac [terminal-last] [{gemm_mode}]: worst loss {worst.loss:.2e}, grads {worst.grad:.2e}, params {e_forced:.2e}")
    finally:
        L.close()


# ------------------------------------------------------------------------------- C. row counts
ROWS = [
    pytest.param(127, 1, "auto", id="cta1-rows127"),             # partial 128-row tile; t = 1: every loss-head chunk is 1 step
    pytest.param(4, 32, "auto", id="cta1-rows128"),              # one exact tile; t = 32 one exact loss-head chunk
    pytest.param(3, 43, "auto", id="cta1-rows129"),              # a 1-row tail tile
    pytest.param(5, 51, "auto", id="cta1-rows255"),              # the last row count on single CTAs
    pytest.param(4, 64, "auto", id="pair-rows256"),              # CTA pairs: one exact 256-row pair tile
    pytest.param(1, 257, "auto", id="pair-rows257-peer-oob"),    # second pair tile of 1 row; t = 257 ends in a 1-step chunk
    pytest.param(383, 1, "auto", id="pair-rows383-peer-oob"),    # second pair tile: the peer CTA has no row in bounds
    pytest.param(12, 32, "auto", id="pair-rows384"),             # ... exactly 128 rows in it
    pytest.param(5, 77, "auto", id="pair-rows385-peer-1row"),    # ... and 1 row in the peer
    pytest.param(7, 64, "auto", id="splitk1-rows448"),           # 7 k-blocks of 64: one split
    pytest.param(1, 449, "auto", id="splitk2-rows449"),          # 8 k-blocks: two splits, the last k-block holds one row
    pytest.param(16, 32, "auto", id="splitk2-rows512"),
    pytest.param(37, 64, "auto", id="rederive-rows2368"),        # 37 k-blocks: 9 splits re-derived to 8
    pytest.param(7, 32, "tcgen05", id="tf32-splitk1-rows224"),   # 3xTF32: 7 k-blocks of 32, one split
    pytest.param(9, 25, "tcgen05", id="tf32-splitk2-rows225"),   # 8 k-blocks: two splits
]


@pytest.mark.parametrize("m,t,gemm_mode", ROWS)
def test_step_at_row_count_thresholds(fi, oracle, m, t, gemm_mode):
    _check_steps(fi, oracle, f"rows {m * t} ({m} x {t})", t, [m] * 2, gemm_mode=gemm_mode, seed=m * t)


# ------------------------------------------------------------------------------- D. partial batches
def test_step_with_partial_batches(fi, oracle):
    """batch_size 37, t = 64: steps of 36 (2304 rows: 9 full splits), 37 (2368 rows: 8 splits while the ninth slab still holds
    the previous step's partials), 3 (192 rows: single CTAs, no split-K) and 37 trajectories. The loss is a sum over the
    step's own trajectories."""
    _check_steps(fi, oracle, "partial-36-37-3-37", 64, [36, 37, 3, 37], m_cfg=37, gemm_mode="auto", seed=37)


# ------------------------------------------------------------------------------- F. two players
def test_two_players_stay_independent(fi, oracle):
    """num_players = 2, auto, 8 x 40, different parameters and data, steps interleaved p0 p1 p0 p1 p0 p1: each player against
    its own oracles, and player 1's parameters and gradients bit-identical across every step of player 0. Then a 300-row
    inference per player (tensor-core forward on that player's inf_dense) against a float64 forward at its parameters."""
    m, t = 8, 40
    L = _ac(fi, m, t, players=2, gemm_mode="auto")
    try:
        O, F, parity, worst = [], [], [], []
        for p in range(2):
            params = U.ac_params(2000 + p)
            L.set_params(p, params)
            O.append(oracle.actor_critic(params, lr=LR))
            F.append(oracle.actor_critic(params, lr=LR))
            parity.append(U.AdamParity(O[p], F[p]))
            worst.append(Worst())
        for s in range(6):
            p = s % 2
            if p == 0:
                L.sync(1)
                before = L.get_params(1), L.get_grads(1)
            grads = _step_and_check(L, p, O[p], F[p], _batch(500 + 10 * p + s // 2, m, t), s // 2, f"player {p}", worst[p])
            L.apply_update(p)
            parity[p].step(grads)
            if p == 0:
                L.sync(0)
                L.sync(1)
                assert np.array_equal(L.get_params(1), before[0]) and np.array_equal(L.get_grads(1), before[1]), s
        rng = np.random.default_rng(300)
        obs = rng.standard_normal((300, 162)).astype(np.float32)
        outs = []
        for p in range(2):
            e_forced = parity[p].check(L.get_params(p), TOL)[0]
            L.sync(p)
            logits, values = L.infer(p, obs)
            wl, wv = oracle.actor_critic(L.get_params(p)).forward(obs)
            el, ev = U.rel_max(logits, wl), U.rel_max(values, wv)
            print(f"ac [two players] player {p}: worst loss {worst[p].loss:.2e}, grads {worst[p].grad:.2e}, params {e_forced:.2e}; "
                  f"300-row inference logits {el:.2e}, values {ev:.2e}")
            assert el < TOL and ev < TOL, (p, el, ev)
            outs.append(logits)
        assert not np.allclose(outs[0], outs[1], rtol=1e-3)   # the two players' forwards really used their own weights
    finally:
        L.close()


# ------------------------------------------------------------------------------- G. inference row thresholds
@pytest.mark.parametrize("gemm_mode", ["simt", "tcgen05", "tcgen05_f16", "auto"])
def test_inference_across_the_tensor_core_threshold(fi, oracle, gemm_mode):
    """One call per row count, in this order: the workspace grows across kInferTcRows = 256 and is reused at smaller sizes."""
    params = U.ac_params(77)
    L = _ac(fi, 4, 5, gemm_mode=gemm_mode)
    try:
        L.set_params(0, params)
        O = oracle.actor_critic(params)
        worst = 0.0
        for i, rows in enumerate([1, 255, 256, 257, 384, 385, 2000, 255, 1]):
            obs = np.random.default_rng(900 + i).standard_normal((rows, 162)).astype(np.float32)
            logits, values = L.infer(0, obs)
            wl, wv = O.forward(obs)
            el, ev = U.rel_max(logits, wl), U.rel_max(values, wv)
            worst = max(worst, el, ev)
            assert el < TOL and ev < TOL, (gemm_mode, i, rows, el, ev)
        print(f"ac inference [{gemm_mode}] rows 1 ... 2000 ... 1: worst rel_max {worst:.2e}")
    finally:
        L.close()
