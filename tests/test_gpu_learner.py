"""Learner-step parity through the C ABI (fi_learner_*) against the CPU oracle. Needs a B200.

Tolerance (BASELINE.json north_star): loss and parameter relative error <= 1e-5 after N steps.
The actor-critic V-trace step has no counterpart in the reference (parity vs the reference is
unpinned, SURVEY.md section 0); its checker is the float64 oracle. The FarmerLstm step is
checked against the golden fixtures produced by the reference's own libtorch train_step.
"""
import os
import tempfile
import threading

import numpy as np
import pytest

import _util as U
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
TOL = 1e-5
# Free-running parameters against the reference's own after N Adam steps, relative L2 over all sampled elements (no
# trimming). profiles/r2_parity.md has the measured values per case and GEMM mode.
PARAM_TOL_VS_REFERENCE = 1e-5


def _ac_learner(fi, m, t, **kw):
    return fi.Learner(1, max(m, 2), t, m, 0, 0, kw.pop("ckpt", ""), "", 0, model="mlp_actor_critic", **kw)


@pytest.mark.parametrize("gemm_mode", ["simt", "tcgen05", "tcgen05_f16", "auto"])
@pytest.mark.parametrize("m,t,steps", [(4, 7, 3), (64, 100, 3), (9, 33, 2), (2, 1, 2), (1, 130, 1)])
def test_actor_critic_vtrace_step_vs_oracle(fi, oracle, m, t, steps, gemm_mode):
    params = U.ac_params(11)
    L = _ac_learner(fi, m, t, gemm_mode=gemm_mode, entropy_cost=0.01, baseline_cost=0.5)
    assert L.param_count == po.AC_PARAMS
    L.set_params(0, params)
    O = oracle.actor_critic(params, lr=5e-4)          # teacher-forced: fed the CUDA gradients
    F = oracle.actor_critic(params, lr=5e-4)          # free-running
    parity = U.AdamParity(O, F)
    for s in range(steps):
        obs, mu, act, rew, disc, boot = U.vtrace_batch(100 + s, m, t, done_p=0.03)
        slots = po.pack_vtrace_slots(obs, mu, act, rew, disc, boot)
        want_free = F.loss_grad(obs, mu, act, rew, disc, boot)
        batch = L.stage_batch(0, slots)
        L.forward_backward(0, batch)
        got = L.last_losses(0)
        # ReLU kinks: a unit whose pre-activation is within fp32 rounding of zero is legitimately decided
        # differently by an fp32 and a float64 forward, and ONE such unit changes a weight-gradient row by
        # O(1/rows) (measured: 7e-4 of ||dW1|| at 64 x 100). The oracle therefore takes the CUDA run's ReLU
        # decisions; the assertions below prove that only genuinely ambiguous units were overridden.
        masks = L.debug_relu_masks(0, m * t)
        want, n_over, max_over = O.loss_grad_masked(obs, mu, act, rew, disc, boot, masks)
        assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (n_over, max_over)
        np.testing.assert_allclose(got, want, rtol=TOL, atol=1e-6 * abs(want[0]))
        # the free-running oracle drifts after the first update (see AdamParity): sanity bound only
        np.testing.assert_allclose(got, want_free, rtol=TOL if s == 0 else 1e-3, atol=1e-6 * abs(want[0]))
        grads = L.get_grads(0)
        assert U.rel_l2(grads, O.grads()) < TOL
        L.apply_update(0)
        parity.step(grads)
        parity.check(L.get_params(0), TOL)
    assert L.steps_done(0) == steps
    L.close()


@pytest.mark.parametrize("gemm_mode", ["simt", "tcgen05", "tcgen05_f16"])
def test_partial_batch_smaller_than_configured(fi, oracle, gemm_mode):
    """A batch of fewer trajectories than batch_size (the learner's buffers are sized for M) is a valid step."""
    m_cfg, m, t = 6, 3, 5
    params = U.ac_params(8)
    L = _ac_learner(fi, m_cfg, t, gemm_mode=gemm_mode)
    L.set_params(0, params)
    obs, mu, act, rew, disc, boot = U.vtrace_batch(31, m, t)
    O = oracle.actor_critic(params, lr=5e-4)
    L.forward_backward(0, L.stage_batch(0, po.pack_vtrace_slots(obs, mu, act, rew, disc, boot)))
    want, n_over, max_over = O.loss_grad_masked(obs, mu, act, rew, disc, boot, L.debug_relu_masks(0, m * t))
    assert n_over <= 4 and max_over < 1e-5
    np.testing.assert_allclose(L.last_losses(0), want, rtol=TOL, atol=1e-6 * abs(want[0]))
    assert U.rel_l2(L.get_grads(0), O.grads()) < TOL
    with pytest.raises(fi.FiError):
        L.stage_batch(0, np.zeros((m_cfg + 1, t * 1024), np.uint8))      # more than batch_size is rejected
    L.close()


def test_step_through_ring_equals_staged_step(fi, oracle):
    """Ring write -> H2D on the side stream -> gather kernel -> step gives the same bits as the staged
    batch: the ring path moves bytes only."""
    m, t = 8, 12
    params = U.ac_params(3)
    obs, mu, act, rew, disc, boot = U.vtrace_batch(9, m, t)
    slots = po.pack_vtrace_slots(obs, mu, act, rew, disc, boot)
    A = fi.Learner(1, 11, t, m, model="mlp_actor_critic", gemm_mode="simt")
    B = fi.Learner(1, 11, t, m, model="mlp_actor_critic", gemm_mode="simt")
    A.set_params(0, params)
    B.set_params(0, params)
    ring = A.getSharedBuffers()[0]
    for i in range(9):  # advance the ring so that the batch wraps around
        ring.write(np.full(t * 1024, i, np.uint8))
    ring.readBatch(9)
    for i in range(m):
        assert ring.write(slots[i])
    batch = ring.readBatch(m)
    assert np.array_equal(batch.to_host(), slots)
    A.trainModel(0, batch)
    B.trainModel(0, B.stage_batch(0, slots))
    assert np.array_equal(A.get_params(0), B.get_params(0))
    A.close()
    B.close()


def test_next_gather_waits_for_the_consumer_of_the_previous_batch(fi):
    """readBatch with no stream (the gather runs on the ring's own stream), an asynchronous step on the learner's stream,
    and the next readBatch straight away: the second gather must not overwrite the batch buffer under the running step
    (ADVICE r1: write-after-read on dev_batch). The step is long (256 x 100 on the fp32 FFMA path), the gather short."""
    m, t = 256, 100
    params = U.ac_params(4)
    a = po.pack_vtrace_slots(*U.vtrace_batch(41, m, t))
    b = po.pack_vtrace_slots(*U.vtrace_batch(42, m, t))
    L = fi.Learner(1, 2 * m, t, m, model="mlp_actor_critic", gemm_mode="simt")
    R = fi.Learner(1, 2 * m, t, m, model="mlp_actor_critic", gemm_mode="simt")
    for X in (L, R):
        X.set_params(0, params)
    ring = L.getSharedBuffers()[0]
    for slots in (a, b):
        assert ring.write_many(slots) == m
    first = ring.readBatch(m)            # stream=None: the ring's own stream
    L.forward_backward(0, first)         # asynchronous, on the learner's stream
    second = ring.readBatch(m)           # no synchronisation in between
    got_a = L.get_grads(0)
    L.forward_backward(0, second)
    got_b = L.get_grads(0)
    R.forward_backward(0, R.stage_batch(0, a))
    want_a = R.get_grads(0)
    R.forward_backward(0, R.stage_batch(0, b))
    want_b = R.get_grads(0)
    assert np.array_equal(got_a, want_a) and np.array_equal(got_b, want_b)
    L.close()
    R.close()


def test_model_store_versions_and_checkpoint(fi, oracle):
    m, t = 4, 5
    with tempfile.TemporaryDirectory() as d:
        L = _ac_learner(fi, m, t, ckpt=d, gemm_mode="simt")
        mm = L.getModelManager()
        assert mm.getLatestVersion(0) == 1              # Model ctor -> version 1 (data_structures.h:52-58)
        assert mm.getLatestVersion(5) == 0 and mm.getModel(5) is None
        assert not mm.waitForModelUpdate(0, 1, 20)      # times out: nothing newer than 1
        model = mm.getModel(0)
        assert model.getVersion() == 1 and np.array_equal(model.as_float32(), L.get_params(0))
        slots = po.pack_vtrace_slots(*U.vtrace_batch(1, m, t))
        for s in range(3):
            L.trainModel(0, L.stage_batch(0, slots))
        assert mm.waitForModelUpdate(0, 3, 5000)
        L.sync(0)
        model = mm.getModel(0)
        assert model.getVersion() == mm.getLatestVersion(0) == 4   # +1 per step (learner.h:40-45)
        assert np.array_equal(model.as_float32(), L.get_params(0))
        # checkpoint: little-endian u64 version + raw bytes, two files (data_structures.h:105-110,399-419)
        mm.saveModel(0, 7)
        raw = np.fromfile(os.path.join(d, "model_0_7.bin"), np.uint8)
        assert raw.size == 8 + 4 * L.param_count and int(raw[:8].view("<u8")[0]) == 4
        assert np.array_equal(raw[8:].view(np.float32), L.get_params(0))
        assert np.array_equal(raw, np.fromfile(os.path.join(d, "model_0_latest.bin"), np.uint8))
        mm.saveModel(0, 0)                              # iteration 0 -> per-player counter (:405)
        assert os.path.exists(os.path.join(d, "model_0_0.bin"))
        # resume with optimiser state: the continued run equals the uninterrupted one bit for bit
        mm.saveModel(0, 9, with_optimizer_state=True)
        L.trainModel(0, L.stage_batch(0, slots))
        want = L.get_params(0)
        os.remove(os.path.join(d, "model_0_latest.bin"))
        R = _ac_learner(fi, m, t, gemm_mode="simt", seed=99)
        assert R.getModelManager().loadModels(d) == 1   # highest-numbered file (model_0_9.bin)
        assert R.getModelManager().getLatestVersion(0) == 4
        assert R.get_opt_state(0)[2] == 3
        R.trainModel(0, R.stage_batch(0, slots))
        assert np.array_equal(R.get_params(0), want)
        R.close()
        L.close()


def test_worker_threads_with_concurrent_actors(fi):
    """configs[2] in miniature: p=2 players, actors writing from many threads, one worker thread per
    player (learner.h:72-97), total_iterations honoured, versions advance by one per update."""
    p, B, S, M, T = 2, 8, 6, 4, 5
    L = fi.Learner(p, B, S, M, 0, 0, "", "", T, model="mlp_actor_critic", gemm_mode="simt")
    bufs = L.getSharedBuffers()
    L.start()

    def actor(a):
        rng = np.random.default_rng(a)
        for i in range(T * M // 4):
            for pl in range(p):
                obs, mu, act, rew, disc, boot = U.vtrace_batch(int(rng.integers(1 << 30)), 1, S)
                assert bufs[pl].write(po.pack_vtrace_slots(obs, mu, act, rew, disc, boot)[0])

    ts = [threading.Thread(target=actor, args=(a,)) for a in range(4)]
    for th in ts:
        th.start()
    for th in ts:
        th.join(timeout=120)
    for w in list(L.worker_threads):
        w.join(timeout=120)
    L.stop()
    assert not L.errors
    assert L.iterations_done == [T, T]
    mm = L.getModelManager()
    assert [mm.getLatestVersion(i) for i in range(p)] == [1 + T, 1 + T]
    assert np.all(np.isfinite(L.get_params(0)))
    L.close()


def test_batched_actor_inference_vs_oracle(fi, oracle):
    params = U.ac_params(21)
    L = _ac_learner(fi, 4, 5, gemm_mode="simt")
    L.set_params(0, params)
    O = oracle.actor_critic(params)
    obs = np.random.default_rng(2).standard_normal((70, 162)).astype(np.float32)
    logits, values = L.infer(0, obs)
    wl, wv = O.forward(obs)
    assert U.rel_max(logits, wl) < TOL and U.rel_max(values, wv) < TOL
    L.close()


@pytest.mark.parametrize("gemm_mode", ["simt", "tcgen05", "tcgen05_f16", "auto"])
def test_concurrent_actor_inference_is_combined_and_matches_oracle(fi, oracle, gemm_mode):
    """64 actors of one player ask for the policy at the same time (Agent::simulateGame's hook, agent.h:52-56): their
    requests are combined into a few forwards on the published weights (fi_learner_infer_stats), every caller gets its own
    rows, and the rows match the float64 oracle. A single large request (1000 rows) takes the tensor-core forward in the
    fp16 modes; it must meet the same tolerance."""
    import threading
    params = U.ac_params(23)
    L = _ac_learner(fi, 4, 5, gemm_mode=gemm_mode)
    L.set_params(0, params)
    O = oracle.actor_critic(params)
    rng = np.random.default_rng(7)
    actors, rounds = 64, 6
    obs = [rng.standard_normal((rounds, 1 + a % 5, 162)).astype(np.float32) for a in range(actors)]   # 1..5 rows per call
    got = [[None] * rounds for _ in range(actors)]
    barrier = threading.Barrier(actors)

    def actor(a):
        for r in range(rounds):
            barrier.wait()                      # all actors of a round call together
            got[a][r] = L.infer(0, obs[a][r])

    ts = [threading.Thread(target=actor, args=(a,)) for a in range(actors)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=120)
    assert not any(t.is_alive() for t in ts)
    for a in range(actors):
        for r in range(rounds):
            wl, wv = O.forward(obs[a][r])
            logits, values = got[a][r]
            scale = max(np.abs(wl).max(), np.abs(wv).max())      # a call carries 1-5 rows: one scale for the 17 head outputs
            assert np.abs(logits - wl).max() < TOL * scale and np.abs(values - wv).max() < TOL * scale, (a, r)
    st = L.infer_stats(0)
    assert st["calls"] == actors * rounds and st["rows"] == sum(o.shape[0] * o.shape[1] for o in obs)
    print(f"[{gemm_mode}] {st['calls']} concurrent inference calls served by {st['batches']} forwards")
    assert st["batches"] <= st["calls"] // 4    # combining: on average at least 4 callers per forward
    big = rng.standard_normal((1000, 162)).astype(np.float32)
    logits, values = L.infer(0, big)
    wl, wv = O.forward(big)
    assert U.rel_max(logits, wl) < TOL and U.rel_max(values, wv) < TOL
    L.close()


def test_create_rejects_bad_config(fi):
    with pytest.raises(fi.FiError):
        fi.Learner(1, 2, 5, 3)                                  # M > B (validateParameters)
    with pytest.raises(fi.FiError):
        fi.Learner(1, 4, 5, 2, model="mlp_actor_critic", loss="mse")
    L = _ac_learner(fi, 2, 5, gemm_mode="simt")
    bad = fi.Learner(1, 4, 6, 2, model="mlp_actor_critic", gemm_mode="simt")
    with pytest.raises(fi.FiError):
        L.trainModel(0, bad.stage_batch(0, np.zeros((2, 6 * 1024), np.uint8)))   # wrong slot size
    L.close()
    bad.close()


# ------------------------------------------------------------------------------- FarmerLstm step
def _farmer_learner(fi, m, t, **kw):
    return fi.Learner(1, max(m, 2), t, m, 0, 0, "", "", 0, model="farmer_lstm", **kw)


@pytest.mark.parametrize("gemm_mode", ["simt", "auto", "tcgen05_f16"])
@pytest.mark.parametrize("ci", [3, 4, 5, 6, 7])
def test_farmer_step_vs_reference_golden(fi, oracle, ci, gemm_mode):
    """The CUDA FarmerLstm step against the reference's own libtorch train_step
    (cmd/libtorch_bench/main.cpp:117-135; fixtures from tools/make_golden.py). Case 3 is the README
    shape / BASELINE.json configs[0]: batch 64, seq 100, MSE, Adam lr 5e-4; case 7 is the shape bench.py's
    reference arm and `--workload farmer` run: batch 1024, seq 100."""
    if ci == 7 and gemm_mode == "simt":
        pytest.skip("1024 x 100 is checked on the two tensor-core paths the bench runs (auto, tcgen05_f16)")
    g = np.load(os.path.join(U.GOLDEN, "farmer_step.npz"))
    stride = int(g["stride"][0])
    b, t, steps, ps, ys, bs = (int(v) for v in g[f"c{ci}_meta"])
    loss, opt = (str(v) for v in g[f"c{ci}_kind"])
    lr = float(g[f"c{ci}_lr"][0])
    params = U.farmer_params(ps)
    L = _farmer_learner(fi, b, t, loss=loss, optimizer=opt, lr=lr, gemm_mode=gemm_mode)
    assert L.param_count == po.FARMER_PARAMS and len(L.tensor_table()) == 16
    L.set_params(0, params)
    O = oracle.farmer(params, opt=opt, lr=lr, loss=loss)   # teacher-forced
    F = oracle.farmer(params, opt=opt, lr=lr, loss=loss)   # free-running
    z0, x0, _ = U.farmer_batch(ys, b, t)
    np.testing.assert_allclose(L.infer(0, z0, x0), g[f"c{ci}_y0"], rtol=2e-5, atol=2e-6)
    parity = U.AdamParity(O, F)
    for s in range(steps):
        z, x, tg = U.farmer_batch(bs + s, b, t)
        batch = L.stage_batch(0, po.pack_farmer_slots(z, x, tg))
        L.forward_backward(0, batch)
        want_loss = float(g[f"c{ci}_losses"][s])                                    # the reference's own loss
        assert abs(L.last_losses(0)[0] - want_loss) <= TOL * abs(want_loss) + 1e-7
        O.loss_grad(z, x, tg)
        F.loss_grad(z, x, tg)
        grads = L.get_grads(0)
        assert U.rel_l2(grads[::stride], g[f"c{ci}_grads"][s]) < 2e-5               # vs the reference (fp32)
        assert U.rel_l2(grads, O.grads()) < TOL                                     # vs the float64 oracle
        L.apply_update(0)
        parity.step(grads)
    e_forced, e_trim, e_free = parity.check(L.get_params(0), TOL)
    # Against the reference's OWN parameters after N free-running steps (every 997th element is stored), all elements, no
    # trimming -- north_star: "parameter relative error <= 1e-5 after N steps" -- next to the same metric for the float64
    # oracle against the reference (tests/test_oracle_pinned.py holds that one to 1e-5 as well).
    got, ref = L.get_params(0)[::stride], g[f"c{ci}_params"]
    e_ref, e_ref_max, e_orc_ref = U.rel_l2(got, ref), U.rel_max(got, ref), U.rel_l2(F.params()[::stride], ref)
    print(f"farmer c{ci} {b}x{t} {loss}/{opt} x{steps} [{gemm_mode}] params after {steps} steps, untrimmed: cuda~reference rel_l2 "
          f"{e_ref:.2e} (max {e_ref_max:.2e}); oracle~reference {e_orc_ref:.2e}; cuda~oracle free-running {e_free:.2e}, "
          f"teacher-forced {e_forced:.2e}")
    assert e_ref < PARAM_TOL_VS_REFERENCE, (e_ref, e_orc_ref)
    L.close()


@pytest.mark.parametrize("live", ["64", "128"])
@pytest.mark.parametrize("ci", [3, 6, 7])
def test_farmer_step_with_the_tensor_core_recurrence(fi, oracle, ci, live, monkeypatch):
    """The opt-in tcgen05 recurrence (csrc/lstm_tc.cu: clusters of 8 CTAs, h exchanged with bulk copies into distributed
    shared memory, gates and c kept in 64-row blocks) gives the same step as the reference: losses, gradients against the
    reference's goldens and the float64 oracle, with 64 and with 128 batch rows per cluster (case 6, 9 x 33, has padding rows
    in its only cluster; case 7, 1024 x 100, fills 16 / 8 clusters)."""
    from freeimpala_b200 import _lib
    g = np.load(os.path.join(U.GOLDEN, "farmer_step.npz"))
    stride = int(g["stride"][0])
    b, t, steps, ps, ys, bs = (int(v) for v in g[f"c{ci}_meta"])
    loss, opt = (str(v) for v in g[f"c{ci}_kind"])
    lr = float(g[f"c{ci}_lr"][0])
    params = U.farmer_params(ps)
    monkeypatch.setenv("FI_LSTM_LIVE", live)   # batch rows per cluster, read at every launch
    _lib.load().fi_debug_set_lstm_tc(1)
    try:
        L = _farmer_learner(fi, b, t, loss=loss, optimizer=opt, lr=lr, gemm_mode="tcgen05_f16")
        L.set_params(0, params)
        O = oracle.farmer(params, opt=opt, lr=lr, loss=loss)
        for s in range(steps):
            z, x, tg = U.farmer_batch(bs + s, b, t)
            L.forward_backward(0, L.stage_batch(0, po.pack_farmer_slots(z, x, tg)))
            want_loss = float(g[f"c{ci}_losses"][s])
            assert abs(L.last_losses(0)[0] - want_loss) <= TOL * abs(want_loss) + 1e-7
            O.loss_grad(z, x, tg)
            grads = L.get_grads(0)
            assert U.rel_l2(grads[::stride], g[f"c{ci}_grads"][s]) < 2e-5
            assert U.rel_l2(grads, O.grads()) < TOL
            L.apply_update(0)
            O.set_grads(np.asarray(grads, np.float64))   # teacher-forced, as in the test above
            O.opt_step()
        assert U.rel_l2(L.get_params(0)[::stride], g[f"c{ci}_params"]) < PARAM_TOL_VS_REFERENCE
        L.close()
    finally:
        _lib.load().fi_debug_set_lstm_tc(-1)


def test_farmer_step_through_ring_decodes_records(fi, oracle):
    """Batch assembly + record decode: trajectories written through the ring give the oracle's loss."""
    b, t = 6, 10
    params = U.farmer_params(5)
    L = _farmer_learner(fi, b, t, gemm_mode="simt")
    L.set_params(0, params)
    z, x, tg = U.farmer_batch(77, b, t)
    slots = po.pack_farmer_slots(z, x, tg)
    ring = L.getSharedBuffers()[0]
    for i in range(b):
        assert ring.write(slots[i])
    batch = ring.readBatch(b)
    dz, dx, dt = oracle.decode_farmer(batch.to_host(), b, t)
    assert np.array_equal(dz, z) and np.array_equal(dx, x) and np.array_equal(dt, tg)
    L.forward_backward(0, batch)
    O = oracle.farmer(params)
    want = O.loss_grad(z, x, tg)
    assert abs(L.last_losses(0)[0] - want) <= TOL * abs(want)
    L.close()


def test_profiler_brackets_account_for_every_launch(fi):
    """fi_prof_enable / fi_prof_collect (what bench.py's per-kernel rooflines are made of): consecutive launches of one
    kernel share an event bracket, yet every launch is counted, every kernel gets a positive time and its work tag."""
    m, t = 4, 7
    L = _ac_learner(fi, m, t, gemm_mode="simt")
    batch = L.stage_batch(0, po.pack_vtrace_slots(*U.vtrace_batch(5, m, t)))
    L.trainModel(0, batch)
    L.sync(0)
    fi.prof_collect()
    fi.prof_enable(True)
    n0 = fi.kernel_launch_count()
    for _ in range(3):   # (graphs are not used while the profiler is on)
        L.trainModel(0, batch)
    L.sync(0)
    fi.prof_enable(False)
    launched = fi.kernel_launch_count() - n0
    prof = fi.prof_collect()
    assert launched > 0 and sum(r["launches"] for r in prof.values()) == launched
    assert all(r["total_ms"] > 0 and r["work"] > 0 for r in prof.values())
    assert prof["gemm_simt_kernel"]["launches"] % 3 == 0 and prof["fused_opt_kernel"]["launches"] == 3
    assert fi.prof_collect() == {}   # the window was reset
    L.close()


def test_losses_at_reads_back_any_of_the_last_steps(fi):
    """fi_learner_losses_at: per-step loss read-back ring (a host loop logs step s-1 while step s runs)."""
    m, t = 3, 6
    L = _ac_learner(fi, m, t, gemm_mode="simt")
    seen = []
    for s in range(11):
        obs, mu, act, rew, disc, boot = U.vtrace_batch(300 + s, m, t)
        L.trainModel(0, L.stage_batch(0, po.pack_vtrace_slots(obs, mu, act, rew, disc, boot)))
        seen.append(L.last_losses(0))
    assert L.steps_done(0) == 11
    for step in range(4, 12):   # the ring keeps the last 8 steps
        np.testing.assert_allclose(L.losses_at(0, step), seen[step - 1], rtol=1e-6)
    for bad in (0, 3, 12):
        with pytest.raises(fi.FiError):
            L.losses_at(0, bad)
    L.close()


def test_full_size_step_properties(fi):
    """BASELINE.json's bench shape (1024 x 100), where the float64 oracle is too slow to be the checker:
    (1) two independent implementations of the step — fp32 FFMA GEMMs and the tcgen05 3xFP16 path — agree on the
        losses to 1e-5 and on the gradients to fp32 rounding (apart from the ReLU units within rounding of zero that the
        two decide differently; the decisions themselves are compared);
    (2) the losses are sums over trajectories, so the gradient of the full batch equals the sum of the gradients of its
        two halves (every trajectory is processed identically whatever the batch around it: tile position, split-K
        partition and the per-tensor fp16 scales all change with the batch)."""
    m, t = 1024, 100
    params = U.ac_params(5)
    obs, mu, act, rew, disc, boot = U.vtrace_batch(77, m, t, done_p=0.02)
    slots = po.pack_vtrace_slots(obs, mu, act, rew, disc, boot)
    A = _ac_learner(fi, m, t, gemm_mode="auto")
    B = _ac_learner(fi, m, t, gemm_mode="simt")
    res = {}
    for name, L in (("tc", A), ("simt", B)):
        L.set_params(0, params)
        L.forward_backward(0, L.stage_batch(0, slots))
        res[name] = (L.last_losses(0), L.get_grads(0), L.debug_relu_masks(0, m * t))
    B.close()
    (la, ga, ma), (lb, gb, mb) = res["tc"], res["simt"]
    np.testing.assert_allclose(la, lb, rtol=1e-5, atol=1e-6 * abs(lb[0]))
    flips = int(np.count_nonzero(ma != mb))
    assert flips <= 4 + 2e-5 * ma.size / 5, flips       # same budget as the oracle comparison at small sizes
    full_rel, trimmed = U.rel_l2(ga, gb), U.trimmed_rel_l2(ga, gb)
    print(f"full-size cross-path: relu flips {flips}, grads rel_l2 {full_rel:.3e}, trimmed {trimmed:.3e}")
    # a unit decided differently moves a whole weight-gradient row of every layer below it (both are valid subgradients at
    # the kink), so across two implementations the gradients are only held to the flip-limited level; the tight gradient
    # check at this size is (2), where both sides make the same decisions
    assert trimmed < 1e-3 and full_rel < 2e-3
    # (2) halves
    g_sum, l_sum = np.zeros_like(ga, dtype=np.float64), np.zeros(4)
    for half in (slots[: m // 2], slots[m // 2:]):
        A.forward_backward(0, A.stage_batch(0, half))
        g_sum += A.get_grads(0)
        l_sum += A.last_losses(0)
    np.testing.assert_allclose(l_sum, la, rtol=2e-6, atol=1e-6 * abs(la[0]))
    half_rel = U.rel_l2(g_sum, ga)
    print(f"full-size halves: grads rel_l2 {half_rel:.3e}")
    assert half_rel < 1e-5
    A.close()


def test_full_size_step_vs_oracle(fi, oracle):
    """One V-trace learner step at the bench shape (1024 x 100, default tensor-core path) against the float64 oracle
    (tens of seconds of host time): losses, gradients and the parameters after the Adam update within 1e-5."""
    m, t = 1024, 100
    params = U.ac_params(6)
    obs, mu, act, rew, disc, boot = U.vtrace_batch(78, m, t, done_p=0.02)
    L = _ac_learner(fi, m, t)
    L.set_params(0, params)
    L.forward_backward(0, L.stage_batch(0, po.pack_vtrace_slots(obs, mu, act, rew, disc, boot)))
    got, grads, masks = L.last_losses(0), L.get_grads(0), L.debug_relu_masks(0, m * t)
    O = oracle.actor_critic(params, lr=5e-4)
    want, n_over, max_over = O.loss_grad_masked(obs, mu, act, rew, disc, boot, masks)
    assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (n_over, max_over)
    np.testing.assert_allclose(got, want, rtol=TOL, atol=1e-6 * abs(want[0]))
    rel = U.rel_l2(grads, O.grads())
    print(f"full-size vs oracle: overridden relu units {n_over} (max |pre-activation| {max_over:.2e}), grads rel_l2 {rel:.3e}")
    assert rel < TOL
    L.apply_update(0)
    O.set_grads(np.asarray(grads, np.float64))     # teacher-forced Adam step (see _util.AdamParity)
    O.opt_step()
    assert U.rel_l2(L.get_params(0), O.params()) < TOL
    L.close()


@pytest.mark.parametrize("model,partial", [
    pytest.param("mlp_actor_critic", False, id="mlp_actor_critic"),
    pytest.param("farmer_lstm", False, id="farmer_lstm"),
    pytest.param("mlp_actor_critic", True, id="mlp_actor_critic-partial"),
    pytest.param("farmer_lstm", True, id="farmer_lstm-partial"),
])
def test_graph_replayed_steps_equal_stream_launched_steps(fi, model, partial, monkeypatch):
    """fi_learner_step replays the step as one CUDA graph from the third step on (only the optimiser node is re-parameterised:
    step count, snapshot and loss slots). Ten steps through the graph path must give the same bits as ten steps enqueued launch
    by launch (FI_GRAPH=0 is read once per process, so the reference run uses forward_backward + apply_update, which never
    use the graph), with the batch alternating between two buffers so that the graph is re-captured on the way. `partial`:
    steps 5, 6 and 9 stage m/2 trajectories into the SAME staged buffer as the full batches around them, so only the batch
    size changes between captures (a graph replayed for the wrong m would read the stale second half of the buffer)."""
    m, t = 16, 20
    farmer = model == "farmer_lstm"
    mk = (lambda: _farmer_learner(fi, m, t, gemm_mode="auto")) if farmer else (lambda: _ac_learner(fi, m, t, gemm_mode="auto"))
    A, B = mk(), mk()
    params = U.farmer_params(3) if farmer else U.ac_params(3)
    for X in (A, B):
        X.set_params(0, params)
    slots = []
    for s in range(3):
        if farmer:
            slots.append(po.pack_farmer_slots(*U.farmer_batch(500 + s, m, t)))
        else:
            slots.append(po.pack_vtrace_slots(*U.vtrace_batch(500 + s, m, t)))
    n0 = fi.kernel_launch_count()
    ring = A.getSharedBuffers()[0]
    for s in range(10):
        n = m // 2 if partial and s in (5, 6, 9) else m
        if s % 4 == 3:                       # through the ring now and then: another batch buffer -> re-capture
            assert ring.write_many(slots[s % 3]) == m
            A.trainModel(0, ring.readBatch(m))
        else:
            A.trainModel(0, A.stage_batch(0, slots[s % 3][:n]))
        B.forward_backward(0, B.stage_batch(0, slots[s % 3][:n]))
        B.apply_update(0)
        np.testing.assert_allclose(A.last_losses(0), B.last_losses(0), rtol=1e-6)   # loss sums: double atomics, order varies
    assert np.array_equal(A.get_params(0), B.get_params(0))
    assert A.getModelManager().getLatestVersion(0) == 11 and A.steps_done(0) == 10
    assert fi.kernel_launch_count() - n0 > 200      # graph launches are counted kernel by kernel
    A.close()
    B.close()
