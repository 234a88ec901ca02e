"""PopArt value normalisation in the actor-critic V-trace step on the GPU (fi_learner_config.popart_beta, include/fi_learner.h).
Needs a B200.

  1. the PopArt loss head alone (fi_op_vtrace_loss_head_popart) against tests/popart_reference.py, with legal words x lengths,
     sigma from the lower clamp to 50 with mu != 0, and NaN / +-inf in the padding rows and records;
  2. a PopArt learner against the float64 reference over 5 steps in every GEMM mode, with and without legal words and lengths;
  3. the replayed graph and forward_backward + apply_update bit-identical, and two identical runs bit-identical;
  4. publication: the model store holds the reward-unit transform of the arena after a step, set_params and fi_model_load;
     inference equals a plain learner's on that blob; a step with lr = 0 leaves the published values unchanged;
  5. checkpoints: bit-exact resume, files without the PopArt section, a plain learner loading a PopArt file;
  6. two data-parallel ranks (needs 2 GPUs): replicas bit-identical, statistics those of the full batch;
  7. the threaded harness with --popart-beta.
"""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

import _util as U
import length_reference as LenR
import popart_reference as R
import test_gpu_ac_paths as P
import test_gpu_legal_actions as GL
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
A = po.NUM_ACTIONS
MODES = ["simt", "tcgen05", "tcgen05_f16", "auto"]
BETA = 0.01


def _data(seed, m, t):
    """test_gpu_ac_paths batches with rewards scaled x100 around a mean of 50, so that the statistics move."""
    obs, mu, act, rew, disc, boot = P._batch(seed, m, t)
    return obs, mu, act, (100.0 * rew + 50.0).astype(np.float32), disc, (100.0 * boot).astype(np.float32)


def _words(seed, m, t):
    L = np.random.default_rng(seed).integers(1, t + 1, size=m)
    L[0], L[-1] = 1, t
    return L.astype(np.uint32)


def _slots(data, words=None, legal=None):
    if words is None:
        return po.pack_vtrace_slots(*data) if legal is None else R.LR.pack_vtrace_slots_legal(*data, legal)
    return LenR.pack_length_slots(*data, words, legal=legal, pad="garbage")


def _ac(fi, m, t, **kw):
    kw.setdefault("popart_beta", BETA)
    return P._ac(fi, m, t, **kw)


# ------------------------------------------------------------------------------- 1. the loss head alone
@pytest.mark.parametrize("sigma", [1e-4, 0.3, 1.0, 50.0])
@pytest.mark.parametrize("lengths", [False, True])
@pytest.mark.parametrize("legal", [False, True])
def test_popart_loss_head_vs_reference(fi, oracle, legal, lengths, sigma):
    import torch
    m, t = 11, 45
    data = _data(20 + int(sigma * 10), m, t)
    obs, mu_l, act, rew, disc, boot = data
    lw = GL._legal_words(t, act) if legal else None
    words = _words(7, m, t) if lengths else None
    L = R.LenR.lengths_of(words, t) if lengths else np.full(m, t)
    rng = np.random.default_rng(3)
    head = rng.standard_normal((m * t, 17)).astype(np.float32)
    mu = float(np.float32(-37.5))
    sig = float(np.float32(sigma))
    cfg = P._oracle_cfg(P.C1)
    want = R.vtrace_losses_popart(oracle, head[:, :16].reshape(m, t, A).astype(np.float64), head[:, 16].reshape(m, t), mu_l, act, rew,
                                  disc, boot, mu, sig, lw, L, **cfg)
    past = ~LenR.valid_rows(L, t).reshape(-1)
    fills = np.array([np.nan, np.inf, -np.inf, 1e30], np.float32)
    head[past] = fills[np.arange(int(past.sum()))[:, None] % 4 + np.zeros((1, 17), np.int64)]
    batch = LenR.pack_length_slots(*data, words if lengths else np.zeros(m, np.uint32), legal=lw, pad="garbage")
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    d_batch, d_head = dev(batch), dev(head)
    dhead = torch.full((m * t, 17), 7.0, device="cuda")
    vs, adv = torch.full((m * t,), 7.0, device="cuda"), torch.full((m * t,), 7.0, device="cuda")
    losses = torch.zeros(4, dtype=torch.float64, device="cuda")
    sums = torch.full((3,), 7.0, dtype=torch.float64, device="cuda")
    fi.ops.vtrace_loss_head(d_batch.data_ptr(), m, t, d_head.data_ptr(), 17, dhead.data_ptr(), losses.data_ptr(), vs.data_ptr(),
                            adv.data_ptr(), stream=torch.cuda.current_stream().cuda_stream, legal_mask=legal, lengths=lengths,
                            popart=(mu, sig), sums=sums.data_ptr(), **P.C1)
    torch.cuda.synchronize()
    got, got_l, got_vs, got_adv, got_s = (x.cpu().numpy() for x in (dhead, losses, vs, adv, sums))
    for name, a in (("losses", got_l), ("dhead", got), ("vs", got_vs), ("pg_adv", got_adv), ("sums", got_s)):
        assert np.all(np.isfinite(a)), name
    assert np.all(got[past] == 0.0)
    dl = want["dlogits"].reshape(-1, A)
    errs = dict(vs=U.rel_max(got_vs, want["vs"]), pg_adv=U.rel_max(got_adv, want["pg_adv"]), dlogits=U.rel_max(got[:, :16], dl),
                dvalue=U.rel_max(got[:, 16], want["dvalue"].reshape(-1)), S1=U.rel_max(got_s[0], want["sums"][0]),
                S2=U.rel_max(got_s[1], want["sums"][1]))
    print(f"popart loss head legal={legal} lengths={lengths} sigma={sigma}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert got_s[2] == want["sums"][2]
    atol = 1e-6 * (np.abs(want["losses"][1:]).sum() + 1.0)
    np.testing.assert_allclose(got_l, want["losses"], rtol=1e-5, atol=atol)
    assert all(e < 1e-5 for e in errs.values()), errs


# ------------------------------------------------------------------------------- 2. the step against the reference
@pytest.mark.parametrize("opts", ["plain", "legal+lengths"])
@pytest.mark.parametrize("gemm_mode", MODES)
def test_popart_step_vs_reference(fi, oracle, gemm_mode, opts):
    m, t, steps = 9, 33, 5
    on = opts != "plain"
    params = U.ac_params(8100)
    L = _ac(fi, m, t, gemm_mode=gemm_mode, legal_action_mask=on, variable_length=on)
    try:
        L.set_params(0, params)
        O, F = R.PopArtAC(params, BETA, P.LR), R.PopArtAC(params, BETA, P.LR)   # teacher-forced, free-running
        worst = 0.0
        for s in range(steps):
            data = _data(8200 + s, m, t)
            lw = GL._legal_words(8300 + s, data[2]) if on else None
            words = _words(8400 + s, m, t) if on else None
            lens = None if words is None else LenR.lengths_of(words, t)
            L.forward_backward(0, L.stage_batch(0, _slots(data, words, lw)))
            got = L.last_losses(0)
            assert np.all(np.isfinite(got)), (s, got)
            masks = L.debug_relu_masks(0, m * t)
            want, g_want, sums_o, n_over, max_over = R.ac_loss_grad_popart(oracle, O.p, *data, *O.stats32(), lw, lens, relu_mask=masks)
            want_free, g_free, sums_f, _, _ = R.ac_loss_grad_popart(oracle, F.p, *data, *F.stats32(), lw, lens)
            assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (s, n_over, max_over)
            atol = 1e-6 * max(abs(want[0]), abs(want[1]) + 0.5 * abs(want[2]) + 0.01 * abs(want[3]))
            np.testing.assert_allclose(got, want, rtol=P.TOL, atol=atol, err_msg=f"step {s}: teacher-forced")
            np.testing.assert_allclose(got, want_free, rtol=P.TOL if s == 0 else 1e-3, atol=atol, err_msg=f"step {s}: free-running")
            grads = L.get_grads(0)
            e = U.rel_l2(grads, g_want)
            assert e < P.TOL, (s, e)
            worst = max(worst, e)
            L.apply_update(0)
            O.step(grads, sums_o)
            F.step(g_free, sums_f)
            mu, nu, sig = L.popart_stats(0)
            assert abs(mu - O.mu) <= 1e-6 * abs(O.mu) and abs(nu - O.nu) <= 1e-6 * abs(O.nu), (s, mu, O.mu, nu, O.nu)
            assert abs(sig - R.sigma(O.mu, O.nu)) <= 1e-6 * sig and sig == R.sigma(mu, nu)
        assert sig > 3.0, sig   # the statistics did move
        e_forced, e_free = U.rel_l2(L.get_params(0), O.p), U.rel_l2(L.get_params(0), F.p)
        print(f"popart [{opts}] [{gemm_mode}]: grads {worst:.2e}, params teacher-forced {e_forced:.2e}, free {e_free:.2e}, "
              f"mu {mu:.4f} sigma {sig:.4f}")
        assert e_forced < P.TOL and e_free < 5e-3
    finally:
        L.close()


# ------------------------------------------------------------------------------- 3. graph, split form, repeat
def _run_steps(fi, graph, steps=6, m=16, t=20, **kw):
    L = _ac(fi, m, t, gemm_mode="auto", legal_action_mask=True, variable_length=True, **kw)
    L.set_params(0, U.ac_params(8500))
    out = []
    for s in range(steps):
        data = _data(8600 + s, m, t)
        b = L.stage_batch(0, _slots(data, _words(8700 + s, m, t), GL._legal_words(8800 + s, data[2])))
        if graph:
            L.trainModel(0, b)
        else:
            L.forward_backward(0, b)
            L.apply_update(0)
        out.append((L.get_params(0), L.popart_stats(0)))
    return L, out


def test_popart_graph_split_and_repeat_are_bit_identical(fi):
    runs = [_run_steps(fi, True), _run_steps(fi, False), _run_steps(fi, True)]
    try:
        for s in range(6):
            p0, st0 = runs[0][1][s]
            for _, out in runs[1:]:
                assert np.array_equal(out[s][0], p0) and out[s][1] == st0, s
    finally:
        for L, _ in runs:
            L.close()


def test_popart_off_keeps_the_launch_count(fi):
    """A learner with popart_beta = 0 launches what it launched before PopArt existed; PopArt adds its two kernels."""
    counts = []
    for beta in (0.0, BETA):
        L = _ac(fi, 8, 20, gemm_mode="auto", popart_beta=beta)
        try:
            b = L.stage_batch(0, _slots(_data(1, 8, 20)))
            L.trainModel(0, b)
            L.sync(0)
            n0 = fi.load_library().fi_kernel_launch_count()
            L.forward_backward(0, b)
            L.apply_update(0)
            L.sync(0)
            counts.append(fi.load_library().fi_kernel_launch_count() - n0)
        finally:
            L.close()
    assert counts[1] == counts[0] + 2, counts


# ------------------------------------------------------------------------------- 4. publication
def _published(L):
    L.sync(0)
    return L.model_manager.getModel(0).as_float32().copy()


def _assert_published(L):
    mu, nu, _ = L.popart_stats(0)
    assert np.array_equal(_published(L), R.publish(L.get_params(0), mu, nu))


def test_publication_is_the_reward_unit_transform(fi, tmp_path):
    m, t = 8, 20
    L = fi.Learner(1, m, t, m, 0, 0, str(tmp_path), "", 0, model="mlp_actor_critic", lr=P.LR, popart_beta=0.2)
    L2 = plain = None
    try:
        L.set_params(0, U.ac_params(8900))
        for s in range(3):
            L.trainModel(0, L.stage_batch(0, _slots(_data(9000 + s, m, t))))
            _assert_published(L)
        mu, nu, sig = L.popart_stats(0)
        assert sig > 2.0 and mu != 0.0
        L.set_params(0, U.ac_params(8901))
        _assert_published(L)
        assert L.popart_stats(0) == (mu, nu, sig)
        L.model_manager.saveModel(0, 1, with_optimizer_state=True)
        L2 = fi.Learner(1, m, t, m, 0, 0, "", str(tmp_path), 0, model="mlp_actor_critic", lr=P.LR, popart_beta=0.2)
        _assert_published(L2)
        assert np.array_equal(_published(L2), _published(L))
        # inference: the PopArt learner's outputs are a plain learner's on the published blob
        plain = P._ac(fi, m, t)
        plain.set_params(0, _published(L))
        obs = np.random.default_rng(1).standard_normal((300, 162)).astype(np.float32)
        legal = np.random.default_rng(2).integers(1, 1 << 16, size=300).astype(np.uint32)
        for rows in (5, 300):   # the fp32 forward and the tensor-core forward of inference
            a, b = L.infer(0, obs[:rows]), plain.infer(0, obs[:rows])
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
            a, b = L.infer_sample(0, obs[:rows], legal[:rows], seed=9), plain.infer_sample(0, obs[:rows], legal[:rows], seed=9)
            assert all(np.array_equal(x, y) for x, y in zip(a, b))
    finally:
        for x in (L, L2, plain):
            if x is not None:
                x.close()


def test_statistics_update_leaves_the_published_values(fi):
    """With lr = 0 the optimiser changes nothing: across steps the statistics move, the arena's value row is rescaled exactly
    as the reference rescales it, and the published values on a fixed observation set stay what they were. The published row is
    fp32 in reward units, so the value sum carries the rounding of terms of size |mu| + sigma: the bound is 1e-6 of that."""
    m, t = 8, 20
    L = fi.Learner(1, m, t, m, 0, 0, "", "", 0, model="mlp_actor_critic", lr=0.0, popart_beta=0.3, gemm_mode="simt")
    try:
        L.set_params(0, U.ac_params(9100))
        obs = np.random.default_rng(3).standard_normal((64, 162)).astype(np.float32)
        v0 = L.infer(0, obs)[1]
        for s in range(3):
            before, st0 = L.get_params(0), L.popart_stats(0)
            L.trainModel(0, L.stage_batch(0, _slots(_data(9200 + s, m, t))))
            st1 = L.popart_stats(0)
            assert st1[:2] != st0[:2]
            assert np.array_equal(L.get_params(0), R.rescale(before, st0[0], st0[1], st1[0], st1[1]))
            _assert_published(L)
            v = L.infer(0, obs)[1]
            bound = 1e-6 * (abs(st1[0]) + st1[2]) + 1e-5 * np.abs(v0).max()
            assert np.abs(v - v0).max() <= bound, (s, np.abs(v - v0).max(), bound)
    finally:
        L.close()


# ------------------------------------------------------------------------------- 5. checkpoints
def test_checkpoint_resume_is_bit_exact(fi, tmp_path):
    m, t = 8, 20
    mk = lambda loc="", start="", beta=0.05: fi.Learner(1, m, t, m, 0, 0, loc, start, 0, model="mlp_actor_critic",  # noqa: E731
                                                       lr=P.LR, popart_beta=beta)
    a = mk(str(tmp_path / "full"))
    others = []
    try:
        a.set_params(0, U.ac_params(9300))
        batches = [_slots(_data(9400 + s, m, t)) for s in range(6)]
        for s in range(3):
            a.forward_backward(0, a.stage_batch(0, batches[s]))
            a.apply_update(0)
        a.model_manager.saveModel(0, 3, with_optimizer_state=True)
        a.sync(0)
        blob = _published(a)
        b = mk("", str(tmp_path / "full"))
        others.append(b)
        assert b.popart_stats(0) == a.popart_stats(0) and np.array_equal(b.get_params(0), a.get_params(0))
        for s in range(3, 6):
            for x in (a, b):
                x.forward_backward(0, x.stage_batch(0, batches[s]))
                x.apply_update(0)
            assert np.array_equal(a.get_params(0), b.get_params(0)) and a.popart_stats(0) == b.popart_stats(0), s
        # without the section (weights only): mu = 0, nu = 1 and the same published values
        os.makedirs(tmp_path / "plain")
        with open(tmp_path / "full" / "model_0_latest.bin", "rb") as f:
            head = f.read(8 + 4 * blob.size)
        with open(tmp_path / "plain" / "model_0_latest.bin", "wb") as f:
            f.write(head)
        c = mk("", str(tmp_path / "plain"))
        others.append(c)
        assert c.popart_stats(0) == (0.0, 1.0, 1.0)
        assert np.array_equal(c.get_params(0), blob) and np.array_equal(_published(c), blob)
        # a learner without PopArt loads the published weights of a PopArt file
        d = mk("", str(tmp_path / "full"), beta=0.0)
        others.append(d)
        assert np.array_equal(d.get_params(0), blob)
    finally:
        a.close()
        for x in others:
            x.close()


# ------------------------------------------------------------------------------- 6. data parallelism
WORKER = os.path.abspath(__file__)


def _dp_rank(rank, world, port, out):
    """One rank (run as `python test_gpu_popart.py RANK WORLD PORT OUT`): the shard of 4 global batches through fi_learner_step."""
    import torch
    import torch.distributed as dist
    import freeimpala_b200 as fi
    from freeimpala_b200 import dp
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    gm, t = 16, 20
    lo, hi = dp.shard_range(gm, rank, world)
    L = fi.Learner(1, hi - lo, t, hi - lo, 0, 0, "", "", 0, device=rank, model="mlp_actor_critic", lr=P.LR, popart_beta=0.2)
    L.set_params(0, U.ac_params(9500))
    ids = [fi.Learner.dp_create_ids(1) if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    L.dp_init(ids[0], rank, world)
    stats = []
    for s in range(4):
        full = _slots(_data(9600 + s, gm, t)).reshape(gm, -1)
        L.trainModel(0, L.stage_batch(0, np.ascontiguousarray(full[lo:hi])))
        stats.append(L.popart_stats(0))
    np.savez(os.path.join(out, f"rank{rank}.npz"), params=L.get_params(0), stats=np.array(stats))
    dist.barrier()
    L.close()
    dist.destroy_process_group()


def test_popart_data_parallel_ranks_agree(fi, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = [subprocess.Popen([sys.executable, WORKER, str(r), "2", str(port), str(tmp_path)], start_new_session=True)
             for r in range(2)]
    try:
        codes = [p.wait(timeout=300) for p in procs]
    finally:
        for p in procs:
            if p.poll() is None:
                os.killpg(p.pid, 9)
                p.wait()
    assert codes == [0, 0], codes
    r0, r1 = (np.load(tmp_path / f"rank{r}.npz") for r in range(2))
    assert np.array_equal(r0["params"], r1["params"]) and np.array_equal(r0["stats"], r1["stats"])
    # the statistics of the full batch: the single-process learner on the same global batches
    gm, t = 16, 20
    L = fi.Learner(1, gm, t, gm, 0, 0, "", "", 0, model="mlp_actor_critic", lr=P.LR, popart_beta=0.2)
    try:
        L.set_params(0, U.ac_params(9500))
        for s in range(4):
            L.trainModel(0, L.stage_batch(0, _slots(_data(9600 + s, gm, t))))
            np.testing.assert_allclose(r0["stats"][s], L.popart_stats(0), rtol=1e-6)
    finally:
        L.close()


# ------------------------------------------------------------------------------- 7. the harness
def test_harness_popart_variable_length_sampled_actions(fi):
    from freeimpala_b200 import build
    args = ["-p", 2, "-B", 8, "-M", 4, "-a", 8, "-T", 3, "-S", 40, "--game-steps", 30, "--agent-time", 0,
            "--popart-beta", 3e-4, "--variable-length", "--sample-actions"]
    r = subprocess.run([build.HOST_BIN, *map(str, args)], capture_output=True, text=True, timeout=300)
    line = [x for x in r.stdout.splitlines() if x.startswith("{")]
    assert r.returncode == 0 and line, r.stderr[-2000:]
    out = json.loads(line[-1])
    assert out["learner_updates"] == out["expected_updates"] and out["illegal_actions"] == 0
    assert len(out["popart_mu"]) == len(out["popart_sigma"]) == 2
    assert all(np.isfinite(out["popart_mu"])) and all(np.isfinite(out["popart_sigma"])) and min(out["popart_sigma"]) > 0


if __name__ == "__main__":
    for _p in (U.ROOT, os.path.dirname(os.path.abspath(__file__))):
        if _p not in sys.path:
            sys.path.insert(0, _p)
    _dp_rank(int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), sys.argv[4])
