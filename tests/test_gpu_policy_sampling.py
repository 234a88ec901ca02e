"""Policy sampling on the device: fi_op_policy_sample and fi_learner_infer_sample against the float64 rule of
tests/sampling_reference.py. Needs a B200.

policy_sample_kernel draws in fp32 (expf, prefix sums in ascending j); the reference draws in float64. They must agree except
where u lies within BAND of a cumulative boundary, where the neighbouring action across that boundary is accepted too; the
share of such rows is printed and bounded. Greedy actions, empty supports and rows with NaN / +inf / all -inf in the support
have no rounding to hide behind and must match exactly.
"""
import os
import subprocess
import threading

import numpy as np
import pytest
from scipy import stats

import _util as U
import legal_reference as LR
import sampling_reference as R

pytestmark = pytest.mark.gpu
BAND = 1e-5
TOL = 1e-5          # the actor-critic inference tolerance of test_gpu_learner.py
MAX_ROWS = 16384
NAN, INF = np.nan, np.inf


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _op(fi, head, ldh, legal, seed, greedy):
    import torch
    rows = head.shape[0]
    d_head = _dev(head)
    d_legal = None if legal is None else _dev(np.asarray(legal, np.uint32).view(np.int32))
    acts = torch.full((rows,), 99, dtype=torch.int32, device="cuda")
    fi.ops.policy_sample(d_head.data_ptr(), ldh, rows, acts.data_ptr(), None if d_legal is None else d_legal.data_ptr(), seed,
                         greedy, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return acts.cpu().numpy()


def _check(got, z, legal, seed, greedy, what):
    """got against the reference on logits z [n,16]; returns the number of rows settled by the boundary band."""
    want, alt, gap = R.sample(z, legal, seed, greedy)
    n = len(z)
    sup = R.supports(legal, n)
    empty = ~sup.any(1)
    assert np.all(got[empty] == -1), what
    inside = sup[np.arange(n), np.clip(got, 0, 15)] & (got >= 0)
    assert np.all(inside[~empty]), f"{what}: {int((~inside[~empty]).sum())} actions outside their support"
    exact = got == want
    banded = ~exact & (gap < BAND) & (got == alt)
    bad = ~exact & ~banded
    assert not bad.any(), (f"{what}: {int(bad.sum())} rows differ, first {np.flatnonzero(bad)[:5]}: got "
                           f"{got[bad][:5]}, want {want[bad][:5]}, gap {gap[bad][:5]}")
    nb = int(banded.sum())
    print(f"{what}: {n} rows, {nb} settled within {BAND:g} of a cumulative boundary")
    assert nb < 1e-3 * n, what
    return nb


def _random_rows(seed, n, ldh):
    """Logits [n, ldh] (columns 16.. random filler), legal words, and the row kinds: plain, NaN / +inf / all -inf in the
    support, non-finite values outside it, an underflowing spread (> 104 below the maximum), bits 16..31 set, empty."""
    rng = np.random.default_rng(seed)
    head = (rng.standard_normal((n, ldh)) * 2).astype(np.float32)
    legal = rng.integers(1, 1 << 16, n).astype(np.uint32)
    kind = rng.integers(0, 16, n)
    z = head[:, :16]
    sup = R.supports(legal, n)
    first = np.argmax(sup, 1)
    z[kind == 0, :] = np.where(sup[kind == 0], NAN, z[kind == 0])                                   # NaN in S
    r1 = np.flatnonzero(kind == 1)
    z[r1, first[r1]] = INF                                                                          # +inf in S
    z[kind == 2] = -INF                                                                             # all -inf
    z[(kind == 3)[:, None] & ~sup] = NAN                                                            # NaN outside S
    z[(kind == 4)[:, None] & ~sup] = INF                                                            # +inf outside S
    r5 = np.flatnonzero(kind == 5)
    z[r5] = np.where(rng.random((r5.size, 16)) < 0.5, z[r5] - 110.0, z[r5])                         # underflow
    legal[kind == 6] |= rng.integers(1, 1 << 16, int((kind == 6).sum())).astype(np.uint32) << np.uint32(16)
    legal[kind == 7] = 0                                                                            # empty support
    r8 = np.flatnonzero(kind == 8)
    legal[r8] = np.uint32(1) << rng.integers(0, 16, r8.size).astype(np.uint32)                     # one legal action
    return head, legal, kind


# ------------------------------------------------------------------------------- 1. operator: exactness
@pytest.mark.parametrize("seed,ldh", [(1, 17), (0x123456789ABCDEF0, 16), (7, 20)], ids=["s1-ldh17", "s64bit-ldh16", "s7-ldh20"])
def test_op_sample_matches_the_float64_rule(fi, seed, ldh):
    n = 1 << 20
    head, legal, kind = _random_rows(seed & 0xFFFF, n, ldh)
    z = head[:, :16]
    got = _op(fi, head, ldh, legal, seed, False)
    _check(got, z, legal, seed, False, f"sample seed {seed:#x} ldh {ldh}")
    g = _op(fi, head, ldh, legal, seed, True)
    assert np.array_equal(g, R.greedy_actions(z.astype(np.float64), R.supports(legal, n))), "greedy"
    # NaN / +inf / all -inf in the support follow the greedy rule; empty supports give -1
    for k in (0, 1, 2):
        assert np.array_equal(got[kind == k], g[kind == k]), k
    assert np.all(got[kind == 7] == -1)
    # a weight that underflows in fp32 is never drawn
    zg = np.take_along_axis(z, np.maximum(g, 0)[:, None], 1)[:, 0]
    r5 = np.flatnonzero((kind == 5) & np.isfinite(zg))
    assert np.all(z[r5, got[r5]] - zg[r5] > -104.0)
    assert ((z[r5] - zg[r5, None] < -104.0) & R.supports(legal[r5], r5.size)).any(1).mean() > 0.9   # the case is there


def test_op_sample_with_null_legal_is_all_legal(fi):
    head, _, _ = _random_rows(9, 4096, 17)
    head[:, :16] = np.random.default_rng(9).standard_normal((4096, 16)).astype(np.float32)
    a = _op(fi, head, 17, None, 5, False)
    assert np.array_equal(a, _op(fi, head, 17, np.full(4096, 0xFFFF, np.uint32), 5, False))
    _check(a, head[:, :16], None, 5, False, "null legal")


# ------------------------------------------------------------------------------- 2. operator: distribution
def test_op_sample_follows_the_masked_softmax(fi):
    n = 1 << 20
    z = np.array([0.3, -1.2, 0.0, 1.1, -0.4, 0.8, -2.0, 0.5, -0.1, 1.4, -0.7, 0.2, -1.5, 0.9, -0.3, 0.6], np.float32)
    legal = 0b1011_0110_1101_1011
    sup = R.supports(np.array([legal], np.uint32), 1)[0]
    got = _op(fi, np.repeat(z[None], n, 0), 16, np.full(n, legal, np.uint32), 2024, False)
    counts = np.bincount(got, minlength=16)
    assert counts[~sup].sum() == 0
    p = stats.chisquare(counts[sup], n * R.masked_softmax(z, sup)[sup]).pvalue
    print(f"masked softmax over {int(sup.sum())} actions, {n} draws: chi-square p = {p:.3g}")
    assert p > 1e-6
    flat = np.bincount(_op(fi, np.zeros((n, 16), np.float32), 16, None, 31337, False), minlength=16)
    p = stats.chisquare(flat).pvalue
    print(f"equal logits over 16 actions: chi-square p = {p:.3g}")
    assert p > 1e-6


# ------------------------------------------------------------------------------- 3. learner path: the network's own logits
def _ac(fi, gemm_mode="auto", **kw):
    return fi.Learner(1, 2, 5, 2, 0, 0, "", "", 0, model="mlp_actor_critic", gemm_mode=gemm_mode, **kw)


def _obs(seed, rows):
    return np.random.default_rng(seed).standard_normal((rows, 162)).astype(np.float32)


def _legal(seed, rows):
    w = np.random.default_rng(seed).integers(1, 1 << 16, rows).astype(np.uint32)
    w[::7] |= np.uint32(0xABCD0000)
    return w


@pytest.mark.parametrize("gemm_mode", ["simt", "auto"])
def test_infer_sample_against_its_own_logits(fi, gemm_mode):
    L = _ac(fi, gemm_mode)
    try:
        L.set_params(0, U.ac_params(61))
        for rows in (1, 255, 256, 4097, MAX_ROWS):
            obs, legal = _obs(rows, rows), _legal(rows + 1, rows)
            seed = 1000 + rows
            acts, logits, values = L.infer_sample(0, obs, legal, seed)
            _check(acts, logits, legal, seed, False, f"[{gemm_mode}] infer_sample {rows} rows")
            plain_logits, plain_values = L.infer(0, obs)
            assert logits.tobytes() == plain_logits.tobytes() and values.tobytes() == plain_values.tobytes(), rows
            g, glog, _ = L.infer_sample(0, obs, legal, seed, greedy=True)
            assert glog.tobytes() == logits.tobytes()
            assert np.array_equal(g, R.greedy_actions(logits.astype(np.float64), R.supports(legal, rows))), rows
            a_none, l_none, _ = L.infer_sample(0, obs, None, seed)
            a_all, _, _ = L.infer_sample(0, obs, np.full(rows, 0xFFFF, np.uint32), seed)
            assert np.array_equal(a_none, a_all) and l_none.tobytes() == logits.tobytes(), rows
            _check(a_none, logits, None, seed, False, f"[{gemm_mode}] infer_sample {rows} rows, all legal")
    finally:
        L.close()


# ------------------------------------------------------------------------------- 4. reproducibility
def test_same_seed_same_actions_other_seed_other_actions(fi):
    L = _ac(fi)
    try:
        L.set_params(0, U.ac_params(62))
        obs, legal = _obs(5, 3000), _legal(6, 3000)
        a1, l1, v1 = L.infer_sample(0, obs, legal, 42)
        a2, l2, v2 = L.infer_sample(0, obs, legal, 42)
        assert np.array_equal(a1, a2) and l1.tobytes() == l2.tobytes() and v1.tobytes() == v2.tobytes()
        a3, _, _ = L.infer_sample(0, obs, legal, 43)
        assert (a1 != a3).mean() > 0.1
        a4, _, _ = L.infer_sample(0, obs, legal, 42 | (1 << 40))   # the seed's high word is part of the key
        assert (a1 != a4).mean() > 0.1
    finally:
        L.close()


# ------------------------------------------------------------------------------- 5. combining
@pytest.mark.parametrize("gemm_mode", ["simt", "auto"])
def test_concurrent_sampling_and_plain_callers(fi, oracle, gemm_mode):
    params = U.ac_params(63)
    L = _ac(fi, gemm_mode)
    try:
        L.set_params(0, params)
        O = oracle.actor_critic(params)
        callers, rounds = 32, 4
        rng = np.random.default_rng(8)
        reqs = []   # [caller][round] = (kind, obs, legal, seed, greedy)
        for c in range(callers):
            row = []
            for r in range(rounds):
                rows = int(rng.integers(1, 70)) if (c + r) % 5 else 300       # a few large requests: the batch crosses 256
                kind = "p" if c % 4 == 3 else "s"
                row.append((kind, _obs(100 * c + r, rows), _legal(100 * c + r + 7, rows) if c % 3 else None,
                            (c << 20) + r, c % 8 == 5))
            reqs.append(row)
        got = [[None] * rounds for _ in range(callers)]
        barrier = threading.Barrier(callers)

        def caller(c):
            for r in range(rounds):
                kind, obs, legal, seed, greedy = reqs[c][r]
                barrier.wait()
                got[c][r] = L.infer_sample(0, obs, legal, seed, greedy) if kind == "s" else L.infer(0, obs)

        ts = [threading.Thread(target=caller, args=(c,)) for c in range(callers)]
        for th in ts:
            th.start()
        for th in ts:
            th.join(timeout=300)
        assert not any(th.is_alive() for th in ts)
        st = L.infer_stats(0)
        rows = sum(q[1].shape[0] for row in reqs for q in row)
        print(f"[{gemm_mode}] sampling + plain callers: {st['calls']} calls, {st['rows']} rows, {st['batches']} forwards")
        assert st["calls"] == callers * rounds and st["rows"] == rows and st["batches"] < st["calls"]
        for c in range(callers):
            for r in range(rounds):
                kind, obs, legal, seed, greedy = reqs[c][r]
                if kind == "s":
                    acts, logits, values = got[c][r]
                    _check(acts, logits, legal, seed, greedy, f"caller {c} round {r}")
                else:
                    logits, values = got[c][r]
                wl, wv = O.forward(obs)
                scale = max(np.abs(wl).max(), np.abs(wv).max())
                assert np.abs(logits - wl).max() < TOL * scale and np.abs(values - wv).max() < TOL * scale, (c, r)
    finally:
        L.close()


# ------------------------------------------------------------------------------- 6. refusals
def test_refusals_leave_the_learner_usable(fi):
    from freeimpala_b200 import _lib
    lib = _lib.load()
    L = _ac(fi)
    F = fi.Learner(1, 2, 8, 2, 0, 0, "", "", 0, model="farmer_lstm")
    try:
        L.set_params(0, U.ac_params(64))
        rows = 5
        obs, legal = _obs(1, rows), _legal(2, rows)
        acts = np.empty(MAX_ROWS + 1, np.int32)
        big = _obs(3, MAX_ROWS + 1)

        def call(h=L._h, o=obs.ctypes.data, lg=legal.ctypes.data, n=rows, greedy=0, a=acts.ctypes.data):
            return lib.fi_learner_infer_sample(h, 0, o, lg, n, 9, greedy, a, None, None)

        empty_word = legal.copy()
        empty_word[3] = 0xFFFF0000          # bits only above 15: no legal action
        bad = {"farmer learner": dict(h=F._h), "null obs": dict(o=None), "null actions": dict(a=None), "rows 0": dict(n=0),
               "too many rows": dict(o=big.ctypes.data, lg=None, n=MAX_ROWS + 1), "greedy 2": dict(greedy=2),
               "greedy -1": dict(greedy=-1), "a row without a legal action": dict(lg=empty_word.ctypes.data)}
        calls_before = L.infer_stats(0)["calls"]
        for name, kw in bad.items():
            assert call(**kw) == _lib.FI_ERR_ARG, name
        assert L.infer_stats(0)["calls"] == calls_before     # refused before the request is queued
        assert call() == _lib.FI_OK
        a, logits, _ = L.infer_sample(0, obs, legal, 9)
        assert np.array_equal(acts[:rows], a)
        _check(a, logits, legal, 9, False, "after refusals")
        with pytest.raises(ValueError):
            L.infer_sample(0, obs, legal[:-1])
    finally:
        F.close()
        L.close()


# ------------------------------------------------------------------------------- 7. end to end
def test_sampled_records_are_the_masked_learners_behaviour_policy(fi, oracle):
    """Trajectories built from infer_sample: observation, returned logits, sampled action, legal word. With the head set to
    the same logits and values, the masked loss head sees pi = mu, so log rho = 0 and its vs / pg advantages are V-trace's
    with log rho = 0. A masking learner then trains on the same records."""
    import torch
    m, t = 8, 20
    params = U.ac_params(65)
    L = _ac(fi, "auto")
    try:
        L.set_params(0, params)
        obs, _, _, rew, disc, boot = U.vtrace_batch(66, m, t)
        legal = _legal(67, m * t).reshape(m, t)
        acts, logits, values = L.infer_sample(0, obs.reshape(m * t, 162), legal.reshape(-1), 0x5EED)
        assert np.all(R.supports(legal.reshape(-1), m * t)[np.arange(m * t), acts])
        mu = logits.reshape(m, t, 16)
        act = acts.reshape(m, t)
        batch = LR.pack_vtrace_slots_legal(obs, mu, act, rew, disc, boot, legal)
        head = np.concatenate([logits, values[:, None]], 1).astype(np.float32)
        d_batch, d_head = _dev(batch), _dev(head)
        dhead = torch.zeros((m * t, 17), device="cuda")
        vs, adv = torch.zeros(m * t, device="cuda"), torch.zeros(m * t, device="cuda")
        losses = torch.zeros(4, dtype=torch.float64, device="cuda")
        st = torch.cuda.current_stream().cuda_stream
        fi.ops.vtrace_loss_head(d_batch.data_ptr(), m, t, d_head.data_ptr(), 17, dhead.data_ptr(), losses.data_ptr(),
                                vs.data_ptr(), adv.data_ptr(), stream=st, legal_mask=True)
        ins = [_dev(a) for a in (np.zeros((m, t), np.float32), disc, rew, values.reshape(m, t), boot)]
        vs0, adv0 = torch.zeros((m, t), device="cuda"), torch.zeros((m, t), device="cuda")
        fi.ops.vtrace(m, t, *[x.data_ptr() for x in ins], vs0.data_ptr(), adv0.data_ptr(), stream=st)
        torch.cuda.synchronize()
        e_vs = np.abs(vs.cpu().numpy() - vs0.cpu().numpy().reshape(-1)).max() / max(1.0, np.abs(vs0.cpu().numpy()).max())
        e_adv = np.abs(adv.cpu().numpy() - adv0.cpu().numpy().reshape(-1)).max() / max(1.0, np.abs(adv0.cpu().numpy()).max())
        print(f"pi = mu: vs {e_vs:.2e}, pg advantages {e_adv:.2e} against V-trace with log rho = 0")
        assert e_vs < 1e-6 and e_adv < 1e-6
        M = fi.Learner(1, 2 * m, t, m, 0, 0, "", "", 0, model="mlp_actor_critic", legal_action_mask=True)
        try:
            M.set_params(0, params)
            for step in range(3):
                M.trainModel(0, M.stage_batch(0, batch))
                got = M.last_losses(0)
                assert np.all(np.isfinite(got)), (step, got)
            assert np.all(np.isfinite(M.get_params(0)))
        finally:
            M.close()
    finally:
        L.close()


def test_harness_sample_actions(fi):
    import json
    from freeimpala_b200 import build
    out = subprocess.run([build.HOST_BIN, "-p", "1", "-B", "8", "-M", "4", "-a", "8", "-T", "2", "-S", "10", "--game-steps", "10",
                          "--agent-time", "0", "--sample-actions"], capture_output=True, text=True, timeout=300,
                         env={**os.environ, "LD_LIBRARY_PATH": os.path.dirname(build.LIB)})
    assert out.returncode == 0, out.stderr
    res = json.loads(out.stdout.strip().splitlines()[-1])
    print(res)
    assert res["learner_updates"] == res["expected_updates"] == (8 * 2) // 4
    assert res["actor_sampled_rows"] == 8 * 2 * 10
    assert res["illegal_actions"] == 0
    assert res["actor_inference_calls"] == 8 * 2
