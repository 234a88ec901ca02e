"""FarmerLstm move histories on the GPU (fi_learner_config.history_length, record word 183; the rule: include/fi_learner.h,
FI_REC_WORD_LENGTH; its float64 statement: tests/history_reference.py). Needs a B200.

  * padding invariance: two history learners whose batches differ only where nothing may be read (z past L, every word of
    records past max(L, 8)), zeros against NaN / +-inf / 1e30 / random bits, stay bit-identical over three steps in all four
    GEMM modes and through the replayed graph;
  * full length: W = 0 and W = T give the bits of a learner without the option;
  * the step against the float64 statement with test_gpu_farmer_paths.py's criteria, at every shape that changes the path;
  * workspaces that hold a full-length step's data, the tensor-core recurrence switch (a history learner never takes it),
    a T = 100 learner on 37-step histories;
  * fi_learner_infer_grouped_lengths: bit-identical to per-state fi_learner_infer_grouped at t = L, NaN past L, combining
    with plain grouped requests, refusals.
"""
import ctypes as C
import threading

import numpy as np
import pytest

import _util as U
import history_reference as H
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
TOL = 1e-5
KINK_UNITS, KINK_REL, KINK_GRAD_TOL = 4, 1e-5, 2e-3   # as test_gpu_farmer_paths.py (its comment says why)
MODES = ["simt", "auto", "tcgen05", "tcgen05_f16"]


def _farmer(fi, m_cfg, t, history=True, **kw):
    return fi.Learner(1, max(m_cfg, 2), t, m_cfg, 0, 0, "", "", 0, model="farmer_lstm", history_length=history, **kw)


def _lstm_tc(on):
    from freeimpala_b200 import _lib
    _lib.load().fi_debug_set_lstm_tc(on)


def _uniform_lengths(seed, m, t):
    L = np.random.default_rng(seed).integers(1, t + 1, size=m)
    L[0], L[-1] = 1, t
    return L


def _kink_signature(L, m, params_before, z, x, lengths):
    pre = H.dense_preactivations(params_before, z, x, lengths)
    cuda_on = L.debug_relu_masks(0, m).reshape(5, m, 512).astype(bool)
    flips = cuda_on != (pre > 0)
    rel = np.abs(pre) / np.sqrt(np.mean(pre * pre, axis=(1, 2)))[:, None, None]
    return int(flips.sum()), float(rel[flips].max()) if flips.any() else 0.0


def _check_history_steps(fi, oracle, case, t, ms, lengths_of, *, m_cfg=None, gemm_mode="auto", seed=0):
    """test_gpu_farmer_paths._check_steps on a history learner: step s has m = ms[s] samples with lengths lengths_of(s, m),
    the records past them filled with garbage; the oracles run the float64 statement (history_reference.loss_grad_history)."""
    m_cfg = m_cfg or max(ms)
    params = U.farmer_params(1000 + seed)
    L = _farmer(fi, m_cfg, t, gemm_mode=gemm_mode)
    try:
        L.set_params(0, params)
        O, F = oracle.farmer(params), oracle.farmer(params)   # teacher-forced, free-running
        parity = U.AdamParity(O, F)
        e_loss = e_grad = 0.0
        n_kink = 0
        for s, m in enumerate(ms):
            z, x, tg = U.farmer_batch(2000 + 97 * seed + s, m, t)
            lens = np.asarray(lengths_of(s, m), np.int64)
            params_before = O.params()
            L.forward_backward(0, L.stage_batch(0, H.pack_history_slots(z, x, tg, lens.astype(np.uint32), pad="garbage")))
            got = L.last_losses(0)[0]
            want, want_g = H.loss_grad_history(O, z, x, tg, lens)
            want_free, free_g = H.loss_grad_history(F, z, x, tg, lens)
            for w in (want, want_free):
                assert abs(got - w) <= TOL * abs(w) + 1e-7, (case, s, m, got, want, want_free)
                e_loss = max(e_loss, abs(got - w) / abs(w))
            grads = L.get_grads(0)
            e = U.rel_l2(grads, want_g)
            if e >= TOL:   # only the ReLU-kink signature may explain it
                n_flip, worst_rel = _kink_signature(L, m, params_before, z, x, lens)
                print(f"history [{case}] step {s}: grads rel_l2 {e:.2e}, {n_flip} ReLU units decided differently, "
                      f"max |pre-activation| / rms {worst_rel:.2e}")
                assert 0 < n_flip <= KINK_UNITS and worst_rel < KINK_REL, (case, s, m, e, n_flip, worst_rel)
                assert e < KINK_GRAD_TOL, (case, s, m, e)
                n_kink += 1
            else:
                e_grad = max(e_grad, e)
            L.apply_update(0)
            F.set_grads(free_g)   # the free-running oracle steps on its own summed gradient
            parity.step(grads)
        e_forced, e_trim, e_free = parity.check(L.get_params(0), TOL)
        print(f"history [{case}] m={ms} t={t} [{gemm_mode}]: worst loss {e_loss:.2e}, grads {e_grad:.2e} (+{n_kink} ReLU-kink "
              f"steps); params teacher-forced {e_forced:.2e}, free-running {e_free:.2e} (trimmed {e_trim:.2e})")
    finally:
        L.close()


def _run(L, slots_list, graph=False):
    """Steps on `L`; returns (losses f64 per step, grads after the last forward_backward, params)."""
    losses, grads = [], None
    for slots in slots_list:
        b = L.stage_batch(0, slots)
        if graph:
            L.trainModel(0, b)
        else:
            L.forward_backward(0, b)
            grads = L.get_grads(0)
            L.apply_update(0)
        L.sync(0)
        losses.append(L.last_losses(0)[0])
    return np.array(losses), grads, L.get_params(0)


# ------------------------------------------------------------------------------- padding invariance
@pytest.mark.parametrize("graph", [False, True], ids=["forward_backward", "graph"])
@pytest.mark.parametrize("gemm_mode", MODES)
def test_padding_is_never_read(fi, gemm_mode, graph):
    """17 x 33 (m*t = 561: the 3xFP16 projection under auto; a 1-row tail CTA): zeros against garbage past each length."""
    m, t = 17, 33
    params = U.farmer_params(5)
    batches = {}
    for pad in ("zeros", "garbage"):
        batches[pad] = []
        for s in range(3):
            z, x, tg = U.farmer_batch(40 + s, m, t)
            lens = _uniform_lengths(50 + s, m, t).astype(np.uint32)
            lens[3] = 7
            batches[pad].append(H.pack_history_slots(z, x, tg, lens, pad=pad))
    out = {}
    for pad in batches:
        L = _farmer(fi, m, t, gemm_mode=gemm_mode)
        try:
            L.set_params(0, params)
            out[pad] = _run(L, batches[pad], graph=graph)
        finally:
            L.close()
    (la, ga, pa), (lb, gb, pb) = out["zeros"], out["garbage"]
    assert np.all(np.isfinite(la)) and np.array_equal(la, lb)
    assert np.array_equal(pa, pb) and np.all(np.isfinite(pa))
    if not graph:
        assert np.array_equal(ga, gb)


# ------------------------------------------------------------------------------- full length
@pytest.mark.parametrize("gemm_mode", MODES)
def test_full_length_is_the_fixed_length_step(fi, gemm_mode):
    m, t = 17, 33
    params = U.farmer_params(6)
    data = [U.farmer_batch(60 + s, m, t) for s in range(2)]
    plain = [po.pack_farmer_slots(*d) for d in data]
    ref = None
    for history, words in ((False, None), (True, 0), (True, t)):
        slots = plain if words is None else [H.pack_history_slots(*d, np.full(m, words, np.uint32)) for d in data]
        L = _farmer(fi, m, t, history=history, gemm_mode=gemm_mode)
        try:
            L.set_params(0, params)
            got = _run(L, slots)
        finally:
            L.close()
        if ref is None:
            ref = got
        else:
            for a, b in zip(got, ref):
                assert np.array_equal(a, b), (gemm_mode, words)


# ------------------------------------------------------------------------------- against the float64 statement
@pytest.mark.parametrize("m", [1, 7, 9])
def test_step_simt_row_tails(fi, oracle, m):
    _check_history_steps(fi, oracle, f"simt tail m{m}", 8, [m] * 3, lambda s, n: _uniform_lengths(s + n, n, 8),
                         gemm_mode="simt", seed=m)


@pytest.mark.parametrize("gemm_mode", MODES)
def test_step_65x33_in_every_gemm_mode(fi, oracle, gemm_mode):
    _check_history_steps(fi, oracle, f"{gemm_mode} 65x33", 33, [65] * 3, lambda s, n: _uniform_lengths(10 + s, n, 33),
                         gemm_mode=gemm_mode, seed=98)


@pytest.mark.parametrize("m,t", [pytest.param(129, 8, id="dense-f16x3-m129t8"), pytest.param(5, 77, id="auto-proj385-ffma"),
                                 pytest.param(2, 193, id="auto-proj386-tc")])
def test_step_at_the_auto_thresholds(fi, oracle, m, t):
    _check_history_steps(fi, oracle, f"auto {m}x{t}", t, [m] * 3, lambda s, n: _uniform_lengths(20 + s, n, t), seed=m)


def test_step_1024x100_uniform_lengths(fi, oracle):
    _check_history_steps(fi, oracle, "auto 1024x100", 100, [1024] * 2, lambda s, n: _uniform_lengths(30 + s, n, 100), seed=3)


@pytest.mark.parametrize("gemm_mode", ["auto", "simt"])
def test_step_every_length_one(fi, oracle, gemm_mode):
    _check_history_steps(fi, oracle, f"{gemm_mode} all L=1", 100, [64] * 3, lambda s, n: np.ones(n, np.int64),
                         gemm_mode=gemm_mode, seed=4)


def test_step_lengths_around_the_x_records(fi, oracle):
    """L in {7, 8, 9}: records L..7 still carry x, records from max(L, 8) on carry nothing."""
    _check_history_steps(fi, oracle, "auto L 7/8/9", 16, [33] * 3, lambda s, n: np.arange(n) % 3 + 7, gemm_mode="auto", seed=5)


def test_step_with_partial_batches(fi, oracle):
    """batch_size 200, steps of 200, 70, 1 and 200 samples: AUTO moves between the 3xFP16 and plain projections."""
    _check_history_steps(fi, oracle, "partial auto", 8, [200, 70, 1, 200], lambda s, n: _uniform_lengths(40 + s, n, 8),
                         m_cfg=200, seed=200)


def test_step_t100_learner_on_37_step_histories(fi, oracle):
    """Every L = 37 in 100-record slots: the oracle's step at T = 37 (and the reference's own, where oracle/_ref exists)."""
    m, t, n = 16, 100, 37
    params = U.farmer_params(7)
    z, x, tg = U.farmer_batch(70, m, t)
    L = _farmer(fi, m, t)
    try:
        L.set_params(0, params)
        L.forward_backward(0, L.stage_batch(0, H.pack_history_slots(z, x, tg, np.full(m, n, np.uint32), pad="garbage")))
        got, grads = L.last_losses(0)[0], L.get_grads(0)
    finally:
        L.close()
    o = oracle.farmer(params)
    want = o.loss_grad(np.ascontiguousarray(z[:, :n]), x, tg)
    assert abs(got - want) <= TOL * abs(want) + 1e-7 and U.rel_l2(grads, o.grads()) < TOL
    if po.ref_available():
        ref = po.RefNN(seed=1234)
        ref.set_params(params)
        want_ref = ref.train_step(np.ascontiguousarray(z[:, :n]), x, tg)
        assert abs(got - want_ref) <= TOL * abs(want_ref) + 1e-7 and U.rel_l2(grads, ref.grads()) < 2e-5


# ------------------------------------------------------------------------------- stale workspaces
@pytest.mark.parametrize("gemm_mode", MODES)
def test_short_histories_after_a_full_length_step(fi, oracle, gemm_mode):
    """m = 16: a full-length step fills every workspace row with finite data; then rows 0..7 have L = 3 and rows 8..15 L = T
    (one CTA of the recurrence wholly short). Matches the reference and a fresh learner given the same parameters, bit for bit."""
    m, t = 16, 33
    params = U.farmer_params(8)
    z0, x0, tg0 = U.farmer_batch(80, m, t)
    z, x, tg = U.farmer_batch(81, m, t)
    lens = np.where(np.arange(m) < 8, 3, t)
    short = H.pack_history_slots(z, x, tg, lens.astype(np.uint32), pad="garbage")
    L = _farmer(fi, m, t, gemm_mode=gemm_mode)
    F = _farmer(fi, m, t, gemm_mode=gemm_mode)
    try:
        L.set_params(0, params)
        L.forward_backward(0, L.stage_batch(0, H.pack_history_slots(z0, x0, tg0, np.zeros(m, np.uint32))))
        L.apply_update(0)
        p1 = L.get_params(0)
        L.forward_backward(0, L.stage_batch(0, short))
        got, grads = L.last_losses(0)[0], L.get_grads(0)
        F.set_params(0, p1)
        F.forward_backward(0, F.stage_batch(0, short))
        assert got == F.last_losses(0)[0] and np.array_equal(grads, F.get_grads(0))
    finally:
        L.close()
        F.close()
    want, want_g = H.loss_grad_history(oracle.farmer(p1), z, x, tg, lens)
    assert abs(got - want) <= TOL * abs(want) + 1e-7 and U.rel_l2(grads, want_g) < TOL


def test_tensor_core_recurrence_switch_is_ignored(fi):
    """fi_debug_set_lstm_tc(1): a history learner still runs the FFMA recurrence, the bits of the run with it at 0. m = 24:
    regression_loss_kernel adds its warps' partial losses with atomics, so only a batch of one warp has a loss whose bits
    do not depend on timing."""
    m, t = 24, 33
    params = U.farmer_params(9)
    data = [U.farmer_batch(90 + s, m, t) for s in range(2)]
    slots = [H.pack_history_slots(*d, _uniform_lengths(91 + s, m, t).astype(np.uint32), pad="garbage") for s, d in enumerate(data)]
    out = []
    try:
        for on in (0, 1):
            _lstm_tc(on)
            L = _farmer(fi, m, t, gemm_mode="tcgen05_f16")
            try:
                L.set_params(0, params)
                out.append(_run(L, slots))
            finally:
                L.close()
    finally:
        _lstm_tc(-1)
    for a, b in zip(*out):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------------------- inference
def _groups(seed, states, rows):
    """offsets [states + 1] of `rows` candidates spread over `states` groups, each non-empty."""
    rng = np.random.default_rng(seed)
    cuts = np.sort(rng.choice(np.arange(1, rows), size=states - 1, replace=False)) if states > 1 else np.array([], int)
    return np.concatenate([[0], cuts, [rows]]).astype(np.uint32)


def _per_state(L, z, x, off, lens):
    values, best = np.empty(int(off[-1]), np.float32), np.empty(len(lens), np.int32)
    for s, n in enumerate(lens):
        v, b = L.infer_grouped(0, np.ascontiguousarray(z[s:s + 1, :n]), x[off[s]:off[s + 1]], np.array([0, off[s + 1] - off[s]]))
        values[off[s]:off[s + 1]], best[s] = v, b[0]
    return values, best


@pytest.mark.parametrize("states,rows", [(1, 1), (17, 255), (64, 16384)])
@pytest.mark.parametrize("history", [False, True], ids=["plain-learner", "history-learner"])
def test_inference_is_per_state_grouped_inference_at_t_L(fi, states, rows, history):
    t = 100
    params = U.farmer_params(10)
    z, _, _ = U.farmer_batch(100 + rows, states, t)
    x = np.random.default_rng(rows).standard_normal((rows, 484)).astype(np.float32)
    off = _groups(rows, states, rows)
    lens = _uniform_lengths(rows, states, t) if states > 1 else np.array([37])
    L = _farmer(fi, 8, 8, history=history)
    try:
        L.set_params(0, params)
        want_v, want_b = _per_state(L, z, x, off, lens)
        got_v, got_b = L.infer_grouped(0, z, x, off, lengths=lens)
        assert np.array_equal(got_v, want_v) and np.array_equal(got_b, want_b)
        z_nan = z.copy()
        z_nan[np.arange(t)[None, :] >= lens[:, None]] = np.nan
        got_v2, got_b2 = L.infer_grouped(0, z_nan, x, off, lengths=lens)
        assert np.array_equal(got_v2, want_v) and np.array_equal(got_b2, want_b)
        st = L.infer_stats(0)
        assert st["rows"] == sum(int(off[s + 1] - off[s]) for s in range(states)) + 2 * rows
    finally:
        L.close()


def test_concurrent_length_and_plain_requests_are_combined(fi):
    """32 callers, half with per-state lengths, half plain grouped calls, all at t = 40: fewer forwards than calls, and every
    caller's values and best equal the per-state results."""
    t, callers, rounds = 40, 32, 4
    params = U.farmer_params(11)
    L = _farmer(fi, 8, 8)
    try:
        L.set_params(0, params)
        cases, want = [], []
        for a in range(callers):
            row = []
            for r in range(rounds):
                rng = np.random.default_rng(1000 * a + r)
                states = int(rng.integers(1, 5))
                rows = states + int(rng.integers(0, 8))
                z = rng.standard_normal((states, t, 162)).astype(np.float32)
                x = rng.standard_normal((rows, 484)).astype(np.float32)
                off = _groups(a + r, states, rows)
                lens = rng.integers(1, t + 1, size=states) if a % 2 == 0 else None
                row.append((z, x, off, lens))
            cases.append(row)
        before = L.infer_stats(0)
        want = [[_per_state(L, z, x, off, lens if lens is not None else np.full(len(off) - 1, t)) for z, x, off, lens in row]
                for row in cases]
        mid = L.infer_stats(0)
        got = [[None] * rounds for _ in range(callers)]
        barrier = threading.Barrier(callers)

        def caller(a):
            for r in range(rounds):
                barrier.wait()
                z, x, off, lens = cases[a][r]
                got[a][r] = L.infer_grouped(0, z, x, off, lengths=lens)

        ts = [threading.Thread(target=caller, args=(a,)) for a in range(callers)]
        for th in ts:
            th.start()
        for th in ts:
            th.join(timeout=300)
        assert not any(th.is_alive() for th in ts)
        for a in range(callers):
            for r in range(rounds):
                assert np.array_equal(got[a][r][0], want[a][r][0]) and np.array_equal(got[a][r][1], want[a][r][1]), (a, r)
        st = L.infer_stats(0)
        calls, batches = st["calls"] - mid["calls"], st["batches"] - mid["batches"]
        print(f"history inference: {calls} calls served by {batches} forwards ({mid['calls'] - before['calls']} per-state calls before)")
        assert calls == callers * rounds and batches < calls
    finally:
        L.close()


def test_inference_refusals_leave_the_learner_usable(fi):
    from freeimpala_b200 import _lib
    lib = _lib.load()
    t, states = 10, 2
    params = U.farmer_params(12)
    z, _, _ = U.farmer_batch(120, states, t)
    x = np.random.default_rng(1).standard_normal((3, 484)).astype(np.float32)
    off = np.array([0, 1, 3], np.uint32)
    values, best = np.empty(3, np.float32), np.empty(states, np.int32)
    L = _farmer(fi, 8, 8)
    A = fi.Learner(1, 4, 8, 2, model="mlp_actor_critic")
    try:
        L.set_params(0, params)
        want = L.infer_grouped(0, z, x, off, lengths=np.array([3, 10]))

        def call(h, lens, offsets=off):
            return lib.fi_learner_infer_grouped_lengths(h, 0, z.ctypes.data, states, t, None if lens is None else lens.ctypes.data,
                                                        x.ctypes.data, offsets.ctypes.data, values.ctypes.data, best.ctypes.data)
        for lens, offsets, msg in ((None, off, "lengths"), (np.array([0, 3], np.uint32), off, "lengths[0]"),
                                   (np.array([3, t + 1], np.uint32), off, "lengths[1]"),
                                   (np.array([3, 10], np.uint32), np.array([1, 1, 3], np.uint32), "offsets[0]"),
                                   (np.array([3, 10], np.uint32), np.array([0, 2, 2], np.uint32), "increase")):
            assert call(L._h, lens, offsets) == _lib.FI_ERR_ARG and msg in _lib.last_error(), (msg, _lib.last_error())
        assert call(A._h, np.array([3, 10], np.uint32)) == _lib.FI_ERR_ARG and "FarmerLstm model only" in _lib.last_error()
        got = L.infer_grouped(0, z, x, off, lengths=np.array([3, 10]))
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    finally:
        L.close()
        A.close()
