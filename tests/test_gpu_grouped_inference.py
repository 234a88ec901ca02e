"""fi_learner_infer_grouped: FarmerLstm inference of candidate actions grouped by state. Needs a B200.

A state's history z runs through the recurrence once; its candidate rows x run through the dense stack; best[s] is the
argmax within each group, computed on the device. The code paths the cases below drive (csrc/model_farmer.cu):

  tail      the FFMA recurrence owns 8 states per CTA: 7 states is one partial CTA, 9 a full one and a tail CTA of 1
  wave      1185 states = 149 CTAs: one more than the 148 SMs, so a second wave
  wide      one state with 4000 candidates: segment_argmax_kernel's warp loops 125 times over the group
  t1..t100  the recurrence's step count

Farmer inference runs every product on the fp32 FFMA kernels, and the recurrence and the dense stack are row-independent
(no split-K, no reduction across rows). So a candidate's value is the same bits whether its history came once per state or
once per candidate, and whatever other requests shared the forward: the bit-identity tests below rely on that.
"""
import threading

import numpy as np
import pytest

import _util as U

pytestmark = pytest.mark.gpu
RTOL, ATOL = 2e-5, 2e-6   # the farmer inference tolerance of test_gpu_farmer_paths.py
MAX_ROWS = 16384


def _farmer(fi):
    return fi.Learner(1, 2, 8, 2, 0, 0, "", "", 0, model="farmer_lstm")


@pytest.fixture
def learner(fi):
    L = _farmer(fi)
    L.set_params(0, U.farmer_params(41))
    yield L
    L.close()


def _groups(seed, states, t, lo, hi):
    """z [states, t, 162], x [rows, 484] and offsets [states + 1] for group sizes drawn from lo..hi."""
    rng = np.random.default_rng(seed)
    counts = rng.integers(lo, hi + 1, size=states)
    offsets = np.zeros(states + 1, np.uint32)
    offsets[1:] = np.cumsum(counts)
    z, _, _ = U.farmer_batch(seed, states, t)
    x = rng.standard_normal((int(offsets[-1]), 484)).astype(np.float32)
    return z, x, offsets


def _group_argmax(values, offsets):
    return np.array([int(np.argmax(values[offsets[s]:offsets[s + 1]])) for s in range(len(offsets) - 1)], np.int32)


def _same_bits(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


# ------------------------------------------------------------------------------- 1. against the float64 oracle
ORACLE_CASES = [(f"tail-s{s}-t{t}", 100 * s + t, s, t, 1, 64) for s in (1, 7, 9) for t in (1, 5, 33, 100)] + [
    ("wave-s1185-t5", 11855, 1185, 5, 1, 8),
    ("wave-s1185-t100", 118500, 1185, 100, 1, 8),
    ("wide-g4000-t1", 40001, 1, 1, 4000, 4000),
    ("wide-g4000-t100", 40100, 1, 100, 4000, 4000),
]


@pytest.mark.parametrize("case,seed,states,t,lo,hi", ORACLE_CASES, ids=[c[0] for c in ORACLE_CASES])
def test_grouped_inference_vs_oracle(learner, oracle, case, seed, states, t, lo, hi):
    z, x, offsets = _groups(seed, states, t, lo, hi)
    assert offsets[-1] <= MAX_ROWS
    values, best = learner.infer_grouped(0, z, x, offsets)
    want = oracle.farmer(U.farmer_params(41)).forward(np.repeat(z, np.diff(offsets), 0), x)
    np.testing.assert_allclose(values, want, rtol=RTOL, atol=ATOL, err_msg=case)
    assert np.array_equal(best, _group_argmax(values, offsets)), case
    near_ties = 0
    for s in range(states):
        w = want[offsets[s]:offsets[s + 1]]
        top = int(np.argmax(w))
        if best[s] == top:
            continue
        # the GPU's pick may differ only where two oracle values lie within the tolerance of each (both carry its error)
        tol = 2 * (ATOL + RTOL * abs(w[top]))
        assert w[top] - w[best[s]] <= tol, f"{case}: state {s} picked {best[s]} ({w[best[s]]!r}), oracle {top} ({w[top]!r})"
        near_ties += 1
    print(f"{case}: {states} states, {offsets[-1]} rows, rel_max {U.rel_max(values, want):.2e}, {near_ties} near-tie groups")


# ------------------------------------------------------------------------------- 2. bit identity
@pytest.mark.parametrize("states,t,lo,hi", [(9, 33, 1, 16), (64, 100, 16, 16), (300, 5, 1, 40)],
                         ids=["s9-t33", "s64x16-t100", "s300-t5"])
def test_grouped_values_equal_infer_on_repeated_z(learner, states, t, lo, hi):
    z, x, offsets = _groups(states * 7 + t, states, t, lo, hi)
    values, best = learner.infer_grouped(0, z, x, offsets)
    plain = learner.infer(0, np.repeat(z, np.diff(offsets), 0), x)
    assert _same_bits(values, plain)
    assert np.array_equal(best, _group_argmax(plain, offsets))


@pytest.mark.parametrize("rows,t", [(1, 1), (9, 8), (300, 100)], ids=["1x1", "9x8", "300x100"])
def test_identity_offsets_equal_plain_infer(learner, rows, t):
    z, x, _ = U.farmer_batch(rows + t, rows, t)
    values, best = learner.infer_grouped(0, z, x, np.arange(rows + 1, dtype=np.uint32))
    assert _same_bits(values, learner.infer(0, z, x))
    assert np.array_equal(best, np.zeros(rows, np.int32))


# ------------------------------------------------------------------------------- 3. ties
def test_ties_pick_the_lowest_index(fi, learner):
    t = 5
    z, _, _ = U.farmer_batch(77, 1, t)
    base = np.random.default_rng(77).standard_normal((64, 484)).astype(np.float32)
    v, _ = learner.infer_grouped(0, z, base, np.array([0, 64], np.uint32))
    m = int(np.argmax(v))
    others = [i for i in range(64) if i != m]
    # candidate lists (indices into base); identical rows give identical values
    groups = [
        [m, others[0], m, others[1], m],                        # maxima at start, middle and end -> 0
        [others[0], m, others[1], m],                           # -> 1
        [others[0], others[1], others[2], m],                   # the end only -> 3
        [others[0], others[0], others[1]],                      # duplicate rows that are not the maximum
        [m] * 37,                                               # all equal -> 0
        # 100 rows, maxima at 40, 70 and 99: lanes 8, 6 and 3 of the warp, so the tie is settled in the reduction -> 40
        [others[i % len(others)] if i not in (40, 70, 99) else m for i in range(100)],
    ]
    expect = [0, 1, 3, None, 0, 40]
    zz = np.repeat(z, len(groups), 0)
    offsets = np.zeros(len(groups) + 1, np.uint32)
    offsets[1:] = np.cumsum([len(g) for g in groups])
    xx = np.concatenate([base[g] for g in groups])
    values, best = learner.infer_grouped(0, zz, xx, offsets)
    assert np.array_equal(best, _group_argmax(values, offsets))
    for s, e in enumerate(expect):
        if e is not None:
            assert best[s] == e, f"group {s}: {best[s]} != {e}"
    assert best[3] == int(np.argmax(values[offsets[3]:offsets[4]]))
    # a NaN head weight makes every value NaN: numpy's argmax order puts NaN first, so each group's answer is 0
    params = U.farmer_params(41)
    params[-513] = np.nan   # dense6.w[0, 0]: the head's weight row is the last 512 + 1 values before its bias
    L = _farmer(fi)
    try:
        L.set_params(0, params)
        values, best = L.infer_grouped(0, zz, xx, offsets)
        assert np.isnan(values).all() and np.array_equal(best, np.zeros(len(groups), np.int32))
    finally:
        L.close()


# ------------------------------------------------------------------------------- 4. combining
def test_concurrent_grouped_and_plain_calls_are_combined(fi):
    params = U.farmer_params(42)
    L = _farmer(fi)
    try:
        L.set_params(0, params)
        callers, rounds = 16, 4
        rng = np.random.default_rng(5)
        reqs = []   # [caller][round] = ("g", z, x, offsets) | ("p", z, x)
        for a in range(callers):
            row = []
            for r in range(rounds):
                t = int(rng.choice([5, 33]))
                if (a + r) % 2 == 0:
                    row.append(("g",) + _groups(1000 * a + r, int(rng.integers(1, 5)), t, 1, 12))
                else:
                    row.append(("p",) + U.farmer_batch(1000 * a + r, int(rng.integers(1, 6)), t)[:2])
            reqs.append(row)

        def run(q):
            return L.infer_grouped(0, *q[1:]) if q[0] == "g" else (L.infer(0, *q[1:]), None)

        got = [[None] * rounds for _ in range(callers)]
        barrier = threading.Barrier(callers)

        def caller(a):
            for r in range(rounds):
                barrier.wait()
                got[a][r] = run(reqs[a][r])

        ts = [threading.Thread(target=caller, args=(a,)) for a in range(callers)]
        for th in ts:
            th.start()
        for th in ts:
            th.join(timeout=300)
        assert not any(th.is_alive() for th in ts)
        st = L.infer_stats(0)
        rows = sum(int(q[3][-1]) if q[0] == "g" else q[1].shape[0] for row in reqs for q in row)
        print(f"grouped + plain concurrent inference: {st['calls']} calls served by {st['batches']} forwards")
        assert st["calls"] == callers * rounds and st["rows"] == rows
        assert st["batches"] <= st["calls"] // 2
        for a in range(callers):   # the same request issued alone
            for r in range(rounds):
                alone = run(reqs[a][r])
                assert _same_bits(got[a][r][0], alone[0]), f"caller {a} round {r}"
                if reqs[a][r][0] == "g":
                    assert np.array_equal(got[a][r][1], alone[1]), f"caller {a} round {r}"
    finally:
        L.close()


# ------------------------------------------------------------------------------- 5. workspaces
def test_workspaces_grow_and_shrink(fi):
    """The recurrence's workspace grows with states and t, the feature rows and the dense stack with candidate rows; every
    call is compared with the same call on a learner that has served nothing else."""
    params = U.farmer_params(43)
    shapes = [(1, 1, 1), (3, 40, 5), (70, 300, 33), (65, 4000, 8), (600, 700, 100), (9, 9, 100), (2, 130, 5), (1, 1, 1)]
    L = _farmer(fi)
    try:
        L.set_params(0, params)
        for i, (states, rows, t) in enumerate(shapes):
            rng = np.random.default_rng(500 + i)
            cuts = np.sort(rng.choice(np.arange(1, rows), states - 1, replace=False)) if states > 1 else []
            offsets = np.array([0, *cuts, rows], np.uint32)
            z, _, _ = U.farmer_batch(500 + i, states, t)
            x = rng.standard_normal((rows, 484)).astype(np.float32)
            values, best = L.infer_grouped(0, z, x, offsets)
            F = _farmer(fi)
            try:
                F.set_params(0, params)
                fresh_values, fresh_best = F.infer_grouped(0, z, x, offsets)
            finally:
                F.close()
            assert _same_bits(values, fresh_values), (states, rows, t)
            assert np.array_equal(best, fresh_best), (states, rows, t)
    finally:
        L.close()


# ------------------------------------------------------------------------------- 6. refusals
def test_refusals_leave_the_learner_usable(fi, learner):
    from freeimpala_b200 import _lib
    lib = _lib.load()
    z, x, offsets = _groups(9, 3, 5, 1, 4)
    values = np.empty(int(offsets[-1]), np.float32)
    best = np.empty(3, np.int32)

    def call(h=learner._h, zp=z.ctypes.data, states=3, t=5, xp=x.ctypes.data, op=offsets.ctypes.data, vp=values.ctypes.data,
             bp=best.ctypes.data):
        return lib.fi_learner_infer_grouped(h, 0, zp, states, t, xp, op, vp, bp)

    def offs(*v):
        return np.array(v, np.uint32)

    bad = {
        "null z": dict(zp=None), "null x": dict(xp=None), "null offsets": dict(op=None),
        "values and best null": dict(vp=None, bp=None), "states 0": dict(states=0), "t 0": dict(t=0),
    }
    keep = []
    for name, o in [("offsets[0] != 0", offs(1, 2, 3, 4)), ("equal offsets", offs(0, 1, 1, 2)),
                    ("decreasing offsets", offs(0, 2, 1, 3)), ("too many rows", offs(0, 1, 2, MAX_ROWS + 1))]:
        keep.append(o)
        bad[name] = dict(op=o.ctypes.data)
    for name, kw in bad.items():
        assert call(**kw) == _lib.FI_ERR_ARG, name
    ac = fi.Learner(1, 2, 8, 2, 0, 0, "", "", 0)
    try:
        assert call(h=ac._h) == _lib.FI_ERR_ARG, "actor-critic learner"
    finally:
        ac.close()
    assert call() == _lib.FI_OK
    assert _same_bits(values, learner.infer(0, np.repeat(z, np.diff(offsets), 0), x))
    assert np.array_equal(best, _group_argmax(values, offsets))
    # only one of the two outputs
    v2 = np.empty_like(values)
    b2 = np.empty_like(best)
    assert call(vp=v2.ctypes.data, bp=None) == _lib.FI_OK and _same_bits(v2, values)
    assert call(vp=None, bp=b2.ctypes.data) == _lib.FI_OK and np.array_equal(b2, best)
    assert learner.infer_stats(0)["calls"] >= 3
    with pytest.raises(ValueError):
        learner.infer_grouped(0, z, x, offsets[:-1])


# ------------------------------------------------------------------------------- 7. published weights
def test_grouped_inference_follows_published_weights(fi, oracle):
    from oracle import pyoracle as po
    t = 8
    z, x, offsets = _groups(71, 5, t, 2, 9)
    zr = np.repeat(z, np.diff(offsets), 0)
    L = fi.Learner(1, 4, t, 4, 0, 0, "", "", 0, model="farmer_lstm")
    try:
        L.set_params(0, U.farmer_params(44))
        v0, _ = L.infer_grouped(0, z, x, offsets)
        p1 = U.farmer_params(45)
        L.set_params(0, p1)
        v1, _ = L.infer_grouped(0, z, x, offsets)
        assert not np.array_equal(v0, v1)
        assert _same_bits(v1, L.infer(0, zr, x))
        np.testing.assert_allclose(v1, oracle.farmer(p1).forward(zr, x), rtol=RTOL, atol=ATOL)
        bz, bx, btg = U.farmer_batch(72, 4, t)
        L.trainModel(0, L.stage_batch(0, po.pack_farmer_slots(bz, bx, btg)))
        L.sync(0)
        v2, b2 = L.infer_grouped(0, z, x, offsets)
        assert not np.array_equal(v1, v2)
        assert _same_bits(v2, L.infer(0, zr, x))
        assert np.array_equal(b2, _group_argmax(v2, offsets))
        np.testing.assert_allclose(v2, oracle.farmer(L.get_params(0)).forward(zr, x), rtol=RTOL, atol=ATOL)
    finally:
        L.close()
