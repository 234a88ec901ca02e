"""CPU checks of the policy sampling rule (fi_learner_infer_sample / fi_op_policy_sample, include/fi_learner.h): the numpy
Philox4x32-10 of tests/sampling_reference.py against Random123's known answers and a chi-square of its uniforms, the float64
sampler and greedy rule on hand-worked rows, and the operator's refusals, which happen before any device is looked for."""
import numpy as np
import pytest
from scipy import stats

import sampling_reference as R

NAN, INF = np.nan, np.inf


# ------------------------------------------------------------------------------- Philox4x32-10
KAT = [  # Random123's known-answer vectors (kat_vectors, philox4x32 10 rounds): counter, key, output
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


@pytest.mark.parametrize("ctr,key,out", KAT, ids=["zeros", "ones", "pi"])
def test_philox_known_answers(ctr, key, out):
    got = R.philox4x32_10(np.array(ctr, np.uint32), np.array(key, np.uint32))
    assert [int(x) for x in got] == list(out)


def test_philox_vectorises_over_counters():
    ctr = np.array([c for c, _, _ in KAT], np.uint64)
    key = np.array([k for _, k, _ in KAT], np.uint64)
    assert np.array_equal(R.philox4x32_10(ctr, key), np.array([o for _, _, o in KAT], np.uint32))


@pytest.mark.parametrize("seed", [0, 1, 0xDEADBEEF12345678])
def test_uniforms_pass_a_256_bin_chi_square(seed):
    u = R.uniforms(np.arange(1 << 18), seed)
    assert u.min() >= 0.0 and u.max() < 1.0
    assert np.array_equal(u, u.astype(np.float32).astype(np.float64))   # 24 bits: the kernel's fp32 u is the same number
    counts = np.bincount((u * 256).astype(np.int64), minlength=256)
    p = stats.chisquare(counts).pvalue
    print(f"seed {seed:#x}: 256-bin chi-square p = {p:.3g}")
    assert p > 1e-6


def test_seed_high_word_is_the_second_key_word():
    lo = R.uniforms(np.arange(8), 5)
    assert not np.array_equal(lo, R.uniforms(np.arange(8), 5 | (1 << 32)))
    ctr = np.zeros((8, 4), np.uint64)
    ctr[:, 0] = np.arange(8)
    x0 = R.philox4x32_10(ctr, np.array([5, 1], np.uint64))[:, 0]
    assert np.array_equal(R.uniforms(np.arange(8), 5 | (1 << 32)), (x0 >> 8) * 2.0 ** -24)


# ------------------------------------------------------------------------------- the rule on hand-worked rows
def _row(**entries):
    z = np.zeros(16, np.float32)
    for k, v in entries.items():
        z[int(k[1:])] = v
    return z


def _bits(*js):
    return int(sum(1 << j for j in js))


def _one(z, legal, seed=0, greedy=False, r=0):
    a, _, _ = R.sample(np.asarray(z, np.float32)[None], None if legal is None else np.array([legal], np.uint32), seed, greedy,
                       rows=np.array([r]))
    return int(a[0])


def test_single_legal_action_is_always_taken():
    z = np.random.default_rng(0).standard_normal(16).astype(np.float32) * 5
    for r in range(50):
        assert _one(z, _bits(9), r=r) == 9
        assert _one(z, _bits(9), r=r, greedy=True) == 9


def test_greedy_rule():
    z = _row(j3=2.0, j7=2.0, j9=5.0)
    assert _one(z, 0xFFFF, greedy=True) == 9
    assert _one(z, _bits(3, 7, 12), greedy=True) == 3                        # tie: the lowest index
    assert _one(z, None, greedy=True) == 9                                   # NULL legal = all 16
    assert _one(_row(j2=INF, j5=NAN), _bits(2, 5, 6), greedy=True) == 5      # NaN counts as largest, above +inf
    assert _one(_row(j2=INF, j5=NAN), _bits(2, 6), greedy=True) == 2         # ... but not from outside the support
    allneg = np.full(16, -INF, np.float32)
    assert _one(allneg, _bits(4, 11), greedy=True) == 4                      # all -inf in S: the lowest action in S
    assert _one(allneg, _bits(4, 11)) == 4


@pytest.mark.parametrize("fill", [NAN, INF, -INF])
def test_non_finite_logits_outside_the_support_change_nothing(fill):
    z = np.random.default_rng(1).standard_normal(16).astype(np.float32)
    sup = _bits(1, 4, 6, 13)
    zf = z.copy()
    zf[[0, 2, 15]] = fill
    for r in range(64):
        assert _one(zf, sup, r=r) == _one(z, sup, r=r)
    assert _one(zf, sup, greedy=True) == _one(z, sup, greedy=True)


@pytest.mark.parametrize("fill,expect", [(NAN, 6), (INF, 6)])
def test_nan_or_inf_inside_the_support_takes_the_greedy_action(fill, expect):
    z = _row(j1=3.0, j6=fill, j10=1.0)
    for r in range(32):
        assert _one(z, _bits(1, 6, 10), r=r) == expect


def test_minus_inf_inside_the_support_is_never_drawn():
    z = _row(j0=-INF, j5=-INF)
    sup = _bits(0, 3, 5, 8)
    got = {_one(z, sup, r=r) for r in range(400)}
    assert got == {3, 8}


def test_bits_16_to_31_are_ignored():
    z = np.random.default_rng(2).standard_normal(16).astype(np.float32)
    for r in range(64):
        assert _one(z, 0xFFFF0000 | _bits(2, 9), r=r) == _one(z, _bits(2, 9), r=r)


def test_u_on_either_side_of_a_cumulative_boundary():
    """Two legal actions {3, 7}: action 3 is drawn exactly when u < p3, the cumulative boundary. Put p3 just above and just
    below the u of counter r."""
    for r in range(5):
        u = float(R.uniforms(np.array([r]), 77)[0])
        for p3, want in ((u + 1e-4, 3), (u - 1e-4, 7)):
            z = _row(j3=np.log(p3), j7=np.log(1 - p3))
            a, alt, gap = R.sample(z[None], np.array([_bits(3, 7)], np.uint32), 77, rows=np.array([r]))
            assert (int(a[0]), int(alt[0])) == (want, 10 - want), (r, u, p3)
            assert abs(gap[0] - 1e-4) < 1e-6


def test_draws_follow_the_masked_softmax():
    z = _row(j0=1.0, j2=-0.5, j5=0.3, j9=2.0, j15=0.0)
    sup = R.supports(np.array([_bits(0, 2, 5, 9, 15)], np.uint32), 1)[0]
    n = 1 << 16
    a, _, _ = R.sample(np.repeat(z[None], n, 0), np.full(n, _bits(0, 2, 5, 9, 15), np.uint32), 3)
    p = R.masked_softmax(z, sup)
    counts = np.bincount(a, minlength=16)
    assert counts[~sup].sum() == 0
    assert stats.chisquare(counts[sup], n * p[sup]).pvalue > 1e-6


def test_vectorised_reference_equals_a_per_row_restatement():
    """sample() against the rule written out row by row, on rows with -inf / NaN / +inf mixed in and random legal words."""
    rng = np.random.default_rng(3)
    n = 2000
    z = (rng.standard_normal((n, 16)) * 3).astype(np.float32)
    special = rng.random((n, 16))
    z[special < 0.05] = -INF
    z[(special >= 0.05) & (special < 0.06)] = NAN
    z[(special >= 0.06) & (special < 0.065)] = INF
    legal = rng.integers(0, 1 << 16, n).astype(np.uint32)
    legal[::97] = 0
    got, _, _ = R.sample(z, legal, 11)
    u = R.uniforms(np.arange(n), 11)
    for r in range(n):
        idx = [j for j in range(16) if (legal[r] >> j) & 1]
        if not idx:
            assert got[r] == -1
            continue
        zz = z[r, idx].astype(np.float64)
        g = idx[int(np.argmax(zz))]
        if not np.isfinite(z[r, g]):
            assert got[r] == g, r
            continue
        w = np.exp(zz - float(z[r, g]))
        cum = np.cumsum(w)
        pick = next((idx[i] for i in range(len(idx)) if cum[i] > u[r] * cum[-1]), None)
        assert got[r] == pick, r


# ------------------------------------------------------------------------------- operator refusals (no device needed)
def test_op_refuses_narrow_head_and_bad_greedy_before_the_device(fi):
    from freeimpala_b200 import _lib
    lib = _lib.load()
    assert lib.fi_op_policy_sample(None, 15, 4, None, 0, 0, None, None) == _lib.FI_ERR_ARG
    assert "ldh" in _lib.last_error()
    assert lib.fi_op_policy_sample(None, 17, 4, None, 0, 2, None, None) == _lib.FI_ERR_ARG
    assert lib.fi_op_policy_sample(None, 17, 4, None, 0, -1, None, None) == _lib.FI_ERR_ARG
    with pytest.raises(fi.FiError):
        fi.ops.policy_sample(0, 8, 4, 0)
