"""Pins the CPU oracle (oracle/*.c) against the reference.

(1) Against tests/golden/*.npz, produced by tools/make_golden.py from the UNMODIFIED reference
    compiled into oracle/_ref (libtorch train_step, SharedBuffer, ModelManager). These run
    anywhere (the GPU box has no /root/reference).
(2) Live against oracle/_ref when those .so files are present.
The reference itself holds no tests or golden vectors (SURVEY.md section 8c)."""
import os

import numpy as np
import pytest

import _util as U
from oracle import pyoracle as po


def _farmer_case(g, ci):
    b, t, steps, ps, ys, bs = (int(v) for v in g[f"c{ci}_meta"])
    loss, opt = (str(v) for v in g[f"c{ci}_kind"])
    return b, t, steps, ps, ys, bs, loss, opt, float(g[f"c{ci}_lr"][0])


@pytest.mark.parametrize("ci", [0, 1, 2, 3, 4, 5, 6, 7])
def test_farmer_step_matches_reference_golden(oracle, ci):
    g = np.load(os.path.join(U.GOLDEN, "farmer_step.npz"))
    stride = int(g["stride"][0])
    b, t, steps, ps, ys, bs, loss, opt, lr = _farmer_case(g, ci)
    f = oracle.farmer(U.farmer_params(ps), opt=opt, lr=lr, loss=loss)
    z0, x0, _ = U.farmer_batch(ys, b, t)
    np.testing.assert_allclose(f.forward(z0, x0), g[f"c{ci}_y0"], rtol=2e-5, atol=2e-6)
    for s in range(steps):
        z, x, tg = U.farmer_batch(bs + s, b, t)
        l = f.loss_grad(z, x, tg)
        assert abs(l - g[f"c{ci}_losses"][s]) <= 1e-5 * abs(g[f"c{ci}_losses"][s]) + 1e-7
        ref_g = g[f"c{ci}_grads"][s]
        assert U.rel_l2(f.grads()[::stride], ref_g) < 2e-5
        f.opt_step()
    # north_star tolerance: parameter relative error <= 1e-5 after N steps (fp32 reference
    # vs float64 oracle; relative L2 over the sampled parameters)
    assert U.rel_l2(f.params()[::stride], g[f"c{ci}_params"]) < 1e-5
    psum = f.params().sum()
    assert abs(psum - g[f"c{ci}_param_sum"][0]) < 1e-5 * g[f"c{ci}_param_sum"][1]


def test_ring_trace_matches_reference_golden(oracle):
    g = np.load(os.path.join(U.GOLDEN, "ring_trace.npz"))
    ops, blob, lens = g["ops"], g["blob"], g["lens"]
    ring = oracle.ring(int(g["entry"][0]), int(g["cap"][0]))
    off = 0
    for (kind, n, _, res), ln in zip(ops, lens):
        data = blob[off:off + ln]
        off += ln
        if kind in (0, 1):
            assert ring.write(data) == res
        elif kind == 2:
            got_n, got = ring.read_batch(int(n))
            assert got_n == res
            assert np.array_equal(got.reshape(-1), data)
        else:
            ring.set_draining()
            got_n, _ = ring.read_batch(int(n))
            assert got_n == 0 == res


def test_ring_blocking_points(oracle):
    ring = oracle.ring(1, 3)
    assert ring.read_batch(1)[0] == -1          # would block: empty, not draining
    for i in range(3):
        assert ring.write(bytes([i]) * 1024) == 1
    assert ring.write(b"x" * 1024) == -1        # would block: full
    assert ring.write(b"x" * 1025) == -1        # full is checked before size (data_structures.h:223-226)
    n, out = ring.read_batch(2)
    assert n == 2 and out[0, 0] == 0 and out[1, 0] == 1
    assert ring.write(b"y" * 1025) == 0         # too large -> false
    assert ring.write(b"z" * 10) == 1           # short write keeps the stale tail
    n, out = ring.read_batch(2)
    assert bytes(out[1, :10]) == b"z" * 10 and out[1, 10] == 0  # slot 0 tail was bytes([0])


def test_checkpoint_format_golden():
    """File layout = little-endian u64 version + raw blob (data_structures.h:105-110), two files per
    save (:399-419). NOTE a reference quirk this fixture records: saveModel re-creates the Model
    (:404-405), so the reference writes freshly rand()-filled bytes with version 2, not the
    published weights. The product keeps the layout and file names but writes the real version
    and weights (DESIGN.md, deviations)."""
    g = np.load(os.path.join(U.GOLDEN, "model_ckpt.npz"))
    names = [str(n) for n in g["names"]]
    assert sorted(names) == ["model_1_7.bin", "model_1_latest.bin"]
    assert int(g["version"][0]) == 4                     # ctor generateRandomData -> 1, then 3 publishes
    files = [g[f"file_{i}"] for i in range(len(names))]
    for f in files:
        assert f.size == 8 + 4096                        # u64 version + raw bytes
        assert int(f[:8].view("<u8")[0]) == 2            # the quirk above
    assert np.array_equal(files[0], files[1])            # "latest" is a copy of the versioned file


# ---------------------------------------------------------------- live against oracle/_ref
needs_ref = pytest.mark.skipif(not po.ref_available(), reason="oracle/_ref is not in this tree (built from the reference's sources)")


@needs_ref
def test_live_ring_against_reference(oracle):
    host = po.RefHost()
    rng = np.random.default_rng(0)
    a, b = host.ring(2, 4), oracle.ring(2, 4)
    count = 0
    for _ in range(300):
        if rng.random() < 0.55 and count < 4:
            d = rng.integers(0, 256, size=int(rng.choice([2048, 100, 2049])), dtype=np.uint8)
            ra, rb = a.write(d), b.write(d)
            assert ra == rb
            count += int(ra and d.size <= 2048)
        elif count:
            m = int(rng.integers(1, count + 1))
            (na, oa), (nb, ob) = a.read_batch(m), b.read_batch(m)
            assert na == nb == m and np.array_equal(oa, ob)
            count -= m
        assert a.filled_count() == b.filled_count() == count


@needs_ref
def test_live_farmer_against_reference(oracle):
    r = po.RefNN(seed=3)
    p = r.params()                                      # libtorch's own random init
    z, x, tg = r.make_batch(11, 6, 9)                   # the reference's own generator
    f = oracle.farmer(p)
    np.testing.assert_allclose(f.forward(z, x), r.forward(z, x), rtol=2e-5, atol=2e-6)
    for s in range(3):
        lref = r.loss(z, x, tg)
        l = f.train_step(z, x, tg.reshape(-1))
        r.train_step(z, x, tg)
        assert abs(l - lref) < 1e-5 * abs(lref)
    assert U.rel_l2(f.params(), r.params()) < 1e-5


def test_adam_f32_tracks_f64(oracle):
    rng = np.random.default_rng(1)
    n = 10007
    p = rng.standard_normal(n).astype(np.float32)
    m = np.zeros(n, np.float32); v = np.zeros(n, np.float32)
    pd, md, vd = p.astype(np.float64), m.astype(np.float64), v.astype(np.float64)
    for step in range(1, 6):
        g = rng.standard_normal(n).astype(np.float32)
        oracle.opt_update_f32("adam", 5e-4, step, p, g, m, v)
        oracle.opt_update("adam", 5e-4, step, pd, g.astype(np.float64), md, vd)
    assert U.rel_l2(p, pd) < 1e-6
