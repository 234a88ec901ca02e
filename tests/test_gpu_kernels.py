"""Kernel-level parity (operator layer of the C ABI) against the CPU oracle. Needs a B200.

Integer/byte work (ring gather, ring protocol) is bit-exact. Floating point: Adam is
bit-exact against the oracle's fp32 restatement of libtorch's update; V-trace and the GEMMs
are compared with the float64 oracle at the tolerance written in each test.
"""
import os
import threading

import numpy as np
import pytest

import _util as U

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------- gather
@pytest.mark.parametrize("cap,slot,first,m", [(5, 1024, 0, 5), (5, 1024, 3, 4), (32, 102400, 20, 32),
                                              (7, 2048, 6, 1), (1, 1024, 0, 1), (64, 16, 63, 64),
                                              (1500, 102400, 1000, 1024)])
def test_gather_bit_exact(fi, torch_cuda, cap, slot, first, m):
    torch = torch_cuda
    rng = np.random.default_rng(cap * 31 + first)
    ring = rng.integers(0, 256, size=(cap, slot), dtype=np.uint8)
    d_ring = _dev(torch, ring)
    d_out = torch.zeros((m, slot), dtype=torch.uint8, device="cuda")
    n0 = fi.kernel_launch_count()
    fi.ops.gather(d_ring.data_ptr(), cap, slot, first, m, d_out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert fi.kernel_launch_count() == n0 + 1
    want = ring[(first + np.arange(m)) % cap]
    assert np.array_equal(d_out.cpu().numpy(), want)


def test_gather_rejects_bad_arguments(fi, torch_cuda):
    torch = torch_cuda
    d = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    with pytest.raises(fi.FiError):
        fi.ops.gather(d.data_ptr(), 4, 1024, 4, 1, d.data_ptr())      # first >= capacity
    with pytest.raises(fi.FiError):
        fi.ops.gather(d.data_ptr(), 4, 1000, 0, 1, d.data_ptr())      # slot not a multiple of 16
    with pytest.raises(fi.FiError):
        fi.ops.gather(d.data_ptr(), 2, 1024, 0, 3, d.data_ptr())      # m > capacity


# ------------------------------------------------------------------------------- ring protocol
def test_ring_replays_reference_trace(fi, torch_cuda):
    """The golden trace was recorded from the reference's SharedBuffer (tools/make_golden.py)."""
    g = np.load(os.path.join(U.GOLDEN, "ring_trace.npz"))
    ops, blob, lens = g["ops"], g["blob"], g["lens"]
    ring = fi.SharedBuffer(int(g["entry"][0]), int(g["cap"][0]))
    off = 0
    for (kind, n, _, res), ln in zip(ops, lens):
        data = blob[off:off + ln]
        off += ln
        if kind == 0:
            assert int(ring.write(data)) == res
        elif kind == 1:
            assert int(ring.try_write(data)) == res
        elif kind == 2:
            b = ring.readBatch(int(n))
            assert len(b) == res
            assert np.array_equal(b.to_host().reshape(-1), data)
        else:
            ring.setDraining()
            assert ring.readBatch(int(n)).empty() and res == 0
    ring.close()


def test_ring_matches_oracle_random_ops(fi, oracle, torch_cuda):
    rng = np.random.default_rng(7)
    entry, cap = 3, 6
    a, b = fi.SharedBuffer(entry, cap), oracle.ring(entry, cap)
    count = 0
    for _ in range(400):
        if rng.random() < 0.55 and count < cap:
            n = int(rng.choice([entry * 1024, entry * 1024, 1000, 16, entry * 1024 + 1, 0]))
            d = rng.integers(0, 256, size=n, dtype=np.uint8)
            ra, rb = a.write(d), b.write(d)
            assert int(ra) == rb
            count += int(rb == 1)
        elif count:
            m = int(rng.integers(1, count + 1))
            ba = a.readBatch(m)
            nb, ob = b.read_batch(m)
            assert len(ba) == nb == m
            assert np.array_equal(ba.to_host(), ob)
            count -= m
        assert a.getFilledCount() == b.filled_count() == count
    a.close()


def test_ring_try_write_full_and_oversize(fi, torch_cuda):
    ring = fi.SharedBuffer(1, 2)
    assert ring.try_write(b"a" * 1024) and ring.try_write(b"b" * 1024)
    assert not ring.try_write(b"c" * 1024)            # full -> false, never blocks
    assert len(ring.readBatch(1)) == 1
    assert not ring.try_write(b"c" * 1025)            # too large -> false
    assert not ring.write(b"c" * 1025)
    assert ring.getFilledCount() == 1
    with pytest.raises(fi.FiError):
        ring.readBatch(3)                             # M > capacity can never be served
    ring.close()


def test_ring_blocking_writers_and_drain(fi, torch_cuda):
    """64 writers x 2 rings like configs[2] (SURVEY.md 8d config 3): every trajectory arrives exactly
    once, per-writer order is preserved, blocked writers are released by reads, and a reader blocked
    on a drained ring gets the empty batch (data_structures.h:278-280)."""
    entry, cap, m, writers, per = 1, 8, 4, 16, 12
    ring = fi.SharedBuffer(entry, cap)

    def writer(w):
        for i in range(per):
            d = np.zeros(1024, np.uint8)
            d[:8] = np.frombuffer(np.array([w, i], np.uint32).tobytes(), np.uint8)
            d[8:] = (w * 7 + i) % 251
            assert ring.write(d)

    ts = [threading.Thread(target=writer, args=(w,)) for w in range(writers)]
    for t in ts:
        t.start()
    seen = {}
    for _ in range(writers * per // m):
        b = ring.readBatch(m).to_host()
        for row in b:
            w, i = np.frombuffer(row[:8].tobytes(), np.uint32)
            assert np.all(row[8:] == (w * 7 + i) % 251)
            assert seen.get(int(w), -1) == int(i) - 1   # FIFO per writer
            seen[int(w)] = int(i)
    for t in ts:
        t.join()
    assert all(seen[w] == per - 1 for w in range(writers)) and ring.getFilledCount() == 0
    got = []
    rd = threading.Thread(target=lambda: got.append(ring.readBatch(m)))
    rd.start()
    ring.setDraining()
    rd.join(timeout=10)
    assert got and got[0].empty()
    ring.close()


def test_ring_zero_copy_reserve_commit(fi, torch_cuda):
    ring = fi.SharedBuffer(1, 4)
    views = []
    for i in range(3):
        v, t = ring.reserve()
        v[:] = i + 1
        views.append((v, t))
    assert ring.getFilledCount() == 0
    ring.commit(views[1][1])                  # out-of-order commit: not visible before ticket 0
    assert ring.getFilledCount() == 0
    ring.commit(views[0][1])
    assert ring.getFilledCount() == 2
    ring.commit(views[2][1], 10)              # short commit keeps the slot's tail
    out = ring.readBatch(3).to_host()
    assert np.all(out[0] == 1) and np.all(out[1] == 2) and np.all(out[2, :10] == 3) and np.all(out[2, 10:] == 0)
    ring.close()


def test_ring_reserve_many_commit_many(fi, torch_cuda):
    import ctypes as C
    ring = fi.SharedBuffer(1, 8)
    ptrs, ticket = ring.reserve_many(5)
    assert len(ptrs) == 5 and ring.getFilledCount() == 0
    for i, p in enumerate(ptrs):
        C.memset(p, i + 1, 1024)
    assert ring.commit_many(ticket, 5)
    assert ring.getFilledCount() == 5
    out = ring.readBatch(5).to_host()
    assert all(np.all(out[i] == i + 1) for i in range(5))
    ptrs, ticket = ring.reserve_many(6)            # wraps around the ring end (slots 5,6,7,0,1,2)
    for i, p in enumerate(ptrs):
        C.memset(p, 10 + i, 1024)
    ring.commit_many(ticket, 6, 100)               # short commit: bytes [100, 1024) keep the previous occupant
    out = ring.readBatch(6).to_host()
    assert all(np.all(out[i, :100] == 10 + i) for i in range(6))
    # only the committed bytes travel: the tail is the slot's previous content in HBM (first batch / zero-initialised)
    assert np.all(out[3, 100:] == 1) and np.all(out[0, 100:] == 0)
    with pytest.raises(fi.FiError):
        ring.reserve_many(9)                       # more than the capacity can never be reserved
    ring.close()


def test_ring_posted_receives_complete_out_of_order(fi, torch_cuda):
    """Stand-in for the MPI receiver of freeimpala_mpi_async (cmd/freeimpala_mpi_async/main.cpp:283-297: NUM_SLOTS posted
    MPI_Irecv's, MPI_Waitany, handle, repost) with the zero-copy producer API (SURVEY.md 8f rank 1): every "receive" is
    posted straight into a reserved pinned ring slot, the "network" (a pool of threads with random delays) completes them out
    of order, and each completion commits its own ticket. The learner must see the trajectories in POSTING order, byte for
    byte, whatever the completion order, across many ring wrap-arounds, while it consumes batches concurrently."""
    import ctypes as C
    import threading
    cap, entry, m, total, posted_max = 16, 2, 4, 160, 8
    ring = fi.SharedBuffer(entry, cap)
    slot = ring.slot_bytes
    rng = np.random.default_rng(11)
    payload = rng.integers(0, 256, size=(total, slot), dtype=np.uint8)
    delays = rng.random(total) * 2e-3
    sem = threading.Semaphore(posted_max)           # at most posted_max receives outstanding, like NUM_SLOTS
    done_order, lock = [], threading.Lock()

    def complete(i, view, ticket):                  # the "network": fills the posted buffer some time later, then Waitany fires
        import time
        time.sleep(delays[i])
        view[:] = payload[i]
        with lock:
            done_order.append(i)
        assert ring.commit(ticket)
        sem.release()

    def receiver():                                 # posts receives in order; completions run on their own threads
        ts = []
        for i in range(total):
            sem.acquire()
            view, ticket = ring.reserve()           # blocks while the ring is full: back-pressure on the posting side
            t = threading.Thread(target=complete, args=(i, view, ticket))
            t.start()
            ts.append(t)
        for t in ts:
            t.join()

    rx = threading.Thread(target=receiver)
    rx.start()
    got = [ring.readBatch(m).to_host() for _ in range(total // m)]
    rx.join(timeout=60)
    assert not rx.is_alive()
    assert done_order != sorted(done_order), "the completions were meant to be out of order"
    assert np.array_equal(np.concatenate(got), payload)
    ring.close()


# ------------------------------------------------------------------------------- Adam
@pytest.mark.parametrize("kind,n", [("adam", 1514497), ("adamw", 10007), ("sgd", 4099), ("adam", 3), ("adam", 1142801)])
def test_fused_optimizer_bit_exact_vs_f32_oracle(fi, oracle, torch_cuda, kind, n):
    torch = torch_cuda
    rng = np.random.default_rng(n)
    p = rng.standard_normal(n).astype(np.float32)
    m = np.zeros(n, np.float32)
    v = np.zeros(n, np.float32)
    dp, dm, dv = _dev(torch, p), _dev(torch, m), _dev(torch, v)
    for step in range(1, 5):
        g = (rng.standard_normal(n) * 10.0 ** rng.integers(-4, 2)).astype(np.float32)
        dg = _dev(torch, g)
        fi.ops.adam(kind, 5e-4, step, n, dp.data_ptr(), dg.data_ptr(), dm.data_ptr(), dv.data_ptr(),
                    stream=torch.cuda.current_stream().cuda_stream)
        oracle.opt_update_f32(kind, 5e-4, step, p, g, m, v)
    torch.cuda.synchronize()
    assert np.array_equal(dp.cpu().numpy(), p)
    if kind != "sgd":
        assert np.array_equal(dm.cpu().numpy(), m) and np.array_equal(dv.cpu().numpy(), v)


def test_fused_adam_tracks_float64(fi, oracle, torch_cuda):
    """north_star tolerance: parameter relative error <= 1e-5 after N steps (float64 oracle)."""
    torch = torch_cuda
    rng = np.random.default_rng(3)
    n = 200003
    p = rng.standard_normal(n).astype(np.float32)
    dp, dm, dv = _dev(torch, p), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    pd, md, vd = p.astype(np.float64), np.zeros(n), np.zeros(n)
    for step in range(1, 11):
        g = rng.standard_normal(n).astype(np.float32)
        fi.ops.adam("adam", 5e-4, step, n, dp.data_ptr(), _dev(torch, g).data_ptr(), dm.data_ptr(), dv.data_ptr(),
                    stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        oracle.opt_update("adam", 5e-4, step, pd, g.astype(np.float64), md, vd)
    assert U.rel_l2(dp.cpu().numpy(), pd) < 1e-6


# ------------------------------------------------------------------------------- V-trace scan
@pytest.mark.parametrize("m,t", [(64, 100), (1, 1), (3, 31), (5, 32), (7, 33), (33, 400), (1024, 100), (2, 1000)])
@pytest.mark.parametrize("clip", [(1.0, 1.0, 1.0, 1.0), (2.0, 0.7, 1.5, 0.95)])
def test_vtrace_scan_vs_float64_oracle(fi, oracle, torch_cuda, m, t, clip):
    torch = torch_cuda
    rho_bar, c_bar, pg_rho_bar, lam = clip
    rng = np.random.default_rng(m * 1000 + t)
    log_rho = (0.5 * rng.standard_normal((m, t))).astype(np.float32)
    disc = (0.99 * (rng.random((m, t)) >= 0.02)).astype(np.float32)
    rew = rng.standard_normal((m, t)).astype(np.float32)
    val = rng.standard_normal((m, t)).astype(np.float32)
    boot = rng.standard_normal(m).astype(np.float32)
    d = [_dev(torch, a) for a in (log_rho, disc, rew, val, boot)]
    vs = torch.empty((m, t), device="cuda")
    adv = torch.empty((m, t), device="cuda")
    fi.ops.vtrace(m, t, *[x.data_ptr() for x in d], vs.data_ptr(), adv.data_ptr(), rho_bar, c_bar, pg_rho_bar, lam,
                  stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    want_vs, want_adv = oracle.vtrace(log_rho, disc, rew, val, boot, rho_bar, c_bar, pg_rho_bar, lam)
    # fp32 scan (re-associated in 32-step chunks) against the float64 recurrence: 1e-5 relative
    # to the largest target in the batch (the north_star's fp32 tolerance)
    assert U.rel_max(vs.cpu().numpy(), want_vs) < 1e-5
    assert U.rel_max(adv.cpu().numpy(), want_adv) < 1e-5


def test_vtrace_on_policy_reduces_to_nstep_returns(fi, torch_cuda):
    """Size-independent property at the BASELINE size (1024 x 100): with log_rho = 0 and
    rho_bar = c_bar = 1, vs_s is the discounted n-step return and pg_adv_s = vs_s... - V_s form."""
    torch = torch_cuda
    m, t = 1024, 100
    rng = np.random.default_rng(0)
    rew = rng.standard_normal((m, t)).astype(np.float32)
    val = rng.standard_normal((m, t)).astype(np.float32)
    boot = rng.standard_normal(m).astype(np.float32)
    disc = np.full((m, t), 0.9, np.float32)
    d = [_dev(torch, a) for a in (np.zeros((m, t), np.float32), disc, rew, val, boot)]
    vs = torch.empty((m, t), device="cuda")
    adv = torch.empty((m, t), device="cuda")
    fi.ops.vtrace(m, t, *[x.data_ptr() for x in d], vs.data_ptr(), adv.data_ptr())
    torch.cuda.synchronize()
    ret = np.empty((m, t))
    nxt = boot.astype(np.float64)
    for s in range(t - 1, -1, -1):
        nxt = rew[:, s] + 0.9 * nxt
        ret[:, s] = nxt
    assert U.rel_max(vs.cpu().numpy(), ret) < 1e-5
    vs_next = np.concatenate([ret[:, 1:], boot[:, None]], axis=1)
    assert U.rel_max(adv.cpu().numpy(), rew + 0.9 * vs_next - val) < 1e-5


# ------------------------------------------------------------------------------- fused loss head
LH_BASE = dict(rho_bar=1.0, c_bar=1.0, pg_rho_bar=1.0, lambda_=0.97, baseline_cost=0.5, entropy_cost=0.01)
# the V-trace constant sets of tests/test_gpu_ac_paths.py (distinct values, lambda = 0, c_bar > rho_bar, no clipping)
LH_C1 = dict(rho_bar=2.0, c_bar=0.7, pg_rho_bar=1.5, lambda_=0.95, baseline_cost=0.25, entropy_cost=0.05)
LH_SETS = {"c1-distinct": LH_C1, "c2-lambda0": dict(LH_BASE, lambda_=0.0, entropy_cost=0.0),
           "c3-cbar-gt-rhobar": dict(LH_BASE, rho_bar=0.5, c_bar=3.0, pg_rho_bar=0.35, lambda_=1.0, baseline_cost=1.0),
           "c4-unclipped": dict(LH_BASE, rho_bar=float("inf"), c_bar=float("inf"), pg_rho_bar=float("inf"), lambda_=1.0)}
# (m, t, constants, ldh, behaviour-logit scale, learner-logit scale)
LOSS_HEAD_CASES = (
    [pytest.param(4, 7, LH_BASE, 17, 1, 1, id="4-7"), pytest.param(64, 100, LH_BASE, 17, 1, 1, id="64-100"),
     pytest.param(3, 65, LH_BASE, 17, 1, 1, id="3-65")] +
    # 32-step chunks: one partial / exact / exact + 1-step chunk, two exact, two + 1 step, a 4-step last chunk
    [pytest.param(5, t, LH_C1, 17, 1, 1, id=f"chunks-t{t}") for t in (1, 31, 32, 33, 64, 65, 100)] +
    [pytest.param(6, 65, c, 17, 1, 1, id=f"vtrace-{k}") for k, c in LH_SETS.items()] +
    [pytest.param(5, 40, LH_C1, 20, 1, 1, id="padded-ldh20"),          # head rows of 20 floats, 3 of them padding
     # |log rho| up to ~15: every threshold clips. (Not unclipped: the trace products c_s c_{s+1} ... then reach 1e70, far
     # beyond fp32, and the targets themselves overflow.)
     pytest.param(6, 65, LH_C1, 17, 4, 1, id="mu-x4"),
     pytest.param(6, 65, LH_C1, 17, 1, 50, id="logits-x50")])          # fp32 softmax probabilities underflow to 0


@pytest.mark.parametrize("m,t,cfg,ldh,mu_scale,logit_scale", LOSS_HEAD_CASES)
def test_vtrace_loss_head_vs_oracle(fi, oracle, torch_cuda, m, t, cfg, ldh, mu_scale, logit_scale):
    from oracle import pyoracle as po
    torch = torch_cuda
    rng = np.random.default_rng(m + t)
    obs, mu, act, rew, disc, boot = U.vtrace_batch(5, m, t, done_p=0.05)
    mu = mu * np.float32(mu_scale)
    batch = po.pack_vtrace_slots(obs, mu, act, rew, disc, boot)
    head = np.full((m * t, ldh), np.nan, np.float32)     # padding columns are NaN: a kernel that reads them shows it
    head[:, :17] = rng.standard_normal((m * t, 17)).astype(np.float32)
    head[:, :16] *= np.float32(logit_scale)
    want = oracle.vtrace_losses(head[:, :16].reshape(m, t, 16), head[:, 16].reshape(m, t), mu, act, rew, disc, boot,
                                **{k: float(np.float32(v)) for k, v in cfg.items()})
    d_batch, d_head = _dev(torch, batch), _dev(torch, head)
    dhead = torch.full((m * t, ldh), 7.0, device="cuda")  # padding columns must keep this
    vs = torch.zeros(m * t, device="cuda")
    adv = torch.zeros(m * t, device="cuda")
    losses = torch.zeros(4, dtype=torch.float64, device="cuda")
    fi.ops.vtrace_loss_head(d_batch.data_ptr(), m, t, d_head.data_ptr(), ldh, dhead.data_ptr(), losses.data_ptr(),
                            vs.data_ptr(), adv.data_ptr(), stream=torch.cuda.current_stream().cuda_stream, **cfg)
    torch.cuda.synchronize()
    got = dhead.cpu().numpy()
    got_losses, got_vs, got_adv = losses.cpu().numpy(), vs.cpu().numpy(), adv.cpu().numpy()
    for name, a in (("losses", got_losses), ("dhead", got[:, :17]), ("vs", got_vs), ("pg_adv", got_adv)):
        assert np.all(np.isfinite(a)), name
    assert np.all(got[:, 17:] == 7.0)
    # Each loss is a sum over transitions. The baseline and entropy terms have one sign; the policy-gradient terms
    # -log pi(a) * adv do not, and their sum (and the total's) can cancel: 515-fold for vtrace-c1-distinct (36.7-fold at most
    # in the first three cases). fp32 terms cannot give that sum 1e-5 of itself, so a loss is held to 1e-5 relative but never
    # to less than 1e-7 of the summed term magnitudes, which is looser only where a sum cancels more than 100-fold.
    z = head[:, :16].astype(np.float64)
    z = z - z.max(axis=1, keepdims=True)
    logp = z - np.log(np.exp(z).sum(axis=1, keepdims=True))
    pg_abs = np.abs(np.take_along_axis(logp, act.reshape(-1, 1), 1)[:, 0] * want["pg_adv"].reshape(-1)).sum()
    bl_sum = 0.5 * ((want["vs"] - head[:, 16].reshape(m, t)) ** 2).sum()
    ent_abs = np.abs((np.exp(logp) * logp).sum(axis=1)).sum()
    magnitude = np.array([pg_abs + cfg["baseline_cost"] * bl_sum + cfg["entropy_cost"] * ent_abs, pg_abs, bl_sum, ent_abs])
    loss_tol = 1e-5 * np.maximum(np.abs(want["losses"]), magnitude / 100)
    errs = dict(losses=float(np.max(np.abs(got_losses - want["losses"]) / np.abs(want["losses"]))),
                vs=U.rel_max(got_vs, want["vs"]), pg_adv=U.rel_max(got_adv, want["pg_adv"]),
                dlogits=U.rel_max(got[:, :16], want["dlogits"].reshape(-1, 16)),
                dvalue=U.rel_max(got[:, 16], want["dvalue"].reshape(-1)))
    print(f"loss head m={m} t={t} ldh={ldh} mu x{mu_scale} logits x{logit_scale}: " +
          ", ".join(f"{k} {v:.2e}" for k, v in errs.items()) +
          f" (pg sum cancels {magnitude[1] / abs(want['losses'][1]):.0f}-fold)")
    assert np.all(np.abs(got_losses - want["losses"]) <= loss_tol), (got_losses, want["losses"], loss_tol)
    assert errs["vs"] < 1e-5 and errs["pg_adv"] < 1e-5
    assert errs["dlogits"] < 1e-5 and errs["dvalue"] < 1e-5


# ------------------------------------------------------------------------------- GEMM
GEMM_CASES = [("NT", 640, 512, 162, 256), ("NT", 6400, 512, 512, 512), ("NT", 100, 17, 512, 512), ("NT", 64, 1, 512, 512),
              ("NN", 640, 512, 17, 17), ("NN", 1000, 512, 512, 512), ("NN", 64, 612, 512, 512),
              ("TN", 512, 162, 6400, 512), ("TN", 512, 512, 6400, 512), ("TN", 17, 512, 3000, 17), ("TN", 512, 612, 64, 512),
              ("NT", 1, 1, 1, 1), ("NT", 129, 130, 19, 19),
              ("NT", 4096, 512, 512, 512), ("NN", 2048, 512, 512, 512), ("TN", 512, 512, 20000, 512), ("TN", 512, 162, 3333, 512),
              ("NT", 300, 100, 70, 72), ("NN", 260, 40, 33, 36), ("TN", 130, 60, 77, 132)]


@pytest.mark.parametrize("mode", ["simt", "tcgen05", "tcgen05_f16"])
@pytest.mark.parametrize("trans,m,n,k,lda", GEMM_CASES)
def test_gemm_fp32_accuracy(fi, torch_cuda, trans, m, n, k, lda, mode):
    """C = op(A) op(B) (+bias, ReLU) within fp32 rounding of the float64 product: the learner's
    1e-5 end-to-end tolerance needs every GEMM at ~1e-6, which excludes plain TF32/bf16."""
    torch = torch_cuda
    rng = np.random.default_rng(m * 7 + n * 3 + k)
    if trans == "NT":
        A = rng.standard_normal((m, lda)).astype(np.float32); B = rng.standard_normal((n, k)).astype(np.float32)
        ref = A[:, :k].astype(np.float64) @ B.astype(np.float64).T
        ldb = k
    elif trans == "NN":
        A = rng.standard_normal((m, lda)).astype(np.float32); B = rng.standard_normal((k, n)).astype(np.float32)
        ref = A[:, :k].astype(np.float64) @ B.astype(np.float64)
        ldb = n
    else:
        A = rng.standard_normal((k, lda)).astype(np.float32); B = rng.standard_normal((k, n)).astype(np.float32)
        ref = A[:, :m].astype(np.float64).T @ B.astype(np.float64)
        ldb = n
    use_epi = trans == "NT"
    bias = rng.standard_normal(n).astype(np.float32)
    if use_epi:
        ref = np.maximum(ref + bias, 0.0)
    dA, dB, dbias = _dev(torch, A), _dev(torch, B), _dev(torch, bias)
    dC = torch.full((m, n), float("nan"), device="cuda")
    ws_bytes = fi.ops.gemm_workspace_bytes(trans, m, n, k, mode)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device="cuda")
    fi.ops.gemm(trans, m, n, k, dA.data_ptr(), lda, dB.data_ptr(), ldb, dC.data_ptr(), n,
                dbias.data_ptr() if use_epi else None, use_epi, mode, ws.data_ptr(), ws_bytes,
                torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    got = dC.cpu().numpy()
    scale = np.sqrt(k) * 1.0  # |sum of k products of N(0,1)| ~ sqrt(k)
    assert np.abs(got - ref).max() < 2e-6 * scale * 4


@pytest.mark.gpu
@pytest.mark.parametrize("trans", ["NT", "NN", "TN"])
@pytest.mark.parametrize("sa,sb", [(1e-7, 3e4), (1e6, 1e-9), (1.0, 1.0)])
def test_gemm_f16_format_dynamic_range(fi, torch_cuda, trans, sa, sb):
    """3xFP16 format: per-tensor power-of-two scales keep fp32-level accuracy when the operands sit far from fp16's
    range (gradients ~1e-7, large activations) and when a few outliers set the scale 1000x above the bulk."""
    torch = torch_cuda
    m, n, k = 384, 256, 700
    rng = np.random.default_rng(5)
    shape_a = (m, k) if trans != "TN" else (k, m)
    shape_b = (n, k) if trans == "NT" else (k, n)
    A = (rng.standard_normal(shape_a) * sa).astype(np.float32)
    B = (rng.standard_normal(shape_b) * sb).astype(np.float32)
    A.flat[::977] *= 1000.0   # outliers: the scale follows max |x|, the bulk sits 10 bits lower
    B.flat[::1013] *= 1000.0
    A64, B64 = A.astype(np.float64), B.astype(np.float64)
    ref = A64 @ B64.T if trans == "NT" else (A64 @ B64 if trans == "NN" else A64.T @ B64)
    absprod = np.abs(A64) @ np.abs(B64).T if trans == "NT" else (np.abs(A64) @ np.abs(B64) if trans == "NN" else np.abs(A64).T @ np.abs(B64))
    dA, dB = _dev(torch, A), _dev(torch, B)
    dC = torch.full((m, n), float("nan"), device="cuda")
    ws_bytes = fi.ops.gemm_workspace_bytes(trans, m, n, k, "tcgen05_f16")
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device="cuda")
    fi.ops.gemm(trans, m, n, k, dA.data_ptr(), shape_a[1], dB.data_ptr(), shape_b[1], dC.data_ptr(), n, None, False,
                "tcgen05_f16", ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    got = dC.cpu().numpy().astype(np.float64)
    # element-wise: within a few fp32 ulps of the sum of |products| (what an fp32 dot product guarantees)
    assert np.all(np.abs(got - ref) <= 4e-6 * absprod / np.sqrt(k) * 8 + 1e-30), float(np.max(np.abs(got - ref) / (absprod + 1e-300)))
    assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 1e-6
