"""The data-parallel learner step on two or three B200s against the float64 full-batch reference. Needs >= 2 GPUs.

Every case starts W ranks of tests/dp_worker.py (one process and one GPU each, NCCL inside fi_learner_step) that step their
shards of the same global batches through fi_learner_step with step graphs on: from the third step on, the step is one replayed
CUDA graph with the gradient all-reduce captured inside it. The ranks only record; this file judges, at every step of every case:

  1. the all-reduced gradient arena against the teacher-forced float64 gradient of the WHOLE global batch, relative L2 < 1e-5
     (the actor-critic reference takes the ranks' ReLU decisions concatenated in shard order; FarmerLstm may miss only with
     the ReLU-kink signature of test_gpu_farmer_paths.py, computed from the saved decisions);
  2. the losses are the global ones: actor-critic sums over every rank's transitions, FarmerLstm means over the global batch;
  3. gradient arena and parameters bit-identical on every rank;
  4. with clipping, the pre-clip norm has the same bits on every rank and is the float64 norm of the reduced arena;
  5. after the last step, the teacher-forced parameters within 1e-5 and the free-running bound of _util.AdamParity.

A rank that fails before a collective leaves its peers waiting in NCCL, so the launcher runs every case under one deadline and
kills every rank's process group when the deadline passes or any rank fails.
"""
import os
import signal
import socket
import subprocess
import sys
import time

import numpy as np
import pytest

import _util as U
import dp_worker as W
import history_reference as H
from freeimpala_b200 import dp
from test_gpu_farmer_paths import KINK_GRAD_TOL, KINK_REL, KINK_UNITS, _f64_dense_preactivations, kink_signature

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEADLINE_S = 300
WORKER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "dp_worker.py")


def _device_count():
    import torch
    return torch.cuda.device_count()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _tail(path, n=40):
    with open(path, errors="replace") as f:
        return "".join(f.readlines()[-n:])


def _launch(case, world, out_dir):
    """Run the W ranks of `case`; returns their recordings. Any failure kills every rank before the test fails."""
    port = _free_port()
    procs, errs = [], []
    try:
        for r in range(world):
            errs.append(os.path.join(out_dir, f"rank{r}.stderr"))
            with open(errs[-1], "w") as ef, open(os.path.join(out_dir, f"rank{r}.stdout"), "w") as of:
                procs.append(subprocess.Popen([sys.executable, WORKER, case, str(r), str(world), str(port), out_dir],
                                              stdout=of, stderr=ef, start_new_session=True))
        deadline = time.monotonic() + DEADLINE_S
        failed = None
        while failed is None and any(p.poll() is None for p in procs):
            if time.monotonic() > deadline:
                failed = f"deadline of {DEADLINE_S} s passed"
            elif any(p.poll() not in (None, 0) for p in procs):
                failed = "a rank exited with " + str([p.returncode for p in procs])
            else:
                time.sleep(0.2)
        if failed is None and any(p.returncode != 0 for p in procs):
            failed = "a rank exited with " + str([p.returncode for p in procs])
    finally:
        for p in procs:   # every rank, also when the launcher itself is interrupted
            if p.poll() is None:
                try:
                    os.killpg(p.pid, signal.SIGKILL)
                except ProcessLookupError:
                    pass
        for p in procs:
            p.wait()
    tails = "\n".join(f"--- rank {r} stderr ---\n{_tail(e)}" for r, e in enumerate(errs))
    assert failed is None, f"{case}: {failed}\n{tails}"
    for r, e in enumerate(errs):   # the stream-launch fallback would pass without testing the captured all-reduce
        with open(e, errors="replace") as f:
            assert "step graph capture failed" not in f.read(), f"{case} rank {r}: the step ran without its graph\n{tails}"
    return [dict(np.load(os.path.join(out_dir, f"rank{r}.npz"))) for r in range(world)]


def _farmer_kinks(run, masks, params_before, batch):
    z, x = batch["data"][:2]
    pre = (H.dense_preactivations(params_before, z, x, batch["lengths"]) if "lengths" in batch else
           _f64_dense_preactivations(params_before, z, x))
    return kink_signature(masks, pre)


def _check_losses(run, got, want, what):
    if run["model"] == W.FARMER:   # the mean over the global batch
        assert abs(got[0] - want[0]) <= TOL * abs(want[0]) + 1e-7, (what, got, want)
        assert not np.any(got[1:]), (what, got)
        return
    # sums over every rank's transitions: test_gpu_optim.py's rule, with the length tests' allowance for the cancelling terms
    atol = 1e-6 * max(abs(want[0]), abs(want[1]) + 0.5 * abs(want[2]) + 0.01 * abs(want[3]))
    np.testing.assert_allclose(got, want, rtol=TOL, atol=atol, err_msg=what)


def _check_run(oracle, case, ri, run, world, ranks):
    pre, P = f"r{ri}_", run["players"]
    shards = [dp.shard_range(run["gm"], r, world) for r in range(world)]
    clip = float(ranks[0][pre + "max_grad_norm"])   # the bound the ranks computed (float64 sums may round differently here)
    assert abs(clip - W.max_grad_norm(oracle, run, 0)) <= 1e-9 * clip
    for p in range(P):
        O, F = W.new_reference(oracle, run, p), W.new_reference(oracle, run, p)   # teacher-forced, free-running
        e_grad = e_loss = 0.0
        for s in range(run["steps"]):
            k = f"{pre}p{p}_s{s}_"
            what = f"{case} run {ri} player {p} step {s}"
            batch = W.global_batch(run, p, s)[0]
            # 3. one reduced arena, one optimiser result: every rank holds the same bits
            grads, params = ranks[0][k + "grads"], ranks[0][k + "params"]
            for r in range(1, world):
                assert np.array_equal(ranks[r][k + "grads"], grads), (what, "gradient arena differs on rank", r)
                assert np.array_equal(ranks[r][k + "params"], params), (what, "parameters differ on rank", r)
            for r in range(world):
                assert int(ranks[r][k + "steps_done"]) == s + 1 + run["warmup"], what
            # 1. against the full-batch gradient, at the teacher-forced parameters
            masks = np.concatenate([ranks[r][k + "masks"] for r in range(world)], axis=1)
            params_before = O.params()
            want, g_want, n_over, max_over = W.reference_loss_grad(
                oracle, run, O, batch, relu_mask=masks if run["model"] == W.AC else None)
            assert n_over <= 4 + 2e-5 * masks.size and max_over < 1e-5, (what, n_over, max_over)
            e = U.rel_l2(grads, g_want)
            if e >= TOL and run["model"] == W.FARMER:
                n_flip, worst = _farmer_kinks(run, masks, params_before, batch)
                print(f"[{what}] grads {e:.2e} with {n_flip} ReLU kinks ({worst:.1e})")
                assert 0 < n_flip <= KINK_UNITS and worst < KINK_REL and e < KINK_GRAD_TOL, (what, e, n_flip, worst)
            else:
                assert e < TOL, (what, "all-reduced gradient vs the full batch", e)
                e_grad = max(e_grad, e)
            # 2. the global losses, f64 and the f32 read-back ring
            for r in range(world):
                _check_losses(run, ranks[r][k + "losses"], want, f"{what} rank {r} losses")
                _check_losses(run, ranks[r][k + "losses_at"], want, f"{what} rank {r} losses_at")
            e_loss = max(e_loss, U.rel_max(ranks[0][k + "losses"], want))
            # 4. the pre-clip norm: of the reduced arena, the same on every rank
            if clip:
                norm = ranks[0][k + "norm"]
                g64 = float(np.linalg.norm(grads.astype(np.float64)))
                for r in range(1, world):
                    assert ranks[r][k + "norm"].tobytes() == norm.tobytes(), (what, "norm differs on rank", r)
                assert abs(float(norm) - g64) <= 1e-6 * g64, (what, float(norm), g64)
                if s == 0:
                    assert g64 > clip, (what, "step 0 is not clipped", g64, clip)
            # the optimiser step of both references under the learner's options of this step
            F_loss, F_g = W.reference_loss_grad(oracle, run, F, batch)[:2]
            F.set_grads(F_g)
            for X in (O, F):
                X.set_opt(W.lr_at(run, s), max_grad_norm=clip, rmsprop_eps=run.get("rmsprop_eps", 1e-8),
                          rmsprop_momentum=run.get("rmsprop_momentum", 0.0))
            O.set_grads(np.asarray(grads, np.float64))
            O.opt_step()
            F.opt_step()
        # 5. the parameters after the last step
        e_forced, e_trim, e_free = U.AdamParity(O, F).check(ranks[0][k + "params"], TOL)
        print(f"[{case} run {ri} player {p}] {run['model']} {run['gm']} x {run['t']} over {world} ranks "
              f"{[hi - lo for lo, hi in shards]}: worst grads {e_grad:.2e}, losses {e_loss:.2e}; params teacher-forced "
              f"{e_forced:.2e}, free-running {e_free:.2e} (trimmed {e_trim:.2e})")


@pytest.mark.parametrize("case", list(W.CASES))
def test_data_parallel_step_vs_full_batch_reference(fi, oracle, case, tmp_path):
    world, runs = W.CASES[case]
    have = _device_count()
    if have < world:
        pytest.skip(f"{case} needs {world} CUDA devices, {have} visible")
    ranks = _launch(case, world, str(tmp_path))
    for ri, run in enumerate(runs):
        pre = f"r{ri}_"
        if run["warmup"]:   # the graph was captured before the learner joined
            assert all(np.all(r[pre + "warm_steps"] == run["warmup"]) for r in ranks)
        if run["refusals"]:   # a partial batch, then a second fi_learner_dp_init: refused alike on every rank
            err = int(ranks[0][pre + "err_state"])
            for r in range(world):
                assert list(ranks[r][pre + "codes"]) == [err, err], (r, ranks[r][pre + "codes"])
        _check_run(oracle, case, ri, run, world, ranks)
