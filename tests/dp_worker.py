"""One rank of one data-parallel case of tests/test_gpu_dp.py (not collected by pytest: the test starts W of these).

    python tests/dp_worker.py CASE RANK WORLD PORT OUT_DIR

The rank runs on device RANK among the visible devices. A gloo process group on 127.0.0.1 carries the NCCL ids of
fi_learner_dp_init and the barriers; the gradients travel over the learner's own NCCL communicators. The rank steps its shard
(dp.shard_range) of every global batch through fi_learner_step with step graphs on (FI_GRAPH unset) and writes rank{RANK}.npz
with what each step left behind: losses, the all-reduced gradient arena, the parameters, the ReLU decisions, the pre-clip norm
and steps_done. It judges nothing: a rank that stopped between collectives would leave its peers waiting in NCCL, so every
comparison happens in the parent, after all ranks have exited.

The cases and their global batches are defined here and nowhere else; the parent rebuilds the same batches from the same seeds.
"""
from __future__ import annotations

import os
import sys
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

import _util as U  # noqa: E402
import history_reference as H  # noqa: E402
import length_reference as LR  # noqa: E402
from freeimpala_b200 import dp  # noqa: E402
from oracle import pyoracle as po  # noqa: E402

AC, FARMER = "mlp_actor_critic", "farmer_lstm"
LR0 = {"adam": 5e-4, "sgd": 1e-2, "rmsprop": 2e-4}


def _run(model, gm, t, steps=4, opt="adam", gemm_mode="auto", loss=None, players=1, seed=0, **extra):
    """One learner's part of a case. extra: lengths / legal (batch contents), clip (bound = clip x the step-0 norm of the
    full-batch gradient), lr_schedule, feed ("stage" or "ring"), warmup (local steps before fi_learner_dp_init),
    refusals (a refused partial step first, a refused second fi_learner_dp_init after step 1)."""
    return dict(model=model, gm=gm, t=t, steps=steps, opt=opt, gemm_mode=gemm_mode, loss=loss, players=players, seed=seed,
                lengths=extra.pop("lengths", False), legal=extra.pop("legal", False), clip=extra.pop("clip", 0.0),
                lr_schedule=extra.pop("lr_schedule", False), feed=extra.pop("feed", "stage"),
                warmup=extra.pop("warmup", 0), refusals=extra.pop("refusals", False), **extra)


AC_UNEVEN = dict(model=AC, gm=9, t=33, seed=11)
FARMER_UNEVEN = [dict(model=FARMER, gm=9, t=33, loss="mse", gemm_mode="simt", seed=21),
                 dict(model=FARMER, gm=9, t=33, loss="huber", gemm_mode="auto", seed=22)]

# case -> (world, runs)
CASES = {
    "ac-uneven": (2, [_run(**AC_UNEVEN)]),
    "ac-options": (2, [_run(AC, 64, 100, opt="rmsprop", gemm_mode="tcgen05_f16", seed=31, lengths=True, legal=True, clip=0.1,
                            lr_schedule=True, rmsprop_momentum=0.9, rmsprop_eps=0.01)]),
    "farmer-uneven": (2, [_run(**r) for r in FARMER_UNEVEN]),
    "farmer-history": (2, [_run(FARMER, 65, 33, seed=41, lengths=True, clip=0.1)]),
    "ring-fed": (2, [_run(AC, 16, 33, seed=51, feed="ring")]),
    "two-players": (2, [_run(AC, 9, 33, seed=61, players=2)]),
    "join-after-capture": (2, [_run(AC, 9, 33, opt="sgd", seed=71, warmup=3, steps=3),
                               _run(FARMER, 9, 33, opt="sgd", seed=72, warmup=3, steps=3)]),
    "refusals": (2, [_run(AC, 9, 33, seed=81, refusals=True)]),
    "world-3": (3, [_run(**dict(AC_UNEVEN, gm=10)), _run(**dict(FARMER_UNEVEN[0], gm=10))]),
}


def params_of(run, player):
    return (U.ac_params if run["model"] == AC else U.farmer_params)(run["seed"] * 10 + player)


def _length_words(seed, m, t):
    """Length words with L = 1 and L = t in every shard of two (both ends and the middle), full lengths also written as
    W = 0 and W > t; for the FarmerLstm histories also L = 7, 8, 9 (x spans records 0..7)."""
    rng = np.random.default_rng(seed)
    L = rng.integers(1, t + 1, size=m)
    fixed = [1, t, 7, 8, 9]
    for i, v in enumerate(fixed):
        L[i] = L[m // 2 + i] = v
    L[-1] = t
    words = L.astype(np.uint32)
    words[m // 2 + 1] = 0
    words[-1] = t + 5
    return words


def global_batch(run, player, step):
    """(data, slots) of the global batch of `step` (negative: warm-up steps). data are the arrays the float64 reference
    takes, slots the packed records [gm, t * record bytes]; rank r steps slots[lo:hi] of dp.shard_range."""
    m, t = run["gm"], run["t"]
    seed = 1000 * run["seed"] + 100 * player + step + 50
    if run["model"] == AC:
        data = U.vtrace_batch(seed, m, t, done_p=0.03)
        if not (run["lengths"] or run["legal"]):
            return dict(data=data), po.pack_vtrace_slots(*data)
        import test_gpu_legal_actions as GL
        legal = GL._legal_words(seed + 7, data[2]) if run["legal"] else None
        words = _length_words(seed + 3, m, t) if run["lengths"] else np.zeros(m, np.uint32)
        return (dict(data=data, legal=legal, lengths=LR.lengths_of(words, t)),
                LR.pack_length_slots(*data, words, legal=legal, pad="garbage"))
    z, x, tg = U.farmer_batch(seed, m, t)
    if not run["lengths"]:
        return dict(data=(z, x, tg)), po.pack_farmer_slots(z, x, tg)
    words = _length_words(seed + 3, m, t)
    return (dict(data=(z, x, tg), lengths=H.lengths_of(words, t)),
            H.pack_history_slots(z, x, tg, words, pad="garbage"))


def reference_loss_grad(oracle, run, model, batch, relu_mask=None):
    """(losses, grads) of the float64 reference on a whole global batch at the parameters of `model` (an
    optim_reference.OptOracle). Actor-critic: relu_mask pins the ReLU decisions (C oracle, or length_reference with legal
    words / lengths); also returns (units overridden, largest |z|/rms among them)."""
    data = batch["data"]
    if run["model"] == FARMER:
        if "lengths" in batch:
            loss, g = H.loss_grad_history(model, *data, batch["lengths"])
            return np.array([loss, 0, 0, 0]), g, 0, 0.0
        loss = model.loss_grad(*data)
        return np.array([loss, 0, 0, 0]), model.grads(), 0, 0.0
    if "lengths" in batch:
        return LR.ac_loss_grad_length(oracle, model.params(), *data, batch["legal"], batch["lengths"], relu_mask=relu_mask)
    if relu_mask is None:
        return model.loss_grad(*data), model.grads(), 0, 0.0
    losses, n_over, max_over = model.loss_grad_masked(*data, relu_mask)
    return losses, model.grads(), n_over, max_over


def new_reference(oracle, run, player):
    import optim_reference as R
    make = R.OptOracle.actor_critic if run["model"] == AC else R.OptOracle.farmer
    kw = {} if run["model"] == AC else dict(loss=run["loss"] or "mse")
    return make(oracle, params_of(run, player), opt=run["opt"], lr=LR0[run["opt"]], **kw)


def max_grad_norm(oracle, run, player):
    """The clipping bound: run["clip"] x the norm of the full-batch gradient of step 0 (0 = no clipping)."""
    if not run["clip"]:
        return 0.0
    g = reference_loss_grad(oracle, run, new_reference(oracle, run, player), global_batch(run, player, 0)[0])[1]
    return run["clip"] * float(np.linalg.norm(g))


def lr_at(run, step):
    """The learning rate of `step`: constant, or changed before every step (lr_schedule)."""
    lr0 = LR0[run["opt"]]
    return lr0 * (1.0 - 0.2 * step) if run["lr_schedule"] else lr0


def _learner_kwargs(run, clip):
    kw = dict(model=run["model"], optimizer=run["opt"], lr=LR0[run["opt"]], gemm_mode=run["gemm_mode"], max_grad_norm=clip,
              rmsprop_momentum=run.get("rmsprop_momentum", 0.0), rmsprop_eps=run.get("rmsprop_eps", 1e-8))
    if run["loss"]:
        kw["loss"] = run["loss"]
    if run["model"] == AC:
        kw.update(legal_action_mask=run["legal"], variable_length=run["lengths"])
    else:
        kw["history_length"] = run["lengths"]
    return kw


def run_rank(case, rank, world, out_dir):
    import torch.distributed as dist

    import freeimpala_b200 as fi
    from freeimpala_b200 import _lib
    oracle = po.Oracle()
    out = {}
    for ri, run in enumerate(CASES[case][1]):
        lo, hi = dp.shard_range(run["gm"], rank, world)
        m, t, P = hi - lo, run["t"], run["players"]
        clip = max_grad_norm(oracle, run, 0)
        L = fi.Learner(P, max(m, 2), t, m, device=rank, **_learner_kwargs(run, clip))
        pre = f"r{ri}_"
        for p in range(P):
            L.set_params(p, params_of(run, p))
        for w in range(run["warmup"]):   # local steps on this rank's shard: the step graph is captured before joining
            for p in range(P):
                L.trainModel(p, L.stage_batch(p, global_batch(run, p, -1 - w)[1][lo:hi]))
        if run["warmup"]:
            out[pre + "warm_steps"] = np.array([L.steps_done(p) for p in range(P)])
            for p in range(P):   # every rank starts the data-parallel steps from the same parameters (SGD keeps no state)
                L.set_params(p, params_of(run, p))
        dp.init_learner_dp(L, rank, world)
        codes = []
        if run["refusals"]:   # every rank makes the same refused call: nothing collective runs
            try:
                L.trainModel(0, L.stage_batch(0, global_batch(run, 0, 0)[1][lo:hi - 1]))
                codes.append(0)
            except fi.FiError as e:
                codes.append(e.code)
        for s in range(run["steps"]):
            for p in range(P):
                if run["lr_schedule"]:
                    L.set_lr(p, lr_at(run, s))
                slots = global_batch(run, p, s)[1][lo:hi]
                if run["feed"] == "ring":
                    ring = L.getSharedBuffers()[p]
                    assert ring.write_many(slots) == m
                    batch = ring.readBatch(m)
                else:
                    batch = L.stage_batch(p, slots)
                L.trainModel(p, batch)
                L.sync(p)
                k = f"{pre}p{p}_s{s}_"
                out[k + "losses"] = L.last_losses(p)
                out[k + "losses_at"] = L.losses_at(p, L.steps_done(p))
                out[k + "grads"] = L.get_grads(p)
                out[k + "params"] = L.get_params(p)
                out[k + "masks"] = L.debug_relu_masks(p, m * t if run["model"] == AC else m)
                out[k + "steps_done"] = np.array(L.steps_done(p))
                if clip:
                    out[k + "norm"] = np.array(L.grad_norm_at(p, L.steps_done(p)))
            if run["refusals"] and s == 1:
                try:
                    dp.init_learner_dp(L, rank, world)
                    codes.append(0)
                except fi.FiError as e:
                    codes.append(e.code)
        out[pre + "codes"] = np.array(codes, np.int64)
        out[pre + "max_grad_norm"] = np.array(clip)
        out[pre + "err_state"] = np.array(_lib.FI_ERR_STATE)
        L.close()
        dist.barrier()
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **out)


def main(argv):
    case, rank, world, port, out_dir = argv[0], int(argv[1]), int(argv[2]), int(argv[3]), argv[4]
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        run_rank(case, rank, world, out_dir)
    except BaseException:
        # No cleanup: closing the learner would wait on collectives the other ranks may never join. The parent kills the
        # remaining ranks and reports this trace.
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1:])
