#!/usr/bin/env python
"""Data-parallel parity on real GPUs (run under torchrun, one rank per GPU):
every rank steps on its shard of the global batch; after fi_learner_step the all-reduced gradient arena must
equal the float64 oracle's full-batch gradient (1e-5), the all-reduced losses the full-batch losses, and the
parameters must be bit-identical on every rank.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/dp_check.py

Optimiser options (default: Adam, no clipping), e.g. RMSProp with momentum and global-norm clipping:

    ... tools/dp_check.py --optimizer rmsprop --rmsprop-momentum 0.9 --rmsprop-eps 0.01 --max-grad-norm 0.5

With clipping, every rank must also report the same pre-clip norm (fi_learner_grad_norm_at): the norm is taken after the
all-reduce, so all ranks clip with the same coefficient.
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch
import torch.distributed as dist

import _util as U
import optim_reference as R
import freeimpala_b200 as fi
from freeimpala_b200 import dp
from oracle import pyoracle as po

ap = argparse.ArgumentParser()
ap.add_argument("--optimizer", default="adam", choices=["adam", "adamw", "sgd", "rmsprop"])
ap.add_argument("--lr", type=float, default=5e-4)
ap.add_argument("--max-grad-norm", type=float, default=0.0)
ap.add_argument("--rmsprop-alpha", type=float, default=0.99)
ap.add_argument("--rmsprop-eps", type=float, default=1e-8)
ap.add_argument("--rmsprop-momentum", type=float, default=0.0)
args = ap.parse_args()
opt_kw = dict(optimizer=args.optimizer, lr=args.lr, max_grad_norm=args.max_grad_norm, rmsprop_alpha=args.rmsprop_alpha,
              rmsprop_eps=args.rmsprop_eps, rmsprop_momentum=args.rmsprop_momentum)
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ok = True
for model, mode in (("mlp_actor_critic", "simt"), ("mlp_actor_critic", "auto"), ("farmer_lstm", "simt")):
    gm, t = 4 * world, 9
    lo, hi = dp.shard_range(gm, rank, world)
    L = fi.Learner(1, max(hi - lo, 2), t, hi - lo, model=model, device=local, gemm_mode=mode, **opt_kw)
    dp.init_learner_dp(L, rank, world)
    o = po.Oracle()
    if model == "mlp_actor_critic":
        params = U.ac_params(4)
        full = U.vtrace_batch(21, gm, t)
        slots = po.pack_vtrace_slots(*[a[lo:hi] for a in full])
        O = R.OptOracle.actor_critic(o, params, opt=args.optimizer, lr=args.lr)
        want = O.loss_grad(*full)
    else:
        params = U.farmer_params(4)
        z, x, tg = U.farmer_batch(22, gm, t)
        slots = po.pack_farmer_slots(z[lo:hi], x[lo:hi], tg[lo:hi])
        O = R.OptOracle.farmer(o, params, opt=args.optimizer, lr=args.lr)
        want = np.array([O.loss_grad(z, x, tg), 0, 0, 0])
    O.set_opt(args.lr, max_grad_norm=args.max_grad_norm, rmsprop_alpha=args.rmsprop_alpha, rmsprop_eps=args.rmsprop_eps,
              rmsprop_momentum=args.rmsprop_momentum)
    L.set_params(0, params)
    L.trainModel(0, L.stage_batch(0, slots))
    got_l, got_g, got_p = L.last_losses(0), L.get_grads(0), L.get_params(0)
    e_g = U.rel_l2(got_g, O.grads())
    e_l = np.abs(got_l - want).max() / np.abs(want).max()
    O.opt_step()
    e_p = U.rel_l2(got_p, O.params())
    p_all = [torch.zeros(got_p.size, device="cuda") for _ in range(world)]
    dist.all_gather(p_all, torch.from_numpy(got_p).cuda())
    same = all(torch.equal(p_all[0], q) for q in p_all)
    norm_txt = ""
    if args.max_grad_norm > 0:   # every rank clipped with the norm of the same all-reduced arena
        n_all = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(n_all, torch.tensor([L.grad_norm_at(0, 1)], dtype=torch.float64, device="cuda"))
        same_norm = all(torch.equal(n_all[0], q) for q in n_all)
        same &= same_norm
        norm_txt = f"norm {float(n_all[0].item()):.6e} on every rank {same_norm} "
    good = e_g < 1e-5 and e_l < 1e-5 and same
    ok &= good
    if rank == 0:
        print(f"dp_check world={world} {model}/{mode} {args.optimizer} clip={args.max_grad_norm}: grads rel_l2 {e_g:.2e} "
              f"losses {e_l:.2e} params(after the update) {e_p:.2e} {norm_txt}replicas bit-identical {same} -> "
              f"{'OK' if good else 'FAIL'}", flush=True)
    L.close()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
