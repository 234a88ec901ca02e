#!/usr/bin/env python
"""What PopArt value normalisation costs on the B200 (fi_learner_config.popart_beta).

The whole actor-critic step at 1024 x 100 (graph-replayed fi_learner_step) in gemm_mode auto and simt, with popart_beta = 0 and
3e-4 in one process per mode: host clock around K steps that end in a synchronisation, the two alternated over R rounds. Then
one profiled window (fi_prof: CUDA events around every launch) per learner for the kernels PopArt changes or adds: the loss
head (its kPopArt instantiation), popart_sums_kernel and popart_update_kernel.

    python tools/popart_cost.py [--quick] [--out profiles/r3_popart.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import _util as U
import freeimpala_b200 as fi
from oracle import pyoracle as po

KERNELS = ["vtrace_loss_head_kernel", "vtrace_loss_head_kernel_popart", "popart_sums_kernel", "popart_update_kernel",
           "fused_opt_kernel"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def whole_step(mode, m, t, K, R):
    obs, mu, act, rew, disc, boot = U.vtrace_batch(1, m, t)
    slots = po.pack_vtrace_slots(obs, mu, act, (100.0 * rew).astype(np.float32), disc, (100.0 * boot).astype(np.float32))
    Ls = {"off": fi.Learner(1, m, t, m, model="mlp_actor_critic", gemm_mode=mode),
          "popart": fi.Learner(1, m, t, m, model="mlp_actor_critic", gemm_mode=mode, popart_beta=3e-4)}
    try:
        batches = {k: L.stage_batch(0, slots) for k, L in Ls.items()}
        for k, L in Ls.items():                       # warm-up: first launches, graph capture
            for _ in range(4):
                L.trainModel(0, batches[k])
            L.sync(0)
        ms = {k: [] for k in Ls}
        for _ in range(R):                            # alternated rounds
            for k, L in Ls.items():
                L.sync(0)
                t0 = time.perf_counter()
                for _ in range(K):
                    L.trainModel(0, batches[k])
                L.sync(0)
                ms[k].append((time.perf_counter() - t0) / K * 1e3)
        kern = {}
        for k, L in Ls.items():                       # the kernels inside the step (stream launches while profiling)
            fi.prof_collect()
            fi.prof_enable(True)
            for _ in range(5):
                L.trainModel(0, batches[k])
            L.sync(0)
            fi.prof_enable(False)
            got = fi.prof_collect()
            kern[k] = {n: round(got[n]["total_ms"] * 1e3 / got[n]["launches"], 3) for n in KERNELS if n in got}
        med = {k: float(np.median(v)) for k, v in ms.items()}
        row = {"m": m, "t": t, "gemm_mode": mode, "steps_per_round": K, "rounds": R,
               "ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
               "ms_per_step_all": {k: [round(x, 4) for x in v] for k, v in ms.items()},
               "popart_over_off_us": round(1e3 * (med["popart"] - med["off"]), 1),
               "popart_over_off_pct": round(100.0 * (med["popart"] / med["off"] - 1.0), 2),
               "popart_stats": list(Ls["popart"].popart_stats(0)),
               "kernel_us_in_step": kern}
        print(json.dumps(row), file=sys.stderr, flush=True)
        return row
    finally:
        for L in Ls.values():
            L.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_popart.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "popart_cost measures the GPU: no device"
    K, R = (5, 2) if a.quick else (30, 7)
    res = {"card": card(), "steps": [whole_step("auto", 1024, 100, K, R), whole_step("simt", 1024, 100, max(K // 3, 3), R)]}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
