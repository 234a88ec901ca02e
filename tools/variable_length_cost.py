#!/usr/bin/env python
"""What variable-length trajectories cost on the B200 (fi_learner_config.variable_length, record word 183).

The whole actor-critic step at 1024 x 100 (graph-replayed fi_learner_step) in gemm_mode auto and simt, three ways in one
process per mode: a learner with the option off on full trajectories, and one with it on, fed trajectories of full length
(W = 0) and of lengths uniform in 1..100 (mean ~T/2; the records past each length hold random bits). Host clock around K steps
that end in a synchronisation, the three alternated over R rounds. Then one profiled window (fi_prof: CUDA events around every
launch) per way for the kernels the option changes: the observation pre-pass (amax_split_h_kernel in auto; obs_length_kernel,
the copy the simt path adds) and the loss head.

Padding rows still run through the trunk and the head (fixed shapes), so the option is not expected to save time at mean T/2.

    python tools/variable_length_cost.py [--quick] [--out profiles/r3_variable_length.json]
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
import length_reference
from oracle import pyoracle as po

KERNELS = ["amax_split_h_kernel", "amax_split_h_kernel_length", "obs_length_kernel", "vtrace_loss_head_kernel",
           "vtrace_loss_head_kernel_length"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def whole_step(mode, m, t, K, R):
    data = U.vtrace_batch(1, m, t)
    half = np.random.default_rng(2).integers(1, t + 1, size=m).astype(np.uint32)
    slots = {"off": po.pack_vtrace_slots(*data),
             "on_full": length_reference.pack_length_slots(*data, np.zeros(m, np.uint32)),
             "on_half": length_reference.pack_length_slots(*data, half, pad="garbage")}
    Ls = {"off": fi.Learner(1, m, t, m, model="mlp_actor_critic", gemm_mode=mode),
          "on": fi.Learner(1, m, t, m, model="mlp_actor_critic", gemm_mode=mode, variable_length=True)}
    learner = {k: Ls["off" if k == "off" else "on"] for k in slots}
    try:
        batches = {k: learner[k].stage_batch(0, s) for k, s in slots.items()}
        for k in slots:                               # warm-up: first launches, graph capture
            for _ in range(4):
                learner[k].trainModel(0, batches[k])
            learner[k].sync(0)
        ms = {k: [] for k in slots}
        for _ in range(R):                            # alternated rounds
            for k in slots:
                L = learner[k]
                L.sync(0)
                t0 = time.perf_counter()
                for _ in range(K):
                    L.trainModel(0, batches[k])
                L.sync(0)
                ms[k].append((time.perf_counter() - t0) / K * 1e3)
        kern = {}
        for k in slots:                               # the changed kernels inside the step (stream launches while profiling)
            fi.prof_collect()
            fi.prof_enable(True)
            for _ in range(5):
                learner[k].trainModel(0, batches[k])
            learner[k].sync(0)
            fi.prof_enable(False)
            got = fi.prof_collect()
            kern[k] = {n: round(got[n]["total_ms"] * 1e3 / got[n]["launches"], 3) for n in KERNELS if n in got}
        med = {k: float(np.median(v)) for k, v in ms.items()}
        row = {"m": m, "t": t, "gemm_mode": mode, "steps_per_round": K, "rounds": R,
               "mean_length_on_half": float(length_reference.lengths_of(half, t).mean()),
               "ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
               "ms_per_step_all": {k: [round(x, 4) for x in v] for k, v in ms.items()},
               "on_full_over_off_pct": round(100.0 * (med["on_full"] / med["off"] - 1.0), 2),
               "on_half_over_off_pct": round(100.0 * (med["on_half"] / med["off"] - 1.0), 2),
               "kernel_us_in_step": kern}
        print(json.dumps(row), file=sys.stderr, flush=True)
        return row
    finally:
        for L in Ls.values():
            L.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_variable_length.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "variable_length_cost measures the GPU: no device"
    K, R = (5, 2) if a.quick else (30, 7)
    res = {"card": card(), "steps": [whole_step("auto", 1024, 100, K, R), whole_step("simt", 1024, 100, max(K // 3, 3), R)]}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
