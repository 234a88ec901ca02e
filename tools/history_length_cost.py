#!/usr/bin/env python
"""What variable-length move histories cost on the B200 (fi_learner_config.history_length, record word 183).

The FarmerLstm step at 1024 x 100 (graph-replayed fi_learner_step) in gemm_mode auto and simt, four ways in one process per
mode: a learner with the option off on full histories, and three with it on, fed histories of full length (W = 0), of lengths
uniform in 1..100 and of length 25 everywhere (the records past each length hold random bits). Host clock around K steps
that end in a synchronisation, the four alternated over R rounds. Then one profiled window (fi_prof: CUDA events around every
launch) per way for the recurrent kernels and the z pre-passes the option changes.

Inference: 64 states x 16 candidates with lengths uniform in 1..100, one fi_learner_infer_grouped_lengths call against one
fi_learner_infer_grouped call per distinct length (host clock, median of R rounds).

    python tools/history_length_cost.py [--quick] [--out profiles/r3_history_length.json]
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
import history_reference as H
from oracle import pyoracle as po

KERNELS = ["lstm_forward_kernel", "lstm_forward_kernel_length", "lstm_backward_kernel", "lstm_backward_kernel_length",
           "amax_split_h_kernel", "amax_split_h_kernel_length", "obs_length_kernel"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def whole_step(mode, m, t, K, R):
    z, x, tg = U.farmer_batch(1, m, t)
    uniform = np.random.default_rng(2).integers(1, t + 1, size=m).astype(np.uint32)
    slots = {"off": po.pack_farmer_slots(z, x, tg),
             "on_full": H.pack_history_slots(z, x, tg, np.zeros(m, np.uint32)),
             "on_uniform": H.pack_history_slots(z, x, tg, uniform, pad="garbage"),
             "on_25": H.pack_history_slots(z, x, tg, np.full(m, 25, np.uint32), pad="garbage")}
    kw = dict(model="farmer_lstm", gemm_mode=mode)
    # one learner per way: stage_batch copies into the learner's one device batch buffer
    learner = {k: fi.Learner(1, m, t, m, history_length=k != "off", **kw) for k in slots}
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
               "mean_length_on_uniform": float(uniform.mean()),
               "ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
               "ms_per_step_all": {k: [round(v, 4) for v in vs] for k, vs in ms.items()},
               "over_off_pct": {k: round(100.0 * (med[k] / med["off"] - 1.0), 2) for k in slots if k != "off"},
               "kernel_us_in_step": kern}
        print(json.dumps(row), file=sys.stderr, flush=True)
        return row
    finally:
        for L in learner.values():
            L.close()


def inference(R):
    states, cand, t = 64, 16, 100
    rng = np.random.default_rng(3)
    z = rng.standard_normal((states, t, 162)).astype(np.float32)
    x = rng.standard_normal((states * cand, 484)).astype(np.float32)
    lens = rng.integers(1, t + 1, size=states)
    off = np.arange(0, states * cand + 1, cand, dtype=np.uint32)
    groups = {int(n): np.flatnonzero(lens == n) for n in np.unique(lens)}
    L = fi.Learner(1, 8, 8, 8, model="farmer_lstm")
    try:
        L.set_params(0, U.farmer_params(4))

        def one_call():
            return L.infer_grouped(0, z, x, off, lengths=lens)

        def per_length():
            for n, idx in groups.items():
                xs = np.concatenate([x[off[s]:off[s + 1]] for s in idx])
                L.infer_grouped(0, np.ascontiguousarray(z[idx, :n]), xs, np.arange(0, len(idx) * cand + 1, cand, dtype=np.uint32))

        ways = {"lengths_one_call": one_call, "grouped_per_length": per_length}
        for f in ways.values():
            for _ in range(3):
                f()
        ms = {k: [] for k in ways}
        for _ in range(R):
            for k, f in ways.items():
                t0 = time.perf_counter()
                for _ in range(10):
                    f()
                ms[k].append((time.perf_counter() - t0) / 10 * 1e3)
        med = {k: float(np.median(v)) for k, v in ms.items()}
        row = {"states": states, "candidates_per_state": cand, "t": t, "distinct_lengths": len(groups),
               "ms_per_decision_batch_median": {k: round(v, 4) for k, v in med.items()},
               "ms_all": {k: [round(v, 4) for v in vs] for k, vs in ms.items()}}
        print(json.dumps(row), file=sys.stderr, flush=True)
        return row
    finally:
        L.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_history_length.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "history_length_cost measures the GPU: no device"
    K, R = (5, 2) if a.quick else (20, 5)
    res = {"card": card(), "steps": [whole_step("auto", 1024, 100, K, R), whole_step("simt", 1024, 100, max(K // 4, 3), R)],
           "inference": inference(R)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
