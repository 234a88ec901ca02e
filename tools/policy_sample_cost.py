#!/usr/bin/env python
"""What drawing the action on the GPU costs an actor-critic actor (fi_learner_infer_sample against fi_learner_infer on the
same observations).

At 64, 1024 and 16384 rows (below and above the 256-row switch to the tensor-core forward), on one actor-critic learner in
gemm_mode auto:
1. Call time: a host clock around each call, which ends in the library's stream synchronisation. Both calls are warmed up
   first (module load, workspace growth), then they alternate for N calls each on the same observations.
2. Kernel time: one profiled window per call (fi_prof_enable brackets every launch with CUDA events), taken after the timed
   calls: per-launch device time of every kernel, among them policy_sample_kernel.
Each shape also checks that infer_sample returns the logits and values of infer bit for bit, and only legal actions.

    python tools/policy_sample_cost.py [--quick] [--out profiles/r3_policy_sample.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import freeimpala_b200 as fi


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def profile(call, n):
    fi.prof_collect()
    fi.prof_enable(True)
    for _ in range(n):
        call()
    fi.prof_enable(False)
    return {k: {"us_per_launch": round(e["total_ms"] * 1e3 / e["launches"], 3), "launches": e["launches"]}
            for k, e in sorted(fi.prof_collect().items())}


def shape(L, rows, calls, seed):
    rng = np.random.default_rng(seed)
    obs = rng.standard_normal((rows, 162)).astype(np.float32)
    legal = rng.integers(1, 1 << 16, rows).astype(np.uint32)
    run = {"infer": lambda: L.infer(0, obs), "infer_sample": lambda: L.infer_sample(0, obs, legal, seed)}
    out = {}
    for name, f in run.items():   # warm-up
        for _ in range(3):
            out[name] = f()
    (logits, values), (acts, s_logits, s_values) = out["infer"], out["infer_sample"]
    assert logits.tobytes() == s_logits.tobytes() and values.tobytes() == s_values.tobytes(), "logits / values differ"
    assert np.all((legal >> acts.astype(np.uint32)) & 1), "an action outside its legal set"
    ms = {name: [] for name in run}
    for _ in range(calls):        # alternated
        for name, f in run.items():
            t0 = time.perf_counter()
            f()
            ms[name].append((time.perf_counter() - t0) * 1e3)
    kernels = {name: profile(f, 5) for name, f in run.items()}
    med = {n: float(np.median(v)) for n, v in ms.items()}
    row = {"rows": rows, "calls": calls,
           "h2d_bytes": {"infer": rows * 162 * 4, "infer_sample": rows * (162 * 4 + 16)},
           "d2h_bytes": {"infer": rows * 17 * 4, "infer_sample": rows * (17 * 4 + 4)},
           "ms_median": {n: round(v, 4) for n, v in med.items()},
           "ms_p10_p90": {n: [round(float(np.percentile(v, 10)), 4), round(float(np.percentile(v, 90)), 4)] for n, v in ms.items()},
           "extra_ms_median": round(med["infer_sample"] - med["infer"], 4),
           "kernels": kernels}
    print(json.dumps({k: row[k] for k in ("rows", "ms_median", "extra_ms_median")}), file=sys.stderr, flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_policy_sample.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "policy_sample_cost measures the GPU: no device"
    calls = 5 if a.quick else 200
    L = fi.Learner(1, 2, 5, 2, 0, 0, "", "", 0, model="mlp_actor_critic", gemm_mode="auto")
    try:
        shapes = [shape(L, rows, calls, seed=rows) for rows in (64, 1024, 16384)]
    finally:
        L.close()
    res = {"card": card(), "what": "host clock around each call (ends in a stream synchronisation), median of alternated calls; "
                                   "kernel times from fi_prof_enable in a separate window",
           "shapes": shapes}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
