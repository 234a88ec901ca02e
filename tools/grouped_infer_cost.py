#!/usr/bin/env python
"""What grouped FarmerLstm inference saves on the B200 (fi_learner_infer_grouped against fi_learner_infer on z repeated per
candidate, the way a DouZero actor scores its legal actions today).

For states in {1, 64, 1024} x candidates per state in {1, 4, 16} x t in {5, 100} (shapes over 16384 candidate rows are
skipped and listed as such), on one FarmerLstm learner:
1. Call time: a host clock around each call, which ends in the library's stream synchronisation. Both calls are warmed up
   first (module load, workspace growth), then they alternate for N calls each on the same inputs.
2. Kernel time: one profiled window per path (fi_prof_enable brackets every launch with CUDA events), taken after the timed
   calls: per-launch device time of every kernel, among them farmer_assemble_grouped_kernel and segment_argmax_kernel.
The values of the two calls are compared bit for bit, and best with the argmax of the values, on every shape.

    python tools/grouped_infer_cost.py [--quick] [--out profiles/r3_grouped_infer.json]
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

MAX_ROWS = 16384
Z_DIM, X_DIM = 162, 484


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
    return {k: round(e["total_ms"] * 1e3 / e["launches"], 3) for k, e in sorted(fi.prof_collect().items())}


def shape(L, states, k, t, calls, seed):
    rng = np.random.default_rng(seed)
    rows = states * k
    z = rng.standard_normal((states, t, Z_DIM)).astype(np.float32)
    x = rng.standard_normal((rows, X_DIM)).astype(np.float32)
    offsets = np.arange(0, rows + 1, k, dtype=np.uint32)
    z_rep = np.repeat(z, k, 0)
    run = {"replicated": lambda: (L.infer(0, z_rep, x), None), "grouped": lambda: L.infer_grouped(0, z, x, offsets)}
    out = {}
    for name, f in run.items():   # warm-up
        for _ in range(3):
            out[name] = f()
    v_rep, (v_grp, best) = out["replicated"][0], out["grouped"]
    assert v_rep.tobytes() == v_grp.tobytes(), "grouped values differ from fi_learner_infer on repeated z"
    assert np.array_equal(best, v_grp.reshape(states, k).argmax(1)), "best is not the argmax of the values"
    ms = {name: [] for name in run}
    for _ in range(calls):        # alternated
        for name, f in run.items():
            t0 = time.perf_counter()
            f()
            ms[name].append((time.perf_counter() - t0) * 1e3)
    kernels = {name: profile(f, 5) for name, f in run.items()}
    med = {n: float(np.median(v)) for n, v in ms.items()}
    row = {"states": states, "candidates": k, "t": t, "rows": rows, "calls": calls,
           "h2d_bytes": {"replicated": rows * (t * Z_DIM + X_DIM) * 4,
                         "grouped": states * t * Z_DIM * 4 + rows * X_DIM * 4 + (states + 1 + rows) * 4},
           "ms_median": {n: round(v, 4) for n, v in med.items()},
           "ms_p10_p90": {n: [round(float(np.percentile(v, 10)), 4), round(float(np.percentile(v, 90)), 4)] for n, v in ms.items()},
           "replicated_over_grouped": round(med["replicated"] / med["grouped"], 3),
           "kernel_us_per_launch": kernels}
    print(json.dumps({k: row[k] for k in ("states", "candidates", "t", "ms_median", "replicated_over_grouped")}),
          file=sys.stderr, flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_grouped_infer.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "grouped_infer_cost measures the GPU: no device"
    calls = 5 if a.quick else 50
    L = fi.Learner(1, 2, 8, 2, 0, 0, "", "", 0, model="farmer_lstm")
    rows, skipped = [], []
    try:
        for t in (5, 100):
            for states in (1, 64, 1024):
                for k in (1, 4, 16):
                    if states * k > MAX_ROWS:
                        skipped.append({"states": states, "candidates": k, "t": t, "rows": states * k})
                        continue
                    rows.append(shape(L, states, k, t, calls, seed=states * 1000 + k * 10 + t))
    finally:
        L.close()
    res = {"card": card(), "what": "host clock around each call (ends in a stream synchronisation), median of alternated calls; "
                                   "kernel times from fi_prof_enable in a separate window",
           "shapes": rows, "skipped": skipped}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
