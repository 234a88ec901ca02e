#!/usr/bin/env python
"""What legal-action masking costs on the B200 (fi_learner_config.legal_action_mask, record word 182).

1. The fused loss head alone (vtrace_loss_head_kernel against vtrace_loss_head_kernel_legal) on a gathered 1024 x 100 batch
   with random legal words: fi_prof_enable brackets every launch with CUDA events; the two kernels alternate in rounds of
   N launches each, in one process, on the same batch and head rows (105 MB of records, so the L2 state is the same for
   both). The masked kernel reads no extra bytes: word 182 sits in the 16-byte load of words 180..183.
2. The whole actor-critic step at 1024 x 100 (gemm_mode auto, graph-replayed fi_learner_step): a learner with the mask
   off against one with it on, host clock around K steps that end in a synchronisation, alternated over R rounds; then one
   profiled window per learner for the loss head's time inside the step.

    python tools/legal_mask_cost.py [--quick] [--out profiles/r3_legal_mask.json]
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
import legal_reference

HEADS = {"unmasked": "vtrace_loss_head_kernel", "masked": "vtrace_loss_head_kernel_legal"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def legal_words(seed, act):
    """Random legal sets that contain the action taken, one transition in eight a forced move."""
    rng = np.random.default_rng(seed)
    legal = rng.integers(0, 1 << 16, size=act.shape).astype(np.uint32) | (np.uint32(1) << act.astype(np.uint32))
    legal[rng.random(act.shape) < 0.125] = 0
    return legal


def head_alone(m, t, rounds, n):
    obs, mu, act, rew, disc, boot = U.vtrace_batch(1, m, t)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
    batch = dev(legal_reference.pack_vtrace_slots_legal(obs, mu, act, rew, disc, boot, legal_words(2, act)))
    head = dev(np.random.default_rng(3).standard_normal((m * t, 17)).astype(np.float32))
    dhead = torch.empty((m * t, 17), device="cuda")
    losses = torch.zeros(4, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def launch(masked):
        fi.ops.vtrace_loss_head(batch.data_ptr(), m, t, head.data_ptr(), 17, dhead.data_ptr(), losses.data_ptr(),
                                stream=st, legal_mask=masked)

    for masked in (False, True):          # warm-up: module load, first launches
        for _ in range(5):
            launch(masked)
    torch.cuda.synchronize()
    us = {k: [] for k in HEADS}
    for _ in range(rounds):
        for k, name in HEADS.items():
            fi.prof_collect()
            fi.prof_enable(True)
            for _ in range(n):
                launch(k == "masked")
            torch.cuda.synchronize()
            fi.prof_enable(False)
            e = fi.prof_collect()[name]
            us[k].append(e["total_ms"] * 1e3 / e["launches"])
    bytes_per_launch = 212.0 * m * t
    med = {k: float(np.median(v)) for k, v in us.items()}
    row = {"m": m, "t": t, "rounds": rounds, "launches_per_round": n, "algorithmic_bytes": bytes_per_launch,
           "us_median": {k: round(v, 3) for k, v in med.items()},
           "us_all": {k: [round(x, 3) for x in v] for k, v in us.items()},
           "gbs_median": {k: round(bytes_per_launch / v / 1e3, 1) for k, v in med.items()},
           "masked_minus_unmasked_us": round(med["masked"] - med["unmasked"], 3)}
    print(json.dumps(row), file=sys.stderr, flush=True)
    return row


def whole_step(m, t, K, R):
    data = U.vtrace_batch(1, m, t)
    slots = legal_reference.pack_vtrace_slots_legal(*data, legal_words(2, data[2]))
    Ls = {"unmasked": fi.Learner(1, m, t, m, model="mlp_actor_critic"),
          "masked": fi.Learner(1, m, t, m, model="mlp_actor_critic", legal_action_mask=True)}
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
        head_us = {}
        for k, L in Ls.items():                       # the loss head inside the step (stream launches while profiling)
            fi.prof_collect()
            fi.prof_enable(True)
            for _ in range(5):
                L.trainModel(0, batches[k])
            L.sync(0)
            fi.prof_enable(False)
            e = fi.prof_collect()[HEADS[k]]
            head_us[k] = round(e["total_ms"] * 1e3 / e["launches"], 3)
        med = {k: float(np.median(v)) for k, v in ms.items()}
        row = {"m": m, "t": t, "gemm_mode": "auto", "steps_per_round": K, "rounds": R,
               "ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
               "ms_per_step_all": {k: [round(x, 4) for x in v] for k, v in ms.items()},
               "masked_over_unmasked_pct": round(100.0 * (med["masked"] / med["unmasked"] - 1.0), 2),
               "loss_head_us_in_step": head_us}
        print(json.dumps(row), file=sys.stderr, flush=True)
        return row
    finally:
        for L in Ls.values():
            L.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_legal_mask.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "legal_mask_cost measures the GPU: no device"
    rounds, n, K, R = (3, 20, 5, 2) if a.quick else (9, 200, 30, 7)
    res = {"card": card(), "loss_head_alone": head_alone(1024, 100, rounds, n), "step": whole_step(1024, 100, K, R)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
