#!/usr/bin/env python
"""RMSProp and gradient clipping on the B200: the two kernels against the HBM roofline, and what they cost in the step.

1. grad_norm_clip_kernel (4 B/param) and fused_opt_kernel as RMSProp (20 B/param, 28 with momentum; Adam's 28 beside them)
   at P = 1,142,801 (actor-critic) and 1,514,497 (FarmerLstm), 8 M and 64 M parameters. The two model sizes are timed the way
   the learner runs them: one arena, re-read every launch, so it is L2-resident (4.6 / 6.1 MB of gradient). 8 M and 64 M
   rotate over buffer sets whose footprint exceeds the 126 MB L2, so every launch reads HBM. Launches are captured into
   one CUDA graph and timed with CUDA events; the roofline is the 7.7 TB/s of NVIDIA's B200 data sheet.
2. The V-trace actor-critic and the FarmerLstm step at 1024 x 100, batch resident in HBM, graph-replayed steps, host clock
   around K steps ending in a synchronisation: Adam without clipping against RMSProp (eps 0.01) with clipping at a global
   norm of 40, alternated in one process, R rounds each; then one profiled window per configuration for the per-kernel times.

    python tools/optim_sweep.py [--quick] > optim.json
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

L2_BYTES = 126 * 2 ** 20
HBM_GBS = 7700.0   # NVIDIA B200 data sheet (one GPU of an HGX B200)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def time_graph(launch, nsets, iters):
    """Mean microseconds per launch of `iters` launches captured into one CUDA graph (launch(i, stream): buffer set i % nsets)."""
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for i in range(min(nsets, 3)):
            launch(i, side.cuda_stream)           # warm-up outside the capture (also creates the op's per-stream scratch)
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for i in range(iters):
                launch(i, side.cuda_stream)
        g.replay()
        side.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = float("inf")
        for _ in range(3):
            e0.record(side)
            g.replay()
            e1.record(side)
            side.synchronize()
            best = min(best, e0.elapsed_time(e1) * 1e3 / iters)
    return best


def kernel_rows(quick):
    rows = []
    for n in (1142801, 1514497, 8 << 20, 64 << 20):
        resident = n < 4 << 20
        for name, per_param in (("grad_norm_clip_kernel", 4), ("rmsprop", 20), ("rmsprop+momentum", 28), ("adam", 28)):
            bytes_per_set = per_param * n
            nsets = 1 if resident else int(min(max(2, np.ceil(1.5 * L2_BYTES / bytes_per_set) + 1), max(2, (6 << 30) // bytes_per_set)))
            sets = []
            for _ in range(nsets):
                b = {k: torch.randn(n, device="cuda") * 1e-3 for k in ("p", "g")}
                b.update({k: torch.zeros(n, device="cuda") for k in ("m", "v")})
                b["norm"] = torch.zeros(1, dtype=torch.float64, device="cuda")
                b["coef"] = torch.full((1,), 0.5, device="cuda")
                sets.append(b)

            def launch(i, st, name=name, sets=sets, n=n):
                b = sets[i % len(sets)]
                if name == "grad_norm_clip_kernel":
                    fi.ops.grad_norm_clip(n, b["g"].data_ptr(), 40.0, b["norm"].data_ptr(), b["coef"].data_ptr(), stream=st)
                elif name == "adam":
                    fi.ops.adam("adam", 5e-4, 1, n, b["p"].data_ptr(), b["g"].data_ptr(), b["m"].data_ptr(), b["v"].data_ptr(), stream=st)
                else:
                    mom = 0.9 if name == "rmsprop+momentum" else 0.0
                    fi.ops.rmsprop(6e-4, n, b["p"].data_ptr(), b["g"].data_ptr(), b["v"].data_ptr(), b["m"].data_ptr(), eps=0.01,
                                   momentum=mom, coef=b["coef"].data_ptr(), stream=st)
            iters = 20 if quick else (200 if n < 16 << 20 else 50)
            us = time_graph(launch, nsets, iters)
            gbs = bytes_per_set / us / 1e3
            rows.append({"kernel": name, "params": n, "l2_resident": resident, "bytes": bytes_per_set, "us": round(us, 2),
                         "gbs": round(gbs, 1), "frac_of_7.7TBs": round(gbs / HBM_GBS, 3)})
            print(f"{name:24s} P={n:>9d} {'L2-resident' if resident else 'HBM (rotating)':15s} {bytes_per_set / 1e6:8.2f} MB "
                  f"{us:9.2f} us {gbs:8.1f} GB/s {gbs / HBM_GBS:.3f}", file=sys.stderr, flush=True)
            del sets
            torch.cuda.empty_cache()
    return rows


CONFIGS = {"adam": dict(optimizer="adam", lr=5e-4),
           "rmsprop+clip40": dict(optimizer="rmsprop", lr=6e-4, rmsprop_eps=0.01, max_grad_norm=40.0)}


def step_rows(quick):
    m, t = 1024, 100
    K, R = (5, 2) if quick else (30, 7)
    out = []
    for model in ("mlp_actor_critic", "farmer_lstm"):
        if model == "farmer_lstm":
            slots = po.pack_farmer_slots(*U.farmer_batch(1, m, t))
        else:
            slots = po.pack_vtrace_slots(*U.vtrace_batch(1, m, t))
        Ls = {k: fi.Learner(1, m, t, m, model=model, **kw) for k, kw in CONFIGS.items()}
        batches = {k: L.stage_batch(0, slots) for k, L in Ls.items()}
        for k, L in Ls.items():                       # warm-up: first launches, graph capture
            for _ in range(4):
                L.trainModel(0, batches[k])
            L.sync(0)
        times = {k: [] for k in Ls}
        for _ in range(R):                            # alternated rounds
            for k, L in Ls.items():
                L.sync(0)
                t0 = time.perf_counter()
                for _ in range(K):
                    L.trainModel(0, batches[k])
                L.sync(0)
                times[k].append((time.perf_counter() - t0) / K * 1e3)
        prof = {}
        for k, L in Ls.items():                       # per-kernel device times (stream launches: graphs are off while profiling)
            fi.prof_collect()
            fi.prof_enable(True)
            for _ in range(5):
                L.trainModel(0, batches[k])
            L.sync(0)
            fi.prof_enable(False)
            pr = fi.prof_collect()
            prof[k] = {n: round(v["total_ms"] * 1e3 / v["launches"], 2) for n, v in pr.items()
                       if n in ("grad_norm_clip_kernel", "fused_opt_kernel")}
        med = {k: float(np.median(v)) for k, v in times.items()}
        row = {"model": model, "m": m, "t": t, "steps_per_round": K, "rounds": R,
               "ms_per_step_median": {k: round(v, 4) for k, v in med.items()},
               "ms_per_step_all": {k: [round(x, 4) for x in v] for k, v in times.items()},
               "overhead_pct": round(100.0 * (med["rmsprop+clip40"] / med["adam"] - 1.0), 2),
               "kernel_us_per_launch": prof}
        print(json.dumps(row), file=sys.stderr, flush=True)
        out.append(row)
        for L in Ls.values():
            L.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "optim_sweep measures the GPU: no device"
    res = {"card": card(), "kernels": kernel_rows(a.quick), "steps": step_rows(a.quick), "configs": CONFIGS}
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
