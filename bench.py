#!/usr/bin/env python
"""Learner hot-path benchmark (BASELINE.json metric: learner transitions/s).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's CPU learner
    python bench.py [--gpus N] ... --dump-outputs DIR              # CUDA path: also the last timed step's results as .npy

A "step" is one pass of the learner hot path over one batch of synthetic trajectories: ring
gather -> MLP actor-critic forward -> fused V-trace loss head -> backward -> (gradient
all-reduce) -> fused Adam. Workload (BASELINE.json configs[3] / north_star target): batch 1024
trajectories x T=100 transitions per GPU, 1024-byte records. `value` is timed with the
trajectories already resident in HBM; `e2e` goes through the reference-facing API with host
buffers: SharedBuffer.write (actor threads) -> Learner.trainModel -> loss read-back.
Under torchrun every rank runs the same per-GPU batch (weak scaling) and the gradient arena is
sum-all-reduced with NCCL; rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import datetime
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the source tree: it imports modules the build never
                                 # imported (freeimpala_b200.dp), whose bytecode caches would otherwise land there

METRIC = "learner_transitions_per_s"
UNIT = "transitions/s"
REC_WORDS, Z_DIM, NUM_ACTIONS = 256, 162, 16
W_MU, W_ACTION, W_REWARD, W_DISCOUNT, W_AUX = 162, 178, 179, 180, 181
AC_FWD_FLOPS_PER_TRANSITION = 2.0 * (162 * 512 + 4 * 512 * 512 + 17 * 512)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--batch", type=int, default=1024, help="trajectories per GPU per step (M)")
    ap.add_argument("--seq", type=int, default=100, help="transitions per trajectory (T = entry size S)")
    ap.add_argument("--publish-every", type=int, default=1, help="publish the weights to the model store every N steps (reference: every step)")
    ap.add_argument("--gemm-mode", default="auto", choices=["auto", "simt", "tcgen05", "tcgen05_f16"])
    ap.add_argument("--workload", default="vtrace", choices=["vtrace", "farmer"],
                    help="vtrace: MLP actor-critic V-trace step (headline); farmer: the reference's FarmerLstm/MSE/Adam step")
    ap.add_argument("--writers", type=int, default=0, help="actor threads feeding the ring in the e2e leg (0: min(16, host cores / ranks))")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch trajectories per GPU (default); strong: --batch is the GLOBAL batch, sharded over the ranks")
    ap.add_argument("--no-reference-workload", action="store_true", help="skip the FarmerLstm leg of the default (V-trace) run")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg of a multi-GPU weak-scaling run")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work budget of the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="CUDA path (--impl b200) only: write what the last step of the headline timed pass computed (losses, "
                         "parameters, gradients; rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
    return args


def synth_slots(seed: int, m: int, t: int) -> np.ndarray:
    """Synthetic trajectories in the record layout of DESIGN.md (SURVEY.md 8d config 2): obs and
    behaviour logits ~N(0,1), uniform actions, rewards ~N(0,1), done~Bernoulli(0.01) ->
    discount 0.99(1-done), bootstrap ~N(0,1). Returns uint8 [m, t*1024]."""
    rng = np.random.default_rng(seed)
    w = np.zeros((m, t, REC_WORDS), np.float32)
    w[:, :, :Z_DIM] = rng.standard_normal((m, t, Z_DIM), dtype=np.float32)
    w[:, :, W_MU:W_MU + NUM_ACTIONS] = rng.standard_normal((m, t, NUM_ACTIONS), dtype=np.float32)
    w[:, :, W_ACTION] = rng.integers(0, NUM_ACTIONS, size=(m, t)).astype(np.int32).view(np.float32)
    w[:, :, W_REWARD] = rng.standard_normal((m, t), dtype=np.float32)
    w[:, :, W_DISCOUNT] = (0.99 * (rng.random((m, t)) >= 0.01)).astype(np.float32)
    w[:, t - 1, W_AUX] = rng.standard_normal(m, dtype=np.float32)
    return w.reshape(m, t * REC_WORDS).view(np.uint8)


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    # nvidia-smi block-buffers its output when piped, so lines are dated by nvidia-smi's own `timestamp` field (wall clock,
    # millisecond resolution), not by when they are read; the timed windows are wall-clock (time.time()) intervals
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, devices):
        self.devices, self.proc, self.lines = set(devices), None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self, windows):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.thread.join(timeout=5)   # drain what nvidia-smi had buffered
        sm, mx, pw, reasons = [], [], [], set()
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 10 or not f[1].isdigit() or int(f[1]) not in self.devices:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                continue
            f = f[1:]
            if not any(a <= ts <= b for a, b in windows):
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------
def cpu_baseline_port(seq: int, budget_s: float):
    """The oracle's float64 restatement of the V-trace actor-critic step on the host cores: a bounded sample of
    8-trajectory steps (kind "port"). Reported beside the reference figure; the reference has no V-trace step."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import pyoracle as po
    o = po.Oracle()
    rng = np.random.default_rng(0)
    params = (rng.standard_normal(po.AC_PARAMS) * 0.04).astype(np.float32)
    O = o.actor_critic(params, lr=5e-4)
    m = 8
    slots = synth_slots(99, m, seq)
    dec = o.decode_vtrace(slots, m, seq)
    t0 = time.perf_counter()
    n = 0
    while True:
        O.loss_grad(*dec)
        O.opt_step()
        n += 1
        if time.perf_counter() - t0 >= budget_s or n >= 64:
            break
    dt = time.perf_counter() - t0
    return {"value": n * m * seq / dt, "unit": UNIT, "cores": o.num_threads, "kind": "port",
            "sample": f"{n} V-trace actor-critic steps of {m} x {seq} transitions (float64 C port, OpenMP), {dt:.1f} s"}


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def reference_libtorch(batch: int, seq: int, warmup: int, steps: int):
    """The reference's own learner math: cmd/libtorch_bench train_step (FarmerLstm, MSE, Adam lr 5e-4) compiled from the
    reference's sources into oracle/_ref, on ALL the host cores this process may use (torchrun exports OMP_NUM_THREADS=1
    to its workers: the thread count is set explicitly, VERDICT r1 weak #11)."""
    from oracle import pyoracle as po
    if not os.path.exists(po.REF_NN_SO):
        return None
    r = po.RefNN(seed=1, opt="adam", lr=5e-4, loss="mse")
    r.lib.ref_nn_set_num_threads(host_cores())
    ms = r.bench(batch, seq, warmup, steps)
    return {"ms_per_step": ms, "value": batch * seq / (ms / 1e3), "cores": r.num_threads}


def run_reference_arm(args):
    """--impl reference: the reference's CPU learner step on this box's host cores. The reference has
    no V-trace (SURVEY.md section 0): its learner math is libtorch_bench's FarmerLstm/MSE/Adam
    train_step, timed here at the same batch x seq through oracle/_ref. If oracle/_ref is missing
    the oracle's C port of the V-trace step is timed instead."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ["OMP_NUM_THREADS"] = str(host_cores())   # before libtorch's OpenMP runtime starts
    cfg = {"workload": f"learner step, batch {args.batch} x T={args.seq} (reference arm: libtorch_bench FarmerLstm "
                       f"MSE/Adam train_step on CPU; the reference has no V-trace)",
           "batch_per_gpu": args.batch, "seq_len": args.seq}
    ref = reference_libtorch(args.batch, args.seq, args.warmup, args.steps)
    if ref is not None:
        value, ms, kind, cores = ref["value"], ref["ms_per_step"], "reference", ref["cores"]
        sample = f"{args.steps} train_step calls at batch {args.batch} x seq {args.seq} after {args.warmup} warm-ups"
    else:
        b = cpu_baseline_port(args.seq, max(args.cpu_seconds, 10.0))
        value, kind, cores, sample = b["value"], "port", b["cores"], b["sample"]
        ms = args.batch * args.seq / value * 1e3
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": cfg,
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------
def bind_to_gpu_cpus(torch, local: int):
    """sched_setaffinity to the CPUs NVML reports as local to CUDA device `local` (matched by PCI bus id); None if NVML, the
    device or the cpuset does not allow it."""
    try:
        import pynvml
        pr = torch.cuda.get_device_properties(local)
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByPciBusId(f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0".encode())
        before = os.sched_getaffinity(0)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = os.sched_getaffinity(0)
        if len(after) < min(4, len(before)):   # a binding that leaves no room for the rank's actor threads is worse than none
            os.sched_setaffinity(0, before)
            return None
        return {"cpus": len(after), "of": len(before)}
    except Exception:   # no NVML, no permission, CPUs outside the cpuset: stay where the launcher put us
        return None


class Job:
    """Process-wide state of the b200 arm: rank / world, torch, barriers, reductions over ranks."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            if self.world == 1 and args.gpus > 1:  # convenience: relaunch under torchrun
                cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                       "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29511"), *sys.argv]
                sys.exit(subprocess.call(cmd))
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        # Several ranks on one node: keep this rank's threads (actor threads included: they inherit it) and therefore its
        # pinned ring (first touch) on the CPUs next to its GPU, as a deployment would (numactl / the launcher's binding).
        # FI_BENCH_NUMA=0 leaves the process where the launcher put it.
        self.cpu_binding = None
        self.total_cores = host_cores()   # before any binding: what the node gives the whole job
        if self.world > 1 and os.environ.get("FI_BENCH_NUMA", "1") != "0":
            self.cpu_binding = bind_to_gpu_cpus(torch, self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def all_ranks(self, x: float) -> list:
        if self.world == 1:
            return [x]
        t = self.torch.zeros(self.world, dtype=self.torch.float64, device="cuda")
        t[self.rank] = x
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def measure(job: Job, args, workload: str, M: int, windows: list, *, with_e2e: bool, with_prof: bool,
            with_outputs: bool = False):
    """One workload at M trajectories per GPU: `value` (inputs resident in HBM, EXACTLY K steps between two events on the
    learner's stream, max over ranks), the per-kernel profile of a second, instrumented pass, and `e2e` (host buffers through
    SharedBuffer::write -> readBatch -> trainModel -> loss read-back, wall clock, max over ranks). `with_outputs` keeps
    what the last step of the headline pass computed in res["outputs"]."""
    import freeimpala_b200 as fi
    from freeimpala_b200 import dp
    from freeimpala_b200._lib import FiBatch
    torch = job.torch
    rank, world, local = job.rank, job.world, job.local
    T = args.seq
    slot_bytes = T * 1024
    K, W = args.steps, max(args.warmup, 3)
    cap = 2 * M
    farmer = workload == "farmer"
    ring_cap = 4 * M   # learner's pinned-host/HBM ring: producers may run up to three batches ahead of the learner
    L = fi.Learner(1, ring_cap, T, M, model="farmer_lstm" if farmer else "mlp_actor_critic", device=local,
                   gemm_mode=args.gemm_mode, seed=1, lr=5e-4, publish_every=args.publish_every)
    dp.init_learner_dp(L, rank, world)
    lib = fi.load_library()
    stream_ptr = lib.fi_learner_stream(L._h, 0)
    ext = torch.cuda.ExternalStream(stream_ptr, device=torch.device("cuda", local))

    # two distinct synthetic batches per rank, in pinned host memory and (for `value`) in an HBM ring
    host_ptr = lib.fi_host_alloc(cap * slot_bytes)
    host = np.ctypeslib.as_array((C.c_uint8 * (cap * slot_bytes)).from_address(host_ptr)).reshape(cap, slot_bytes)
    host[:M] = synth_slots(1000 + rank, M, T)   # z / obs ~ N(0,1) in words 0..161 of every record for both workloads;
    host[M:] = synth_slots(2000 + rank, M, T)   # the farmer step also reads x (words 192..255, zeros here) and the target
    ring_dev = torch.empty((cap, slot_bytes), dtype=torch.uint8, device="cuda")
    ring_dev.copy_(torch.from_numpy(host))
    batch_dev = torch.empty((M, slot_bytes), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def device_step(i: int):
        first = (i * M + M // 2) % cap  # every other step wraps around the ring end
        fi.ops.gather(ring_dev.data_ptr(), cap, slot_bytes, first, M, batch_dev.data_ptr(), stream_ptr)
        raw = FiBatch(batch_dev.data_ptr(), M, slot_bytes, stream_ptr, 0)
        L.trainModel(0, fi.Batch(raw))

    # ---------------- value: inputs resident in HBM -------------------------------------------
    for i in range(W):
        device_step(i)
    L.sync(0)
    job.barrier()
    torch.cuda.synchronize()
    per_rank_ms = []   # [pass][rank]: every rank's own device time per step (the headline is the max)

    def timed_pass(profiled: bool):
        L.sync(0)
        job.barrier()
        torch.cuda.synchronize()
        fi.prof_collect()
        fi.prof_enable(profiled)
        n0 = fi.kernel_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        ev0.record(ext)
        for i in range(K):
            device_step(i)
        ev1.record(ext)
        L.sync(0)
        torch.cuda.synchronize()
        job.barrier()
        windows.append((w0, time.time()))
        fi.prof_enable(False)
        per_rank_ms.append(job.all_ranks(ev0.elapsed_time(ev1) / K))
        return max(per_rank_ms[-1]) * K, fi.kernel_launch_count() - n0, fi.prof_collect()

    # Pass 1 is the headline: EXACTLY K steps, two events on the learner's stream, no instrumentation in between.
    # Pass 2 repeats the same K steps with the launches bracketed by CUDA events (fi_prof_enable) for the per-kernel
    # rooflines: consecutive launches of the same kernel share one bracket (an event record between two kernels exposes the
    # launch set-up of the next one, +25-40 us on the cluster GEMMs, which back-to-back launches hide; csrc/fi_common.cuh).
    # The instrumented step is still ~20 % longer than the headline step, which is why the headline does not come from it;
    # kernel shares are quoted against pass 2's own step time.
    ms_total, launches, _ = timed_pass(False)
    res = {"M": M, "ms_per_step": ms_total / K, "value": world * M * T / (ms_total / K / 1e3), "launches": int(launches),
           "per_rank_ms": per_rank_ms[0], "param_count": L.param_count, "ring_cap": ring_cap, "prof": None, "e2e": None}
    if with_outputs:
        # what a caller of the step receives after step W + K: its losses and the updated weights, with the gradients that
        # produced them; read before the instrumented pass moves the weights on
        res["outputs"] = {"losses": L.last_losses(0), "params": L.get_params(0), "grads": L.get_grads(0)}
    if with_prof:
        ms_prof_total, _, prof = timed_pass(True)
        res["prof"], res["ms_per_step_prof"] = prof, ms_prof_total / K
    res["losses"] = [float(x) for x in L.last_losses(0)]

    # ---------------- e2e: host buffers through SharedBuffer.write -> trainModel -> loss read-back ---
    if with_e2e:
        ring = L.getSharedBuffers()[0]
        cores_per_rank = max(1, job.total_cores // world)
        nw_copy = args.writers if args.writers > 0 else max(2, min(14, cores_per_rank - 2))
        nw_zc = int(os.environ.get("FI_BENCH_ZC_THREADS", "2"))  # in-place producers only take the ring lock: two threads keep the ring full
        zc_burst = int(os.environ.get("FI_BENCH_ZC_BURST", "64"))

        def copy_writer(j: int, steps: int, nw: int):
            # actor thread j owns trajectories [j*per, (j+1)*per) of every step: SharedBuffer::write semantics (the ring
            # copies EVERY byte of the caller's trajectory into the pinned slot), handed over in bursts of 32
            per = (M + nw - 1) // nw
            for s in range(steps):
                base = (s % 2) * M
                lo, hi = j * per, min(M, (j + 1) * per)
                for i in range(lo, hi, 32):
                    ring.write_many(host[base + i:base + min(i + 32, hi)])

        def inplace_writer(j: int, steps: int, nw: int):
            # zero-copy producer (fi_ring_reserve_many / fi_ring_commit_many): the trajectory is produced IN the pinned slot
            # (what an MPI_Irecv posted into the slot does); here the slot keeps the synthetic trajectory written during
            # warm-up and the producer stamps the step number into an unused word of the first record of each burst
            burst = zc_burst
            for s in range(steps):
                for i in range(j * burst, M, nw * burst):
                    n = min(burst, M - i)
                    ptrs, ticket = ring.reserve_many(n)
                    C.c_uint32.from_address(ptrs[0] + 4 * 255).value = s
                    ring.commit_many(ticket, n)

        e2e_losses = []
        host_ms = {"readBatch": 0.0, "trainModel": 0.0}

        def e2e_steps(steps: int, writer, nw: int, lead: int = 0):
            """`steps` learner steps fed by `nw` producer threads. Returns the time from the moment the loss of step `lead`
            - 1 has reached the host to the moment the loss of the last step has: the steps [lead, steps) in the steady state
            of the producer -> H2D -> gather -> step pipeline (lead = 0: from the call, thread start-up and pipeline fill
            included)."""
            ts = [threading.Thread(target=writer, args=(j, steps, nw)) for j in range(nw)]
            t_start = time.perf_counter()
            for t in ts:
                t.start()
            base = L.steps_done(0)
            for s in range(steps):
                t0 = time.perf_counter()
                b = ring.readBatch(M, stream_ptr)
                t1 = time.perf_counter()
                L.trainModel(0, b)
                t2 = time.perf_counter()
                host_ms["readBatch"] += (t1 - t0) * 1e3
                host_ms["trainModel"] += (t2 - t1) * 1e3
                # device -> host read of a step's result, every step: the copy of step s is enqueued by trainModel; the host
                # picks up step s-1's losses here (one step behind, as an asynchronous learner's logging is) so that the
                # stream never drains between steps, and the last step's after the loop
                if s > 0:
                    e2e_losses.append(L.losses_at(0, base + s)[0])
                if s == lead and lead > 0:
                    t_start = time.perf_counter()   # the loss of step lead - 1 is on the host
            e2e_losses.append(L.losses_at(0, base + steps)[0])
            t_end = time.perf_counter()
            for t in ts:
                t.join()
            return t_end - t_start

        E2E_LEAD = 3   # untimed steps of the SAME continuous run in front of the K timed ones (producer threads started,
                       # ring filled, the pipeline in its steady state: bench.py's W warm-up steps, for the e2e loop)

        def timed(writer, nw):
            L.sync(0)
            job.barrier()
            torch.cuda.synchronize()
            tw0 = time.time()
            dt = e2e_steps(E2E_LEAD + K, writer, nw, lead=E2E_LEAD)
            L.sync(0)
            torch.cuda.synchronize()
            tw1 = time.time()
            job.barrier()
            windows.append((tw0, tw1))
            return job.max_over_ranks(dt)

        e2e_steps(max(W, 4), copy_writer, nw_copy)   # warm-up; also leaves a valid trajectory in each pinned slot
        host_ms.update(readBatch=0.0, trainModel=0.0)
        copy_s = timed(copy_writer, nw_copy)
        copy_host = {k: v / (E2E_LEAD + K) for k, v in host_ms.items()}   # rank 0's host time per step inside the two calls (blocking included)
        zc_s = timed(inplace_writer, nw_zc)
        res["e2e"] = {
            "value": world * M * T * K / copy_s, "unit": UNIT, "ms_per_step": copy_s / K * 1e3,
            "h2d_bytes_per_step": world * M * slot_bytes, "d2h_bytes_per_step": world * (32 + 4 * L.param_count),
            "actor_threads": nw_copy, "host_cores_per_rank": cores_per_rank,
            "path": f"{nw_copy} actor threads per rank call SharedBuffer::write semantics (fi_ring_write_many: every byte of every "
                    f"trajectory is copied from the actor's buffer into a pinned ring slot) -> cudaMemcpyAsync per run of slots on the "
                    f"side stream -> readBatch (gather kernel) -> Learner.trainModel -> losses D2H every step; weights published D2H "
                    f"every step; the loss of step s is read by the host while step s+1 runs (fi_learner_losses_at). Timed: "
                    f"{K} consecutive steps of one continuous run, from the moment the loss of the step before them has reached the "
                    f"host to the moment the loss of the last one has ({E2E_LEAD} untimed steps of the same run in front: producer "
                    f"threads started, ring filled); every timed step's H2D copy and loss read-back fall inside the region",
            "losses_read": len(e2e_losses), "host_ms_per_step": copy_host,
            "inplace": {"value": world * M * T * K / zc_s, "ms_per_step": zc_s / K * 1e3, "producer_threads": nw_zc,
                        "path": "zero-copy producer API (fi_ring_reserve_many / fi_ring_commit_many): the trajectory already sits in the "
                                "pinned slot (an MPI_Irecv posted into it); the producer only stamps one word per burst, so this leg "
                                "measures the ring + H2D + step without the host memcpy"}}
    L.close()
    lib.fi_host_free(host_ptr)
    return res


def kernel_table(prof, K, ms_per_step_prof, world, peaks, ms_per_step=None):
    """Per-kernel rooflines from the event-bracketed pass.

    The brackets (CUDA events; consecutive launches of one kernel share a bracket, csrc/fi_common.cuh) tile the instrumented
    step, and that step is ~20 % longer than the headline step: every bracket boundary costs GPU time the graph-launched step
    does not pay (the event record drains the stream and flushes the previous kernel's dirty lines out of L2; the next kernel
    starts cold). Against the ncu launch list of the same step (profiles/r2_launches.md) a bracketed average reads +25..35 us
    on every kernel that moves 100 MB or more -- the cluster GEMMs as much as the gather -- and +4 us on a 2 us kernel.
    `avg_us_bracketed` is that raw average. `avg_us` takes the overhead out with the one-parameter model those numbers
    suggest: overhead per launch = min(c, half the bracketed average), c chosen so that the kernels add up to the HEADLINE
    step (both measured with CUDA events on the learner's stream). At the bench shape c comes out at ~16 us and the dominant
    GEMM at ~134 us per launch (ncu: 120 us isolated); on the FarmerLstm step c is ~7 us. `achieved` / `frac` use `avg_us`;
    `frac_bracketed` is the same from the raw average. With more than one rank only rank 0's brackets exist: no correction.
    """
    rows = {n: r for n, r in (prof or {}).items() if r["launches"] > 0 and r["total_ms"] > 0}
    c_us = 0.0
    if world == 1 and ms_per_step and rows:
        target = ms_per_step * 1e3 * K   # us of the headline pass
        def total(c):
            return sum(r["launches"] * (r["total_ms"] * 1e3 / r["launches"] - min(c, 0.5 * r["total_ms"] * 1e3 / r["launches"]))
                       for r in rows.values())
        if total(0.0) > target:
            lo, hi = 0.0, max(r["total_ms"] * 1e3 / r["launches"] for r in rows.values())
            for _ in range(60):
                mid = 0.5 * (lo + hi)
                lo, hi = (mid, hi) if total(mid) > target else (lo, mid)
            c_us = hi
    kernels = {}
    for name, r in rows.items():
        bracketed_us = r["total_ms"] * 1e3 / r["launches"]
        avg_us = bracketed_us - min(c_us, 0.5 * bracketed_us)
        per_launch = r["work"] / r["launches"]
        if r["unit"] == "bytes":
            scale, peak, unit, bound = 1e9, peaks["hbm_gbs"], "GB/s", "hbm"
        else:
            scale, peak, unit, bound = 1e12, peaks["bf16_tflops_sustained"], "TFLOP/s", "tensor"
        ach = per_launch / (avg_us / 1e6) / scale
        kernels[name] = {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                         "frac_bracketed": per_launch / (bracketed_us / 1e6) / scale / peak,
                         "launches_per_step": r["launches"] / K, "avg_us": avg_us, "avg_us_bracketed": bracketed_us,
                         "bracket_overhead_us": min(c_us, 0.5 * bracketed_us),
                         "share_of_step": r["total_ms"] / (ms_per_step_prof * K) if world == 1 else None}
    return kernels


def run_b200_arm(args):
    job = Job(args)
    rank, world = job.rank, job.world
    T, K = args.seq, args.steps
    farmer = args.workload == "farmer"
    strong = args.scaling == "strong"
    if strong and args.batch % world:
        raise SystemExit(f"--scaling strong needs --batch {args.batch} divisible by the {world} ranks")
    M = args.batch // world if strong else args.batch

    sampler = ClockSampler(range(world))   # rank 0 samples every GPU of the job: the slowest one sets the step time
    windows = []
    if rank == 0:
        sampler.start()
    main = measure(job, args, args.workload, M, windows, with_e2e=not args.no_e2e, with_prof=True,
                   with_outputs=bool(args.dump_outputs) and rank == 0)
    # the reference's own learner step (FarmerLstm / MSE / Adam) at the same batch x seq, in the same run: the like-for-like
    # partner of `bench.py --impl reference` (VERDICT r1: the headline V-trace step has no counterpart in the reference)
    ref_wl = None
    if not farmer and not args.no_reference_workload:
        try:
            ref_wl = measure(job, args, "farmer", M, windows, with_e2e=not args.no_e2e, with_prof=False)
        except Exception as e:
            # an auxiliary leg must not cost the headline line. One process only: with several ranks a rank that gave up
            # alone would leave the others in a collective, so there the failure stays fatal
            if world > 1:
                raise
            sys.stderr.write(f"reference_workload leg failed: {e!r}\n")
    # strong scaling (SURVEY.md 8d config 4: batch 1024 GLOBAL, sharded M/N per GPU) beside the weak-scaling headline
    strong_wl = None
    if world > 1 and not strong and not farmer and args.batch % world == 0 and not args.no_strong:
        strong_wl = measure(job, args, args.workload, args.batch // world, windows, with_e2e=False, with_prof=False)
    clocks = sampler.stop(windows) if rank == 0 else None

    ms_per_step, value, launches = main["ms_per_step"], main["value"], main["launches"]
    peaks = measured_peaks()
    kernels = kernel_table(main["prof"], K, main["ms_per_step_prof"], world, peaks, ms_per_step)
    own = [k for k in kernels if not k.startswith("nccl_")]   # the all-reduce entry is skew + transfer, not one of our kernels
    dominant = max(own, key=lambda k: main["prof"][k]["total_ms"]) if own else None
    roofline = None
    if dominant:
        d = kernels[dominant]
        # DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/), if any
        traffic, traffic_src = None, None
        for prof_name in ("r2_gemm_traffic", "r1_gemm_f16x3_traffic"):
            tpath = os.path.join(ROOT, "profiles", prof_name + ".json")
            if traffic is None and os.path.exists(tpath) and not farmer:
                tj = json.load(open(tpath))
                key = next((k for k in tj if k.startswith(dominant.split(">")[0].rsplit(",", 1)[0] if dominant.count(",") > 1 else dominant)), None)
                if key:
                    traffic, traffic_src = tj[key]["dram_bytes_per_launch"], f"profiles/{prof_name}.json ({key})"
        roofline = {"kernel": dominant, "bound": d["bound"], "achieved": d["achieved"], "peak": d["peak"], "unit": d["unit"],
                    "frac": d["frac"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peaks["source"],
                    "avg_launch_us": d["avg_us"], "avg_launch_us_bracketed": d["avg_us_bracketed"], "frac_bracketed": d["frac_bracketed"],
                    "duration": ("CUDA-event brackets over K steps on the learner's stream; `avg_launch_us` = the bracketed average "
                                 "minus the per-bracket overhead that makes the kernels add up to the headline step "
                                 f"({d['bracket_overhead_us']:.1f} us here; bench.py kernel_table, DESIGN.md section 3); "
                                 "`frac_bracketed` uses the raw bracketed average; profiles/r2_launches.md is the ncu launch list"),
                    "note": ("tensor peak = cuBLAS bf16 sustained; `achieved` counts the 2mnk algorithmic flops, and every "
                             "fp32-accurate product costs three tensor-core products (3xFP16: fp16 hi/lo pairs at the bf16 rate, "
                             "ceiling 1/3 of the peak; 3xTF32: 1/6), so tensor-pipe work is 3 x achieved"
                             if d["bound"] == "tensor" else "HBM copy peak")}
        if d["bound"] == "tensor":
            mult = 3.0 if "f16x3" in dominant else 6.0
            roofline["frac_of_fp32_accurate_ceiling"] = d["frac"] * mult

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # the reference's own CPU learner step (libtorch_bench train_step, FarmerLstm/MSE/Adam) at this batch x seq on the box's
        # host cores: a bounded sample (~0.15 s per step on 16 cores); falls back to the oracle's port if oracle/_ref is absent
        try:
            n_ref = max(3, min(20, int(args.cpu_seconds / 0.4)))
            ref = reference_libtorch(args.batch, T, 2, n_ref)
        except Exception as e:  # the reference build is optional on the GPU box
            ref = None
            sys.stderr.write(f"cpu_baseline: reference libtorch step unavailable: {e}\n")
        if ref:
            cpu = {"value": ref["value"], "unit": UNIT, "cores": ref["cores"], "kind": "reference",
                   "ms_per_step": ref["ms_per_step"],
                   "sample": f"{n_ref} libtorch_bench train_step calls (FarmerLstm, MSE, Adam) at batch {args.batch} x seq {T} after 2 warm-ups; "
                             f"the reference has no V-trace step: compare with reference_workload"}
            cpu["vtrace_port"] = cpu_baseline_port(T, min(args.cpu_seconds, 4.0))
        else:
            cpu = cpu_baseline_port(T, args.cpu_seconds)

    if rank == 0:
        def wl_block(w, name):
            return None if w is None else {
                "workload": name, "value": w["value"], "unit": UNIT, "ms_per_step": w["ms_per_step"], "batch_per_gpu": w["M"],
                "gpu_launches": w["launches"], "params": w["param_count"], "e2e": w["e2e"], "losses_last_step": w["losses"]}
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
               "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
               "dtype": "f32", "data": "synthetic",
               "config": {"workload": (f"farmer_lstm MSE/Adam learner step (the reference's train_step), batch {M} x T={T} per GPU"
                                       if farmer else f"vtrace_mlp_actor_critic learner step, batch {M} x T={T} per GPU "
                                                      f"(BASELINE.json configs[3]; records of 1024 B)"),
                          "batch_per_gpu": M, "global_batch": M * world, "ring_capacity_slots": main["ring_cap"], "seq_len": T,
                          "params": main["param_count"], "optimizer": "adam lr 5e-4", "gemm_mode": args.gemm_mode,
                          "parallelism": f"dp{world} (batch sharded, NCCL sum-allreduce of the flat gradient arena)",
                          "l2": "inputs (105 MB) and activations (>1 GB) per step exceed the 126 MB L2; no explicit flush",
                          "flops_per_step": None if farmer else 3.0 * AC_FWD_FLOPS_PER_TRANSITION * M * T},
               "gpu_launches": int(launches), "ms_per_step_instrumented": main["ms_per_step_prof"],
               "ms_per_step_by_rank": main["per_rank_ms"], "clocks": clocks, "cpu_binding": job.cpu_binding, "e2e": main["e2e"], "roofline": roofline, "kernels": kernels,
               "cpu_baseline": cpu, "losses_last_step": main["losses"],
               "reference_workload": wl_block(ref_wl, f"farmer_lstm MSE/Adam learner step (cmd/libtorch_bench train_step), batch {M} x T={T} "
                                                      f"per GPU: the configuration `bench.py --impl reference` times on the CPU"),
               "strong_scaling": wl_block(strong_wl, f"vtrace_mlp_actor_critic learner step, GLOBAL batch {args.batch} x T={T} sharded over "
                                                     f"{world} GPUs (SURVEY.md 8d config 4)")}
        print(json.dumps(out), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, main["outputs"])
    if world > 1:
        job.dist.destroy_process_group()


def dump_outputs(out_dir: str, arrays: dict):
    """DIR/<name>.npy: losses (float64), params and grads (float32, the whole arena: 4.6 MB each for the actor-critic,
    6.1 MB for FarmerLstm). Inputs and initial weights are seeded, so two builds run with the same arguments can be
    compared array by array."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_b200_arm(a)
