"""Learner / ModelManager / Model: the reference's host interfaces
(include/freeimpala/learner.h:100-207, data_structures.h:43-157, 310-481) on top of the C ABI.

`Learner(p, B, S, M, r, c, l, m, T)` keeps the reference's constructor order. `r` (the
simulated training time the reference sleeps for, learner.h:36) is accepted and ignored: the
step is real work on the GPU. One worker thread per player loops readBatch -> step ->
checkpoint exactly like Learner::workerThread (learner.h:72-97); ctypes releases the GIL
during every call, so the p workers and any number of writer threads run concurrently.
"""
from __future__ import annotations

import ctypes as C
import threading

import numpy as np

from . import _lib
from ._lib import FiBatch, FiLearnerConfig, check
from .shared_buffer import Batch, SharedBuffer


class Model:
    """A published (version, bytes) pair (data_structures.h:43-157)."""

    def __init__(self, data: np.ndarray, version: int):
        self._data, self._version = data, version

    def getVersion(self) -> int:
        return self._version

    def getData(self) -> bytes:
        return self._data.tobytes()

    def as_float32(self) -> np.ndarray:
        return self._data.view(np.float32)


class ModelManager:
    def __init__(self, learner: "Learner"):
        self._l = learner
        self._lib = learner._lib

    def getModel(self, player_index: int):  # :433-438
        if not 0 <= player_index < self._l.num_players:
            return None
        buf = np.empty(self._lib.fi_model_bytes(self._l._h), np.uint8)
        ver = C.c_uint64()
        check(self._lib.fi_model_get(self._l._h, player_index, buf.ctypes.data, buf.nbytes, C.byref(ver)), "fi_model_get")
        return Model(buf, ver.value)

    def getLatestVersion(self, player_index: int) -> int:  # :475-480
        if not 0 <= player_index < self._l.num_players:
            return 0
        return self._lib.fi_model_version(self._l._h, player_index)

    def waitForModelUpdate(self, player_index: int, current_version: int, timeout_ms: int) -> bool:  # :454-472
        if not 0 <= player_index < self._l.num_players:
            return False
        return bool(self._lib.fi_model_wait_update(self._l._h, player_index, current_version, timeout_ms))

    def saveModel(self, player_index: int, current_iteration: int = 0, with_optimizer_state: bool = False) -> None:  # :388-423
        if not 0 <= player_index < self._l.num_players:
            return  # the reference logs and returns
        check(self._lib.fi_model_save(self._l._h, player_index, current_iteration, int(with_optimizer_state)), "fi_model_save")

    def saveAllModels(self, current_iteration: int = 0, with_optimizer_state: bool = False) -> None:  # :426-430
        for p in range(self._l.num_players):
            self.saveModel(p, current_iteration, with_optimizer_state)

    def loadModels(self, model_path: str) -> int:  # :337-385
        if not model_path:
            return 0
        return check(self._lib.fi_model_load(self._l._h, model_path.encode()), "fi_model_load")


class Learner:
    def __init__(self, p: int, B: int, S: int, M: int, r: int = 0, c: int = 0, l: str = "", m: str = "",
                 T: int = 0, *, device: int = 0, model: str = "mlp_actor_critic", loss: str | None = None,
                 optimizer: str = "adam", lr: float = 5e-4, seed: int = 0, gemm_mode: str = "auto",
                 publish_every: int = 1, rho_bar: float = 1.0, c_bar: float = 1.0, pg_rho_bar: float = 1.0,
                 lambda_: float = 1.0, baseline_cost: float = 0.5, entropy_cost: float = 0.01,
                 max_grad_norm: float = 0.0, rmsprop_alpha: float = 0.99, rmsprop_eps: float = 1e-8,
                 rmsprop_momentum: float = 0.0, legal_action_mask: bool = False, variable_length: bool = False,
                 history_length: bool = False, popart_beta: float = 0.0):
        self._lib = _lib.load()
        self.num_players, self.buffer_capacity, self.entry_size, self.batch_size = p, B, S, M
        self.train_time_ms, self.checkpoint_frequency = r, c
        self.checkpoint_location, self.starting_model, self.total_iterations = l, m, T
        cfg = FiLearnerConfig()
        self._lib.fi_learner_config_default(C.byref(cfg))
        cfg.device, cfg.num_players, cfg.buffer_capacity, cfg.entry_size, cfg.batch_size = device, p, B, S, M
        cfg.model = _lib.MODEL[model]
        cfg.loss = _lib.LOSS[loss or ("vtrace" if model == "mlp_actor_critic" else "mse")]
        cfg.optimizer, cfg.lr, cfg.seed = _lib.OPT[optimizer], lr, seed
        cfg.rho_bar, cfg.c_bar, cfg.pg_rho_bar, cfg.lambda_ = rho_bar, c_bar, pg_rho_bar, lambda_
        cfg.baseline_cost, cfg.entropy_cost = baseline_cost, entropy_cost
        cfg.gemm_mode, cfg.publish_every = _lib.GEMM[gemm_mode], publish_every
        cfg.max_grad_norm = max_grad_norm   # global-norm gradient clipping; 0 = off
        cfg.rmsprop_alpha, cfg.rmsprop_eps, cfg.rmsprop_momentum = rmsprop_alpha, rmsprop_eps, rmsprop_momentum
        cfg.legal_action_mask = int(legal_action_mask)   # records carry the legal-action word (fi_learner.h)
        cfg.variable_length = int(variable_length)       # record 0 of a trajectory carries its length (fi_learner.h)
        cfg.history_length = int(history_length)         # FarmerLstm: record 0 of a slot carries its history's length
        cfg.popart_beta = popart_beta                     # PopArt value normalisation; 0 = off (fi_learner.h)
        self._ckpt = l.encode() if l else None
        cfg.checkpoint_location = self._ckpt
        self._h = self._lib.fi_learner_create(C.byref(cfg))
        if not self._h:
            raise _lib.FiError(_lib.FI_ERR_CUDA, "fi_learner_create", _lib.last_error())
        self.model_manager = ModelManager(self)
        if m:  # learner.h:129-132
            self.model_manager.loadModels(m)
        self.shared_buffers = [SharedBuffer(S, B, _handle=self._lib.fi_learner_ring(self._h, i), _owner=self)
                               for i in range(p)]
        self.should_stop = threading.Event()
        self.worker_threads: list[threading.Thread] = []
        self.checkpoint_threads: list[threading.Thread] = []
        self._checkpoint_lock = threading.Lock()
        self.iterations_done = [0] * p
        self.errors: list[str] = []

    # ---- reference interface ----------------------------------------------------------------
    def getSharedBuffers(self):  # learner.h:200-202
        return self.shared_buffers

    def getModelManager(self):  # learner.h:205-207
        return self.model_manager

    def start(self) -> None:  # learner.h:158-163
        for p in range(self.num_players):
            t = threading.Thread(target=self._worker_thread, args=(p,), daemon=True)
            self.worker_threads.append(t)
            t.start()

    def stop(self) -> None:  # learner.h:166-197
        if self._h is None:
            return
        self.should_stop.set()
        for b in self.shared_buffers:
            b.setDraining()
        for t in self.worker_threads:
            t.join()
        self.worker_threads.clear()
        for p in range(self.num_players):
            self.sync(p)
        with self._checkpoint_lock:   # in-progress checkpoints finish before the final save (one writer per file)
            for t in self.checkpoint_threads:
                t.join()
            self.checkpoint_threads.clear()
        if self.checkpoint_location:
            self.model_manager.saveAllModels(self.total_iterations)

    def close(self) -> None:
        if self._h is not None:
            self.stop()
            self._lib.fi_learner_destroy(self._h)
            self._h = None
            self.shared_buffers = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- workerThread / trainModel ----------------------------------------------------------------
    def _worker_thread(self, p: int) -> None:  # learner.h:72-97
        it = 0
        stream = self._lib.fi_learner_stream(self._h, p)
        while not self.should_stop.is_set() and it < self.total_iterations:
            try:
                batch = self.shared_buffers[p].readBatch(self.batch_size, stream)
                if batch.empty():
                    if self.should_stop.is_set():
                        break
                    continue
                self.trainModel(p, batch)
            except _lib.FiError as e:  # reference style: log and stop (SURVEY.md 8b); a failed read would fail again at once
                self.errors.append(str(e))
                self.should_stop.set()
                break
            it += 1
            self.iterations_done[p] = it
            if self.checkpoint_frequency > 0 and it % self.checkpoint_frequency == 0 and self.checkpoint_location:
                self._checkpoint_model(p, it)

    def _checkpoint_model(self, p: int, it: int) -> None:  # learner.h:52-69: reap finished checkpoint threads, start one
        with self._checkpoint_lock:
            for t in self.checkpoint_threads:
                t.join()
            self.checkpoint_threads.clear()
            t = threading.Thread(target=self._save_logged, args=(p, it))
            self.checkpoint_threads.append(t)
            t.start()

    def _save_logged(self, p: int, it: int) -> None:
        try:
            self.model_manager.saveModel(p, it)
        except _lib.FiError as e:   # the reference logs a failed save and carries on
            self.errors.append(str(e))

    def trainModel(self, player_index: int, batch: Batch) -> None:  # learner.h:32-49
        check(self._lib.fi_learner_step(self._h, player_index, C.byref(batch.raw)), "fi_learner_step")

    # ---- pieces of the step, for tests / benchmarks -------------------------------------------------
    def stage_batch(self, player_index: int, host: np.ndarray, ptr: int | None = None, num_slots: int | None = None) -> Batch:
        raw = FiBatch()
        if ptr is None:
            host = np.ascontiguousarray(host)
            ptr, num_slots = host.ctypes.data, host.nbytes // (self.entry_size * _lib.ELEMENT_SIZE)
        check(self._lib.fi_learner_stage_batch(self._h, player_index, ptr, num_slots, C.byref(raw)), "fi_learner_stage_batch")
        return Batch(raw)

    def forward_backward(self, player_index: int, batch: Batch) -> None:
        check(self._lib.fi_learner_forward_backward(self._h, player_index, C.byref(batch.raw)), "fi_learner_forward_backward")

    def apply_update(self, player_index: int) -> None:
        check(self._lib.fi_learner_apply_update(self._h, player_index), "fi_learner_apply_update")

    def sync(self, player_index: int) -> None:
        check(self._lib.fi_learner_sync(self._h, player_index), "fi_learner_sync")

    def last_losses(self, player_index: int) -> np.ndarray:
        out = (C.c_double * 4)()
        check(self._lib.fi_learner_last_losses_f64(self._h, player_index, out), "fi_learner_last_losses_f64")
        return np.array(list(out))

    def losses_at(self, player_index: int, step: int) -> np.ndarray:
        """Losses of optimiser step `step` (1-based, one of the last 8): waits only for that step's read-back."""
        out = (C.c_float * 4)()
        check(self._lib.fi_learner_losses_at(self._h, player_index, step, out), "fi_learner_losses_at")
        return np.array(list(out), dtype=np.float64)

    def grad_norm_at(self, player_index: int, step: int) -> float:
        """Pre-clip gradient L2 norm of optimiser step `step` (one of the last 8; needs max_grad_norm > 0)."""
        out = C.c_double()
        check(self._lib.fi_learner_grad_norm_at(self._h, player_index, step, C.byref(out)), "fi_learner_grad_norm_at")
        return out.value

    def set_lr(self, player_index: int, lr: float) -> None:
        """Learning rate of this player's optimiser from its next update on (e.g. a linear decay, one call per step)."""
        check(self._lib.fi_learner_set_lr(self._h, player_index, lr), "fi_learner_set_lr")

    def debug_relu_masks(self, player_index: int, rows: int) -> np.ndarray:
        out = np.empty((5, rows * 512), np.uint8)
        check(self._lib.fi_learner_debug_relu_masks(self._h, player_index, out.ctypes.data, out.size),
              "fi_learner_debug_relu_masks")
        return out

    def popart_stats(self, player_index: int) -> tuple[float, float, float]:
        """PopArt statistics (mu, nu, sigma) after the updates enqueued so far (synchronises the player's stream)."""
        out = (C.c_double * 3)()
        check(self._lib.fi_learner_popart_stats(self._h, player_index, out), "fi_learner_popart_stats")
        return out[0], out[1], out[2]

    def steps_done(self, player_index: int) -> int:
        return self._lib.fi_learner_steps_done(self._h, player_index)

    @property
    def param_count(self) -> int:
        return self._lib.fi_learner_param_count(self._h)

    def tensor_table(self):
        out = []
        for i in range(self._lib.fi_learner_num_tensors(self._h)):
            v = [C.c_size_t() for _ in range(4)]
            check(self._lib.fi_learner_tensor_info(self._h, i, *[C.byref(x) for x in v]), "fi_learner_tensor_info")
            out.append(tuple(x.value for x in v))
        return out

    def _arena(self, fn, player_index):
        out = np.empty(self.param_count, np.float32)
        check(fn(self._h, player_index, out.ctypes.data, out.size), fn.__name__)
        return out

    def get_params(self, player_index: int) -> np.ndarray:
        return self._arena(self._lib.fi_learner_get_params, player_index)

    def get_grads(self, player_index: int) -> np.ndarray:
        return self._arena(self._lib.fi_learner_get_grads, player_index)

    def set_params(self, player_index: int, params: np.ndarray) -> None:
        params = np.ascontiguousarray(params, dtype=np.float32)
        check(self._lib.fi_learner_set_params(self._h, player_index, params.ctypes.data, params.size), "fi_learner_set_params")

    def set_grads(self, player_index: int, grads: np.ndarray) -> None:
        grads = np.ascontiguousarray(grads, dtype=np.float32)
        check(self._lib.fi_learner_set_grads(self._h, player_index, grads.ctypes.data, grads.size), "fi_learner_set_grads")

    def get_opt_state(self, player_index: int):
        m = np.empty(self.param_count, np.float32)
        v = np.empty(self.param_count, np.float32)
        step = C.c_int64()
        check(self._lib.fi_learner_get_opt_state(self._h, player_index, m.ctypes.data, v.ctypes.data, m.size, C.byref(step)),
              "fi_learner_get_opt_state")
        return m, v, step.value

    def infer(self, player_index: int, obs_or_z: np.ndarray, x: np.ndarray | None = None):
        """Batched actor policy inference: (logits [rows,16], values [rows]) for the actor-critic
        model, values [rows] for the farmer model (z [rows,T,162], x [rows,484])."""
        a = np.ascontiguousarray(obs_or_z, dtype=np.float32)
        if x is None:
            rows = a.size // 162
            logits = np.empty((rows, 16), np.float32)
            values = np.empty(rows, np.float32)
            check(self._lib.fi_learner_infer(self._h, player_index, a.ctypes.data, None, rows, 0, logits.ctypes.data,
                                             values.ctypes.data), "fi_learner_infer")
            return logits, values
        xx = np.ascontiguousarray(x, dtype=np.float32)
        rows, t = a.shape[0], a.shape[1]
        values = np.empty(rows, np.float32)
        check(self._lib.fi_learner_infer(self._h, player_index, a.ctypes.data, xx.ctypes.data, rows, t, None,
                                         values.ctypes.data), "fi_learner_infer")
        return values

    def infer_grouped(self, player_index: int, z: np.ndarray, x: np.ndarray, offsets: np.ndarray, lengths: np.ndarray | None = None):
        """FarmerLstm inference of candidate actions grouped by state: z [S,T,162] is each state's history, x [R,484] the
        candidate rows, rows offsets[s] .. offsets[s+1]-1 belonging to state s (offsets [S+1], offsets[0] = 0, R = offsets[S]).
        lengths [S] (fi_learner_infer_grouped_lengths): state s's history is z[s, :lengths[s]], 1 <= lengths[s] <= T, and the
        rest of z[s] is not read; None runs fi_learner_infer_grouped (every history T steps).
        Returns (values [R], best [S]): best[s] is the index within state s's group of its largest value, lowest on ties."""
        zz = np.ascontiguousarray(z, dtype=np.float32)
        xx = np.ascontiguousarray(x, dtype=np.float32)
        off = np.ascontiguousarray(offsets, dtype=np.uint32)
        if zz.ndim != 3 or zz.shape[2] != 162 or xx.ndim != 2 or xx.shape[1] != 484 or off.shape != (zz.shape[0] + 1,):
            raise ValueError(f"infer_grouped: z {zz.shape}, x {xx.shape}, offsets {off.shape}: "
                             "expected z [S,T,162], x [R,484], offsets [S+1]")
        if off[-1] > xx.shape[0]:
            raise ValueError(f"infer_grouped: offsets[-1] = {off[-1]} but x has {xx.shape[0]} rows")
        states, t = zz.shape[0], zz.shape[1]
        values = np.empty(int(off[-1]), np.float32)
        best = np.empty(states, np.int32)
        if lengths is None:
            check(self._lib.fi_learner_infer_grouped(self._h, player_index, zz.ctypes.data, states, t, xx.ctypes.data,
                                                     off.ctypes.data, values.ctypes.data, best.ctypes.data),
                  "fi_learner_infer_grouped")
            return values, best
        ln = np.ascontiguousarray(lengths, dtype=np.uint32)
        if ln.shape != (states,):
            raise ValueError(f"infer_grouped: lengths {ln.shape}, expected [{states}]")
        check(self._lib.fi_learner_infer_grouped_lengths(self._h, player_index, zz.ctypes.data, states, t, ln.ctypes.data,
                                                         xx.ctypes.data, off.ctypes.data, values.ctypes.data, best.ctypes.data),
              "fi_learner_infer_grouped_lengths")
        return values, best

    def infer_sample(self, player_index: int, obs: np.ndarray, legal: np.ndarray | None = None, seed: int = 0,
                     greedy: bool = False):
        """Actor-critic inference with each row's action drawn on the device from the softmax of its logits over its legal
        set (fi_learner_infer_sample: the rule, Philox4x32-10 at counter = row index, key = seed). obs [rows,162], legal
        [rows] uint32 words (bit j = action j legal; None = all 16). Returns (actions [rows] int32, logits [rows,16],
        values [rows])."""
        a = np.ascontiguousarray(obs, dtype=np.float32)
        rows = a.size // 162
        if a.size != rows * 162 or rows == 0:
            raise ValueError(f"infer_sample: obs {a.shape}: expected [rows,162]")
        lg = None
        if legal is not None:
            lg = np.ascontiguousarray(legal, dtype=np.uint32)
            if lg.shape != (rows,):
                raise ValueError(f"infer_sample: legal {lg.shape}: expected [{rows}]")
        actions = np.empty(rows, np.int32)
        logits = np.empty((rows, 16), np.float32)
        values = np.empty(rows, np.float32)
        check(self._lib.fi_learner_infer_sample(self._h, player_index, a.ctypes.data, None if lg is None else lg.ctypes.data,
                                                rows, seed, int(greedy), actions.ctypes.data, logits.ctypes.data,
                                                values.ctypes.data), "fi_learner_infer_sample")
        return actions, logits, values

    # ---- data parallelism (SURVEY.md 8e) ------------------------------------------------------------
    def infer_stats(self, player_index: int) -> dict:
        """Counters of the combining inference path: calls made, forwards run, rows served."""
        c, b, r = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(self._lib.fi_learner_infer_stats(self._h, player_index, C.byref(c), C.byref(b), C.byref(r)), "fi_learner_infer_stats")
        return {"calls": c.value, "batches": b.value, "rows": r.value}

    def dp_init(self, ids: bytes, rank: int, world_size: int) -> None:
        assert len(ids) == self.num_players * _lib.DP_ID_BYTES
        buf = C.create_string_buffer(ids, len(ids))
        check(self._lib.fi_learner_dp_init(self._h, buf, rank, world_size), "fi_learner_dp_init")

    @staticmethod
    def dp_create_ids(num_players: int) -> bytes:
        lib = _lib.load()
        out = b""
        for _ in range(num_players):
            buf = C.create_string_buffer(_lib.DP_ID_BYTES)
            check(lib.fi_dp_create_id(buf), "fi_dp_create_id")
            out += buf.raw
        return out
