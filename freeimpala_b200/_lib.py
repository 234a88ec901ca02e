"""ctypes binding of the C ABI in include/fi_learner.h (the drop-in boundary).

The library is the product: if it is missing this module raises (there is no CPU or PyTorch
fallback anywhere in the package). Build it with `python -m freeimpala_b200.build`.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

c_void_p, c_int, c_size_t, c_u64, c_i64, c_float, c_double, c_char_p = (
    C.c_void_p, C.c_int, C.c_size_t, C.c_uint64, C.c_int64, C.c_float, C.c_double, C.c_char_p)

FI_OK, FI_ERR_CUDA, FI_ERR_ARG, FI_ERR_STATE, FI_ERR_IO, FI_ERR_NCCL = 0, -1, -2, -3, -4, -5
ELEMENT_SIZE = 1024
DP_ID_BYTES = 128
MODEL = {"farmer_lstm": 0, "mlp_actor_critic": 1}
LOSS = {"mse": 0, "mae": 1, "huber": 2, "vtrace": 3}
OPT = {"adam": 0, "sgd": 1, "adamw": 2, "rmsprop": 3}
GEMM = {"auto": 0, "simt": 1, "tcgen05": 2, "tcgen05_f16": 3}


class FiBatch(C.Structure):
    _fields_ = [("dev_ptr", c_void_p), ("num_slots", c_size_t), ("slot_bytes", c_size_t),
                ("stream", c_void_p), ("seq", c_u64)]


class FiLearnerConfig(C.Structure):
    _fields_ = [("device", c_int), ("num_players", c_int), ("buffer_capacity", c_size_t),
                ("entry_size", c_size_t), ("batch_size", c_size_t), ("model", c_int), ("loss", c_int),
                ("optimizer", c_int), ("lr", c_double), ("seed", c_u64),
                ("rho_bar", c_float), ("c_bar", c_float), ("pg_rho_bar", c_float), ("lambda_", c_float),
                ("baseline_cost", c_float), ("entropy_cost", c_float),
                ("gemm_mode", c_int), ("publish_every", c_int), ("checkpoint_location", c_char_p),
                ("max_grad_norm", c_double), ("rmsprop_alpha", c_double), ("rmsprop_eps", c_double),
                ("rmsprop_momentum", c_double), ("legal_action_mask", c_int)]


class FiProfEntry(C.Structure):
    _fields_ = [("name", C.c_char * 48), ("launches", c_u64), ("total_ms", c_double), ("work", c_double),
                ("unit", c_int)]


_P = c_void_p
# name -> (restype, argtypes); every FI_API symbol of include/fi_learner.h
SIGNATURES = {
    "fi_last_error": (c_char_p, []),
    "fi_version": (c_char_p, []),
    "fi_kernel_launch_count": (c_u64, []),
    "fi_prof_enable": (None, [c_int]),
    "fi_prof_collect": (c_int, [C.POINTER(FiProfEntry), c_int]),
    "fi_debug_tc_trace": (c_int, [_P, c_size_t]),
    "fi_debug_set_lstm_tc": (None, [c_int]),
    "fi_ring_create": (_P, [c_int, c_size_t, c_size_t]),
    "fi_ring_destroy": (None, [_P]),
    "fi_ring_write": (c_int, [_P, _P, c_size_t]),
    "fi_ring_try_write": (c_int, [_P, _P, c_size_t]),
    "fi_ring_write_many": (c_size_t, [_P, _P, c_size_t, c_size_t, c_size_t]),
    "fi_ring_reserve": (_P, [_P, C.POINTER(c_u64)]),
    "fi_ring_commit": (c_int, [_P, c_u64, c_size_t]),
    "fi_ring_reserve_many": (c_size_t, [_P, c_size_t, _P, C.POINTER(c_u64)]),
    "fi_ring_commit_many": (c_int, [_P, c_u64, c_size_t, c_size_t]),
    "fi_ring_read_batch": (c_int, [_P, c_size_t, _P, C.POINTER(FiBatch)]),
    "fi_ring_set_draining": (None, [_P]),
    "fi_ring_filled_count": (c_size_t, [_P]),
    "fi_ring_slot_bytes": (c_size_t, [_P]),
    "fi_ring_capacity": (c_size_t, [_P]),
    "fi_batch_to_host": (c_int, [C.POINTER(FiBatch), _P, c_size_t]),
    "fi_learner_config_default": (None, [C.POINTER(FiLearnerConfig)]),
    "fi_learner_create": (_P, [C.POINTER(FiLearnerConfig)]),
    "fi_learner_destroy": (None, [_P]),
    "fi_learner_ring": (_P, [_P, c_int]),
    "fi_learner_stream": (_P, [_P, c_int]),
    "fi_learner_step": (c_int, [_P, c_int, C.POINTER(FiBatch)]),
    "fi_learner_forward_backward": (c_int, [_P, c_int, C.POINTER(FiBatch)]),
    "fi_learner_apply_update": (c_int, [_P, c_int]),
    "fi_learner_stage_batch": (c_int, [_P, c_int, _P, c_size_t, C.POINTER(FiBatch)]),
    "fi_learner_last_losses": (c_int, [_P, c_int, C.POINTER(c_float)]),
    "fi_learner_last_losses_f64": (c_int, [_P, c_int, C.POINTER(c_double)]),
    "fi_learner_losses_at": (c_int, [_P, c_int, c_u64, C.POINTER(c_float)]),
    "fi_learner_grad_norm_at": (c_int, [_P, c_int, c_u64, C.POINTER(c_double)]),
    "fi_learner_set_lr": (c_int, [_P, c_int, c_double]),
    "fi_learner_sync": (c_int, [_P, c_int]),
    "fi_learner_steps_done": (c_u64, [_P, c_int]),
    "fi_learner_debug_relu_masks": (c_int, [_P, c_int, _P, c_size_t]),
    "fi_learner_param_count": (c_size_t, [_P]),
    "fi_learner_num_tensors": (c_int, [_P]),
    "fi_learner_tensor_info": (c_int, [_P, c_int] + [C.POINTER(c_size_t)] * 4),
    "fi_learner_set_params": (c_int, [_P, c_int, _P, c_size_t]),
    "fi_learner_get_params": (c_int, [_P, c_int, _P, c_size_t]),
    "fi_learner_get_grads": (c_int, [_P, c_int, _P, c_size_t]),
    "fi_learner_set_grads": (c_int, [_P, c_int, _P, c_size_t]),
    "fi_learner_get_opt_state": (c_int, [_P, c_int, _P, _P, c_size_t, C.POINTER(c_i64)]),
    "fi_learner_grad_ptr": (_P, [_P, c_int]),
    "fi_learner_param_ptr": (_P, [_P, c_int]),
    "fi_learner_infer": (c_int, [_P, c_int, _P, _P, c_size_t, c_size_t, _P, _P]),
    "fi_learner_infer_stats": (c_int, [_P, c_int, C.POINTER(c_u64), C.POINTER(c_u64), C.POINTER(c_u64)]),
    "fi_learner_infer_grouped": (c_int, [_P, c_int, _P, c_size_t, c_size_t, _P, _P, _P, _P]),
    "fi_model_bytes": (c_size_t, [_P]),
    "fi_model_version": (c_u64, [_P, c_int]),
    "fi_model_get": (c_int, [_P, c_int, _P, c_size_t, C.POINTER(c_u64)]),
    "fi_model_wait_update": (c_int, [_P, c_int, c_u64, c_int]),
    "fi_model_save": (c_int, [_P, c_int, c_u64, c_int]),
    "fi_model_load": (c_int, [_P, c_char_p]),
    "fi_dp_create_id": (c_int, [_P]),
    "fi_learner_dp_init": (c_int, [_P, _P, c_int, c_int]),
    "fi_learner_dp_world": (c_int, [_P]),
    "fi_host_alloc": (_P, [c_size_t]),
    "fi_host_free": (None, [_P]),
    "fi_op_gather": (c_int, [_P, c_size_t, c_size_t, c_size_t, c_size_t, _P, _P]),
    "fi_op_vtrace": (c_int, [c_int, c_int] + [_P] * 5 + [c_float] * 4 + [_P, _P, _P]),
    "fi_op_vtrace_loss_head": (c_int, [_P, c_int, c_int, _P, c_int] + [c_float] * 6 + [_P] * 5),
    "fi_op_vtrace_loss_head_legal": (c_int, [_P, c_int, c_int, _P, c_int] + [c_float] * 6 + [_P] * 5),
    "fi_op_adam": (c_int, [c_int, c_double, c_i64, c_size_t, _P, _P, _P, _P, c_float, _P]),
    "fi_op_grad_norm_clip": (c_int, [c_size_t, _P, c_double, _P, _P, _P]),
    "fi_op_rmsprop": (c_int, [c_double] * 4 + [c_size_t] + [_P] * 6),
    "fi_op_gemm_workspace_bytes": (c_size_t, [c_int] * 5),
    "fi_op_gemm": (c_int, [c_int] * 4 + [_P, c_int, _P, c_int, _P, c_int, _P, c_int, c_int, _P, c_size_t, _P]),
}


class FiError(RuntimeError):
    def __init__(self, code: int, where: str, msg: str):
        super().__init__(f"{where}: fi_status {code}: {msg}")
        self.code = code


def library_path() -> str:
    return os.environ.get("FI_LIBRARY", _build.LIB)


_lib = None


def load() -> C.CDLL:
    """dlopen the CUDA library and declare every signature. Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(f"{path} not found: the CUDA library is the product and there is no fallback; "
                          f"run `python -m freeimpala_b200.build`")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return (load().fi_last_error() or b"").decode(errors="replace")


def check(code: int, where: str) -> int:
    if code < 0:
        raise FiError(code, where, last_error())
    return code
