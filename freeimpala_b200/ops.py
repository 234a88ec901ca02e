"""Operator layer: stream-ordered launches of the individual sm_100a kernels on DEVICE
pointers (ints, e.g. torch.Tensor.data_ptr()). Used by the kernel-level parity tests and the
roofline sweeps; `stream` is a cudaStream_t handle (torch.cuda.current_stream().cuda_stream)
or None for the legacy default stream."""
from __future__ import annotations

from . import _lib
from ._lib import check


def gather(ring_ptr: int, capacity: int, slot_bytes: int, first: int, m: int, dst_ptr: int, stream=None) -> None:
    check(_lib.load().fi_op_gather(ring_ptr, capacity, slot_bytes, first, m, dst_ptr, stream), "fi_op_gather")


def vtrace(m: int, t: int, log_rho: int, discount: int, reward: int, value: int, bootstrap: int, vs: int,
           pg_adv: int, rho_bar=1.0, c_bar=1.0, pg_rho_bar=1.0, lambda_=1.0, stream=None) -> None:
    check(_lib.load().fi_op_vtrace(m, t, log_rho, discount, reward, value, bootstrap, rho_bar, c_bar, pg_rho_bar,
                                   lambda_, vs, pg_adv, stream), "fi_op_vtrace")


def vtrace_loss_head(batch: int, m: int, t: int, head: int, ldh: int, dhead: int, losses: int, vs: int = None,
                     pg_adv: int = None, rho_bar=1.0, c_bar=1.0, pg_rho_bar=1.0, lambda_=1.0, baseline_cost=0.5,
                     entropy_cost=0.01, stream=None, legal_mask=False, lengths=False, popart=None, sums: int = None) -> None:
    """legal_mask: the softmaxes, entropy and d(head) run over each record's legal-action word (fi_learner.h).
    lengths: each trajectory holds as many steps as word 183 of its record 0 says; the rows past them get zero d(head),
    vs and pg_adv.
    popart: (mu, sigma) runs PopArt normalisation (fi_op_vtrace_loss_head_popart): head column 16 is the normalised value and
    `sums` (device double[3]) receives {sum vs, sum vs^2, valid steps}."""
    if popart is not None:
        if sums is None:
            raise ValueError("vtrace_loss_head: popart needs a sums pointer")
        mu, sigma = popart
        check(_lib.load().fi_op_vtrace_loss_head_popart(batch, m, t, head, ldh, rho_bar, c_bar, pg_rho_bar, lambda_, baseline_cost,
                                                        entropy_cost, int(legal_mask), int(lengths), dhead, vs, pg_adv, losses, mu,
                                                        sigma, sums, stream), "fi_op_vtrace_loss_head_popart")
        return
    if lengths:
        check(_lib.load().fi_op_vtrace_loss_head_opts(batch, m, t, head, ldh, rho_bar, c_bar, pg_rho_bar, lambda_, baseline_cost,
                                                      entropy_cost, int(legal_mask), 1, dhead, vs, pg_adv, losses, stream),
              "fi_op_vtrace_loss_head_opts")
        return
    name = "fi_op_vtrace_loss_head_legal" if legal_mask else "fi_op_vtrace_loss_head"
    check(getattr(_lib.load(), name)(batch, m, t, head, ldh, rho_bar, c_bar, pg_rho_bar, lambda_,
                                     baseline_cost, entropy_cost, dhead, vs, pg_adv, losses, stream), name)


def policy_sample(head: int, ldh: int, rows: int, actions: int, legal: int = None, seed=0, greedy=False, stream=None) -> None:
    """actions[r] (int32) drawn from head row r (columns 0..15 of [rows, ldh]) over legal[r] (uint32 words; None = all 16),
    RNG counter r (fi_op_policy_sample); an empty support gives -1."""
    check(_lib.load().fi_op_policy_sample(head, ldh, rows, legal, seed, int(greedy), actions, stream), "fi_op_policy_sample")


def adam(kind: str, lr: float, step: int, n: int, p: int, g: int, m: int, v: int, grad_scale=1.0, stream=None) -> None:
    check(_lib.load().fi_op_adam(_lib.OPT[kind], lr, step, n, p, g, m, v, grad_scale, stream), "fi_op_adam")


def rmsprop(lr: float, n: int, p: int, g: int, square_avg: int, momentum_buf: int = None, alpha=0.99, eps=1e-8,
            momentum=0.0, coef: int = None, stream=None) -> None:
    """torch.optim.RMSprop (centered=False, weight_decay=0) over n fp32 values; `coef` (device float) multiplies g first."""
    check(_lib.load().fi_op_rmsprop(lr, alpha, eps, momentum, n, p, g, square_avg, momentum_buf, coef, stream), "fi_op_rmsprop")


def grad_norm_clip(n: int, g: int, max_norm: float, norm: int, coef: int, stream=None) -> None:
    """*norm (device double) = ||g||_2, *coef (device float) = min(1, max_norm / (norm + 1e-6))."""
    check(_lib.load().fi_op_grad_norm_clip(n, g, max_norm, norm, coef, stream), "fi_op_grad_norm_clip")


TRANS = {"NT": 0, "NN": 1, "TN": 2}


def gemm_workspace_bytes(trans: str, m: int, n: int, k: int, mode="auto") -> int:
    return _lib.load().fi_op_gemm_workspace_bytes(TRANS[trans], m, n, k, _lib.GEMM[mode])


def gemm(trans: str, m: int, n: int, k: int, a: int, lda: int, b: int, ldb: int, c: int, ldc: int, bias: int = None,
         relu=False, mode="auto", workspace: int = None, workspace_bytes: int = 0, stream=None) -> None:
    check(_lib.load().fi_op_gemm(TRANS[trans], m, n, k, a, lda, b, ldb, c, ldc, bias, int(relu), _lib.GEMM[mode],
                                 workspace, workspace_bytes, stream), "fi_op_gemm")
