"""TEST INFRASTRUCTURE ONLY: references for RMSProp, global-norm gradient clipping and learning-rate changes.

  * float64: torch.optim.RMSprop (centered=False, weight_decay=0) and torch.nn.utils.clip_grad_norm_ on one flat array;
  * float32: the CUDA kernel's RMSProp (freeimpala_b200/csrc/adam.cu rmsprop_elem) restated operation for operation, each
    numpy float32 operation rounding once, so the kernel can be held to it bit for bit;
  * OptOracle: a model oracle of oracle/pyoracle.py (which only knows Adam / AdamW / SGD at a fixed learning rate) driven
    with any of the four optimisers, a learning rate that may change between steps and optional clipping.

Adam / AdamW / SGD updates are the oracle's own float64 orc_opt_update; only clipping and RMSProp are computed here.
"""
from __future__ import annotations

import numpy as np

OPTS = ("adam", "sgd", "adamw", "rmsprop")


def clip_coef(g, max_norm: float):
    """(coefficient, norm) of clip_grad_norm_: norm = ||g||_2 in float64, coefficient = min(1, max_norm / (norm + 1e-6))."""
    g = np.asarray(g, np.float64)
    norm = float(np.sqrt(np.dot(g, g)))
    return min(1.0, max_norm / (norm + 1e-6)), norm


def rmsprop_f64(lr, alpha, eps, momentum, p, g, sa, buf=None):
    """One torch.optim.RMSprop step in float64, in place on p, sa (and buf when momentum > 0)."""
    sa *= alpha
    sa += (1.0 - alpha) * g * g
    avg = np.sqrt(sa) + eps
    if momentum > 0:
        buf *= momentum
        buf += g / avg
        p -= lr * buf
    else:
        p -= lr * (g / avg)


def rmsprop_f32(lr, alpha, eps, momentum, p, g, sa, buf=None, gscale=1.0):
    """The kernel's RMSProp in float32, in place: g = g*gscale; sa = alpha*sa + ((1-alpha)*g)*g; avg = sqrt(sa) + eps;
    momentum: buf = mu*buf + g/avg, p = p - lr*buf; otherwise p = p - lr*(g/avg)."""
    f = np.float32
    g = np.asarray(g, f) * f(gscale)
    sa[...] = f(alpha) * sa + (f(1.0 - alpha) * g) * g
    q = g / (np.sqrt(sa) + f(eps))
    if momentum > 0:
        buf[...] = f(momentum) * buf + q
        p[...] = p - f(lr) * buf
    else:
        p[...] = p - f(lr) * q


class OptOracle:
    """Wraps a model oracle (pyoracle OracleAC / OracleFarmer) so that its optimiser step is `opt` with the options set by
    set_opt: the gradient stays as loss_grad / set_grads left it (clipping works on a copy), the new parameters are computed
    here in float64 and written into the model oracle through its SGD step with lr = 1 (p - (p - p_new) is p_new)."""

    def __init__(self, oracle, model, opt="adam", lr=5e-4, max_grad_norm=0.0, rmsprop_alpha=0.99, rmsprop_eps=1e-8,
                 rmsprop_momentum=0.0):
        assert opt in OPTS, opt
        self.o, self.m, self.opt = oracle, model, opt
        self.set_opt(lr, max_grad_norm, rmsprop_alpha, rmsprop_eps, rmsprop_momentum)
        n = model.params().size
        self.m1, self.v = np.zeros(n), np.zeros(n)   # Adam: the two moments; RMSProp: momentum buffer, square average
        self.step = 0
        self.last_norm = None

    @classmethod
    def actor_critic(cls, oracle, params, opt="adam", lr=5e-4, **kw):
        return cls(oracle, oracle.actor_critic(params, opt="sgd", lr=1.0), opt, lr, **kw)

    @classmethod
    def farmer(cls, oracle, params, opt="adam", lr=5e-4, loss="mse", **kw):
        return cls(oracle, oracle.farmer(params, opt="sgd", lr=1.0, loss=loss), opt, lr, **kw)

    def set_opt(self, lr, max_grad_norm=0.0, rmsprop_alpha=0.99, rmsprop_eps=1e-8, rmsprop_momentum=0.0):
        """Options of the next opt_step: learning rate, clipping bound (0 = off) and the RMSProp constants."""
        self.lr, self.max_grad_norm = lr, max_grad_norm
        self.alpha, self.eps, self.momentum = rmsprop_alpha, rmsprop_eps, rmsprop_momentum

    def opt_step(self):
        self.step += 1
        g = self.m.grads()
        p = self.m.params()
        ge = g
        self.last_norm = None
        if self.max_grad_norm > 0:
            coef, self.last_norm = clip_coef(g, self.max_grad_norm)
            ge = g * coef
        new = p.copy()
        if self.opt == "rmsprop":
            rmsprop_f64(self.lr, self.alpha, self.eps, self.momentum, new, ge, self.v, self.m1)
        else:
            self.o.opt_update(self.opt, self.lr, self.step, new, np.ascontiguousarray(ge), self.m1, self.v)
        self.m.set_grads(p - new)
        self.m.opt_step()
        self.m.set_grads(g)

    def opt_state(self):
        return self.m1.copy(), self.v.copy()

    # the model oracle's own interface
    def loss_grad(self, *a, **kw):
        return self.m.loss_grad(*a, **kw)

    def loss_grad_masked(self, *a, **kw):
        return self.m.loss_grad_masked(*a, **kw)

    def params(self):
        return self.m.params()

    def grads(self):
        return self.m.grads()

    def set_grads(self, g):
        self.m.set_grads(g)
