"""numpy restatements of AdamW, RAdam and Adamax (core/optimizer.py), in the RefOptimizer style of
ref_numpy.py and in the kernel's order of operations (csrc/fused.cu, AdamRule), so that float64
agreement with the device is at the level of machine precision.  tests/test_optimizers_host.py pins
them against torch.optim."""
import math

import numpy as np

from ref_numpy import RefAdam, RefOptimizer


class RefAdamW(RefAdam):
    """p = p * (1 - lr*wd) + Adam's step.  `apply(p, g)` is the fused arena update; `_step(g, p)`
    is the compute_step form, Adam's step minus (lr*wd) * p"""

    def __init__(self, lr=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8, weight_decay=0.01):
        RefAdam.__init__(self, lr, beta1, beta2, epsilon)
        self.wd = weight_decay

    def apply(self, p, g):
        step = RefAdam._step(self, g)
        return p * (1.0 - self.lr * self.wd) + step

    def _step(self, g, p=None):
        step = RefAdam._step(self, g)
        return step - (self.lr * self.wd) * (self._flat_p if p is None else p)

    def compute_steps(self, params):
        self._flat_p = np.concatenate([np.ravel(p.values) for p in params])
        return RefOptimizer.compute_steps(self, params)


class RefRAdam(RefOptimizer):
    def __init__(self, lr=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8):
        self.lr, self.b1, self.b2, self.eps = lr, beta1, beta2, epsilon
        self.t, self.m, self.v = 0, 0, 0

    def rect(self, t):
        """r_t: the rectification term while rho_t > 5, else 0"""
        bc2 = 1.0 - self.b2 ** t
        rho_inf = 2.0 / (1.0 - self.b2) - 1.0
        rho_t = rho_inf - 2.0 * t * self.b2 ** t / bc2
        if rho_t <= 5.0:
            return 0.0
        return math.sqrt((rho_t - 4.0) * (rho_t - 2.0) * rho_inf / ((rho_inf - 4.0) * (rho_inf - 2.0) * rho_t))

    def _step(self, g):
        self.t += 1
        self.m += (1.0 - self.b1) * (g - self.m)
        self.v += (1.0 - self.b2) * (g * g - self.v)
        mh = self.m / (1.0 - self.b1 ** self.t)
        r = self.rect(self.t)
        if r > 0.0:
            return -self.lr * r * mh * math.sqrt(1.0 - self.b2 ** self.t) / (np.sqrt(self.v) + self.eps)
        return -self.lr * mh


class RefAdamax(RefOptimizer):
    def __init__(self, lr=0.002, beta1=0.9, beta2=0.999, epsilon=1e-8):
        self.lr, self.b1, self.b2, self.eps = lr, beta1, beta2, epsilon
        self.t, self.m, self.u = 0, 0, 0

    def _step(self, g):
        self.t += 1
        self.m += (1.0 - self.b1) * (g - self.m)
        # np.maximum propagates NaN, as the kernel's max does
        self.u = np.maximum(self.b2 * self.u, np.abs(g) + self.eps)
        return -(self.lr / (1.0 - self.b1 ** self.t)) * self.m / self.u
