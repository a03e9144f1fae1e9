"""Optimisers (interface of the reference's core/optimizer.py) running on flat device buffers.

compute_step(grads, params) keeps the reference contract: gradients are flattened in layer
order, `w` before `b` (optimizer.py:14-15), one `_compute_step` runs over the flat vector, and
the result is handed back per parameter.  Here the flat vector is a device buffer and
`_compute_step` is one fused kernel (tnn_opt_step).  When core.model.Model keeps parameters and
gradients in flat arenas, apply_fused() updates the parameters in place with that same kernel:
read g, state, p and write state, p in one pass (28 B/param for Adam).

weight_decay: the reference accepts it and never applies it (the line that would,
`_step -= self.weight_decay * v`, is commented out at optimizer.py:28-29).  Same here by default;
setting `optimizer.apply_weight_decay = True` turns exactly that line on (fused path: inside the
optimiser kernel, hyper-parameter slot 7; compute_step path: on the per-parameter step views).
AdamW is the exception: its decoupled decay is always on and `apply_weight_decay` has no effect on it.

`optimizer.lr` is read whenever a step's coefficients are formed, so core/lr_scheduler.py can change
it between steps, recorded steps included.

The fused arena path is only taken for the built-in update rules: an optimiser whose class
overrides `_compute_step` or `compute_step` (the reference's extension point) always goes
through compute_step(), see core.model.Model.step.
"""
import math

import numpy as np

import core._backend as be


def _as_darray(g):
    if isinstance(g, be.DArray):
        return g
    if hasattr(g, "_data"):
        return g._data
    return be.from_numpy(np.asarray(g))


class BaseOptimizer(object):

    opt_code = None
    n_state = 0

    apply_weight_decay = False   # opt-in: the reference has the decay line commented out

    def __init__(self, lr, weight_decay):
        self.lr = lr
        self.weight_decay = weight_decay
        self._state = None  # list of flat device vectors, allocated at the first step
        self._hyper_dev = None  # device copy of the hyper-parameters while a captured step uses them

    # ---- reference interface ------------------------------------------------------------
    def compute_step(self, grads, params):
        flat_list = [_as_darray(v) for grad in grads for v in grad.values()]
        if not flat_list:
            return [dict() for _ in params]
        dt = be.F64 if any(g.dtype == be.F64 for g in flat_list) else be.F32
        total = sum(g.size for g in flat_list)
        flat = be.empty((total,), dt)
        p = 0
        for g in flat_list:
            if g.size:
                be.copy_into(flat.view((g.size,), p), be.astype(g, dt).view((g.size,)))
            p += g.size
        # a user-defined _compute_step may hand back a numpy array (the reference's contract)
        flat_step = _as_darray(self._compute_step(flat))
        if flat_step.dtype != dt:
            flat_step = be.astype(flat_step, dt)
        if flat_step.size != total:
            raise ValueError("_compute_step returned %d elements for %d gradients" % (flat_step.size, total))
        flat_step = flat_step.view((total,))
        wd = self._step_decay()

        p = 0
        steps = []
        for param in params:
            layer = dict()
            for k, v in param.items():
                block = int(np.prod(v.shape))
                step = flat_step.view(tuple(v.shape), p)
                if wd:      # optimizer.py:28-29, opt-in
                    vd = be.astype(_as_darray(v), dt)
                    step = be.ew(be.SUB, step, be.ew(be.MUL, be.full((), wd, dt), vd))
                layer[k] = step
                p += block
            steps.append(layer)
        return steps

    def uses_builtin_rule(self):
        """True when the update is one of this module's fused kernels and nobody overrode the
        reference's extension points (_compute_step / compute_step) in a subclass"""
        cls = type(self)
        return (self.opt_code is not None
                and cls._compute_step is BaseOptimizer._compute_step
                and cls.compute_step is BaseOptimizer.compute_step)

    def _decay_coefficient(self):
        return float(self.weight_decay) if (self.apply_weight_decay and self.weight_decay) else 0.0

    def _step_decay(self):
        """c of `step -= c * v`, which compute_step applies to each parameter's step"""
        return self._decay_coefficient()

    def _hyper8(self):
        """this step's kernel coefficients: the rule's own in slots 0-6, weight decay in slot 7"""
        vals = list(self._hyper())
        vals += [0.0] * (8 - len(vals))
        vals[7] = self._decay_coefficient()
        return vals

    def _compute_step(self, grad):
        """flat device gradient -> flat device step (optimizer.py:37-38)"""
        grad = _as_darray(grad)
        step = be.empty(grad.shape, grad.dtype)
        self._run(None, step, grad)
        return step

    # ---- fused path -----------------------------------------------------------------------
    def apply_fused(self, param_flat, grad_flat):
        """param_flat += step(grad_flat), in place, one kernel"""
        self._run(param_flat, None, grad_flat)

    def step_hyper(self):
        """this step's hyper-parameters (Adam: advances t); a captured step reads them from device"""
        return self._hyper_dev if self._hyper_dev is not None else self._hyper8()

    def apply_fused_range(self, param_flat, grad_flat, lo, hi, hyper):
        """the fused update on elements [lo, hi) of the flat arenas, with hyper from step_hyper()"""
        self._ensure_state(grad_flat)
        n = hi - lo
        s = [st.view((n,), lo) for st in self._state] + [None, None]
        be.opt_step(self.opt_code, param_flat.view((n,), lo), None, grad_flat.view((n,), lo),
                    s[0], s[1], hyper)

    def _ensure_state(self, grad):
        if self.opt_code is None:
            raise NotImplementedError
        if self._state is None:
            self._state = [be.zeros(grad.shape, grad.dtype) for _ in range(self.n_state)]
        elif self._state and (self._state[0].size != grad.size or self._state[0].dtype != grad.dtype):
            raise ValueError("optimizer state was built for %d parameters of %s, got %d of %s"
                             % (self._state[0].size, self._state[0].dtype, grad.size, grad.dtype))

    def _run(self, param, step_out, grad):
        if self.opt_code is None:
            raise NotImplementedError
        if self._state is None:
            self._state = [be.zeros(grad.shape, grad.dtype) for _ in range(self.n_state)]
        elif self._state and (self._state[0].size != grad.size or self._state[0].dtype != grad.dtype):
            raise ValueError("optimizer state was built for %d parameters of %s, got %d of %s"
                             % (self._state[0].size, self._state[0].dtype, grad.size, grad.dtype))
        s = self._state + [None, None]
        hyper = self._hyper_dev if self._hyper_dev is not None else self._hyper8()
        be.opt_step(self.opt_code, param, step_out, grad, s[0], s[1], hyper)

    def upload_hyper(self, dst):
        """advance to the next step (Adam: t += 1) and put its coefficients into the 8-double device
        vector a captured step reads them from"""
        be.upload_into(dst, np.asarray(self._hyper8(), dtype=np.float64))

    def _hyper(self):
        raise NotImplementedError


class SGD(BaseOptimizer):
    """step = -lr * g (optimizer.py:41-47)"""
    opt_code = be.OPT_SGD

    def __init__(self, lr, weight_decay=0.0):
        super().__init__(lr, weight_decay)

    def _hyper(self):
        return [self.lr]


class Adam(BaseOptimizer):
    """optimizer.py:50-79: m += (1-b1)(g-m); v += (1-b2)(g*g-v);
    step = -lr * (m/(1-b1^t)) / (sqrt(v/(1-b2^t)) + eps)"""
    opt_code = be.OPT_ADAM
    n_state = 2

    def __init__(self, lr=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8, weight_decay=0.0):
        super().__init__(lr, weight_decay)
        self._b1 = beta1
        self._b2 = beta2
        self._eps = epsilon
        self._t = 0

    def _hyper(self):
        self._t += 1
        return [self.lr, self._b1, self._b2, self._eps,
                1.0 - self._b1 ** self._t, 1.0 - self._b2 ** self._t]


class RMSProp(BaseOptimizer):
    """optimizer.py:82-112: ms += (1-decay)(g*g-ms); mom = momentum*mom + lr*g/sqrt(ms+eps);
    step = -mom"""
    opt_code = be.OPT_RMSPROP
    n_state = 2

    def __init__(self, lr=0.01, decay=0.99, momentum=0.0, epsilon=1e-8, weight_decay=0.0):
        super().__init__(lr, weight_decay)
        self._decay = decay
        self._momentum = momentum
        self._eps = epsilon

    def _hyper(self):
        return [self.lr, self._decay, self._momentum, self._eps]


class Momentum(BaseOptimizer):
    """optimizer.py:115-128: acc = momentum*acc + g; step = -lr*acc"""
    opt_code = be.OPT_MOMENTUM
    n_state = 1

    def __init__(self, lr, momentum=0.9, weight_decay=0.0):
        super().__init__(lr, weight_decay)
        self._momentum = momentum

    def _hyper(self):
        return [self.lr, self._momentum]


class Adagrad(BaseOptimizer):
    """optimizer.py:131-146: G += g*g; step = -(lr / sqrt(G + eps)) * g"""
    opt_code = be.OPT_ADAGRAD
    n_state = 1

    def __init__(self, lr, weight_decay=0.0, epsilon=1e-8):
        super().__init__(lr, weight_decay)
        self._eps = epsilon

    def _hyper(self):
        return [self.lr, self._eps]


class Adadelta(BaseOptimizer):
    """optimizer.py:149-164"""
    opt_code = be.OPT_ADADELTA
    n_state = 2

    def __init__(self, lr=1.0, weight_decay=0.0, decay=0.9, epsilon=1e-8):
        super().__init__(lr, weight_decay)
        self._eps = epsilon
        self._decay = decay

    def _hyper(self):
        return [self.lr, self._decay, self._eps]


def _check_adam_args(lr, beta1, beta2, epsilon):
    for name, v in (("lr", lr), ("epsilon", epsilon)):
        if not (math.isfinite(v) and v >= 0.0):
            raise ValueError("%s must be finite and non-negative, got %r" % (name, v))
    for name, v in (("beta1", beta1), ("beta2", beta2)):
        if not 0.0 <= v < 1.0:
            raise ValueError("%s must lie in [0, 1), got %r" % (name, v))


class AdamW(Adam):
    """Adam with decoupled weight decay (torch.optim.AdamW): p = p * (1 - lr*wd) + Adam's step.

    The decay is always on; `apply_weight_decay` has no effect on this rule.  On the fused path the
    kernel scales the parameter; on the compute_step path `(lr*wd) * v` is subtracted from each
    parameter's step."""
    opt_code = be.OPT_ADAMW

    def __init__(self, lr=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8, weight_decay=0.01):
        _check_adam_args(lr, beta1, beta2, epsilon)
        super().__init__(lr, beta1, beta2, epsilon, weight_decay)

    def _decay_coefficient(self):
        return 0.0

    def _step_decay(self):
        return float(self.lr) * float(self.weight_decay)

    def _hyper(self):
        return super()._hyper() + [1.0 - float(self.lr) * float(self.weight_decay)]


class RAdam(Adam):
    """Rectified Adam (torch.optim.RAdam): with mh = m/(1-b1^t),
    step = -lr * r_t * mh * sqrt(1-b2^t) / (sqrt(v) + eps) once the variance is tractable
    (rho_t > 5), step = -lr * mh before.  Weight decay is opt-in, as for the reference's rules."""
    opt_code = be.OPT_RADAM

    def __init__(self, lr=0.001, beta1=0.9, beta2=0.999, epsilon=1e-8, weight_decay=0.0):
        _check_adam_args(lr, beta1, beta2, epsilon)
        super().__init__(lr, beta1, beta2, epsilon, weight_decay)

    def _hyper(self):
        self._t += 1
        t, b2 = self._t, self._b2
        bc2 = 1.0 - b2 ** t
        rho_inf = 2.0 / (1.0 - b2) - 1.0
        rho_t = rho_inf - 2.0 * t * b2 ** t / bc2
        r_t = 0.0
        if rho_t > 5.0:
            r_t = math.sqrt((rho_t - 4.0) * (rho_t - 2.0) * rho_inf / ((rho_inf - 4.0) * (rho_inf - 2.0) * rho_t))
        return [self.lr, self._b1, b2, self._eps, 1.0 - self._b1 ** t, math.sqrt(bc2), r_t]


class Adamax(Adam):
    """Adam's infinity-norm variant (torch.optim.Adamax): u = max(b2*u, |g| + eps);
    step = -(lr/(1-b1^t)) * m / u.  Weight decay is opt-in, as for the reference's rules."""
    opt_code = be.OPT_ADAMAX

    def __init__(self, lr=0.002, beta1=0.9, beta2=0.999, epsilon=1e-8, weight_decay=0.0):
        _check_adam_args(lr, beta1, beta2, epsilon)
        super().__init__(lr, beta1, beta2, epsilon, weight_decay)

    def _hyper(self):
        self._t += 1
        return [self.lr, self._b1, self._b2, self._eps, self.lr / (1.0 - self._b1 ** self._t)]
