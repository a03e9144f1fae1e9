"""Learning-rate schedules for the optimisers of core/optimizer.py.

A scheduler only writes `optimizer.lr`.  Every optimiser reads that attribute when it forms a step's
coefficients (BaseOptimizer._hyper8), on the eager step and in the upload before each replay of a
recorded step, so a schedule needs nothing from the engine.

Construction records `base_lr = optimizer.lr` and sets `optimizer.lr` to the epoch-0 value;
`step()` advances `last_epoch` by one and sets the new value.  Each schedule is a closed form of
the epoch, equal to what `torch.optim.lr_scheduler` gives when its `step()` is called once per
epoch.
"""
import math
import numbers


def _positive_int(name, v):
    if isinstance(v, bool) or not isinstance(v, numbers.Integral) or v <= 0:
        raise ValueError("%s must be a positive int, got %r" % (name, v))
    return int(v)


def _finite(name, v, lo=None, hi=None):
    if not (isinstance(v, numbers.Real) and math.isfinite(v)):
        raise ValueError("%s must be a finite number, got %r" % (name, v))
    if (lo is not None and v < lo) or (hi is not None and v > hi):
        raise ValueError("%s must lie in [%s, %s], got %r" % (name, lo, hi, v))
    return float(v)


class LRScheduler(object):

    def __init__(self, optimizer):
        self.optimizer = optimizer
        self.base_lr = optimizer.lr
        self.last_epoch = 0
        optimizer.lr = self._lr_at(0)

    def step(self):
        self.last_epoch += 1
        self.optimizer.lr = self._lr_at(self.last_epoch)

    def get_lr(self):
        """the learning rate of the current epoch"""
        return self._lr_at(self.last_epoch)

    def _lr_at(self, epoch):
        raise NotImplementedError


class StepLR(LRScheduler):
    """base_lr * gamma ** (epoch // step_size)"""

    def __init__(self, optimizer, step_size, gamma=0.1):
        self.step_size = _positive_int("step_size", step_size)
        self.gamma = _finite("gamma", gamma, lo=0.0)
        super().__init__(optimizer)

    def _lr_at(self, e):
        return self.base_lr * self.gamma ** (e // self.step_size)


class MultiStepLR(LRScheduler):
    """base_lr * gamma ** (number of milestones <= epoch)"""

    def __init__(self, optimizer, milestones, gamma=0.1):
        ms = [_positive_int("milestone", m) for m in milestones]
        if any(a >= b for a, b in zip(ms, ms[1:])):
            raise ValueError("milestones must be strictly increasing, got %r" % (list(milestones),))
        self.milestones = ms
        self.gamma = _finite("gamma", gamma, lo=0.0)
        super().__init__(optimizer)

    def _lr_at(self, e):
        return self.base_lr * self.gamma ** sum(1 for m in self.milestones if m <= e)


class ExponentialLR(LRScheduler):
    """base_lr * gamma ** epoch"""

    def __init__(self, optimizer, gamma):
        self.gamma = _finite("gamma", gamma, lo=0.0)
        super().__init__(optimizer)

    def _lr_at(self, e):
        return self.base_lr * self.gamma ** e


class CosineAnnealingLR(LRScheduler):
    """eta_min + (base_lr - eta_min) * (1 + cos(pi * epoch / T_max)) / 2; past T_max the cosine
    rises again, as torch's does"""

    def __init__(self, optimizer, T_max, eta_min=0.0):
        self.T_max = _positive_int("T_max", T_max)
        self.eta_min = _finite("eta_min", eta_min, lo=0.0)
        super().__init__(optimizer)

    def _lr_at(self, e):
        return self.eta_min + (self.base_lr - self.eta_min) * (1.0 + math.cos(math.pi * e / self.T_max)) / 2.0


class LinearLR(LRScheduler):
    """base_lr * (start + (end - start) * min(epoch, total_iters) / total_iters)"""

    def __init__(self, optimizer, start_factor=1.0 / 3, end_factor=1.0, total_iters=5):
        if not (isinstance(start_factor, numbers.Real) and 0.0 < start_factor <= 1.0):
            raise ValueError("start_factor must lie in (0, 1], got %r" % (start_factor,))
        self.start_factor = float(start_factor)
        self.end_factor = _finite("end_factor", end_factor, lo=0.0, hi=1.0)
        self.total_iters = _positive_int("total_iters", total_iters)
        super().__init__(optimizer)

    def _lr_at(self, e):
        s, f = self.start_factor, self.end_factor
        return self.base_lr * (s + (f - s) * min(e, self.total_iters) / self.total_iters)
