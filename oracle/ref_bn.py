"""CPU oracle for BatchNormalization: float64 numpy batch normalisation as a RefTensor node, in both
phases, with the running-statistics update.

TEST INFRASTRUCTURE ONLY (same rules as oracle/ref_numpy.py: imported by tests/ and scripts only).
The semantics restated here are the ones core/layers.py documents for BatchNormalization (the torch
conventions: biased variance for the normalisation, unbiased for the running variance).
tests/test_batchnorm_host.py pins this module against torch.nn.functional.batch_norm on the CPU.
"""
import numpy as np

from ref_numpy import _node


class RefBNState(object):
    """running statistics (float64, C values each) and the layer's constants"""

    def __init__(self, C, momentum=0.1, eps=1e-5, running_mean=None, running_var=None):
        self.momentum, self.eps = float(momentum), float(eps)
        self.running_mean = np.zeros(C) if running_mean is None else np.array(running_mean, np.float64).ravel()
        self.running_var = np.ones(C) if running_var is None else np.array(running_var, np.float64).ravel()


def batchnorm(x, gamma, beta, state, training, stats=None):
    """x (..., C), gamma and beta (1, C) RefTensors -> y of x's shape, normalised over every axis but
    the last.  TRAIN updates `state` in place.  `stats` = (n, mean, M2) replaces the batch's own
    statistics (the global ones of a data-parallel run); backward then expects its `sums` hook to
    be given the global sums (see vjp_x.sums) -- None keeps the single-process maths."""
    xv = np.asarray(x.values, np.float64)
    shape = xv.shape
    C = shape[-1]
    x2 = xv.reshape(-1, C)
    M = x2.shape[0]
    g = np.asarray(gamma.values, np.float64).reshape(C)
    b = np.asarray(beta.values, np.float64).reshape(C)
    if training:
        if stats is None:
            n, mean = M, x2.mean(axis=0)
            m2 = ((x2 - mean) ** 2).sum(axis=0)
        else:
            n, mean, m2 = stats
        var = m2 / n
        state.running_mean = (1 - state.momentum) * state.running_mean + state.momentum * mean
        state.running_var = (1 - state.momentum) * state.running_var + state.momentum * (m2 / (n - 1))
    else:
        n, mean, var = M, state.running_mean.copy(), state.running_var.copy()
    r = 1.0 / np.sqrt(var + state.eps)
    xhat = (x2 - mean) * r
    y = (xhat * g + b).reshape(shape)

    def local_sums(dy):
        d2 = np.asarray(dy, np.float64).reshape(-1, C)
        return d2.sum(axis=0), (d2 * xhat).sum(axis=0)

    def vjp_x(dy):
        d2 = np.asarray(dy, np.float64).reshape(-1, C)
        if not training:
            return (d2 * g * r).reshape(shape)
        s_dy, s_dyx = vjp_x.sums(dy) if vjp_x.sums is not None else local_sums(dy)
        return (g * r * (d2 - s_dy / n - xhat * s_dyx / n)).reshape(shape)

    vjp_x.sums = None

    def vjp_gamma(dy):
        return local_sums(dy)[1].reshape(1, C)

    def vjp_beta(dy):
        return local_sums(dy)[0].reshape(1, C)

    node = _node(y, [(x, vjp_x), (gamma, vjp_gamma), (beta, vjp_beta)])
    node.bn_vjp_x = vjp_x
    node.bn_local_sums = local_sums
    return node


def local_stats(x2):
    """(n, mean[C], M2[C]) of the rows of x2 (M, C), the triple a rank contributes to the merge"""
    x2 = np.asarray(x2, np.float64)
    n = x2.shape[0]
    if n == 0:
        return 0, np.zeros(x2.shape[1]), np.zeros(x2.shape[1])
    mean = x2.mean(axis=0)
    return n, mean, ((x2 - mean) ** 2).sum(axis=0)
