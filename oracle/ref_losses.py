"""CPU oracle for the pointwise losses of core/losses.py (MSELoss, MAELoss, HuberLoss,
SigmoidCrossEntropyLoss): float64 numpy values and gradients, and the loss as a RefTensor node.

TEST INFRASTRUCTURE ONLY (same rules as oracle/ref_numpy.py: imported by tests/ and scripts only).
The semantics restated here are the ones core/losses.py documents:

    L = (1/m) * sum over every element of l(p, t),  m = p.shape[0] (the global batch's rows)

with e = p - t and
    mse         l = e^2                                                 dl/dp = 2e
    mae         l = |e|                                                 dl/dp = sign(e)
    huber       l = e^2/2 if |e| < delta else delta (|e| - delta/2)     dl/dp = e or delta sign(e)
    sigmoid_ce  l = max(z, 0) - z t + log1p(exp(-|z|))                 dl/dz = sigmoid(z) - t

tests/test_losses_host.py pins this module against torch's mse_loss, l1_loss, huber_loss and
binary_cross_entropy_with_logits (reduction="sum", divided by m) on the CPU.
"""
import numpy as np

from ref_numpy import _node

KINDS = ("mse", "mae", "huber", "sigmoid_ce")


def terms(p, t, kind, delta=1.0):
    """(l, dl/dp) per element, float64 arrays of p's shape"""
    p = np.asarray(p, np.float64)
    t = np.asarray(t, np.float64)
    with np.errstate(all="ignore"):
        if kind == "sigmoid_ce":
            en = np.exp(-np.abs(p))
            l = (np.maximum(p, 0.0) - p * t) + np.log1p(en)
            d = np.where(p >= 0.0, 1.0, en) / (1.0 + en) - t
            return l, d
        e = p - t
        if kind == "mse":
            return e * e, 2.0 * e
        if kind == "mae":
            return np.abs(e), np.sign(e)
        if kind == "huber":
            a = np.abs(e)
            quad = a < delta
            return (np.where(quad, 0.5 * e * e, delta * (a - 0.5 * delta)),
                    np.where(quad, e, delta * np.sign(e)))
    raise ValueError("unknown loss kind %r" % (kind,))


def loss_and_grad(p, t, kind, delta=1.0, m=None, g=1.0):
    """(L, dL/dp for the upstream gradient g); m defaults to p.shape[0]"""
    p = np.asarray(p, np.float64)
    m = p.shape[0] if m is None else m
    l, d = terms(p, t, kind, delta)
    with np.errstate(all="ignore"):
        return l.sum() / m, d * (g / m)


def pointwise_loss(pred, target, kind, delta=1.0, m=None):
    """the loss of a RefTensor prediction against a fixed target, as a RefTensor node"""
    m = pred.values.shape[0] if m is None else m
    l, d = terms(pred.values, target, kind, delta)
    return _node(np.asarray(l.sum() / m), [(pred, lambda g: d * (np.asarray(g, np.float64) / m))])
