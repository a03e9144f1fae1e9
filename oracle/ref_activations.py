"""CPU oracle for the elementwise activations of core/layers.py (LeakyReLU, ELU, GELU in both forms,
Softplus, SiLU): float64 numpy values and derivatives, and each activation as a RefTensor node.

TEST INFRASTRUCTURE ONLY (same rules as oracle/ref_numpy.py: imported by tests/ and scripts only).
The semantics restated here are the ones core/layers.py and include/tnn_b200.h document:

    leaky_relu  y = x if x >= 0 else slope x                  y' = 1 if x >= 0 else slope
    elu         y = x if x >= 0 else alpha expm1(x)           y' = 1 if x >= 0 else alpha exp(x)
    gelu        y = x Phi(x), Phi(x) = erfc(-x/sqrt2)/2       y' = Phi(x) + x phi(x)
    gelu_tanh   y = x s, s = sigma(2u),                       y' = s + 2x s(1-s) sqrt(2/pi)(1 + 0.134145 x^2)
                u = sqrt(2/pi)(x + 0.044715 x^3)
    softplus    y = max(x, 0) + log1p(exp(-|x|))              y' = sigma(x)
    silu        y = x sigma(x)                                y' = sigma(x)(1 + x(1 - sigma(x)))

with the kink at 0 in the x >= 0 branch, NaN -> NaN, +-inf -> the limits of the function and of its
derivative, and a product whose weight underflowed to 0 taken as 0 (never inf * 0).

tests/test_activations_host.py pins this module against torch's float64 autograd away from x = 0.
"""
import numpy as np
from scipy.special import erfc

from ref_numpy import _node

KINDS = ("leaky_relu", "elu", "gelu", "gelu_tanh", "softplus", "silu")
DEFAULT_PARAM = {"leaky_relu": 0.01, "elu": 1.0}

_SQRT_2_OVER_PI = np.sqrt(2.0 / np.pi)


def _sigmoid2(v):
    """(sigma(v), sigma(-v)) without overflow"""
    e = np.exp(-np.abs(v))
    lo, hi = e / (1.0 + e), 1.0 / (1.0 + e)
    pos = v >= 0.0
    return np.where(pos, hi, lo), np.where(pos, lo, hi)


def _mul_or_zero(x, w):
    return np.where(w == 0.0, 0.0, x * w)


def terms(x, kind, param=None):
    """(y, dy/dx) per element, float64 arrays of x's shape; param is slope / alpha"""
    x = np.asarray(x, np.float64)
    p = DEFAULT_PARAM.get(kind, 0.0) if param is None else float(param)
    nan = np.full(x.shape, np.nan)
    with np.errstate(all="ignore"):
        if kind == "leaky_relu":
            neg = x < 0.0
            return (np.where(neg, _mul_or_zero(x, p), x),
                    np.where(neg, p, np.where(x >= 0.0, 1.0, nan)))
        if kind == "elu":
            pos = x >= 0.0
            return np.where(pos, x, p * np.expm1(x)), np.where(pos, 1.0, p * np.exp(x))
        if kind == "gelu":
            cdf = 0.5 * erfc(-x / np.sqrt(2.0))
            pdf = np.exp(-0.5 * (x * x)) / np.sqrt(2.0 * np.pi)
            return _mul_or_zero(x, cdf), cdf + _mul_or_zero(x, pdf)
        if kind == "gelu_tanh":
            s, sn = _sigmoid2(2.0 * _SQRT_2_OVER_PI * (x + 0.044715 * (x * x * x)))
            w = s * sn
            t = np.where(w == 0.0, 0.0, 2.0 * x * w * _SQRT_2_OVER_PI * (1.0 + 0.134145 * (x * x)))
            return _mul_or_zero(x, s), s + t
        if kind == "softplus":
            return np.where(x > 0.0, x, 0.0) + np.log1p(np.exp(-np.abs(x))), _sigmoid2(x)[0]
        if kind == "silu":
            s, sn = _sigmoid2(x)
            return _mul_or_zero(x, s), s + _mul_or_zero(x, s * sn)
    raise ValueError("unknown activation %r" % (kind,))


def value_and_grad(x, kind, param=None, g=1.0):
    """(y, dL/dx for the upstream gradient g)"""
    y, d = terms(x, kind, param)
    with np.errstate(all="ignore"):
        return y, np.asarray(g, np.float64) * d


def activation(a, kind, param=None):
    """the activation of a RefTensor as a RefTensor node"""
    y, d = terms(a.values, kind, param)
    return _node(y, [(a, lambda g: np.asarray(g, np.float64) * d)])
