"""Loss functions (interface of the reference's core/losses.py: BaseLoss, SoftmaxCrossEntropyLoss).

The reference's softmax cross-entropy is unusual and the engine reproduces it exactly: the maximum
that is subtracted and the sum that normalises the exponentials are taken over the WHOLE
batch x class matrix (losses.py:26-27 call .max() and .sum() without an axis), so

    p_ij = exp(z_ij - max z) / sum_kl exp(z_kl - max z)
    L    = -(1/m) sum_i log( sum_j p_ij * labels_ij )

and the initial loss of an untrained classifier is about log(m * C), not log(C).  The fused node
(ops.softmax_ce_) computes this with three streaming passes forward and one backward; under data
parallelism the max / sum pair is merged across ranks so the normaliser still spans the global
batch.

Four elementwise losses have no reference counterpart (new): MSELoss, MAELoss, HuberLoss and
SigmoidCrossEntropyLoss.  Each is L = (1/m) sum over every element of l(p, t), m = the prediction's
row count (of the global batch under data parallelism): the per-sample convention of
MSEEvaluator / MAEEvaluator, sum over each row, mean over rows.  They run as one fused node
(ops.pointwise_loss_): one launch for the loss and, with backward()'s default seed, its gradient.
"""
import math

import numpy as np

import core._backend as be
import core.ops as ops
from core.tensor import Tensor, as_tensor


class BaseLoss(object):

    def loss(self, predicted, actual):
        raise NotImplementedError


class SoftmaxCrossEntropyLoss(BaseLoss):

    def __init__(self, weight=None):
        # `weight` ([n_classes]) is part of the reference signature; its weighted path indexes a
        # numpy array with a one-hot Tensor (losses.py:30-31) and cannot execute, so a weight is
        # accepted here only to be refused at call time with a clear message.
        self._weight = None if weight is None else np.asarray(weight)

    def loss(self, logits, labels):
        if type(logits) is not Tensor and isinstance(logits, Tensor):
            # a prediction Model.forward postponed (core/_deferred.py): the loss is postponed with it
            import core._deferred as deferred
            if type(logits) is deferred.LazyTensor:
                lazy = deferred.defer_loss(self, logits, labels)
                if lazy is not None:
                    return lazy
        if self._weight is not None:
            raise NotImplementedError(
                "class weights are not supported (the reference's weighted path is broken, "
                "losses.py:30-31)")
        z, y = as_tensor(logits), as_tensor(labels)
        fused_ok = z.ndim == 2 and tuple(y.shape) == tuple(z.shape)
        return ops.softmax_ce_(z, y) if fused_ok else self.loss_composed(z, y)

    @staticmethod
    def loss_composed(logits, labels):
        """The same quantity assembled from the primitive differentiable ops (eleven graph nodes,
        the way losses.py:25-32 builds it).  Serves shapes the fused kernel does not take and is
        the cross-check the test-suite runs against the fused node."""
        batch = logits.shape[0]
        shifted = ops.sub_(logits, ops.max_(logits, axis=None))        # z - max(z), global max
        unnormalised = ops.exp_(shifted)
        probs = ops.div_(unnormalised, ops.sum_(unnormalised, axis=None))   # global normaliser
        picked = ops.sum_(ops.mul_(probs, as_tensor(labels)), axis=1)   # q_i = sum_j p_ij y_ij
        total = ops.sum_(ops.neg_(ops.log_(picked)), axis=None)
        return total / batch


class _PointwiseLoss(BaseLoss):
    """L = (1/m) sum_all l(predicted, actual), m = predicted.shape[0]; dL/dpredicted only.

    Prediction and target have the same shape (any rank >= 1, no broadcasting) and the same dtype,
    float32 or float64; the target must not require a gradient.  NaN and +-inf propagate as in numpy;
    target values are not range-checked (that would need a read back to the host)."""

    _kind = None
    _delta = 1.0         # read by the Huber kind only

    def _config(self):
        """the fixed configuration a recorded step depends on beyond the class (Model._step_key)"""
        return ()

    def loss(self, predicted, actual):
        self._check(predicted, actual)
        if type(predicted) is not Tensor and isinstance(predicted, Tensor):
            # a prediction Model.forward postponed (core/_deferred.py): the loss is postponed with it
            import core._deferred as deferred
            if type(predicted) is deferred.LazyTensor:
                lazy = deferred.defer_loss(self, predicted, actual)
                if lazy is not None:
                    return lazy
        return ops.pointwise_loss_(as_tensor(predicted), as_tensor(actual), self._kind, self._delta)

    @staticmethod
    def _describe(x):
        """(shape, dtype on the device, requires_grad) without touching the device"""
        if isinstance(x, np.ndarray) or not (hasattr(x, "shape") and hasattr(x, "dtype")):
            arr = np.asarray(x)
            try:
                return arr.shape, be.device_dtype(arr.dtype), False
            except TypeError as exc:
                raise ValueError(str(exc))
        return tuple(x.shape), np.dtype(x.dtype), bool(getattr(x, "requires_grad", False))

    def _check(self, predicted, actual):
        name = type(self).__name__
        p_shape, p_dtype, _ = self._describe(predicted)
        t_shape, t_dtype, t_grad = self._describe(actual)
        if p_shape != t_shape:
            raise ValueError("%s: prediction %s and target %s must have the same shape (no broadcasting)"
                             % (name, p_shape, t_shape))
        if len(p_shape) < 1:
            raise ValueError("%s: the prediction needs at least one axis (the batch rows)" % name)
        if p_shape[0] < 1:
            raise ValueError("%s: the batch has no rows" % name)
        if p_dtype not in (be.F32, be.F64) or t_dtype != p_dtype:
            raise ValueError("%s: prediction (%s) and target (%s) must both be float32 or both float64"
                             % (name, p_dtype, t_dtype))
        if t_grad:
            raise ValueError("%s: the target requires a gradient; the loss differentiates the "
                             "prediction only" % name)


class MSELoss(_PointwiseLoss):
    """l = (p - t)^2; for a 2-D prediction L equals MSEEvaluator's "mse" (new)"""
    _kind = be.LOSS_MSE


class MAELoss(_PointwiseLoss):
    """l = |p - t|, gradient sign(p - t) with 0 at p = t (new)"""
    _kind = be.LOSS_MAE


class HuberLoss(_PointwiseLoss):
    """l = (p - t)^2 / 2 where |p - t| < delta, else delta * (|p - t| - delta / 2) (new).  delta is
    fixed at construction: it is part of what a recorded training step computes."""
    _kind = be.LOSS_HUBER

    def __init__(self, delta=1.0):
        if isinstance(delta, (bool, np.bool_)) or not isinstance(delta, (int, float, np.integer, np.floating)):
            raise ValueError("HuberLoss: delta must be a number, got %r" % (delta,))
        delta = float(delta)
        if not (math.isfinite(delta) and delta > 0.0):
            raise ValueError("HuberLoss: delta must be finite and > 0, got %r" % delta)
        self._delta = delta

    @property
    def delta(self):
        return self._delta

    def _config(self):
        return (self._delta,)


class SigmoidCrossEntropyLoss(_PointwiseLoss):
    """Binary cross-entropy of logits z against targets t in [0, 1] (soft targets allowed), one
    independent sigmoid per element -- multi-label classification (new):
    l = max(z, 0) - z t + log1p(exp(-|z|)), gradient sigmoid(z) - t."""
    _kind = be.LOSS_SIGMOID_CE
