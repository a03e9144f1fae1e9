"""Differentiable tensor operations: the function table of the reference's core/ops.py, with every
forward value and gradient product computed by a CUDA kernel (core/_backend.py ->
libtnn_b200.so).  Names, arguments and gradient conventions follow the reference; citations are
to /root/reference/core/ops.py.

A grad_fn receives the incoming gradient as a device array and returns a device array; the
un-broadcast reduction the reference inlines twelve times (ops.py:41-46 ...) is one backend call.
Three fused nodes are added for the training path (dense_, relu_, softmax_ce_); they are what
core/layers.py and core/losses.py use.  Two more serve the NHWC image layers: im2col_ (Conv2D's
window matrix) and maxpool2d_; batchnorm_ is BatchNormalization, and pointwise_loss_ the MSE, MAE,
Huber and sigmoid cross-entropy losses.
"""
import builtins as _bi

import numpy as np

import os

import core._backend as be

# ReLU-backward mask fused into the dX GEMM epilogue.  Correct and bit-identical (tested).  On the
# tensor-core path it is 6 fewer launches per wide-MLP step (3 relu_bwd + 3 operand splits: the
# masked gradient leaves the epilogue with its planes).  r01 measured no gain (11.58 vs 11.58 ms);
# with r02's longer accumulator chunks the epilogue has more slack and the A/B is 11.07 / 11.08 ms
# fused against 11.19 ms unfused (same box, alternating runs), so it is on by default
# (TNN_FUSE_RELU_BWD=0 turns it off).  On the SIMT path (MNIST-sized layers, launch-bound) it is
# always on: one launch less per hidden layer.
FUSE_RELU_BWD = os.environ.get("TNN_FUSE_RELU_BWD", "1") != "0"
# dX, dW and db of a small Dense layer as one grouped launch (tnn_dense_bwd_simt)
GROUP_SMALL_DENSE_BWD = os.environ.get("TNN_GROUP_DENSE_BWD", "1") != "0"
WRITTEN_IN_PLACE = object()   # returned by a node's _fused_bwd for gradients it wrote into their slot


_GRAD_ENABLED = True


class no_grad(object):
    """Context manager: ops run inside it build no autograd graph (outputs have requires_grad =
    False and hold no references to their inputs), the way an evaluation forward pass wants it
    (run.py:87-91).  Not part of the reference's interface; Model.predict() uses it."""

    def __enter__(self):
        global _GRAD_ENABLED
        self._prev = _GRAD_ENABLED
        _GRAD_ENABLED = False
        return self

    def __exit__(self, *exc):
        global _GRAD_ENABLED
        _GRAD_ENABLED = self._prev
        return False


def as_tensor(obj, like=None):
    # avoid looping import
    from core.tensor import as_tensor
    return as_tensor(obj, like)


def build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values):
    """ops.py:12-20"""
    requires_grad = (ts1.requires_grad or ts2.requires_grad) and _GRAD_ENABLED
    dependency = []
    if ts1.requires_grad and requires_grad:
        dependency.append(dict(tensor=ts1, grad_fn=grad_fn_ts1))
    if ts2.requires_grad and requires_grad:
        dependency.append(dict(tensor=ts2, grad_fn=grad_fn_ts2))
    tensor_cls = ts1.__class__
    return tensor_cls(values, requires_grad, dependency)


def build_unary_ops_tensor(ts, grad_fn, values):
    """ops.py:23-29"""
    requires_grad = ts.requires_grad and _GRAD_ENABLED
    dependency = []
    if requires_grad:
        dependency.append(dict(tensor=ts, grad_fn=grad_fn))
    tensor_cls = ts.__class__
    return tensor_cls(values, requires_grad, dependency)


# ------------------------------------------------------------------------------ binary ops
def add_(ts1, ts2):
    """ops.py:32-58"""
    a, b = ts1._data, ts2._data
    values = be.ew(be.ADD, a, b)

    def grad_fn_ts1(grad):
        return be.unbroadcast(grad, a.shape)

    def grad_fn_ts2(grad):
        return be.unbroadcast(grad, b.shape)

    return build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values)


def sub_(ts1, ts2):
    """ops.py:61-62 builds add(ts1, neg(ts2)); here one kernel and one node, same gradients"""
    a, b = ts1._data, ts2._data
    values = be.ew(be.SUB, a, b)

    def grad_fn_ts1(grad):
        return be.unbroadcast(grad, a.shape)

    def grad_fn_ts2(grad):
        return be.unbroadcast(be.ew(be.NEG, grad), b.shape)

    return build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values)


def mul_(ts1, ts2):
    """ops.py:65-90"""
    a, b = ts1._data, ts2._data
    values = be.ew(be.MUL, a, b)

    def grad_fn_ts1(grad):
        return be.unbroadcast(be.ew(be.MUL, grad, b), a.shape)

    def grad_fn_ts2(grad):
        return be.unbroadcast(be.ew(be.MUL, grad, a), b.shape)

    return build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values)


def div_(ts1, ts2):
    """ops.py:93-118: d/da = g / b, d/db = -g * a / b**2"""
    a, b = ts1._data, ts2._data
    values = be.ew(be.DIV, a, b)

    def grad_fn_ts1(grad):
        return be.unbroadcast(be.ew(be.DIV, grad, b), a.shape)

    def grad_fn_ts2(grad):
        return be.unbroadcast(be.ew(be.DIV_BWD_B, grad, a, b), b.shape)

    return build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values)


def pow_(ts1, ts2):
    """ops.py:121-147: d/da = g * b * a**(b-1), d/db = g * ln(a) * a**b"""
    a, b = ts1._data, ts2._data
    values = be.ew(be.POW, a, b)

    def grad_fn_ts1(grad):
        return be.unbroadcast(be.ew(be.POW_BWD_A, grad, a, b), a.shape)

    def grad_fn_ts2(grad):
        return be.unbroadcast(be.ew(be.POW_BWD_B, grad, a, values), b.shape)

    return build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values)


def dot_(ts1, ts2):
    """ops.py:150-163: C = A @ B, dA = g @ B.T, dB = A.T @ g"""
    a, b = ts1._data, ts2._data
    values = be.matmul(a, b, reuse_a=ts2.requires_grad, reuse_b=ts1.requires_grad)

    def grad_fn_ts1(grad, out=None, accumulate=False):
        return be.matmul(grad, b, tb=True, out=out, accumulate=accumulate,
                         reuse_a=ts2.requires_grad)

    def grad_fn_ts2(grad, out=None, accumulate=False):
        return be.matmul(a, grad, ta=True, out=out, accumulate=accumulate,
                         reuse_b=ts1.requires_grad)

    grad_fn_ts1.supports_out = True
    grad_fn_ts2.supports_out = True
    return build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values)


def maximum_(ts1, ts2):
    """ops.py:166-188: ties go to ts1 (>= for ts1, > for ts2)"""
    a, b = ts1._data, ts2._data
    values = be.ew(be.MAXIMUM, a, b)

    def grad_fn_ts1(grad):
        return be.unbroadcast(be.ew(be.MUL_GE, grad, a, b), a.shape)

    def grad_fn_ts2(grad):
        return be.unbroadcast(be.ew(be.MUL_GT, grad, b, a), b.shape)

    return build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values)


def minimum_(ts1, ts2):
    """ops.py:191-213: ties go to ts1 (<= for ts1, < for ts2)"""
    a, b = ts1._data, ts2._data
    values = be.ew(be.MINIMUM, a, b)

    def grad_fn_ts1(grad):
        return be.unbroadcast(be.ew(be.MUL_LE, grad, a, b), a.shape)

    def grad_fn_ts2(grad):
        return be.unbroadcast(be.ew(be.MUL_LT, grad, b, a), b.shape)

    return build_binary_ops_tensor(ts1, ts2, grad_fn_ts1, grad_fn_ts2, values)


# ------------------------------------------------------------------------------ unary ops
def exp_(ts):
    """ops.py:216-222: the gradient reuses the forward values"""
    values = be.ew(be.EXP, ts._data)

    def grad_fn(grad):
        return be.ew(be.MUL, values, grad)

    return build_unary_ops_tensor(ts, grad_fn, values)


def log_(ts):
    """ops.py:243-249"""
    x = ts._data
    values = be.ew(be.LOG, x)

    def grad_fn(grad):
        return be.ew(be.DIV, grad, x)

    return build_unary_ops_tensor(ts, grad_fn, values)


def neg_(ts):
    """ops.py:293-299"""
    values = be.ew(be.NEG, ts._data)

    def grad_fn(grad):
        return be.ew(be.NEG, grad)

    return build_unary_ops_tensor(ts, grad_fn, values)


def _extreme(ts, axis, red_op):
    x = ts._data
    values = be.reduce(red_op, x, axis)
    if axis is None:
        keep_shape = (1,) * x.ndim
    else:
        ax = axis % x.ndim
        keep_shape = x.shape[:ax] + (1,) + x.shape[ax + 1:]

    def grad_fn(grad):
        # ops.py:228-229: grad * (x.max(axis, keepdims=1) == x); every tied element gets the
        # full gradient.  The incoming gradient is expanded with keepdims, which also makes
        # axis >= 1 well defined (the reference mis-broadcasts there, SURVEY Q10).
        g = grad.view(keep_shape) if grad.size == values.size else grad
        return be.ew(be.MUL_EQ, g, x, values.view(keep_shape))

    return build_unary_ops_tensor(ts, grad_fn, values)


def max_(ts, axis=None):
    """ops.py:225-231"""
    return _extreme(ts, axis, be.RED_MAX)


def min_(ts, axis=None):
    """ops.py:234-240"""
    return _extreme(ts, axis, be.RED_MIN)


def sum_(ts, axis):
    """ops.py:252-265"""
    x = ts._data
    values = be.reduce(be.RED_SUM, x, axis)
    if axis is None:
        keep_shape = (1,) * x.ndim
    else:
        ax = axis % x.ndim
        keep_shape = x.shape[:ax] + (1,) + x.shape[ax + 1:]

    def grad_fn(grad):
        g = grad.view(keep_shape) if grad.size == values.size else grad
        return be.broadcast_to(g, x.shape)

    return build_unary_ops_tensor(ts, grad_fn, values)


def transpose_(ts, axes=None):
    """ops.py:268-279"""
    x = ts._data
    if axes is None:
        axes = list(reversed(range(x.ndim)))
    axes = [int(a) for a in axes]
    values = be.permute(x, axes)
    inverse = [int(i) for i in np.argsort(axes)]

    def grad_fn(grad):
        return be.permute(grad, inverse)

    return build_unary_ops_tensor(ts, grad_fn, values)


def _as_index_array(key):
    """a 1-D integer index vector (list / ndarray / Tensor) or None"""
    if hasattr(key, "_data"):
        key = key.values
    if isinstance(key, (list, np.ndarray)):
        arr = np.asarray(key)
        if arr.ndim == 1 and arr.dtype.kind in "iu":
            return arr.astype(np.int64)
        if arr.ndim == 1 and arr.size == 0:
            return arr.astype(np.int64)
    return None


def _last_writer(idx, modulus):
    """numpy's `out[idx] = g` lets the LAST occurrence of a repeated index win.  A parallel scatter
    would race, so repeated indices are resolved here: returns (unique indices, position of the
    last occurrence of each) or None when every index is distinct."""
    norm = np.where(idx < 0, idx + modulus, idx)
    uniq, first_rev = np.unique(norm[::-1], return_index=True)
    if uniq.size == norm.size:
        return None
    return uniq.astype(np.int64), (norm.size - 1 - first_rev).astype(np.int64)


def getitem_(ts, key):
    """ops.py:282-290: x[key]; backward writes the gradient into zeros_like(x) at key
    (assignment, duplicates are not accumulated).

    Row slices are zero-copy views, integer row vectors use the row-gather kernel (the two
    access patterns of utils/data_iterator.py:27-33); any other numpy key is resolved to a flat
    element index map on the host and executed by the flat gather/scatter kernels."""
    x = ts._data
    shape = x.shape
    if x.ndim >= 1 and isinstance(key, slice):
        start, stop, step = key.indices(shape[0])
        if step == 1:
            n = _bi.max(stop - start, 0)
            row = be._prod(shape[1:])
            values = x.view((n,) + shape[1:], start * row)

            def grad_fn(grad):
                out = be.zeros(shape, x.dtype)
                if n:
                    be.copy_into(out.view((n,) + shape[1:], start * row), grad)
                return out

            return build_unary_ops_tensor(ts, grad_fn, values)
    if x.ndim >= 1 and isinstance(key, (int, np.integer)) and not isinstance(key, bool):
        k = int(key)
        if not -shape[0] <= k < shape[0]:
            raise IndexError("index %d is out of bounds for axis 0 with size %d" % (k, shape[0]))
        k %= shape[0]
        row = be._prod(shape[1:])
        values = x.view(shape[1:], k * row)

        def grad_fn(grad):
            out = be.zeros(shape, x.dtype)
            be.copy_into(out.view(shape[1:], k * row), grad)
            return out

        return build_unary_ops_tensor(ts, grad_fn, values)
    idx = _as_index_array(key) if x.ndim >= 1 else None
    if idx is not None:
        if idx.size and (idx.min() < -shape[0] or idx.max() >= shape[0]):
            raise IndexError("index out of bounds for axis 0 with size %d" % shape[0])
        n_idx = int(idx.size)
        idx_dev = be.upload_index(idx)
        values = be.gather_rows(x, idx_dev, n_idx)
        dup = _last_writer(idx, shape[0]) if n_idx > 1 else None

        def grad_fn(grad):
            if dup is None:
                return be.scatter_rows(grad, idx_dev, n_idx, shape)
            uniq, last = dup   # deterministic "last write wins", as numpy's assignment
            winners = be.gather_rows(grad, be.upload_index(last), int(last.size))
            return be.scatter_rows(winners, be.upload_index(uniq), int(uniq.size), shape)

        return build_unary_ops_tensor(ts, grad_fn, values)
    # general numpy key
    if hasattr(key, "_data"):
        key = key.values
    if isinstance(key, tuple):
        key = tuple(k.values if hasattr(k, "_data") else k for k in key)
    flat = np.arange(x.size, dtype=np.int64).reshape(shape)[key]
    oshape = flat.shape
    flat_idx = np.ascontiguousarray(flat).ravel()
    idx_dev = be.upload_index(flat_idx)
    values = be.gather_flat(x, idx_dev, oshape)
    dup = _last_writer(flat_idx, x.size) if flat_idx.size > 1 else None

    def grad_fn(grad):
        if dup is None:
            return be.scatter_flat(grad, idx_dev, shape)
        uniq, last = dup
        winners = be.gather_flat(grad.view((grad.size,)), be.upload_index(last), (int(last.size),))
        return be.scatter_flat(winners, be.upload_index(uniq), shape)

    return build_unary_ops_tensor(ts, grad_fn, values)


def _resolve_shape(size, newshape):
    """numpy's reshape rules (one -1 allowed) without touching any data"""
    if isinstance(newshape, (int, np.integer)):
        newshape = (newshape,)
    dims = [int(d) for d in newshape]
    if dims.count(-1) > 1:
        raise ValueError("can only specify one unknown dimension")
    known = 1
    for d in dims:
        if d != -1:
            if d < 0:
                raise ValueError("negative dimensions not allowed")
            known *= d
    if -1 in dims:
        if known == 0 or size % known != 0:
            raise ValueError("cannot reshape array of size %d into shape %s" % (size, tuple(newshape)))
        dims[dims.index(-1)] = size // known
    elif known != size:
        raise ValueError("cannot reshape array of size %d into shape %s" % (size, tuple(newshape)))
    return tuple(dims)


def reshape_(ts, newshape):
    """ops.py:302-309: a view, no kernel"""
    x = ts._data
    shape = x.shape
    target = _resolve_shape(x.size, newshape)
    values = x.view(target)

    def grad_fn(grad):
        return grad.view(shape)

    return build_unary_ops_tensor(ts, grad_fn, values)


def pad_(ts, pad_width, mode):
    """ops.py:312-321.  Constant (zero) padding only: the reference's backward is a plain slice,
    which is only the right gradient for that mode (SURVEY Q17)."""
    if mode != "constant":
        raise NotImplementedError("pad_: only mode='constant' is supported on the device")
    x = ts._data
    pw = np.broadcast_to(np.asarray(pad_width, dtype=np.int64), (x.ndim, 2))
    if (pw < 0).any():
        raise ValueError("index can't contain negative values")
    oshape = tuple(int(s + b + a) for s, (b, a) in zip(x.shape, pw))
    ostr = be._cstrides(oshape)
    xstr = be._cstrides(x.shape)
    offset = int(_bi.sum(int(b) * st for (b, _), st in zip(pw, ostr)))
    values = be.zeros(oshape, x.dtype)
    be.strided_copy(values, offset, ostr, x, 0, xstr, x.shape)

    def grad_fn(grad):
        out = be.empty(x.shape, grad.dtype)
        be.strided_copy(out, 0, xstr, grad, offset, ostr, x.shape)
        return out

    return build_unary_ops_tensor(ts, grad_fn, values)


def flatten_(ts):
    """ops.py:324-330"""
    x = ts._data
    shape = x.shape
    values = x.view((x.size,))

    def grad_fn(grad):
        return grad.view(shape)

    return build_unary_ops_tensor(ts, grad_fn, values)


def clip_(ts, min, max):
    """ops.py:333-344: x.clip(min, max); gradient mask is (x >= min) & (x <= max), inclusive on
    both sides, taken from the pre-clip values (so ReLU'(0) = 1)."""
    x = ts._data
    if min is None and max is None:
        raise ValueError("One of max or min must be given")
    if min is not None and max is None and float(min) == 0.0:
        return relu_(ts)
    flags = (1 if min is not None else 0) | (2 if max is not None else 0)
    p0 = float(min) if min is not None else 0.0
    p1 = float(max) if max is not None else 0.0
    values = be.ew(be.CLIP, x, p0=p0, p1=p1, flags=flags)

    def grad_fn(grad):
        return be.ew(be.CLIP_BWD, grad, x, p0=p0, p1=p1, flags=flags)

    return build_unary_ops_tensor(ts, grad_fn, values)


# ------------------------------------------------------------------------------ fused nodes
def relu_(ts):
    """clip(x, 0.0) as used by layers.py:97-98, one kernel each way; mask = (x >= 0)"""
    x = ts._data
    values = be.relu_fwd(x)

    def grad_fn(grad):
        return be.relu_bwd(grad, x)

    return build_unary_ops_tensor(ts, grad_fn, values)


def dense_(ts_x, ts_w, ts_b):
    """inputs @ w + b of layers.py:49 as one node: the bias add runs in the GEMM epilogue, the
    bias gradient is the column sum of the incoming gradient (ops.py:49-55 on the (1, N) bias)."""
    x, w, b = ts_x._data, ts_w._data, ts_b._data
    if b.shape != (1, w.shape[1]) or x.dtype != w.dtype or b.dtype != w.dtype:
        return ts_x @ ts_w + ts_b
    values = be.matmul(x, w, bias=b, reuse_a=ts_w.requires_grad, reuse_b=ts_x.requires_grad)
    return _dense_node(ts_x, ts_w, ts_b, values)


def _dense_node(ts_x, ts_w, ts_b, values):
    """graph node of x@w+b: dX = g@w.T, dW = x.T@g, db = column sum of g"""
    x, w = ts_x._data, ts_w._data

    pre = getattr(ts_x, "_relu_pre", None)   # x = relu(pre) from dense_relu_

    def grad_fn_x(grad, out=None, accumulate=False):
        fuse_mask = pre is not None and out is None and pre.dtype == grad.dtype and (
            FUSE_RELU_BWD or not be.use_tensor_cores(grad.shape[0], w.shape[0], w.shape[1], grad.dtype))
        if fuse_mask:
            # x came out of a ReLU: the dX launch also applies that ReLU's mask and leaves the masked
            # gradient (with its tf32 planes) on the side for the ReLU node, which then has no
            # kernel of its own to run.  dX itself (dL/dx, unmasked) is returned as always.
            dx, masked = be.matmul(grad, w, tb=True, reuse_a=ts_w.requires_grad, act=True, mask_src=pre)
            dx.aux = (pre, masked)
            return dx
        return be.matmul(grad, w, tb=True, out=out, accumulate=accumulate,
                         reuse_a=ts_w.requires_grad)

    def grad_fn_w(grad, out=None, accumulate=False):
        return be.matmul(x, grad, ta=True, out=out, accumulate=accumulate,
                         reuse_b=ts_x.requires_grad)

    def grad_fn_b(grad, out=None, accumulate=False):
        if out is not None and not accumulate:
            return be.colsum(grad, out=out)
        s = be.colsum(grad)
        return be.add_inplace(out, s) if out is not None else s

    def fused_bwd(grad, direct):
        """All three gradients from ONE grouped launch when the layer is small (MNIST-sized: a launch
        costs more than the arithmetic).  `direct` maps id(tensor) -> (arena slot, accumulate) for the
        leaves the kernel may write in place; returns {id(tensor): gradient or WRITTEN_IN_PLACE}, or
        None when this node should go through the per-input functions instead."""
        b = ts_b._data
        if not (ts_w.requires_grad and ts_b.requires_grad and id(ts_w) in direct and id(ts_b) in direct):
            return None
        if ts_w is ts_b or not (grad.dtype == x.dtype == w.dtype == b.dtype) or grad.ndim != 2:
            return None
        if not be.dense_bwd_grouped_ok(grad.shape[0], w.shape[0], w.shape[1], grad.dtype):
            return None
        mask = pre if (pre is not None and pre.dtype == grad.dtype) else None
        (w_slot, w_acc), (b_slot, b_acc) = direct[id(ts_w)], direct[id(ts_b)]
        dx, masked = be.dense_bwd_grouped(grad, x, w, mask, ts_x.requires_grad, w_slot, w_acc, b_slot, b_acc)
        out = {id(ts_w): WRITTEN_IN_PLACE, id(ts_b): WRITTEN_IN_PLACE}
        if ts_x.requires_grad:
            if masked is not None:
                dx.aux = (pre, masked)
            out[id(ts_x)] = dx
        return out

    grad_fn_x.supports_out = grad_fn_w.supports_out = grad_fn_b.supports_out = True
    dependency = []
    requires_grad = (ts_x.requires_grad or ts_w.requires_grad or ts_b.requires_grad) and _GRAD_ENABLED
    for t, fn in ((ts_x, grad_fn_x), (ts_w, grad_fn_w), (ts_b, grad_fn_b)):
        if t.requires_grad and requires_grad:
            dependency.append(dict(tensor=t, grad_fn=fn))
    node = ts_x.__class__(values, requires_grad, dependency)
    if requires_grad and GROUP_SMALL_DENSE_BWD and ts_x is not ts_w and ts_x is not ts_b:
        node._fused_bwd = fused_bwd
    return node


def dense_relu_(ts_x, ts_w, ts_b):
    """Dense followed by ReLU (layers.py:49 then layers.py:97-98) computed by ONE GEMM launch whose
    epilogue writes both the pre-activation z = x@w+b and a = clip(z, 0).  The graph is the same two
    nodes the unfused layers build (z depends on x, w, b; a depends on z with the x >= 0 mask), so
    gradients, non-leaf .grad and Activation.inputs are unchanged.  Returns (z, a)."""
    x, w, b = ts_x._data, ts_w._data, ts_b._data
    if b.shape != (1, w.shape[1]) or x.dtype != w.dtype or b.dtype != w.dtype:
        z = ts_x @ ts_w + ts_b
        return z, relu_(z)
    zv, av = be.matmul(x, w, bias=b, reuse_a=ts_w.requires_grad, reuse_b=ts_x.requires_grad, act=True)
    ts_z = _dense_node(ts_x, ts_w, ts_b, zv)

    def relu_grad(grad):
        aux = grad.aux
        if aux is not None and aux[0] is zv:
            return aux[1]            # already masked by the dX epilogue that produced `grad`
        return be.relu_bwd(grad, zv)

    ts_a = build_unary_ops_tensor(ts_z, relu_grad, av)
    ts_a._relu_pre = zv
    return ts_z, ts_a


def im2col_(ts, KH, KW, stride, pads, out_hw):
    """NHWC x (N, H, W, C) -> col (N*OH*OW, KH*KW*C): row (n, oh, ow) holds the window of output pixel
    (oh, ow), columns in (kh, kw, c) order, zeros where the window reaches into the padding.  `pads` is
    the padding before the first row and column.  Backward is the adjoint (tnn_col2im, a gather)."""
    x = ts._data
    geom = (KH, KW, stride[0], stride[1], pads[0], pads[1], out_hw[0], out_hw[1])
    values = be.im2col(x, geom)

    def grad_fn(grad):
        if grad.dtype != x.dtype:
            grad = be.astype(grad, x.dtype)
        return be.col2im(grad, x.shape, geom)

    return build_unary_ops_tensor(ts, grad_fn, values)


def maxpool2d_(ts, pool, stride, pads, out_hw):
    """NHWC window maxima; the selected element of each window (the first maximum in row-major window
    order, or the first NaN) is kept as an int32 offset for backward, which hands each output's
    gradient wholly to it (summed where windows overlap)."""
    x = ts._data
    geom = (pool[0], pool[1], stride[0], stride[1], pads[0], pads[1], out_hw[0], out_hw[1])
    values, arg = be.maxpool_fwd(x, geom)

    def grad_fn(grad):
        if grad.dtype != x.dtype:
            grad = be.astype(grad, x.dtype)
        return be.maxpool_bwd(grad, arg, x.shape, geom)

    return build_unary_ops_tensor(ts, grad_fn, values)


def batchnorm_(ts_x, ts_gamma, ts_beta, layer_state, training):
    """Batch normalisation of x (..., C) over every axis but the last, viewed as (M, C):

        y = (x - mean) * gamma / sqrt(var + eps) + beta

    `layer_state` carries `buffers` (running_mean, running_var: (1, C) tensors without gradients),
    `momentum` and `epsilon` -- the BatchNormalization layer.  TRAIN (`training`): mean and the biased
    variance of this batch (of the global batch under data parallelism), and the running statistics
    are updated in place, running = (1 - momentum) * running + momentum * batch value with the
    unbiased variance.  TEST: the running statistics, left unchanged.  Two launches forward (TRAIN;
    one in TEST), two backward.

    The node depends on x, gamma and beta and keeps x and mr -- the per-column mean, r = 1/sqrt(var +
    eps) and row count -- for backward, which recomputes xhat = (x - mean) * r from them: dbeta =
    sum dy, dgamma = sum dy * xhat (one reduction whose fold writes them straight into the arena slots
    through _fused_bwd), dx = gamma * r * (dy - sum dy / M - xhat * sum(dy * xhat) / M), or gamma * r * dy
    in TEST.  Under data parallelism the two sums are all-reduced before dx, and the slots receive this
    rank's partials: Model.step's gradient all-reduce completes them."""
    import core._dist as dist
    x = ts_x._data
    shape = x.shape
    C = shape[-1]
    M = x.size // C
    x2 = x.view((M, C))
    gamma, beta = ts_gamma._data, ts_beta._data
    rm, rv = layer_state.buffers["running_mean"], layer_state.buffers["running_var"]
    eps = layer_state.epsilon
    world = dist.world_size()
    if training:
        if world > 1:
            mr = dist.bn_global_stats(x2, layer_state.momentum, eps, rm._data, rv._data)
        else:
            mr = be.bn_stats(x2, layer_state.momentum, eps, rm._data, rv._data)
        rm._touch()
        rv._touch()
        values, _ = be.bn_apply(x2, gamma, beta, mr=mr)
    else:
        values, mr = be.bn_apply(x2, gamma, beta, running=(rm._data, rv._data), eps=eps)
    values = values.view(shape)
    cache = {}

    def _as_x(grad):
        if grad.dtype != x.dtype:
            grad = be.astype(grad, x.dtype)
        return grad.view((M, C))

    def _sums(grad, dgamma=None, acc_gamma=False, dbeta=None, acc_beta=False):
        sums = be.bn_bwd_reduce(_as_x(grad), x2, mr, dgamma, acc_gamma, dbeta, acc_beta)
        if training and world > 1:
            dist.allreduce_sum(sums)     # after the local partials went to dgamma / dbeta
        return sums

    def _dx(grad, sums):
        return be.bn_dx(_as_x(grad), x2, mr, gamma, sums if training else None).view(shape)

    def _param_grads(grad):
        """(dgamma, dbeta, sums) from one reduction shared by the per-input functions below"""
        if cache.get("grad") is not grad:
            dg, db = be.empty((1, C), x.dtype), be.empty((1, C), x.dtype)
            cache.update(grad=grad, dg=dg, db=db, sums=_sums(grad, dg, False, db, False))
        return cache

    def grad_fn_x(grad):
        return _dx(grad, _param_grads(grad)["sums"] if training else None)

    def grad_fn_gamma(grad):
        return _param_grads(grad)["dg"]

    def grad_fn_beta(grad):
        return _param_grads(grad)["db"]

    def fused_bwd(grad, direct):
        """dgamma and dbeta written (or added) into their arena slots by the reduction's fold"""
        if ts_gamma is ts_beta or id(ts_gamma) not in direct or id(ts_beta) not in direct:
            return None
        (g_slot, g_acc), (b_slot, b_acc) = direct[id(ts_gamma)], direct[id(ts_beta)]
        sums = _sums(grad, g_slot, g_acc, b_slot, b_acc)
        out = {id(ts_gamma): WRITTEN_IN_PLACE, id(ts_beta): WRITTEN_IN_PLACE}
        if ts_x.requires_grad:
            out[id(ts_x)] = _dx(grad, sums)
        return out

    dependency = []
    requires_grad = (ts_x.requires_grad or ts_gamma.requires_grad or ts_beta.requires_grad) and _GRAD_ENABLED
    for t, fn in ((ts_x, grad_fn_x), (ts_gamma, grad_fn_gamma), (ts_beta, grad_fn_beta)):
        if t.requires_grad and requires_grad:
            dependency.append(dict(tensor=t, grad_fn=fn))
    node = ts_x.__class__(values, requires_grad, dependency)
    if requires_grad and ts_gamma.requires_grad and ts_beta.requires_grad:
        node._fused_bwd = fused_bwd
    return node


def softmax_ce_(ts_logits, ts_labels):
    """SoftmaxCrossEntropyLoss.loss of losses.py:24-32 as one node, reproducing its batch-global
    max and normaliser (SURVEY 0.4): M = max(z), S = sum_all exp(z - M), q_i = sum_j p_ij y_ij,
    L = -(1/m) sum_i ln q_i;  dL/dz = p - y p / (m q_i).

    Under data parallelism (core/_dist.py) the (M, S) pair is all-gathered and merged so the
    normaliser spans the global batch, m is the global batch size, and the returned loss is the
    all-reduced global value."""
    import core._dist as dist
    z, y = ts_logits._data, ts_labels._data
    B, C = z.shape
    world = dist.world_size()
    m_global = B * world
    dz_seed1 = None
    if world == 1 and be.ce_small_ok(B, C):
        # one launch instead of three; it also leaves dL/dz for backward()'s default seed
        stats, loss, q, dz_seed1 = be.ce_fwd_small(z, y, m_global,
                                                   want_dz=ts_logits.requires_grad and _GRAD_ENABLED)
    else:
        stats = be.ce_stats(z)
        if world > 1:
            stats = dist.merge_ce_stats(stats)
        loss, q = be.ce_loss(z, y, stats, m_global)
        if world > 1:
            dist.allreduce_sum(loss)

    def grad_fn(grad):
        if dz_seed1 is not None and be.is_ones_scalar(grad):
            return dz_seed1              # bit-identical to ce_bwd with g = 1, no launch
        return be.ce_bwd(z, y, stats, q, m_global, grad)

    return build_unary_ops_tensor(ts_logits, grad_fn, loss)


def pointwise_loss_(ts_pred, ts_target, kind, delta=1.0):
    """MSELoss / MAELoss / HuberLoss / SigmoidCrossEntropyLoss (core/losses.py) as one node:
    L = (1/m) sum over every element of l(p, t), m = pred.shape[0] rows of the global batch, `kind` one
    of be.LOSS_*.  The forward launch also writes dL/dp for backward()'s default seed, so the loss's
    forward and backward together are one launch; any other upstream gradient takes a second one.
    The gradient flows to the prediction only (the caller refuses a target that requires one).

    Under data parallelism m is the global batch (equal shards, the cross-entropy's convention), so
    1/m_global is inside dL/dp and Model.step's SUM all-reduce of the gradients completes them; the
    returned loss is the all-reduced global value."""
    import core._dist as dist
    p, t = ts_pred._data, ts_target._data
    world = dist.world_size()
    m_global = p.shape[0] * world
    loss, dp_seed1 = be.pointwise_loss(p, t, kind, m_global, delta,
                                       want_dp=ts_pred.requires_grad and _GRAD_ENABLED)
    if world > 1:
        dist.allreduce_sum(loss)

    def grad_fn(grad):
        if dp_seed1 is not None and be.is_ones_scalar(grad):
            return dp_seed1              # bit-identical to pointwise_loss_bwd with g = 1, no launch
        return be.pointwise_loss_bwd(p, t, kind, m_global, delta, grad)

    return build_unary_ops_tensor(ts_pred, grad_fn, loss)


# ------------------------------------------------------------------------------ coercing wrappers
def max(obj, axis=None):
    return max_(as_tensor(obj), axis=axis)


def maximum(obj1, obj2):
    return maximum_(as_tensor(obj1), as_tensor(obj2))


def minimum(obj1, obj2):
    return minimum_(as_tensor(obj1), as_tensor(obj2))


def exp(obj):
    return exp_(as_tensor(obj))


def sum(obj, axis=None):
    return sum_(as_tensor(obj), axis=axis)


def log(obj):
    return log_(as_tensor(obj))


def reshape(obj, newshape):
    return reshape_(as_tensor(obj), newshape)


def pad(obj, pad_width, mode="constant"):
    return pad_(as_tensor(obj), pad_width, mode=mode)


def flatten(obj):
    return flatten_(as_tensor(obj))


def clip(obj, min=None, max=None):
    return clip_(as_tensor(obj), min, max)
