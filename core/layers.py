"""Layers (interface of the reference's core/layers.py: Layer, Dense, Activation, Sigmoid, Tanh,
ReLU; `params` dicts, `inputs` bookkeeping, lazy Dense initialisation), plus the NHWC image layers
Conv2D, MaxPool2D and Flatten and the activations LeakyReLU, ELU, GELU, Softplus and SiLU of the
tinynn family.

Dense is one fused GEMM(+bias) node; together with a following ReLU it is one launch (see
core/nn.py).  ReLU, Sigmoid and Tanh are compositions of the op library, which routes `clip(x, 0.0)`
to the fused ReLU kernels; the other activations are one elementwise launch each way
(ops.activation_).  Conv2D is im2col + that same Dense node.
"""
import math

import numpy as np

import core._backend as be
import core.ops as ops
from core.initializer import ConstantInit
from core.initializer import XavierUniformInit
from core.initializer import ZerosInit
from core.tensor import Tensor


class Layer(object):
    """Base class: a name, a dict of parameter tensors, a dict of state tensors that are not
    parameters (`buffers`: saved and loaded with the parameters, never optimised) and the
    TRAIN/TEST flag."""

    def __init__(self, name):
        self.name = name
        self.params = {}
        self.buffers = {}
        self.grads = {}
        self.is_training = True

    def forward(self, inputs):
        raise NotImplementedError

    def __call__(self, inputs):
        return self.forward(inputs)

    def set_phase(self, phase):
        self.is_training = (phase == "TRAIN")


class Dense(Layer):
    """y = x @ w + b with w of shape (num_in, num_out) and b of shape (1, num_out), both float32
    device tensors.  num_in may be left out: it is then taken from the first input (layers.py:45-46),
    which also fixes WHEN the weights are drawn from numpy's global RNG."""

    def __init__(self, num_out, num_in=None, w_init=XavierUniformInit(), b_init=ZerosInit()):
        Layer.__init__(self, "Linear")
        self.initializers = {"w": w_init, "b": b_init}
        self.shapes = {"w": [num_in, num_out], "b": [1, num_out]}
        self.params = {"w": None, "b": None}
        self.inputs = None
        self.is_init = False
        if num_in is not None:
            self._init_parameters(num_in)

    def _init_parameters(self, input_size):
        self.shapes["w"][0] = input_size
        for key in ("w", "b"):          # draw order w, b: layers.py:53-56
            tensor = self.initializers[key](shape=self.shapes[key])
            tensor.zero_grad()
            self.params[key] = tensor
        self.is_init = True

    def _prepare(self, inputs):
        if not self.is_init:
            self._init_parameters(inputs.shape[1])
        self.inputs = inputs
        return self.params["w"], self.params["b"]

    def forward(self, inputs):
        w, b = self._prepare(inputs)
        return ops.dense_(inputs, w, b)

    def forward_fused_relu(self, inputs, relu_layer):
        """this layer followed by `relu_layer` in one GEMM launch; both record their inputs"""
        w, b = self._prepare(inputs)
        pre_activation, activated = ops.dense_relu_(inputs, w, b)
        relu_layer.inputs = pre_activation
        return activated


def _pair(v, what):
    """an int or a pair of ints -> (rows, columns), both >= 1"""
    pair = (v, v) if isinstance(v, (int, np.integer)) else tuple(v)
    if len(pair) != 2 or not all(isinstance(p, (int, np.integer)) and p >= 1 for p in pair):
        raise ValueError("%s must be a positive int or a pair of them, got %r" % (what, v))
    return int(pair[0]), int(pair[1])


def _check_padding(padding):
    if padding not in ("SAME", "VALID"):
        raise ValueError("padding must be 'SAME' or 'VALID', got %r" % (padding,))
    return padding


def window_geometry(in_hw, window_hw, stride_hw, padding):
    """Output extent and leading padding of a sliding window over an (H, W) image, per dimension:

      "VALID": no padding, O = (I - K) // S + 1; a ValueError if I < K.
      "SAME":  K - 1 padded positions in total, (K - 1) // 2 before the first row / column and the rest
               after it (an even window pads one more after than before), O = ceil(I / S).

    Returns ((OH, OW), (PH0, PW0)).  Used by Conv2D and MaxPool2D."""
    _check_padding(padding)
    out, before = [], []
    for i, k, s in zip(in_hw, window_hw, stride_hw):
        if padding == "VALID":
            if i < k:
                raise ValueError("VALID padding: input extent %d is smaller than the window %d" % (i, k))
            out.append((i - k) // s + 1)
            before.append(0)
        else:
            out.append(-(-i // s))
            before.append((k - 1) // 2)
    return tuple(out), tuple(before)


def _check_nhwc(layer, inputs, channels=None):
    shape = tuple(inputs.shape)
    if len(shape) != 4 or (channels is not None and shape[3] != channels):
        want = "(N, H, W, %d)" % channels if channels is not None else "(N, H, W, C)"
        raise ValueError("%s: input of shape %s does not match %s" % (layer, shape, want))
    return shape


class Conv2D(Layer):
    """2-D convolution over NHWC float32 / float64 inputs:

        y[n, oh, ow, o] = b[o] + sum_{kh, kw, c} xpad[n, oh*SH + kh, ow*SW + kw, c] * w[kh, kw, c, o]

    kernel = (KH, KW, C_in, C_out); params["w"] has that shape and params["b"] is (1, C_out), as for
    Dense; both are drawn at construction, w then b, by calling the initialisers with those shapes.
    stride is an int or an (SH, SW) pair.  padding is "SAME" or "VALID" (see window_geometry: SAME
    pads K - 1 positions per dimension, (K - 1) // 2 of them before, and gives ceil(I / S) outputs).
    An input that is not 4-D or whose channel count is not C_in is a ValueError.

    The layer is a composition of existing nodes: im2col_ lays the windows out as rows of a
    (N*OH*OW, KH*KW*C_in) matrix, which is multiplied by w viewed as (KH*KW*C_in, C_out) through the
    Dense node (bias in the GEMM epilogue, the usual tensor-core / SIMT routing), and the product is
    viewed as (N, OH, OW, C_out).  The col matrix lives until backward, as a Dense input does."""

    def __init__(self, kernel, stride=(1, 1), padding="SAME", w_init=XavierUniformInit(), b_init=ZerosInit()):
        Layer.__init__(self, "Conv2D")
        kernel = tuple(kernel)
        if len(kernel) != 4 or not all(isinstance(k, (int, np.integer)) and k >= 1 for k in kernel):
            raise ValueError("kernel must be (KH, KW, C_in, C_out) positive ints, got %r" % (kernel,))
        self.kernel = tuple(int(k) for k in kernel)
        self.stride = _pair(stride, "stride")
        self.padding = _check_padding(padding)
        self.initializers = {"w": w_init, "b": b_init}
        shapes = {"w": list(self.kernel), "b": [1, self.kernel[3]]}
        for key in ("w", "b"):
            tensor = self.initializers[key](shape=shapes[key])
            tensor.zero_grad()
            self.params[key] = tensor
        self.inputs = None

    def forward(self, inputs):
        KH, KW, C, O = self.kernel
        N, H, W, _ = _check_nhwc("Conv2D", inputs, C)
        out_hw, pads = window_geometry((H, W), (KH, KW), self.stride, self.padding)
        self.inputs = inputs
        col = ops.im2col_(inputs, KH, KW, self.stride, pads, out_hw)
        w2 = ops.reshape_(self.params["w"], (KH * KW * C, O))
        z = ops.dense_(col, w2, self.params["b"])
        return ops.reshape_(z, (N, out_hw[0], out_hw[1], O))


class MaxPool2D(Layer):
    """Window maxima over NHWC inputs.  stride=None means stride = pool_size; padding as Conv2D's
    (window_geometry), and padded positions are never selected (SAME leaves at least one real element
    in every window).  The selected element is the first maximum in row-major window order -- np.argmax
    over the flattened window -- or the first NaN, which makes the output NaN, as np.max does.  Each
    output's gradient goes wholly to its selected input; where windows overlap (stride < pool_size)
    the contributions are summed.  (Unlike the reference's max_, tied elements do not all receive it.)"""

    def __init__(self, pool_size=(2, 2), stride=None, padding="VALID"):
        Layer.__init__(self, "MaxPool2D")
        self.pool_size = _pair(pool_size, "pool_size")
        self.stride = self.pool_size if stride is None else _pair(stride, "stride")
        self.padding = _check_padding(padding)
        self.inputs = None

    def forward(self, inputs):
        N, H, W, C = _check_nhwc("MaxPool2D", inputs)
        out_hw, pads = window_geometry((H, W), self.pool_size, self.stride, self.padding)
        self.inputs = inputs
        return ops.maxpool2d_(inputs, self.pool_size, self.stride, pads, out_hw)


class BatchNormalization(Layer):
    """Batch normalisation over every axis but the last: a (N, C) Dense output or an (N, H, W, C)
    NHWC Conv2D output is normalised per channel over its N (or N*H*W) rows M,

        y = (x - mean) * gamma / sqrt(var + epsilon) + beta

    params["gamma"] and params["beta"] are (1, C), drawn at construction in that order through the
    initialisers.  layer.buffers holds the running statistics, running_mean (starts at 0) and
    running_var (starts at 1): (1, C) device tensors of the parameters' dtype without gradients, not
    parameters (the optimiser does not see them), saved and loaded with them by Model.save / load.

    TRAIN phase: mean and the biased variance of the batch (of the global batch under data
    parallelism), and running = (1 - momentum) * running + momentum * batch value with the unbiased
    variance (* M / (M - 1)) -- the torch conventions.  The phase decides, not the grad mode: a
    forward under no_grad() in TRAIN also updates them.  M < 2 is a ValueError there.
    TEST phase: the running statistics, unchanged; gradients still flow.  An empty batch is allowed.

    The input must be 2-D or 4-D with a last axis of num_features and share gamma's dtype (float32
    or float64); anything else is a ValueError.  momentum and epsilon are fixed at construction."""

    def __init__(self, num_features, momentum=0.1, epsilon=1e-5, gamma_init=ConstantInit(1.0),
                 beta_init=ZerosInit()):
        Layer.__init__(self, "BatchNormalization")
        if not isinstance(num_features, (int, np.integer)) or num_features < 1:
            raise ValueError("num_features must be a positive int, got %r" % (num_features,))
        self.num_features = int(num_features)
        self.momentum = float(momentum)
        self.epsilon = float(epsilon)
        self.initializers = {"gamma": gamma_init, "beta": beta_init}
        for key in ("gamma", "beta"):
            tensor = self.initializers[key](shape=[1, self.num_features])
            tensor.zero_grad()
            self.params[key] = tensor
        dt = self.params["gamma"].dtype
        self.buffers = {"running_mean": Tensor(np.zeros((1, self.num_features), dt), dtype=dt),
                        "running_var": Tensor(np.ones((1, self.num_features), dt), dtype=dt)}
        self.inputs = None

    def _check(self, inputs):
        shape = tuple(inputs.shape)
        if len(shape) not in (2, 4) or shape[-1] != self.num_features:
            raise ValueError("BatchNormalization: input of shape %s does not match (N, %d) or (N, H, W, %d)"
                             % (shape, self.num_features, self.num_features))
        dt = self.params["gamma"].dtype
        if inputs.dtype != dt or self.params["beta"].dtype != dt:
            raise ValueError("BatchNormalization: input dtype %s and gamma / beta dtype %s / %s differ"
                             % (inputs.dtype, dt, self.params["beta"].dtype))
        rows = int(np.prod(shape[:-1], dtype=np.int64))
        if self.is_training and rows < 2:
            raise ValueError("BatchNormalization: TRAIN phase needs at least 2 values per channel, got %d "
                             "(input of shape %s)" % (rows, shape))

    def forward(self, inputs):
        self._check(inputs)
        dt = self.params["gamma"].dtype
        for buf in self.buffers.values():
            if buf.dtype != dt:          # gamma / beta were replaced by tensors of another dtype
                buf.values = np.asarray(buf.values, dt)
        self.inputs = inputs
        return ops.batchnorm_(inputs, self.params["gamma"], self.params["beta"], self, self.is_training)


class Flatten(Layer):
    """(N, ...) -> (N, prod(...)), a view (no kernel)"""

    def __init__(self):
        Layer.__init__(self, "Flatten")
        self.inputs = None

    def forward(self, inputs):
        self.inputs = inputs
        shape = tuple(inputs.shape)
        return ops.reshape_(inputs, (shape[0], int(np.prod(shape[1:], dtype=np.int64))))


class Activation(Layer):

    def __init__(self, name):
        Layer.__init__(self, name)
        self.inputs = None

    def forward(self, inputs):
        self.inputs = inputs
        return self.func(inputs)

    def func(self, x):
        raise NotImplementedError


class ReLU(Activation):
    """clip(x, 0.0): the backward mask is x >= 0, so ReLU'(0) = 1 (layers.py:97-98, ops.py:336-343)"""

    def __init__(self):
        Activation.__init__(self, "ReLU")

    def func(self, x):
        return ops.clip(x, 0.0)


class Tanh(Activation):
    """(1 - e^-x) / (1 + e^-x), which is tanh(x / 2) -- the formula at layers.py:88-89"""

    def __init__(self):
        Activation.__init__(self, "Tanh")

    def func(self, x):
        decay = ops.exp(-x)
        return (1.0 - decay) / (1.0 + decay)


class Sigmoid(Activation):
    """1 / (1 + e^-x).  The reference's version calls np.exp on a Tensor and raises
    (layers.py:79-80); no test pins that, so this one works."""

    def __init__(self):
        Activation.__init__(self, "Sigmoid")

    def func(self, x):
        return 1.0 / (1.0 + ops.exp(-x))


# ---------------------------------------------------------------------------- elementwise activations
# Conventions shared by LeakyReLU, ELU, GELU, Softplus and SiLU (include/tnn_b200.h states them
# beside the op codes):
#   - the kink at 0 goes to the x >= 0 branch, as ReLU's (ReLU'(0) = 1), so LeakyReLU(0.0) equals
#     ReLU in value and gradient on non-NaN inputs (torch gives slope / alpha there instead);
#   - NaN in x gives NaN in y and in dx; +-inf give the function's limit and the derivative's limit;
#   - every finite x gives a finite y and dx;
#   - the computation is in the input's dtype (float32 or float64);
#   - slope / alpha / approximate are fixed at construction (read-only properties): a recorded
#     training step bakes them into its kernel arguments.
# Each layer is one node, ops.activation_: one launch forward, one backward.

def _finite_number(layer, what, value):
    if isinstance(value, (bool, np.bool_)) or not isinstance(value, (int, float, np.integer, np.floating)):
        raise ValueError("%s: %s must be a number, got %r" % (layer, what, value))
    value = float(value)
    if not math.isfinite(value):
        raise ValueError("%s: %s must be finite, got %r" % (layer, what, value))
    return value


class LeakyReLU(Activation):
    """y = x if x >= 0 else slope * x;  dy/dx = 1 if x >= 0 else slope.

    slope (default 0.01) is any finite number, fixed at construction.  The kink at 0 goes to the
    x >= 0 branch, so LeakyReLU(0.0) is ReLU on non-NaN inputs; LeakyReLU(-inf) is 0 when slope = 0.
    NaN gives NaN in y and dx."""

    def __init__(self, slope=0.01):
        Activation.__init__(self, "LeakyReLU")
        self._slope = _finite_number("LeakyReLU", "slope", slope)

    @property
    def slope(self):
        return self._slope

    def func(self, x):
        return ops.activation_(ops.as_tensor(x), be.LEAKY_RELU, be.LEAKY_RELU_BWD, self._slope)


class ELU(Activation):
    """y = x if x >= 0 else alpha * expm1(x);  dy/dx = 1 if x >= 0 else alpha * exp(x).

    alpha (default 1.0) is any finite number, fixed at construction.  dy/dx(0) = 1 (the x >= 0
    branch); ELU(-inf) = -alpha with gradient 0.  NaN gives NaN in y and dx."""

    def __init__(self, alpha=1.0):
        Activation.__init__(self, "ELU")
        self._alpha = _finite_number("ELU", "alpha", alpha)

    @property
    def alpha(self):
        return self._alpha

    def func(self, x):
        return ops.activation_(ops.as_tensor(x), be.ELU, be.ELU_BWD, self._alpha)


class GELU(Activation):
    """approximate="none" (default): y = x * Phi(x), Phi(x) = erfc(-x / sqrt 2) / 2, the normal CDF;
        dy/dx = Phi(x) + x * phi(x), phi(x) = exp(-x^2 / 2) / sqrt(2 pi).
    approximate="tanh": y = x * s, s = sigma(2u) (= (1 + tanh u) / 2), u = sqrt(2/pi) (x + 0.044715 x^3);
        dy/dx = s + 2x * s(1 - s) * sqrt(2/pi) (1 + 0.134145 x^2), s(1 - s) as sigma(2u) sigma(-2u).

    sigma is the logistic function evaluated without overflow.  GELU(-inf) = 0, GELU(+inf) = +inf,
    with gradients 0 and 1; in float32 the tanh form's x^3 and x^2 overflow for large finite |x|,
    and the value and gradient there are still finite (x and 1, or 0 and 0).  NaN gives NaN.
    approximate is "none" or "tanh", fixed at construction."""

    def __init__(self, approximate="none"):
        Activation.__init__(self, "GELU")
        if not isinstance(approximate, str) or approximate not in ("none", "tanh"):
            raise ValueError("GELU: approximate must be 'none' or 'tanh', got %r" % (approximate,))
        self._approximate = approximate

    @property
    def approximate(self):
        return self._approximate

    def func(self, x):
        if self._approximate == "tanh":
            return ops.activation_(ops.as_tensor(x), be.GELU_TANH, be.GELU_TANH_BWD)
        return ops.activation_(ops.as_tensor(x), be.GELU, be.GELU_BWD)


class Softplus(Activation):
    """y = max(x, 0) + log1p(exp(-|x|)) (= log(1 + e^x) without overflow);  dy/dx = sigma(x).

    Softplus(-inf) = 0, Softplus(+inf) = +inf, with gradients 0 and 1.  NaN gives NaN."""

    def __init__(self):
        Activation.__init__(self, "Softplus")

    def func(self, x):
        return ops.activation_(ops.as_tensor(x), be.SOFTPLUS, be.SOFTPLUS_BWD)


class SiLU(Activation):
    """y = x * sigma(x);  dy/dx = sigma(x) (1 + x (1 - sigma(x))), x (1 - sigma(x)) sigma(x) as
    x sigma(x) sigma(-x).  sigma is the logistic function evaluated without overflow.

    SiLU(-inf) = 0, SiLU(+inf) = +inf, with gradients 0 and 1.  NaN gives NaN."""

    def __init__(self):
        Activation.__init__(self, "SiLU")

    def func(self, x):
        return ops.activation_(ops.as_tensor(x), be.SILU, be.SILU_BWD)
