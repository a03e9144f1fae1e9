"""CPU oracle for the NHWC image layers: float64 numpy conv2d and maxpool2d as RefTensor nodes, so a
whole CNN step (with ref_numpy's matmul / clip / reshape, softmax_cross_entropy and RefAdam) runs in
the oracle.

TEST INFRASTRUCTURE ONLY (same rules as oracle/ref_numpy.py: imported by tests/ and scripts only).
The reference has no convolution; the semantics restated here are the ones core/layers.py documents
for Conv2D / MaxPool2D (NHWC; SAME pads K - 1 positions per dimension, (K - 1) // 2 before; pooling
selects np.argmax of the real elements of each flattened window).  tests/test_conv_host.py pins this
module against torch's conv2d / max_pool2d on the CPU.
"""
import numpy as np

from ref_numpy import _node


def geometry(size, k, s, padding):
    """(output extent, padding before, padding after) of one spatial dimension"""
    if padding == "VALID":
        if size < k:
            raise ValueError("VALID: input %d smaller than window %d" % (size, k))
        return (size - k) // s + 1, 0, 0
    if padding == "SAME":
        out = -(-size // s)
        return out, (k - 1) // 2, k - 1 - (k - 1) // 2
    raise ValueError(padding)


def _windows(xp, KH, KW, SH, SW, OH, OW):
    """xp (N, Hp, Wp, C) -> (N, OH, OW, KH, KW, C) view-copy of every window"""
    N, _, _, C = xp.shape
    out = np.empty((N, OH, OW, KH, KW, C), xp.dtype)
    for kh in range(KH):
        for kw in range(KW):
            out[:, :, :, kh, kw, :] = xp[:, kh:kh + SH * (OH - 1) + 1:SH, kw:kw + SW * (OW - 1) + 1:SW, :]
    return out


def _scatter_windows(dwin, shape_p, SH, SW):
    """adjoint of _windows: (N, OH, OW, KH, KW, C) -> (N, Hp, Wp, C), overlapping windows summed"""
    N, OH, OW, KH, KW, C = dwin.shape
    out = np.zeros(shape_p, dwin.dtype)
    for kh in range(KH):
        for kw in range(KW):
            out[:, kh:kh + SH * (OH - 1) + 1:SH, kw:kw + SW * (OW - 1) + 1:SW, :] += dwin[:, :, :, kh, kw, :]
    return out


def conv2d(x, w, b, stride=(1, 1), padding="SAME"):
    """x (N, H, W, C), w (KH, KW, C, O), b (1, O) RefTensors -> (N, OH, OW, O), in float64"""
    xv = np.asarray(x.values, np.float64)
    wv = np.asarray(w.values, np.float64)
    bv = np.asarray(b.values, np.float64)
    N, H, W, C = xv.shape
    KH, KW, _, O = wv.shape
    SH, SW = stride
    OH, ph0, ph1 = geometry(H, KH, SH, padding)
    OW, pw0, pw1 = geometry(W, KW, SW, padding)
    pad = ((0, 0), (ph0, ph1), (pw0, pw1), (0, 0))
    xp = np.pad(xv, pad)
    col = _windows(xp, KH, KW, SH, SW, OH, OW).reshape(N * OH * OW, KH * KW * C)
    w2 = wv.reshape(KH * KW * C, O)
    y = (col @ w2 + bv).reshape(N, OH, OW, O)

    def vjp_x(g):
        dcol = g.reshape(N * OH * OW, O) @ w2.T
        dxp = _scatter_windows(dcol.reshape(N, OH, OW, KH, KW, C), xp.shape, SH, SW)
        return dxp[:, ph0:ph0 + H, pw0:pw0 + W, :]

    def vjp_w(g):
        return (col.T @ g.reshape(N * OH * OW, O)).reshape(KH, KW, C, O)

    def vjp_b(g):
        return g.reshape(N * OH * OW, O).sum(axis=0, keepdims=True)

    return _node(y, [(x, vjp_x), (w, vjp_w), (b, vjp_b)])


def maxpool2d(x, pool=(2, 2), stride=None, padding="VALID"):
    """x (N, H, W, C) RefTensor -> (N, OH, OW, C) window maxima over the real elements; the selected
    element is np.argmax of the flattened window (first maximum, or first NaN) and receives the
    whole gradient, summed where windows overlap"""
    xv = np.asarray(x.values, np.float64)
    N, H, W, C = xv.shape
    PH, PW = pool
    SH, SW = pool if stride is None else stride
    OH, ph0, ph1 = geometry(H, PH, SH, padding)
    OW, pw0, pw1 = geometry(W, PW, SW, padding)
    pad = ((0, 0), (ph0, ph1), (pw0, pw1), (0, 0))
    win = _windows(np.pad(xv, pad, constant_values=-np.inf), PH, PW, SH, SW, OH, OW)
    valid = _windows(np.pad(np.ones((1, H, W, 1), bool), pad), PH, PW, SH, SW, OH, OW)
    win = win.reshape(N, OH, OW, PH * PW, C)
    valid = np.broadcast_to(valid.reshape(1, OH, OW, PH * PW, 1), win.shape)
    sel = np.argmax(win, axis=3)[:, :, :, None, :]
    # a padded position is only ever the argmax when every real element is -inf; the first real one wins
    first_real = np.argmax(valid, axis=3)[:, :, :, None, :]
    sel = np.where(np.take_along_axis(valid, sel, axis=3), sel, first_real)
    y = np.take_along_axis(win, sel, axis=3)[:, :, :, 0, :]
    onehot = np.arange(PH * PW)[None, None, None, :, None] == sel

    def vjp(g):
        dwin = (onehot * g[:, :, :, None, :]).reshape(N, OH, OW, PH, PW, C)
        dxp = _scatter_windows(dwin, (N, H + ph0 + ph1, W + pw0 + pw1, C), SH, SW)
        return dxp[:, ph0:ph0 + H, pw0:pw0 + W, :]

    return _node(y, [(x, vjp)])
