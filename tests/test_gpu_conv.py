"""Conv2D, MaxPool2D and Flatten on the device (csrc/conv.cu + the GEMM routes) against the float64
oracle of oracle/ref_conv.py: forward values and every gradient over a grid of kernels, strides,
paddings and channel counts in float32 and float64, the tensor-core route, the im2col / col2im
adjoint pair, the pooling edge cases, and a small MNIST CNN trained eagerly, through the recorded
train_step and through the recorded five-line loop."""
import os

import numpy as np
import pytest

import op_cases
import ref_conv as RC
import ref_fp32
import ref_numpy as R
from support import params

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    import core._backend as be
    be.init()
    return be


def _rel(a, b):
    return op_cases.rel_err(a, b)


def _conv_case(kernel, stride, padding, dtype, N, H, W, seed):
    """device Conv2D forward + backward with a random upstream gradient, and the oracle's"""
    from core.layers import Conv2D
    from core.tensor import Tensor
    rng = np.random.RandomState(seed)
    KH, KW, C, O = kernel
    x = rng.standard_normal((N, H, W, C)).astype(dtype)
    w = rng.standard_normal(kernel).astype(dtype)
    b = rng.standard_normal((1, O)).astype(dtype)
    layer = Conv2D(kernel, stride=stride, padding=padding)
    layer.params["w"] = Tensor(w, requires_grad=True, dtype=dtype)
    layer.params["b"] = Tensor(b, requires_grad=True, dtype=dtype)
    for p in layer.params.values():
        p.zero_grad()
    tx = Tensor(x, requires_grad=True, dtype=dtype)
    tx.zero_grad()
    y = layer.forward(tx)
    g = rng.standard_normal(y.shape).astype(dtype)
    y.backward(g)
    rx, rw, rb = R.RefTensor(x, True), R.RefTensor(w, True), R.RefTensor(b, True)
    ry = RC.conv2d(rx, rw, rb, stride, padding)
    ry.backward(g.astype(np.float64))
    got = dict(y=y.values, dx=tx.grad, dw=layer.params["w"].grad, db=layer.params["b"].grad)
    ref = dict(y=ry.values, dx=rx.grad, dw=rw.grad, db=rb.grad)
    return got, ref, y


# (C_in, batch): every channel count (scalar and 16-byte vector paths) and both batch sizes
CHANNELS_BATCH = [(1, 1), (3, 7), (8, 1), (64, 7)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("padding", ["SAME", "VALID"])
@pytest.mark.parametrize("stride", [1, 2, 3])
@pytest.mark.parametrize("khw", [(1, 1), (2, 2), (3, 3), (5, 5), (3, 1)])
def test_conv2d_matches_oracle(be, khw, stride, padding, dtype):
    """forward, dx, dw, db on the SIMT route (f32: rel 1e-5 of max|ref|; f64: 1e-12), 11 x 8 images"""
    tol = 1e-5 if dtype == np.float32 else 1e-12
    for C, N in CHANNELS_BATCH:
        kernel = (khw[0], khw[1], C, 5)
        got, ref, _ = _conv_case(kernel, (stride, stride), padding, dtype, N, 11, 8, seed=C * 31 + N)
        for k in ("y", "dx", "dw", "db"):
            assert got[k].shape == ref[k].shape, (k, C, N)
            assert got[k].dtype == dtype
            assert _rel(got[k], ref[k]) <= tol, (k, C, N, _rel(got[k], ref[k]))


def test_conv2d_rectangular_stride_and_shape_checks(be):
    """(SH, SW) = (2, 3) with a 4 x 2 kernel (asymmetric SAME padding); bad inputs raise"""
    from core.layers import Conv2D
    from core.tensor import Tensor
    got, ref, _ = _conv_case((4, 2, 3, 6), (2, 3), "SAME", np.float64, 3, 9, 13, seed=5)
    for k in ("y", "dx", "dw", "db"):
        assert _rel(got[k], ref[k]) <= 1e-12, k
    layer = Conv2D((3, 3, 4, 2))
    for shape in [(2, 8, 8, 3), (8, 8, 4), (1, 2, 8, 8, 4)]:
        with pytest.raises(ValueError, match=r"\(N, H, W, 4\)"):
            layer.forward(Tensor(np.zeros(shape, np.float32)))
    with pytest.raises(ValueError):
        Conv2D((5, 5, 1, 2), padding="VALID").forward(Tensor(np.zeros((1, 4, 9, 1), np.float32)))


def test_conv2d_tensor_core_route(be):
    """batch 8, 32 x 32 x 64 input, 3 x 3 x 64 x 128 SAME kernel: the forward, dW and dcol products
    all have M*N*K >= TC_MIN_MNK and run on the tcgen05 f16-split kernel"""
    M, K, O = 8 * 32 * 32, 3 * 3 * 64, 128
    for m, n, k in ((M, O, K), (K, O, M), (M, K, O)):
        assert be.use_tensor_cores(m, n, k, be.F32)
    got, ref, y = _conv_case((3, 3, 64, 128), (1, 1), "SAME", np.float32, 8, 32, 32, seed=11)
    col = y.dependency[0]["tensor"].dependency[0]["tensor"]        # reshape <- dense <- im2col
    assert col.shape == (M, K) and "f" in col._data.split           # planes of the f16 split route
    for k in ("y", "dx", "dw", "db"):
        assert _rel(got[k], ref[k]) <= 1e-5, (k, _rel(got[k], ref[k]))


@pytest.mark.parametrize("geom", [
    # (N, H, W, C, KH, KW, SH, SW, padding)
    (2, 9, 7, 3, 3, 3, 1, 1, "SAME"), (3, 10, 6, 8, 4, 2, 2, 3, "SAME"), (1, 12, 12, 64, 5, 5, 3, 2, "VALID"),
    (4, 7, 9, 2, 2, 3, 2, 1, "VALID"),
])
def test_im2col_col2im_adjoint_and_reproducible(be, geom):
    from core.layers import window_geometry
    N, H, W, C, KH, KW, SH, SW, padding = geom
    (OH, OW), (PH0, PW0) = window_geometry((H, W), (KH, KW), (SH, SW), padding)
    g_ = (KH, KW, SH, SW, PH0, PW0, OH, OW)
    rng = np.random.RandomState(H * W + C)
    x = rng.standard_normal((N, H, W, C))
    g = rng.standard_normal((N * OH * OW, KH * KW * C))
    dx_, dg = be.from_numpy(x), be.from_numpy(g)
    cols = [be.im2col(dx_, g_).numpy() for _ in range(2)]
    dxs = [be.col2im(dg, x.shape, g_).numpy() for _ in range(2)]
    lhs = float(np.sum(cols[0] * g))
    rhs = float(np.sum(x * dxs[0]))
    assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), np.sum(np.abs(cols[0] * g)))
    assert np.array_equal(cols[0], cols[1]) and np.array_equal(dxs[0], dxs[1])
    # and im2col equals the oracle's layout
    xp = np.pad(x, ((0, 0), (PH0, KH - 1 - PH0 if padding == "SAME" else 0),
                    (PW0, KW - 1 - PW0 if padding == "SAME" else 0), (0, 0)))
    assert np.array_equal(cols[0], RC._windows(xp, KH, KW, SH, SW, OH, OW).reshape(cols[0].shape))


def _pool_case(x, pool, stride, padding, g=None):
    from core.layers import MaxPool2D
    from core.tensor import Tensor
    dtype = x.dtype.type
    tx = Tensor(x, requires_grad=True, dtype=dtype)
    tx.zero_grad()
    y = MaxPool2D(pool, stride, padding).forward(tx)
    if g is None:
        g = np.random.RandomState(1).standard_normal(y.shape).astype(dtype)
    y.backward(g)
    rx = R.RefTensor(x, True)
    ry = RC.maxpool2d(rx, pool, stride, padding)
    ry.backward(np.asarray(g, np.float64))
    return y.values, tx.grad, ry.values, rx.grad


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("pool,stride,padding", [
    ((2, 2), None, "VALID"), ((3, 3), (2, 2), "VALID"), ((3, 3), (1, 1), "SAME"), ((2, 3), (1, 2), "SAME"),
])
@pytest.mark.parametrize("C", [3, 8])
def test_maxpool_matches_oracle(be, pool, stride, padding, dtype, C):
    """values exactly; gradients (sums over overlapping windows) to the last bits"""
    rng = np.random.RandomState(C)
    x = rng.standard_normal((3, 9, 10, C)).astype(dtype)
    y, dx, ry, rdx = _pool_case(x, pool, stride, padding)
    assert np.array_equal(y, ry.astype(dtype))
    tol = 1e-6 if dtype == np.float32 else 1e-14
    np.testing.assert_allclose(dx, rdx, rtol=tol, atol=tol)


def test_maxpool_ties_nan_inf_and_empty_batch(be):
    # constant input: every window hands its gradient to its first element
    x = np.full((2, 6, 6, 4), 0.5, np.float32)
    y, dx, ry, rdx = _pool_case(x, (3, 3), (2, 2), "VALID", g=np.ones((2, 2, 2, 4), np.float32))
    assert np.array_equal(dx, rdx)
    assert dx[0, 0, 0, 0] == 1.0 and dx[0, 2, 2, 0] == 1.0 and dx.sum() == 2 * 2 * 2 * 4
    # NaN and -inf: the first NaN of a window is selected and the output is NaN; an all -inf window
    # (also one reaching into SAME padding) selects its first real element
    rng = np.random.RandomState(3)
    for dtype in (np.float32, np.float64):
        x = rng.standard_normal((2, 7, 8, 4)).astype(dtype)
        x[0, 1, 1, 0] = x[0, 0, 1, 0] = np.nan
        x[1, 3:6, 2:5, :] = -np.inf
        x[0, :3, :3, 3] = -np.inf
        x[1, 6, 7, 2] = np.nan
        for pool, stride, padding in (((2, 2), None, "VALID"), ((3, 3), (1, 1), "SAME"), ((3, 3), (2, 2), "SAME")):
            y, dx, ry, rdx = _pool_case(x, pool, stride, padding)
            np.testing.assert_array_equal(y, ry.astype(dtype))            # NaN == NaN here
            tol = 1e-6 if dtype == np.float32 else 1e-14
            np.testing.assert_allclose(dx, rdx, rtol=tol, atol=tol)
            assert np.isnan(y).any()
    # a batch of 0
    y, dx, ry, rdx = _pool_case(np.zeros((0, 6, 6, 3), np.float32), (2, 2), None, "VALID")
    assert y.shape == (0, 3, 3, 3) and dx.shape == (0, 6, 6, 3)


def test_maxpool_backward_is_reproducible(be):
    from core.layers import window_geometry
    rng = np.random.RandomState(9)
    x = be.from_numpy(rng.standard_normal((4, 15, 13, 8)).astype(np.float32))
    (OH, OW), (PH0, PW0) = window_geometry((15, 13), (3, 3), (1, 2), "SAME")
    geom = (3, 3, 1, 2, PH0, PW0, OH, OW)
    y, arg = be.maxpool_fwd(x, geom)
    a = arg.numpy()
    assert a.dtype == np.int32 and a.min() >= 0 and a.max() < 9
    g = be.from_numpy(rng.standard_normal(y.shape).astype(np.float32))
    outs = [be.maxpool_bwd(g, arg, x.shape, geom).numpy() for _ in range(2)]
    assert np.array_equal(outs[0], outs[1])


# ---------------------------------------------------------------------------- small MNIST CNN
def _cnn(seed):
    from core.layers import Conv2D, Dense, Flatten, MaxPool2D, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    np.random.seed(seed)
    net = Net([Conv2D((5, 5, 1, 8), stride=2), ReLU(), MaxPool2D(), Conv2D((3, 3, 8, 16)), ReLU(), Flatten(),
               Dense(10, num_in=7 * 7 * 16)])
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))


def _data(n):
    x, _, onehot = ref_fp32.learnable_mnist(n, seed=0)
    return x.reshape(n, 28, 28, 1), onehot


class _RefCNN(object):
    """the same network in the float64 oracle, starting from the engine model's parameters"""

    def __init__(self, net):
        vals = params(net)
        self.p = [R.RefTensor(v, True) for v in vals]
        self.opt = R.RefAdam(lr=1e-3)

    def loss(self, x, y):
        w1, b1, w2, b2, w3, b3 = self.p
        h = R.clip(RC.conv2d(R.lift(x), w1, b1, (2, 2), "SAME"), 0.0)
        h = RC.maxpool2d(h, (2, 2))
        h = R.clip(RC.conv2d(h, w2, b2, (1, 1), "SAME"), 0.0)
        h = R.reshape(h, (x.shape[0], -1))
        return R.softmax_cross_entropy(R.matmul(h, w3) + b3, y)

    def step(self, x, y):
        for p in self.p:
            p.zero_grad()
        loss = self.loss(x, y)
        loss.backward()
        grads = [p.grad.copy() for p in self.p]
        for p, s in zip(self.p, self.opt.compute_steps(self.p)):
            p.assign(p.values + s)
            p.zero_grad()
        return float(loss.values), grads


def _eager(model, x, y):
    model.zero_grad()
    loss = model.loss.loss(model.forward(x), y)
    loss.backward()
    model.step()
    return loss


def test_cnn_one_step_matches_oracle(be):
    """teacher forced: the loss and every parameter gradient within 1e-5 of the oracle (f32)"""
    from core.tensor import Tensor
    x, y = _data(128)
    net, model = _cnn(0)
    ref = _RefCNN(net)
    model.zero_grad()
    loss = model.loss.loss(model.forward(Tensor(x)), Tensor(y))
    loss.backward()
    grads = [p.grad.copy() for layer in net.get_parameters() for p in layer.values()]
    rloss, rgrads = ref.step(x, y)
    assert abs(float(loss.values) - rloss) <= 1e-5 * abs(rloss)
    assert [g.shape for g in grads] == [(5, 5, 1, 8), (1, 8), (3, 3, 8, 16), (1, 16), (784, 10), (1, 10)]
    for g, rg in zip(grads, rgrads):
        assert _rel(g, rg) <= 1e-5, _rel(g, rg)


def test_cnn_loss_trajectory_matches_oracle(be):
    """50 free-running Adam steps in float32 against the float64 oracle: within 1e-4 at every step,
    and the network learns"""
    from core.tensor import Tensor
    steps, B = 50, 128
    x, y = _data(steps * B)
    net, model = _cnn(0)
    ref = _RefCNN(net)
    losses, rlosses = [], []
    for i in range(steps):
        xb, yb = x[i * B:(i + 1) * B], y[i * B:(i + 1) * B]
        losses.append(float(_eager(model, Tensor(xb), Tensor(yb)).values))
        rlosses.append(ref.step(xb, yb)[0])
    diff = np.abs(np.array(losses) - np.array(rlosses))
    assert np.max(diff) <= 1e-4, (int(np.argmax(diff)), float(np.max(diff)))
    assert np.mean(losses[-5:]) < np.mean(losses[:5]) - 0.1


def test_cnn_train_step_replay_is_bit_identical(be):
    """Model.train_step records the layer-by-layer step (no fused MLP plan for this network) and its
    replays give the eager five lines' bits, across a change of batch shape"""
    from core.tensor import Tensor
    x, y = _data(128 * 8)
    sizes = [128] * 5 + [80, 80, 80] + [128] * 2
    net_a, model_a = _cnn(3)
    net_b, model_b = _cnn(3)
    assert model_b._fused_mlp_plan(Tensor(x[:128]), Tensor(y[:128])) is None
    start = 0
    for b in sizes:
        xb, yb = Tensor(x[start:start + b]), Tensor(y[start:start + b])
        start = (start + b) % (len(x) - 128)
        la = float(_eager(model_a, xb, yb).values)
        lb = float(model_b.train_step(xb, yb).values)
        assert la == lb
    states = [s for s in model_b._captured.values() if hasattr(s, "graph")]
    assert len(states) == 2
    assert model_b._fused_mlp_plan(Tensor(x[:128]), Tensor(y[:128])) is None
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.array_equal(pa, pb)


def test_cnn_five_line_loop_recording_is_bit_identical(be):
    """the unmodified loop with its iterations replayed from a recording (core/_deferred.py) gives
    the bits of the same loop run eagerly"""
    from core.losses import SoftmaxCrossEntropyLoss
    from core.tensor import Tensor
    x, y = _data(128 * 8)
    net_a, model_a = _cnn(4)
    net_b, model_b = _cnn(4)
    model_a.defer_loop, model_b.defer_loop = False, True
    out = []
    for model in (model_a, model_b):
        loss_layer = SoftmaxCrossEntropyLoss()
        losses = []
        for i in range(8):
            xb, yb = Tensor(x[i * 128:(i + 1) * 128]), Tensor(y[i * 128:(i + 1) * 128])
            model.zero_grad()
            pred = model.forward(xb)
            loss = loss_layer.loss(pred, yb)
            loss.backward()
            model.step()
            losses.append(float(loss.values))
        out.append(losses)
    assert out[0] == out[1]
    assert [s for s in model_b._captured.values() if hasattr(s, "graph")]
    assert not [s for s in model_a._captured.values() if hasattr(s, "graph")]
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.array_equal(pa, pb)


def test_cnn_predict_and_checkpoint(be, tmp_path):
    """predict equals forward and builds no graph; save / load round-trips the 4-D weights"""
    from core.tensor import Tensor
    x, y = _data(64)
    net, model = _cnn(5)
    for i in range(2):
        _eager(model, Tensor(x), Tensor(y))
    pred = model.predict(Tensor(x))
    assert not pred.requires_grad and not pred.dependency
    assert np.array_equal(pred.values, net.forward(Tensor(x)).values)
    path = os.path.join(str(tmp_path), "cnn.pkl")
    model.save(path)
    net2, model2 = _cnn(6)
    assert not np.array_equal(params(net)[0], params(net2)[0])
    model2.load(path)
    for pa, pb in zip(params(net), params(net2)):
        assert np.array_equal(pa, pb)
    assert net2.layers[0].params["w"].shape == (5, 5, 1, 8)
    assert np.array_equal(model2.predict(Tensor(x)).values, pred.values)
