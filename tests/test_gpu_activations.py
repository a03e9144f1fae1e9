"""The elementwise activations on the device (LeakyReLU, ELU, GELU in both forms, Softplus, SiLU: the
activation op codes of csrc/elementwise.cu) against the float64 oracle of oracle/ref_activations.py:
values and gradients over activation x dtype x shape with aligned and offset pointers (the vector and
the scalar path), special values, LeakyReLU(0) against ReLU, one launch each way, the empty batch;
then training through the model -- an MLP with GELU and LeakyReLU and an NHWC CNN with ELU and SiLU --
against the oracle, train_step and the recorded five-line loop against the eager step, predict in the
TEST phase and a checkpoint round trip."""
import os

import numpy as np
import pytest

import ref_activations as RA
import ref_conv as RC
import ref_numpy as R
from support import params

pytestmark = pytest.mark.gpu

CASES = [("leaky_relu", 0.0), ("leaky_relu", 0.01), ("leaky_relu", 0.2), ("elu", 0.5), ("elu", 1.0), ("elu", 2.0),
         ("gelu", None), ("gelu_tanh", None), ("softplus", None), ("silu", None)]


def _ids(case):
    return case[0] if case[1] is None else "%s-%g" % case


@pytest.fixture(scope="module")
def be():
    import core._backend as be
    be.init()
    return be


def _layer(kind, param):
    from core.layers import ELU, GELU, LeakyReLU, SiLU, Softplus
    if kind == "leaky_relu":
        return LeakyReLU(param)
    if kind == "elu":
        return ELU(param)
    if kind in ("gelu", "gelu_tanh"):
        return GELU("tanh" if kind == "gelu_tanh" else "none")
    return {"softplus": Softplus, "silu": SiLU}[kind]()


def _err(a, b, floor=0.0):
    """max |a - b| relative to max |b| (or `floor` where that is larger)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(np.max(np.abs(b), initial=0.0), floor)
    return np.max(np.abs(a - b), initial=0.0) / scale if scale > 0 else np.max(np.abs(a - b), initial=0.0)


def _device(be, host, offset=0):
    """host array on the device, starting `offset` elements into its allocation"""
    buf = be.zeros((host.size + offset,), host.dtype)
    d = buf.view(host.shape, offset)
    be.upload_into(d, host)
    return d                        # (the view keeps the allocation alive)


def _bounds(dtype):
    """normwise bounds (values, gradients)"""
    return (1e-12, 1e-12) if dtype == np.float64 else (1e-6, 2e-6)


def _run(be, layer, x, g, offset=0):
    """(y, dx) of `layer` on the device for input x and upstream gradient g, both host arrays"""
    from core.tensor import Tensor
    tx = Tensor(_device(be, x, offset), requires_grad=True)
    y = layer(tx)
    y.backward(_device(be, g, offset))
    return y.values, tx.grad


SHAPES = [(1,), (1001,), (37, 11), (3, 5, 7, 2), (256, 32, 32, 64)]


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_values_and_gradients_match_oracle(be, case, dtype, shape, offset):
    kind, param = case
    rng = np.random.RandomState(sum(shape) + offset)
    x = (rng.standard_normal(shape) * 3.0).astype(dtype)
    g = rng.standard_normal(shape).astype(dtype)        # a non-unit upstream gradient
    y, dx = _run(be, _layer(kind, param), x, g, offset)
    assert y.dtype == dtype and y.shape == shape and dx.dtype == dtype and dx.shape == shape
    ry, rdx = RA.value_and_grad(x, kind, param, g)
    tol_y, tol_g = _bounds(dtype)
    assert _err(y, ry) <= tol_y, _err(y, ry)
    assert _err(dx, rdx) <= tol_g, _err(dx, rdx)


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_special_values(be, case, dtype):
    """+-0, +-inf, NaN and large finite inputs: NaN exactly where the oracle has it, infinities equal,
    every finite input gives a finite value and gradient, close to the oracle's element by element"""
    kind, param = case
    big = [3e38, -3e38, 1e20, -1e20, 7e12, -7e12] + ([1e300, -1e300] if dtype == np.float64 else [])
    x = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1.0, -1.0, 30.0, -30.0, 200.0, -200.0] + big, dtype)
    x = np.tile(x, 3)                                 # long enough for the vector path too
    g = np.full(x.shape, 1.5, dtype)
    finite = np.isfinite(x)
    for offset in (0, 1):
        y, dx = _run(be, _layer(kind, param), x, g, offset)
        ry, rdx = RA.value_and_grad(x, kind, param, g)
        for got, want in ((y, ry), (dx, rdx)):
            assert np.array_equal(np.isnan(got), np.isnan(want)), (x, got, want)
            assert np.all(np.isfinite(got[finite])), (x[finite], got[finite])
            inf = np.isinf(want)
            assert np.array_equal(got[inf], want[inf].astype(dtype))
            ok = np.isfinite(want)
            tol = 1e-12 if dtype == np.float64 else 2e-6
            assert np.all(np.abs(got[ok] - want[ok]) <= tol * np.maximum(1.0, np.abs(want[ok]))), (x[ok], got[ok],
                                                                                                    want[ok])
        # the kink at 0 goes to the x >= 0 branch
        if kind in ("leaky_relu", "elu"):
            assert np.all(dx[:2] == 1.5)


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_leaky_relu_zero_slope_equals_relu(be, dtype):
    from core.layers import ReLU
    rng = np.random.RandomState(7)
    for shape in ((1001,), (64, 33), (8, 5, 5, 16)):
        x = (rng.standard_normal(shape) * 2.0).astype(dtype)
        x.ravel()[:4] = [0.0, -0.0, 3e38, -3e38]
        g = rng.standard_normal(shape).astype(dtype)
        y, dx = _run(be, _layer("leaky_relu", 0.0), x, g)
        ry, rdx = _run(be, ReLU(), x, g)
        assert np.array_equal(y, ry)
        assert np.array_equal(dx, rdx)


@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_one_launch_forward_and_one_backward(be, case):
    from core.tensor import Tensor
    for dtype in (np.float32, np.float64):
        for shape in ((1024, 256), (1001,)):
            rng = np.random.RandomState(0)
            tx = Tensor(_device(be, rng.standard_normal(shape).astype(dtype)), requires_grad=True)
            g = _device(be, rng.standard_normal(shape).astype(dtype))
            layer = _layer(*case)
            be.sync()
            n0 = be.launch_count()
            y = layer(tx)
            assert be.launch_count() - n0 == 1
            y.backward(g)
            assert be.launch_count() - n0 == 2
            tx.grad         # (a read back, not a launch)
            assert be.launch_count() - n0 == 2


@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_empty_batch(be, case):
    from core.tensor import Tensor
    tx = Tensor(be.zeros((0, 16), np.float32), requires_grad=True)
    be.sync()
    n0 = be.launch_count()
    y = _layer(*case)(tx)
    assert y.shape == (0, 16) and y.dtype == np.float32
    y.backward(be.zeros((0, 16), np.float32))
    assert tx.grad.shape == (0, 16)
    assert be.launch_count() == n0


def test_no_grad_builds_no_graph(be):
    import core.ops as ops
    from core.tensor import Tensor
    tx = Tensor(_device(be, np.linspace(-3, 3, 64, dtype=np.float32)), requires_grad=True)
    with ops.no_grad():
        y = _layer("gelu", None)(tx)
    assert not y.requires_grad and not y.dependency


# ---------------------------------------------------------------------------- through the model
B, DIN, DH, C = 128, 20, 48, 10


def _class_data(n, seed=0):
    rng = np.random.RandomState(seed)
    x = rng.standard_normal((n, DIN)).astype(np.float32)
    w = rng.standard_normal((DIN, C))
    labels = np.argmax(x @ w + 0.5 * rng.standard_normal((n, C)), axis=1)
    return x, np.eye(C, dtype=np.float32)[labels]


def _mlp(seed):
    from core.layers import GELU, Dense, LeakyReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    np.random.seed(seed)
    net = Net([Dense(DH, num_in=DIN), GELU(), Dense(DH, num_in=DH), LeakyReLU(0.1), Dense(C, num_in=DH)])
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))


class _RefMLP(object):
    def __init__(self, net):
        self.p = [R.RefTensor(v, True) for v in params(net)]
        self.opt = R.RefAdam(lr=1e-3)

    def loss(self, x, y):
        w1, b1, w2, b2, w3, b3 = self.p
        h = RA.activation(R.matmul(R.lift(x), w1) + b1, "gelu")
        h = RA.activation(R.matmul(h, w2) + b2, "leaky_relu", 0.1)
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


H_IMG, W_IMG, CIN, C1, C2 = 8, 8, 3, 8, 12


def _img_data(n, seed=0):
    rng = np.random.RandomState(seed)
    x = rng.standard_normal((n, H_IMG, W_IMG, CIN)).astype(np.float32)
    score = x[:, :4, :4, 0].mean(axis=(1, 2))[:, None] * np.arange(-2.0, 3.0)[None, :] \
        + x[:, 4:, 4:, 1].mean(axis=(1, 2))[:, None] * np.array([1.0, -1.0, 0.5, 2.0, -0.5])[None, :]
    return x, np.eye(5, dtype=np.float32)[np.argmax(score, axis=1)]


def _cnn(seed):
    from core.layers import ELU, Conv2D, Dense, Flatten, MaxPool2D, SiLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    np.random.seed(seed)
    net = Net([Conv2D((3, 3, CIN, C1)), ELU(0.5), MaxPool2D(), Conv2D((3, 3, C1, C2)), SiLU(), Flatten(),
               Dense(5, num_in=4 * 4 * C2)])
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))


class _RefCNN(_RefMLP):
    def loss(self, x, y):
        w1, b1, w2, b2, w3, b3 = self.p
        h = RA.activation(RC.conv2d(R.lift(x), w1, b1, (1, 1), "SAME"), "elu", 0.5)
        h = RC.maxpool2d(h, (2, 2))
        h = RA.activation(RC.conv2d(h, w2, b2, (1, 1), "SAME"), "silu")
        return R.softmax_cross_entropy(R.matmul(R.reshape(h, (x.shape[0], -1)), w3) + b3, y)


NETS = {"mlp_gelu_leaky": (_mlp, _RefMLP, _class_data, B), "cnn_elu_silu": (_cnn, _RefCNN, _img_data, 64)}


def _eager(model, x, y):
    model.zero_grad()
    loss = model.loss.loss(model.forward(x), y)
    loss.backward()
    model.step()
    return loss


@pytest.mark.parametrize("which", sorted(NETS))
def test_one_step_and_trajectory_match_oracle(be, which):
    from core.tensor import Tensor
    build, ref_cls, data, n = NETS[which]
    steps = 50
    x, y = data(n * steps)
    net, model = build(0)
    model.defer_loop = False
    assert model._fused_mlp_plan(Tensor(x[:n]), Tensor(y[:n])) is None
    ref = ref_cls(net)
    model.zero_grad()
    loss = model.loss.loss(model.forward(Tensor(x[:n])), Tensor(y[:n]))
    loss.backward()
    grads = [p.grad.copy() for layer in net.get_parameters() for p in layer.values()]
    rloss, rgrads = ref.step(x[:n], y[:n])
    assert abs(float(loss.values) - rloss) <= 1e-5 * abs(rloss)
    for g, rg in zip(grads, rgrads):
        assert _err(g, rg) <= 1e-5, _err(g, rg)
    model.step()
    losses, rlosses = [float(loss.values)], [rloss]
    for i in range(1, steps):
        xb, yb = x[i * n:(i + 1) * n], y[i * n:(i + 1) * n]
        losses.append(float(_eager(model, Tensor(xb), Tensor(yb)).values))
        rlosses.append(ref.step(xb, yb)[0])
    diff = np.abs(np.array(losses) - np.array(rlosses))
    assert np.max(diff) <= 1e-4, (int(np.argmax(diff)), float(np.max(diff)))
    assert np.mean(losses[-5:]) < np.mean(losses[:5])


@pytest.mark.parametrize("which", sorted(NETS))
def test_train_step_and_recorded_loop_are_bit_identical_to_eager(be, which):
    from core.tensor import Tensor
    build, _, data, n = NETS[which]
    x, y = data(n * 8, seed=1)
    batches = [(Tensor(x[i * n:(i + 1) * n]), Tensor(y[i * n:(i + 1) * n])) for i in range(8)]
    (net_a, model_a), (net_b, model_b), (net_c, model_c) = build(5), build(5), build(5)
    model_a.defer_loop, model_c.defer_loop = False, True
    la = [float(_eager(model_a, xb, yb).values) for xb, yb in batches]
    lb = [float(model_b.train_step(xb, yb).values) for xb, yb in batches]
    lc = [float(_eager(model_c, xb, yb).values) for xb, yb in batches]
    assert la == lb == lc
    assert [s for s in model_b._captured.values() if hasattr(s, "graph")]
    assert [s for s in model_c._captured.values() if hasattr(s, "graph")]
    assert not [s for s in model_a._captured.values() if hasattr(s, "graph")]
    for pa, pb, pc in zip(params(net_a), params(net_b), params(net_c)):
        assert np.array_equal(pa, pb) and np.array_equal(pa, pc)


@pytest.mark.parametrize("which", sorted(NETS))
def test_predict_in_test_phase_and_checkpoint(be, which, tmp_path):
    from core.tensor import Tensor
    build, _, data, n = NETS[which]
    x, y = data(n, seed=2)
    net, model = build(6)
    for _ in range(2):
        _eager(model, Tensor(x), Tensor(y))
    model.set_phase("TEST")
    pred = model.predict(Tensor(x))
    assert not pred.requires_grad and not pred.dependency
    assert np.array_equal(pred.values, net.forward(Tensor(x)).values)
    path = os.path.join(str(tmp_path), which + ".pkl")
    model.save(path)
    net2, model2 = build(7)
    model2.load(path)
    model2.set_phase("TEST")
    for pa, pb in zip(params(net), params(net2)):
        assert np.array_equal(pa, pb)
    assert np.array_equal(model2.predict(Tensor(x)).values, pred.values)
