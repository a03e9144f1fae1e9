"""The pointwise losses on the device (csrc/loss.cu: MSELoss, MAELoss, HuberLoss,
SigmoidCrossEntropyLoss) against the float64 oracle of oracle/ref_losses.py: loss and gradient over a
grid of loss x dtype x shape with aligned and offset pointers (the vector and the scalar path), the
seeded gradient against the backward launch, a non-unit upstream gradient, the launch count, bit
reproducibility, NaN / inf, an empty row and a 2^26-element case; then training through the model --
a regression MLP with MSELoss and an NHWC CNN head with SigmoidCrossEntropyLoss against the oracle,
train_step and the recorded five-line loop against the eager step, and a loop alternating two Huber
deltas."""
import numpy as np
import pytest

import ref_conv as RC
import ref_losses as RL
import ref_numpy as R
from support import gpu_count, params, run_two_ranks

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    import core._backend as be
    be.init()
    return be


def _err(a, b, floor=0.0):
    """max |a - b| relative to max |b| (or `floor` where that is larger)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(np.max(np.abs(b), initial=0.0), floor)
    return np.max(np.abs(a - b), initial=0.0) / scale if scale > 0 else np.max(np.abs(a - b), initial=0.0)


def _loss_obj(kind, delta=1.0):
    from core.losses import HuberLoss, MAELoss, MSELoss, SigmoidCrossEntropyLoss
    return {"mse": MSELoss, "mae": MAELoss, "sigmoid_ce": SigmoidCrossEntropyLoss}[kind]() if kind != "huber" \
        else HuberLoss(delta)


def _inputs(kind, shape, dtype, seed, delta=1.0):
    rng = np.random.RandomState(seed)
    if kind == "sigmoid_ce":
        p = rng.standard_normal(shape) * 6.0
        t = rng.rand(*shape)
    else:
        t = rng.standard_normal(shape)
        p = t + rng.standard_normal(shape) * 1.5 * delta
    return p.astype(dtype), t.astype(dtype)


def _device(be, host, offset):
    """host array on the device, starting `offset` elements into its allocation"""
    buf = be.zeros((host.size + offset,), host.dtype)
    d = buf.view(host.shape, offset)
    be.upload_into(d, host)
    return d                        # (the view keeps the allocation alive)


def _tensors(be, p, t, offset=0):
    from core.tensor import Tensor
    tp = Tensor(_device(be, p, offset), requires_grad=True)
    tt = Tensor(_device(be, t, offset))
    return tp, tt


def _bounds(dtype):
    return (1e-12, 1e-12) if dtype == np.float64 else (1e-6, 1e-6)


SHAPES = [(1,), (1001,), (1, 1), (5, 3), (37, 11), (128, 10), (3, 5, 7, 2), (256, 32, 32, 64)]


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kind", RL.KINDS)
def test_loss_and_gradient_match_oracle(be, kind, dtype, shape, offset):
    delta = 0.8
    p, t = _inputs(kind, shape, dtype, seed=sum(shape) + offset)
    tp, tt = _tensors(be, p, t, offset)
    loss = _loss_obj(kind, delta).loss(tp, tt)
    assert loss.shape == () and loss.dtype == dtype
    loss.backward()
    L, d = RL.loss_and_grad(p, t, kind, delta)
    tol_l, tol_g = _bounds(dtype)
    assert abs(float(loss.values) - L) <= tol_l * max(abs(L), 1e-30), (float(loss.values), L)
    grad = tp.grad
    assert grad.dtype == dtype and grad.shape == shape
    assert _err(grad, d) <= tol_g


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kind", RL.KINDS)
def test_seeded_gradient_is_bit_identical_to_backward_launch(be, kind, dtype):
    for shape, offset in (((128, 10), 0), ((1000, 33), 1), ((64, 8, 8, 16), 0)):
        p, t = _inputs(kind, shape, dtype, seed=3)
        dp_, dt_ = _device(be, p, offset), _device(be, t, offset)
        code = getattr(be, "LOSS_" + kind.upper())
        loss, seeded = be.pointwise_loss(dp_, dt_, code, shape[0], 0.8, want_dp=True)
        loss_only, none = be.pointwise_loss(dp_, dt_, code, shape[0], 0.8)
        assert none is None and np.array_equal(loss.numpy(), loss_only.numpy())
        explicit = be.pointwise_loss_bwd(dp_, dt_, code, shape[0], 0.8, be.full((), 1.0, dtype))
        assert np.array_equal(seeded.numpy(), explicit.numpy())


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kind", RL.KINDS)
def test_non_unit_upstream_gradient(be, kind, dtype):
    p, t = _inputs(kind, (96, 7), dtype, seed=9)
    tp, tt = _tensors(be, p, t)
    (_loss_obj(kind, 0.8).loss(tp, tt) * 2.5).backward()
    _, d = RL.loss_and_grad(p, t, kind, 0.8, g=2.5)
    assert _err(tp.grad, d) <= _bounds(dtype)[1]
    # and through backward() with an explicit gradient of 1: the backward launch, the seeded bits
    tp2, tt2 = _tensors(be, p, t)
    tp3, tt3 = _tensors(be, p, t)
    _loss_obj(kind, 0.8).loss(tp2, tt2).backward()
    _loss_obj(kind, 0.8).loss(tp3, tt3).backward(np.ones((), dtype))
    assert np.array_equal(tp2.grad, tp3.grad)


@pytest.mark.parametrize("kind", RL.KINDS)
def test_forward_and_seeded_backward_are_one_launch(be, kind):
    for shape in ((128, 10), (64, 8, 8, 16), (1 << 20,)):
        p, t = _inputs(kind, shape, np.float32, seed=1)
        tp, tt = _tensors(be, p, t)
        be.sync()
        n0 = be.launch_count()
        loss = _loss_obj(kind).loss(tp, tt)
        loss.backward()
        assert be.launch_count() - n0 == 1
        tp.grad        # (a read back, not a launch)
        assert be.launch_count() - n0 == 1


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_bit_reproducible_over_many_ctas(be, dtype):
    n = (1 << 22) + 3
    for kind in RL.KINDS:
        p, t = _inputs(kind, (n,), dtype, seed=4)
        for offset in (0, 1):
            dp_, dt_ = _device(be, p, offset), _device(be, t, offset)
            code = getattr(be, "LOSS_" + kind.upper())
            runs = [be.pointwise_loss(dp_, dt_, code, 1024, 0.8, want_dp=True) for _ in range(4)]
            losses = [r[0].numpy().tobytes() for r in runs]
            grads = [r[1].numpy() for r in runs]
            assert len(set(losses)) == 1
            assert all(np.array_equal(g, grads[0]) for g in grads[1:])


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kind", RL.KINDS)
def test_nan_and_inf_propagate_like_numpy(be, kind, dtype):
    special = np.array([np.nan, np.inf, -np.inf, 0.0, 1.0, -2.0])
    p = np.repeat(special, 6).reshape(6, 6).astype(dtype)
    t = np.tile(np.array([0.0, 1.0, 0.5, np.nan, np.inf, -np.inf]), 6).reshape(6, 6).astype(dtype)
    with np.errstate(all="ignore"):
        _, d = RL.loss_and_grad(p, t, kind, 0.8)
    for offset in (0, 1):
        dp_, dt_ = _device(be, p, offset), _device(be, t, offset)
        code = getattr(be, "LOSS_" + kind.upper())
        _, got = be.pointwise_loss(dp_, dt_, code, 6, 0.8, want_dp=True)
        got = got.numpy()
        assert np.array_equal(np.isnan(got), np.isnan(d)), (got, d)
        finite = np.isfinite(d)
        assert np.array_equal(got[~finite & ~np.isnan(d)], d[~finite & ~np.isnan(d)].astype(dtype))
        assert _err(got[finite], d[finite]) <= _bounds(dtype)[1]
    # any NaN term makes the loss NaN
    tp, tt = _tensors(be, p, t)
    assert np.isnan(float(_loss_obj(kind, 0.8).loss(tp, tt).values))
    # a finite loss with an infinite term: inf
    q = np.zeros((2, 3), dtype)
    q[1, 2] = np.inf
    tp, tt = _tensors(be, q, np.zeros((2, 3), dtype))
    with np.errstate(all="ignore"):
        expect, _ = RL.loss_and_grad(q, np.zeros((2, 3)), kind, 0.8)
    got = float(_loss_obj(kind, 0.8).loss(tp, tt).values)
    assert got == expect or (np.isnan(got) and np.isnan(expect)), (got, expect)    # (inf * 0 in sigmoid_ce)


@pytest.mark.parametrize("kind", RL.KINDS)
def test_rows_without_columns(be, kind):
    tp, tt = _tensors(be, np.zeros((4, 0), np.float32), np.zeros((4, 0), np.float32))
    loss = _loss_obj(kind).loss(tp, tt)
    assert float(loss.values) == 0.0
    loss.backward()
    assert tp.grad.shape == (4, 0)
    tp, tt = _tensors(be, np.zeros((4, 0), np.float32), np.zeros((4, 0), np.float32))
    (_loss_obj(kind).loss(tp, tt) * 3.0).backward()
    assert tp.grad.shape == (4, 0)


def test_two_to_the_26_elements(be):
    n = 1 << 26
    rng = np.random.RandomState(2)
    t = rng.standard_normal(n).astype(np.float32)
    p = (t + rng.standard_normal(n).astype(np.float32)).astype(np.float32)
    for kind in ("mse", "sigmoid_ce"):
        tp, tt = _tensors(be, p.reshape(1 << 13, 1 << 13), t.reshape(1 << 13, 1 << 13))
        loss = _loss_obj(kind).loss(tp, tt)
        loss.backward()
        L, d = RL.loss_and_grad(p.reshape(1 << 13, 1 << 13), t.reshape(1 << 13, 1 << 13), kind)
        assert abs(float(loss.values) - L) <= 1e-6 * abs(L)
        assert _err(tp.grad, d) <= 1e-6
        del tp, tt, loss, d


# ---------------------------------------------------------------------------- through the model
B, DIN, DH, DOUT = 128, 16, 32, 4


def _regression_data(n, seed=0):
    rng = np.random.RandomState(seed)
    x = rng.standard_normal((n, DIN)).astype(np.float32)
    w = rng.standard_normal((DIN, DOUT)) / 4.0
    y = (np.tanh(x @ w) * 2.0 + 0.1 * rng.standard_normal((n, DOUT))).astype(np.float32)
    return x, y


def _mlp(seed, loss):
    from core.layers import Dense, ReLU
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    np.random.seed(seed)
    net = Net([Dense(DH, num_in=DIN), ReLU(), Dense(DOUT, num_in=DH)])
    return net, Model(net=net, loss=loss, optimizer=Adam(lr=1e-3))


class _RefMLP(object):
    def __init__(self, net, kind, delta=1.0):
        self.p = [R.RefTensor(v, True) for v in params(net)]
        self.kind, self.delta = kind, delta
        self.opt = R.RefAdam(lr=1e-3)

    def step(self, x, y, delta=None):
        w1, b1, w2, b2 = self.p
        for p in self.p:
            p.zero_grad()
        h = R.clip(R.matmul(R.lift(x), w1) + b1, 0.0)
        loss = RL.pointwise_loss(R.matmul(h, w2) + b2, y, self.kind, self.delta if delta is None else delta)
        loss.backward()
        grads = [p.grad.copy() for p in self.p]
        for p, s in zip(self.p, self.opt.compute_steps(self.p)):
            p.assign(p.values + s)
            p.zero_grad()
        return float(loss.values), grads


def _eager(model, x, y, loss_obj=None):
    model.zero_grad()
    loss = (loss_obj or model.loss).loss(model.forward(x), y)
    loss.backward()
    model.step()
    return loss


def test_regression_mlp_one_step_and_trajectory_match_oracle(be):
    from core.losses import MSELoss
    from core.tensor import Tensor
    steps = 40
    x, y = _regression_data(B * steps)
    net, model = _mlp(0, MSELoss())
    model.defer_loop = False
    ref = _RefMLP(net, "mse")
    model.zero_grad()
    loss = model.loss.loss(model.forward(Tensor(x[:B])), Tensor(y[:B]))
    loss.backward()
    grads = [p.grad.copy() for layer in net.get_parameters() for p in layer.values()]
    rloss, rgrads = ref.step(x[:B], y[:B])
    assert abs(float(loss.values) - rloss) <= 1e-5 * abs(rloss)
    for g, rg in zip(grads, rgrads):
        assert _err(g, rg) <= 1e-5
    model.step()
    losses, rlosses = [float(loss.values)], [rloss]
    for i in range(1, steps):
        xb, yb = x[i * B:(i + 1) * B], y[i * B:(i + 1) * B]
        losses.append(float(_eager(model, Tensor(xb), Tensor(yb)).values))
        rlosses.append(ref.step(xb, yb)[0])
    diff = np.abs(np.array(losses) - np.array(rlosses))
    assert np.max(diff) <= 1e-4, (int(np.argmax(diff)), float(np.max(diff)))
    assert np.mean(losses[-5:]) < np.mean(losses[:5])


H_IMG, W_IMG, CIN, CMID, COUT = 8, 8, 2, 6, 3


def _cnn_data(n, seed=0):
    rng = np.random.RandomState(seed)
    x = rng.standard_normal((n, H_IMG, W_IMG, CIN)).astype(np.float32)
    # multi-label per pixel: soft targets from a fixed smooth function of the input
    y = (1.0 / (1.0 + np.exp(-(x[..., :1] * np.array([1.0, -2.0, 0.5]) + x[..., 1:] * 0.7)))).astype(np.float32)
    return x, y


def _cnn(seed):
    from core.layers import Conv2D, ReLU
    from core.losses import SigmoidCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    np.random.seed(seed)
    net = Net([Conv2D((3, 3, CIN, CMID)), ReLU(), Conv2D((3, 3, CMID, COUT))])
    return net, Model(net=net, loss=SigmoidCrossEntropyLoss(), optimizer=Adam(lr=1e-3))


class _RefCNN(object):
    def __init__(self, net):
        self.p = [R.RefTensor(v, True) for v in params(net)]
        self.opt = R.RefAdam(lr=1e-3)

    def step(self, x, y):
        w1, b1, w2, b2 = self.p
        for p in self.p:
            p.zero_grad()
        h = R.clip(RC.conv2d(R.lift(x), w1, b1, (1, 1), "SAME"), 0.0)
        loss = RL.pointwise_loss(RC.conv2d(h, w2, b2, (1, 1), "SAME"), y, "sigmoid_ce")
        loss.backward()
        grads = [p.grad.copy() for p in self.p]
        for p, s in zip(self.p, self.opt.compute_steps(self.p)):
            p.assign(p.values + s)
            p.zero_grad()
        return float(loss.values), grads


def test_nhwc_cnn_head_one_step_and_trajectory_match_oracle(be):
    from core.tensor import Tensor
    steps, n = 30, 64
    x, y = _cnn_data(n * steps)
    net, model = _cnn(0)
    model.defer_loop = False
    ref = _RefCNN(net)
    model.zero_grad()
    pred = model.forward(Tensor(x[:n]))
    assert pred.shape == (n, H_IMG, W_IMG, COUT)
    loss = model.loss.loss(pred, Tensor(y[:n]))
    loss.backward()
    grads = [p.grad.copy() for layer in net.get_parameters() for p in layer.values()]
    rloss, rgrads = ref.step(x[:n], y[:n])
    assert abs(float(loss.values) - rloss) <= 1e-5 * abs(rloss)
    for g, rg in zip(grads, rgrads):
        assert _err(g, rg) <= 1e-5
    model.step()
    losses, rlosses = [float(loss.values)], [rloss]
    for i in range(1, steps):
        xb, yb = x[i * n:(i + 1) * n], y[i * n:(i + 1) * n]
        losses.append(float(_eager(model, Tensor(xb), Tensor(yb)).values))
        rlosses.append(ref.step(xb, yb)[0])
    diff = np.abs(np.array(losses) - np.array(rlosses))
    assert np.max(diff) <= 1e-4, (int(np.argmax(diff)), float(np.max(diff)))


@pytest.mark.parametrize("which", ["mlp_mse", "mlp_mae", "mlp_huber", "cnn_sigmoid_ce"])
def test_train_step_and_recorded_loop_are_bit_identical_to_eager(be, which):
    """train_step records the layer-by-layer step (the fused small-MLP plan declines these losses);
    the five-line loop records it too where the prediction is 2-D, and runs eagerly for the 4-D head.
    Every variant gives the eager bits."""
    from core.losses import HuberLoss, MAELoss, MSELoss
    from core.tensor import Tensor
    if which.startswith("mlp"):
        loss_cls = {"mlp_mse": MSELoss, "mlp_mae": MAELoss, "mlp_huber": lambda: HuberLoss(0.5)}[which]
        x, y = _regression_data(B * 8)
        build, n = (lambda seed: _mlp(seed, loss_cls())), B
    else:
        x, y = _cnn_data(64 * 8)
        build, n = _cnn, 64
    batches = [(Tensor(x[i * n:(i + 1) * n]), Tensor(y[i * n:(i + 1) * n])) for i in range(8)]
    (net_a, model_a), (net_b, model_b), (net_c, model_c) = build(5), build(5), build(5)
    model_a.defer_loop, model_c.defer_loop = False, True
    assert model_b._fused_mlp_plan(*batches[0]) is None
    la = [float(_eager(model_a, xb, yb).values) for xb, yb in batches]
    lb = [float(model_b.train_step(xb, yb).values) for xb, yb in batches]
    lc = [float(_eager(model_c, xb, yb).values) for xb, yb in batches]
    assert la == lb == lc
    assert [s for s in model_b._captured.values() if hasattr(s, "graph")]
    if which.startswith("mlp"):
        assert [s for s in model_c._captured.values() if hasattr(s, "graph")]
    for pa, pb, pc in zip(params(net_a), params(net_b), params(net_c)):
        assert np.array_equal(pa, pb) and np.array_equal(pa, pc)


def test_alternating_huber_deltas_in_the_recorded_loop(be):
    """two HuberLoss objects with different deltas alternate on the same model and batch shape: each
    gets its own recording, and the losses follow the oracle"""
    from core.losses import HuberLoss
    from core.tensor import Tensor
    x, y = _regression_data(B * 10, seed=1)
    batches = [(x[i * B:(i + 1) * B], y[i * B:(i + 1) * B]) for i in range(10)]
    deltas = (1.0, 2.0)
    net_a, model_a = _mlp(2, HuberLoss(1.0))
    net_b, model_b = _mlp(2, HuberLoss(1.0))
    model_a.defer_loop, model_b.defer_loop = False, True
    ref = _RefMLP(net_a, "huber")
    losses_fns = [HuberLoss(d) for d in deltas]
    out_a, out_b, rl = [], [], []
    for i, (xb, yb) in enumerate(batches):
        fn = losses_fns[i % 2]
        out_a.append(float(_eager(model_a, Tensor(xb), Tensor(yb), fn).values))
        out_b.append(float(_eager(model_b, Tensor(xb), Tensor(yb), fn).values))
        rl.append(ref.step(xb, yb, delta=deltas[i % 2])[0])
    assert out_a == out_b
    assert np.max(np.abs(np.array(out_a) - np.array(rl))) <= 1e-4
    recorded = [k for k, s in model_b._captured.items() if hasattr(s, "graph")]
    assert sorted(k[-1] for k in recorded) == [(1.0,), (2.0,)]
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.array_equal(pa, pb)
    # train_step with the model's loss swapped between the two deltas: the same bits again
    net_c, model_c = _mlp(2, HuberLoss(1.0))
    out_c = []
    for i, (xb, yb) in enumerate(batches):
        model_c.loss = losses_fns[i % 2]
        out_c.append(float(model_c.train_step(Tensor(xb), Tensor(yb)).values))
    assert out_c == out_a


# ---------------------------------------------------------------------------- two ranks
def test_two_rank_losses_equal_full_batch_oracle():
    if gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    assert "LOSS_DIST_OK world=2" in run_two_ranks("loss_dist_worker.py", timeout=200)
