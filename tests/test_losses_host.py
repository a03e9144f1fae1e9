"""Pointwise losses (MSELoss, MAELoss, HuberLoss, SigmoidCrossEntropyLoss) without a GPU: the float64
oracle (oracle/ref_losses.py) pinned against torch's mse_loss, l1_loss, huber_loss and
binary_cross_entropy_with_logits on the CPU, every argument the losses refuse, the data-parallel
scheme (two ranks over gloo with oracle compute: 1/m_global inside each rank's gradient, losses and
gradients SUM-reduced, equal to the full batch), and the recorded-step key.  torch is test
infrastructure here; nothing on the product path imports it."""
import os
import socket
import sys

import numpy as np
import pytest

import ref_losses as RL
import ref_numpy as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _close(a, b, tol=1e-12):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape
    assert np.max(np.abs(a - b), initial=0.0) <= tol * max(1.0, np.max(np.abs(b), initial=0.0))


def _torch_loss(p, t, kind, delta=1.0):
    """(L, dL/dp) from torch, reduction="sum" divided by the row count"""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    tp = torch.tensor(p, dtype=torch.float64, requires_grad=True)
    tt = torch.tensor(t, dtype=torch.float64)
    if kind == "mse":
        s = F.mse_loss(tp, tt, reduction="sum")
    elif kind == "mae":
        s = F.l1_loss(tp, tt, reduction="sum")
    elif kind == "huber":
        s = F.huber_loss(tp, tt, reduction="sum", delta=delta)
    else:
        s = F.binary_cross_entropy_with_logits(tp, tt, reduction="sum")
    L = s / p.shape[0]
    L.backward()
    return L.item(), tp.grad.numpy()


def _case(kind, shape, seed, delta=1.0):
    rng = np.random.RandomState(seed)
    if kind == "sigmoid_ce":
        p = rng.standard_normal(shape) * 30.0
        t = rng.rand(*shape)                        # soft targets in [0, 1)
        return p, t
    t = rng.standard_normal(shape)
    return t + rng.standard_normal(shape) * 2.0 * delta, t


SHAPES = [(7,), (1, 1), (5, 3), (4, 3, 2, 6)]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("kind", RL.KINDS)
def test_oracle_matches_torch(kind, shape):
    p, t = _case(kind, shape, seed=len(shape) * 7 + sum(shape))
    L, d = RL.loss_and_grad(p, t, kind)
    tL, td = _torch_loss(p, t, kind)
    _close(L, tL)
    _close(d, td)
    # the RefTensor node agrees with the plain function
    rp = R.RefTensor(p, True)
    node = RL.pointwise_loss(rp, t, kind)
    node.backward()
    assert float(node.values) == L
    assert np.array_equal(rp.grad, d)


@pytest.mark.parametrize("delta", [0.25, 1.0, 2.5])
def test_oracle_huber_both_sides_and_at_delta(delta):
    t = np.array([[0.5, -1.0, 2.0, 0.0, 0.25, -0.75, 3.0, 1.0]])
    t = np.repeat(t, 3, axis=0)
    # row 0: inside (|e| = delta / 2), row 1: outside (|e| = 3 delta), row 2: exactly at +-delta
    e = np.array([[0.5], [3.0], [1.0]]) * delta * np.array([1, -1, 1, -1, 1, -1, 1, -1])
    p = t + e
    assert np.array_equal(np.abs(p[2] - t[2]), np.full(8, delta))    # exact in binary
    L, d = RL.loss_and_grad(p, t, "huber", delta)
    tL, td = _torch_loss(p, t, "huber", delta)
    _close(L, tL)
    _close(d, td)
    # at |e| = delta both branches meet: l = delta^2 / 2, dl/dp = e
    l, dl = RL.terms(p[2], t[2], "huber", delta)
    _close(l, np.full(8, 0.5 * delta * delta))
    _close(dl, p[2] - t[2])


def test_oracle_mae_gradient_is_zero_where_prediction_equals_target():
    t = np.array([[0.0, 1.5, -2.0], [3.0, 0.0, 0.125]])
    p = t.copy()
    p[0, 1] += 1.0
    L, d = RL.loss_and_grad(p, t, "mae")
    tL, td = _torch_loss(p, t, "mae")
    _close(L, tL)
    _close(d, td)
    assert np.array_equal(d, [[0.0, 0.5, 0.0], [0.0, 0.0, 0.0]])


def test_oracle_sigmoid_ce_large_logits_and_soft_targets():
    z = np.array([[-100.0, -40.0, -5.0, -1e-3, 0.0, 1e-3, 5.0, 40.0, 100.0]] * 3)
    t = np.array([[0.0] * 9, [1.0] * 9, [0.3, 0.9, 0.5, 0.1, 0.5, 0.7, 0.2, 0.05, 0.99]])
    L, d = RL.loss_and_grad(z, t, "sigmoid_ce")
    tL, td = _torch_loss(z, t, "sigmoid_ce")
    assert np.isfinite(L) and np.all(np.isfinite(d))
    _close(L, tL)
    _close(d, td)


def test_mse_loss_equals_mse_evaluator():
    from core.evaluator import MSEEvaluator
    rng = np.random.RandomState(5)
    p, t = rng.standard_normal((9, 4)), rng.standard_normal((9, 4))
    L, _ = RL.loss_and_grad(p, t, "mse")
    _close(L, MSEEvaluator.evaluate(p, t)["mse"])


# ---------------------------------------------------------------------------- refusals
class _Stub(object):
    """stands in for a device tensor: shape, dtype and requires_grad, no device memory"""

    def __init__(self, shape, dtype=np.float32, requires_grad=False):
        self.shape, self.dtype, self.requires_grad = tuple(shape), np.dtype(dtype), requires_grad


def _losses():
    from core.losses import HuberLoss, MAELoss, MSELoss, SigmoidCrossEntropyLoss
    return [MSELoss(), MAELoss(), HuberLoss(0.5), SigmoidCrossEntropyLoss()]


@pytest.mark.parametrize("pred,target,match", [
    ((4, 3), (4, 2), "same shape"),
    ((4, 3), (1, 3), "same shape"),            # no broadcasting
    ((4, 3), (3,), "same shape"),
    ((4, 1), (4,), "same shape"),
    ((), (), "at least one axis"),
    ((0, 3), (0, 3), "no rows"),
    ((0,), (0,), "no rows"),
])
def test_shape_refusals(pred, target, match):
    for loss in _losses():
        with pytest.raises(ValueError, match=match):
            loss.loss(_Stub(pred), _Stub(target))


def test_dtype_refusals():
    for loss in _losses():
        for pd, td in [(np.float32, np.float64), (np.float64, np.float32), (np.int32, np.int32),
                       (np.float16, np.float16)]:
            with pytest.raises(ValueError, match="float32 or both float64"):
                loss.loss(_Stub((4, 3), pd), _Stub((4, 3), td))
        # a host array is typed as the device would hold it: integers become float64
        with pytest.raises(ValueError, match="float32 or both float64"):
            loss.loss(_Stub((4, 3), np.float32), np.zeros((4, 3), np.int64))
        with pytest.raises(ValueError, match="same shape"):
            loss.loss(_Stub((4, 3), np.float32), np.zeros((4, 2), np.float32))


def test_target_requiring_a_gradient_is_refused():
    for loss in _losses():
        with pytest.raises(ValueError, match="target requires a gradient"):
            loss.loss(_Stub((4, 3), requires_grad=True), _Stub((4, 3), requires_grad=True))
    # (the prediction may, of course)
    # a (4, 0) batch has rows and is accepted by the checks: its loss is 0 and its gradient empty
    from core.losses import MSELoss
    MSELoss()._check(_Stub((4, 0)), _Stub((4, 0)))


@pytest.mark.parametrize("delta", [0, 0.0, -1.0, float("nan"), float("inf"), -float("inf"), "1", None, True])
def test_huber_delta_refusals(delta):
    from core.losses import HuberLoss
    with pytest.raises(ValueError, match="delta"):
        HuberLoss(delta)


def test_huber_delta_is_fixed_at_construction():
    from core.losses import HuberLoss
    h = HuberLoss(np.float32(2.0))
    assert h.delta == 2.0 and type(h.delta) is float
    with pytest.raises(AttributeError):
        h.delta = 3.0
    assert HuberLoss().delta == 1.0 and HuberLoss(3).delta == 3.0


# ---------------------------------------------------------------------------- recorded-step key
def _model(loss):
    from core.layers import Dense, ReLU
    from core.model import Model
    from core.nn import Net
    from core.optimizer import SGD
    return Model(net=Net([Dense(5), ReLU(), Dense(2)]), loss=loss, optimizer=SGD(lr=0.1))


def test_step_key_distinguishes_huber_deltas():
    from core.losses import HuberLoss, MAELoss, MSELoss
    model = _model(MSELoss())
    x, y = np.zeros((8, 3), np.float32), np.zeros((8, 2), np.float32)
    k1, k1b, k2 = (model._step_key(x, y, HuberLoss(d)) for d in (1.0, 1.0, 2.0))
    assert k1 == k1b
    assert k1 != k2
    assert model._step_key(x, y, MSELoss()) == model._step_key(x, y, MSELoss())
    assert model._step_key(x, y, MSELoss()) != model._step_key(x, y, MAELoss())
    assert model._step_key(x, y, HuberLoss(1.0), "loop") != k1


def test_step_key_of_softmax_cross_entropy_is_unchanged():
    import core._dist as dist
    from core.losses import SoftmaxCrossEntropyLoss
    loss = SoftmaxCrossEntropyLoss()
    model = _model(loss)
    x, y = np.zeros((8, 3), np.float32), np.zeros((8, 2), np.float32)
    expect = ("train_step", x.shape, x.dtype.str, y.shape, y.dtype.str, dist.world_size(), id(model.optimizer),
              SoftmaxCrossEntropyLoss, id(None), model._phase,
              tuple((id(layer), type(layer)) for layer in model.net.layers))
    assert model._step_key(x, y, loss) == expect


def test_fused_small_mlp_plan_declines_pointwise_losses():
    for loss in _losses():
        model = _model(loss)
        x, y = np.zeros((8, 3), np.float32), np.zeros((8, 2), np.float32)
        assert model._fused_mlp_plan(x, y, loss) is None


# ---------------------------------------------------------------------------- data parallel scheme
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dp_problem():
    """a linear model pred = x @ w on 8 rows, per loss kind"""
    rng = np.random.RandomState(11)
    x = rng.standard_normal((8, 5))
    w = rng.standard_normal((5, 3))
    t = {"sigmoid_ce": rng.rand(8, 3)}
    base = rng.standard_normal((8, 3))
    for k in ("mse", "mae", "huber"):
        t[k] = base
    return x, w, t


def _dp_worker(rank, world, port, queue):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    for p in (ROOT, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    import torch.distributed as td
    import core._dist as dist
    import ref_losses as RL
    td.init_process_group("gloo", init_method="env://")
    try:
        x, w, t = _dp_problem()
        lo, hi = dist.shard_bounds(x.shape[0], rank, world)    # equal shards of 4
        out = {}
        for kind in RL.KINDS:
            pred = x[lo:hi] @ w
            m_global = (hi - lo) * world
            L, dp = RL.loss_and_grad(pred, t[kind][lo:hi], kind, delta=0.7, m=m_global)
            loss = torch.tensor([L])
            td.all_reduce(loss)                    # the loss node's all-reduce
            dw = torch.tensor(x[lo:hi].T @ dp)
            td.all_reduce(dw)                      # the gradient arena's SUM all-reduce
            out[kind] = (float(loss[0]), dw.numpy().copy())
        queue.put((rank, out))
    finally:
        td.destroy_process_group()


def test_sharded_losses_equal_full_batch():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    x, w, t = _dp_problem()
    for kind in RL.KINDS:
        L, dp = RL.loss_and_grad(x @ w, t[kind], kind, delta=0.7)
        dw = x.T @ dp
        for r in (0, 1):
            _close(got[r][kind][0], L)
            _close(got[r][kind][1], dw)
        assert got[0][kind][0] == got[1][kind][0]
        assert np.array_equal(got[0][kind][1], got[1][kind][1])
