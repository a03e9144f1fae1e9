"""BatchNormalization host logic without a GPU: the float64 oracle (oracle/ref_bn.py) pinned against
torch.nn.functional.batch_norm on the CPU, the layer's argument checks, the data-parallel merge of
the statistics (two ranks over gloo with oracle compute, equal to the full-batch maths) and the
checkpoint layout.  torch is test infrastructure here; nothing on the product path imports it."""
import os

import numpy as np
import pytest

import ref_bn as RB
import ref_numpy as R
from support import spawn_gloo


def _close(a, b, tol=1e-12):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape
    assert np.max(np.abs(a - b), initial=0.0) <= tol * max(1.0, np.max(np.abs(b), initial=0.0))


@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("shape", [(7, 3), (64, 1), (2, 5, 4, 6), (3, 1, 1, 8)])
def test_oracle_matches_torch(shape, training):
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    rng = np.random.RandomState(sum(shape))
    C = shape[-1]
    x = rng.standard_normal(shape) * 3.0 + 1.5
    gamma = rng.standard_normal((1, C))
    beta = rng.standard_normal((1, C))
    rm0, rv0 = rng.standard_normal(C), rng.rand(C) + 0.5
    g = rng.standard_normal(shape)
    state = RB.RefBNState(C, momentum=0.3, eps=1e-3, running_mean=rm0, running_var=rv0)
    rx, rg, rb = R.RefTensor(x, True), R.RefTensor(gamma, True), R.RefTensor(beta, True)
    y = RB.batchnorm(rx, rg, rb, state, training)
    y.backward(g)

    # torch: channels on axis 1
    perm = (0, 3, 1, 2) if len(shape) == 4 else (0, 1)
    inv = (0, 2, 3, 1) if len(shape) == 4 else (0, 1)
    tx = torch.tensor(x.transpose(perm), requires_grad=True)
    tg = torch.tensor(gamma[0], requires_grad=True)
    tb = torch.tensor(beta[0], requires_grad=True)
    trm, trv = torch.tensor(rm0), torch.tensor(rv0)
    ty = F.batch_norm(tx, trm, trv, tg, tb, training=training, momentum=0.3, eps=1e-3)
    ty.backward(torch.tensor(g.transpose(perm)))
    _close(y.values, ty.detach().numpy().transpose(inv))
    _close(state.running_mean, trm.numpy())
    _close(state.running_var, trv.numpy())
    _close(rx.grad, tx.grad.numpy().transpose(inv))
    _close(rg.grad, tg.grad.numpy()[None])
    _close(rb.grad, tb.grad.numpy()[None])
    if not training:
        assert np.array_equal(state.running_mean, rm0) and np.array_equal(state.running_var, rv0)


class _Stub(object):
    """stands in for a device tensor: shape, dtype and host values"""

    def __init__(self, arr):
        self.values = np.asarray(arr)
        self.shape = self.values.shape
        self.dtype = self.values.dtype


def _stub_bn(C, dtype=np.float32):
    from core.layers import BatchNormalization
    layer = BatchNormalization.__new__(BatchNormalization)
    layer.name, layer.grads, layer.is_training, layer.inputs = "BatchNormalization", {}, True, None
    layer.num_features, layer.momentum, layer.epsilon = C, 0.1, 1e-5
    layer.params = {"gamma": _Stub(np.arange(C, dtype=dtype)[None] + 1), "beta": _Stub(np.zeros((1, C), dtype))}
    layer.buffers = {"running_mean": _Stub(np.full((1, C), 0.25, dtype)), "running_var": _Stub(np.full((1, C), 2.0, dtype))}
    return layer


def test_layer_argument_checks():
    from core.layers import BatchNormalization
    for bad in (0, -3, 2.5, "4"):
        with pytest.raises(ValueError):
            BatchNormalization(bad)
    layer = _stub_bn(4)
    for shape in [(8, 3), (8,), (2, 3, 4), (1, 2, 2, 2, 4), (2, 5, 5, 3)]:
        with pytest.raises(ValueError, match=r"\(N, 4\) or \(N, H, W, 4\)"):
            layer.forward(_Stub(np.zeros(shape, np.float32)))
    for shape in [(1, 4), (1, 1, 1, 4), (0, 4)]:            # M < 2 in TRAIN
        with pytest.raises(ValueError, match="at least 2"):
            layer.forward(_Stub(np.zeros(shape, np.float32)))
    with pytest.raises(ValueError, match="float64.*float32|float32.*float64"):
        layer.forward(_Stub(np.zeros((8, 4), np.float64)))


def test_checkpoint_layout_holds_buffers(tmp_path):
    import pickle
    from core.layers import Dense
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import SGD
    bn = _stub_bn(3)
    model = Model(net=Net([Dense(3), bn]), loss=SoftmaxCrossEntropyLoss(), optimizer=SGD(lr=0.1))
    path = os.path.join(str(tmp_path), "bn.pkl")
    model.save(path)
    with open(path, "rb") as f:
        state = pickle.load(f)
    assert state[0] == {}
    assert list(state[1]) == ["gamma", "beta", "running_mean", "running_var"]
    assert np.array_equal(state[1]["gamma"], [[1, 2, 3]]) and np.array_equal(state[1]["running_var"], [[2, 2, 2]])


# ---------------------------------------------------------------------------- data parallel scheme
def _problem():
    rng = np.random.RandomState(0)
    x = rng.standard_normal((9, 3, 2, 5)) * 2.0 + 40.0
    g = rng.standard_normal(x.shape)
    gamma = rng.standard_normal((1, 5))
    beta = rng.standard_normal((1, 5))
    return x, g, gamma, beta


def _dp_worker(rank, world):
    import torch
    import torch.distributed as td
    import core._dist as dist
    x, g, gamma, beta = _problem()
    lo, hi = dist.shard_bounds(x.shape[0], rank, world)      # 9 images: shards of 5 and 4
    xs, gs = x[lo:hi], g[lo:hi]
    C = x.shape[-1]
    # forward: gather every rank's (count, mean, M2), merge in rank order
    n, mean, m2 = RB.local_stats(xs.reshape(-1, C))
    mine = torch.tensor(np.concatenate([[n], mean, m2]))
    gathered = [torch.zeros(1 + 2 * C, dtype=torch.float64) for _ in range(world)]
    td.all_gather(gathered, mine)
    parts = [(float(t[0]), t[1:1 + C].numpy(), t[1 + C:].numpy()) for t in gathered]
    stats = dist.merge_bn_stats_host(parts)
    state = RB.RefBNState(C, momentum=0.2)
    rx, rg, rb = R.RefTensor(xs, True), R.RefTensor(gamma, True), R.RefTensor(beta, True)
    y = RB.batchnorm(rx, rg, rb, state, True, stats=stats)

    # backward: SUM all-reduce of the two per-column sums before dx; local dgamma / dbeta
    def global_sums(dy):
        s = torch.tensor(np.concatenate(y.bn_local_sums(dy)))
        td.all_reduce(s)
        return s[:C].numpy(), s[C:].numpy()

    y.bn_vjp_x.sums = global_sums
    y.backward(gs)
    flat = torch.tensor(np.concatenate([rg.grad.ravel(), rb.grad.ravel()]))
    td.all_reduce(flat)       # the gradient arena's all-reduce completes the local partials
    return y.values, rx.grad, flat.numpy().copy(), state.running_mean, state.running_var


def test_sharded_statistics_equal_full_batch():
    got = spawn_gloo(_dp_worker)
    x, g, gamma, beta = _problem()
    state = RB.RefBNState(5, momentum=0.2)
    rx, rg, rb = R.RefTensor(x, True), R.RefTensor(gamma, True), R.RefTensor(beta, True)
    y = RB.batchnorm(rx, rg, rb, state, True)
    y.backward(g)
    flat = np.concatenate([rg.grad.ravel(), rb.grad.ravel()])
    y_dp = np.concatenate([got[0][0], got[1][0]])
    dx_dp = np.concatenate([got[0][1], got[1][1]])
    _close(y_dp, y.values)
    _close(dx_dp, rx.grad)
    for r in (0, 1):
        _close(got[r][2], flat)
        _close(got[r][3], state.running_mean)
        _close(got[r][4], state.running_var)
    # replicas agree bit for bit on what they share
    for k in (2, 3, 4):
        assert np.array_equal(got[0][k], got[1][k])


def test_host_merge_matches_direct_statistics():
    import core._dist as dist
    rng = np.random.RandomState(3)
    x = rng.standard_normal((23, 4)) + 1000.0
    parts = [RB.local_stats(x[a:b]) for a, b in ((0, 0), (0, 7), (7, 8), (8, 23))]
    n, mean, m2 = dist.merge_bn_stats_host(parts)
    assert n == 23
    _close(mean, x.mean(axis=0))
    _close(m2, ((x - x.mean(axis=0)) ** 2).sum(axis=0), tol=1e-9)
