"""BatchNormalization on the device (csrc/batchnorm.cu) against the float64 oracle of
oracle/ref_bn.py: y, dx, dgamma, dbeta and the running statistics over a grid of channel counts, row
counts (up to many split CTAs), layouts, phases and dtypes; offset data, a constant channel, the
empty TEST batch, reproducibility, accumulation into an arena slot; and a small CNN with two
BatchNormalization layers trained eagerly, through the recorded train_step and the recorded
five-line loop, predicted in the TEST phase and checkpointed."""
import os

import numpy as np
import pytest

import ref_bn as RB
import ref_conv as RC
import ref_fp32
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


def _layer(C, dtype, gamma, beta, rm, rv, momentum=0.1, eps=1e-5):
    from core.layers import BatchNormalization
    from core.tensor import Tensor
    layer = BatchNormalization(C, momentum=momentum, epsilon=eps)
    layer.params["gamma"] = Tensor(gamma, requires_grad=True, dtype=dtype)
    layer.params["beta"] = Tensor(beta, requires_grad=True, dtype=dtype)
    for p in layer.params.values():
        p.zero_grad()
    layer.buffers["running_mean"].values = np.asarray(rm, dtype).reshape(1, C)
    layer.buffers["running_var"].values = np.asarray(rv, dtype).reshape(1, C)
    return layer


def _bn_case(shape, dtype, training, seed, x=None, slots=None):
    """device forward + backward with a random upstream gradient, and the oracle's.  `slots`: prior
    gradients for gamma and beta held in arena-style slots, which the fused backward accumulates into."""
    from core.tensor import Tensor
    rng = np.random.RandomState(seed)
    C = shape[-1]
    if x is None:
        x = (rng.standard_normal(shape) * 2.0 + 0.5).astype(dtype)
    gamma = rng.standard_normal((1, C)).astype(dtype)
    beta = rng.standard_normal((1, C)).astype(dtype)
    rm, rv = rng.standard_normal(C).astype(dtype), (rng.rand(C) + 0.5).astype(dtype)
    g = rng.standard_normal(shape).astype(dtype)
    layer = _layer(C, dtype, gamma, beta, rm, rv)
    layer.set_phase("TRAIN" if training else "TEST")
    if slots is not None:
        import core._backend as be
        for k, prior in zip(("gamma", "beta"), slots):
            p = layer.params[k]
            p._gslot = be.from_numpy(np.asarray(prior, dtype))
            p._grad, p._grad_zero = p._gslot, False
    tx = Tensor(x, requires_grad=True, dtype=dtype)
    tx.zero_grad()
    y = layer.forward(tx)
    y.backward(g)
    state = RB.RefBNState(C, running_mean=rm, running_var=rv)
    rx, rg, rb = R.RefTensor(x, True), R.RefTensor(gamma, True), R.RefTensor(beta, True)
    ry = RB.batchnorm(rx, rg, rb, state, training)
    ry.backward(g.astype(np.float64))
    got = dict(y=y.values, dx=tx.grad, dgamma=layer.params["gamma"].grad, dbeta=layer.params["beta"].grad,
               running_mean=layer.buffers["running_mean"].values[0],
               running_var=layer.buffers["running_var"].values[0])
    ref = dict(y=ry.values, dx=rx.grad, dgamma=rg.grad, dbeta=rb.grad, running_mean=state.running_mean,
               running_var=state.running_var)
    if slots is not None:
        ref["dgamma"] = ref["dgamma"] + slots[0]
        ref["dbeta"] = ref["dbeta"] + slots[1]
    # dx can vanish analytically (M = 2 in TRAIN): measure it against the size of gamma * r * dy
    var = state.running_var if not training else x.reshape(-1, C).astype(np.float64).var(axis=0)
    floors = dict(dx=np.max(np.abs(g), initial=0.0) * np.max(np.abs(gamma) / np.sqrt(var + 1e-5), initial=0.0))
    return got, ref, floors, rm, rv


def _check(got, ref, floors, tol, what):
    for k in ("y", "dx", "dgamma", "dbeta", "running_mean", "running_var"):
        assert got[k].shape == ref[k].shape, (k, what)
        e = _err(got[k], ref[k], floors.get(k, 0.0))
        assert e <= tol, (k, what, e)


CHANNELS = [1, 3, 8, 64, 130]
SHAPES = [(2,), (37,), (3001,), (20000,), (2, 1, 1), (3, 5, 7), (16, 12, 10)]   # leading axes: M rows


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("lead", SHAPES)
def test_batchnorm_matches_oracle(be, lead, training, dtype):
    tol = 1e-5 if dtype == np.float32 else 1e-12
    for C in CHANNELS:
        got, ref, floors, _, _ = _bn_case(lead + (C,), dtype, training, seed=C * 7 + len(lead))
        _check(got, ref, floors, tol, (lead, C))
        assert got["y"].dtype == dtype and got["dx"].dtype == dtype


def test_batchnorm_full_size_float32(be):
    got, ref, floors, _, _ = _bn_case((256, 32, 32, 64), np.float32, True, seed=1)
    _check(got, ref, floors, 1e-5, "256x32x32x64")


def test_batchnorm_offset_data_float32(be):
    """x = 1000 + N(0, 1): a float32 one-pass sum of squares would lose the variance entirely"""
    rng = np.random.RandomState(2)
    x = (1000.0 + rng.standard_normal((64, 16, 16, 8))).astype(np.float32)
    got, ref, floors, _, _ = _bn_case(x.shape, np.float32, True, seed=2, x=x)
    assert _err(got["y"], ref["y"]) <= 1e-5
    assert _err(got["running_var"], ref["running_var"]) <= 1e-5
    assert _err(got["running_mean"], ref["running_mean"]) <= 1e-5


def test_batchnorm_constant_channel(be):
    """sigma^2 = 0: y = beta exactly and every gradient finite"""
    for dtype in (np.float32, np.float64):
        rng = np.random.RandomState(4)
        x = rng.standard_normal((300, 5)).astype(dtype)
        x[:, 2] = 3.0
        got, ref, floors, _, _ = _bn_case(x.shape, dtype, True, seed=4, x=x)
        beta = ref["y"][0, 2]
        assert np.all(got["y"][:, 2] == got["y"][0, 2]) and abs(got["y"][0, 2] - beta) <= 1e-6 * max(1, abs(beta))
        for k in ("dx", "dgamma", "dbeta"):
            assert np.all(np.isfinite(got[k])), k
        tol = 1e-5 if dtype == np.float32 else 1e-12
        for k in ("dbeta", "running_mean", "running_var"):
            assert _err(got[k], ref[k]) <= tol, k


def test_batchnorm_empty_batch_in_test_phase(be):
    for shape in [(0, 5), (0, 4, 4, 5)]:
        got, ref, floors, rm, rv = _bn_case(shape, np.float32, False, seed=5)
        assert got["y"].shape == shape and got["dx"].shape == shape
        assert np.all(got["dgamma"] == 0) and np.all(got["dbeta"] == 0)
        assert np.array_equal(got["running_mean"], rm) and np.array_equal(got["running_var"], rv)


def test_batchnorm_is_bit_reproducible(be):
    for training in (True, False):
        a = _bn_case((12, 9, 11, 64), np.float32, training, seed=6)[0]
        b = _bn_case((12, 9, 11, 64), np.float32, training, seed=6)[0]
        for k in a:
            assert np.array_equal(a[k], b[k]), (k, training)


def test_batchnorm_accumulates_into_a_slot(be):
    """gamma / beta in arena-style slots that already hold a gradient: the fold adds to them"""
    rng = np.random.RandomState(7)
    for dtype, tol in ((np.float32, 1e-5), (np.float64, 1e-12)):
        for training in (True, False):
            prior = (rng.standard_normal((1, 12)), rng.standard_normal((1, 12)))
            got, ref, floors, _, _ = _bn_case((500, 12), dtype, training, seed=8, slots=prior)
            _check(got, ref, floors, tol, (dtype, training))


def test_single_rank_merge_path_equals_direct_statistics(be):
    """the data-parallel route (local (count, mean, M2) + the device merge) on one rank gives the
    statistics of the direct route to rounding"""
    import core._dist as dist
    rng = np.random.RandomState(9)
    x = be.from_numpy((rng.standard_normal((4000, 24)) * 3 + 7).astype(np.float32))
    rm_a, rv_a = be.zeros((1, 24), be.F32), be.full((1, 24), 1.0, be.F32)
    rm_b, rv_b = be.zeros((1, 24), be.F32), be.full((1, 24), 1.0, be.F32)
    mr_a = be.bn_stats(x, 0.1, 1e-5, rm_a, rv_a).numpy()
    mr_b = dist.bn_global_stats(x, 0.1, 1e-5, rm_b, rv_b).numpy()
    assert mr_a[-1] == mr_b[-1] == 4000
    np.testing.assert_allclose(mr_b, mr_a, rtol=1e-13)
    np.testing.assert_allclose(rv_b.numpy(), rv_a.numpy(), rtol=1e-6)


# ---------------------------------------------------------------------------- small MNIST CNN
def _cnn(seed, optimizer=None):
    from core.layers import BatchNormalization, Conv2D, Dense, Flatten, MaxPool2D, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    np.random.seed(seed)
    net = Net([Conv2D((5, 5, 1, 8), stride=2), BatchNormalization(8), ReLU(), MaxPool2D(),
               Conv2D((3, 3, 8, 16)), BatchNormalization(16), ReLU(), Flatten(), Dense(10, num_in=7 * 7 * 16)])
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=optimizer or Adam(lr=1e-3))


def _data(n):
    x, _, onehot = ref_fp32.learnable_mnist(n, seed=0)
    return x.reshape(n, 28, 28, 1), onehot


def _buffers(net):
    return [b.values.copy() for layer in net.layers for b in layer.buffers.values()]


class _RefCNN(object):
    """the same network in the float64 oracle, starting from the engine model's parameters and
    running statistics"""

    def __init__(self, net):
        self.p = [R.RefTensor(v, True) for v in params(net)]
        bufs = _buffers(net)
        self.st = [RB.RefBNState(8, running_mean=bufs[0], running_var=bufs[1]),
                   RB.RefBNState(16, running_mean=bufs[2], running_var=bufs[3])]
        self.opt = R.RefAdam(lr=1e-3)

    def forward(self, x, training=True):
        w1, b1, g1, be1, w2, b2, g2, be2, w3, b3 = self.p
        h = RC.conv2d(R.lift(x), w1, b1, (2, 2), "SAME")
        h = R.clip(RB.batchnorm(h, g1, be1, self.st[0], training), 0.0)
        h = RC.maxpool2d(h, (2, 2))
        h = RC.conv2d(h, w2, b2, (1, 1), "SAME")
        h = R.clip(RB.batchnorm(h, g2, be2, self.st[1], training), 0.0)
        h = R.reshape(h, (x.shape[0], -1))
        return R.matmul(h, w3) + b3

    def step(self, x, y):
        for p in self.p:
            p.zero_grad()
        loss = R.softmax_cross_entropy(self.forward(x), y)
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
    assert len(grads) == 10 and grads[2].shape == (1, 8) and grads[6].shape == (1, 16)
    # a conv bias that feeds a BatchNormalization has gradient 0 analytically (the batch mean absorbs
    # it): measure what rounding leaves there against its conv weight's gradient
    floors = {1: np.max(np.abs(rgrads[0])), 5: np.max(np.abs(rgrads[4]))}
    for i, (g, rg) in enumerate(zip(grads, rgrads)):
        assert _err(g, rg, floors.get(i, 0.0)) <= 1e-5, (i, _err(g, rg, floors.get(i, 0.0)))
    rbufs = [ref.st[0].running_mean, ref.st[0].running_var, ref.st[1].running_mean, ref.st[1].running_var]
    for b, rb in zip(_buffers(net), rbufs):
        assert _err(b[0], rb) <= 1e-5


def test_cnn_loss_trajectory_matches_oracle(be):
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
    # the running variances follow the oracle's.  The running means are not compared: the conv biases
    # before each BatchNormalization get rounding-level gradients (0 analytically), which Adam's
    # normalised step turns into lr-sized moves, and the batch means -- not the loss -- follow them
    for b, rb in zip(_buffers(net)[1::2], [ref.st[0].running_var, ref.st[1].running_var]):
        assert _err(b[0], rb) <= 1e-4


def test_cnn_train_step_replay_is_bit_identical(be):
    """train_step records the layer-by-layer step (the fused small-MLP plan declines this network);
    replays give the eager bits, running statistics included, across a change of batch shape"""
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
        assert float(_eager(model_a, xb, yb).values) == float(model_b.train_step(xb, yb).values)
        for ba, bb in zip(_buffers(net_a), _buffers(net_b)):
            assert np.array_equal(ba, bb)
    assert len([s for s in model_b._captured.values() if hasattr(s, "graph")]) == 2
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.array_equal(pa, pb)
    # TRAIN and TEST recordings are kept apart
    keys = [k for k in model_b._captured]
    assert all(k[9] == "TRAIN" for k in keys)


def test_cnn_five_line_loop_recording_is_bit_identical(be):
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
            loss = loss_layer.loss(model.forward(xb), yb)
            loss.backward()
            model.step()
            losses.append(float(loss.values))
        out.append(losses)
    assert out[0] == out[1]
    assert [s for s in model_b._captured.values() if hasattr(s, "graph")]
    for pa, pb in zip(params(net_a) + _buffers(net_a), params(net_b) + _buffers(net_b)):
        assert np.array_equal(pa, pb)


def test_cnn_test_phase_prediction_uses_running_statistics(be):
    from core.tensor import Tensor
    x, y = _data(256)
    net, model = _cnn(5)
    for i in range(3):
        model.train_step(Tensor(x[:128]), Tensor(y[:128]))
    model.set_phase("TEST")
    before = _buffers(net)
    pred = model.predict(Tensor(x[128:]))
    assert all(np.array_equal(a, b) for a, b in zip(before, _buffers(net)))
    ref = _RefCNN(net)
    rpred = ref.forward(x[128:], training=False).values
    assert _err(pred.values, rpred) <= 1e-5
    # a batch of one is fine in TEST
    assert model.predict(Tensor(x[:1])).shape == (1, 10)
    model.set_phase("TRAIN")
    # the phase decides, not the grad mode: a TRAIN-phase predict updates the statistics
    model.predict(Tensor(x[:64]))
    assert not np.array_equal(before[0], _buffers(net)[0])


def test_cnn_checkpoint_round_trip_and_replay_from_loaded_statistics(be, tmp_path):
    """save writes gamma, beta, running_mean, running_var per BatchNormalization; load copies the
    statistics into the existing device arrays; recorded steps afterwards continue from them"""
    import pickle
    from core.optimizer import SGD
    from core.tensor import Tensor
    x, y = _data(128 * 9)
    batches = [(Tensor(x[i * 128:(i + 1) * 128]), Tensor(y[i * 128:(i + 1) * 128])) for i in range(9)]
    net_a, model_a = _cnn(6, SGD(lr=0.05))
    for xb, yb in batches[:3]:
        model_a.train_step(xb, yb)
    path = os.path.join(str(tmp_path), "bn_cnn.pkl")
    model_a.save(path)
    with open(path, "rb") as f:
        state = pickle.load(f)
    assert list(state[1]) == ["gamma", "beta", "running_mean", "running_var"]
    saved = params(net_a) + _buffers(net_a)
    for xb, yb in batches[3:6]:
        model_a.train_step(xb, yb)
    bufs = [b._data for layer in net_a.layers for b in layer.buffers.values()]
    model_a.load(path)
    assert [b._data for layer in net_a.layers for b in layer.buffers.values()] == bufs   # in place
    for a, b in zip(params(net_a) + _buffers(net_a), saved):
        assert np.array_equal(a, b)
    net_b, model_b = _cnn(7, SGD(lr=0.05))
    model_b.load(path)
    for a, b in zip(params(net_b) + _buffers(net_b), saved):
        assert np.array_equal(a, b)
    for xb, yb in batches[6:]:
        la = float(model_a.train_step(xb, yb).values)
        lb = float(_eager(model_b, xb, yb).values)
        assert la == lb
    assert [s for s in model_a._captured.values() if hasattr(s, "graph")]
    for a, b in zip(params(net_a) + _buffers(net_a), params(net_b) + _buffers(net_b)):
        assert np.array_equal(a, b)


# ---------------------------------------------------------------------------- two ranks
def test_two_rank_batchnorm_equals_full_batch_oracle():
    if gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    assert "BN_DIST_OK world=2" in run_two_ranks("bn_dist_worker.py", timeout=200)
