"""Captured training step (Model.train_step -> CUDA graph replay) against the eager step.

The generic recorded step is the same arithmetic as the five lines of the reference's loop
(run.py:78-83) issued kernel by kernel: losses and parameters are compared bit for bit, across a
change of batch shape (the short last batch of an epoch), on the SIMT path (MNIST-sized layers)
and on the tcgen05 path (TMA descriptors, split-K counters and fused epilogues inside a graph).
For small Dense/ReLU MLPs train_step records the fused small-MLP pass instead (csrc/mlp_fused.cu:
other summation orders, so it is held to rounding-level agreement with the eager loop and to the
oracle / golden trajectories)."""
import numpy as np
import pytest

import ref_numpy as R
from support import gemm_route, params

pytestmark = pytest.mark.gpu


def _model(widths, seed, opt="adam", d_in=None):
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    import core.optimizer as O
    if seed is not None:
        np.random.seed(seed)
    layers = []
    dims = [d_in] + list(widths)
    for i, w in enumerate(widths):
        # with d_in the weights are drawn here (not lazily at the first forward), so two models
        # built with the same seed are identical
        layers.append(Dense(w, num_in=dims[i] if d_in is not None else None))
        if i + 1 < len(widths):
            layers.append(ReLU())
    net = Net(layers)
    optimizer = {"adam": lambda: O.Adam(lr=1e-3), "sgd": lambda: O.SGD(lr=1e-2),
                 "rmsprop": lambda: O.RMSProp(lr=1e-3), "momentum": lambda: O.Momentum(lr=1e-2)}[opt]()
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=optimizer)


def _eager(model, x, y):
    model.zero_grad()
    pred = model.forward(x)
    loss = model.loss.loss(pred, y)
    loss.backward()
    model.step()
    return loss


def _batches(n_rows, d_in, classes, sizes, seed=0):
    from core.tensor import Tensor
    rng = np.random.RandomState(seed)
    out = []
    for b in sizes:
        x = rng.rand(b, d_in).astype(np.float32)
        lab = rng.randint(0, classes, b)
        out.append((Tensor(x), Tensor(np.eye(classes)[lab])))   # float64 one-hot, as run.py:27-28
    return out


@pytest.mark.parametrize("opt", ["adam", "sgd", "rmsprop", "momentum"])
def test_captured_mnist_step_is_bit_identical(opt):
    widths = [200, 100, 70, 30, 10]
    sizes = [128] * 6 + [80, 80, 80] + [128] * 4 + [80]
    batches = _batches(0, 784, 10, sizes)
    net_a, model_a = _model(widths, 3, opt, d_in=784)
    net_b, model_b = _model(widths, 3, opt, d_in=784)
    model_b.fuse_small_mlp = False          # the layer-by-layer recording (the fused pass is tested below)
    for x, y in batches:
        la = float(_eager(model_a, x, y).values)
        lb = float(model_b.train_step(x, y).values)
        assert la == lb
    states = [s for s in model_b._captured.values()]
    assert len(states) == 2 and all(hasattr(s, "graph") for s in states)   # both shapes were recorded
    info = states[0].info()
    assert info["kernel_nodes"] >= 10 and info["blocks"] > 0
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.array_equal(pa, pb)


@pytest.mark.parametrize("label_dtype", [np.float64, np.float32])
@pytest.mark.parametrize("opt", ["adam", "sgd"])
def test_fused_small_mlp_step_matches_eager(opt, label_dtype):
    """examples/mnist network: train_step records the fused pass (first-layer product, ONE launch
    for layers 2..5 forward + global-softmax CE + backward, first-layer gradients, optimiser: 6
    kernels instead of 13).  Other summation orders than the eager loop, so: every loss within
    2e-6 relative, parameters within 1e-5 after 16 steps, across the short last batch."""
    from core.tensor import Tensor
    widths = [200, 100, 70, 30, 10]
    sizes = [128] * 6 + [80, 80, 80] + [128] * 4 + [80, 80, 80]
    rng = np.random.RandomState(0)
    batches = []
    for b in sizes:
        x = rng.rand(b, 784).astype(np.float32)
        batches.append((Tensor(x), Tensor(np.eye(10, dtype=label_dtype)[rng.randint(0, 10, b)])))
    net_a, model_a = _model(widths, 3, opt, d_in=784)
    net_b, model_b = _model(widths, 3, opt, d_in=784)
    for x, y in batches:
        la = float(_eager(model_a, x, y).values)
        lb = float(model_b.train_step(x, y).values)
        assert abs(la - lb) <= 2e-6 * abs(la), (la, lb)
    states = [s for s in model_b._captured.values()]
    assert len(states) == 2 and all(hasattr(s, "graph") for s in states)
    assert all(s.info()["kernel_nodes"] <= 8 for s in states)          # the fused pass was recorded
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.max(np.abs(pa - pb)) <= 1e-5 * np.max(np.abs(pa))


@pytest.mark.parametrize("widths,d_in,batch", [([50, 33, 7], 20, 37), ([64, 10], 32, 16), ([256, 128, 3], 9, 130)])
def test_fused_small_mlp_other_shapes(widths, d_in, batch):
    """batches that are not a multiple of the 4 rows a CTA takes, widths up to the 256 limit, a
    two-Dense network (tail of one layer)"""
    from core.tensor import Tensor
    rng = np.random.RandomState(4)
    net_a, model_a = _model(widths, 6, d_in=d_in)
    net_b, model_b = _model(widths, 6, d_in=d_in)
    for _ in range(6):
        x = Tensor(rng.standard_normal((batch, d_in)).astype(np.float32))
        y = Tensor(np.eye(widths[-1], dtype=np.float32)[rng.randint(0, widths[-1], batch)])
        la = float(_eager(model_a, x, y).values)
        lb = float(model_b.train_step(x, y).values)
        assert abs(la - lb) <= 2e-6 * abs(la), (la, lb)
    assert all(s.info()["kernel_nodes"] <= 8 for s in model_b._captured.values() if hasattr(s, "graph"))
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.max(np.abs(pa - pb)) <= 1e-5 * np.max(np.abs(pa))


def test_fused_small_mlp_is_not_used_where_it_does_not_apply():
    """a Tanh in the stack, a tail too wide for shared memory, or a subclassed loss: train_step
    records the generic step (and still equals the eager loop bit for bit)"""
    from core.layers import Dense, ReLU, Tanh
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    from core.tensor import Tensor

    class MyLoss(SoftmaxCrossEntropyLoss):
        pass

    rng = np.random.RandomState(1)
    x = Tensor(rng.rand(32, 24).astype(np.float32))
    y = Tensor(np.eye(6, dtype=np.float32)[rng.randint(0, 6, 32)])
    for make, loss in ((lambda: [Dense(16, num_in=24), Tanh(), Dense(6, num_in=16)], SoftmaxCrossEntropyLoss()),
                       (lambda: [Dense(300, num_in=24), ReLU(), Dense(6, num_in=300)], SoftmaxCrossEntropyLoss()),
                       (lambda: [Dense(16, num_in=24), ReLU(), Dense(6, num_in=16)], MyLoss())):
        out = []
        for use_graph in (False, True):
            np.random.seed(2)
            net = Net(make())
            model = Model(net=net, loss=loss, optimizer=Adam(lr=1e-3))
            losses = [float((model.train_step(x, y) if use_graph else _eager(model, x, y)).values)
                      for _ in range(5)]
            out.append((losses, params(net)))
            if use_graph:
                assert model._fused_mlp_plan(x, y) is None
        assert out[0][0] == out[1][0]
        for pa, pb in zip(out[0][1], out[1][1]):
            assert np.array_equal(pa, pb)


def test_fused_small_mlp_holds_the_reference_trajectory(golden_dir):
    """north_star's 100-step loss trajectory within 1e-4 of the real reference's, on the recorded
    fused path, free running: BatchIterator (same shuffle draw, before the lazy weight init) ->
    train_step, on the random-label golden (measured 1.5e-6)."""
    import os
    from core.tensor import Tensor
    from utils.data_iterator import BatchIterator
    gold = np.load(os.path.join(golden_dir, "mnist_traj.npz"))["losses"]
    np.random.seed(0)
    x, y, onehot = R.synthetic_mnist(12800, seed=0)
    net, model = _model([200, 100, 70, 30, 10], None)      # seed stays: weights are drawn lazily
    losses = []
    for batch in BatchIterator(batch_size=128)(Tensor(x), Tensor(onehot)):
        losses.append(float(model.train_step(batch.inputs, batch.targets).values))
        if len(losses) == 100:
            break
    assert any(hasattr(s, "graph") and s.info()["kernel_nodes"] <= 8 for s in model._captured.values())
    diff = np.abs(np.array(losses) - gold)
    assert np.max(diff) <= 1e-4, (int(np.argmax(diff)), float(np.max(diff)))


def test_fused_small_mlp_teacher_forced_on_learnable_data():
    """The learnable golden is held by the eager engine free running (test_gpu_train.py: 7e-7).  The
    fused pass sums in another order; on this data one near-zero ReLU pre-activation lands on the
    other side of the kink at step 13 and the two runs then follow different (equally valid) float32
    trajectories, so the fused pass is held to the eager step with teacher forcing instead (SURVEY
    7.3): before each of 40 steps it gets the eager model's parameters and Adam state; loss within
    1e-6 relative and every parameter within 1e-6 of max|p| after the step (measured 1e-7)."""
    import core._backend as be
    import ref_fp32
    from core.tensor import Tensor
    x, y, onehot = ref_fp32.learnable_mnist(128 * 40, seed=0)
    net_a, a = _model([200, 100, 70, 30, 10], 0, d_in=784)
    net_b, b = _model([200, 100, 70, 30, 10], 0, d_in=784)
    compared = 0
    for k in range(40):
        xb, yb = Tensor(x[k * 128:(k + 1) * 128]), Tensor(onehot[k * 128:(k + 1) * 128])
        if a._arena is not None and b._arena is not None:
            be.copy_into(b._arena["p"], a._arena["p"])
            for sb, sa in zip(b.optimizer._state, a.optimizer._state):
                be.copy_into(sb, sa)
            b.optimizer._t = a.optimizer._t
            for p in b._arena["params"]:
                p._touch()
        la = float(_eager(a, xb, yb).values)
        lb = float(b.train_step(xb, yb).values)
        assert abs(la - lb) <= 1e-6 * abs(la), (k, la, lb)
        if k >= 2:                                   # from the third call on the fused recording runs
            compared += 1
            for pa, pb in zip(params(net_a), params(net_b)):
                assert np.max(np.abs(pa - pb)) <= 1e-6 * np.max(np.abs(pa)), k
    assert compared == 38 and any(hasattr(s, "graph") and s.info()["kernel_nodes"] <= 8
                                  for s in b._captured.values())


def test_captured_tensor_core_step_is_bit_identical():
    """256-wide layers at batch 1024: every product is above the tensor-core threshold"""
    import core._backend as be
    widths = [256, 256, 256]
    with gemm_route(TC_MIN_MNK=1 << 26):
        assert be.use_tensor_cores(1024, 256, 256, be.F32)
        batches = _batches(0, 256, 256, [1024] * 6)
        net_a, model_a = _model(widths, 5, d_in=256)
        net_b, model_b = _model(widths, 5, d_in=256)
        for x, y in batches:
            la = float(_eager(model_a, x, y).values)
            lb = float(model_b.train_step(x, y).values)
            assert la == lb
        for pa, pb in zip(params(net_a), params(net_b)):
            assert np.array_equal(pa, pb)


def test_replay_does_not_touch_other_tensors():
    """blocks a recorded step uses stay out of the pool: tensors made between replays survive"""
    from core.tensor import Tensor
    widths = [64, 10]
    batches = _batches(0, 32, 10, [16] * 8)
    net, model = _model(widths, 1)
    keep, expect = [], []
    rng = np.random.RandomState(9)
    for i, (x, y) in enumerate(batches):
        model.train_step(x, y)
        for shape in ((16, 64), (16, 10), (32, 64), (1, 64), (16,)):
            a = rng.rand(*shape).astype(np.float32)
            t = Tensor(a) + 0.0      # result block comes from the pool
            keep.append(t)
            expect.append(a)
    for t, a in zip(keep, expect):
        t._host = None
        assert np.array_equal(t.values, a)


def test_captured_step_loss_copies_are_independent():
    batches = _batches(0, 32, 10, [16] * 6)
    net, model = _model([64, 10], 2)
    held = [model.train_step(x, y) for x, y in batches]
    vals = [float(t.values) for t in held]
    assert len(set(vals)) == len(vals)      # not all aliases of the graph's loss buffer


def test_captured_step_tracks_oracle_trajectory():
    """the replayed MNIST-MLP loop against the oracle's 20-step trajectory: same initial weights
    (np.random.seed(0) draw order), float32 engine vs the oracle's float64 path, rel 1e-4"""
    from core.tensor import Tensor
    x, y, onehot = R.synthetic_mnist(2560, seed=0)
    widths = [200, 100, 70, 30, 10]
    np.random.seed(0)
    mlp = R.RefMLP(widths, R.RefAdam(lr=1e-3))
    want = [float(mlp.train_step(x[i * 128:(i + 1) * 128], onehot[i * 128:(i + 1) * 128]))
            for i in range(20)]
    net, model = _model(widths, 0)
    got = []
    for i in range(20):
        xb, yb = Tensor(x[i * 128:(i + 1) * 128]), Tensor(onehot[i * 128:(i + 1) * 128])
        got.append(float(model.train_step(xb, yb).values))
    assert hasattr(list(model._captured.values())[0], "graph")
    assert np.max(np.abs(np.array(got) - np.array(want)) / np.abs(want)) < 1e-4


def test_host_transfer_inside_capture_fails_loudly():
    import core._backend as be
    g = be.StepGraph()
    with pytest.raises(be.BackendError):
        with g.capture():
            be.from_numpy(np.ones(4, dtype=np.float32))
    # the aborted capture left the stream usable
    a = be.from_numpy(np.arange(4, dtype=np.float32))
    assert np.array_equal(be.to_numpy(be.ew(be.ADD, a, a)), 2 * np.arange(4, dtype=np.float32))


def test_graph_destroyed_during_another_capture_is_deferred():
    """a recorded step released while a second capture is running (the garbage collector can do
    that) must not synchronise the stream: its destruction waits for the capture to end"""
    import core._backend as be
    a = be.from_numpy(np.arange(8, dtype=np.float32))
    g1 = be.StepGraph()
    with g1.capture():
        b = be.ew(be.ADD, a, a)
    g1.replay()
    assert np.array_equal(be.to_numpy(b), 2 * np.arange(8, dtype=np.float32))
    g2 = be.StepGraph()
    with g2.capture():
        c = be.ew(be.MUL, a, a)
        g1.destroy()                       # in the middle of g2's capture
        d = be.ew(be.ADD, c, a)
    g2.replay()
    x = np.arange(8, dtype=np.float32)
    assert np.array_equal(be.to_numpy(d), x * x + x)
    g2.destroy()


def test_recorded_step_is_dropped_when_a_parameter_is_rebound():
    """p.values = ... moves a parameter out of the arena a recorded step names: the next
    train_step must notice, fall back to the eager lines and record again -- same numbers as a
    model that never used a graph"""
    batches = _batches(0, 32, 10, [16] * 10)
    net_a, model_a = _model([64, 10], 7, d_in=32)
    net_b, model_b = _model([64, 10], 7, d_in=32)
    model_b.fuse_small_mlp = False
    for i, (x, y) in enumerate(batches):
        if i == 5:
            for net in (net_a, net_b):
                w = net.layers[0].params["w"]
                w.values = w.values * 0.5
                w.zero_grad()
        la = float(_eager(model_a, x, y).values)
        lb = float(model_b.train_step(x, y).values)
        assert la == lb, i
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.array_equal(pa, pb)
    assert any(hasattr(s, "graph") for s in model_b._captured.values())
