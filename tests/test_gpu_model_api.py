"""Model / optimiser interface behaviours around the fused arena step: the reference's extension
points keep working (core/optimizer.py:12-38, core/model.py:45-61), gradients assigned by user code
are honoured, weight decay is opt-in, host views are read-only, reference-format checkpoints load."""
import os

import numpy as np
import pytest

import op_cases
import ref_numpy as R
from support import params

pytestmark = pytest.mark.gpu


def _mlp(widths, optimizer):
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    layers = []
    for i, w in enumerate(widths):
        layers.append(Dense(w))
        if i + 1 < len(widths):
            layers.append(ReLU())
    net = Net(layers)
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=optimizer)


def _pair(widths, optimizer, ref_optimizer, seed, x):
    """engine model and oracle MLP with the same reference-style initial parameters (both draw from
    numpy's global RNG at their first forward, so each gets its own freshly seeded stream)"""
    from core.tensor import Tensor
    np.random.seed(seed)
    net, model = _mlp(widths, optimizer)
    model.forward(Tensor(x))
    np.random.seed(seed)
    ref = R.RefMLP(widths, ref_optimizer)
    ref.forward(R.lift(x))
    for p, rp in zip(_param_tensors(net), ref.params()):
        assert np.array_equal(p.values, rp.values)
    return net, model, ref


def _data(seed=2, B=16, D=20, C=10):
    rng = np.random.RandomState(seed)
    return rng.rand(B, D).astype(np.float32), np.eye(C, dtype=np.float32)[rng.randint(0, C, B)]


def _param_tensors(net):
    return [p for layer in net.get_parameters() for p in layer.values()]


def _one_step(model, x, y):
    from core.tensor import Tensor
    model.zero_grad()
    loss = model.loss.loss(model.forward(Tensor(x)), Tensor(y))
    loss.backward()
    model.step()
    return float(loss.values)


def test_user_defined_optimizer_is_called():
    """an optimiser written against the reference's contract -- subclass BaseOptimizer, implement
    _compute_step(flat numpy-like gradient) -> flat step -- must drive Model.step (ADVICE r1)"""
    from core.optimizer import BaseOptimizer

    class SignSGD(BaseOptimizer):
        calls = 0

        def __init__(self, lr):
            super().__init__(lr, 0.0)

        def _compute_step(self, grad):
            SignSGD.calls += 1
            g = grad.numpy() if hasattr(grad, "numpy") else np.asarray(grad)
            return -self.lr * np.sign(g)          # a plain numpy array, as in the reference

    x, y = _data()
    np.random.seed(3)
    net, model = _mlp([13, 10], SignSGD(lr=0.01))
    model.forward(__import__("core.tensor", fromlist=["Tensor"]).Tensor(x))
    before = params(net)
    from core.tensor import Tensor
    model.zero_grad()
    loss = model.loss.loss(model.forward(Tensor(x)), Tensor(y))
    loss.backward()
    grads = [p.grad.copy() for p in _param_tensors(net)]
    model.step()
    assert SignSGD.calls == 1
    for b, g, p in zip(before, grads, _param_tensors(net)):
        assert np.allclose(p.values, b - 0.01 * np.sign(g), atol=1e-7)


def test_subclass_overriding_compute_step_is_not_bypassed():
    """a subclass of a built-in rule that post-processes the step (here: clips it) is honoured for
    every step, and its Adam state stays consistent although bias sizes are not multiples of 64"""
    from core.optimizer import Adam

    class ClippedAdam(Adam):
        def _compute_step(self, grad):
            step = super()._compute_step(grad)
            return np.clip(step.numpy(), -5e-4, 5e-4)

    x, y = _data()
    net, model, ref = _pair([13, 7, 10], ClippedAdam(lr=1e-3), R.RefAdam(lr=1e-3), 3, x)
    for _ in range(3):
        _one_step(model, x, y)
        ref.zero_grad()
        R.softmax_cross_entropy(ref.forward(R.lift(x)), y).backward()
        params = ref.params()
        for p, s in zip(params, ref.optimizer.compute_steps(params)):
            p.assign((p.values + np.clip(s, -5e-4, 5e-4)).astype(np.float32))
    for p, rp in zip(_param_tensors(net), ref.params()):
        assert op_cases.rel_err(p.values, rp.values) <= 1e-5


def test_assigned_gradient_stays_on_the_fused_path():
    """`p.grad = clipped` between backward() and step() (ordinary gradient clipping): the step uses
    the assigned gradient and the fused Adam state carries over (ADVICE r1: this used to fall to the
    generic path and raise on the padded state)"""
    from core.optimizer import Adam
    from core.tensor import Tensor
    x, y = _data()
    net, model, ref = _pair([13, 7, 10], Adam(lr=1e-3), R.RefAdam(lr=1e-3), 5, x)
    for it in range(4):
        model.zero_grad()
        loss = model.loss.loss(model.forward(Tensor(x)), Tensor(y))
        loss.backward()
        ref.zero_grad()
        R.softmax_cross_entropy(ref.forward(R.lift(x)), y).backward()
        if it >= 1:                                  # the arenas exist from the first step on
            for p in _param_tensors(net):
                p.grad = np.clip(p.grad, -1e-3, 1e-3)
            for rp in ref.params():
                rp.grad = np.clip(rp.grad, -1e-3, 1e-3)
        model.step()
        assert model._arena is not None and all(p._gslot is not None for p in _param_tensors(net))
        ref.step()
        for rp in ref.params():
            rp.assign(rp.values.astype(np.float32).astype(np.float64))
    for p, rp in zip(_param_tensors(net), ref.params()):
        assert op_cases.rel_err(p.values, rp.values) <= 1e-5


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("name", ["sgd", "adam", "momentum"])
def test_weight_decay_is_opt_in(name, fused):
    """optimizer.py:28-29: weight_decay is accepted and ignored (the reference's line is commented
    out); with apply_weight_decay = True the line `_step -= weight_decay * v` is applied -- in the
    fused kernel and on the compute_step path alike"""
    import core.optimizer as O
    make = {"sgd": lambda: O.SGD(lr=0.05, weight_decay=0.1),
            "adam": lambda: O.Adam(lr=1e-3, weight_decay=0.1),
            "momentum": lambda: O.Momentum(lr=0.02, weight_decay=0.1)}[name]
    rmake = {"sgd": lambda: R.RefSGD(0.05), "adam": lambda: R.RefAdam(1e-3),
             "momentum": lambda: R.RefMomentum(0.02)}[name]
    x, y = _data()
    for apply in (False, True):
        opt = make()
        opt.apply_weight_decay = apply
        net, model, ref = _pair([13, 10], opt, rmake(), 7, x)
        for _ in range(3):
            if fused:
                _one_step(model, x, y)
            else:
                from core.tensor import Tensor
                model.zero_grad()
                model.loss.loss(model.forward(Tensor(x)), Tensor(y)).backward()
                model._step_generic()
            ref.zero_grad()
            R.softmax_cross_entropy(ref.forward(R.lift(x)), y).backward()
            params = ref.params()
            for p, s in zip(params, ref.optimizer.compute_steps(params)):
                if apply:
                    s = s - 0.1 * p.values
                p.assign((p.values + s).astype(np.float32))
        for p, rp in zip(_param_tensors(net), ref.params()):
            assert op_cases.rel_err(p.values, rp.values) <= 1e-5, (name, apply)


def test_host_views_are_read_only():
    """.values / .grad are host copies; an in-place edit could never reach the device, so it must
    fail loudly (the reference hands out live arrays, tensor.py:20,31-33)"""
    from core.tensor import Tensor
    t = Tensor(np.arange(6, dtype=np.float32).reshape(2, 3), requires_grad=True)
    with pytest.raises(ValueError):
        t.values[0, 0] = 5.0
    with pytest.raises(ValueError):
        t.grad[0, 0] = 1.0
    (t * 2.0).sum().backward()
    with pytest.raises(ValueError):
        t.grad *= 0.5            # numpy refuses the in-place multiply on the read-only array
    with pytest.raises(ValueError):
        np.clip(t.grad, -1, 1, out=t.grad)
    # the setters are the way in
    t.grad = t.grad * 0.5
    assert t.grad.tolist() == [[1.0, 1.0, 1.0], [1.0, 1.0, 1.0]]
    t.values = t.values + 1.0
    assert t.values[0, 0] == 1.0 and t.grad is None


def test_reference_format_checkpoint_loads(golden_dir):
    """a file written by the reference's Model.save (the pickled Net, model.py:18-21) restores the
    same forward values here, also into a lazily initialised network"""
    from core.optimizer import Adam
    from core.tensor import Tensor
    io = np.load(os.path.join(golden_dir, "ref_checkpoint_io.npz"))
    np.random.seed(1)
    net, model = _mlp([3, 2], Adam())
    model.load(os.path.join(golden_dir, "ref_checkpoint.pkl"))      # layers not initialised yet
    assert net.layers[0].shapes["w"] == [4, 3]
    out = model.forward(Tensor(io["x"]))
    assert op_cases.rel_err(out.values, io["y"]) <= 1e-6
    np.random.seed(2)
    net2, model2 = _mlp([3, 2], Adam())
    model2.forward(Tensor(io["x"]))                                  # initialised with other values
    model2.load(os.path.join(golden_dir, "ref_checkpoint.pkl"))
    assert op_cases.rel_err(model2.forward(Tensor(io["x"])).values, io["y"]) <= 1e-6
    np.random.seed(3)
    net3, model3 = _mlp([5, 2], Adam())
    model3.forward(Tensor(io["x"]))
    with pytest.raises(ValueError):
        model3.load(os.path.join(golden_dir, "ref_checkpoint.pkl"))


def test_failed_capture_falls_back_to_eager():
    """train_step with a loss that reads a device value on the host while the step is being
    recorded: the recording is abandoned, this and later batches run eagerly, results unchanged"""
    from core.losses import SoftmaxCrossEntropyLoss
    from core.optimizer import Adam
    from core.tensor import Tensor

    class PeekingLoss(SoftmaxCrossEntropyLoss):
        def loss(self, predicted, actual):
            out = super().loss(predicted, actual)
            float(out.values)                  # D2H read: not recordable
            return out

    x, y = _data()
    results = []
    for peek in (True, False):
        np.random.seed(9)
        net, model = _mlp([13, 10], Adam(lr=1e-3))
        if peek:
            model.loss = PeekingLoss()
        losses = [float(model.train_step(Tensor(x), Tensor(y)).values) for _ in range(5)]
        results.append((losses, params(net)))
    assert np.allclose(results[0][0], results[1][0], rtol=0, atol=1e-6)
    for a, b in zip(results[0][1], results[1][1]):
        assert op_cases.rel_err(a, b) <= 1e-6


def test_values_async_matches_values():
    """Tensor.values_async(): the read-back runs on its own stream after the work queued so far;
    several can be outstanding, results equal the synchronous .values (scalars and matrices)"""
    from core.tensor import Tensor
    rng = np.random.RandomState(3)
    x = rng.rand(64, 33).astype(np.float32)
    t = Tensor(x)
    reads, want = [], []
    for k in range(6):
        u = t * float(k) + 1.0
        reads.append((u.values_async(), u.sum().values_async()))
        want.append(x * np.float32(k) + np.float32(1.0))
        t = t + 0.0                       # more work queued behind the pending reads
    for (rm, rs), w in zip(reads, want):
        assert np.array_equal(rm.result(), w)
        assert abs(float(rs.result()) - float(w.astype(np.float64).sum())) <= 1e-3 * abs(float(w.sum()))
        assert rm.result() is rm.result()          # cached after the first wait


def test_optimizer_that_only_offers_compute_step():
    """an optimiser object that does not derive from BaseOptimizer and offers just what the
    reference's Model.step calls (model.py:55 `compute_step(grads, params)` -> per-layer dicts of
    steps): Model.step applies its steps, nothing is postponed or recorded for such a model"""
    from core.tensor import Tensor

    class Plain(object):
        def compute_step(self, grads, params):
            return [{k: -0.05 * (g.numpy() if hasattr(g, "numpy") else np.asarray(g)) for k, g in layer.items()}
                    for layer in grads]

    x, y = _data()
    np.random.seed(4)
    net, model = _mlp([13, 10], Plain())
    losses = []
    for _ in range(4):
        before = params(net) if net.layers[0].is_init else None
        model.zero_grad()
        pred = model.forward(Tensor(x))
        assert type(pred) is Tensor
        loss = model.loss.loss(pred, Tensor(y))
        loss.backward()
        grads = [p.grad.copy() for p in _param_tensors(net)]
        model.step()
        if before is not None:
            for b, g, p in zip(before, grads, _param_tensors(net)):
                assert np.allclose(p.values, b - 0.05 * g, atol=1e-7)
        losses.append(float(loss.values))
    assert losses[-1] < losses[0] and not model._captured
