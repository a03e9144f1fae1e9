"""The reference's five-line training iteration (run.py:78-83) reaching the recorded step without a
change to the loop (core/_deferred.py): Model.forward / SoftmaxCrossEntropyLoss.loss / backward()
are postponed and Model.step() replays the recording.  Everything observable must equal the eager
loop: bit for bit where the recording is the generic one (same kernels), to rounding level where it
is the fused small-MLP pass (other summation orders, as in test_gpu_graph.py)."""
import numpy as np
import pytest

from support import params

pytestmark = pytest.mark.gpu

MNIST = [200, 100, 70, 30, 10]


def _model(widths, seed, d_in, defer, fuse=True, opt="adam"):
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    import core.optimizer as O
    np.random.seed(seed)
    layers = []
    dims = [d_in] + list(widths)
    for i, w in enumerate(widths):
        layers.append(Dense(w, num_in=dims[i]))
        if i + 1 < len(widths):
            layers.append(ReLU())
    net = Net(layers)
    optimizer = {"adam": lambda: O.Adam(lr=1e-3), "sgd": lambda: O.SGD(lr=1e-2)}[opt]()
    model = Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=optimizer)
    model.defer_loop = defer
    model.defer_loop_may_fuse = fuse
    return net, model


def _batches(d_in, classes, sizes, seed=0):
    from core.tensor import Tensor
    rng = np.random.RandomState(seed)
    return [(Tensor(rng.rand(b, d_in).astype(np.float32)), Tensor(np.eye(classes)[rng.randint(0, classes, b)]))
            for b in sizes]


def _recordings(model):
    return [s for s in model._captured.values() if hasattr(s, "graph")]


def _loop(model, batches, loss_layer=None, probe=None):
    """run.py:78-83 verbatim; probe(i, model, pred, loss, when) may look at things on the way"""
    from core.losses import SoftmaxCrossEntropyLoss
    loss_layer = loss_layer or SoftmaxCrossEntropyLoss()
    losses = []
    for i, (x, y) in enumerate(batches):
        model.zero_grad()
        pred = model.forward(x)
        if probe:
            probe(i, model, pred, None, "forward")
        loss = loss_layer.loss(pred, y)
        if probe:
            probe(i, model, pred, loss, "loss")
        loss.backward()
        if probe:
            probe(i, model, pred, loss, "backward")
        model.step()
        if probe:
            probe(i, model, pred, loss, "step")
        losses.append(loss.values.copy())
    return losses


@pytest.mark.parametrize("opt", ["adam", "sgd"])
def test_five_line_loop_replays_the_generic_recording_bit_identically(opt):
    """layer-by-layer recording (fuse_small_mlp off): the unmodified loop with postponement on gives
    the same bits as with it off, across the short last batch of an epoch, and really replayed"""
    import core._backend as be
    sizes = [128] * 6 + [80, 80, 80] + [128] * 4 + [80]
    batches = _batches(784, 10, sizes)
    net_a, model_a = _model(MNIST, 3, 784, defer=False, fuse=False, opt=opt)
    net_b, model_b = _model(MNIST, 3, 784, defer=True, fuse=False, opt=opt)
    la = _loop(model_a, batches)
    n0 = be.launch_count()
    lb = _loop(model_b, batches)
    assert [float(v) for v in la] == [float(v) for v in lb]
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.array_equal(pa, pb)
    assert len(_recordings(model_b)) == 2 and not _recordings(model_a)
    assert all(v.dtype == np.float32 and v.shape == () for v in lb)


def test_defaults_record_layer_by_layer():
    """a Model as the example builds it (no attribute touched): the loop is recorded kernel by kernel
    (>= 10 kernel nodes), NOT as the fused small-MLP pass, so its numbers are the eager loop's"""
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    batches = _batches(784, 10, [128] * 6)
    out = []
    for defer in (False, True):
        np.random.seed(1)
        net = Net([Dense(200), ReLU(), Dense(100), ReLU(), Dense(70), ReLU(), Dense(30), ReLU(), Dense(10)])
        model = Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))
        if not defer:
            model.defer_loop = False
        out.append(([float(v) for v in _loop(model, batches)], params(net)))
    assert Model.defer_loop is True and Model.defer_loop_may_fuse is False
    rec = _recordings(model)
    assert len(rec) == 1 and rec[0].info()["kernel_nodes"] >= 10
    assert out[0][0] == out[1][0]
    for pa, pb in zip(out[0][1], out[1][1]):
        assert np.array_equal(pa, pb)


def test_five_line_loop_can_reach_the_fused_small_mlp_pass():
    """opt-in (defer_loop_may_fuse): from the third iteration of a shape on, step() replays the
    fused pass (<= 8 kernels); losses within 2e-6 of the eager loop, parameters within 1e-5; the
    loss object is the loop's own (run.py:73 `loss_layer`), not model.loss"""
    sizes = [128] * 8 + [80, 80, 80] + [128] * 5
    batches = _batches(784, 10, sizes)
    net_a, model_a = _model(MNIST, 3, 784, defer=False)
    net_b, model_b = _model(MNIST, 3, 784, defer=True)
    la = _loop(model_a, batches)
    lb = _loop(model_b, batches)
    for a, b in zip(la, lb):
        assert abs(float(a) - float(b)) <= 2e-6 * abs(float(a))
    rec = _recordings(model_b)
    assert len(rec) == 2 and all(s.info()["kernel_nodes"] <= 8 for s in rec)
    for pa, pb in zip(params(net_a), params(net_b)):
        assert np.max(np.abs(pa - pb)) <= 1e-5 * np.max(np.abs(pa))


@pytest.mark.parametrize("fuse", [False, True])
def test_values_and_gradients_read_around_a_replayed_step(fuse):
    """whatever the loop looks at is what the eager loop shows: the prediction and its gradient read
    AFTER step() (served from the recording), the loss's gradient, a prediction kept across the
    next replay, parameter gradients read between backward() and step() (runs that iteration
    eagerly)"""
    sizes = [64] * 9
    batches = _batches(96, 10, sizes, seed=4)
    widths = [48, 32, 10]
    tol = 1e-5 if fuse else 0.0
    seen = {False: {}, True: {}}

    def make_probe(store):
        def probe(i, model, pred, loss, when):
            if when == "step" and i in (3, 5, 6):
                store[("pred", i)] = pred.values.copy()
                store[("dpred", i)] = pred.grad.copy()
                store[("dloss", i)] = np.array(loss.grad)
                assert pred.shape == (64, 10) and pred.requires_grad
            if when == "step" and i == 4:
                store["kept"] = pred                      # read two replays later
            if when == "step" and i == 6:
                store[("pred", "kept")] = store["kept"].values.copy()
                store[("dpred", "kept")] = store["kept"].grad.copy()
            if when == "backward" and i == 7:
                store["pgrads"] = [p.grad.copy() for layer in model.net.get_parameters() for p in layer.values()]
            if when == "forward" and i == 8:
                store[("pred", "early")] = pred.values.copy()   # before the loss exists
        return probe

    out = {}
    for defer in (False, True):
        net, model = _model(widths, 5, 96, defer=defer, fuse=fuse)
        losses = _loop(model, batches, probe=make_probe(seen[defer]))
        out[defer] = (losses, params(net))
        if defer:
            assert len(_recordings(model)) == 1
            if fuse:
                assert _recordings(model)[0].info()["kernel_nodes"] <= 8
    a, b = seen[False], seen[True]
    for key in a:
        if key == "kept":
            continue
        va, vb = (a[key], b[key])
        if isinstance(va, list):
            for x, y in zip(va, vb):
                assert np.max(np.abs(x - y)) <= tol * max(np.max(np.abs(x)), 1e-30), key
        else:
            assert va.shape == vb.shape and va.dtype == vb.dtype, key
            assert np.max(np.abs(va - vb)) <= tol * max(np.max(np.abs(va)), 1e-30), key
    for la, lb in zip(out[False][0], out[True][0]):
        assert abs(float(la) - float(lb)) <= (2e-6 if fuse else 0.0) * abs(float(la))
    for pa, pb in zip(out[False][1], out[True][1]):
        assert np.max(np.abs(pa - pb)) <= tol * np.max(np.abs(pa))


def test_anything_else_runs_the_postponed_lines_as_written():
    """uses of a postponed tensor that are not the five lines: operators on the prediction, a second
    loss on it, backward with a seed, backward twice -- all bit-identical to the eager engine"""
    from core.losses import SoftmaxCrossEntropyLoss
    import core.tensor as T
    batches = _batches(40, 6, [32] * 8, seed=9)
    res = {}
    for defer in (False, True):
        net, model = _model([24, 6], 11, 40, defer=defer, fuse=False)
        ce = SoftmaxCrossEntropyLoss()
        log = []
        for i, (x, y) in enumerate(batches):
            model.zero_grad()
            pred = model.forward(x)
            if i == 3:
                extra = (pred * pred).sum()                     # an operator on the prediction
                loss = ce.loss(pred, y) + extra * 0.01
            elif i == 4:
                loss = ce.loss(pred, y)
                other = ce.loss(pred, y)                        # a second loss on the same prediction
                log.append(float(other.values))
            else:
                loss = ce.loss(pred, y)
            if i == 5:
                loss.backward(2.0)                              # seeded
            elif i == 6:
                loss.backward()
                loss.backward()                                 # accumulates twice
            else:
                loss.backward()
            model.step()
            log.append(float(loss.values))
            assert T._DEFERRED[0] is None
        res[defer] = (log, params(net))
    assert res[False][0] == res[True][0]
    for pa, pb in zip(res[False][1], res[True][1]):
        assert np.array_equal(pa, pb)


def test_loops_that_must_not_be_postponed():
    """no zero_grad() before forward (the reference then fails in backward: tensor.py:163 on a None
    gradient -- same TypeError here), TEST phase, a user-defined update rule, defer_loop off, a loss
    with soft labels of another shape: Model.forward returns an ordinary computed Tensor"""
    import core.optimizer as O
    from core.losses import SoftmaxCrossEntropyLoss
    from core.tensor import Tensor
    from core._deferred import LazyTensor
    batches = _batches(40, 6, [32] * 6, seed=2)
    net, model = _model([24, 6], 1, 40, defer=True, fuse=False)
    _loop(model, batches[:4])
    assert len(_recordings(model)) == 1
    x, y = batches[4]
    # TEST phase
    model.set_phase("TEST")
    assert type(model.forward(x)) is Tensor
    model.set_phase("TRAIN")
    # gradients not zeroed since the last step
    pred = model.forward(x)
    assert type(pred) is Tensor
    with pytest.raises(TypeError):
        SoftmaxCrossEntropyLoss().loss(pred, y).backward()
    # switched off
    model.defer_loop = False
    model.zero_grad()
    assert type(model.forward(x)) is Tensor
    model.defer_loop = True
    model.zero_grad()
    lazy = model.forward(x)
    assert type(lazy) is LazyTensor and lazy.shape == (32, 6)
    assert np.array_equal(np.asarray(lazy), model.predict(x).values)      # resolves on first use
    assert type(lazy) is Tensor

    class Mine(O.SGD):
        def _compute_step(self, grad):           # the reference's extension point, overridden
            return super()._compute_step(grad)

    net2, model2 = _model([24, 6], 1, 40, defer=True, fuse=False)
    model2.optimizer = Mine(lr=1e-2)
    _loop(model2, batches)
    assert not _recordings(model2)


def test_batch_iterator_epochs_through_the_postponed_loop():
    """run.py's loop fed by BatchIterator (rows gathered by permutation window straight into the
    recording's input buffer, 80-row last batch): two epochs equal the eager loop bit for bit"""
    from core.tensor import Tensor
    from utils.data_iterator import BatchIterator
    rng = np.random.RandomState(0)
    n = 128 * 5 + 80
    x = Tensor(rng.rand(n, 60).astype(np.float32))
    y = Tensor(np.eye(10)[rng.randint(0, 10, n)])
    res = {}
    for defer in (False, True):
        net, model = _model([32, 10], 7, 60, defer=defer, fuse=False)
        np.random.seed(21)
        it = BatchIterator(batch_size=128)
        losses = []
        for epoch in range(3):
            losses += _loop(model, [(b.inputs, b.targets) for b in it(x, y)])
        res[defer] = ([float(v) for v in losses], params(net))
        if defer:
            assert len(_recordings(model)) == 2
    assert res[False][0] == res[True][0]
    for pa, pb in zip(res[False][1], res[True][1]):
        assert np.array_equal(pa, pb)


def test_recordings_are_capped_for_loops_over_many_shapes():
    """every recording pins its temporaries: a loop whose batch shape keeps changing stops being
    recorded after defer_loop_max_recordings shapes and runs as written -- same numbers either way"""
    sizes = [b for b in (16, 24, 32, 40, 48) for _ in range(4)]
    batches = _batches(40, 6, sizes, seed=3)
    res = {}
    for defer in (False, True):
        net, model = _model([24, 6], 2, 40, defer=defer, fuse=False)
        model.defer_loop_max_recordings = 3
        res[defer] = ([float(v) for v in _loop(model, batches)], params(net))
        if defer:
            assert len(_recordings(model)) == 3
    assert res[False][0] == res[True][0]
    for pa, pb in zip(res[False][1], res[True][1]):
        assert np.array_equal(pa, pb)


_PDL_SCRIPT = r"""
import sys, json
import numpy as np
sys.path.insert(0, %(root)r)
sys.path.insert(0, %(tests)r)
import test_gpu_deferred as td
net, model = td._model(td.MNIST, 3, 784, defer=True, fuse=False)
losses = td._loop(model, td._batches(784, 10, [128] * 8))
print("RESULT " + json.dumps([float(v).hex() for v in losses]
                             + [float(np.sum(p.astype(np.float64))).hex() for p in td.params(net)]))
"""


def test_programmatic_dependent_launch_is_bit_identical():
    """TNN_PDL=1 (experiment, profiles/r02h_pdl_experiment.md): the small kernels of the recorded step
    are launched with the programmatic-dependency attribute and wait at their top for their
    predecessor; same bits as the ordinary launches (the switch is read once per process, hence the
    two child processes)"""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = _PDL_SCRIPT % {"root": root, "tests": os.path.join(root, "tests")}
    out = {}
    for flag in ("0", "1"):
        env = dict(os.environ, TNN_PDL=flag)
        r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
        out[flag] = json.loads(line[len("RESULT "):])
    assert out["0"] == out["1"]


def test_gradient_accumulation_over_prefetched_batches():
    """a loop that is NOT the five lines: backward() on two consecutive PrefetchIterator batches,
    then one step().  The first batch's postponed lines must run before the iterator reuses that
    batch's device buffers (the iterator flushes them when it is resumed); same bits as the eager
    engine"""
    from core.losses import SoftmaxCrossEntropyLoss
    from utils.data_iterator import PrefetchIterator
    rng = np.random.RandomState(6)
    n, D, C = 64 * 12, 40, 6
    x = rng.rand(n, D).astype(np.float32)
    lab = rng.randint(0, C, n)
    res = {}
    for defer in (False, True):
        net, model = _model([24, C], 13, D, defer=defer, fuse=False)
        ce = SoftmaxCrossEntropyLoss()
        losses = []
        for i, batch in enumerate(PrefetchIterator(batch_size=64, num_classes=C)(x, lab)):
            if i % 2 == 0:
                model.zero_grad()
            loss = ce.loss(model.forward(batch.inputs), batch.targets)
            loss.backward()
            if i % 2 == 1:
                model.step()
            losses.append(float(loss.values) if i % 3 == 0 else None)
        res[defer] = (losses, params(net))
    assert res[False][0] == res[True][0]
    for pa, pb in zip(res[False][1], res[True][1]):
        assert np.array_equal(pa, pb)


def test_a_changed_layer_list_is_not_served_by_an_old_recording():
    """swapping an activation between iterations leaves every parameter in place (the arena stays
    valid) but changes the network: the recording of the old layer list must not be replayed --
    the loop and train_step both give the eager engine's bits"""
    from core.layers import Tanh
    batches = _batches(40, 6, [32] * 12, seed=8)
    res = {}
    for mode in ("eager", "loop", "train_step"):
        net, model = _model([24, 16, 6], 17, 40, defer=(mode == "loop"), fuse=False)
        model.fuse_small_mlp = False
        losses = []
        for i, (x, y) in enumerate(batches):
            if i == 6:
                net.layers[1] = Tanh()
            if mode == "train_step":
                losses.append(float(model.train_step(x, y).values))
            else:
                losses += [float(v) for v in _loop(model, [(x, y)])]
        res[mode] = (losses, params(net))
        if mode != "eager":
            assert len(_recordings(model)) == 2
    for mode in ("loop", "train_step"):
        assert res["eager"][0] == res[mode][0], mode
        for pa, pb in zip(res["eager"][1], res[mode][1]):
            assert np.array_equal(pa, pb)
