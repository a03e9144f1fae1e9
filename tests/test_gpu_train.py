"""End-to-end parity of the training path (Dense/ReLU layers, fused CE, autograd sweep, flat
arenas, fused Adam) against goldens recorded from the real reference and against the oracle."""
import os

import numpy as np
import pytest

import op_cases
import ref_numpy as R
from support import gemm_route

pytestmark = pytest.mark.gpu


def _build(widths, lr=1e-3):
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    layers = []
    for i, w in enumerate(widths):
        layers.append(Dense(w))
        if i + 1 < len(widths):
            layers.append(ReLU())
    net = Net(layers)
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=lr)), SoftmaxCrossEntropyLoss()


def _mnist_trajectory(param_dtype, steps=100, kind="mnist_traj"):
    """examples/mnist/run.py's loop (run.py:78-84) on synthetic MNIST-shaped data, np.random.seed(0).
    kind = "mnist_traj" (random labels) or "mnist_learn_traj" (learnable class templates).
    Returns (losses, first-step gradient norms, final parameter sums)."""
    import ref_fp32
    import core.initializer as I
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    from core.tensor import Tensor
    from utils.data_iterator import BatchIterator

    class Xavier(I.XavierUniformInit):
        # the reference stores float32 draws; float64 mode keeps those (float32-rounded) values
        def __call__(self, shape):
            return Tensor(self.init(shape).astype(np.float32), requires_grad=True, dtype=param_dtype)

    class Zeros(I.ZerosInit):
        def __call__(self, shape):
            return Tensor(self.init(shape), requires_grad=True, dtype=param_dtype)

    np.random.seed(0)
    if kind == "mnist_traj":
        x, y, onehot = R.synthetic_mnist(12800, seed=0)
    else:
        x, y, onehot = ref_fp32.learnable_mnist(12800, seed=0)
    train_x, train_y = Tensor(x.astype(param_dtype)), Tensor(onehot)
    widths = [200, 100, 70, 30, 10]
    layers = []
    for i, w in enumerate(widths):
        layers.append(Dense(w, w_init=Xavier(), b_init=Zeros()))
        if i + 1 < len(widths):
            layers.append(ReLU())
    net = Net(layers)
    model = Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))
    loss_layer = SoftmaxCrossEntropyLoss()
    losses, first_norms = [], None
    for batch in BatchIterator(batch_size=128)(train_x, train_y):
        model.zero_grad()
        pred = model.forward(batch.inputs)
        loss = loss_layer.loss(pred, batch.targets)
        loss.backward()
        if first_norms is None:
            first_norms = np.array([float(np.linalg.norm(p.grad)) for layer in net.get_parameters()
                                    for p in layer.values()])
        model.step()
        losses.append(float(loss.values))
        if len(losses) == steps:
            break
    sums = np.array([float(np.sum(p.values)) for layer in net.get_parameters() for p in layer.values()])
    return np.array(losses), first_norms, sums


@pytest.mark.parametrize("kind", ["mnist_traj", "mnist_learn_traj"])
def test_mnist_mlp_loss_trajectory_float64_engine(golden_dir, kind):
    """The reference is a float64 computation from its second step on (SURVEY 0.4); with the
    engine's parameters kept in float64 every kernel on the path (SIMT GEMM, bias/ReLU, fused CE,
    column sums, arena Adam) runs in its float64 instantiation and the 100-step trajectory agrees
    to <= 1e-6 (measured <= 1e-7)."""
    gold = np.load(os.path.join(golden_dir, kind + ".npz"))
    losses, first_norms, sums = _mnist_trajectory(np.float64, kind=kind)
    assert np.max(np.abs(losses - gold["losses"])) <= 1e-6
    assert np.allclose(first_norms, gold["first_grad_norms"], rtol=1e-5, atol=1e-12)
    # parameter sums: Adam's first steps are +-lr on entries whose gradient is ~eps, so a 1e-12
    # gradient difference moves individual entries by O(lr); the sums agree to ~1e-6 relative
    assert np.allclose(sums, gold["final_param_sums"], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("kind", ["mnist_traj", "mnist_learn_traj"])
def test_mnist_mlp_loss_trajectory_float32_engine(golden_dir, kind):
    """north_star: "the loss trajectory over 100 steps within 1e-4" on the PRODUCTION path: float32
    parameters, gradients and Adam state, free running for all 100 steps, against the trajectory
    the real reference recorded (random-label data, where the loss stays near ln(B*C), and
    learnable data, where it falls from 7.13 to 4.87).  oracle/ref_fp32.py shows plain single
    precision holds 2e-6 here (tests/test_oracle_golden.py), so 1e-4 is asserted over every step."""
    gold = np.load(os.path.join(golden_dir, kind + ".npz"))
    losses, first_norms, _ = _mnist_trajectory(np.float32, kind=kind)
    diff = np.abs(losses - gold["losses"])
    assert np.max(diff) <= 1e-4, (int(np.argmax(diff)), float(np.max(diff)))
    assert np.allclose(first_norms, gold["first_grad_norms"], rtol=1e-5, atol=1e-9)


def test_mnist_mlp_teacher_forced_float32(golden_dir):
    """float32 engine vs oracle with the oracle's parameters loaded every step (SURVEY 7.3):
    loss within 1e-5 and every gradient within rel 1e-5 (north_star's per-op bound) at each of 20
    steps, so errors cannot compound."""
    from core.losses import SoftmaxCrossEntropyLoss
    from core.tensor import Tensor
    np.random.seed(0)
    x, y, onehot = R.synthetic_mnist(2560, seed=0)
    mlp = R.RefMLP([200, 100, 70, 30, 10], R.RefAdam(lr=1e-3))
    net, model, loss_layer = _build([200, 100, 70, 30, 10])
    for it in range(20):
        xb, yb = x[it * 128:(it + 1) * 128], onehot[it * 128:(it + 1) * 128]
        mlp.zero_grad()
        rloss = R.softmax_cross_entropy(mlp.forward(R.lift(xb)), yb)
        rloss.backward()
        if it == 0:
            model.forward(Tensor(xb))          # lazy initialisation of the engine's layers
        params = [p for layer in net.get_parameters() for p in layer.values()]
        for p, rp in zip(params, mlp.params()):
            p.values = rp.values.astype(np.float32)
            p.requires_grad = True
        model.zero_grad()
        loss = loss_layer.loss(model.forward(Tensor(xb)), Tensor(yb))
        loss.backward()
        assert abs(float(loss.values) - float(rloss.values)) <= 1e-5, it
        for k, (p, rp) in enumerate(zip(params, mlp.params())):
            assert op_cases.rel_err(p.grad, rp.grad) <= 1e-5, (it, k)
        mlp.step()
        # both sides start the next step from bit-identical parameters
        for rp in mlp.params():
            rp.assign(rp.values.astype(np.float32).astype(np.float64))


def test_wide_style_mlp_steps(golden_dir):
    """3 Adam steps of a 4 x Dense(64) MLP with fp32 one-hot labels: losses, first-step gradients
    and final parameters against the reference golden"""
    from core.tensor import Tensor
    gold = np.load(os.path.join(golden_dir, "mlp_step.npz"))
    np.random.seed(0)
    rng = np.random.RandomState(0)
    B, D = 32, 64
    x = rng.rand(B, D).astype(np.float32)
    labels = np.eye(D, dtype=np.float32)[rng.randint(0, D, B)]
    net, model, loss_layer = _build([D, D, D, D])
    losses = []
    for it in range(3):
        model.zero_grad()
        loss = loss_layer.loss(model.forward(Tensor(x)), Tensor(labels))
        loss.backward()
        if it == 0:
            k = 0
            for layer in net.get_parameters():
                for p in layer.values():
                    assert op_cases.rel_err(p.grad, gold["grad%d" % k]) <= 1e-5, k
                    k += 1
        model.step()
        losses.append(float(loss.values))
    assert np.max(np.abs(np.array(losses) - gold["losses"])) <= 1e-5
    k = 0
    for layer in net.get_parameters():
        for p in layer.values():
            assert op_cases.rel_err(p.values, gold["param%d" % k]) <= 1e-5, k
            k += 1


@pytest.mark.parametrize("cg", [1, 2])
def test_tensor_core_mlp_step_teacher_forced(cg):
    """a 4-layer 512-wide MLP at batch 1024 runs its 11 GEMMs on the tcgen05 path; one step is
    compared with the oracle started from the same parameters (teacher forcing, SURVEY 7.3)"""
    import core._backend as be
    from core.tensor import Tensor
    with gemm_route(cta_group=cg, TC_MIN_MNK=1 << 20):
        np.random.seed(1)
        rng = np.random.RandomState(1)
        B, D = 1024, 512
        x = rng.rand(B, D).astype(np.float32)
        labels = np.eye(D, dtype=np.float32)[rng.randint(0, D, B)]
        net, model, loss_layer = _build([D, D, D, D])
        model.zero_grad()
        loss = loss_layer.loss(model.forward(Tensor(x)), Tensor(labels))
        # oracle with the very same initial parameters
        mlp = R.RefMLP([D, D, D, D], R.RefAdam(lr=1e-3))
        params = [p for layer in net.get_parameters() for p in layer.values()]
        k = 0
        for layer in mlp.layers:
            if isinstance(layer, R.RefDense):
                layer.w = R.RefTensor(params[k].values.copy(), True)
                layer.b = R.RefTensor(params[k + 1].values.copy(), True)
                k += 2
        rloss = R.softmax_cross_entropy(mlp.forward(R.lift(x)), labels)
        assert abs(float(loss.values) - float(rloss.values)) <= 1e-5
        loss.backward()
        rloss.backward()
        for p, rp in zip(params, mlp.params()):
            assert op_cases.rel_err(p.grad, rp.grad) <= 1e-5
        # the fused arena Adam, checked against the reference update applied to the engine's own
        # gradients (Adam's first step is -lr*g/(|g|+eps): for entries with |g| ~ eps = 1e-8 it
        # turns a 1e-8 absolute gradient difference into an O(lr) step difference, so feeding
        # both sides the same gradient is the meaningful comparison)
        p0 = [p.values.astype(np.float64) for p in params]
        g0 = [p.grad.astype(np.float64) for p in params]
        model.step()
        adam = R.RefAdam(lr=1e-3)
        flat_step = adam._step(np.concatenate([g.ravel() for g in g0]))
        pos = 0
        for p, a, g in zip(params, p0, g0):
            expect = a + flat_step[pos:pos + g.size].reshape(g.shape)
            pos += g.size
            assert op_cases.rel_err(p.values, expect) <= 1e-5


@pytest.mark.parametrize("fuse_bwd", [False, True])
@pytest.mark.parametrize("size", [(16, 20, 12, 8), (512, 256, 384, 128)])
def test_dense_relu_fusion_is_transparent(size, fuse_bwd):
    """Net.forward runs Dense+ReLU as one GEMM launch (ReLU and the next layer's tf32 planes come
    out of the epilogue); values, recorded layer inputs and every gradient are bit-identical to
    calling the layers one by one (small = SIMT kernel, large = tcgen05 kernel)"""
    import core._backend as be
    import core.ops as ops
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.nn import Net
    from core.tensor import Tensor
    B, D, H, C = size
    rng = np.random.RandomState(7)
    x = rng.standard_normal((B, D)).astype(np.float32)
    labels = np.eye(C, dtype=np.float32)[rng.randint(0, C, B)]
    old_bwd = ops.FUSE_RELU_BWD
    ops.FUSE_RELU_BWD = fuse_bwd   # also fold the ReLU-backward mask into the dX launch
    try:
        with gemm_route(TC_MIN_MNK=1 << 22):
            outs = []
            for fused in (True, False):
                np.random.seed(11)
                layers = [Dense(H), ReLU(), Dense(H), ReLU(), Dense(C)]
                net = Net(layers)
                be.new_split_epoch()
                if fused:
                    pred = net.forward(Tensor(x))
                else:
                    pred = Tensor(x)
                    for layer in layers:
                        pred = layer.forward(pred)
                loss = SoftmaxCrossEntropyLoss().loss(pred, Tensor(labels))
                loss.backward()
                grads = [p.grad.copy() for layer in net.get_parameters() for p in layer.values()]
                outs.append((pred.values.copy(), layers[1].inputs.values.copy(), layers[2].inputs.values.copy(), grads))
            a, b = outs
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
            for ga, gb in zip(a[3], b[3]):
                assert np.array_equal(ga, gb)
    finally:
        ops.FUSE_RELU_BWD = old_bwd


def test_generic_step_path_equals_fused():
    """Model.step through compute_step()/`param += step` (the reference's three stages) gives the
    same parameters as the fused arena kernel"""
    from core.tensor import Tensor
    rng = np.random.RandomState(2)
    x = rng.rand(16, 20).astype(np.float32)
    labels = np.eye(8, dtype=np.float32)[rng.randint(0, 8, 16)]
    results = []
    for generic in (False, True):
        np.random.seed(3)
        net, model, loss_layer = _build([12, 8])
        for _ in range(3):
            model.zero_grad()
            loss = loss_layer.loss(model.forward(Tensor(x)), Tensor(labels))
            loss.backward()
            if generic:
                model._step_generic()
            else:
                model.step()
        results.append([p.values.copy() for layer in net.get_parameters() for p in layer.values()])
    for a, b in zip(*results):
        assert op_cases.rel_err(a, b) <= 1e-6


def test_save_load_roundtrip(tmp_path):
    from core.tensor import Tensor
    np.random.seed(4)
    net, model, _ = _build([6, 3])
    x = Tensor(np.random.rand(5, 4).astype(np.float32))
    y0 = model.forward(x).values.copy()
    path = str(tmp_path / "m.pkl")
    model.save(path)
    np.random.seed(5)
    net2, model2, _ = _build([6, 3])
    model2.forward(x)
    model2.load(path)
    assert np.array_equal(model2.forward(x).values, y0)


def test_bench_dump_outputs_hold_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs on the MNIST workload, eager steps: the loss is the JSON line's
    final_loss, and loss, prediction and every parameter equal those of the same seeded steps run
    here (step 0 and warm-up, then exactly --steps timed steps: one step more or less moves every
    parameter by about Adam's lr)"""
    import json
    import subprocess
    import sys
    import bench
    import core._backend as be
    from core.tensor import Tensor
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    steps, warmup = 3, 4
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "mnist", "--graph", "off",
                          "--steps", str(steps), "--warmup", str(warmup), "--no-extras", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path / "bench")],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warmup

    cfg = dict(bench.MNIST)
    B, C = cfg["batch"], cfg["widths"][-1]
    xs, ys = bench.synthetic_shard(cfg, B, 0)
    x_dev = [be.from_numpy(x) for x in xs]
    y_dev = [be.from_numpy(bench.one_hot_host(y, C)) for y in ys]
    stepper = bench.Stepper(cfg, use_graph=False)
    stepper.keep_outputs = True
    for i in list(range(warmup)) + list(range(steps)):
        stepper(Tensor(x_dev[i % 2]), Tensor(y_dev[i % 2]))
    names = bench.dump_outputs(stepper, str(tmp_path / "here"))
    assert names == ["layer%d_%s" % (i, k) for i in (0, 2, 4, 6, 8) for k in ("b", "w")] + ["loss", "prediction"]
    assert sorted(f[:-len(".npy")] for f in os.listdir(str(tmp_path / "bench"))) == names
    for n in names:
        got = np.load(str(tmp_path / "bench" / (n + ".npy")))
        want = np.load(str(tmp_path / "here" / (n + ".npy")))
        assert got.dtype == np.float32 and got.shape == want.shape, n
        assert op_cases.rel_err(got, want) <= 1e-6, n
    assert float(np.load(str(tmp_path / "bench" / "loss.npy"))) == line["final_loss"]
    assert np.load(str(tmp_path / "bench" / "prediction.npy")).shape == (B, C)


def test_prefetch_iterator_delivers_the_right_rows():
    """utils.data_iterator.PrefetchIterator: host data set -> device batches over the copy stream
    (pinned in place without shuffling, staged with shuffling); every batch must hold exactly the
    rows the equivalent numpy indexing gives, including the short last batch and loop mode"""
    from utils.data_iterator import PrefetchIterator
    rng = np.random.RandomState(0)
    x = rng.rand(1000, 37).astype(np.float32)
    y = rng.rand(1000, 5).astype(np.float32)
    got = [(b.inputs.values.copy(), b.targets.values.copy()) for b in PrefetchIterator(batch_size=128)(x, y)]
    assert [len(a) for a, _ in got] == [128] * 7 + [104]
    assert np.array_equal(np.concatenate([a for a, _ in got]), x)
    assert np.array_equal(np.concatenate([b for _, b in got]), y)
    np.random.seed(5)
    got = [(b.inputs.values.copy(), b.targets.values.copy())
           for b in PrefetchIterator(batch_size=128, shuffle=True)(x, y)]
    np.random.seed(5)
    order = np.arange(1000)
    np.random.shuffle(order)
    assert np.array_equal(np.concatenate([a for a, _ in got]), x[order])
    assert np.array_equal(np.concatenate([b for _, b in got]), y[order])
    feed = iter(PrefetchIterator(batch_size=400, loop=True)(x, y))
    sizes = [len(next(feed).inputs) for _ in range(7)]
    assert sizes == [400, 400, 200, 400, 400, 200, 400]
    feed.close()


def test_batch_iterator_gathers_by_permutation_window():
    """utils/data_iterator.py:22-34 on device Tensors: each batch is rows perm[start:end] of the data
    set, gathered on demand (no shuffled copy of the whole set is ever made), identical to the
    reference's `inputs[idx]` then `inputs[start:end]` with the same seed, short last batch included"""
    import core._backend as be
    from core.tensor import Tensor
    from utils.data_iterator import BatchIterator
    rng = np.random.RandomState(3)
    n, d = 50000, 784
    x = rng.rand(n, d).astype(np.float32)
    y = np.eye(10)[rng.randint(0, 10, n)]
    tx, ty = Tensor(x), Tensor(y)
    be.sync()
    before = be.pool_stats()["reserved"]
    np.random.seed(11)
    sizes, checked = [], 0
    for k, batch in enumerate(BatchIterator(batch_size=128)(tx, ty)):
        sizes.append(len(batch.inputs))
        if k in (0, 1, 200, 390):
            if k == 0:
                np.random.seed(11)
                order = np.arange(n)
                np.random.shuffle(order)
            lo = k * 128
            assert np.array_equal(batch.inputs.values, x[order[lo:lo + 128]])
            assert np.array_equal(batch.targets.values, y[order[lo:lo + 128]])
            checked += 1
    assert sizes == [128] * 390 + [80] and checked == 4
    # the epoch allocated the permutation (400 KB) and a few batches, not a second copy of x (157 MB)
    assert be.pool_stats()["reserved"] - before < 16 * 1024 * 1024
    # a tensor that takes part in autograd keeps the reference's differentiable getitem path
    np.random.seed(11)
    tg = Tensor(x[:300], requires_grad=True)
    first = next(iter(BatchIterator(batch_size=128)(tg, Tensor(y[:300]))))
    assert first.inputs.requires_grad and len(first.inputs.dependency) == 1


def test_train_step_takes_gathered_batches_directly():
    """Model.train_step on BatchIterator batches: the recorded step gathers rows perm[start:end]
    straight into its input buffers; same losses and parameters as feeding materialised batches"""
    from core.tensor import Tensor
    from utils.data_iterator import BatchIterator
    rng = np.random.RandomState(5)
    x = rng.rand(1000, 48).astype(np.float32)
    y = np.eye(10)[rng.randint(0, 10, 1000)]
    results = []
    for lazy in (True, False):
        np.random.seed(7)
        net, model, _ = _build([32, 16, 10])
        np.random.seed(9)
        losses = []
        for batch in BatchIterator(batch_size=128)(Tensor(x), Tensor(y)):
            xb, yb = batch.inputs, batch.targets
            if not lazy:
                xb, yb = Tensor(xb.values), Tensor(yb.values)
            losses.append(float(model.train_step(xb, yb).values))
        results.append((losses, [p.values.copy() for layer in net.get_parameters() for p in layer.values()]))
    assert results[0][0] == results[1][0] and len(results[0][0]) == 8
    for a, b in zip(results[0][1], results[1][1]):
        assert np.array_equal(a, b)


def test_prefetch_iterator_integer_labels_become_one_hot_on_device():
    """PrefetchIterator(num_classes=C): targets are the integer label vector; the batches carry the
    dense one-hot rows `np.eye(C)[labels]` (run.py:27-28) built by tnn_one_hot, for class counts that
    are and are not multiples of 4, shuffled and not, short last batch included"""
    from utils.data_iterator import PrefetchIterator
    rng = np.random.RandomState(1)
    for C in (10, 4096, 7):
        n = 300
        x = rng.rand(n, 12).astype(np.float32)
        lab = rng.randint(0, C, n)
        got = [(b.inputs.values.copy(), b.targets.values.copy())
               for b in PrefetchIterator(batch_size=128, num_classes=C)(x, lab)]
        assert [len(a) for a, _ in got] == [128, 128, 44]
        assert np.array_equal(np.concatenate([a for a, _ in got]), x)
        assert np.array_equal(np.concatenate([b for _, b in got]), np.eye(C, dtype=np.float32)[lab])
        np.random.seed(3)
        got = [(b.inputs.values.copy(), b.targets.values.copy())
               for b in PrefetchIterator(batch_size=128, shuffle=True, num_classes=C)(x, lab)]
        np.random.seed(3)
        order = np.arange(n)
        np.random.shuffle(order)
        assert np.array_equal(np.concatenate([a for a, _ in got]), x[order])
        assert np.array_equal(np.concatenate([b for _, b in got]), np.eye(C, dtype=np.float32)[lab[order]])
    with pytest.raises(ValueError):
        next(iter(PrefetchIterator(batch_size=8, num_classes=3)(x, np.eye(3)[lab % 3])))


def test_cross_entropy_takes_class_indices_bit_identically():
    """A one-hot target matrix that exists only as int32 class indices (be.LazyOneHot, what
    PrefetchIterator(num_classes=C) yields): the fused cross-entropy reads the indices
    (tnn_ce_loss / tnn_ce_bwd `labels_dev`) and its loss and dz are bit-identical to the dense-row
    path (losses.py:24-32 on np.eye(C)[labels], run.py:27-28); the dense rows are never written
    unless somebody asks for them; labels outside [0, C) behave like an all-zero row"""
    import core._backend as be
    from core.losses import SoftmaxCrossEntropyLoss
    from core.tensor import Tensor
    rng = np.random.RandomState(5)
    for B, C, bad in ((300, 7, False), (4096, 10, False), (64, 4096, False), (513, 1001, False), (40, 12, True),
                       (3000, 12, True)):
        z = (rng.randn(B, C) * 3).astype(np.float32)
        lab = rng.randint(0, C, B).astype(np.int32)
        if bad:
            lab[3], lab[17] = -1, C + 2
        dense = np.zeros((B, C), np.float32)
        ok = (lab >= 0) & (lab < C)
        dense[np.arange(B)[ok], lab[ok]] = 1.0
        out = []
        for mode in ("dense", "lazy"):
            zt = Tensor(z, requires_grad=True)
            if mode == "dense":
                yt = Tensor(dense)
            else:
                dl = be.from_numpy(lab.view(np.float32))
                lazy = be.LazyOneHot(dl, C, be.empty((B, C), be.F32))
                yt = Tensor(lazy)
            zt.zero_grad()
            loss = SoftmaxCrossEntropyLoss().loss(zt, yt)
            loss.backward()
            if mode == "lazy" and not be.ce_small_ok(B, C):
                assert lazy._real is None          # the B x C rows were never written
            out.append((np.array(loss.values), zt.grad.copy()))
        if bad:
            # -log(0) rows: inf loss on both paths, identical NaN/inf pattern
            assert np.array_equal(out[0][0], out[1][0], equal_nan=True)
            assert np.array_equal(out[0][1], out[1][1], equal_nan=True)
            continue
        assert np.array_equal(out[0][0], out[1][0])
        assert np.array_equal(out[0][1], out[1][1])
        # and both equal the oracle on the dense rows
        rz = R.RefTensor(z.astype(np.float64), requires_grad=True)
        rz.zero_grad()
        rl = R.softmax_cross_entropy(rz, dense.astype(np.float64))
        rl.backward()
        assert abs(float(out[1][0]) - float(rl.values)) <= 1e-5 * max(1.0, abs(float(rl.values)))
        assert np.max(np.abs(out[1][1] - rz.grad)) <= 1e-5 * np.max(np.abs(rz.grad))
        # the rows appear on demand and are exactly np.eye(C)[labels]
        assert np.array_equal(yt.values, dense)


def test_training_on_index_labels_equals_training_on_dense_rows():
    """three steps of an MLP fed by PrefetchIterator(num_classes=C) (class indices into the fused
    loss) and by PrefetchIterator on the dense one-hot matrix: identical losses and parameters"""
    from core.tensor import Tensor
    from utils.data_iterator import PrefetchIterator
    rng = np.random.RandomState(2)
    n, D, C = 384, 40, 130
    x = rng.rand(n, D).astype(np.float32)
    lab = rng.randint(0, C, n)
    dense = np.eye(C, dtype=np.float32)[lab]
    res = []
    for mode in ("dense", "index"):
        np.random.seed(4)
        net, model, loss_fn = _build([64, C])
        it = (PrefetchIterator(batch_size=128)(x, dense) if mode == "dense"
              else PrefetchIterator(batch_size=128, num_classes=C)(x, lab))
        losses = []
        for batch in it:
            model.zero_grad()
            loss = loss_fn.loss(model.forward(batch.inputs), batch.targets)
            loss.backward()
            model.step()
            losses.append(float(loss.values))
        res.append((losses, [p.values.copy() for layer in net.get_parameters() for p in layer.values()]))
    assert res[0][0] == res[1][0]
    for a, b in zip(res[0][1], res[1][1]):
        assert np.array_equal(a, b)


def test_one_hot_kernel_edge_cases():
    """tnn_one_hot: float32 / float64 outputs, labels outside [0, C) give all-zero rows"""
    import core._backend as be
    lab = np.array([0, 3, 2, -1, 4, 7, 1], dtype=np.int32)
    dl = be.from_numpy(lab.view(np.float32))           # raw 4-byte device vector
    for dt, C in ((be.F32, 4), (be.F32, 5), (be.F64, 4)):
        out = be.empty((len(lab), C), dt)
        be.one_hot_into(out, dl.ptr, len(lab), C)
        want = np.zeros((len(lab), C))
        for r, v in enumerate(lab):
            if 0 <= v < C:
                want[r, v] = 1.0
        assert np.array_equal(out.numpy(), want.astype(out.numpy().dtype))


def test_split_column_reduction_is_deterministic_and_exact_on_integers():
    """the one-launch split column reduction (last CTA folds the partials in split order): integer
    data sums exactly whatever the split, repeated launches are bit-identical, max / min take the
    same path"""
    import core._backend as be
    rng = np.random.RandomState(2)
    for R_, C_ in ((20000, 1024), (4099, 260), (70000, 33)):
        a = rng.randint(-8, 9, (R_, C_)).astype(np.float32)
        d = be.from_numpy(a)
        s1 = be.colsum(d).numpy()
        s2 = be.colsum(d).numpy()
        assert np.array_equal(s1, s2)
        assert np.array_equal(s1, a.sum(axis=0, keepdims=True, dtype=np.float64).astype(np.float32))
        assert np.array_equal(be.reduce(be.RED_MAX, d, axis=0).numpy(), a.max(axis=0))
        assert np.array_equal(be.reduce(be.RED_MIN, d, axis=0).numpy(), a.min(axis=0))
    x = rng.standard_normal((30000, 512)).astype(np.float32)
    got = be.colsum(be.from_numpy(x)).numpy()
    assert op_cases.rel_err(got, x.astype(np.float64).sum(axis=0, keepdims=True)) <= 1e-5


def test_predict_builds_no_graph_and_matches_forward():
    """Model.predict / ops.no_grad: same values as forward(), no autograd graph, training unaffected"""
    import core.ops as ops
    from core.tensor import Tensor
    rng = np.random.RandomState(2)
    x = rng.rand(64, 48).astype(np.float32)
    labels = np.eye(10)[rng.randint(0, 10, 64)]
    np.random.seed(4)
    net, model, loss_layer = _build([32, 16, 10])
    ref = model.forward(Tensor(x))
    out = model.predict(x)
    assert np.array_equal(out.values, ref.values)
    assert ref.requires_grad and len(ref.dependency) > 0
    assert not out.requires_grad and out.dependency == []
    with pytest.raises(AssertionError):
        out.backward()
    with ops.no_grad():
        t = Tensor(x, requires_grad=True) * 2.0 + 1.0
    assert not t.requires_grad
    assert np.argmax(out, axis=1).shape == (64,)          # run.py:89 consumes a Tensor through __array__
    # the graph machinery is back on afterwards
    model.zero_grad()
    loss = loss_layer.loss(model.forward(Tensor(x)), Tensor(labels))
    loss.backward()
    model.step()
    assert np.isfinite(float(loss.values))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_grouped_dense_backward_matches_separate_launches(dtype):
    """small Dense layers: dX / dW / db from one grouped launch (tnn_dense_bwd_simt) against the
    three separate products, through the whole MLP backward, including a second backward() that
    accumulates into the arena slots"""
    import core.initializer as I
    import core.ops as ops
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import SGD
    from core.tensor import Tensor

    class Xavier(I.XavierUniformInit):
        def __call__(self, shape):
            return Tensor(self.init(shape).astype(np.float32), requires_grad=True, dtype=dtype)

    class Zeros(I.ZerosInit):
        def __call__(self, shape):
            return Tensor(self.init(shape), requires_grad=True, dtype=dtype)

    rng = np.random.RandomState(3)
    x = rng.rand(80, 50).astype(dtype)
    labels = np.eye(10)[rng.randint(0, 10, 80)]
    tol = 2e-6 if dtype == np.float32 else 1e-12
    old = ops.GROUP_SMALL_DENSE_BWD
    out = {}
    try:
        for grouped in (True, False):
            ops.GROUP_SMALL_DENSE_BWD = grouped
            np.random.seed(5)
            widths = [70, 33, 10]
            layers = []
            for i, wd in enumerate(widths):
                layers.append(Dense(wd, w_init=Xavier(), b_init=Zeros()))
                if i + 1 < len(widths):
                    layers.append(ReLU())
            net = Net(layers)
            model = Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=SGD(lr=0.1))
            xin = Tensor(x, requires_grad=True)
            # step 1 builds the arenas; afterwards gradients are written straight into their slots
            model.zero_grad()
            model.loss.loss(model.forward(Tensor(x)), Tensor(labels)).backward()
            model.step()
            model.zero_grad()
            loss = model.loss.loss(model.forward(xin), Tensor(labels))
            loss.backward()
            first = [p.grad.copy() for layer in net.get_parameters() for p in layer.values()]
            loss2 = model.loss.loss(model.forward(xin), Tensor(labels))
            loss2.backward()                      # accumulates on top
            second = [p.grad.copy() for layer in net.get_parameters() for p in layer.values()]
            out[grouped] = (first, second, xin.grad.copy(), layers[1].inputs.grad.copy())
    finally:
        ops.GROUP_SMALL_DENSE_BWD = old
    for a, b in zip(out[True][0] + out[True][1], out[False][0] + out[False][1]):
        assert op_cases.rel_err(a, b) <= tol
    assert op_cases.rel_err(out[True][2], out[False][2]) <= tol      # dL/dx of the input batch
    assert op_cases.rel_err(out[True][3], out[False][3]) <= tol      # non-leaf .grad of a pre-activation
    for a, b in zip(out[True][0], out[True][1]):
        assert op_cases.rel_err(b, 2 * a) <= 10 * tol                # second backward doubled it


@pytest.mark.parametrize("split", ["f16", "mix", "tf32x3"])
def test_tensor_core_mlp_teacher_forced_over_steps(split):
    """the tcgen05 path along a training run: 12 steps of a 3-layer 256-wide MLP at batch 512, the
    oracle's (Adam-updated, float32-rounded) parameters loaded into the engine before every step,
    loss within 1e-5 and every gradient within rel 1e-5 of the oracle's at each step -- for both
    operand splits.  A step on which a pre-activation sits so close to zero that float32 and
    float64 arithmetic put it on different sides of the ReLU kink (one unit in ~10^6, seen about
    once per run) compares the loss only: there the gradients differ by the discontinuity, not by
    the arithmetic."""
    import core._backend as be
    from core.tensor import Tensor
    with gemm_route(TC_MIN_MNK=1 << 20, TC_SPLIT=split):
        rng = np.random.RandomState(8)
        B, D = 512, 256
        np.random.seed(8)
        mlp = R.RefMLP([D, D, D], R.RefAdam(lr=1e-3))
        net, model, loss_layer = _build([D, D, D])
        compared = 0
        for it in range(12):
            x = rng.rand(B, D).astype(np.float32)
            labels = np.eye(D, dtype=np.float32)[rng.randint(0, D, B)]
            mlp.zero_grad()
            h, ref_pre = R.lift(x), []
            for layer in mlp.layers:
                h = layer.forward(h)
                if isinstance(layer, R.RefDense):
                    ref_pre.append(h.values)
            rloss = R.softmax_cross_entropy(h, labels)
            rloss.backward()
            if it == 0:
                model.forward(Tensor(x))          # lazy initialisation of the engine's layers
            params = [p for layer in net.get_parameters() for p in layer.values()]
            for p, rp in zip(params, mlp.params()):
                p.values = rp.values.astype(np.float32)
                p.requires_grad = True
            model.zero_grad()
            assert be.use_tensor_cores(B, D, D, be.F32)
            loss = loss_layer.loss(model.forward(Tensor(x)), Tensor(labels))
            loss.backward()
            assert abs(float(loss.values) - float(rloss.values)) <= 1e-5, it
            pre = [layer.inputs.values for layer in net.layers if layer.name == "ReLU"]
            same_side = all(np.array_equal(z >= 0, zr >= 0) for z, zr in zip(pre, ref_pre))
            for z, zr in zip(pre, ref_pre):
                assert op_cases.rel_err(z, zr) <= 1e-5, it
            if same_side:
                compared += 1
                for p, rp in zip(params, mlp.params()):
                    assert op_cases.rel_err(p.grad, rp.grad) <= 1e-5, it
            mlp.step()
            # both sides start the next step from bit-identical parameters: the oracle keeps the
            # float32 rounding of its update
            for rp in mlp.params():
                rp.assign(rp.values.astype(np.float32).astype(np.float64))
        assert compared >= 9


@pytest.mark.parametrize("dtype,tol", [(np.float32, 2e-6), (np.float64, 1e-12)])
def test_tanh_and_sigmoid_layers(dtype, tol):
    """layers.py:74-89: Tanh is (1 - e^-x) / (1 + e^-x) = tanh(x / 2) (the reference's formula, kept),
    Sigmoid is 1 / (1 + e^-x) (raises upstream; works here): values and gradients in closed form"""
    from core.layers import Sigmoid, Tanh
    from core.tensor import Tensor
    rng = np.random.RandomState(6)
    x = (rng.standard_normal((37, 21)) * 2).astype(dtype)
    g = rng.standard_normal((37, 21)).astype(dtype)
    x64, g64 = x.astype(np.float64), g.astype(np.float64)
    t = Tensor(x, requires_grad=True)
    out = Tanh().forward(t)
    out.backward(g)
    ref = np.tanh(x64 / 2)
    assert op_cases.rel_err(out.values, ref) <= tol
    assert op_cases.rel_err(t.grad, g64 * 0.5 * (1 - ref ** 2)) <= 10 * tol
    s = Tensor(x, requires_grad=True)
    out = Sigmoid().forward(s)
    out.backward(g)
    ref = 1 / (1 + np.exp(-x64))
    assert op_cases.rel_err(out.values, ref) <= tol
    assert op_cases.rel_err(s.grad, g64 * ref * (1 - ref)) <= 10 * tol
