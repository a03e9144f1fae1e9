"""AdamW, RAdam and Adamax on the device, and learning-rate schedules driving recorded steps.

The kernels against the float64 oracle (oracle/ref_optim.py) on the compute_step and the fused arena
paths; the 128-bit and the scalar path giving the same bits; NaN staying in its element; MLP training
against the oracle; recorded steps (CUDA graph replays, which read the coefficients from device memory)
against the eager loop while a schedule changes the learning rate and RAdam's rectification switches
on; two ranks through the chunked all-reduce."""
import numpy as np
import pytest

import op_cases
import ref_numpy as R
import ref_optim as RO
from support import gpu_count, params, run_two_ranks

pytestmark = pytest.mark.gpu

RULES = ["adamw", "radam", "adamax"]
FAMILY = ["adam"] + RULES


def _make(name, lr=None, **kw):
    import core.optimizer as O
    cls = {"adam": O.Adam, "adamw": O.AdamW, "radam": O.RAdam, "adamax": O.Adamax}[name]
    return cls(**kw) if lr is None else cls(lr=lr, **kw)


def _ref(name, lr=None, **kw):
    cls = {"adam": R.RefAdam, "adamw": RO.RefAdamW, "radam": RO.RefRAdam, "adamax": RO.RefAdamax}[name]
    return cls(**kw) if lr is None else cls(lr=lr, **kw)


def _ref_update(ref, p, g):
    """the fused arena update p <- p + step in the oracle"""
    return ref.apply(p, g) if isinstance(ref, RO.RefAdamW) else p + ref._step(g)


def _grads(n, steps, seed, dt):
    rng = np.random.RandomState(seed)
    return [(rng.standard_normal(n) * 10.0 ** rng.uniform(-2, 1)).astype(dt) for _ in range(steps)]


@pytest.mark.parametrize("name", RULES)
def test_compute_step_matches_oracle(name):
    """the flat step of _compute_step (AdamW: Adam's part alone; compute_step adds the decay)"""
    import core._backend as be
    kw = dict(weight_decay=0.1) if name == "adamw" else {}
    for dt, tol in ((np.float64, 1e-12), (np.float32, 2e-5)):
        opt, ref = _make(name, **kw), _ref(name, **kw)
        for g in _grads(1000, 8, 3, dt):              # RAdam is rectified from t = 6
            step = opt._compute_step(be.from_numpy(g)).numpy()
            g64 = g.astype(np.float64)
            rstep = ref._step(g64, np.zeros_like(g64)) if name == "adamw" else ref._step(g64)
            assert op_cases.rel_err(step, rstep) <= tol


@pytest.mark.parametrize("n", [1, 3, 4 * 1000 + 3, (1 << 20) + 5])
@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("name", RULES)
def test_apply_fused_matches_oracle(name, dt, n):
    import core._backend as be
    kw = dict(weight_decay=0.05) if name == "adamw" else {}
    tol = 1e-12 if dt == np.float64 else 2e-5
    opt, ref = _make(name, **kw), _ref(name, **kw)
    p = np.random.RandomState(n).standard_normal(n).astype(dt)
    pd = be.from_numpy(p)
    p = p.astype(np.float64)
    for g in _grads(n, 7, n + 1, dt):
        opt.apply_fused(pd, be.from_numpy(g))
        p = _ref_update(ref, p, g.astype(np.float64))
        assert op_cases.rel_err(pd.numpy(), p) <= tol


def _run_arena(opt, n, dt, offset, steps=8, nan_at=None):
    """`steps` fused updates on views that start `offset` elements into their buffers: param, state
    and the launches of the first update"""
    import core._backend as be
    rng = np.random.RandomState(5)
    p = np.zeros(n + offset, dt)
    p[offset:] = rng.standard_normal(n)
    pbuf = be.from_numpy(p)
    pv = pbuf.view((n,), offset)
    launches = None
    for k, g in enumerate(_grads(n, steps, 9, dt)):
        if nan_at is not None and k == 2:
            g[nan_at] = np.nan
        gh = np.zeros(n + offset, dt)
        gh[offset:] = g
        gbuf = be.from_numpy(gh)
        be.sync()
        n0 = be.launch_count()
        opt.apply_fused(pv, gbuf.view((n,), offset))
        if launches is None:
            launches = be.launch_count() - n0
    return pv.numpy(), [s.numpy() for s in opt._state], launches


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("name", FAMILY)
def test_vector_and_scalar_paths_are_bit_identical(name, dt):
    """aligned views take the 128-bit kernel plus a scalar tail (two launches), views one element off
    take the scalar kernel (one launch); every parameter and state bit agrees"""
    n = 4 * 1000 + 3
    kw = dict(weight_decay=0.05) if name == "adamw" else {}
    pa, sa, la = _run_arena(_make(name, **kw), n, dt, 0)
    pb, sb, lb = _run_arena(_make(name, **kw), n, dt, 1)
    assert (la, lb) == (2, 1)
    assert np.array_equal(pa, pb)
    for x, y in zip(sa, sb):
        assert np.array_equal(x, y)
    assert np.all(np.isfinite(pa))


@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_adamw_without_decay_is_adam(dt):
    for offset in (0, 1):
        pa, sa, _ = _run_arena(_make("adam"), 4099, dt, offset)
        pb, sb, _ = _run_arena(_make("adamw", weight_decay=0.0), 4099, dt, offset)
        assert np.array_equal(pa, pb)
        for x, y in zip(sa, sb):
            assert np.array_equal(x, y)


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("name", FAMILY)
def test_nan_gradient_stays_in_its_element(name, offset):
    """a NaN gradient element makes that parameter and its state NaN (Adamax's max included) and
    leaves every other element as a clean run leaves it"""
    n, bad = 4099, 1234
    clean_p, clean_s, _ = _run_arena(_make(name), n, np.float32, offset)
    p, s, _ = _run_arena(_make(name), n, np.float32, offset, nan_at=bad)
    keep = np.arange(n) != bad
    assert np.isnan(p[bad]) and all(np.isnan(x[bad]) for x in s)
    assert np.array_equal(p[keep], clean_p[keep])
    for x, y in zip(s, clean_s):
        assert np.array_equal(x[keep], y[keep])


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


@pytest.mark.parametrize("name", RULES)
def test_mlp_training_matches_oracle(name):
    """10 steps through Model.step (the fused arena kernel) and through Model._step_generic
    (compute_step, where AdamW's decay is added on the host) against RefMLP with the oracle rule,
    whose parameters are rounded to float32 after each step as the engine's are, and against each
    other"""
    from core.tensor import Tensor
    kw = dict(weight_decay=0.1) if name == "adamw" else {}
    rng = np.random.RandomState(2)
    x = rng.rand(16, 20).astype(np.float32)
    y = np.eye(10, dtype=np.float32)[rng.randint(0, 10, 16)]
    np.random.seed(7)
    ref = R.RefMLP([13, 7, 10], _ref(name, lr=1e-2, **kw))
    ref.forward(R.lift(x))
    for _ in range(10):
        ref.zero_grad()
        R.softmax_cross_entropy(ref.forward(R.lift(x)), y).backward()
        ps = ref.params()
        for p, s in zip(ps, ref.optimizer.compute_steps(ps)):
            p.assign((p.values + s).astype(np.float32))
    want = [p.values for p in ref.params()]
    got = []
    for generic in (False, True):
        np.random.seed(7)
        net, model = _mlp([13, 7, 10], _make(name, lr=1e-2, **kw))
        model.defer_loop = False
        for _ in range(10):
            model.zero_grad()
            model.loss.loss(model.forward(Tensor(x)), Tensor(y)).backward()
            if generic:
                model._step_generic()
            else:
                model.step()
        assert (model._arena is None) == generic
        got.append(params(net))
        for a, b in zip(got[-1], want):
            assert op_cases.rel_err(a, b) <= 1e-5
    for a, b in zip(*got):
        assert op_cases.rel_err(a, b) <= 1e-5


# ---- recorded steps -------------------------------------------------------------------------------
SIZES = [128] * 6 + [80, 80, 80] + [128] * 4 + [80]      # test_gpu_graph.py's sequence, short batches included


def _model(opt_factory, seed=3, widths=(200, 100, 70, 30, 10), d_in=784):
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    np.random.seed(seed)
    layers = []
    dims = [d_in] + list(widths)
    for i, w in enumerate(widths):
        layers.append(Dense(w, num_in=dims[i]))
        if i + 1 < len(widths):
            layers.append(ReLU())
    net = Net(layers)
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=opt_factory())


def _batches(sizes=SIZES, d_in=784, classes=10, seed=0):
    from core.tensor import Tensor
    rng = np.random.RandomState(seed)
    return [(Tensor(rng.rand(b, d_in).astype(np.float32)), Tensor(np.eye(classes)[rng.randint(0, classes, b)]))
            for b in sizes]


def _eager(model, x, y):
    model.zero_grad()
    loss = model.loss.loss(model.forward(x), y)
    loss.backward()
    model.step()
    return float(loss.values)


def _schedule(kind):
    from core import lr_scheduler as S
    return {"none": None,
            "step": lambda o: S.StepLR(o, 3, gamma=0.5),
            "multistep": lambda o: S.MultiStepLR(o, [2, 5, 11], gamma=0.3),
            "exponential": lambda o: S.ExponentialLR(o, 0.8),
            "cosine": lambda o: S.CosineAnnealingLR(o, 6, eta_min=1e-5),
            "linear": lambda o: S.LinearLR(o, 0.1, 1.0, 8)}[kind]


def _eager_and_recorded(opt_name, sched_kind, mode):
    """the eager loop against the same loop through train_step ('graph'), the fused small-MLP pass
    ('fused') or the postponed five-line loop ('deferred'); the scheduler is stepped every iteration"""
    kw = dict(weight_decay=0.1) if opt_name == "adamw" else {}
    make = lambda: _make(opt_name, lr=3e-3, **kw)      # noqa: E731
    sched = _schedule(sched_kind)
    net_a, model_a = _model(make)
    net_b, model_b = _model(make)
    model_a.defer_loop = False
    model_b.fuse_small_mlp = mode == "fused"
    model_b.defer_loop = mode == "deferred"
    model_b.defer_loop_may_fuse = False
    sa = sched(model_a.optimizer) if sched else None
    sb = sched(model_b.optimizer) if sched else None
    la, lb, lrs = [], [], []
    for x, y in _batches():
        la.append(_eager(model_a, x, y))
        lb.append(_eager(model_b, x, y) if mode == "deferred" else float(model_b.train_step(x, y).values))
        lrs.append(model_b.optimizer.lr)
        if sched:
            sa.step()
            sb.step()
    rec = [s for s in model_b._captured.values() if hasattr(s, "graph")]
    assert len(rec) == 2, "both batch shapes were recorded and replayed"
    assert all((s.info()["kernel_nodes"] <= 8) == (mode == "fused") for s in rec)
    if sched:
        assert len(set(lrs)) > 2
    return (la, params(net_a)), (lb, params(net_b))


@pytest.mark.parametrize("mode", ["graph", "deferred"])
def test_recorded_radam_switches_to_the_rectified_step(mode):
    """RAdam's branch is taken from the uploaded r_t: the recording made at t = 2 is replayed through
    t = 6, where the rectified form starts, and gives the eager loop's bits"""
    (la, pa), (lb, pb) = _eager_and_recorded("radam", "none", mode)
    assert la == lb
    for a, b in zip(pa, pb):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("sched", ["step", "multistep", "exponential", "cosine", "linear"])
@pytest.mark.parametrize("opt_name", ["adam", "adamw"])
def test_recorded_step_follows_the_schedule(opt_name, sched):
    (la, pa), (lb, pb) = _eager_and_recorded(opt_name, sched, "graph")
    assert la == lb
    for a, b in zip(pa, pb):
        assert np.array_equal(a, b)


def test_deferred_loop_follows_the_schedule():
    (la, pa), (lb, pb) = _eager_and_recorded("adamw", "cosine", "deferred")
    assert la == lb
    for a, b in zip(pa, pb):
        assert np.array_equal(a, b)


def test_schedule_changes_the_replayed_step():
    """a control: the same recorded loop without the schedule ends elsewhere"""
    (_, pa), _ = _eager_and_recorded("adamw", "exponential", "graph")
    (_, pc), _ = _eager_and_recorded("adamw", "none", "graph")
    assert not all(np.array_equal(a, c) for a, c in zip(pa, pc))


@pytest.mark.parametrize("opt_name,sched", [("radam", "cosine"), ("adamw", "linear"), ("adamax", "step")])
def test_fused_small_mlp_pass_with_new_rules(opt_name, sched):
    """the fused small-MLP recording, held to test_gpu_graph.py's tolerances"""
    (la, pa), (lb, pb) = _eager_and_recorded(opt_name, sched, "fused")
    for a, b in zip(la, lb):
        assert abs(a - b) <= 2e-6 * abs(a), (a, b)
    for a, b in zip(pa, pb):
        assert np.max(np.abs(a - b)) <= 1e-5 * np.max(np.abs(a))


def test_two_rank_radam_with_schedule_equals_full_batch_oracle():
    if gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    assert "OPT_DIST_OK world=2" in run_two_ranks("opt_dist_worker.py", timeout=200)
