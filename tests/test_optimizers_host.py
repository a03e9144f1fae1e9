"""AdamW, RAdam, Adamax and the learning-rate schedulers on the host: the float64 oracle rules
(oracle/ref_optim.py) against torch.optim, the schedules against torch.optim.lr_scheduler, the
coefficients the optimisers hand the kernel, and argument checking.  No GPU needed."""
import math

import numpy as np
import pytest

import ref_optim as RO

torch = pytest.importorskip("torch")

# (beta1, beta2, eps): RAdam's rectification switches on at t = 6, 7 and 10 respectively
SETTINGS = [(0.9, 0.999, 1e-8), (0.8, 0.8, 1e-6), (0.5, 0.7, 1e-3)]


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def _grads(n, steps, seed):
    rng = np.random.RandomState(seed)
    return [rng.standard_normal(n) * 10.0 ** rng.uniform(-3, 1) for _ in range(steps)]


def _torch_rule(name, b1, b2, eps, wd):
    if name == "adamw":
        return lambda p: torch.optim.AdamW([p], lr=1e-2, betas=(b1, b2), eps=eps, weight_decay=wd)
    if name == "radam":
        return lambda p: torch.optim.RAdam([p], lr=1e-2, betas=(b1, b2), eps=eps)
    return lambda p: torch.optim.Adamax([p], lr=2e-2, betas=(b1, b2), eps=eps)


def _ref_rule(name, b1, b2, eps, wd):
    if name == "adamw":
        return RO.RefAdamW(lr=1e-2, beta1=b1, beta2=b2, epsilon=eps, weight_decay=wd)
    if name == "radam":
        return RO.RefRAdam(lr=1e-2, beta1=b1, beta2=b2, epsilon=eps)
    return RO.RefAdamax(lr=2e-2, beta1=b1, beta2=b2, epsilon=eps)


@pytest.mark.parametrize("setting", SETTINGS)
@pytest.mark.parametrize("name,wd", [("adamw", 0.01), ("adamw", 0.5), ("radam", 0.0), ("adamax", 0.0)])
def test_oracle_rules_match_torch(name, wd, setting):
    b1, b2, eps = setting
    rng = np.random.RandomState(7)
    p0 = rng.standard_normal(257)
    tp = torch.tensor(p0.copy(), dtype=torch.float64, requires_grad=True)
    topt = _torch_rule(name, b1, b2, eps, wd)(tp)
    ref = _ref_rule(name, b1, b2, eps, wd)
    p = p0.copy()
    for g in _grads(p0.size, 20, 11):
        tp.grad = torch.tensor(g, dtype=torch.float64)
        topt.step()
        p = ref.apply(p, g) if name == "adamw" else p + ref._step(g)
        assert _rel(p, tp.detach().numpy()) <= 1e-12


def test_adamw_compute_step_form_equals_apply():
    """the compute_step form (Adam's step minus (lr*wd) p) and the fused form (p*(1-lr*wd) + step)"""
    a, b = RO.RefAdamW(lr=1e-2, weight_decay=0.1), RO.RefAdamW(lr=1e-2, weight_decay=0.1)
    p = np.random.RandomState(1).standard_normal(64)
    pa = pb = p
    for g in _grads(64, 5, 2):
        pa = a.apply(pa, g)
        pb = pb + b._step(g, pb)
        assert _rel(pa, pb) <= 1e-14


def _sched_pairs():
    from core import lr_scheduler as S
    T = torch.optim.lr_scheduler
    return [
        ("step", lambda o: S.StepLR(o, 7, gamma=0.5), lambda o: T.StepLR(o, 7, gamma=0.5)),
        ("multistep", lambda o: S.MultiStepLR(o, [3, 50, 51, 200], gamma=0.3),
         lambda o: T.MultiStepLR(o, [3, 50, 51, 200], gamma=0.3)),
        ("exponential", lambda o: S.ExponentialLR(o, 0.98), lambda o: T.ExponentialLR(o, 0.98)),
        ("cosine", lambda o: S.CosineAnnealingLR(o, 40, eta_min=1e-4), lambda o: T.CosineAnnealingLR(o, 40, eta_min=1e-4)),
        ("cosine_zero_floor", lambda o: S.CosineAnnealingLR(o, 77), lambda o: T.CosineAnnealingLR(o, 77)),
        ("linear", lambda o: S.LinearLR(o), lambda o: T.LinearLR(o)),
        ("linear_decay", lambda o: S.LinearLR(o, 1.0, 0.05, 120), lambda o: T.LinearLR(o, 1.0, 0.05, 120)),
    ]


@pytest.mark.parametrize("case", range(7))
def test_schedulers_match_torch(case):
    import core.optimizer as O
    name, mine, theirs = _sched_pairs()[case]
    opt = O.Adam(lr=0.1)
    sched = mine(opt)
    tp = torch.zeros(1, requires_grad=True)
    topt = torch.optim.SGD([tp], lr=0.1)
    tsched = theirs(topt)
    got, want = [opt.lr], [topt.param_groups[0]["lr"]]
    for _ in range(300):
        topt.step()
        tsched.step()
        sched.step()
        assert sched.get_lr() == opt.lr
        got.append(opt.lr)
        want.append(topt.param_groups[0]["lr"])
    assert sched.last_epoch == 300 and sched.base_lr == 0.1
    assert _rel(np.array(got), np.array(want)) <= 1e-12, name


@pytest.mark.parametrize("make", ["SGD", "Adam", "RMSProp", "Momentum", "Adagrad", "Adadelta", "AdamW", "RAdam",
                                  "Adamax"])
def test_scheduler_drives_every_optimizer(make):
    """the coefficients handed to the kernel carry the scheduled lr"""
    import core.optimizer as O
    from core.lr_scheduler import StepLR
    opt = getattr(O, make)(lr=0.4)
    sched = StepLR(opt, 2, gamma=0.5)
    for e in range(6):
        assert opt._hyper8()[0] == 0.4 * 0.5 ** (e // 2)
        sched.step()


def test_radam_rectification_term():
    import core.optimizer as O
    opt = O.RAdam()
    ref = RO.RefRAdam()
    for t in range(1, 40):
        h = opt._hyper8()
        assert len(h) == 8 and h[7] == 0.0
        assert (h[6] == 0.0) == (t <= 5)
        assert h[6] == ref.rect(t)
        assert h[4] == 1.0 - 0.9 ** t and h[5] == math.sqrt(1.0 - 0.999 ** t)


def test_adamw_and_adamax_coefficients():
    import core.optimizer as O
    w = O.AdamW(lr=0.01, weight_decay=0.2)
    w.apply_weight_decay = True          # no effect: AdamW's decay is the decoupled one
    h = w._hyper8()
    assert h[6] == 1.0 - 0.01 * 0.2 and h[7] == 0.0
    assert w._step_decay() == 0.01 * 0.2
    m = O.Adamax(lr=0.002, beta1=0.8)
    for t in (1, 2, 3):
        assert m._hyper8()[4] == 0.002 / (1.0 - 0.8 ** t)
    r = O.RAdam(weight_decay=0.1)
    assert r._hyper8()[7] == 0.0 and r._step_decay() == 0.0
    r.apply_weight_decay = True          # opt-in, as for the reference's rules
    assert r._hyper8()[7] == 0.1 and r._step_decay() == 0.1


@pytest.mark.parametrize("name", ["AdamW", "RAdam", "Adamax"])
@pytest.mark.parametrize("kw", [dict(lr=-1e-3), dict(lr=float("nan")), dict(lr=float("inf")),
                                dict(epsilon=-1.0), dict(epsilon=float("nan")), dict(beta1=1.0),
                                dict(beta1=-0.1), dict(beta2=1.0), dict(beta2=float("nan"))])
def test_optimizer_arguments_are_checked(name, kw):
    import core.optimizer as O
    with pytest.raises(ValueError):
        getattr(O, name)(**kw)


def test_scheduler_arguments_are_checked():
    import core.optimizer as O
    from core import lr_scheduler as S
    opt = O.SGD(lr=0.1)
    bad = [lambda: S.StepLR(opt, 0), lambda: S.StepLR(opt, 2.5), lambda: S.StepLR(opt, 3, gamma=float("nan")),
           lambda: S.MultiStepLR(opt, [3, 3]), lambda: S.MultiStepLR(opt, [5, 2]), lambda: S.MultiStepLR(opt, [0, 2]),
           lambda: S.MultiStepLR(opt, [1.5]), lambda: S.ExponentialLR(opt, -0.5),
           lambda: S.ExponentialLR(opt, float("inf")), lambda: S.CosineAnnealingLR(opt, 0),
           lambda: S.CosineAnnealingLR(opt, 10, eta_min=-1.0), lambda: S.LinearLR(opt, start_factor=0.0),
           lambda: S.LinearLR(opt, start_factor=1.5), lambda: S.LinearLR(opt, end_factor=2.0),
           lambda: S.LinearLR(opt, total_iters=0)]
    for make in bad:
        with pytest.raises(ValueError):
            make()
    assert opt.lr == 0.1                  # a refused scheduler leaves the learning rate alone
