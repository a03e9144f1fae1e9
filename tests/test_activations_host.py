"""Elementwise activations (LeakyReLU, ELU, GELU, Softplus, SiLU) without a GPU: the float64 oracle
(oracle/ref_activations.py) pinned against torch's float64 autograd on the CPU away from x = 0, the
oracle's conventions at 0, +-inf and NaN, every argument the layers refuse and their read-only
configuration.  torch is test infrastructure here; nothing on the product path imports it."""
import numpy as np
import pytest

import ref_activations as RA
import ref_numpy as R

# (kind, param): the slopes and alphas the device tests use
CASES = [("leaky_relu", 0.0), ("leaky_relu", 0.01), ("leaky_relu", 0.2), ("elu", 0.5), ("elu", 1.0), ("elu", 2.0),
         ("gelu", None), ("gelu_tanh", None), ("softplus", None), ("silu", None)]


def _ids(case):
    return case[0] if case[1] is None else "%s-%g" % case


def _torch(x, kind, param):
    """(y, dy/dx) from torch's float64 autograd"""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    t = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    y = {"leaky_relu": lambda: F.leaky_relu(t, param),
         "elu": lambda: F.elu(t, param),
         "gelu": lambda: F.gelu(t),
         "gelu_tanh": lambda: F.gelu(t, approximate="tanh"),
         "softplus": lambda: torch.logaddexp(t, torch.zeros_like(t)),
         "silu": lambda: F.silu(t)}[kind]()
    y.sum().backward()
    return y.detach().numpy(), t.grad.numpy()


def _close(a, b, tol):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape
    assert np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)), initial=0.0) <= tol


@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_oracle_matches_torch_away_from_zero(case):
    kind, param = case
    rng = np.random.RandomState(len(kind))
    x = np.concatenate([rng.standard_normal(400) * 3.0, rng.uniform(-40.0, 40.0, 200),
                        [-700.0, -35.0, -9.0, 9.0, 35.0, 700.0]])
    x = x[np.abs(x) > 1e-3]
    y, d = RA.terms(x, kind, param)
    ty, td = _torch(x, kind, RA.DEFAULT_PARAM.get(kind) if param is None else param)
    _close(y, ty, 1e-14)
    _close(d, td, 1e-13)
    # the RefTensor node agrees with the plain function, for a non-unit upstream gradient
    g = rng.standard_normal(x.shape)
    a = R.RefTensor(x, True)
    node = RA.activation(a, kind, param)
    node.backward(g)
    assert np.array_equal(node.values, y)
    assert np.array_equal(a.grad, RA.value_and_grad(x, kind, param, g)[1])
    assert np.array_equal(a.grad, g * d)


def test_kink_goes_to_the_nonnegative_branch():
    for z in (0.0, -0.0):
        x = np.array([z])
        for kind, param in CASES:
            y, d = RA.terms(x, kind, param)
            if kind in ("leaky_relu", "elu"):
                assert y[0] == 0.0 and d[0] == 1.0, (kind, param)
            elif kind == "softplus":
                assert y[0] == np.log(2.0) and d[0] == 0.5
            else:
                assert y[0] == 0.0 and d[0] == 0.5, kind
    # LeakyReLU(0.0) is the reference's ReLU, clip(x, 0.0) with the x >= 0 mask, on finite inputs
    rng = np.random.RandomState(1)
    x = np.concatenate([rng.standard_normal(200), [0.0, -0.0, 1e300, -1e300, 5e-324, -5e-324]])
    g = rng.standard_normal(x.shape)
    a, b = R.RefTensor(x, True), R.RefTensor(x, True)
    la, lb = RA.activation(a, "leaky_relu", 0.0), R.clip(b, 0.0)
    la.backward(g)
    lb.backward(g)
    assert np.array_equal(la.values, lb.values) and np.array_equal(a.grad, b.grad)


@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_oracle_nan_inf_and_large_finite_inputs(case):
    kind, param = case
    p = RA.DEFAULT_PARAM.get(kind, 0.0) if param is None else param
    # NaN in, NaN out, in the value and the derivative
    y, d = RA.terms(np.array([np.nan]), kind, param)
    assert np.isnan(y[0]) and np.isnan(d[0])
    # +-inf: the limits of the function and of its derivative
    y, d = RA.terms(np.array([np.inf, -np.inf]), kind, param)
    lim_y = {"leaky_relu": [np.inf, -np.inf * p if p else 0.0], "elu": [np.inf, -p]}.get(kind, [np.inf, 0.0])
    lim_d = {"leaky_relu": [1.0, p], "elu": [1.0, 0.0]}.get(kind, [1.0, 0.0])
    assert np.array_equal(y, lim_y) and np.array_equal(d, lim_d), (y, d)
    # every finite x gives a finite value and derivative
    big = np.array([1e300, -1e300, 3e38, -3e38, 1e20, -1e20, 7e12, -7e12, 1e-300, -1e-300])
    y, d = RA.terms(big, kind, param)
    assert np.all(np.isfinite(y)) and np.all(np.isfinite(d))


def test_oracle_gelu_tanh_matches_its_tanh_form():
    x = np.linspace(-6.0, 6.0, 1001)
    u = np.sqrt(2.0 / np.pi) * (x + 0.044715 * x ** 3)
    y, _ = RA.terms(x, "gelu_tanh")
    _close(y, 0.5 * x * (1.0 + np.tanh(u)), 1e-15)


# ---------------------------------------------------------------------------- the layers
def _layers():
    from core.layers import ELU, GELU, LeakyReLU, SiLU, Softplus
    return LeakyReLU, ELU, GELU, Softplus, SiLU


@pytest.mark.parametrize("value", [float("nan"), float("inf"), -float("inf"), "1", None, True, [0.1]])
def test_slope_and_alpha_refusals(value):
    LeakyReLU, ELU, _, _, _ = _layers()
    with pytest.raises(ValueError, match="slope"):
        LeakyReLU(value)
    with pytest.raises(ValueError, match="alpha"):
        ELU(value)


@pytest.mark.parametrize("value", ["exact", "TANH", "", None, 1, True])
def test_gelu_approximate_refusals(value):
    GELU = _layers()[2]
    with pytest.raises(ValueError, match="approximate"):
        GELU(value)


def test_configuration_is_read_only_and_fixed_at_construction():
    LeakyReLU, ELU, GELU, Softplus, SiLU = _layers()
    leaky, elu, gelu = LeakyReLU(np.float32(0.25)), ELU(2), GELU("tanh")
    assert leaky.slope == 0.25 and type(leaky.slope) is float
    assert elu.alpha == 2.0 and type(elu.alpha) is float
    assert gelu.approximate == "tanh"
    assert LeakyReLU().slope == 0.01 and ELU().alpha == 1.0 and GELU().approximate == "none"
    assert LeakyReLU(-0.5).slope == -0.5 and ELU(0).alpha == 0.0
    for layer, attr, value in ((leaky, "slope", 0.5), (elu, "alpha", 1.0), (gelu, "approximate", "none")):
        with pytest.raises(AttributeError):
            setattr(layer, attr, value)
        assert getattr(layer, attr) == {"slope": 0.25, "alpha": 2.0, "approximate": "tanh"}[attr]
    for cls in (LeakyReLU, ELU, GELU, Softplus, SiLU):
        layer = cls()
        assert layer.params == {} and layer.inputs is None

