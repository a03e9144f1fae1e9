"""Conv2D / MaxPool2D host logic without a GPU: the padding / output-shape helper the layers share,
the argument checks, and the float64 numpy oracle (oracle/ref_conv.py) pinned against torch's
conv2d / max_pool2d on the CPU (torch is test infrastructure here; nothing on the product path
imports it)."""
import numpy as np
import pytest

import ref_conv as RC
import ref_numpy as R
from core.layers import window_geometry


@pytest.mark.parametrize("size", [1, 2, 5, 7, 8, 28])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("s", [1, 2, 3])
def test_window_geometry_matches_its_definition(size, k, s):
    (o_same, _), (p_same, _) = window_geometry((size, 1), (k, 1), (s, 1), "SAME")
    assert o_same == int(np.ceil(size / s)) and p_same == (k - 1) // 2
    # every SAME window holds at least one real element and lies within the K - 1 padded positions
    after = k - 1 - p_same
    for o in range(o_same):
        start = o * s - p_same
        assert start <= size - 1 and start + k - 1 >= 0 and start + k - 1 <= size - 1 + after
    if size < k:
        with pytest.raises(ValueError):
            window_geometry((size, 1), (k, 1), (s, 1), "VALID")
    else:
        (o_valid, _), (p_valid, _) = window_geometry((size, 1), (k, 1), (s, 1), "VALID")
        assert o_valid == (size - k) // s + 1 and p_valid == 0
        assert (o_valid - 1) * s + k <= size


def test_window_geometry_two_dimensions():
    # H != W, each dimension on its own window and stride; an even window pads more after than before
    assert window_geometry((28, 20), (5, 2), (2, 3), "SAME") == ((14, 7), (2, 0))
    assert window_geometry((28, 20), (5, 2), (2, 3), "VALID") == ((12, 7), (0, 0))
    assert window_geometry((6, 9), (4, 3), (1, 2), "SAME") == ((6, 5), (1, 1))
    with pytest.raises(ValueError):
        window_geometry((28, 1), (3, 2), (1, 1), "VALID")
    with pytest.raises(ValueError):
        window_geometry((28, 28), (3, 3), (1, 1), "same")


def test_layer_argument_checks():
    from core.layers import Conv2D, MaxPool2D
    for bad in [dict(kernel=(3, 3, 1)), dict(kernel=(3, 0, 1, 4)), dict(kernel=(3, 3, 1, 4), stride=0),
                dict(kernel=(3, 3, 1, 4), stride=(1, 2, 3)), dict(kernel=(3, 3, 1, 4), padding="FULL")]:
        with pytest.raises(ValueError):
            Conv2D(**bad)
    for bad in [dict(pool_size=0), dict(stride=(2, -1)), dict(padding="valid")]:
        with pytest.raises(ValueError):
            MaxPool2D(**bad)


def _torch_same_pad(k):
    return (k - 1) // 2, k - 1 - (k - 1) // 2


@pytest.mark.parametrize("kernel,stride,padding", [
    ((3, 3, 3, 4), (1, 1), "SAME"), ((2, 2, 2, 3), (1, 1), "SAME"), ((4, 2, 3, 5), (2, 3), "SAME"),
    ((5, 5, 1, 8), (2, 2), "SAME"), ((3, 1, 2, 2), (3, 1), "VALID"), ((1, 1, 4, 3), (2, 2), "VALID"),
    ((3, 3, 2, 4), (2, 1), "VALID"),
])
def test_oracle_conv2d_matches_torch(kernel, stride, padding):
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    rng = np.random.RandomState(sum(kernel) + 7 * stride[0] + stride[1])
    KH, KW, C, O = kernel
    x = rng.standard_normal((2, 9, 7, C))
    w = rng.standard_normal(kernel)
    b = rng.standard_normal((1, O))
    g = None
    rx, rw, rb = R.RefTensor(x, True), R.RefTensor(w, True), R.RefTensor(b, True)
    y = RC.conv2d(rx, rw, rb, stride, padding)
    g = rng.standard_normal(y.values.shape)
    y.backward(g)

    tx = torch.tensor(x.transpose(0, 3, 1, 2), requires_grad=True)
    tw = torch.tensor(w.transpose(3, 2, 0, 1), requires_grad=True)
    tb = torch.tensor(b[0], requires_grad=True)
    inp = tx
    if padding == "SAME":
        ph, pw = _torch_same_pad(KH), _torch_same_pad(KW)
        inp = F.pad(tx, (pw[0], pw[1], ph[0], ph[1]))
    ty = F.conv2d(inp, tw, tb, stride=stride)
    ty.backward(torch.tensor(g.transpose(0, 3, 1, 2)))
    np.testing.assert_allclose(y.values, ty.detach().numpy().transpose(0, 2, 3, 1), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(rx.grad, tx.grad.numpy().transpose(0, 2, 3, 1), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(rw.grad, tw.grad.numpy().transpose(2, 3, 1, 0), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(rb.grad, tb.grad.numpy()[None], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("pool,stride,padding", [
    ((2, 2), None, "VALID"), ((3, 3), (2, 2), "VALID"), ((3, 3), (1, 1), "SAME"), ((2, 2), (2, 2), "SAME"),
    ((2, 3), (1, 2), "SAME"),
])
def test_oracle_maxpool2d_matches_torch(pool, stride, padding):
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    rng = np.random.RandomState(pool[0] * 3 + pool[1])
    x = rng.permutation(2 * 9 * 8 * 3).reshape(2, 9, 8, 3).astype(np.float64) - 100.0   # tie-free
    rx = R.RefTensor(x, True)
    y = RC.maxpool2d(rx, pool, stride, padding)
    g = rng.standard_normal(y.values.shape)
    y.backward(g)

    s = pool if stride is None else stride
    tx = torch.tensor(x.transpose(0, 3, 1, 2), requires_grad=True)
    inp = tx
    if padding == "SAME":
        ph, pw = _torch_same_pad(pool[0]), _torch_same_pad(pool[1])
        inp = F.pad(tx, (pw[0], pw[1], ph[0], ph[1]), value=-np.inf)
    ty = F.max_pool2d(inp, pool, stride=s)
    ty.backward(torch.tensor(g.transpose(0, 3, 1, 2)))
    assert np.array_equal(y.values, ty.detach().numpy().transpose(0, 2, 3, 1))
    np.testing.assert_allclose(rx.grad, tx.grad.numpy().transpose(0, 2, 3, 1), rtol=1e-12, atol=1e-12)


def test_oracle_maxpool2d_ties_nan_and_inf():
    """ties go to the first element of the row-major window, a NaN is selected (first one) and
    propagates, an all -inf window selects its first real element even under SAME padding"""
    x = np.zeros((1, 2, 2, 1))
    rx = R.RefTensor(x, True)
    y = RC.maxpool2d(rx, (2, 2))
    y.backward(np.ones((1, 1, 1, 1)))
    assert rx.grad[0, :, :, 0].tolist() == [[1.0, 0.0], [0.0, 0.0]]
    x = np.array([1.0, np.nan, 5.0, np.nan]).reshape(1, 2, 2, 1)
    rx = R.RefTensor(x, True)
    y = RC.maxpool2d(rx, (2, 2))
    y.backward(np.full((1, 1, 1, 1), 2.0))
    assert np.isnan(y.values).all() and rx.grad[0, :, :, 0].tolist() == [[0.0, 2.0], [0.0, 0.0]]
    x = np.full((1, 3, 3, 1), -np.inf)
    rx = R.RefTensor(x, True)
    y = RC.maxpool2d(rx, (3, 3), (1, 1), "SAME")
    y.backward(np.ones((1, 3, 3, 1)))
    # window of output (0, 0) covers rows/cols -1..1: its first real element is (0, 0)
    assert rx.grad[0, 0, 0, 0] == 4.0 and rx.grad.sum() == 9.0
