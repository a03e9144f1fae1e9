"""Size-independent properties at BASELINE.json's full sizes (configs 3 and 4), where the oracle
would take too long: linearity, round trips, row/column-sum consistency, and spot checks of
random entries of the big GEMM against float64 dot products."""
import numpy as np
import pytest

import op_cases
from support import gemm_route

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    import core._backend as be
    be.init()
    return be


def test_elementwise_sweep_2e27(be):
    n_rows, n_cols = (1 << 27) // 1024, 1024
    rng = np.random.RandomState(0)
    a = rng.rand(n_rows, n_cols).astype(np.float32)
    bias = rng.rand(1, n_cols).astype(np.float32)
    da, dbias = be.from_numpy(a), be.from_numpy(bias)
    # add / mul, same shape: compare a strided sample with numpy
    s = be.ew(be.ADD, da, da)
    m = be.ew(be.MUL, da, da)
    hs, hm = s.numpy(), m.numpy()
    assert np.array_equal(hs[::997], a[::997] + a[::997])
    assert np.array_equal(hm[::997], a[::997] * a[::997])
    # bias add (row broadcast) and its un-broadcast: sum_rows(a + b) == sum_rows(a) + R*b
    ab = be.ew(be.ADD, da, dbias)
    assert np.array_equal(ab.numpy()[::997], a[::997] + bias)
    cs = be.unbroadcast(ab, (1, n_cols)).numpy()
    ref = a.astype(np.float64).sum(axis=0, keepdims=True) + n_rows * bias.astype(np.float64)
    assert op_cases.rel_err(cs, ref) <= 1e-5
    # relu forward/backward: idempotent, mask consistent
    x = be.ew(be.SCALE, da, p0=2.0, p1=-1.0)            # values in [-1, 1)
    r = be.relu_fwd(x)
    rr = be.relu_fwd(r)
    hx, hr = x.numpy(), r.numpy()
    assert np.array_equal(hr, rr.numpy())
    assert np.array_equal(hr[::997], np.maximum(hx[::997], 0))
    g = be.relu_bwd(da, x).numpy()
    assert np.array_equal(g[::997], a[::997] * (hx[::997] >= 0))
    # full reductions
    assert op_cases.rel_err(be.reduce(be.RED_SUM, da).numpy(), a.astype(np.float64).sum()) <= 1e-5
    assert be.reduce(be.RED_MAX, da).numpy() == a.max()


def test_row_gather_permutation_roundtrip(be):
    """BatchIterator's shuffle on a 50000 x 784 table: gather by a permutation then by its inverse
    is the identity; scatter is the inverse of gather"""
    rng = np.random.RandomState(1)
    x = rng.rand(50000, 784).astype(np.float32)
    perm = rng.permutation(50000)
    inv = np.argsort(perm)
    dx = be.from_numpy(x)
    g = be.gather_rows(dx, be.upload_index(perm), 50000)
    assert np.array_equal(g.numpy()[:64], x[perm[:64]])
    back = be.gather_rows(g, be.upload_index(inv), 50000)
    assert np.array_equal(back.numpy(), x)
    sc = be.scatter_rows(g, be.upload_index(perm), 50000, x.shape)
    assert np.array_equal(sc.numpy(), x)


@pytest.mark.parametrize("cg", [1, 2])
def test_wide_gemm_spot_check(be, cg):
    """config 4's GEMM shape (8192 x 4096 x 4096) in all three orientations of a Dense layer;
    512 random output entries checked against float64 dot products, plus linearity in A"""
    with gemm_route(cta_group=cg):
        rng = np.random.RandomState(2)
        M, N, K = 8192, 4096, 4096
        a = rng.rand(M, K).astype(np.float32)
        w = ((rng.rand(K, N) - 0.5) * 0.05).astype(np.float32)
        g = rng.standard_normal((M, N)).astype(np.float32)
        da, dw, dg = be.from_numpy(a), be.from_numpy(w), be.from_numpy(g)
        ii, jj = rng.randint(0, M, 512), rng.randint(0, N, 512)
        a64, w64, g64 = a.astype(np.float64), w.astype(np.float64), g.astype(np.float64)

        y = be.matmul(da, dw).numpy()                                    # forward  X @ W
        ref = np.einsum("ik,ki->i", a64[ii], w64[:, jj])
        assert op_cases.rel_err(y[ii, jj], ref) <= 1e-5
        dx = be.matmul(dg, dw, tb=True).numpy()                          # dX = G @ W.T
        kk = rng.randint(0, K, 512)
        ref = np.einsum("ij,ij->i", g64[ii], w64[kk])
        assert op_cases.rel_err(dx[ii, kk], ref) <= 1e-5
        dwt = be.matmul(da, dg, ta=True).numpy()                         # dW = X.T @ G
        ref = np.einsum("ki,ki->i", a64[:, kk], g64[:, jj])
        assert op_cases.rel_err(dwt[kk, jj], ref) <= 1e-5
        # linearity: (2a) @ w == 2 (a @ w) exactly (scaling by 2 is exact in every split plane)
        y2 = be.matmul(be.ew(be.SCALE, da, p0=2.0, p1=0.0), dw).numpy()
        assert np.array_equal(y2, 2.0 * y)
