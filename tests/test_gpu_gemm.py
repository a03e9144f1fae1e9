"""tcgen05 3xTF32 GEMM and its tf32 split pre-pass against numpy float64 products, through the
C ABI.  Tolerance: rel 1e-5 of max|ref| (north_star per-op tolerance; the 3xTF32 error model is
~2^-21 per product term)."""
import numpy as np
import pytest

import op_cases
from support import gemm_route

pytestmark = pytest.mark.gpu

TOL = 1e-5


@pytest.fixture(scope="module")
def be():
    import core._backend as be
    be.init()
    return be


def _ref(a, b, ta, tb, bias):
    A = a.astype(np.float64).T if ta else a.astype(np.float64)
    B = b.astype(np.float64).T if tb else b.astype(np.float64)
    out = A @ B
    if bias is not None:
        out = out + bias.astype(np.float64)
    return out


def test_split_planes_reconstruct(be):
    rng = np.random.RandomState(0)
    for R_, C_ in ((64, 64), (130, 70), (257, 33), (5, 1000)):
        x = (rng.standard_normal((R_, C_)) * 10 ** rng.uniform(-3, 3, (R_, C_))).astype(np.float32)
        d = be.from_numpy(x)
        hi, lo, ldp = be.split_planes(d, transposed=False, also_other=True)
        hit, lot, ldt = be.split_planes(d, transposed=True)
        H, L = hi.numpy()[:, :C_], lo.numpy()[:, :C_]
        HT, LT = hit.numpy()[:, :R_], lot.numpy()[:, :R_]
        # hi/lo are tf32 values (13 low mantissa bits clear) and hi + lo ~= x to ~2^-21
        assert np.all(H.view(np.uint32) & 0x1FFF == 0) and np.all(L.view(np.uint32) & 0x1FFF == 0)
        assert np.max(np.abs((H.astype(np.float64) + L) - x) / np.maximum(np.abs(x), 1e-30)) < 2.0 ** -20
        assert np.array_equal(HT, H.T) and np.array_equal(LT, L.T)


def _bf16_rn(x):
    b = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    b = (b + 0x7FFF + ((b >> 16) & 1)) >> 16
    return b.astype(np.uint16)


def test_mixed_split_planes(be):
    """hi = tf32(x) in an fp32 plane, h16 = bf16(x), l16 = bf16(x - hi); pad columns are zero"""
    rng = np.random.RandomState(0)
    for R_, C_ in ((64, 64), (130, 70), (257, 33), (5, 1000), (3, 1)):
        x = (rng.standard_normal((R_, C_)) * 10 ** rng.uniform(-3, 3, (R_, C_))).astype(np.float32)
        d = be.from_numpy(x)
        hi, h16, l16, ld = be.split_planes_mix(d)
        assert ld % 8 == 0 and ld >= C_
        H = hi.numpy()
        H16 = h16.numpy().view(np.uint16).reshape(R_, ld)
        L16 = l16.numpy().view(np.uint16).reshape(R_, ld)
        assert np.all(H[:, C_:] == 0) and np.all(H16[:, C_:] == 0) and np.all(L16[:, C_:] == 0)
        H = H[:, :C_]
        assert np.all(H.view(np.uint32) & 0x1FFF == 0)
        assert np.max(np.abs(H.astype(np.float64) - x) / np.abs(x)) <= 2.0 ** -11
        assert np.array_equal(H16[:, :C_], _bf16_rn(x))
        assert np.array_equal(L16[:, :C_], _bf16_rn(x - H))


@pytest.mark.parametrize("split,mn_major", [("mix", True), ("tf32x3", True), ("tf32x3", False)])
@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("shape", [
    (128, 256, 32), (128, 256, 64), (256, 256, 128), (256, 512, 96), (384, 768, 200),
    (100, 300, 52), (129, 257, 36), (1000, 520, 260), (2048, 1024, 512),
])
def test_tf32x3_gemm_shapes(be, cg, shape, split, mn_major):
    """NN / NT / TN products.  split = "mix": tf32 main term + bf16 cross terms (the default path);
    "tf32x3": three tf32 MMAs.  mn_major=True feeds transposed operands MN-major from the plain
    planes (default), False goes through transposed planes (both operands K-major)"""
    M, N, K = shape
    with gemm_route(cta_group=cg, TC_MN_MAJOR=mn_major, TC_SPLIT=split, TC_MIN_MNK=0):
        rng = np.random.RandomState(M * 7 + N * 3 + K)
        a = rng.standard_normal((M, K)).astype(np.float32)
        b = rng.standard_normal((K, N)).astype(np.float32)
        bias = rng.standard_normal((1, N)).astype(np.float32)
        da, db, dbias = be.from_numpy(a), be.from_numpy(b), be.from_numpy(bias)
        out = be.matmul(da, db, bias=dbias).numpy()
        ref = _ref(a, b, False, False, bias)
        assert op_cases.rel_err(out, ref) <= TOL
        # NT: (M,K) @ (N,K)^T
        bt = np.ascontiguousarray(b.T)
        out = be.matmul(da, be.from_numpy(bt), tb=True).numpy()
        assert op_cases.rel_err(out, _ref(a, bt, False, True, None)) <= TOL
        # TN: (K,M)^T @ (K,N), accumulate into an existing buffer
        at = np.ascontiguousarray(a.T)
        c0 = rng.standard_normal((M, N)).astype(np.float32)
        dc = be.from_numpy(c0)
        be.matmul(be.from_numpy(at), db, ta=True, out=dc, accumulate=True)
        assert op_cases.rel_err(dc.numpy(), _ref(at, b, True, False, None) + c0) <= TOL
        # relu epilogue
        out = be.matmul(da, db, bias=dbias, relu=True).numpy()
        assert op_cases.rel_err(out, np.maximum(ref, 0)) <= TOL


@pytest.mark.parametrize("split", ["mix", "tf32x3"])
def test_fused_activation_outputs(be, split):
    """act=True: one launch returns the pre-activation, its ReLU and the ReLU's operand planes,
    which the next product consumes as-is; mask_src form returns out * (mask_src >= 0)"""
    rng = np.random.RandomState(5)
    M, N, K = 300, 264, 136
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = rng.standard_normal((K, N)).astype(np.float32)
    bias = rng.standard_normal((1, N)).astype(np.float32)
    w2 = rng.standard_normal((N, 72)).astype(np.float32)
    with gemm_route(TC_MIN_MNK=0, TC_SPLIT=split):
        z, act = be.matmul(be.from_numpy(a), be.from_numpy(b), bias=be.from_numpy(bias), act=True)
        zr = _ref(a, b, False, False, bias)
        assert op_cases.rel_err(z.numpy(), zr) <= TOL
        assert np.array_equal(act.numpy(), np.maximum(z.numpy(), 0))
        # the planes attached to `act` must equal a fresh split of it
        key = "m" if split == "mix" else "p"
        fused = [p.numpy() for p in act.split[key][:-1]]
        act.split = None
        fresh_planes = be.split_planes_mix(act) if split == "mix" else be.split_planes(act, transposed=False)
        N_ = act.shape[1]
        for f, g in zip(fused, [p.numpy() for p in fresh_planes[:-1]]):
            w = N_ if f.shape[1] >= N_ else N_ // 2       # bf16 planes are kept as half-width fp32
            assert np.array_equal(f[:, :w], g[:, :w])
        # and the next product consumes them
        act2 = be.from_numpy(np.maximum(z.numpy(), 0))
        y_fused = be.matmul(act, be.from_numpy(w2)).numpy()
        y_plain = be.matmul(act2, be.from_numpy(w2)).numpy()
        assert np.array_equal(y_fused, y_plain)
        pre = rng.standard_normal((M, N)).astype(np.float32)
        g, masked = be.matmul(be.from_numpy(a), be.from_numpy(b), act=True, mask_src=be.from_numpy(pre))
        assert np.array_equal(masked.numpy(), g.numpy() * (pre >= 0))


def _meta(rec):
    w = rec.numpy().view(np.uint32)
    return dict(absmax=w[0:1].view(np.float32)[0], need_stats=int(w[1]), exp=int(w[2:3].view(np.int32)[0]),
                safe=int(w[3]), n_small=int(w[4]), n_nz=int(w[5]))


def test_f16_split_planes(be):
    """scaled fp16 hi/lo planes (gemm_f16.cu): bit-identical to the numpy model of
    oracle/split_error_model.py, pad columns zero, record = (absmax, exponent, counts, safe)"""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import split_error_model as S
    rng = np.random.RandomState(0)
    for R_, C_, scale in ((64, 64, 1.0), (130, 70, 3e-4), (257, 33, 7e5), (5, 1000, 1e-12), (3, 1, 2.0)):
        x = (rng.standard_normal((R_, C_)) * scale * np.exp2(rng.randint(-12, 1, (R_, C_)))).astype(np.float32)
        d = be.from_numpy(x)
        hf, l16, ld, meta, _, relu_mode = be.split_planes_f16(d)
        assert ld % 8 == 0 and ld >= C_ and relu_mode == 0
        H = hf.numpy().view(np.float16).reshape(R_, ld)
        L = l16.numpy().view(np.float16).reshape(R_, ld)
        m = _meta(meta)
        rh, rl, e = S.f16_planes(x)
        assert m["exp"] == e and m["safe"] == 1 and m["absmax"] == np.max(np.abs(x))
        assert m["n_nz"] == int(np.sum(x != 0))
        assert np.all(H[:, C_:] == 0) and np.all(L[:, C_:] == 0)
        assert np.array_equal(H[:, :C_].astype(np.float32), rh)
        assert np.array_equal(L[:, :C_].astype(np.float32), rl)
    # relu applied on load (a LazyReLU is split from its pre-activation)
    z = be.from_numpy(rng.standard_normal((64, 96)).astype(np.float32))
    lazy = be.LazyReLU(z)
    hf, l16, ld, meta, src, relu_mode = be.split_planes_f16(lazy)
    assert relu_mode == 1 and src is z and lazy._real is None
    rh, rl, e = S.f16_planes(np.maximum(z.numpy(), 0))
    assert np.array_equal(hf.numpy().view(np.float16).reshape(64, ld)[:, :96].astype(np.float32), rh)


@pytest.mark.parametrize("shape", [
    (128, 256, 64), (256, 256, 128), (256, 512, 96), (384, 768, 200), (100, 300, 52), (129, 257, 36),
    (1000, 520, 260), (2048, 1024, 512), (64, 64, 32), (300, 72, 4100),
])
def test_f16_gemm_shapes(be, shape):
    """default path: NN / NT / TN (+ accumulate) / relu epilogue on operands of very different
    magnitudes (the per-tensor scale exponents are exercised), rel 1e-5 of max|ref|"""
    M, N, K = shape
    with gemm_route(TC_MIN_MNK=0, TC_SPLIT="f16"):
        rng = np.random.RandomState(M * 7 + N * 3 + K)
        a = (rng.standard_normal((M, K)) * 3.7e-6).astype(np.float32)
        b = (rng.standard_normal((K, N)) * 4.1e4).astype(np.float32)
        bias = rng.standard_normal((1, N)).astype(np.float32)
        da, db, dbias = be.from_numpy(a), be.from_numpy(b), be.from_numpy(bias)
        assert be.use_tensor_cores(M, N, K, be.F32)
        ref = _ref(a, b, False, False, bias)
        assert op_cases.rel_err(be.matmul(da, db, bias=dbias).numpy(), ref) <= TOL
        assert _meta(da.split["f"][3])["safe"] == 1 and _meta(db.split["f"][3])["safe"] == 1
        bt = np.ascontiguousarray(b.T)
        assert op_cases.rel_err(be.matmul(da, be.from_numpy(bt), tb=True).numpy(), _ref(a, bt, False, True, None)) <= TOL
        at = np.ascontiguousarray(a.T)
        c0 = rng.standard_normal((M, N)).astype(np.float32)
        outs = []
        for _ in range(2):
            dc = be.from_numpy(c0)
            be.matmul(be.from_numpy(at), db, ta=True, out=dc, accumulate=True)
            outs.append(dc.numpy())
        assert op_cases.rel_err(outs[0], _ref(at, b, True, False, None) + c0) <= TOL
        assert np.array_equal(outs[0], outs[1])                       # run-to-run identical
        out = be.matmul(da, db, bias=dbias, relu=True).numpy()
        assert op_cases.rel_err(out, np.maximum(ref, 0)) <= TOL


@pytest.mark.parametrize("shape", [(256, 512, 128), (384, 768, 200), (300, 300, 96), (1000, 520, 260),
                                   (2048, 1024, 512), (512, 1280, 4100)])
def test_f16_gemm_multicast_clusters(be, shape):
    """optional cluster shape of the default kernel: two CTA pairs on adjacent tile columns share
    their A rows by TMA multicast (odd tile-column counts leave the second pair of the last cluster
    without a tile).  Bit-identical to the pair kernel: same products, same order."""
    M, N, K = shape
    with gemm_route(TC_MIN_MNK=0, TC_SPLIT="f16"):
        rng = np.random.RandomState(M + 5 * N + K)
        a = rng.standard_normal((M, K)).astype(np.float32)
        b = rng.standard_normal((K, N)).astype(np.float32)
        bias = rng.standard_normal((1, N)).astype(np.float32)
        at, bt = np.ascontiguousarray(a.T), np.ascontiguousarray(b.T)
        res = {}
        for cl in (2, 4):
            with gemm_route(f16_cluster=cl):
                da, db = be.from_numpy(a), be.from_numpy(b)
                res[cl] = [be.matmul(da, db, bias=be.from_numpy(bias)).numpy(),
                           be.matmul(da, be.from_numpy(bt), tb=True).numpy(),
                           be.matmul(be.from_numpy(at), db, ta=True).numpy()]
        assert op_cases.rel_err(res[4][0], _ref(a, b, False, False, bias)) <= TOL
        for x, y in zip(res[2], res[4]):
            assert np.array_equal(x, y)


def test_f16_fused_outputs(be):
    """act=True on the default path: the launch stores the pre-activation and records max|relu(z)| for
    the next split (the fp32 activation is a LazyReLU, never written); the next product consumes it.
    mask_src form: second output = out * (mask_src >= 0), with its statistics"""
    rng = np.random.RandomState(5)
    M, N, K = 300, 264, 136
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = rng.standard_normal((K, N)).astype(np.float32)
    bias = rng.standard_normal((1, N)).astype(np.float32)
    w2 = rng.standard_normal((N, 72)).astype(np.float32)
    with gemm_route(TC_MIN_MNK=0, TC_SPLIT="f16"):
        z, act = be.matmul(be.from_numpy(a), be.from_numpy(b), bias=be.from_numpy(bias), act=True)
        assert op_cases.rel_err(z.numpy(), _ref(a, b, False, False, bias)) <= TOL
        assert type(act) is be.LazyReLU and act._real is None
        m = _meta(act.split["stat"])
        assert m["absmax"] == np.max(np.maximum(z.numpy(), 0)) and m["need_stats"] == 0
        y_fused = be.matmul(act, be.from_numpy(w2)).numpy()
        assert act._real is None                                   # still never materialised
        y_plain = be.matmul(be.from_numpy(np.maximum(z.numpy(), 0)), be.from_numpy(w2)).numpy()
        assert np.array_equal(y_fused, y_plain)
        assert np.array_equal(act.numpy(), np.maximum(z.numpy(), 0))
        pre = rng.standard_normal((M, N)).astype(np.float32)
        g, masked = be.matmul(be.from_numpy(a), be.from_numpy(b), act=True, mask_src=be.from_numpy(pre))
        assert np.array_equal(masked.numpy(), g.numpy() * (pre >= 0))
        assert _meta(masked.split["stat"])["absmax"] == np.max(np.abs(masked.numpy()))
        y1 = be.matmul(masked, be.from_numpy(w2)).numpy()
        y2 = be.matmul(be.from_numpy(masked.numpy()), be.from_numpy(w2)).numpy()
        assert np.array_equal(y1, y2)


def test_f16_guard_falls_back_on_device(be):
    """operands outside the guard (rows scaled by 1e-30, Inf) are flagged by the split kernel and the
    product is done by the conditional mixed-split launches: componentwise accuracy as the mixed
    split's, non-finite values propagate like numpy's, and a fused relu output of a fallback product
    still feeds the next product (statistics recomputed on demand).  All-zero operands are safe."""
    rng = np.random.RandomState(1)
    M, N, K = 512, 384, 512
    a = rng.standard_normal((M, K)).astype(np.float32)
    a[::2] *= np.float32(1e-30)
    b = rng.standard_normal((K, N)).astype(np.float32)
    with gemm_route(TC_MIN_MNK=0, TC_SPLIT="f16"):
        da, db = be.from_numpy(a), be.from_numpy(b)
        z, act = be.matmul(da, db, act=True)
        assert _meta(da.split["f"][3])["safe"] == 0 and _meta(db.split["f"][3])["safe"] == 1
        a64, b64 = a.astype(np.float64), b.astype(np.float64)
        comp = np.max(np.abs(z.numpy() - a64 @ b64) / (np.abs(a64) @ np.abs(b64)))
        assert comp <= 5e-6, comp
        assert _meta(act.split["stat"])["need_stats"] == 1
        w2 = rng.standard_normal((N, 128)).astype(np.float32)
        nxt = be.matmul(act, be.from_numpy(w2)).numpy()
        assert _meta(act.split["f"][3])["absmax"] == np.max(np.maximum(z.numpy(), 0))
        ref2 = np.maximum(z.numpy().astype(np.float64), 0) @ w2.astype(np.float64)
        comp2 = np.max(np.abs(nxt - ref2) / (np.maximum(z.numpy().astype(np.float64), 0) @ np.abs(w2.astype(np.float64)) + 1e-300))
        assert comp2 <= 5e-6, comp2
        bad = rng.standard_normal((M, K)).astype(np.float32)
        bad[3, 5] = np.inf
        out = be.matmul(be.from_numpy(bad), db).numpy()
        assert np.all(~np.isfinite(out[3])) and np.all(np.isfinite(np.delete(out, 3, axis=0)))
        zero = be.matmul(be.from_numpy(np.zeros((M, K), np.float32)), db)
        assert np.all(zero.numpy() == 0)


def test_f16_tensor_relative_bound(be):
    """the documented limit of the default split: an element further than 19 binades below its
    tensor's largest is held to 2^-39 of that largest, not to 2^-20 of itself.  One row in 512 scaled
    by 2^-25 stays inside the guard (1/512 of the non-zeros); its entries meet
    |err| <= 2^-19 (|A| @ |B|) + 2^-38 max|A| sum_k |b_kj| and every other row the componentwise 5e-6"""
    rng = np.random.RandomState(2)
    M, N, K = 512, 256, 512
    a = rng.standard_normal((M, K)).astype(np.float32)
    a[7] *= np.float32(2.0 ** -25)
    b = rng.standard_normal((K, N)).astype(np.float32)
    with gemm_route(TC_MIN_MNK=0, TC_SPLIT="f16"):
        da = be.from_numpy(a)
        c = be.matmul(da, be.from_numpy(b)).numpy().astype(np.float64)
        assert _meta(da.split["f"][3])["safe"] == 1
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    err = np.abs(c - a64 @ b64)
    comp = np.abs(a64) @ np.abs(b64)
    bound = 2.0 ** -19 * comp + 2.0 ** -38 * np.max(np.abs(a64)) * np.sum(np.abs(b64), axis=0)[None, :]
    assert np.all(err <= bound)
    others = np.delete(np.arange(M), 7)
    assert np.max(err[others] / comp[others]) <= 5e-6


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("ks", [2, 4])
def test_tf32x3_ordered_split_k(be, cg, ks):
    """forced split-K: same result as the unsplit kernel to rounding, bit-identical run to run"""
    rng = np.random.RandomState(11 * ks + cg)
    M, N, K = 700, 520, 2304
    a = rng.standard_normal((M, K)).astype(np.float32)
    b = rng.standard_normal((K, N)).astype(np.float32)
    bias = rng.standard_normal((1, N)).astype(np.float32)
    c0 = rng.standard_normal((M, N)).astype(np.float32)
    da, db, dbias = be.from_numpy(a), be.from_numpy(b), be.from_numpy(bias)
    ref = _ref(a, b, False, False, bias) + c0
    with gemm_route(TC_MIN_MNK=0, TC_SPLIT="mix", cta_group=cg, ksplit=ks):
        outs = []
        for _ in range(3):
            dc = be.from_numpy(c0)
            be.matmul(da, db, bias=dbias, out=dc, accumulate=True)
            outs.append(dc.numpy())
        assert op_cases.rel_err(outs[0], ref) <= TOL
        assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])


def test_tf32x3_better_than_plain_tf32(be):
    """the split really buys fp32-level accuracy: error well below single-pass TF32 (~5e-4)"""
    rng = np.random.RandomState(1)
    M, N, K = 512, 512, 4096
    a = rng.rand(M, K).astype(np.float32)
    b = rng.rand(K, N).astype(np.float32)
    with gemm_route(TC_MIN_MNK=0):
        out = be.matmul(be.from_numpy(a), be.from_numpy(b)).numpy()
    ref = a.astype(np.float64) @ b.astype(np.float64)
    # all-positive data is the worst case for the tensor core's round-toward-zero accumulation
    # inside a chunk (8 K-blocks = 256 k since r02: between 2e-6 and 3e-6 here, 1.3e-6 on signed data)
    assert op_cases.rel_err(out, ref) <= 3e-6
    # and it is at least as good as numpy's own float32 product on the same data
    assert op_cases.rel_err(out, ref) <= 4 * op_cases.rel_err(a @ b, ref) + 1e-7


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", [(1, 1, 1), (3, 5, 7), (128, 200, 784), (80, 10, 30), (257, 65, 33), (64, 64, 0),
                                   (128, 100, 200), (64, 32, 1000), (30, 30, 4100), (33, 31, 129)])
def test_simt_gemm(be, dtype, shape):
    M, N, K = shape
    rng = np.random.RandomState(M + N + K)
    a = rng.standard_normal((M, K)).astype(dtype)
    b = rng.standard_normal((K, N)).astype(dtype)
    bias = rng.standard_normal((1, N)).astype(dtype)
    tol = 2e-6 if dtype == np.float32 else 1e-13
    with gemm_route(TC_ENABLED=False):
        da, db = be.from_numpy(a), be.from_numpy(b)
        assert op_cases.rel_err(be.matmul(da, db, bias=be.from_numpy(bias)).numpy(), _ref(a, b, False, False, bias)) <= tol
        at, bt = np.ascontiguousarray(a.T), np.ascontiguousarray(b.T)
        assert op_cases.rel_err(be.matmul(be.from_numpy(at), db, ta=True).numpy(), _ref(at, b, True, False, None)) <= tol
        assert op_cases.rel_err(be.matmul(da, be.from_numpy(bt), tb=True).numpy(), _ref(a, bt, False, True, None)) <= tol


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", [(128, 200, 100), (80, 70, 30), (128, 784, 200), (16, 1000, 24)])
def test_simt_gemm_fused_outputs(be, dtype, shape):
    """SIMT path: act=True returns (z, relu(z)); with mask_src (dX form, also through the cluster
    split-K variant) the second output is z * (mask_src >= 0); repeated runs are bit-identical"""
    M, N, K = shape
    rng = np.random.RandomState(M + 3 * N + K)
    a = rng.standard_normal((M, K)).astype(dtype)
    bt = rng.standard_normal((N, K)).astype(dtype)
    pre = rng.standard_normal((M, N)).astype(dtype)
    pre[0, 0] = 0.0
    tol = 2e-6 if dtype == np.float32 else 1e-13
    with gemm_route(TC_ENABLED=False):
        da, dbt = be.from_numpy(a), be.from_numpy(bt)
        ref = a.astype(np.float64) @ bt.astype(np.float64).T
        z, act = be.matmul(da, dbt, tb=True, act=True)
        assert op_cases.rel_err(z.numpy(), ref) <= tol
        assert np.array_equal(act.numpy(), np.maximum(z.numpy(), 0))
        g, masked = be.matmul(da, dbt, tb=True, act=True, mask_src=be.from_numpy(pre))
        assert np.array_equal(g.numpy(), z.numpy())
        assert np.array_equal(masked.numpy(), g.numpy() * (pre >= 0))
