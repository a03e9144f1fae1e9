"""Whole-step parity at BASELINE.json configs[3]'s real width (VERDICT r1, item 3): a 4 x Dense(4096)
MLP, D_in = C = 4096, on the tcgen05 path with the production settings (CTA pairs, tail split-K,
fused Dense+ReLU epilogue chain, fused CE, arena Adam over 67 M parameters) against the oracle --
the batch is 1024 rows so the oracle's float64 step finishes in seconds -- plus the fused
cross-entropy at the config's full 8192 x 4096 logits, and adversarial operands for the TF32+BF16
operand split.  References: /root/reference/core/ops.py:150-163 (dot_), core/losses.py:24-32,
core/optimizer.py:50-79, core/layers.py:43-49,97-98."""
import numpy as np
import pytest

import op_cases
import ref_numpy as R
from support import gemm_route

pytestmark = pytest.mark.gpu

D = 4096
B = 1024


@pytest.fixture(scope="module")
def wide_case():
    """inputs, reference-style initial parameters, and the oracle's forward (float64 parameters
    holding the float32 values: the reference's own state from its second step on)"""
    rng = np.random.RandomState(0)
    x = rng.rand(B, D).astype(np.float32)
    labels = np.eye(D, dtype=np.float32)[rng.randint(0, D, B)]
    np.random.seed(0)
    mlp = R.RefMLP([D, D, D, D], R.RefAdam(lr=1e-3))
    h = D
    init = []
    for layer in mlp.layers:
        if isinstance(layer, R.RefDense):
            layer._init(h)
            h = layer.num_out
            # biases away from zero so the bias path is exercised (the reference starts them at 0)
            b = (rng.standard_normal((1, h)) * 0.05).astype(np.float32)
            init += [layer.w.values.copy(), b]
            layer.w = R.RefTensor(layer.w.values.astype(np.float64), True)
            layer.b = R.RefTensor(b.astype(np.float64), True)
    return dict(x=x, labels=labels, mlp=mlp, init=init)


def _engine_model(init):
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    from core.tensor import Tensor
    layers = []
    for i in range(4):
        d = Dense(D, num_in=D)
        d.params["w"] = Tensor(init[2 * i], requires_grad=True)
        d.params["b"] = Tensor(init[2 * i + 1], requires_grad=True)
        layers.append(d)
        if i < 3:
            layers.append(ReLU())
    net = Net(layers)
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))


@pytest.mark.parametrize("split", ["f16", "mix", "tf32x3"])
def test_wide_mlp_step_matches_oracle(wide_case, split):
    import core._backend as be
    from core.tensor import Tensor
    x, labels, mlp = wide_case["x"], wide_case["labels"], wide_case["mlp"]
    try:
        # cta_group 0 is the production default: CTA pairs, tail split-K on ragged waves
        with gemm_route(TC_SPLIT=split, cta_group=0):
            np.random.seed(1)
            net, model = _engine_model(wide_case["init"])
            params = [p for layer in net.get_parameters() for p in layer.values()]
            assert be.use_tensor_cores(B, D, D, be.F32)
            model.zero_grad()
            loss = model.loss.loss(model.forward(Tensor(x)), Tensor(labels))
            pre = [layer.inputs.values for layer in net.layers if layer.name == "ReLU"]

            # ---- oracle forward; pre-activations within rounding distance of the ReLU kink -------------
            relus = [layer for layer in mlp.layers if isinstance(layer, R.RefReLU)]
            for r in relus:
                r.keep_override = None
            mlp.zero_grad()
            hcur, ref_pre = R.lift(x), []
            for layer in mlp.layers:
                hcur = layer.forward(hcur)
                if isinstance(layer, R.RefDense):
                    ref_pre.append(hcur.values)
            flips = 0
            for z, zr in zip(pre, ref_pre[:3]):
                assert op_cases.rel_err(z, zr) <= 1e-5
                differ = (z >= 0) != (zr >= 0)
                flips += int(differ.sum())
                # only entries that are zero to rounding may land on the other side of the kink
                assert np.all(np.abs(zr[differ]) <= 1e-5 * np.max(np.abs(zr)))
            assert flips <= 256, flips          # of 12.6 M pre-activations (expected: a few tens)

            # ---- oracle backward with the device's masks on those few entries -------------------------
            for r, z in zip(relus, pre):
                r.keep_override = (z >= 0)
            mlp.zero_grad()
            rloss = R.softmax_cross_entropy(mlp.forward(R.lift(x)), labels)
            assert abs(float(loss.values) - float(rloss.values)) <= 1e-5
            loss.backward()
            rloss.backward()
            for k, (p, rp) in enumerate(zip(params, mlp.params())):
                assert op_cases.rel_err(p.grad, rp.grad) <= 1e-5, (split, k)

            # ---- fused arena Adam over all 67 M parameters, fed the engine's own gradients (Adam's
            # first step is -lr*g/(|g|+eps): entries with |g| ~ eps turn a 1e-9 gradient difference into
            # an O(lr) step difference, so both sides get the same gradient) ---------------------------
            p0 = [p.values.astype(np.float64) for p in params]
            g0 = [p.grad.astype(np.float64) for p in params]
            model.step()
            assert model._arena is not None and model._arena["p"].size >= 4 * D * D + 4 * D
            flat_step = R.RefAdam(lr=1e-3)._step(np.concatenate([g.ravel() for g in g0]))
            pos = 0
            for p, a, g in zip(params, p0, g0):
                expect = a + flat_step[pos:pos + g.size].reshape(g.shape)
                pos += g.size
                assert op_cases.rel_err(p.values, expect) <= 1e-5
    finally:
        for r in [layer for layer in mlp.layers if isinstance(layer, R.RefReLU)]:
            r.keep_override = None


def test_cross_entropy_at_config_size():
    """losses.py:24-32 on the wide MLP's full logits (8192 x 4096, float32 one-hot labels): loss
    within 1e-5 and dL/dz within rel 1e-5 of the oracle's 11-node graph"""
    from core.losses import SoftmaxCrossEntropyLoss
    from core.tensor import Tensor
    rng = np.random.RandomState(5)
    Bf, C = 8192, 4096
    z = (rng.standard_normal((Bf, C)) * 2.0).astype(np.float32)
    lab = rng.randint(0, C, Bf)
    y = np.zeros((Bf, C), np.float32)
    y[np.arange(Bf), lab] = 1.0
    zt = Tensor(z, requires_grad=True)
    loss = SoftmaxCrossEntropyLoss().loss(zt, Tensor(y))
    loss.backward()
    rz = R.RefTensor(z.astype(np.float64), True)
    rloss = R.softmax_cross_entropy(rz, y)
    rloss.backward()
    assert abs(float(loss.values) - float(rloss.values)) <= 1e-5
    assert op_cases.rel_err(zt.grad, rz.grad) <= 1e-5
    # closed form of the same thing (SURVEY 8a/a30): dz = p - y/m
    e = np.exp(z.astype(np.float64) - z.max())
    assert op_cases.rel_err(zt.grad, e / e.sum() - y / Bf) <= 1e-5


def _componentwise_err(c, a64, b64):
    """max |C - A@B| / (|A| @ |B|): the error measure that is meaningful under cancellation and
    wide dynamic range (float32 sgemm itself only promises K*2^-24 in this measure)"""
    exact = a64 @ b64
    scale = np.abs(a64) @ np.abs(b64)
    return float(np.max(np.abs(c.astype(np.float64) - exact) / np.maximum(scale, 1e-300)))


@pytest.mark.parametrize("split", ["f16", "mix", "tf32x3"])
@pytest.mark.parametrize("case", ["wide_exponents", "cancellation", "tiny_and_huge_rows", "bf16_unfriendly"])
def test_operand_split_on_adversarial_data(split, case):
    """The default operand split (TF32 main term + two BF16 cross terms) on data chosen to hurt it:
    exponents spread over 2^-30..2^30 inside every row, products that cancel to 1e-6 of their
    magnitude, rows scaled by 1e-30 / 1e+25, and mantissas whose low 13 bits are all ones (the
    worst case for the bf16 rounding of the residual).  Measure: error per entry over (|A|@|B|)
    of that entry, the componentwise bound under which cancellation and dynamic range do not hide
    anything (float32 accumulation of a K=1024 dot product alone is allowed 6e-5 in it).  Bound:
    5e-6 for the mixed split, 2e-6 for 3xTF32, both inside north_star's 1e-5.  Measured (r02):
    mixed 3.6e-6 on wide_exponents -- single products dominate an entry there, so the two bf16
    cross terms' 2^-20 relative error shows unaveraged -- and <= 1e-6 elsewhere."""
    import core._backend as be
    rng = np.random.RandomState(11)
    M, N, K = 512, 384, 1024
    if case == "wide_exponents":
        a = rng.standard_normal((M, K)) * np.exp2(rng.randint(-30, 31, (M, K)))
        b = rng.standard_normal((K, N)) * np.exp2(rng.randint(-30, 31, (K, N)))
    elif case == "cancellation":
        half = rng.standard_normal((M, K // 2))
        a = np.concatenate([half, -half * (1 + 1e-6 * rng.standard_normal((M, K // 2)))], axis=1)
        col = rng.standard_normal((K // 2, N))
        b = np.concatenate([col, col], axis=0)
    elif case == "tiny_and_huge_rows":
        a = rng.standard_normal((M, K)) * np.where(np.arange(M) % 2 == 0, 1e-30, 1e25)[:, None]
        b = rng.standard_normal((K, N)) * np.where(np.arange(N) % 2 == 0, 1e-7, 1e7)[None, :]
    else:
        def ones_tail(shape):
            v = rng.standard_normal(shape).astype(np.float32)
            return (v.view(np.uint32) | np.uint32(0x1FFF)).view(np.float32)
        a, b = ones_tail((M, K)), ones_tail((K, N))
    a, b = a.astype(np.float32), b.astype(np.float32)
    assert np.all(np.isfinite(a)) and np.all(np.isfinite(b))
    with gemm_route(TC_MIN_MNK=0, TC_SPLIT=split):
        assert be.use_tensor_cores(M, N, K, be.F32)
        c = be.matmul(be.from_numpy(a), be.from_numpy(b)).numpy()
    assert np.all(np.isfinite(c))
    err = _componentwise_err(c, a.astype(np.float64), b.astype(np.float64))
    # ("f16", the default: wide_exponents and tiny_and_huge_rows are outside its guard and are done
    # by the on-device fallback to the mixed split; the other two run on the fp16 planes)
    assert err <= (2e-6 if split == "tf32x3" else 5e-6), (case, split, err)
