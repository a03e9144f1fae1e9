"""Conv2D / MaxPool2D measurements on one GPU, one JSON line per measurement.

    python scripts/conv_bench.py > profiles/<run>_conv_bench.jsonl

1. kernel bandwidth of the four passes of csrc/conv.cu on a 256 x 32 x 32 x 64 float32 input (3 x 3
   SAME im2col / col2im: a 604 MB col buffer; 2 x 2 / s2 pooling), timed with bench_common.timed_rotating
   (rotating buffer sets that together exceed twice the L2, recorded into one graph).  Algorithmic
   bytes: every input read once, every output written once.  The copy bandwidth they are compared
   with is a device-to-device copy of the col buffer measured the same way in the same run.
2. one 3 x 3 x 64 x 128 SAME conv layer, forward + backward (dx, dW, db) on that batch: the three
   products take the tcgen05 route.  Reports ms, algorithmic TFLOP/s (3 products of 2*M*N*K) and the
   share of the time spent outside the GEMM kernels (per-family event brackets, in a separate pass).
3. the small MNIST CNN of tests/test_gpu_conv.py at batch 128: Model.train_step (recorded, replayed)
   against the five eager lines, ms per step and samples/s.
The card's name and power limit are read in the same run (first line)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import core._backend as be  # noqa: E402
from bench_common import alternate, card, emit, timed_rotating  # noqa: E402
from core.layers import window_geometry  # noqa: E402


def kernel_bandwidth(l2):
    N, H, W, C = 256, 32, 32, 64
    (OH, OW), (PH0, PW0) = window_geometry((H, W), (3, 3), (1, 1), "SAME")
    conv_geom = (3, 3, 1, 1, PH0, PW0, OH, OW)
    (PO, QO), (pp, qp) = window_geometry((H, W), (2, 2), (2, 2), "VALID")
    pool_geom = (2, 2, 2, 2, pp, qp, PO, QO)
    x_bytes = N * H * W * C * 4
    col_bytes = N * OH * OW * 9 * C * 4
    y_bytes = N * PO * QO * C * 4
    rng = np.random.RandomState(0)
    x_host = rng.standard_normal((N, H, W, C)).astype(np.float32)

    def n_sets(set_bytes):
        return int(max(2, -(-2 * l2 // set_bytes)))

    results = {}
    k_conv = n_sets(x_bytes + col_bytes)
    sets = [dict(x=be.from_numpy(x_host), col=be.empty((N * OH * OW, 9 * C), be.F32)) for _ in range(k_conv)]
    for s in sets:
        s["dx"] = be.empty((N, H, W, C), be.F32)
        s["cp"] = be.empty((N * OH * OW, 9 * C), be.F32)

    def im2col(k):
        s = sets[k]
        if be._lib.tnn_im2col(0, s["col"].ptr, s["x"].ptr, N, H, W, C, *conv_geom):
            be._raise("tnn_im2col")

    def col2im(k):
        s = sets[k]
        if be._lib.tnn_col2im(0, s["dx"].ptr, s["col"].ptr, N, H, W, C, *conv_geom):
            be._raise("tnn_col2im")

    results["copy"] = (timed_rotating(lambda k: be.copy_into(sets[k]["cp"], sets[k]["col"]), k_conv),
                       2 * col_bytes, k_conv)
    results["im2col"] = (timed_rotating(im2col, k_conv), x_bytes + col_bytes, k_conv)
    results["col2im"] = (timed_rotating(col2im, k_conv), col_bytes + x_bytes, k_conv)
    del sets
    k_pool = n_sets(2 * x_bytes + 2 * y_bytes)
    psets = [dict(x=be.from_numpy(x_host), y=be.empty((N, PO, QO, C), be.F32),
                  arg=be.empty((N, PO, QO, C), np.int32), dx=be.empty((N, H, W, C), be.F32))
             for _ in range(k_pool)]

    def pool_fwd(k):
        s = psets[k]
        if be._lib.tnn_maxpool_fwd(0, s["y"].ptr, s["arg"].ptr, s["x"].ptr, N, H, W, C, *pool_geom):
            be._raise("tnn_maxpool_fwd")

    def pool_bwd(k):
        s = psets[k]
        if be._lib.tnn_maxpool_bwd(0, s["dx"].ptr, s["y"].ptr, s["arg"].ptr, N, H, W, C, *pool_geom):
            be._raise("tnn_maxpool_bwd")

    results["maxpool_fwd"] = (timed_rotating(pool_fwd, k_pool), x_bytes + 2 * y_bytes, k_pool)
    results["maxpool_bwd"] = (timed_rotating(pool_bwd, k_pool), 2 * y_bytes + x_bytes, k_pool)
    del psets
    copy_gbs = results["copy"][1] / (results["copy"][0] * 1e-3) / 1e9
    for name, (ms, nbytes, k) in results.items():
        gbs = nbytes / (ms * 1e-3) / 1e9
        emit(section="kernel_bandwidth", op=name, shape="256x32x32x64 f32", ms=ms, algorithmic_bytes=nbytes,
             gbs=gbs, share_of_measured_copy=gbs / copy_gbs, rotating_sets=k)


def conv_layer(iters=20):
    from core.layers import Conv2D
    from core.tensor import Tensor
    N, H, W, C, O = 256, 32, 32, 64, 128
    rng = np.random.RandomState(1)
    np.random.seed(1)
    layer = Conv2D((3, 3, C, O))
    x = Tensor(rng.standard_normal((N, H, W, C)).astype(np.float32), requires_grad=True)
    g = be.from_numpy(rng.standard_normal((N, H, W, O)).astype(np.float32))
    M, K = N * H * W, 9 * C
    assert all(be.use_tensor_cores(m, n, k, be.F32) for m, n, k in ((M, O, K), (K, O, M), (M, K, O)))

    def one():
        be.new_split_epoch()
        for t in (x, layer.params["w"], layer.params["b"]):
            t.zero_grad()
        layer.forward(x).backward(g)

    for _ in range(3):
        one()
    be.sync()
    e0, e1 = be.Event(), be.Event()
    e0.record()
    for _ in range(iters):
        one()
    e1.record()
    ms = e1.elapsed_ms_since(e0) / iters
    fams = {}
    for fam, name in ((1, "tcgen05_gemm_ms"), (3, "operand_split_ms")):
        be.prof_enable(fam)
        for _ in range(iters):
            one()
        fams[name] = be.prof_collect()[0] / iters
        be.prof_enable(0)
    flops = 3 * 2.0 * M * O * K
    emit(section="conv_layer", layer="3x3x64x128 SAME, batch 256x32x32x64 f32, fwd+bwd (dx, dW, db)", ms=ms,
         algorithmic_tflops=flops / (ms * 1e-3) / 1e12, share_outside_gemm=1.0 - fams["tcgen05_gemm_ms"] / ms,
         col_bytes=M * K * 4, **fams)


def mnist_cnn(steps=200):
    from core.layers import Conv2D, Dense, Flatten, MaxPool2D, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    from core.tensor import Tensor
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_fp32
    B = 128
    x, _, onehot = ref_fp32.learnable_mnist(B, seed=0)
    xb, yb = Tensor(x.reshape(B, 28, 28, 1)), Tensor(onehot)

    def eager(model):
        model.zero_grad()
        loss = model.loss.loss(model.forward(xb), yb)
        loss.backward()
        model.step()

    def build(step):
        np.random.seed(0)
        net = Net([Conv2D((5, 5, 1, 8), stride=2), ReLU(), MaxPool2D(), Conv2D((3, 3, 8, 16)), ReLU(), Flatten(),
                   Dense(10, num_in=784)])
        model = Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))
        model.defer_loop = False
        for _ in range(10):
            step(model)
        return lambda: step(model)

    runs = {"train_step": build(lambda m: m.train_step(xb, yb)), "eager": build(eager)}
    out = {}
    for mode, ms in alternate(runs, steps, 1, lambda run: run()):
        out[mode] = ms
        emit(section="mnist_cnn", mode=mode, batch=B, ms_per_step=ms, samples_per_s=B / (ms * 1e-3),
             steps=steps)
    emit(section="mnist_cnn", speedup_train_step_over_eager=out["eager"] / out["train_step"])


def main():
    be.init()
    info = be.device_info()
    emit(section="device", l2_bytes=info["l2_bytes"], sm_count=info["sm_count"], **card())
    kernel_bandwidth(info["l2_bytes"])
    conv_layer()
    mnist_cnn()


if __name__ == "__main__":
    main()
