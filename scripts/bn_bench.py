"""BatchNormalization measurements on one GPU, one JSON line per measurement, each carrying the
card's name and power limit (read in the same run).

    python scripts/bn_bench.py > profiles/bn_bench_b200.jsonl

1. kernel bandwidth of the four passes of csrc/batchnorm.cu -- statistics (with the running update),
   apply, backward reduction, dx (TRAIN) -- on a 256 x 32 x 32 x 64 NHWC input (an (262144, 64)
   problem) and on (8192, 4096), float32, timed with bench_common.timed_rotating (rotating buffer sets
   that together exceed twice the L2, recorded into one graph and replayed).  Algorithmic bytes: every
   (M, C) operand read once, every (M, C) output written once (the C-sized vectors are left out).
   The yardstick is a device-to-device copy of one (M, C) buffer measured the same way in the same run.
2. the MNIST-sized CNN of tests/test_gpu_batchnorm.py at batch 128 through Model.train_step (recorded,
   replayed), ms per step, beside the same CNN without its two BatchNormalization layers, alternating
   the two models twice."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import core._backend as be  # noqa: E402
from bench_common import CARD, alternate, card, emit, timed_rotating  # noqa: E402


def kernel_bandwidth(l2, M, C, label):
    nbytes = M * C * 4
    k = int(max(2, -(-2 * l2 // (4 * nbytes))))
    rng = np.random.RandomState(0)
    x_host = rng.standard_normal((M, C)).astype(np.float32)
    g_host = rng.standard_normal((M, C)).astype(np.float32)
    gamma, beta = be.from_numpy(rng.standard_normal((1, C)).astype(np.float32)), be.zeros((1, C), be.F32)
    rm, rv = be.zeros((1, C), be.F32), be.full((1, C), 1.0, be.F32)
    dgamma, dbeta = be.empty((1, C), be.F32), be.empty((1, C), be.F32)
    sets = [dict(x=be.from_numpy(x_host), g=be.from_numpy(g_host), y=be.empty((M, C), be.F32),
                 dx=be.empty((M, C), be.F32), mr=be.empty((2 * C + 1,), be.F64), sums=be.empty((2 * C,), be.F64))
            for _ in range(k)]
    for s in sets:
        s["mr"] = be.bn_stats(s["x"], 0.1, 1e-5, rm, rv)

    def stats(i):
        s = sets[i]
        if be._lib.tnn_bn_stats(0, s["x"].ptr, M, C, 0.1, 1e-5, rm.ptr, rv.ptr, s["mr"].ptr, None):
            be._raise("tnn_bn_stats")

    def apply(i):
        s = sets[i]
        if be._lib.tnn_bn_apply(0, s["y"].ptr, s["x"].ptr, M, C, gamma.ptr, beta.ptr, s["mr"].ptr, None, None, 0.0):
            be._raise("tnn_bn_apply")

    def bwd_reduce(i):
        s = sets[i]
        if be._lib.tnn_bn_bwd_reduce(0, s["g"].ptr, s["x"].ptr, M, C, s["mr"].ptr, s["sums"].ptr, dgamma.ptr, 0,
                                     dbeta.ptr, 0):
            be._raise("tnn_bn_bwd_reduce")

    def dx(i):
        s = sets[i]
        if be._lib.tnn_bn_dx(0, s["dx"].ptr, s["g"].ptr, s["x"].ptr, M, C, s["mr"].ptr, gamma.ptr, s["sums"].ptr):
            be._raise("tnn_bn_dx")

    results = [("copy", timed_rotating(lambda i: be.copy_into(sets[i]["y"], sets[i]["x"]), k), 2 * nbytes)]
    for name, fn, reads_writes in (("stats", stats, 1), ("apply", apply, 2), ("bwd_reduce", bwd_reduce, 2),
                                   ("dx", dx, 3)):
        results.append((name, timed_rotating(fn, k), reads_writes * nbytes))
    copy_gbs = results[0][2] / (results[0][1] * 1e-3) / 1e9
    for name, ms, nb in results:
        gbs = nb / (ms * 1e-3) / 1e9
        emit(section="kernel_bandwidth", op=name, shape=label, ms=ms, algorithmic_bytes=nb, gbs=gbs,
             share_of_measured_copy=gbs / copy_gbs, rotating_sets=k)


def mnist_cnn(steps=200, rounds=2):
    from core.layers import BatchNormalization, Conv2D, Dense, Flatten, MaxPool2D, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    from core.tensor import Tensor
    import ref_fp32
    B = 128
    x, _, onehot = ref_fp32.learnable_mnist(B, seed=0)
    xb, yb = Tensor(x.reshape(B, 28, 28, 1)), Tensor(onehot)

    def build(with_bn):
        np.random.seed(0)
        bn = (lambda c: [BatchNormalization(c)]) if with_bn else (lambda c: [])
        layers = ([Conv2D((5, 5, 1, 8), stride=2)] + bn(8) + [ReLU(), MaxPool2D(), Conv2D((3, 3, 8, 16))] + bn(16)
                  + [ReLU(), Flatten(), Dense(10, num_in=784)])
        model = Model(net=Net(layers), loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))
        for _ in range(10):
            model.train_step(xb, yb)
        return model

    models = {"with_batchnorm": build(True), "without_batchnorm": build(False)}
    out = {k: [] for k in models}
    for name, ms in alternate(models, steps, rounds, lambda m: m.train_step(xb, yb)):
        out[name].append(ms)
        emit(section="mnist_cnn", model=name, mode="train_step", batch=B, ms_per_step=ms, steps=steps)
    emit(section="mnist_cnn", ms_with_batchnorm=min(out["with_batchnorm"]),
         ms_without_batchnorm=min(out["without_batchnorm"]),
         added_ms=min(out["with_batchnorm"]) - min(out["without_batchnorm"]))


def main():
    be.init()
    CARD.update(card())
    info = be.device_info()
    emit(section="device", l2_bytes=info["l2_bytes"], sm_count=info["sm_count"])
    kernel_bandwidth(info["l2_bytes"], 256 * 32 * 32, 64, "256x32x32x64 f32")
    kernel_bandwidth(info["l2_bytes"], 8192, 4096, "8192x4096 f32")
    mnist_cnn()


if __name__ == "__main__":
    main()
