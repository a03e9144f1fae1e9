"""Activation-layer measurements on one GPU, one JSON line per measurement, each carrying the card's name
and power limit (read in the same run).

    python scripts/act_bench.py > profiles/act_bench_b200.jsonl

1. each activation's forward pass (x read, y written: 8 bytes an element) and backward pass (g and x
   read, dx written: 12 bytes an element) on 2^24 and 2^26 float32 elements, timed with
   bench_common.timed_rotating (rotating buffer sets that together exceed twice the L2, recorded into
   one graph and replayed).  The yardstick is a device-to-device copy (8 bytes an element) measured
   the same way in the same run.
2. the 64-256-256-8 regression MLP of loss_bench.py at batch 1024 through Model.train_step (recorded,
   replayed), with SiLU layers beside SiLU composed from ops (x * Sigmoid()(x)), alternating the two
   models twice: ms per step, and the kernels one eager step launches.
3. the flagship 4 x Dense(4096) step at batch 8192 through Model.train_step with ReLU (fused into the
   GEMM epilogue) beside GELU (its own forward and backward passes), alternating: what an activation
   outside the epilogue costs at that size."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import core._backend as be  # noqa: E402
from bench_common import CARD, alternate, card, emit, timed_rotating  # noqa: E402

# (name, forward code, backward code, p0)
ACTS = (("leaky_relu", be.LEAKY_RELU, be.LEAKY_RELU_BWD, 0.01), ("elu", be.ELU, be.ELU_BWD, 1.0),
        ("gelu", be.GELU, be.GELU_BWD, 0.0), ("gelu_tanh", be.GELU_TANH, be.GELU_TANH_BWD, 0.0),
        ("softplus", be.SOFTPLUS, be.SOFTPLUS_BWD, 0.0), ("silu", be.SILU, be.SILU_BWD, 0.0))


def kernel_bandwidth(l2, log2n):
    n = 1 << log2n
    k = int(max(2, -(-2 * l2 // (12 * n))))
    rng = np.random.RandomState(0)
    x_host = (rng.standard_normal(n) * 3.0).astype(np.float32)
    g_host = rng.standard_normal(n).astype(np.float32)
    sets = [dict(x=be.from_numpy(x_host), g=be.from_numpy(g_host), y=be.empty((n,), be.F32)) for _ in range(k)]

    copy_ms = timed_rotating(lambda i: be.copy_into(sets[i]["y"], sets[i]["x"]), k)
    copy_gbs = 8 * n / (copy_ms * 1e-3) / 1e9
    emit(section="kernel_bandwidth", op="copy", elements=n, ms=copy_ms, algorithmic_bytes=8 * n, gbs=copy_gbs,
         rotating_sets=k)
    for name, fwd, bwd, p0 in ACTS:
        for direction, nbytes, launch in (
                ("forward", 8 * n, lambda i: be.ew(fwd, sets[i]["x"], p0=p0, out=sets[i]["y"])),
                ("backward", 12 * n, lambda i: be.ew(bwd, sets[i]["g"], sets[i]["x"], p0=p0, out=sets[i]["y"]))):
            ms = timed_rotating(launch, k)
            gbs = nbytes / (ms * 1e-3) / 1e9
            emit(section="kernel_bandwidth", op=name, direction=direction, dtype="float32", elements=n, ms=ms,
                 algorithmic_bytes=nbytes, gbs=gbs, share_of_measured_copy=gbs / copy_gbs, rotating_sets=k)


def _composed_silu():
    from core.layers import Activation, Sigmoid

    class ComposedSiLU(Activation):
        """x * sigmoid(x) assembled from the primitive differentiable ops"""

        def __init__(self):
            Activation.__init__(self, "ComposedSiLU")
            self.sigmoid = Sigmoid()

        def func(self, x):
            return x * self.sigmoid(x)

    return ComposedSiLU()


def _timed_models(section, builders, xb, yb, steps, rounds, **fields):
    """train_step timings of the named models, alternating; launches of one eager step each"""
    models = {}
    for name, build in builders.items():
        model = build()
        model.defer_loop = False
        model._eager_step(xb, yb)
        be.sync()
        n0 = be.launch_count()
        model._eager_step(xb, yb)
        launches = be.launch_count() - n0
        for _ in range(5):
            model.train_step(xb, yb)
        models[name] = (model, launches)
    out = {k: [] for k in models}
    for name, ms in alternate(models, steps, rounds, lambda m: m[0].train_step(xb, yb)):
        out[name].append(ms)
        emit(section=section, variant=name, mode="train_step", ms_per_step=ms,
             launches_per_eager_step=models[name][1], steps=steps, **fields)
    emit(section=section, **{"ms_" + k: min(v) for k, v in out.items()},
         **{"launches_" + k: models[k][1] for k in models}, **fields)


def regression_mlp(steps=200, rounds=2):
    from core.layers import Dense, SiLU
    from core.losses import MSELoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    from core.tensor import Tensor
    B, dims = 1024, (64, 256, 256, 8)
    rng = np.random.RandomState(0)
    xb = Tensor(rng.standard_normal((B, dims[0])).astype(np.float32))
    yb = Tensor(rng.standard_normal((B, dims[-1])).astype(np.float32))

    def build(act):
        def make():
            np.random.seed(0)
            layers = []
            for i in range(len(dims) - 1):
                layers += [Dense(dims[i + 1], num_in=dims[i])] + ([act()] if i < len(dims) - 2 else [])
            return Model(net=Net(layers), loss=MSELoss(), optimizer=Adam(lr=1e-3))
        return make

    _timed_models("regression_mlp", {"silu_layer": build(SiLU), "silu_composed": build(_composed_silu)},
                  xb, yb, steps, rounds, batch=B, dims=list(dims))


def wide_mlp(steps=20, rounds=2):
    from core.layers import GELU, Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    from core.tensor import Tensor
    B, D, widths = 8192, 4096, (4096, 4096, 4096, 4096)
    rng = np.random.RandomState(1000)
    xb = Tensor(rng.rand(B, D).astype(np.float32))
    yb = Tensor(np.eye(widths[-1], dtype=np.float32)[rng.randint(0, widths[-1], B)])

    def build(act):
        def make():
            np.random.seed(0)
            layers = []
            for i, w in enumerate(widths):
                layers += [Dense(w)] + ([act()] if i + 1 < len(widths) else [])
            return Model(net=Net(layers), loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))
        return make

    _timed_models("wide_mlp", {"relu_fused": build(ReLU), "gelu": build(GELU)}, xb, yb, steps, rounds,
                  batch=B, widths=list(widths))


def main():
    be.init()
    CARD.update(card())
    info = be.device_info()
    emit(section="device", l2_bytes=info["l2_bytes"], sm_count=info["sm_count"])
    for log2n in (24, 26):
        kernel_bandwidth(info["l2_bytes"], log2n)
    regression_mlp()
    wide_mlp()


if __name__ == "__main__":
    main()
