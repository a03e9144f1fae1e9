"""Pointwise-loss measurements on one GPU, one JSON line per measurement, each carrying the card's name
and power limit (read in the same run).

    python scripts/loss_bench.py > profiles/loss_bench_b200.jsonl

1. the fused pass of csrc/loss.cu -- the loss and the seeded dL/dp in one launch, float32 -- for each
   loss on 2^24 and 2^26 elements, timed with sweep_ops.timed_rotating (rotating buffer sets that
   together exceed twice the L2, recorded into one graph and replayed).  Algorithmic bytes: p and t
   read once, dp written once (12 bytes an element).  The yardstick is a device-to-device copy of p
   (8 bytes an element) measured the same way in the same run.
2. a regression MLP step through Model.train_step (recorded, replayed) with the fused MSELoss beside
   the same loss composed from ops (sub_, mul_, sum_, / m), alternating the two models twice: ms per
   step, and the kernels one eager step launches."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import core._backend as be  # noqa: E402
from sweep_ops import timed_rotating  # noqa: E402

CARD = {}
KINDS = (("mse", be.LOSS_MSE), ("mae", be.LOSS_MAE), ("huber", be.LOSS_HUBER), ("sigmoid_ce", be.LOSS_SIGMOID_CE))


def emit(**row):
    row.update(CARD)
    print(json.dumps(row), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def kernel_bandwidth(l2, log2n):
    n = 1 << log2n
    k = int(max(2, -(-2 * l2 // (12 * n))))
    rng = np.random.RandomState(0)
    t_host = rng.standard_normal(n).astype(np.float32)
    p_host = (t_host + rng.standard_normal(n)).astype(np.float32)
    sets = [dict(p=be.from_numpy(p_host), t=be.from_numpy(t_host), dp=be.empty((n,), be.F32),
                 loss=be.empty((), be.F32), c=be.empty((n,), be.F32)) for _ in range(k)]

    def fused(code):
        def launch(i):
            s = sets[i]
            if be._lib.tnn_pointwise_loss(0, code, s["p"].ptr, s["t"].ptr, n, float(n >> 6), 1.0, s["loss"].ptr,
                                          s["dp"].ptr):
                be._raise("tnn_pointwise_loss")
        return launch

    copy_ms = timed_rotating(lambda i: be.copy_into(sets[i]["c"], sets[i]["p"]), k)
    copy_gbs = 8 * n / (copy_ms * 1e-3) / 1e9
    emit(section="kernel_bandwidth", op="copy", elements=n, ms=copy_ms, algorithmic_bytes=8 * n, gbs=copy_gbs,
         rotating_sets=k)
    for name, code in KINDS:
        ms = timed_rotating(fused(code), k)
        gbs = 12 * n / (ms * 1e-3) / 1e9
        emit(section="kernel_bandwidth", op="fused_loss_dp", loss=name, dtype="float32", elements=n, ms=ms,
             algorithmic_bytes=12 * n, gbs=gbs, share_of_measured_copy=gbs / copy_gbs, rotating_sets=k)


class ComposedMSE(object):
    """the same quantity as MSELoss assembled from the primitive differentiable ops"""

    def loss(self, predicted, actual):
        import core.ops as ops
        from core.tensor import as_tensor
        d = ops.sub_(predicted, as_tensor(actual))
        return ops.sum_(ops.mul_(d, d), axis=None) / predicted.shape[0]


def regression_mlp(steps=200, rounds=2):
    from core.layers import Dense, ReLU
    from core.losses import MSELoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    from core.tensor import Tensor
    B, dims = 1024, (64, 256, 256, 8)
    rng = np.random.RandomState(0)
    xb = Tensor(rng.standard_normal((B, dims[0])).astype(np.float32))
    yb = Tensor(rng.standard_normal((B, dims[-1])).astype(np.float32))

    def build(loss):
        np.random.seed(0)
        layers = []
        for i in range(len(dims) - 1):
            layers += [Dense(dims[i + 1], num_in=dims[i])] + ([ReLU()] if i < len(dims) - 2 else [])
        model = Model(net=Net(layers), loss=loss, optimizer=Adam(lr=1e-3))
        model.defer_loop = False
        # launches of one eager step (what the recording replays)
        model._eager_step(xb, yb)
        be.sync()
        n0 = be.launch_count()
        model._eager_step(xb, yb)
        launches = be.launch_count() - n0
        for _ in range(10):
            model.train_step(xb, yb)
        return model, launches

    models = {"fused_mse": build(MSELoss()), "composed_mse": build(ComposedMSE())}
    out = {k: [] for k in models}
    for _ in range(rounds):
        for name, (model, launches) in models.items():
            be.sync()
            t0 = time.perf_counter()
            for _ in range(steps):
                model.train_step(xb, yb)
            be.sync()
            ms = (time.perf_counter() - t0) * 1e3 / steps
            out[name].append(ms)
            emit(section="regression_mlp", loss=name, mode="train_step", batch=B, dims=list(dims), ms_per_step=ms,
                 launches_per_eager_step=launches, steps=steps)
    emit(section="regression_mlp", ms_fused=min(out["fused_mse"]), ms_composed=min(out["composed_mse"]),
         launches_fused=models["fused_mse"][1], launches_composed=models["composed_mse"][1])


def main():
    be.init()
    CARD.update(card())
    info = be.device_info()
    emit(section="device", l2_bytes=info["l2_bytes"], sm_count=info["sm_count"])
    for log2n in (24, 26):
        kernel_bandwidth(info["l2_bytes"], log2n)
    regression_mlp()


if __name__ == "__main__":
    main()
