"""Optimiser measurements on one GPU, one JSON line per measurement, each carrying the card's name and
power limit (read in the same run).

    python scripts/opt_bench.py > profiles/opt_bench_b200.jsonl

1. each rule's fused arena update (Adam, AdamW, RAdam, Adamax, and SGD as the low-byte reference) on
   2^26 float32 parameters, timed with bench_common.timed_rotating (rotating buffer sets that together
   exceed twice the L2, recorded into one graph and replayed).  Bytes per parameter: 28 for the Adam
   family (g, m, v, p read; m, v, p written), 12 for SGD (g, p read; p written).  The yardstick is a
   device-to-device copy (8 bytes an element) measured the same way in the same run.  The coefficients
   are those of step 10, where RAdam is rectified.
2. the flagship 4 x Dense(4096) step at batch 8192 through Model.train_step with Adam, AdamW and
   RAdam, alternating: what the rule costs in the whole step."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import core._backend as be  # noqa: E402
import core.optimizer as O  # noqa: E402
from bench_common import CARD, alternate, card, emit, timed_rotating  # noqa: E402

RULES = (("sgd", O.SGD, 12), ("adam", O.Adam, 28), ("adamw", O.AdamW, 28), ("radam", O.RAdam, 28),
         ("adamax", O.Adamax, 28))


def kernel_bandwidth(l2, log2n=26):
    n = 1 << log2n
    k = int(max(2, -(-2 * l2 // (16 * n))))
    rng = np.random.RandomState(0)
    g_host = (rng.standard_normal(n) * 1e-2).astype(np.float32)
    p_host = rng.standard_normal(n).astype(np.float32)
    sets = [dict(g=be.from_numpy(g_host), p=be.from_numpy(p_host), m=be.zeros((n,), be.F32),
                 v=be.zeros((n,), be.F32)) for _ in range(k)]
    copy_ms = timed_rotating(lambda i: be.copy_into(sets[i]["p"], sets[i]["g"]), k)
    copy_gbs = 8 * n / (copy_ms * 1e-3) / 1e9
    emit(section="kernel_bandwidth", op="copy", elements=n, ms=copy_ms, algorithmic_bytes=8 * n, gbs=copy_gbs,
         rotating_sets=k)
    for name, cls, nbytes in RULES:
        opt = cls(lr=1e-3)
        for _ in range(10):
            hyper = opt._hyper8()
        s1 = (lambda i: sets[i]["v"]) if opt.n_state == 2 else (lambda i: None)
        s0 = (lambda i: sets[i]["m"]) if opt.n_state >= 1 else (lambda i: None)
        ms = timed_rotating(lambda i: be.opt_step(opt.opt_code, sets[i]["p"], None, sets[i]["g"], s0(i), s1(i), hyper), k)
        gbs = nbytes * n / (ms * 1e-3) / 1e9
        emit(section="kernel_bandwidth", op=name, dtype="float32", elements=n, ms=ms, algorithmic_bytes=nbytes * n,
             gbs=gbs, share_of_measured_copy=gbs / copy_gbs, rotating_sets=k)


def wide_mlp(steps=20, rounds=3):
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.tensor import Tensor
    B, D, widths = 8192, 4096, (4096, 4096, 4096, 4096)
    rng = np.random.RandomState(1000)
    xb = Tensor(rng.rand(B, D).astype(np.float32))
    yb = Tensor(np.eye(widths[-1], dtype=np.float32)[rng.randint(0, widths[-1], B)])
    models = {}
    for name, make in (("adam", O.Adam), ("adamw", O.AdamW), ("radam", O.RAdam)):
        np.random.seed(0)
        layers = []
        for i, w in enumerate(widths):
            layers += [Dense(w)] + ([ReLU()] if i + 1 < len(widths) else [])
        model = Model(net=Net(layers), loss=SoftmaxCrossEntropyLoss(), optimizer=make(lr=1e-3))
        for _ in range(5):
            model.train_step(xb, yb)
        models[name] = model
    out = {k: [] for k in models}
    for name, ms in alternate(models, steps, rounds, lambda m: m.train_step(xb, yb)):
        out[name].append(ms)
        emit(section="wide_mlp", variant=name, mode="train_step", ms_per_step=ms, steps=steps, batch=B,
             widths=list(widths))
    emit(section="wide_mlp", **{"ms_min_" + k: min(v) for k, v in out.items()},
         **{"ms_max_" + k: max(v) for k, v in out.items()}, batch=B, widths=list(widths))


def main():
    be.init()
    CARD.update(card())
    info = be.device_info()
    emit(section="device", l2_bytes=info["l2_bytes"], sm_count=info["sm_count"])
    kernel_bandwidth(info["l2_bytes"])
    wide_mlp()


if __name__ == "__main__":
    main()
