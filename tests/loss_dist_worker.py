"""Worker for tests/test_gpu_losses.py (launched by torch.distributed.run, one rank per GPU): a small
regression MLP trained data-parallel through the public API with MSELoss and with
SigmoidCrossEntropyLoss.  Checks that 1/m covers the GLOBAL batch (losses and parameters equal the
single-process oracle on the full batch), that replicas hold bit-identical parameters, and that the
recorded step (the loss all-reduce and the gradient all-reduce inside the graph) gives the eager
loop's bits."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import core._backend as be  # noqa: E402
import core._dist as dist  # noqa: E402
import ref_losses as RL  # noqa: E402
import ref_numpy as R  # noqa: E402
from core.layers import Dense, ReLU  # noqa: E402
from core.losses import MSELoss, SigmoidCrossEntropyLoss  # noqa: E402
from core.model import Model  # noqa: E402
from core.nn import Net  # noqa: E402
from core.optimizer import SGD  # noqa: E402
from core.tensor import Tensor  # noqa: E402

B, DIN, DH, DOUT = 16, 6, 12, 3     # 16 rows: shards of 8 per rank


def _model(seed, loss):
    np.random.seed(seed)
    net = Net([Dense(DH, num_in=DIN), ReLU(), Dense(DOUT, num_in=DH)])
    return net, Model(net=net, loss=loss, optimizer=SGD(lr=0.2))


def _state(net):
    return [p.values.copy() for layer in net.get_parameters() for p in layer.values()]


def _same_on_every_rank(arrays, world):
    flat = np.concatenate([a.ravel() for a in arrays]).astype(np.float64)
    mine = be.from_numpy(flat)
    dist.allreduce_sum(mine)
    return np.array_equal(mine.numpy(), flat * world)


def check(kind, loss_cls, x, y, rank, world):
    lo, hi = dist.shard_bounds(B, rank, world)
    xs, ys = Tensor(x[lo:hi]), Tensor(y[lo:hi])
    net, model = _model(0, loss_cls())
    start = _state(net)
    eager = []
    for _ in range(4):
        model.zero_grad()
        loss = model.loss.loss(model.forward(xs), ys)
        loss.backward()
        model.step()
        eager.append(float(loss.values))
    final = _state(net)
    assert _same_on_every_rank(final, world), "replicas diverged"
    assert _same_on_every_rank([np.array(eager)], world), "ranks report different losses"

    # the single-process oracle on the full batch
    p = [R.RefTensor(v, True) for v in start]
    opt = R.RefSGD(lr=0.2)
    rlosses = []
    for _ in range(4):
        for t in p:
            t.zero_grad()
        h = R.clip(R.matmul(R.lift(x), p[0]) + p[1], 0.0)
        loss = RL.pointwise_loss(R.matmul(h, p[2]) + p[3], y, kind)
        loss.backward()
        rlosses.append(float(loss.values))
        for t, s in zip(p, opt.compute_steps(p)):
            t.assign(t.values + s)
            t.zero_grad()
    assert np.max(np.abs(np.array(eager) - np.array(rlosses))) <= 1e-5 * max(1.0, max(rlosses)), (eager, rlosses)
    for a, b in zip(final, [t.values for t in p]):
        err = np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-2)
        assert err <= 1e-5, err

    # the recorded step, collectives inside the graph, gives the eager bits
    net_g, model_g = _model(0, loss_cls())
    replayed = [float(model_g.train_step(xs, ys).values) for _ in range(4)]
    assert any(hasattr(v, "graph") for v in model_g._captured.values()), "step was not recorded"
    assert replayed == eager, (replayed, eager)
    for a, b in zip(_state(net_g), final):
        assert np.array_equal(a, b)
    if rank == 0:
        print("LOSS_DIST_%s_OK world=%d losses=%s" % (kind.upper(), world, eager))


def main():
    dist.init_process_group()
    rank, world = dist.rank(), dist.world_size()
    rng = np.random.RandomState(0)
    x = rng.standard_normal((B, DIN)).astype(np.float32)
    y_reg = rng.standard_normal((B, DOUT)).astype(np.float32)
    y_multi = rng.rand(B, DOUT).astype(np.float32)
    check("mse", MSELoss, x, y_reg, rank, world)
    check("sigmoid_ce", SigmoidCrossEntropyLoss, x, y_multi, rank, world)
    if rank == 0:
        print("LOSS_DIST_OK world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
