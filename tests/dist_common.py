"""Blocks the two-rank workers share (dist_worker.py, bn_dist_worker.py, loss_dist_worker.py).
torch.distributed.run starts a worker with tests/ first on sys.path; importing this module puts the
repository root and oracle/ there too."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import core._backend as be  # noqa: E402
import core._dist as dist  # noqa: E402
from support import params  # noqa: E402


def state(net):
    """host copies of the parameters, then of the buffers (running statistics)"""
    return params(net) + [b.values.copy() for layer in net.layers for b in layer.buffers.values()]


def same_on_every_rank(arrays, world):
    flat = np.concatenate([a.ravel() for a in arrays]).astype(np.float64)
    mine = be.from_numpy(flat)
    dist.allreduce_sum(mine)
    return np.array_equal(mine.numpy(), flat * world)


def eager_steps(model, xs, ys, n):
    """n eager training steps on this rank's shard; the losses"""
    losses = []
    for _ in range(n):
        model.zero_grad()
        loss = model.loss.loss(model.forward(xs), ys)
        loss.backward()
        model.step()
        losses.append(float(loss.values))
    return losses


def assert_replay_matches(make_model, xs, ys, eager, final):
    """the recorded step (collectives inside the graph), replayed from a fresh make_model() as many
    times as the eager loop ran, gives the eager losses and the final state bit for bit"""
    net, model = make_model()
    replayed = [float(model.train_step(xs, ys).values) for _ in range(len(eager))]
    assert any(hasattr(v, "graph") for v in model._captured.values()), "step was not recorded"
    assert replayed == eager, (replayed, eager)
    for a, b in zip(state(net), final):
        assert np.array_equal(a, b)
