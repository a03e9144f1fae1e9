"""The data-parallel scheme on CPU, world_size 2 over gloo: batch rows are sharded across ranks,
the cross-entropy's (max, sum-exp) pair is exchanged and merged exactly as core/_dist.py and
tnn_ce_merge_stats do, per-rank gradients are SUM-all-reduced -- and the result must equal the
single-process reference maths on the full batch (SURVEY 8e).  The per-rank compute is the numpy
oracle here (no GPU in this container); the N>1 GPU path runs the same host logic over NCCL."""
import numpy as np

import ref_numpy as R
from support import spawn_gloo


def _worker(rank, world):
    import torch
    import torch.distributed as td
    import core._dist as dist
    rng = np.random.RandomState(0)
    B, D, C = 48, 20, 12
    x = rng.rand(B, D)
    labels = np.eye(C)[rng.randint(0, C, B)]
    w = rng.standard_normal((D, C)) * 0.3
    b = rng.standard_normal((1, C)) * 0.1
    lo, hi = dist.shard_bounds(B, rank, world)
    xs, ys = x[lo:hi], labels[lo:hi]
    # local forward up to the logits
    W, Bv = R.RefTensor(w, True), R.RefTensor(b, True)
    z = R.matmul(R.lift(xs), W) + Bv
    # stage 1: local stats, all-gather, merge
    m_r = z.values.max()
    s_r = np.exp(z.values - m_r).sum()
    gathered = [torch.zeros(2, dtype=torch.float64) for _ in range(world)]
    td.all_gather(gathered, torch.tensor([m_r, s_r], dtype=torch.float64))
    M, S = dist.merge_stats_host([g.numpy() for g in gathered])
    # stage 2: local loss share and dz with the GLOBAL normaliser and batch size
    e = np.exp(z.values - M)
    p = e / S
    q = (p * ys).sum(1)
    loss_part = torch.tensor([-(np.log(q)).sum() / B], dtype=torch.float64)
    dz = p - ys * p / (B * q[:, None])
    z.backward(dz)
    flat = torch.from_numpy(np.concatenate([W.grad.ravel(), Bv.grad.ravel()]))
    td.all_reduce(flat)            # SUM, not mean
    td.all_reduce(loss_part)
    return float(loss_part[0]), flat.numpy().copy()


def test_sharded_ce_and_grad_allreduce_equals_full_batch():
    loss_dp, flat_dp = spawn_gloo(_worker)[0]
    # single-process reference maths on the full batch
    rng = np.random.RandomState(0)
    B, D, C = 48, 20, 12
    x = rng.rand(B, D)
    labels = np.eye(C)[rng.randint(0, C, B)]
    W = R.RefTensor(rng.standard_normal((D, C)) * 0.3, True)
    Bv = R.RefTensor(rng.standard_normal((1, C)) * 0.1, True)
    loss = R.softmax_cross_entropy(R.matmul(R.lift(x), W) + Bv, labels)
    loss.backward()
    flat = np.concatenate([W.grad.ravel(), Bv.grad.ravel()])
    assert abs(loss_dp - float(loss.values)) <= 1e-12
    assert np.max(np.abs(flat_dp - flat)) <= 1e-12 * max(1.0, np.max(np.abs(flat)))
