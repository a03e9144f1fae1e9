"""Worker for tests/test_gpu_dist.py (launched by torch.distributed.run, one rank per GPU):
trains a small MLP data-parallel through the public API and checks, on rank 0, that losses and
parameters equal the single-process oracle on the FULL batch (SURVEY 8e)."""
import numpy as np

from dist_common import assert_replay_matches, eager_steps, same_on_every_rank, state  # sets sys.path
import core._dist as dist
import ref_numpy as R
from core.layers import Dense, ReLU
from core.losses import SoftmaxCrossEntropyLoss
from core.model import Model
from core.nn import Net
from core.optimizer import SGD
from core.tensor import Tensor


def main():
    dist.init_process_group()
    rank, world = dist.rank(), dist.world_size()
    rng = np.random.RandomState(0)
    B, D, C = 96, 40, 12
    x = rng.rand(B, D).astype(np.float32)
    labels = np.eye(C, dtype=np.float32)[rng.randint(0, C, B)]
    lo, hi = dist.shard_bounds(B, rank, world)

    np.random.seed(0)
    net = Net([Dense(24), ReLU(), Dense(C)])
    model = Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=SGD(lr=0.5))
    xs, ys = Tensor(x[lo:hi]), Tensor(labels[lo:hi])
    losses = eager_steps(model, xs, ys, 4)
    params = state(net)
    # every rank must hold bit-identical parameters after the all-reduced update
    assert same_on_every_rank(params, world), "replicas diverged"

    if rank == 0:
        np.random.seed(0)
        ref = R.RefMLP([24, C], R.RefSGD(lr=0.5))
        rlosses = [float(ref.train_step(x, labels)) for _ in range(4)]
        assert np.max(np.abs(np.array(losses) - np.array(rlosses))) <= 1e-5, (losses, rlosses)
        for p, rp in zip(params, ref.params()):
            err = np.max(np.abs(p - rp.values)) / max(np.max(np.abs(rp.values)), 1e-30)
            assert err <= 1e-5, err
        print("DIST_OK world=%d losses=%s" % (world, losses))
    # the captured step (CUDA graph holding the NCCL all-gather / all-reduces) must reproduce the
    # eager data-parallel loop bit for bit
    def fresh():
        np.random.seed(1)
        n = Net([Dense(24, num_in=D), ReLU(), Dense(C, num_in=24)])
        return n, Model(net=n, loss=SoftmaxCrossEntropyLoss(), optimizer=SGD(lr=0.5))

    net_e, model_e = fresh()
    eager = eager_steps(model_e, xs, ys, 6)
    assert_replay_matches(fresh, xs, ys, eager, state(net_e))
    if rank == 0:
        print("GRAPH_DIST_OK world=%d" % world)

    # chunked all-reduce pipelined with the optimiser kernel (what the wide MLP uses): force it on
    # this small model; with two ranks a SUM is order-independent, so it must match bit for bit
    from core.optimizer import Adam
    results = []
    for min_elems, n_chunks in ((1 << 20, 1), (64, 4)):
        dist.MIN_CHUNK_ELEMS, dist.ALLREDUCE_CHUNKS = min_elems, n_chunks
        np.random.seed(2)
        n = Net([Dense(24, num_in=D), ReLU(), Dense(C, num_in=24)])
        m = Model(net=n, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-2))
        results.append((eager_steps(m, xs, ys, 5), state(n)))
    dist.MIN_CHUNK_ELEMS, dist.ALLREDUCE_CHUNKS = 1 << 20, 1
    assert results[0][0] == results[1][0], (results[0][0], results[1][0])
    for a, b in zip(results[0][1], results[1][1]):
        assert np.array_equal(a, b)
    if rank == 0:
        print("CHUNKED_DIST_OK world=%d" % world)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
