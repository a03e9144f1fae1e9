"""Worker for tests/test_gpu_optimizers.py (launched by torch.distributed.run, one rank per GPU): a small
MLP trained data-parallel with RAdam under a cosine schedule, the gradient all-reduce cut into chunks
that are pipelined with the optimiser kernel (core/_dist.reduce_and_apply).  Replicas must hold
bit-identical parameters, and losses and parameters must equal the single-process oracle on the full
batch; the rectified form starts at step 6 of the 8."""
import numpy as np

from dist_common import eager_steps, same_on_every_rank, state  # sets sys.path
import core._dist as dist
import ref_numpy as R
import ref_optim as RO
from core.layers import Dense, ReLU
from core.losses import SoftmaxCrossEntropyLoss
from core.lr_scheduler import CosineAnnealingLR
from core.model import Model
from core.nn import Net
from core.optimizer import RAdam
from core.tensor import Tensor

STEPS = 8


def main():
    dist.init_process_group()
    rank, world = dist.rank(), dist.world_size()
    rng = np.random.RandomState(0)
    B, D, C = 96, 40, 12
    x = rng.rand(B, D).astype(np.float32)
    labels = np.eye(C, dtype=np.float32)[rng.randint(0, C, B)]
    lo, hi = dist.shard_bounds(B, rank, world)
    xs, ys = Tensor(x[lo:hi]), Tensor(labels[lo:hi])

    dist.MIN_CHUNK_ELEMS, dist.ALLREDUCE_CHUNKS = 64, 4
    np.random.seed(0)
    net = Net([Dense(24), ReLU(), Dense(C)])
    model = Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=RAdam(lr=3e-3))
    sched = CosineAnnealingLR(model.optimizer, 5, eta_min=1e-4)
    losses = []
    for _ in range(STEPS):
        losses += eager_steps(model, xs, ys, 1)
        sched.step()
    dist.MIN_CHUNK_ELEMS, dist.ALLREDUCE_CHUNKS = 1 << 20, 1
    final = state(net)
    n_param = sum(p.size for p in final)
    assert n_param >= 4 * 64, "the arena is cut into several chunks"
    assert same_on_every_rank(final, world), "replicas diverged"

    np.random.seed(0)
    ref = R.RefMLP([24, C], RO.RefRAdam(lr=3e-3))
    rsched = CosineAnnealingLR(ref.optimizer, 5, eta_min=1e-4)   # a scheduler writes only `.lr`
    rlosses = []
    for _ in range(STEPS):
        rlosses.append(float(ref.train_step(x, labels)))
        rsched.step()
    assert np.max(np.abs(np.array(losses) - np.array(rlosses))) <= 1e-5, (losses, rlosses)
    for p, rp in zip(final, ref.params()):
        err = np.max(np.abs(p - rp.values)) / max(np.max(np.abs(rp.values)), 1e-30)
        assert err <= 1e-5, err
    if rank == 0:
        print("OPT_DIST_OK world=%d losses=%s" % (world, losses))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
