"""Worker for tests/test_gpu_batchnorm.py (launched by torch.distributed.run, one rank per GPU): a
small CNN with BatchNormalization trained data-parallel through the public API.  Checks that the
statistics are those of the GLOBAL batch (losses, parameters and running statistics equal the
single-process oracle on the full batch), that replicas hold bit-identical parameters and running
statistics, and that the recorded step (the all-gather and all-reduces inside the graph) gives the
eager loop's bits."""
import numpy as np

from dist_common import assert_replay_matches, eager_steps, same_on_every_rank, state  # sets sys.path
import core._dist as dist
import ref_bn as RB
import ref_conv as RC
import ref_numpy as R
from core.layers import BatchNormalization, Conv2D, Dense, Flatten, ReLU
from core.losses import SoftmaxCrossEntropyLoss
from core.model import Model
from core.nn import Net
from core.optimizer import SGD
from core.tensor import Tensor

B, H, W, CIN, C, K = 10, 6, 5, 2, 4, 3     # 10 images: shards of 5 per rank


def _model(seed):
    np.random.seed(seed)
    net = Net([Conv2D((3, 3, CIN, C)), BatchNormalization(C, momentum=0.2), ReLU(), Flatten(),
               Dense(K, num_in=H * W * C)])
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=SGD(lr=0.3))


def main():
    dist.init_process_group()
    rank, world = dist.rank(), dist.world_size()
    rng = np.random.RandomState(0)
    x = (rng.standard_normal((B, H, W, CIN)) * 2 + 3).astype(np.float32)
    labels = np.eye(K, dtype=np.float32)[rng.randint(0, K, B)]
    lo, hi = dist.shard_bounds(B, rank, world)
    xs, ys = Tensor(x[lo:hi]), Tensor(labels[lo:hi])

    net, model = _model(0)
    start = state(net)
    eager = eager_steps(model, xs, ys, 4)
    final = state(net)
    assert same_on_every_rank(final, world), "replicas diverged"

    # the single-process oracle on the full batch
    p = [R.RefTensor(v, True) for v in start[:6]]
    st = RB.RefBNState(C, momentum=0.2, running_mean=start[6], running_var=start[7])
    opt = R.RefSGD(lr=0.3)
    rlosses = []
    for _ in range(4):
        for t in p:
            t.zero_grad()
        h = RC.conv2d(R.lift(x), p[0], p[1], (1, 1), "SAME")
        h = R.clip(RB.batchnorm(h, p[2], p[3], st, True), 0.0)
        h = R.reshape(h, (B, -1))
        loss = R.softmax_cross_entropy(R.matmul(h, p[4]) + p[5], labels)
        loss.backward()
        rlosses.append(float(loss.values))
        for t, s in zip(p, opt.compute_steps(p)):
            t.assign(t.values + s)
            t.zero_grad()
    assert np.max(np.abs(np.array(eager) - np.array(rlosses))) <= 1e-5, (eager, rlosses)
    ref = [t.values for t in p] + [st.running_mean[None], st.running_var[None]]
    for a, b in zip(final, ref):
        # (the conv bias before the BatchNormalization stays near 0: its gradient is 0 analytically)
        err = np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-2)
        assert err <= 1e-5, err
    if rank == 0:
        print("BN_DIST_EAGER_OK world=%d losses=%s" % (world, eager))

    # the recorded step, collectives inside the graph, gives the eager bits
    assert_replay_matches(lambda: _model(0), xs, ys, eager, final)
    if rank == 0:
        print("BN_DIST_OK world=%d" % world)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
