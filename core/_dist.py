"""Data-parallel plumbing (new: the reference is single-process, SURVEY 2.1 / 8e).

One process per GPU.  torch.distributed (gloo) is used only as the control plane that hands the
NCCL unique id from rank 0 to the others; every data-path collective is NCCL on this process's
compute stream, driven through libtnn_b200.so:
  * allreduce_sum(flat gradient arena) -- once per step, SUM (the loss already divides by the
    global batch size, so no averaging)
  * merge_ce_stats -- all-gather of the (max, sum-exp) pair so SoftmaxCrossEntropyLoss keeps the
    reference's batch-global normaliser under row sharding.
  * bn_global_stats / an all-reduce of 2C sums -- BatchNormalization's TRAIN statistics and their
    backward sums span the global batch (core/ops.py batchnorm_).
"""
import ctypes
import os

import numpy as np

import core._backend as be

_world = 1
_rank = 0
_nccl_ready = False


def world_size():
    return _world


def rank():
    return _rank


def shard_bounds(n_rows, rank_, world_):
    """rows [start, stop) of a global batch owned by a rank (contiguous, near-equal shards)"""
    base, rem = divmod(n_rows, world_)
    start = rank_ * base + min(rank_, rem)
    return start, start + base + (1 if rank_ < rem else 0)


def merge_stats_host(pairs):
    """[(M_r, S_r)] -> (M, S) with M = max M_r, S = sum S_r * exp(M_r - M) (host mirror of
    tnn_ce_merge_stats, used by the CPU tests of the sharding scheme)"""
    pairs = np.asarray(pairs, dtype=np.float64).reshape(-1, 2)
    m = pairs[:, 0].max()
    return m, float(np.sum(pairs[:, 1] * np.exp(pairs[:, 0] - m)))


def init_process_group(control_backend="gloo"):
    """Read RANK / WORLD_SIZE / LOCAL_RANK / MASTER_ADDR / MASTER_PORT (torchrun's contract), bind
    this process to its GPU and create the NCCL communicator."""
    global _world, _rank, _nccl_ready
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank_ = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", str(rank_)))
    be.init(local)
    if world == 1:
        _world, _rank = 1, 0
        return
    import torch.distributed as td
    if not td.is_initialized():
        td.init_process_group(control_backend, init_method="env://")
    payload = [None]
    if rank_ == 0:
        buf = ctypes.create_string_buffer(128)
        if be._lib.tnn_nccl_unique_id(buf):
            be._raise("tnn_nccl_unique_id")
        payload = [buf.raw]
    td.broadcast_object_list(payload, src=0)
    idbuf = ctypes.create_string_buffer(payload[0], 128)
    if be._lib.tnn_nccl_init(rank_, world, idbuf):
        be._raise("tnn_nccl_init")
    _world, _rank, _nccl_ready = world, rank_, True


def _parse_cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def bind_to_local_numa_node(local_rank=None):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (sysfs `local_cpulist` of
    the GPU's PCI function), so pinned staging buffers are allocated in that node's memory and the
    per-step H2D traffic of 8 ranks does not all come out of one socket.  Returns a short
    description, or None when the topology is not visible (then nothing is changed)."""
    if not hasattr(os, "sched_setaffinity"):
        return None
    if local_rank is None:
        local_rank = int(os.environ.get("LOCAL_RANK", os.environ.get("TNN_DEVICE", "0")))
    try:
        import subprocess
        out = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=20)
        bus = out.stdout.strip().splitlines()[0].strip().lower()
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:     # 00000000:1B:00.0 -> 0000:1b:00.0
            bus = bus[4:]
        base = "/sys/bus/pci/devices/%s/" % bus
        with open(base + "local_cpulist") as f:
            cpus = _parse_cpulist(f.read())
        node = None
        if os.path.exists(base + "numa_node"):
            with open(base + "numa_node") as f:
                node = int(f.read().strip())
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus or cpus == allowed:
            return "numa node %s: affinity unchanged (%d cpus)" % (node, len(allowed))
        os.sched_setaffinity(0, cpus)
        return "numa node %s: bound to %d of %d cpus" % (node, len(cpus), len(allowed))
    except Exception:        # no nvidia-smi / sysfs entry: leave the affinity alone
        return None


def destroy_process_group():
    global _world, _rank, _nccl_ready
    if _nccl_ready:
        be.destroy_all_graphs()   # graphs holding NCCL nodes must not outlive the communicator
        be._lib.tnn_nccl_destroy()
    _world, _rank, _nccl_ready = 1, 0, False


def allreduce_sum(d):
    """in-place SUM all-reduce of a device array on the compute stream"""
    if _world == 1:
        return d
    if be._lib.tnn_allreduce_sum(be._DT_CODE[d.dtype], d.ptr, d.size):
        be._raise("tnn_allreduce_sum")
    return d


# Measured on 2 B200s (wide MLP, 30 steps): 1 chunk 11.83 / 11.91 ms per step, 4 chunks 11.89 / 11.92,
# 8 chunks 11.96 -- the step is power-bound, hiding the optimiser behind the all-reduce buys nothing,
# so the default is one all-reduce on the compute stream and the pipeline stays a knob.
ALLREDUCE_CHUNKS = int(os.environ.get("TNN_ALLREDUCE_CHUNKS", "1"))
MIN_CHUNK_ELEMS = 1 << 20     # pieces below this are not worth a launch of their own


def chunk_bounds(n, chunks, align):
    """[(lo, hi)] covering [0, n) in at most `chunks` pieces whose starts are multiples of `align`"""
    per = -(-n // chunks)
    per = (per + align - 1) // align * align
    return [(lo, min(lo + per, n)) for lo in range(0, n, per)]


def reduce_and_apply(optimizer, param_flat, grad_flat, align=64):
    """SUM all-reduce of the flat gradient arena pipelined with the fused optimiser: the arena is
    cut into ALLREDUCE_CHUNKS pieces, piece i+1 is reduced on the comm stream while the optimiser
    kernel updates piece i on the compute stream.  Every rank cuts identically, so replicas stay
    bit-identical."""
    n = grad_flat.size
    chunks = max(1, min(ALLREDUCE_CHUNKS, n // MIN_CHUNK_ELEMS))
    if chunks == 1:
        allreduce_sum(grad_flat)
        optimizer.apply_fused(param_flat, grad_flat)
        return
    bounds = chunk_bounds(n, chunks, align)
    if be._lib.tnn_comm_wait_compute():
        be._raise("tnn_comm_wait_compute")
    code = be._DT_CODE[grad_flat.dtype]
    isz = grad_flat.dtype.itemsize
    hyper = optimizer.step_hyper()
    for lo, hi in bounds:
        if be._lib.tnn_allreduce_sum_comm(code, grad_flat.ptr + lo * isz, hi - lo):
            be._raise("tnn_allreduce_sum_comm")
        if be._lib.tnn_compute_wait_comm():
            be._raise("tnn_compute_wait_comm")
        optimizer.apply_fused_range(param_flat, grad_flat, lo, hi, hyper)


def merge_ce_stats(stats):
    """local (max, sum-exp) -> global (max, sum-exp); 2 floats per rank over NCCL"""
    if _world == 1:
        return stats
    gathered = be.empty((2 * _world,), stats.dtype)
    if be._lib.tnn_allgather(be._DT_CODE[stats.dtype], gathered.ptr, stats.ptr, 2):
        be._raise("tnn_allgather")
    return be.ce_merge_stats(gathered, _world)


def bn_global_stats(x, momentum, eps, running_mean, running_var):
    """BatchNormalization's TRAIN statistics over the GLOBAL batch: each rank's (count, mean, M2) per
    column, 1 + 2C float64 values, are all-gathered over NCCL and merged in rank order on the device,
    so every rank gets the same mean, r and running statistics"""
    C = x.shape[1]
    part = be.bn_stats(x, momentum, eps, running_mean, running_var, local=True)
    if _world == 1:
        gathered = part
    else:
        gathered = be.empty((_world * (1 + 2 * C),), be.F64)
        if be._lib.tnn_allgather(be._DT_CODE[be.F64], gathered.ptr, part.ptr, 1 + 2 * C):
            be._raise("tnn_allgather")
    return be.bn_merge(gathered, _world, C, momentum, eps, running_mean, running_var)


def merge_bn_stats_host(parts):
    """[(n_r, mean_r[C], M2_r[C])] in rank order -> (n, mean[C], M2[C]) with Chan's pairwise update,
    the order and formulas of tnn_bn_merge (host mirror, used by the CPU tests of the scheme)"""
    n, mean, m2 = 0.0, 0.0, 0.0
    for nb, mb, m2b in parts:
        if nb == 0:
            continue
        tot = n + nb
        delta = np.asarray(mb, np.float64) - mean
        mean = mean + delta * (nb / tot)
        m2 = m2 + np.asarray(m2b, np.float64) + delta * delta * (n * nb / tot)
        n = tot
    return n, mean, m2


def barrier():
    if _world == 1:
        be.sync()
        return
    token = be.zeros((1,), be.F32)
    allreduce_sum(token)
    be.sync()
