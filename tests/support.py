"""Helpers the test modules share: free ports and GPU counts for the two-rank tests, the launchers of
the torchrun workers and of the gloo harnesses, parameter snapshots and the GEMM route settings."""
import contextlib
import ctypes
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# the library's GEMM knobs have no getter: gemm_route restores these defaults
_KNOB_DEFAULTS = {"cta_group": 0, "ksplit": 0, "f16_cluster": 2}


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def gpu_count():
    import core._backend as be
    n = ctypes.c_int(0)
    if be.load_library().tnn_device_count(ctypes.byref(n)):
        return 0
    return n.value


def params(net):
    """host copies of the parameters, layer by layer"""
    return [p.values.copy() for layer in net.get_parameters() for p in layer.values()]


def run_two_ranks(worker_file, timeout):
    """runs tests/<worker_file> on two ranks through torch.distributed.run; returns its stdout"""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(free_port()),
           os.path.join(ROOT, "tests", worker_file)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


def _gloo_rank(target, rank, world, port, queue):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    for p in (ROOT, os.path.join(ROOT, "oracle")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as td
    td.init_process_group("gloo", init_method="env://")
    try:
        queue.put((rank, target(rank, world)))
    finally:
        td.destroy_process_group()


def spawn_gloo(target, world=2):
    """runs target(rank, world) in `world` spawned processes joined in a gloo process group; returns
    what each rank returned, in rank order"""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=_gloo_rank, args=(target, r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return [got[r] for r in range(world)]


@contextlib.contextmanager
def gemm_route(**settings):
    """routes the products of the with-block: keys starting with TC_ set those globals of
    core._backend, the others (cta_group, ksplit, f16_cluster) call be.set_gemm_<key>.  On exit the
    globals get back their values from entry and the knobs their defaults."""
    import core._backend as be
    knobs = {k: _KNOB_DEFAULTS[k] for k in settings if not k.startswith("TC_")}
    saved = {k: getattr(be, k) for k in settings if k.startswith("TC_")}
    try:
        for k, v in settings.items():
            if k in saved:
                setattr(be, k, v)
            else:
                getattr(be, "set_gemm_" + k)(v)
        yield
    finally:
        for k, v in saved.items():
            setattr(be, k, v)
        for k, v in knobs.items():
            getattr(be, "set_gemm_" + k)(v)
