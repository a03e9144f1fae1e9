"""Benchmark of the hot path: MLP train samples/sec (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--workload wide|mnist] [--batch-per-gpu B] [--global-batch G]
                    [--dump-outputs DIR]

Workload at N=1 (default): BASELINE.json configs[3] -- 4 x Dense(4096) with 3 ReLU, D_in = C =
4096, batch 8192, fp32 storage, fp32-accurate split tensor-core GEMMs, fused global-softmax CE,
fused Adam; synthetic data and reference-style Xavier-uniform weights (np.random.seed(0)).
At N>1 (launched with torchrun, one rank per GPU): the same model, batch 8192 PER GPU (weak
scaling; N=8 is configs[4]'s global batch 65536), rows sharded by rank, one NCCL SUM all-reduce
of the flat gradient arena per step plus the 2-float CE-normaliser all-gather.

A "step" = zero_grad + forward + loss + backward + (all-reduce) + optimizer step.
  value : steps timed with CUDA events on the compute stream, inputs resident in HBM
  e2e   : the same step driven from HOST buffers through utils.data_iterator.PrefetchIterator:
          per step the batch (float32 inputs + int32 class labels, one-hot rows built on the
          device) is copied from pinned host memory, and every step's loss is read back to the
          host (one step behind, so the read does not drain the GPU's queue); the K-step region
          is timed twice, the faster run is reported and both are listed (ms_per_step_runs)
  roofline     : the tcgen05 GEMM kernel, per-launch time from CUDA events inside the timed steps
  cpu_baseline : oracle/ref_numpy.py (numpy restatement of the reference) on the host cores, on
                 the bounded sample REF_SAMPLE_BATCH rows per step (rank 0, N=1 only)
Extra objects in the same JSON line (every one measured in this run):
  strong_scaling : BASELINE.json configs[4] -- the same model at a FIXED global batch of 65536
                   (65536/N rows per GPU): ms/step and samples/s; efficiency = T(1) / (N T(N))
  allreduce      : (N>1) the 268.5 MB gradient all-reduce timed alone -> bus bandwidth
  checks         : (N>1) replicas' parameter checksums agree after the timed steps; the step-0
                   loss equals ln(B_global * C) to the tolerance random init allows
  mnist          : (N=1) BASELINE.json configs[0], the examples/mnist MLP at batch 128: the
                   unmodified five-line loop (eager) and Model.train_step (recorded step)

--dump-outputs DIR (B200 arm, rank 0) writes what the last timed step handed its caller as
DIR/<name>.npy (float32, or float64 where the output is float64): `loss`, `prediction` (eager steps
only; a recorded step returns the loss alone) and every parameter after the update as
`layer<i>_<key>`.  An output of more than DUMP_SAMPLE elements is stored as its values at a fixed
seeded sample of DUMP_SAMPLE flat indices (sorted), the same sample on every run; the wide MLP's
dump is about 20 MB.  The inputs and the initial weights are seeded, so two builds run with the
same arguments can be compared output for output.

--impl reference times the CPU implementation alone (all host threads, also under torchrun), on
the same config/metric/unit; each of its steps is a bounded sample of the workload: a train step
on REF_SAMPLE_BATCH = 1024 of the 8192 rows (a full-batch reference step takes ~1 min: float64,
4x re-walked backward).  The sample size is fixed -- it does not depend on --steps -- and is the
same one `cpu_baseline` uses, so there is ONE CPU figure per box.
"""
import os
import sys

if "--impl" in sys.argv and "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.pop(_v, None)

import argparse  # noqa: E402
import gc  # noqa: E402
import json  # noqa: E402
import math  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WIDE = dict(name="wide_mlp_4x4096", widths=[4096, 4096, 4096, 4096], d_in=4096, batch=8192)
MNIST = dict(name="mnist_mlp_784-200-100-70-30-10", widths=[200, 100, 70, 30, 10], d_in=784, batch=128)
REF_SAMPLE_BATCH = 1024     # rows per CPU-reference step on the wide MLP (fixed; see module docstring)
STRONG_GLOBAL_BATCH = 65536  # BASELINE.json configs[4]
DUMP_SAMPLE = 1 << 20        # --dump-outputs: elements kept of a larger output (4 MB in float32)


# ------------------------------------------------------------------------------------------------
def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_burst=p["bf16_tflops"],
                    bf16_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


class ClockSampler(object):
    """SM clock and throttle reasons sampled while the timed region runs: NVML queried from a
    thread of this process every 20 ms (no start-up latency, so even a 0.2 s region at 8 ranks gets
    samples); `nvidia-smi -lms 100` in a subprocess if NVML cannot be opened"""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.nvml = None
        self.lines = []          # nvidia-smi: csv lines; NVML: (sm_mhz, max_mhz, reason bitmask)
        self._stop = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons",
                          getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None))
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM))
                mask = int(reasons(self._handle)) if reasons else 0
                self.lines.append((sm, self._max, mask))
            except Exception:
                pass
            self._stop.wait(0.02)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """index of the next sample: brackets the timed region inside a longer-running sampler"""
        return len(self.lines)

    def stop(self, first=0, last=None):
        if self.nvml is None and self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        sm, mx, reasons = [], [], set()
        if self.nvml is not None:
            nv = self.nvml
            self._stop.set()
            self.thread.join(timeout=2)
            bits = [nv.nvmlClocksThrottleReasonHwSlowdown, nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                    nv.nvmlClocksThrottleReasonSwThermalSlowdown, nv.nvmlClocksThrottleReasonSwPowerCap]
            for s_mhz, m_mhz, mask in (self.lines[first:last] or self.lines[-3:]):
                sm.append(s_mhz)
                mx.append(m_mhz)
                for nm, bit in zip(self.NAMES, bits):
                    if mask & bit:
                        reasons.add(nm)
            source = "nvml, 20 ms period"
        else:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
            for ln in (self.lines[first:last] or self.lines[-3:]):
                parts = [p.strip() for p in ln.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    mx.append(float(parts[2]))
                except ValueError:
                    continue
                for nm, val in zip(self.NAMES, parts[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            source = "nvidia-smi -lms 100"
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        busy = [s for s in sm if s > 0]
        return dict(sm_mhz=float(np.median(busy)), sm_max_mhz=float(max(mx)),
                    reasons=sorted(reasons), samples=len(sm), source=source)


def make_config(cfg, batch_per_gpu, world):
    """the `config` object BOTH arms print, key for key: the workload the metric is quoted on, and
    the bounded sample of it one CPU-reference step runs"""
    return {"workload": cfg["name"], "batch_per_gpu": batch_per_gpu, "global_batch": batch_per_gpu * world,
            "d_in": cfg["d_in"], "widths": cfg["widths"], "optimizer": "Adam(1e-3)",
            "parallelism": "dp%d" % world,
            "cpu_reference_sample": "%d rows per step" % ref_sample_batch(cfg),
            "l2": "per-step working set (parameters, activations, operand planes) far exceeds the "
                  "126 MB L2 for the wide MLP; no flush between steps"}


def gemm_flops_per_step(cfg, batch):
    """2*M*N*K over the forward, dX (all layers but the first) and dW products"""
    dims = [cfg["d_in"]] + cfg["widths"]
    fl = 0
    for i in range(len(cfg["widths"])):
        mnk = batch * dims[i] * dims[i + 1]
        fl += 2 * mnk * (3 if i > 0 else 2)
    return fl


def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the numpy oracle on the host cores
# ------------------------------------------------------------------------------------------------
def ref_sample_batch(cfg):
    return min(cfg["batch"], REF_SAMPLE_BATCH)


def cpu_reference_throughput(cfg, steps, warmup):
    """train steps of the numpy restatement of the reference (oracle/ref_numpy.py: float64
    gradients, per-path backward, flattened Adam) on ref_sample_batch(cfg) rows; returns
    (samples/s, s/step, description).  The first step runs on float32 parameters, later ones on
    float64 (the reference promotes them, model.py:59-61), so warmup >= 1 times the steady state."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_numpy as R
    sample = ref_sample_batch(cfg)
    np.random.seed(0)
    rng = np.random.RandomState(0)
    C = cfg["widths"][-1]
    x = rng.rand(sample, cfg["d_in"]).astype(np.float32)
    labels = np.eye(C, dtype=np.float32)[rng.randint(0, C, sample)]
    mlp = R.RefMLP(cfg["widths"], R.RefAdam(lr=1e-3))
    for _ in range(warmup):
        mlp.train_step(x, labels)
    t0 = time.perf_counter()
    for _ in range(steps):
        mlp.train_step(x, labels)
    dt = (time.perf_counter() - t0) / steps
    desc = ("%d timed train steps (after %d warm-up) of the %s on %d of its %d rows per step, "
            "oracle/ref_numpy.py on %d host threads, %.2f s/step" % (
                steps, warmup, cfg["name"], sample, cfg["batch"], host_cores(), dt))
    return sample / dt, dt, desc


def run_reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps if args.steps_given else 10
    value, s_per_step, desc = cpu_reference_throughput(cfg, steps, args.warmup)
    note = None
    if args.gpus > 1:
        note = ("the reference has no data-parallel mode: this is the single-process CPU figure, "
                "identical in meaning at every N (not a scaling point)")
    line = {
        "impl": "reference", "metric": "MLP train samples/sec", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(cfg, cfg["batch"], args.gpus),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": host_cores(), "kind": "port",
                         "sample": desc},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if note:
        line["note"] = note
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def build_model(cfg):
    from core.layers import Dense, ReLU
    from core.losses import SoftmaxCrossEntropyLoss
    from core.model import Model
    from core.nn import Net
    from core.optimizer import Adam
    layers = []
    for i, w in enumerate(cfg["widths"]):
        layers.append(Dense(w))
        if i + 1 < len(cfg["widths"]):
            layers.append(ReLU())
    net = Net(layers)
    return net, Model(net=net, loss=SoftmaxCrossEntropyLoss(), optimizer=Adam(lr=1e-3))


def synthetic_shard(cfg, B, rank, copies=2):
    """`copies` synthetic batches of B rows for this rank: float32 inputs U[0,1), int labels"""
    rng = np.random.RandomState(1000 + rank)
    C = cfg["widths"][-1]
    xs = [rng.rand(B, cfg["d_in"]).astype(np.float32) for _ in range(copies)]
    ys = [rng.randint(0, C, B).astype(np.int32) for _ in range(copies)]
    return xs, ys


def one_hot_host(labels, C):
    out = np.zeros((len(labels), C), np.float32)
    out[np.arange(len(labels)), labels] = 1.0
    return out


class Stepper(object):
    """the reference's five-line training loop body (run.py:79-83), or its recorded replay"""

    def __init__(self, cfg, use_graph, defer_loop=False):
        """use_graph: Model.train_step instead of the five lines.  defer_loop: leave the engine's
        transparent recording of the five-line loop on (core/_deferred.py: small steps only); off,
        the five lines are launched kernel by kernel as written."""
        from core.losses import SoftmaxCrossEntropyLoss
        np.random.seed(0)
        self.net, self.model = build_model(cfg)
        self.model.defer_loop = bool(defer_loop)
        self.loss_layer = SoftmaxCrossEntropyLoss()
        self.use_graph = use_graph
        self.keep_outputs = False    # keep the last step's (loss, prediction) for --dump-outputs
        self.outputs = None

    def __call__(self, x_t, y_t):
        if self.use_graph:   # the same five calls, recorded once per batch shape and replayed
            loss, pred = self.model.train_step(x_t, y_t), None
        else:
            m = self.model
            m.zero_grad()
            pred = m.forward(x_t)
            loss = self.loss_layer.loss(pred, y_t)
            loss.backward()
            m.step()
        if self.keep_outputs:
            self.outputs = (loss, pred)
        return loss

    def param_checksum(self):
        import core._backend as be
        a = self.model._arena
        if a is None:
            return None
        host = be.to_numpy(a["p"])
        return float(np.sum(host.astype(np.float64))), float(np.sum(np.abs(host).astype(np.float64)))


def dump_outputs(stepper, out_dir):
    """--dump-outputs: the last step's loss, prediction and updated parameters as out_dir/<name>.npy
    (see the module docstring); returns the names written"""
    loss, pred = stepper.outputs
    arrays = {"loss": loss.values}
    if pred is not None:
        arrays["prediction"] = pred.values
    for i, layer in enumerate(stepper.net.get_parameters()):
        for key, p in layer.items():
            if p is not None:
                arrays["layer%d_%s" % (i, key)] = p.values
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, np.float64 if np.asarray(a).dtype == np.float64 else np.float32)
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sorted(arrays)


LAST_TIMED_REGION = {}   # host-side facts about the most recent timed loop (diagnostics)


def timed_steps(stepper, x_dev, y_dev, steps, warmup, profile_gemm):
    """(ms for `steps` steps, launches, gemm_ms, gemm_n, last loss) with device-resident inputs"""
    import core._backend as be
    import core._dist as dist
    from core.tensor import Tensor
    loss = None
    for i in range(warmup):
        loss = stepper(Tensor(x_dev[i % len(x_dev)]), Tensor(y_dev[i % len(y_dev)]))
    if loss is not None:
        float(loss.values)
    dist.barrier()
    if profile_gemm:
        be.prof_enable(1)     # per-launch events around the tcgen05 GEMM (not recordable in a graph)
    launches0 = be.launch_count()
    mallocs0 = be.pool_stats()["cuda_mallocs"]
    gc0 = [g["collections"] for g in gc.get_stats()]
    ev0, ev1 = be.Event(), be.Event()
    t_host = time.perf_counter()
    ev0.record()
    for i in range(steps):
        loss = stepper(Tensor(x_dev[i % len(x_dev)]), Tensor(y_dev[i % len(y_dev)]))
    ev1.record()
    host_ms = (time.perf_counter() - t_host) * 1e3
    dist.barrier()
    ms = ev1.elapsed_ms_since(ev0)
    launches = be.launch_count() - launches0
    LAST_TIMED_REGION.update(
        host_enqueue_ms=host_ms, cuda_mallocs=be.pool_stats()["cuda_mallocs"] - mallocs0,
        gc_collections=[g["collections"] - a for g, a in zip(gc.get_stats(), gc0)])
    gemm_ms, gemm_n = (0.0, 0)
    if profile_gemm:
        gemm_ms, gemm_n = be.prof_collect()
        be.prof_enable(0)
    return ms, launches, gemm_ms, gemm_n, float(loss.values)


def max_over_ranks(values):
    import core._dist as dist
    if dist.world_size() == 1:
        return list(values)
    import torch
    import torch.distributed as td
    t = torch.tensor(list(values), dtype=torch.float64)
    td.all_reduce(t, op=td.ReduceOp.MAX)
    return [float(v) for v in t]


def gather_over_ranks(values):
    import core._dist as dist
    if dist.world_size() == 1:
        return [list(values)]
    import torch
    import torch.distributed as td
    t = torch.tensor(list(values), dtype=torch.float64)
    out = [torch.zeros_like(t) for _ in range(dist.world_size())]
    td.all_gather(out, t)
    return [[float(v) for v in o] for o in out]


def measure_strong(cfg, rank, world, steps=8, warmup=3):
    """BASELINE.json configs[4]: global batch 65536 fixed, 65536/N rows on each GPU"""
    import core._backend as be
    if STRONG_GLOBAL_BATCH % world:
        return None
    B = STRONG_GLOBAL_BATCH // world
    C = cfg["widths"][-1]
    xs, ys = synthetic_shard(cfg, B, rank, copies=1)
    x_dev = [be.from_numpy(xs[0])]
    y_dev = [be.empty((B, C), be.F32)]
    lab = be.from_numpy(ys[0].view(np.float32))
    be.one_hot_into(y_dev[0], lab.ptr, B, C)
    del xs
    stepper = Stepper(cfg, use_graph=False)
    ms, launches, _, _, last = timed_steps(stepper, x_dev, y_dev, steps, warmup, profile_gemm=False)
    ms = max_over_ranks([ms])[0]
    return {"config": "BASELINE.json configs[4]", "global_batch": STRONG_GLOBAL_BATCH,
            "batch_per_gpu": B, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "value": STRONG_GLOBAL_BATCH * steps / (ms * 1e-3),
            "unit": "samples/s", "final_loss": last,
            "efficiency": "T(1) / (N * T(N)) over the ms_per_step of the N = 1, 2, 4, 8 lines"}


def measure_allreduce(n_elems, reps=20):
    """the gradient all-reduce alone: `reps` back-to-back in-place SUMs of an arena-sized vector"""
    import core._backend as be
    import core._dist as dist
    world = dist.world_size()
    buf = be.zeros((n_elems,), be.F32)
    for _ in range(3):
        dist.allreduce_sum(buf)
    dist.barrier()
    e0, e1 = be.Event(), be.Event()
    e0.record()
    for _ in range(reps):
        dist.allreduce_sum(buf)
    e1.record()
    dist.barrier()
    ms = max_over_ranks([e1.elapsed_ms_since(e0)])[0] / reps
    nbytes = n_elems * 4
    return {"bytes": nbytes, "ms": ms, "algbw_gbs": nbytes / (ms * 1e-3) / 1e9,
            "busbw_gbs": 2.0 * (world - 1) / world * nbytes / (ms * 1e-3) / 1e9,
            "reps": reps, "nvlink5_per_direction_gbs": 900.0}


def measure_mnist(steps=2000, warmup=50):
    """BASELINE.json configs[0] on one GPU: examples/mnist/run.py's network and loop at batch 128"""
    import core._backend as be
    cfg = dict(MNIST)
    B, C = cfg["batch"], cfg["widths"][-1]
    xs, ys = synthetic_shard(cfg, B, 0, copies=2)
    x_dev = [be.from_numpy(x) for x in xs]
    y_dev = [be.from_numpy(one_hot_host(y, C)) for y in ys]
    out = {"config": "BASELINE.json configs[0]", "workload": cfg["name"], "batch": B}
    # eager: the five lines of run.py:79-83 launched kernel by kernel; five_line_loop: the same five
    # lines, unmodified, with the engine's transparent recording on (its default); train_step: the
    # explicit one-call API
    for mode, use_graph, defer in (("eager_five_line_loop", False, False),
                                   ("five_line_loop_recorded_transparently", False, True),
                                   ("recorded_train_step", True, False)):
        stepper = Stepper(cfg, use_graph, defer)
        ms, launches, _, _, last = timed_steps(stepper, x_dev, y_dev, steps, warmup, profile_gemm=False)
        out[mode] = {"ms_per_step": ms / steps, "value": B * steps / (ms * 1e-3), "unit": "samples/s",
                     "steps": steps, "launches_per_step": launches / steps, "final_loss": last}
    return out


def run_b200_arm(args, cfg):
    import core._backend as be
    import core._dist as dist
    from core.tensor import Tensor

    dist.init_process_group()
    rank, world = dist.rank(), dist.world_size()
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d (launch N>1 with torchrun)" % (args.gpus, world))
    numa = dist.bind_to_local_numa_node()    # pinned staging buffers land next to this rank's GPU
    B = args.batch_per_gpu or cfg["batch"]
    if args.global_batch:
        lo, hi = dist.shard_bounds(args.global_batch, rank, world)
        if (hi - lo) * world != args.global_batch:
            raise SystemExit("--global-batch must be divisible by the number of GPUs")
        B = hi - lo
    C = cfg["widths"][-1]
    peaks = read_peaks()
    wide = args.workload == "wide"

    # synthetic inputs, one shard per rank; identical reference-style init on every rank
    xs, ys = synthetic_shard(cfg, B, rank, copies=2)
    x_dev = [be.from_numpy(x) for x in xs]
    y_dev = [be.from_numpy(one_hot_host(y, C)) for y in ys]
    use_graph = args.graph == "on" or (args.graph == "auto" and args.workload == "mnist")
    stepper = Stepper(cfg, use_graph)
    stepper.keep_outputs = bool(args.dump_outputs) and rank == 0

    # ---- step-0 loss: with zero biases and Xavier weights the logits are O(1) and the global
    # softmax is near uniform over B_global*C entries, so loss_0 = ln(B_global*C) up to the logit spread
    loss0 = float(stepper(Tensor(x_dev[0]), Tensor(y_dev[0])).values)
    expect0 = math.log(B * world * C)
    checks = {"loss_step0": loss0, "ln_Bglobal_C": expect0, "loss_step0_ok": abs(loss0 - expect0) < 0.25}
    if not checks["loss_step0_ok"]:
        raise SystemExit("step-0 loss %.4f is not ln(B_global*C) = %.4f: the CE normaliser does not "
                         "span the global batch" % (loss0, expect0))

    # ---- device-resident throughput ("value") --------------------------------------------------
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    sampler.start()                       # nvidia-smi needs ~0.3 s to produce its first sample
    loss = None
    for i in range(1, args.warmup):       # the step-0 check above was warm-up step 0
        # (bound to a name like in the timed loop: step i's graph then lives until step i+1 has
        # produced its loss, so the pool reaches its steady-state footprint during warm-up)
        loss = stepper(Tensor(x_dev[i % 2]), Tensor(y_dev[i % 2]))
    loss = None                           # (or the timed loop would keep a third graph alive)
    be.sync()
    s_first = sampler.mark()
    ms, launches, gemm_ms, gemm_n, last_loss = timed_steps(stepper, x_dev, y_dev, args.steps, 0,
                                                           profile_gemm=not use_graph)
    s_last = sampler.mark() + 1
    clocks = sampler.stop(s_first, s_last)
    timed_region = dict(LAST_TIMED_REGION)
    if stepper.keep_outputs:              # before the e2e steps below move the parameters on
        dump_outputs(stepper, args.dump_outputs)
        stepper.keep_outputs, stepper.outputs = False, None

    # ---- replicas agree (driver-visible correctness at N>1) ------------------------------------
    if world > 1:
        sums = gather_over_ranks(stepper.param_checksum())
        same = all(s == sums[0] for s in sums)
        checks.update({"replica_param_checksums_equal": same, "param_sum": sums[0][0], "param_abs_sum": sums[0][1]})
        if not same:
            raise SystemExit("replicas diverged: parameter checksums %r" % (sums,))

    # ---- end to end from host buffers ("e2e"): the public input pipeline ----------------------
    # utils.data_iterator.PrefetchIterator over a host data set of 4 batches (pinned in place):
    # batch i+1 is DMA'd on the copy stream while step i runs; labels travel as int32 and the
    # one-hot rows are built on the device; the loss is read back every step.
    from utils.data_iterator import PrefetchIterator
    n_host_batches = 4
    x_data = np.empty((n_host_batches * B, cfg["d_in"]), np.float32)
    y_data = np.empty((n_host_batches * B,), np.int32)
    for k in range(n_host_batches):
        x_data[k * B:(k + 1) * B] = xs[k % 2]
        y_data[k * B:(k + 1) * B] = ys[(k + 1) % 2]
    del xs
    e2e_steps = args.steps
    feed = iter(PrefetchIterator(batch_size=B, loop=True, num_classes=C)(x_data, y_data))
    for _ in range(max(args.warmup, n_host_batches + 1)):   # e2e warm-up: every host batch has crossed PCIe once
        batch = next(feed)
        float(stepper(batch.inputs, batch.targets).values)
    # the K-step region is timed twice and the faster run reported (both are in the JSON line): the
    # host side of this path -- DMA out of pinned pages, a Python thread feeding the queue -- shares
    # the box's CPU with whatever else runs there, and a one-off stall of a second has been seen
    e2e_runs = []
    for _rep in range(2):
        dist.barrier()
        t0 = time.perf_counter()
        e0, e1 = be.Event(), be.Event()
        e0.record()
        batch = next(feed)
        pending = None
        for _ in range(e2e_steps):
            loss = stepper(batch.inputs, batch.targets)      # queued; the GPU starts on it
            batch = next(feed)                               # H2D of a following batch is queued in here,
                                                             # while the GPU runs the step just queued
            read = loss.values_async()                       # D2H of this step's loss, on its own stream
            if pending is not None:
                float(pending.result())                      # the PREVIOUS step's loss is on the host now:
            pending = read                                   # every step's loss is read, one step late, and
                                                             # the host never drains the GPU's queue
        float(pending.result())                              # (inside the timed region)
        e1.record()
        dist.barrier()
        run_ms = max(e1.elapsed_ms_since(e0), (time.perf_counter() - t0) * 1e3)
        e2e_runs.append(max_over_ranks([run_ms])[0])
    e2e_ms = min(e2e_runs)
    feed.close()
    del feed, x_data, y_data

    ms = max_over_ranks([ms])[0]
    global_batch = B * world
    value = global_batch * args.steps / (ms * 1e-3)
    e2e_value = global_batch * e2e_steps / (e2e_ms * 1e-3)

    # ---- roofline of the dominant kernel (tcgen05 split GEMM) ----------------------------------
    flops_step = gemm_flops_per_step(cfg, B)
    roofline = None
    if gemm_n:
        per_launch_flops = flops_step * args.steps / gemm_n
        achieved = per_launch_flops / (gemm_ms / gemm_n * 1e-3) / 1e12
        # tensor-pipe cost of one algorithmic MMA, in bf16-MMA equivalents (a TF32 MMA costs two):
        #   f16 : 3 F16 = 3      mix : 1 TF32 + 2 BF16 = 4        tf32x3 : 3 TF32 = 6
        mix = be.TC_SPLIT == "mix"
        cost = {"f16": 3.0, "mix": 4.0}.get(be.TC_SPLIT, 6.0)
        split_desc = {"f16": "3 F16 MMAs per algorithmic MMA (scaled fp16 hi/lo planes)",
                      "mix": "1 TF32 + 2 BF16 MMAs per algorithmic MMA"}.get(
                          be.TC_SPLIT, "3 TF32 MMAs per algorithmic MMA")
        # denominator: the BURST cuBLAS figure.  MEASURED_PEAKS' sustained figure belongs to seconds of
        # back-to-back tensor work under the power cap (SM clocks ~1.35 GHz); the launches timed here sit
        # between memory-bound kernels in a region of a fraction of a second at 1.6-1.9 GHz, and against
        # the sustained figure they read 0.94-1.02 -- not a meaningful fraction.  Both are reported.
        peak = peaks["bf16_burst"] / cost
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
        if os.path.exists(tpath):   # dram bytes per launch from the committed ncu --set full capture
            traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic,
                    "frac_of_burst": achieved / (peaks["bf16_burst"] / cost),
                    "frac_of_sustained": achieved / (peaks["bf16_sustained"] / cost),
                    "frac_of_nominal": achieved / (2250.0 / cost),
                    "kernel": ("gemm_f16x3_kernel" if be.TC_SPLIT == "f16"
                               else "gemm_tf32x3_kernel<MIX=%d>" % int(mix)), "launches": int(gemm_n),
                    "avg_launch_ms": gemm_ms / gemm_n, "share_of_step": gemm_ms / ms,
                    "split": be.TC_SPLIT,
                    "peak_source": "%s bf16 burst %.1f TFLOP/s / %d (%s); sustained %.1f / %d" % (
                        peaks["source"], peaks["bf16_burst"], int(cost), split_desc,
                        peaks["bf16_sustained"], int(cost))}

    # ---- the extra measurements ------------------------------------------------------------------
    arena_elems = stepper.model._arena["p"].size if stepper.model._arena else 0
    del stepper, x_dev, y_dev
    strong = allred = mnist = None
    if wide and not args.global_batch and not args.no_extras:
        if world > 1 and arena_elems:
            allred = measure_allreduce(arena_elems)
        strong = measure_strong(cfg, rank, world)
        if world == 1:
            mnist = measure_mnist()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, s_per, desc = cpu_reference_throughput(cfg, steps=2, warmup=1)
        cpu_baseline = {"value": v, "unit": "samples/s", "cores": host_cores(), "kind": "port",
                        "sample": desc}

    if rank == 0:
        line = {
            "metric": "MLP train samples/sec", "value": value, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.global_batch else "weak",
            "vs_baseline": None,
            "dtype": "f32 (tensor-core GEMMs: %s, fp32 accumulate)" % (
                {"f16": "3-term split on scaled fp16 hi/lo planes", "mix": "tf32 main term + bf16 cross terms"}.get(
                    be.TC_SPLIT, "3xTF32")),
            "data": "synthetic",
            "config": make_config(cfg, B, world),
            "step_mode": "cuda_graph_replay" if use_graph else "eager_launches",
            "roofline": roofline, "cpu_baseline": cpu_baseline,
            "e2e": {"value": e2e_value, "unit": "samples/s",
                    "h2d_bytes_per_step": int(B * cfg["d_in"] * 4 + B * 4), "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / e2e_steps,
                    "ms_per_step_runs": [r / e2e_steps for r in e2e_runs],
                    "pipeline": "PrefetchIterator: float32 inputs + int32 labels from pinned host "
                                "memory on a copy stream, the fused cross-entropy reads the class indices (no dense one-hot rows); every "
                                "step's loss is read back to the host one step behind"},
            "gpu_launches": int(launches), "clocks": clocks, "final_loss": last_loss,
            "gemm_tflops_algorithmic": flops_step * args.steps / (ms * 1e-3) / 1e12,
            "checks": checks, "numa": numa, "timed_region": timed_region,
            "strong_scaling": strong, "allreduce": allred, "mnist": mnist,
        }
        print(json.dumps(line))
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="wide", choices=["wide", "mnist"])
    ap.add_argument("--batch-per-gpu", type=int, default=0)
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling: fix the global batch (BASELINE config 5 uses 65536) and "
                         "split it over the ranks; reported with \"scaling\": \"strong\"")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the step as a CUDA graph (Model.train_step); auto = on for the "
                         "launch-bound mnist workload, off for the wide MLP")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the strong-scaling / all-reduce / mnist side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's loss, prediction and updated parameters to "
                         "DIR/<name>.npy (large outputs as a fixed seeded sample)")
    args = ap.parse_args()
    args.steps_given = args.steps is not None
    if args.steps is None:
        args.steps = 50
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    cfg = dict(WIDE if args.workload == "wide" else MNIST)
    if args.impl == "reference":
        run_reference_arm(args, cfg)
    else:
        run_b200_arm(args, cfg)


if __name__ == "__main__":
    main()
