"""BASELINE.json config 3: elementwise / broadcast / reduce sweep, achieved HBM GB/s per op and
size against the measured copy bandwidth (MEASURED_PEAKS.json hbm_gbs).

    python scripts/sweep_ops.py [--max-log2 30] [--cpu] > gpurun_out/sweep.json

Algorithmic bytes per element (fp32): add/mul 12, bias-add 8, relu fwd 8, relu bwd 12,
unbroadcast (R,1024)->(1,1024) 4, Adam 28.

Timing (r02): for every (op, size) K launches over K ROTATING buffer sets -- K chosen so the sets
together exceed twice the L2, every launch therefore reads cold data from HBM -- are recorded into
one CUDA graph and replayed; time = best of 5 replays / K, CUDA events on the compute stream.  A
replayed graph has no host in the loop, so the small sizes measure the kernel (launch ramp
included), not the Python call that r01's one-launch-per-event-pair timing was bound by.
With --cpu the numpy oracle's ops are timed next to it."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import core._backend as be  # noqa: E402
from bench_common import timed_rotating  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-log2", type=int, default=30)
    ap.add_argument("--cpu", action="store_true")
    args = ap.parse_args()
    be.init()
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6650.0
    l2 = be.device_info()["l2_bytes"]
    rows = []
    for lg in range(20, args.max_log2 + 1, 2):
        n = 1 << lg
        R_, C_ = n // 1024, 1024
        # rotating sets: together more than twice the L2 (4 tensors of n floats per set), 2..48 sets
        n_sets = int(min(48, max(2, -(-2 * l2 // (4 * n * 4)))))
        sets = []
        for k in range(n_sets):
            sets.append(dict(a=be.full((R_, C_), 0.5, be.F32), b=be.full((R_, C_), 0.25, be.F32),
                             out=be.empty((R_, C_), be.F32), cs=be.empty((1, C_), be.F32),
                             v=be.full((R_, C_), 0.25, be.F32)))
        bias = be.full((1, C_), 0.125, be.F32)
        h = [1e-3, 0.9, 0.999, 1e-8, 0.1, 0.001]
        ops = [
            ("add", 12, lambda k: be.ew(be.ADD, sets[k]["a"], sets[k]["b"], out=sets[k]["out"])),
            ("mul", 12, lambda k: be.ew(be.MUL, sets[k]["a"], sets[k]["b"], out=sets[k]["out"])),
            ("bias_add", 8, lambda k: be.ew(be.ADD, sets[k]["a"], bias, out=sets[k]["out"])),
            ("relu_fwd", 8, lambda k: be._lib.tnn_relu_fwd(0, sets[k]["out"].ptr, sets[k]["a"].ptr, n)),
            ("relu_bwd", 12, lambda k: be._lib.tnn_relu_bwd(0, sets[k]["out"].ptr, sets[k]["b"].ptr,
                                                            sets[k]["a"].ptr, n)),
            ("unbroadcast_colsum", 4, lambda k: be.colsum(sets[k]["a"], out=sets[k]["cs"])),
            # Adam: param = out, grad = b, m = a, v = v (28 B/elem: g, m, v, p read; m, v, p written)
            ("adam", 28, lambda k: be.opt_step(be.OPT_ADAM, sets[k]["out"].view((n,)), None,
                                               sets[k]["b"].view((n,)), sets[k]["a"].view((n,)),
                                               sets[k]["v"].view((n,)), h)),
        ]
        for name, bpe, fn in ops:
            ms = timed_rotating(fn, n_sets)
            gbs = n * bpe / (ms * 1e-3) / 1e9
            rows.append(dict(op=name, log2_n=lg, bytes_per_elem=bpe, ms=ms, gbs=gbs,
                             frac_of_measured_hbm=gbs / hbm, rotating_sets=n_sets))
        del sets
    result = dict(hbm_peak_gbs=hbm, rows=rows)
    if args.cpu:
        import ref_numpy as R
        cpu = []
        for lg in (24, 26):
            n = 1 << lg
            x = np.full((n // 1024, 1024), 0.5, np.float32)
            y = np.full((n // 1024, 1024), 0.25, np.float32)
            bias = np.full((1, 1024), 0.125, np.float32)
            tx, ty, tb = R.RefTensor(x), R.RefTensor(y), R.RefTensor(bias, requires_grad=True)
            cases = [("add", 12, lambda: R.add(tx, ty)), ("mul", 12, lambda: R.mul(tx, ty)),
                     ("bias_add", 8, lambda: R.add(tx, tb)), ("relu_fwd", 8, lambda: R.clip(tx, 0.0)),
                     ("unbroadcast_colsum", 4, lambda: R.unbroadcast(x, (1, 1024)))]
            for name, bpe, fn in cases:
                best = 1e30
                for _ in range(3):
                    t0 = time.perf_counter()
                    fn()
                    best = min(best, time.perf_counter() - t0)
                cpu.append(dict(op=name, log2_n=lg, gbs=n * bpe / best / 1e9))
        result["cpu_numpy_oracle"] = cpu
        result["cpu_cores"] = len(os.sched_getaffinity(0))
    print(json.dumps(result))


if __name__ == "__main__":
    main()
