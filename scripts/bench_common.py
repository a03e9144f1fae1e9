"""Measurement helpers the benchmark scripts share: JSON output, the card's identity, rotating-buffer
kernel timing and alternating model timing.  The importing script puts the repository root on
sys.path first."""
import json
import subprocess
import time

import core._backend as be

# added to every emitted row once a script fills it (card() read in the same run)
CARD = {}


def emit(**row):
    row.update(CARD)
    print(json.dumps(row), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock)


def timed_rotating(make_launch, n_sets, reps=5):
    """make_launch(k) issues the op on buffer set k; returns ms per launch"""
    for k in range(n_sets):           # eager warm-up (scratch growth, lazily allocated counters)
        make_launch(k)
    be.sync()
    g = be.StepGraph()
    with g.capture():
        for k in range(n_sets):
            make_launch(k)
    g.replay()
    be.sync()
    best = 1e30
    e0, e1 = be.Event(), be.Event()
    for _ in range(reps):
        e0.record()
        g.replay()
        e1.record()
        best = min(best, e1.elapsed_ms_since(e0))
    g.destroy()
    return best / n_sets


def alternate(models, steps, rounds, run_one):
    """times `steps` calls of run_one(model) for each of the named models in turn, `rounds` times
    over; yields (name, ms per step) after each timing"""
    for _ in range(rounds):
        for name, model in models.items():
            be.sync()
            t0 = time.perf_counter()
            for _ in range(steps):
                run_one(model)
            be.sync()
            yield name, (time.perf_counter() - t0) * 1e3 / steps
