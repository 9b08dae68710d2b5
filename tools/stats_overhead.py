#!/usr/bin/env python
"""Cost of lbm_stats_start (time-averaged rho, u and velocity covariance accumulated inside the step) on three workloads
of bench.py at its size (8192 x 8192, one GPU).

    python tools/stats_overhead.py [--steps K] [--warmup W] [--blocks B] [--profile N] [--out FILE]

For each of `cylinder` (BGK + immersed cylinder), `cylinder_bb` (BGK, staircase body under bounce-back) and `kbc_shear`
(KBC double shear layer) one domain is set up with bench.py's own geometry, rules and initial state.  Three settings
then alternate in B blocks: no record, a record with every = 1 and one with every = 10.  Each block sets the mode, runs
W warm-up steps and times K steps with CUDA events on the domain's stream (lbm_last_step_ms).

Byte model (fp64, bytes per node and step): the plain step reads and writes nine populations, 144 B; a sampled step also
reads and writes the six accumulators, 240 B.  The plain step's rate, 144 B x nodes / its time, is the copy rate this
kernel reaches; the model time of a setting is its bytes at that rate, and `model_over_measured` is the fraction of that
rate the setting reaches.  Prints one JSON object (the card's name and power limit read in the same process) and writes it
to --out when given.  --profile N adds, per workload and setting, the device time of each step kernel over N steps from
a torch.profiler run of its own (after the timed blocks, so the timings are taken with the profiler off).
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

import bench  # noqa: E402  (puts the binding on sys.path)
import lbm_b200 as L  # noqa: E402
from body_force_overhead import card  # noqa: E402

STEP_BYTES, STATS_BYTES = 144.0, 96.0
SETTINGS = (("off", 0), ("every1", 1), ("every10", 10))


def domain(workload, X, Y):
    omega, u_lb = bench.lattice_parameters()
    rho = np.ones((X, Y, 1))
    u = np.zeros((X, Y, 2))
    if workload == "kbc_shear":
        d = L.Domain(L.default_config(model=L.MODEL_KBC, X=X, Y=Y, omega=1.0 / (0.5 + 3.0 * 1.70766666e-4)))
        d.preset_periodic()
        r, c = np.arange(X)[:, None], np.arange(Y)[None, :]
        u[..., 0] = 0.02 * np.tanh(80.0 * (0.25 * X - np.abs(c - 0.5 * X))) + 0.0 * r
        u[..., 1] = 0.02 * 0.05 * np.sin(6.2832 * (r + 0.25 * X) / X) + 0.0 * c
        d.init_equilibrium(rho, u, L.EQ_KBC_FRESH)
        d.set_moments(rho, u)
        return d
    force = L.FORCE_IBM if workload == "cylinder" else L.FORCE_NONE
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=omega, equilibrium=L.EQ_COMPRESSIBLE, force=force))
    d.preset_free_stream(u_lb, 0.0)
    if workload == "cylinder_bb":
        d.bc_add_solid(bench.cylinder_solid(X, Y, X))
        d.bc_commit()
    else:
        d.ibm_set_markers(*bench.cylinder_markers(X, Y))
    u[..., 0] = u_lb
    d.init_equilibrium(rho, u, L.EQ_INCOMPRESSIBLE)
    return d


def kernel_times(d, n_steps):
    """{kernel: (device ms per step, launches per step)} of n_steps steps, from torch.profiler's CUDA activity"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    d.step(2)
    d.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        d.step(n_steps)
        d.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA and ("k_" in e.key):
            name = e.key.split("(")[0].replace("void lbm::", "").replace("lbm::", "")
            total_us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            out[name] = (total_us / 1e3 / n_steps, e.count / n_steps)
    return out


def measure(workload, X, Y, steps, warmup, blocks, profile_steps=0):
    d = domain(workload, X, Y)
    ms = {name: [] for name, _ in SETTINGS}
    samples = {}
    for _ in range(blocks):
        for name, every in SETTINGS:
            if every:
                d.stats_start(every)
            d.step(warmup)
            d.step(steps)
            ms[name].append(d.last_step_ms() / steps)
            if every:
                n, rho_mean, _, _ = d.stats()
                want = len(range(0, warmup + steps, every))
                if n != want:
                    raise RuntimeError(f"{workload} every = {every}: {n} samples, expected {want}")
                samples[name] = dict(n=n, rho_mean_finite=bool(np.isfinite(rho_mean).all()))
                d.stats_stop()
    prof = {}
    for name, every in SETTINGS[:2] if profile_steps else ():
        if every:
            d.stats_start(every)
        prof[name] = kernel_times(d, profile_steps)
        if every:
            d.stats_stop()
    d.close()
    nodes = float(X) * Y
    med = {name: statistics.median(v) for name, v in ms.items()}
    t0 = med["off"]
    rate = STEP_BYTES * nodes / (t0 * 1e-3)  # B/s the plain step moves
    out = dict(workload=workload, X=X, Y=Y, steps_per_block=steps, warmup_per_block=warmup, blocks=blocks,
               ms_per_step=ms, median_ms=med, plain_step_rate_GBps=rate / 1e9, samples=samples, settings={})
    for name, every in SETTINGS[1:]:
        model_bytes = STEP_BYTES + STATS_BYTES / every
        model_ms = model_bytes * nodes / rate * 1e3
        out["settings"][name] = dict(every=every, model_bytes_per_node=model_bytes, model_ms=model_ms,
                                     time_over_plain=med[name] / t0, model_time_over_plain=model_bytes / STEP_BYTES,
                                     model_over_measured=model_ms / med[name])
    # the sampled step alone: every = 1 samples every step
    out["sampled_step_ms"] = med["every1"]
    out["sampled_step_fraction_of_plain_rate"] = out["settings"]["every1"]["model_over_measured"]
    if prof:
        out["profile_ms_per_step"] = prof
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--X", type=int, default=bench.WORKLOADS["cylinder"]["X"])
    ap.add_argument("--Y", type=int, default=bench.WORKLOADS["cylinder"]["Y"])
    ap.add_argument("--workloads", default="cylinder,cylinder_bb,kbc_shear")
    ap.add_argument("--profile", type=int, default=0, help="steps of a torch.profiler run per workload and setting (0: none)")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    out = dict(card=card(), library=L.version(), bytes_per_node=dict(step=STEP_BYTES, sampled_step=STEP_BYTES + STATS_BYTES),
               results=[measure(w, a.X, a.Y, a.steps, a.warmup, a.blocks, a.profile) for w in a.workloads.split(",")])
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
