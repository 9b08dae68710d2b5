#!/usr/bin/env python
"""Cost of lbm_body_force_record on the two cylinder workloads of bench.py, at bench.py's size (8192 x 8192, one GPU).

    python tools/body_force_overhead.py [--steps K] [--warmup W] [--blocks B] [--out FILE]

For each of `cylinder_bb` (staircase body, momentum exchange over its bounce-back links) and `cylinder` (immersed body,
-sum of its force field) one domain is set up with bench.py's own geometry (cylinder_solid, cylinder_markers) and rules.
Recording off and on then alternate in B blocks: each block sets the mode, runs W warm-up steps and times K steps with
CUDA events on the domain's stream (lbm_last_step_ms).  Prints one JSON object (the card's name and power limit read in
the same process) and writes it to --out when given.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (puts the binding on sys.path)
import lbm_b200 as L  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvidia-smi failed: {r.stderr.strip()}")
    name, power, clock = [s.strip() for s in r.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def domain(workload, X, Y):
    omega, u_lb = bench.lattice_parameters()
    force = L.FORCE_IBM if workload == "cylinder" else L.FORCE_NONE
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=omega, equilibrium=L.EQ_COMPRESSIBLE, force=force))
    d.preset_free_stream(u_lb, 0.0)
    solid = None
    if workload == "cylinder_bb":
        solid = bench.cylinder_solid(X, Y, X)
        d.bc_add_solid(solid)
        d.bc_commit()
    else:
        d.ibm_set_markers(*bench.cylinder_markers(X, Y))
    rho = np.ones((X, Y, 1))
    u = np.zeros((X, Y, 2))
    u[..., 0] = u_lb
    d.init_equilibrium(rho, u, L.EQ_INCOMPRESSIBLE)
    return d, solid


def measure(workload, X, Y, steps, warmup, blocks):
    d, solid = domain(workload, X, Y)
    ms = {"off": [], "on": []}
    for _ in range(blocks):
        for mode in ("off", "on"):
            if mode == "on":
                d.body_force_record(solid, capacity=warmup + steps)
            else:
                d.body_force_stop()
            d.step(warmup)
            d.step(steps)
            ms[mode].append(d.last_step_ms() / steps)
            if mode == "on":
                F, first = d.body_force()
                if len(F) != warmup + steps or first != 0:
                    raise RuntimeError(f"{workload}: the record holds {len(F)} steps from {first}, expected {warmup + steps} from 0")
    d.close()
    off, on = statistics.median(ms["off"]), statistics.median(ms["on"])
    finite = np.isfinite(F).all(axis=1)
    # the flow itself may leave the finite range at this Reynolds number; the record says from which step on
    return dict(workload=workload, X=X, Y=Y, steps_per_block=steps, warmup_per_block=warmup, blocks=blocks,
                ms_per_step_off=ms["off"], ms_per_step_on=ms["on"], median_ms_off=off, median_ms_on=on,
                overhead_percent=100.0 * (on - off) / off,
                steps_with_finite_force=int(np.argmin(finite)) if not finite.all() else int(len(F)),
                first_force=[float(v) for v in F[0]], last_finite_force=[float(v) for v in F[finite][-1]] if finite.any() else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--X", type=int, default=bench.WORKLOADS["cylinder"]["X"])
    ap.add_argument("--Y", type=int, default=bench.WORKLOADS["cylinder"]["Y"])
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    out = dict(card=card(), library=L.version(),
               results=[measure(w, a.X, a.Y, a.steps, a.warmup, a.blocks) for w in ("cylinder_bb", "cylinder")])
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
