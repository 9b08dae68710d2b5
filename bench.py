#!/usr/bin/env python
"""bench.py — MLUPS of the fused D2Q9 collide+stream step on B200 (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py --impl reference --steps K --warmup W    (the reference's CPU path, rank 0 only)
    python bench.py --workload mrtcg_rt|rk_droplet|sedimentation|...   (one of the other configs as the headline, nothing else)

A "step" is one lattice-Boltzmann time step of the whole grid.  Headline workload at every N: configs[1] of BASELINE.json —
flow past a cylinder, D2Q9 BGK, compressible equilibrium, immersed-boundary cylinder (multi-direct forcing),
anti-bounce-back inlet/outlet rows, specular side columns (test/cylinder_test.cpp of the reference), 8192 x 8192 nodes PER
GPU (weak scaling: the global grid is (8192 N) x 8192, slab-decomposed along axis 0 like test/decompose_domain.cpp).

After W warm-up steps (at least 4 where the step pair replays as a CUDA graph: its capture takes 4), exactly K steps are
timed as one block with CUDA events on the domain's stream (max over ranks).
--dump-outputs DIR then writes what those steps left in the headline domain (see dump_outputs), so that two builds run
with the same arguments can be compared output for output.  Rank 0 prints ONE JSON line.  Beside the headline the same line carries
  other_workloads  N = 1: every other BASELINE.json config at its named size (device-resident value + roofline of its
                   dominant kernel); every N: `mrtcg_rt_weak`, the MRT colour-gradient step at 8192 x 16384 nodes per GPU —
                   the model with two-row moment-plane halos — so that the 1 -> 8 GPU records hold a curve for it too
  ring_parity      N > 1: before anything is timed, every model on a small grid over THIS ring of N ranks against the
                   monolithic run on rank 0's GPU (bit_exact or the relative error), lbm_comm_check and the ring-wide
                   max of the RK diagnostics included
The CPU baseline (N = 1 only) runs after all GPU work, so no GPU idles in a collective while host cores are timed.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "lattice-boltzmann-method_b200", "python"))

FALLBACK_HBM_GBS = 6650.0        # B200 HBM3e bandwidth assumed where no MEASURED_PEAKS.json gives a measured one
CSF_FUSED_DEFAULT = "1"          # the library's default for LBM_CSF_FUSED (csrc/lbm_two_phase.cu: the single pass, k_csf_staged)

W9 = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
CX9 = np.array([0, 1, 0, -1, 0, 1, -1, -1, 1], dtype=np.float64)
CY9 = np.array([0, 0, 1, 0, -1, 1, 1, -1, -1], dtype=np.float64)

# BASELINE.json configs -> workload; bytes/node = SURVEY §8(d)'s minimal-traffic model (fp64, every population
# read once and written once; two-phase models add their scalar moment planes)
WORKLOADS = {
    # configs[1] — the headline: test/cylinder_test.cpp at 8192 x 8192 per GPU
    "cylinder": dict(X=8192, Y=8192, bytes=144.0, nlat=1, kernel="k_bgk_interior<PULL,COMP,IBM>", driver="test/cylinder_test.cpp",
                     what="cylinder flow, D2Q9 BGK + IBM cylinder, ABB inlet/outlet, specular walls", cpu_sample=1024),
    # configs[1] read literally ("flow past cylinder ... with bounce-back"): the same free-stream channel with a staircase
    # cylinder under link-wise half-way bounce-back instead of the reference driver's immersed-boundary body
    "cylinder_bb": dict(X=8192, Y=8192, bytes=144.0, nlat=1, kernel="k_bgk_interior<PULL,COMP,NONE>",
                        driver="test/cylinder_test.cpp (boundary rows/columns) + the obstacle-wall rule of test/rectangle_sedimentation_test.cpp:186-196",
                        what="flow past a staircase cylinder, D2Q9 BGK compressible, half-way bounce-back links, ABB inlet/outlet, specular side columns",
                        cpu_sample=1024),
    # configs[0] at the parameters.toml grid (the 21 x 21 reference case is a parity test)
    "poiseuille": dict(X=2700, Y=2100, bytes=144.0, nlat=1, kernel="k_bgk_interior<PULL,INCOMP,NONE>",
                       driver="test/horizontal_poiseuille_test.cpp",
                       what="horizontal Poiseuille, D2Q9 BGK incompressible, pressure-periodic rows, bounce-back walls",
                       cpu_sample=1024),
    # configs[2]
    "mrtcg_rt": dict(X=16384, Y=16384, bytes=352.0, nlat=2, kernel="k_tp_staged<MRTCG,3,3,STASH>",
                     driver="test/mrtcg_rayleigh_taylor.cpp",
                     what="MRT colour-gradient Rayleigh-Taylor (mrtcg-rayleigh-taylor-gamma3.toml), two lattices",
                     cpu_sample=512),
    # configs[2] per slab of a ring: what every N runs beside the headline (two-row moment-plane halos at every cut)
    "mrtcg_rt_weak": dict(X=8192, Y=16384, bytes=352.0, nlat=2, kernel="k_tp_staged<MRTCG,3,3,STASH>",
                          driver="test/mrtcg_rayleigh_taylor.cpp",
                          what="MRT colour-gradient Rayleigh-Taylor (mrtcg-rayleigh-taylor-gamma3.toml), two lattices, 8192 rows of 16384 columns per GPU",
                          cpu_sample=512),
    # configs[3]
    "rk_droplet": dict(X=4096, Y=4096, bytes=304.0, nlat=2, kernel="k_tp_staged<RK,5,2>",
                       driver="test/rk_static_droplet_test.cpp",
                       what="Rothman-Keller static droplet, R = L/4, two lattices", cpu_sample=512),
    # configs[4]
    "sedimentation": dict(X=4096, Y=8192, bytes=288.0, nlat=2, kernel="k_bgk_interior<PULL,COMP,NONE,ADE>",
                          driver="test/rectangle_sedimentation_test.cpp",
                          what="rectangle sedimentation: fluid + advection-diffusion lattice, bounce-back rectangle walls",
                          cpu_sample=1024),
    # configs[4] as BASELINE.json words it ("with immersed-boundary coupling (ibm)"): driver 15 has no ibm object (SURVEY §8
    # notes), so this is driver 15's loop plus a cylinder coupled the way driver 11 couples one; not a reference driver
    "sedimentation_ibm": dict(X=4096, Y=8192, bytes=288.0, nlat=2, kernel="k_bgk_interior<PULL,COMP,IBM,ADE>",
                              driver="test/rectangle_sedimentation_test.cpp + ibm as in test/cylinder_test.cpp",
                              what="rectangle sedimentation with an immersed cylinder: fluid (Guo-forced) + advection-diffusion lattice",
                              cpu_sample=1024),
    # not a BASELINE.json config: SURVEY §8(f) rank 2, the continuum-surface-force variant (one pass per step; bytes =
    # both colours' populations read + written once (288) + the carried interfacial tension read + written (32))
    "csf_rt": dict(X=8192, Y=8192, bytes=320.0, nlat=2, kernel="k_csf_staged<3,STASH>",
                   driver="test/mrt_rayleigh_taylor.cpp",
                   what="MRT colour-gradient Rayleigh-Taylor with continuum surface force (curvature from nested 5x5 differences)",
                   cpu_sample=512),
    # not a BASELINE.json config: the SURVEY §8(f) rank-3 collision (ulbm::d2q9::kbc), fully periodic double shear layer
    "kbc_shear": dict(X=8192, Y=8192, bytes=144.0, nlat=1, kernel="k_bgk_interior<PULL,KBC>",
                      driver="test/ulbm_double_shear_flow.cpp",
                      what="double shear layer, D2Q9 entropic central-moment (KBC) collision, fully periodic", cpu_sample=512),
}

RED = dict(rho_0=3.0, alpha=0.7, A=0.5, nu=0.04, beta=0.7)      # configs/mrtcg-rayleigh-taylor-gamma3.toml
BLUE = dict(rho_0=1.0, alpha=0.1, A=0.5, nu=0.04, beta=-0.7)
RK_RED = dict(rho_0=1.2, alpha=1.0 / 3.0, A=1e-4, nu=0.16, beta=0.7)   # rk_static_droplet_test.cpp:504-506
RK_BLUE = dict(rho_0=1.0, alpha=0.2, A=1e-4, nu=0.14, beta=-0.7)
RT_FG = (6.25e-6, 0.0)                                           # SURVEY §8(d) item 3


OTHERS_N1 = ["poiseuille", "mrtcg_rt", "rk_droplet", "sedimentation", "sedimentation_ibm", "kbc_shear", "csf_rt", "cylinder_bb",
             "mrtcg_rt_weak"]
OTHERS_RING = ["mrtcg_rt_weak"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cylinder", choices=sorted(WORKLOADS),
                    help="cylinder = BASELINE.json configs[1] (the headline); the others are the remaining configs")
    ap.add_argument("--X", type=int, default=0, help="rows per GPU (default: the workload's)")
    ap.add_argument("--Y", type=int, default=0, help="columns (default: the workload's)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="edge of the square grid the CPU baseline is timed on")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip other_workloads (they run only beside the default headline)")
    ap.add_argument("--no-ring-parity", action="store_true")
    ap.add_argument("--others", default="", help="comma-separated subset of other_workloads")
    ap.add_argument("--lib", default="", help="development: another build of the library (path) for an A/B run")
    ap.add_argument("--graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the step pair as a CUDA graph (auto: grids up to 2^24 nodes on one GPU, where launches bound the step)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the headline's state after the timed steps to DIR/<name>.npy (float64, sampled nodes on large "
                         "grids); the B200 arm only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the state of the B200 arm's domain: it needs --impl b200")
    wl = WORKLOADS[args.workload]
    args.X = args.X or wl["X"]
    args.Y = args.Y or wl["Y"]
    args.cpu_sample = args.cpu_sample or wl["cpu_sample"]
    return args


# ---------------------------------------------------------------------------------------------
# workload description (shared by both arms)
# ---------------------------------------------------------------------------------------------
PARAMETERS_TOML = os.path.join(ROOT, "configs", "parameters.toml")


def lattice_parameters():
    """B200 arm: omega and u_lb as the product's TOML surface derives them (lbm_params_from_toml = params::lattice)"""
    import lbm_b200 as L

    p = L.params_from_toml(PARAMETERS_TOML, False)
    return p.omega, p.u


def reference_lattice_parameters():
    """CPU arms: the same two numbers WITHOUT the product library — the reference's own params::lattice (oracle/_ref) where it
    compiled, else the C port fed from a plain TOML read"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    if oracle_lib.have_ref():
        p = oracle_lib.Ref().params(PARAMETERS_TOML, False)
        return float(p["omega"]), float(p["u"])
    import tomllib

    with open(PARAMETERS_TOML, "rb") as fh:
        t = tomllib.load(fh)
    fl, la = t["flow"], t["lattice"]
    p = oracle_lib.Oracle().params_lattice(fl["initial_density"], fl["kinematic_viscosity"], fl["characteristic_velocity"],
                                           fl["characteristic_length"], la["relaxation_time"], la["lattice_spacing"],
                                           la["x_multiplier"], la["y_multiplier"])
    return float(p["omega"]), float(p["u"])


def host_threads():
    """host cores this process may use (the CPU arms set their thread count to this explicitly)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def channel_constants(H, W, u_max=0.1030985714):
    """test/horizontal_poiseuille_test.cpp:50-66"""
    tau = np.sqrt(3.0 / 16.0) + 0.5
    nu = (2.0 * tau - 1.0) / 6.0
    p_grad = 8.0 * nu * u_max / (W * W)
    return 1.0 / tau, 3.0 * (H - 1) * p_grad + 1.0, 1.0


def cylinder_markers(X, Y):
    """Cylinder of diameter ~X/9 (the reference's X = 9 l proportion, src/params.cpp:64) centred at
    (X/4, Y/2), markers about one lattice unit apart on the circle."""
    D = max(8.0, X / 9.0)
    n = max(16, int(round(np.pi * D)))
    th = 2.0 * np.pi * np.arange(n) / n
    return X / 4.0 + 0.5 * D * np.cos(th) + 0.37, Y / 2.0 + 0.5 * D * np.sin(th) + 0.21


def cylinder_solid(Xg, Y, X1):
    """GLOBAL {Xg,Y} solid mask of the staircase cylinder: same centre and diameter as cylinder_markers of the first slab"""
    D = max(8.0, X1 / 9.0)
    solid = np.zeros((Xg, Y), dtype=np.uint8)
    lo, hi = max(0, int(X1 / 4.0 - D)), min(Xg, int(X1 / 4.0 + D) + 1)
    r2 = (np.arange(lo, hi)[:, None] - (X1 / 4.0 + 0.37)) ** 2 + (np.arange(Y)[None, :] - (Y / 2.0 + 0.21)) ** 2
    solid[lo:hi] = r2 <= (0.5 * D) ** 2
    return solid


def sedimentation_body(X, Y):
    """sedimentation_ibm: a cylinder of diameter ~X/9 upstream of the rectangle (the flow runs along axis 1), centred at
    (X/2, Y/4) of the first slab, markers about one lattice unit apart"""
    D = max(8.0, X / 9.0)
    n = max(16, int(round(np.pi * D)))
    th = 2.0 * np.pi * np.arange(n) / n
    return X / 2.0 + 0.5 * D * np.cos(th) + 0.37, Y / 4.0 + 0.5 * D * np.sin(th) + 0.21


def write_markers_toml(path, xs, ys):
    with open(path, "w") as fh:
        fh.write("[cylinder-a]\n")
        fh.write("x = [" + ", ".join(repr(float(v)) for v in xs) + "]\n")
        fh.write("y = [" + ", ".join(repr(float(v)) for v in ys) + "]\n")


def sedimentation_geometry(X, Y):
    """rectangle_sedimentation_test.cpp:73-75,89-95 scaled from the parameters.toml grid (2700 x 2100)"""
    R23 = -max(3, int(round(151 * X / 2700)))
    C28 = max(3, int(round(200 * Y / 2100)))
    C38 = max(C28 + 2, int(round(250 * Y / 2100)))
    C_w = np.zeros(X)
    C_w[X - max(1, int(round(50 * X / 2700))):] = 1e-3
    return R23, C28, C38, C_w


def rt_densities(R, C, r0, r1):
    """init_rho_cosine (mrtcg_rayleigh_taylor.cpp:182-210) for global rows [r0, r1)"""
    s = R / 2.0 - 0.1 * C * np.cos(2.0 * 3.141592 * np.arange(C) / C)
    below = np.arange(r0, r1)[:, None] < s[None, :]
    return RED["rho_0"] * below.astype(np.float64), BLUE["rho_0"] * (~below).astype(np.float64)


def droplet_densities(Ln, radius, r0, r1):
    """init_rho (rk_static_droplet_test.cpp:363-396) for global rows [r0, r1)"""
    c = Ln / 2.0
    s = np.sqrt((np.arange(r0, r1)[:, None] - c) ** 2 + (np.arange(Ln)[None, :] - c) ** 2)
    sg = 1.0 / (1.0 + np.exp(-2.0 * (s - radius)))
    return RK_RED["rho_0"] * (1.0 - sg), RK_BLUE["rho_0"] * sg


def workload_config(args, n):
    """the `config` object of both arms' lines (identical for one command line)"""
    wl = WORKLOADS[args.workload]
    gb = args.X * args.Y * 72.0 * wl["nlat"] / 1e9
    return {
        "workload": f"{wl['what']}, {args.X}x{args.Y} nodes per GPU",
        "grid_per_gpu": [args.X, args.Y], "global_grid": [args.X * n, args.Y], "decomposition": f"{n} slab(s) along axis 0",
        "l2": f"inputs larger than L2 (2 x {gb:.1f} GB of populations per GPU), no flush needed" if gb > 0.5 else
              f"populations per GPU: 2 x {gb * 1e3:.0f} MB (fits the 126 MB L2 when below that: reported as such)",
        "reference_driver": wl["driver"],
        "cpu_sample": f"CPU arms (cpu_baseline, --impl reference) time a {args.cpu_sample}x{args.cpu_sample} crop of this workload, not the full grid",
    }


# ---------------------------------------------------------------------------------------------
# CPU arms
# ---------------------------------------------------------------------------------------------
def cpu_reference_mlups(workload, edge, warmup, steps, threads=0):
    """The reference's own CPU implementation (oracle/_ref: unmodified sources on CPU libtorch) where the harness exposes
    the workload's loop; the plain-C oracle port otherwise.  `threads` host threads (0 = all this process may use), set
    EXPLICITLY on both libraries: a launcher's OMP_NUM_THREADS=1 (torch.distributed.run exports it) must not shrink the
    baseline.  Nothing here loads the product library.
    Returns (MLUPS, seconds per step, kind, cores, sample description)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib

    threads = threads or host_threads()
    if workload == "mrtcg_rt_weak":
        workload = "mrtcg_rt"
    omega, u_lb = reference_lattice_parameters()
    if oracle_lib.have_ref():
        oracle_lib.Ref().lib.ref_set_num_threads(threads)
    port_cores = oracle_lib.Oracle().num_threads(threads)  # the port's loops are OpenMP-parallel (oracle/Makefile: -fopenmp when available)

    def timed(step_fn):
        for _ in range(warmup):
            step_fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            step_fn()
        return (time.perf_counter() - t0) / max(steps, 1)

    if workload == "cylinder":
        xs, ys = cylinder_markers(edge, edge)
        desc = f"{edge}x{edge} crop of the cylinder workload"
        if oracle_lib.have_ref():
            ref = oracle_lib.Ref()
            with tempfile.TemporaryDirectory() as td:
                path = os.path.join(td, "boundary.toml")
                write_markers_toml(path, xs, ys)
                sec, _ = ref.cylinder_loop(edge, edge, omega, u_lb, path, warmup, steps)
            return edge * edge / sec / 1e6, sec, "reference", ref.num_threads(), desc
        orc = oracle_lib.Oracle()
        ib = orc.ibm_create(xs, ys)
        u = np.zeros((edge, edge, 2)); u[..., 0] = u_lb
        rho = np.ones((edge, edge, 1))
        f = orc.incomp_equilibrium(u, rho)
        sec = timed(lambda: orc.cylinder_step(f, u, rho, omega, u_lb, ib))
        orc.ibm_destroy(ib)
        return edge * edge / sec / 1e6, sec, "port", port_cores, desc

    if workload == "cylinder_bb":
        # collide + stream through the reference's own solver:: operators (oracle/_ref) where they compiled, the port
        # otherwise; the bounce-back links are the driver-style slice assignments, done here with a mask per direction
        have = oracle_lib.have_ref()
        ops = oracle_lib.Ref() if have else oracle_lib.Oracle()
        solid = cylinder_solid(edge, edge, edge)
        opp = (0, 3, 4, 1, 2, 7, 8, 5, 6)
        cuts = [(q, solid != np.roll(solid, (int(CX9[q]), int(CY9[q])), axis=(0, 1))) for q in range(1, 9)]
        u = np.zeros((edge, edge, 2)); u[..., 0] = u_lb
        state = [ops.incomp_equilibrium(u, np.ones((edge, edge, 1)))]

        def bb_step():
            f = state[0]
            rho = ops.calc_rho(f)
            coll = ops.collision(f, ops.equilibrium(ops.calc_u(f, rho), rho), omega)
            adve = ops.advect(coll)
            for q, cut in cuts:
                adve[cut, q] = coll[cut, opp[q]]
            state[0] = adve

        sec = timed(bb_step)
        return (edge * edge / sec / 1e6, sec, "reference" if have else "port", ops.num_threads() if have else port_cores,
                f"{edge}x{edge} crop of the cylinder_bb workload (solver:: operators + bounce-back links; inlet/outlet rows left out)")

    if workload == "kbc_shear" and oracle_lib.have_ref():
        # the reference's own ulbm::d2q9::kbc object stepped like test/ulbm_double_shear_flow.cpp does (oracle/ref_harness.cpp)
        ref = oracle_lib.Ref()
        r = np.arange(edge)[:, None] + 0.0 * np.arange(edge)[None, :]
        c = np.arange(edge)[None, :] + 0.0 * np.arange(edge)[:, None]
        u = np.zeros((edge, edge, 2))
        u[..., 0] = 0.02 * np.tanh(80.0 * (0.25 * edge - np.abs(c - 0.5 * edge)))
        u[..., 1] = 0.02 * 0.05 * np.sin(6.2832 * (r + 0.25 * edge) / edge)
        m0 = np.ones((edge, edge))
        f = ref.kbc_equilibrium(m0, u)
        s2 = 1.0 / (0.5 + 3.0 * 1.70766666e-4)
        ref.kbc_run(f, m0, u, s2, max(warmup, 1))
        t0 = time.perf_counter()
        ref.kbc_run(f, m0, u, s2, steps)
        sec = (time.perf_counter() - t0) / max(steps, 1)
        return edge * edge / sec / 1e6, sec, "reference", ref.num_threads(), f"{edge}x{edge} crop of the kbc_shear workload"

    if workload == "poiseuille" and oracle_lib.have_ref() and hasattr(oracle_lib.Ref().lib, "ref_poiseuille_loop"):
        ref = oracle_lib.Ref()
        om, rho_in, rho_out = channel_constants(edge, edge)
        sec, _ = ref.poiseuille_loop(edge, edge, om, rho_in, rho_out, max(warmup, 1), steps)
        return edge * edge / sec / 1e6, sec, "reference", ref.num_threads(), f"{edge}x{edge} crop of the poiseuille workload"

    orc = oracle_lib.Oracle()
    if workload == "poiseuille":
        om, rho_in, rho_out = channel_constants(edge, edge)
        u = np.zeros((edge, edge, 2)); rho = np.ones((edge, edge, 1))
        f = orc.incomp_equilibrium(u, rho)
        sec = timed(lambda: orc.poiseuille_step(f, u, rho, om, rho_in, rho_out))
    elif workload in ("sedimentation", "sedimentation_ibm"):
        R23, C28, C38, C_w = sedimentation_geometry(edge, edge)
        f, g, u, rho, Cc = orc.sedimentation_init(edge, edge, u_lb, C_w)
        ib = orc.ibm_create(*sedimentation_body(edge, edge)) if workload == "sedimentation_ibm" else None
        sec = timed(lambda: orc.sedimentation_step(f, g, u, rho, Cc, omega, u_lb, 3e-3, C_w, R23, C28, C38, ib=ib))
        if ib is not None:
            orc.ibm_destroy(ib)
    elif workload == "mrtcg_rt":
        p = oracle_lib.MrtcgParams()
        p.R, p.C = edge, edge
        p.r_rho0, p.r_alpha, p.r_nu, p.r_beta = RED["rho_0"], RED["alpha"], RED["nu"], RED["beta"]
        p.b_rho0, p.b_alpha, p.b_nu, p.b_beta = BLUE["rho_0"], BLUE["alpha"], BLUE["nu"], BLUE["beta"]
        p.sigma, p.delta = 0.1, 0.1
        p.Fg[0], p.Fg[1] = RT_FG
        p.add_force = 1
        st = orc.mrtcg_init(p, "rt")
        sec = timed(lambda: orc.mrtcg_step(p, st))
    elif workload == "csf_rt":
        p = oracle_lib.CsfParams()
        p.R, p.C = edge, edge
        p.r_rho0, p.r_alpha, p.r_nu, p.r_beta, p.r_A = RED["rho_0"], RED["alpha"], RED["nu"], RED["beta"], RED["A"]
        p.b_rho0, p.b_alpha, p.b_nu, p.b_beta, p.b_A = BLUE["rho_0"], BLUE["alpha"], BLUE["nu"], BLUE["beta"], BLUE["A"]
        p.sigma, p.delta = 0.1, 0.1
        p.Fg[0], p.Fg[1] = RT_FG
        st = orc.csf_init(p)
        sec = timed(lambda: orc.csf_step(p, st))
    elif workload == "kbc_shear":
        r = np.arange(edge)[:, None] + 0.0 * np.arange(edge)[None, :]
        c = np.arange(edge)[None, :] + 0.0 * np.arange(edge)[:, None]
        u = np.zeros((edge, edge, 2))
        u[..., 0] = 0.02 * np.tanh(80.0 * (0.25 * edge - np.abs(c - 0.5 * edge)))
        u[..., 1] = 0.02 * 0.05 * np.sin(6.2832 * (r + 0.25 * edge) / edge)
        m0 = np.ones((edge, edge))
        f = orc.kbc_equilibrium(m0, u)
        s2 = 1.0 / (0.5 + 3.0 * 1.70766666e-4)
        sec = timed(lambda: orc.kbc_step(f, m0, u, s2))
    else:  # rk_droplet
        p = oracle_lib.RkParams()
        p.L, p.radius = edge, edge / 4.0
        p.r_rho0, p.r_alpha, p.r_A, p.r_nu = RK_RED["rho_0"], RK_RED["alpha"], RK_RED["A"], RK_RED["nu"]
        p.b_rho0, p.b_alpha, p.b_A, p.b_nu = RK_BLUE["rho_0"], RK_BLUE["alpha"], RK_BLUE["A"], RK_BLUE["nu"]
        p.delta = 0.98
        st = orc.rk_init(p)
        sec = timed(lambda: orc.rk_step(p, st))
    return edge * edge / sec / 1e6, sec, "port", port_cores, f"{edge}x{edge} crop of the {workload} workload"


def cpu_baseline_leg(workload, edge, target_seconds=12.0):
    """The `cpu_baseline` object of the B200 arm's line: the CPU implementation on a crop of the workload, sized from a short
    calibration run to about `target_seconds` of CPU work (the contract asks for 10-30 s; between 5 and 400 steps)."""
    _, sec, _, _, _ = cpu_reference_mlups(workload, edge, 1, 2)
    steps = int(min(400, max(5, round(target_seconds / max(sec, 1e-6)))))
    mlups, sec, kind, cores, desc = cpu_reference_mlups(workload, edge, 1, steps)
    out = {"value": mlups, "unit": "MLUPS", "cores": cores, "kind": kind,
           "sample": f"{desc}, {steps} steps after 1 warm-up ({sec * steps:.1f} s of CPU work)", "ms_per_step": sec * 1e3}
    if kind == "reference":
        # SURVEY §8(d): the reference also on ONE host thread (at::set_num_threads(1)), a few steps of the same crop
        one, _, _, _, _ = cpu_reference_mlups(workload, edge, 1, int(min(steps, max(2, round(4.0 / max(sec * cores, 1e-6))))), threads=1)
        out["single_thread"] = {"value": one, "unit": "MLUPS", "cores": 1}
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    edge = args.cpu_sample
    mlups, sec, kind, cores, desc = cpu_reference_mlups(args.workload, edge, args.warmup, args.steps)
    sample = f"{desc}, {args.steps} steps after {args.warmup} warm-up, {cores} host threads set explicitly"
    line = {
        "impl": "reference", "metric": "MLUPS", "value": mlups, "unit": "MLUPS", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": mlups, "unit": "MLUPS", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": mlups, "unit": "MLUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi polled every 20 ms from before the warm-up; the reported clocks are those of the samples whose
    timestamps fall inside the timed region (mark_begin / mark_end)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        import datetime

        for line in self.proc.stdout:
            c = [x.strip() for x in line.split(",")]
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except Exception:
                ts = time.time()
            self.rows.append([ts] + c[1:])

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        isnum = lambda v: v.replace(".", "").isdigit()
        rows = [r for r in self.rows if len(r) > 2 and isnum(r[1])]
        t0, t1 = self.t0 or 0.0, self.t1 or 1e30
        inside = [r for r in rows if t0 <= r[0] <= t1]
        if not inside and rows:  # region shorter than the polling period: the sample nearest to it
            mid = 0.5 * (t0 + t1)
            inside = [min(rows, key=lambda r: abs(r[0] - mid))]
        sm = [float(r[1]) for r in inside]
        mx = [float(r[2]) for r in inside if isnum(r[2])]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in inside)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "samples_total": len(rows)}


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (FALLBACK_HBM_GBS of bench.py)"


def ncu_traffic_per_launch(workload, X, Y):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu capture
    (profiles/roofline_traffic.json), only when it was taken at this grid size; on the same basis as `achieved`
    (all of a step's launches of that kernel: the single-phase step has an early-rows and a bulk-rows launch)"""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
            return json.load(fh).get(f"{workload}_{X}x{Y}_bytes_per_launch")
    except Exception:
        return None


class Case:
    """One workload on one slab: builds the domain, holds the pinned host state, imports it."""

    def __init__(self, L, torch, args, rank, world, local):
        self.L, self.torch, self.args = L, torch, args
        self.rank, self.world, self.local = rank, world, local
        self.X, self.Y = args.X, args.Y
        self.Xg = args.X * world
        self.x0, self.x1 = rank * args.X, (rank + 1) * args.X
        self.label = args.workload
        self.name = "mrtcg_rt" if args.workload == "mrtcg_rt_weak" else args.workload  # same model, per-slab grid
        self.pin = getattr(args, "pin", True)
        self.omega, self.u_lb = lattice_parameters()
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        slab = dict(X=self.Xg, Y=self.Y, x0=self.x0, x1=self.x1, device=local)
        if self.name == "cylinder":
            cfg = L.default_config(model=L.MODEL_BGK, omega=self.omega, equilibrium=L.EQ_COMPRESSIBLE, force=L.FORCE_IBM, **slab)
        elif self.name == "cylinder_bb":
            cfg = L.default_config(model=L.MODEL_BGK, omega=self.omega, equilibrium=L.EQ_COMPRESSIBLE, **slab)
        elif self.name == "poiseuille":
            om, self.rho_in, self.rho_out = channel_constants(self.Xg, self.Y)
            cfg = L.default_config(model=L.MODEL_BGK, omega=om, equilibrium=L.EQ_INCOMPRESSIBLE, **slab)
        elif self.name == "kbc_shear":
            cfg = L.default_config(model=L.MODEL_KBC, omega=1.0 / (0.5 + 3.0 * 1.70766666e-4), **slab)
        elif self.name in ("sedimentation", "sedimentation_ibm"):
            cfg = L.default_config(model=L.MODEL_BGK_ADE, omega=self.omega, omega_g=self.omega, equilibrium=L.EQ_COMPRESSIBLE,
                                   w_s=3e-3, force=L.FORCE_IBM if self.name == "sedimentation_ibm" else L.FORCE_NONE, **slab)
        elif self.name == "csf_rt":
            cfg = L.default_config(model=L.MODEL_MRT_CSF, red=RED, blue=BLUE, sigma=0.1, delta=0.1, Fg=RT_FG, add_force=1, **slab)
        elif self.name == "mrtcg_rt":
            cfg = L.default_config(model=L.MODEL_MRTCG, red=RED, blue=BLUE, sigma=0.1, delta=0.1, Fg=RT_FG, add_force=1, **slab)
        else:
            cfg = L.default_config(model=L.MODEL_RK, red=RK_RED, blue=RK_BLUE, delta=0.98, **slab)
        self.d = L.Domain(cfg)

    def comm_init(self, ident):
        if self.world > 1:
            self.d.comm_init(ident, self.world, self.rank)

    def pinned(self, shape):
        """host buffer of the state: pinned for the headline (its e2e leg times the copies), pageable otherwise"""
        t = self.torch.empty(shape, dtype=self.torch.float64, pin_memory=self.pin)
        return t, t.numpy()

    def setup(self):
        d, X, Y = self.d, self.X, self.Y
        if self.name in ("cylinder", "cylinder_bb"):
            d.preset_free_stream(self.u_lb, 0.0)
            if self.name == "cylinder_bb":
                d.bc_add_solid(cylinder_solid(self.Xg, Y, self.X))  # appended to the preset's rules; the body sits in rank 0's slab
                d.bc_commit()
            else:
                xs, ys = cylinder_markers(self.X, Y)  # the body sits in rank 0's slab
                if self.rank == 0:
                    d.ibm_set_markers(xs, ys)
            # the drivers' f = incomp_equilibrium(u=(u_lb,0), rho=1) (cylinder_test.cpp:84-86): u and rho are the inputs
            self.ri_t, self.ri = self.pinned((X, Y, 1))
            self.ui_t, self.ui = self.pinned((X, Y, 2))
            self.ri[...] = 1.0
            self.ui[..., 0] = self.u_lb
            self.ui[..., 1] = 0.0
        elif self.name == "poiseuille":
            d.preset_poiseuille(self.rho_in, self.rho_out)
            self.ri_t, self.ri = self.pinned((X, Y, 1))  # incomp_equilibrium(u=0, rho=1) (horizontal_poiseuille_test.cpp:91)
            self.ui_t, self.ui = self.pinned((X, Y, 2))
            self.ri[...] = 1.0
            self.ui[...] = 0.0
        elif self.name == "kbc_shear":
            d.preset_periodic()
            self.ri_t, self.ri = self.pinned((X, Y, 1))
            self.ui_t, self.ui = self.pinned((X, Y, 2))
            self.ri[...] = 1.0   # set_initial_conditions (ulbm_double_shear_flow.cpp:44-67) on global rows [x0, x1)
            r = np.arange(self.x0, self.x1)[:, None]; c = np.arange(Y)[None, :]
            self.ui[..., 0] = 0.02 * np.tanh(80.0 * (0.25 * self.Xg - np.abs(c - 0.5 * self.Xg))) + 0.0 * r
            self.ui[..., 1] = 0.02 * 0.05 * np.sin(6.2832 * (r + 0.25 * self.Xg) / self.Xg) + 0.0 * c
        elif self.name in ("sedimentation", "sedimentation_ibm"):
            R23, C28, C38, C_w = sedimentation_geometry(self.Xg, Y)
            d.preset_sedimentation(self.u_lb, C_w, R23, C28, C38)
            if self.name == "sedimentation_ibm" and self.rank == 0:
                d.ibm_set_markers(*sedimentation_body(self.X, Y))  # the body sits in rank 0's slab
            # rectangle_sedimentation_test.cpp:84-103: u = (0, u_lb); f = incomp_eq(u, 1); g = eq(u, C), C = C_w on column 0
            self.f_t, self.f = self.pinned((X, Y, 9))
            self.g_t, self.g = self.pinned((X, Y, 9))
            self.f[...] = (1.0 + 3.0 * CY9 * self.u_lb) * W9
            cu = CY9 * self.u_lb
            geq = W9 * (1.0 + 3.0 * cu + 4.5 * cu * cu - 1.5 * self.u_lb ** 2)
            self.g[...] = 0.0
            self.g[:, 0, :] = C_w[self.x0:self.x1, None] * geq[None, :]
        else:
            (d.preset_rk if self.name == "rk_droplet" else d.preset_mrtcg)()
            self.rr_t, self.rr = self.pinned((X, Y))
            self.rb_t, self.rb = self.pinned((X, Y))
            self.u_t, self.u = self.pinned((X, Y, 2))
            self.u[...] = 0.0
            if self.name != "rk_droplet":
                self.rr[...], self.rb[...] = rt_densities(self.Xg, Y, self.x0, self.x1)
            else:
                self.rr[...], self.rb[...] = droplet_densities(self.Xg, self.Xg / 4.0, self.x0, self.x1)
        self.rho_t, self.rho = self.pinned((X, Y, 1))
        self.uo_t, self.uo = self.pinned((X, Y, 2))

    def import_state(self):
        """host -> device through the C ABI; returns the bytes copied"""
        d = self.d
        if self.name in ("cylinder", "cylinder_bb", "poiseuille"):
            d.init_equilibrium(self.ri, self.ui, self.L.EQ_INCOMPRESSIBLE)
            return self.ri.nbytes + self.ui.nbytes
        if self.name == "kbc_shear":
            d.init_equilibrium(self.ri, self.ui, self.L.EQ_KBC_FRESH)
            d.set_moments(self.ri, self.ui)
            return 2 * (self.ri.nbytes + self.ui.nbytes)
        if self.name in ("sedimentation", "sedimentation_ibm"):
            d.set_f(self.f, 0)
            d.set_f(self.g, 1)
            return self.f.nbytes + self.g.nbytes
        d.init_two_phase(self.rr, self.rb, self.u)
        return self.rr.nbytes + self.rb.nbytes + self.u.nbytes

    def export_moments(self):
        """device -> host: rho and u of the current state (what every driver snapshots)"""
        lib = self.L.load()
        dp = ctypes.POINTER(ctypes.c_double)
        rc = lib.lbm_get_moments(self.d.h, 0, self.rho.ctypes.data_as(dp), self.uo.ctypes.data_as(dp))
        if rc != 0:
            raise RuntimeError(lib.lbm_last_error().decode())
        return self.rho.nbytes + self.uo.nbytes

    def dominant_classes(self):
        L = self.L
        return [L.PROF_INTERIOR]

    def dominant_nodes(self):
        """nodes per step the dominant kernel owns (every interior-column node; the edge columns are listed nodes).  The
        single-phase step launches it twice, one after the other on the main stream: early rows, then bulk rows"""
        if self.name in ("mrtcg_rt", "rk_droplet", "csf_rt"):
            return self.X * (self.Y - 2)
        return self.X * (2 * ((self.Y - 3) // 2))


# ---------------------------------------------------------------------------------------------
# B200 arm: one measured workload
# ---------------------------------------------------------------------------------------------
class Ctx:
    """process-wide handles of the B200 arm"""

    def __init__(self, L, torch, dist, rank, world, local):
        self.L, self.torch, self.dist, self.rank, self.world, self.local = L, torch, dist, rank, world, local

    anchor = None  # the domain that holds this process's ring communicator (join_ring)

    def fresh_id(self):
        """one NCCL unique id per ring: rank 0 creates it, everyone receives it"""
        ident = [self.L.comm_unique_id() if self.rank == 0 else None]
        self.dist.broadcast_object_list(ident, src=0)
        return ident[0]

    def barrier(self, d=None):
        if d is not None:
            d.synchronize()
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()

    def max_over_ranks(self, v):
        if self.dist is None:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather_rows(self, a):
        out = [None] * self.world
        self.dist.all_gather_object(out, a)
        return np.concatenate(out, axis=0)


def join_ring(ctx, d):
    """d joins the ring of this run.  ONE NCCL communicator per process, created on a tiny anchor domain the first time and
    shared from then on (lbm_comm_share): ncclCommInitRank costs seconds on eight ranks, and this run joins a dozen domains"""
    L = ctx.L
    if getattr(ctx, "anchor", None) is None:
        X = 4 * ctx.world
        x0, x1 = L.decompose_rows(X, ctx.world, ctx.rank)
        ctx.anchor = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=8, x0=x0, x1=x1, omega=1.0, device=ctx.local))
        ctx.anchor.comm_init(ctx.fresh_id(), ctx.world, ctx.rank)
    d.comm_share(ctx.anchor)


def want_graph(mode, X, Y, world):
    """CUDA-graph replay of the step pair (lbm_use_graph): one process, no ring (the library refuses it there)"""
    if world > 1 or mode == "off":
        return False
    return mode == "on" or X * Y <= (1 << 24)


DUMP_NODES = 1 << 17  # nodes written by --dump-outputs, over all ranks: at most 2 x 9 + 3 float64 values each, 22 MB


def dump_outputs(ctx, case, out_dir):
    """What a caller of lbm_step receives after the timed steps: the populations of every lattice (lbm_get_f, `f0`, `f1`)
    and rho, u (lbm_get_moments of lattice 0), as float64 arrays of shape (nodes, components) over the slab's nodes in
    row-major order.  A slab of more than DUMP_NODES / ranks nodes contributes a fixed, seeded, sorted sample of that many
    nodes; rank 0 writes the ranks' rows one after the other."""
    d, n = case.d, case.X * case.Y
    k = DUMP_NODES // ctx.world
    idx = np.arange(n) if n <= k else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    rho, u = d.get_moments(0)
    out = {"rho": rho.reshape(n, 1)[idx], "u": u.reshape(n, 2)[idx]}
    for lat in range(WORKLOADS[case.label]["nlat"]):
        out[f"f{lat}"] = d.get_f(lat).reshape(n, 9)[idx]
    if ctx.world > 1:
        out = {name: ctx.gather_rows(a) for name, a in out.items()}
    if ctx.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for name, a in out.items():
            np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def measure(ctx, workload, X, Y, steps, warmup, *, pin, with_e2e, graph_mode, sampler=None, cpu_sample=0, dump_dir=""):
    """Device-resident MLUPS of one workload (one block of exactly K steps), the roofline of its dominant kernel and, for
    the headline, the end-to-end figure through the C ABI with pinned host buffers.  dump_dir: dump_outputs after the
    timed block."""
    import types

    L, rank, world = ctx.L, ctx.rank, ctx.world
    wl = WORKLOADS[workload]
    a = types.SimpleNamespace(workload=workload, X=X, Y=Y, pin=pin, gpus=world, cpu_sample=cpu_sample or wl["cpu_sample"])
    case = Case(L, ctx.torch, a, rank, world, ctx.local)
    d = case.d
    if world > 1:
        join_ring(ctx, d)
    case.setup()
    if world > 1:
        d.comm_check()  # every rank's setup agrees (grid, model, marker lists of bodies across cuts) or LBM_ERR_COMM — not a hang
    case.import_state()
    graph = want_graph(graph_mode, X, Y, world)
    # W warm-up steps in all; with the graph the last 4 of them reach the steady state and capture the pair (so at least 4)
    d.step(max(warmup - 4, 0) if graph else warmup)
    if graph:
        d.use_graph(True)
        d.step(4)
    ctx.barrier(d)

    # ---- device-resident timed region: exactly K steps in one block, CUDA events on the domain's stream
    d.profile_enable(not graph)
    launches0 = d.kernel_launches()
    if sampler is not None:
        sampler.mark_begin()
    ctx.barrier(d)
    d.step(steps)
    d.synchronize()
    ms = ctx.max_over_ranks(d.last_step_ms())
    ctx.barrier(d)
    if sampler is not None:
        sampler.mark_end()
    launches = d.kernel_launches() - launches0
    prof_steps = steps
    if dump_dir:
        dump_outputs(ctx, case, dump_dir)
    if graph:
        # the graph replays without per-kernel events: the dominant kernel's duration comes from one more K-step block of
        # plain launches of the same kernel (same grid, same launch configuration), right after the timed block
        d.use_graph(False)
        d.profile_enable(True)
        d.step(steps)
        d.synchronize()
        prof_steps = steps
    names = [("interior", L.PROF_INTERIOR), ("early_rows", L.PROF_EARLY), ("boundary", L.PROF_BOUNDARY), ("fixup", L.PROF_FIXUP),
             ("ghost", L.PROF_GHOST), ("ibm", L.PROF_IBM), ("moments", L.PROF_MOMENTS)]
    prof = {n: d.profile_read(c) for n, c in names}
    dom_ms, dom_n = prof["interior"][0] + prof["early_rows"][0], prof["interior"][1] + prof["early_rows"][1]  # both launches of the kernel
    d.profile_enable(False)
    mlups = (case.Xg * case.Y) * steps / (ms * 1e-3) / 1e6

    # ---- end to end through the C ABI with host buffers.  A user's loop: import the fields (H2D from pinned host), K steps,
    #      snapshot rho, u (D2H into pinned host).  Two measurements of the same traffic:
    #        blocking  : lbm_get_moments returns when the copy is done (what round 1 reported) — median of 3 blocks
    #        streaming : lbm_snapshot_async stages rho, u on the device and copies them on the library's copy stream while the
    #                    next block's import and steps run (PCIe is full duplex), lbm_snapshot_wait at the very end — five
    #                    consecutive blocks timed as one region, every byte moved and waited for inside it.  This is how the
    #                    drivers of this repo snapshot (drivers/common.hpp), and it is the `e2e.value` of the line.
    e2e = None
    if with_e2e:
        runs = []
        for _ in range(3):
            ctx.barrier(d)
            t0 = time.perf_counter()
            h2d = case.import_state()
            t1 = time.perf_counter()
            d.step(steps)
            d2h = case.export_moments()
            d.synchronize()
            t2 = time.perf_counter()
            runs.append((ctx.max_over_ranks(t2 - t0), t1 - t0, t2 - t1))
        sec_blocking, imp, rest = sorted(runs)[1]
        R = 5
        ctx.barrier(d)
        t0 = time.perf_counter()
        for _ in range(R):
            case.import_state()
            d.step(steps)
            d.snapshot_async(rho=case.rho, u=case.uo)
        d.snapshot_wait()
        d.synchronize()
        sec_stream = ctx.max_over_ranks(time.perf_counter() - t0) / R
        nodes = case.Xg * case.Y
        e2e = {"value": nodes * steps / sec_stream / 1e6, "unit": "MLUPS",
               "h2d_bytes_per_step": h2d / steps, "d2h_bytes_per_step": d2h / steps,
               "what": f"per block: initial fields from pinned host (the drivers' u, rho -> equilibrium; populations for the ADE / "
                       f"two-phase imports) + lbm_step({steps}) + rho, u to pinned host through lbm_snapshot_async; {R} consecutive "
                       "blocks timed as one region that ends after lbm_snapshot_wait (the snapshot's copy overlaps the next block's "
                       "import and steps), per rank",
               "seconds_per_block": sec_stream,
               "blocking": {"value": nodes * steps / sec_blocking / 1e6, "unit": "MLUPS", "seconds": sec_blocking, "import_seconds": imp,
                            "steps_and_export_seconds": rest,
                            "what": "the same block with lbm_get_moments (returns when the copy is done), median of 3"},
               "rho_mean": float(case.rho_t.mean())}

    peak, peak_src = measured_hbm_peak()
    B = wl["bytes"]
    nodes_per_step = case.dominant_nodes()
    achieved = B * nodes_per_step * prof_steps / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else None
    per_gpu = mlups / world
    kernel = wl["kernel"]
    if case.name == "csf_rt" and os.environ.get("LBM_CSF_FUSED", CSF_FUSED_DEFAULT) != CSF_FUSED_DEFAULT:
        kernel = "k_csf_collide_ring<PULL> (LBM_CSF_FUSED=0: three passes)"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak if achieved else None,
                "traffic": ncu_traffic_per_launch(case.name, X, Y),
                "kernel": kernel, "bytes_per_node": B, "algorithmic_bytes_per_step": B * nodes_per_step,
                "launches_per_step": dom_n / prof_steps if prof_steps else 0, "kernel_ms_per_step": dom_ms / prof_steps,
                "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0 if achieved else None,
                "whole_step_frac_per_gpu": B * per_gpu * 1e6 / 1e9 / peak,
                "whole_step_frac_per_gpu_of_nominal_8TBs": B * per_gpu * 1e6 / 1e9 / 8000.0,
                "share_of_step": (dom_ms / prof_steps) / (ms / steps),
                "other_spans_ms_per_step": {k: v[0] / prof_steps for k, v in prof.items() if v[1] and k not in ("interior", "early_rows")},
                "early_rows_ms_per_step": prof["early_rows"][0] / prof_steps,
                "timed_in": ("one more K-step block of plain launches after the timed block (that one replays a CUDA graph)" if graph
                             else "the timed block itself (CUDA events around every launch of the kernel, rank 0)"),
                "note": f"achieved = {B:.0f} B x nodes the dominant kernel owns per step / summed duration of its launches (single-phase "
                        "family: early rows then bulk rows, one after the other); listed nodes, stages, ghost rows and the IBM "
                        "pre-pass run on a side stream under the bulk launch"}
    out = {"value": mlups, "ms_per_step": ms / steps, "steps": steps, "blocks": 1, "block_ms": [round(ms, 4)],
           "cuda_graph": graph, "grid_per_gpu": [X, Y], "global_grid": [case.Xg, Y], "gpu_launches": launches, "roofline": roofline,
           "e2e": e2e, "what": wl["what"], "reference_driver": wl["driver"]}
    d.close()
    return out


# ---------------------------------------------------------------------------------------------
# B200 arm, N > 1: the ring against the monolithic run, on this ring, before anything is timed
# ---------------------------------------------------------------------------------------------
def ring_parity(ctx):
    """Every model family on a small grid over the ring of `world` ranks (lbm_comm_init: NCCL send/recv ghost rows, moment
    and normal halos, pressure packets, an immersed body across every cut) against the monolithic domain on rank 0's GPU.
    No oracle here: slabs must reproduce the single-GPU run, which the -m gpu tests tie to the oracle.  Returns on rank 0
    {case: "bit_exact" | relative error}; a rank that waits for a message nobody sends ends the process after 300 s."""
    L, rank, world, local = ctx.L, ctx.rank, ctx.world, ctx.local
    t_start = time.perf_counter()
    dog = threading.Timer(300.0, lambda: (sys.stderr.write("bench.py: ring_parity did not finish within 300 s (a rank waits for a "
                                                           "message nobody sends)\n"), sys.stderr.flush(), os._exit(3)))
    dog.daemon = True
    dog.start()
    out = {}
    omega, u_lb = lattice_parameters()

    def verdict(pairs):
        if all(np.array_equal(a, b) for a, b in pairs):
            return "bit_exact"
        return max(float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)) for a, b in pairs)

    def run(name, make, init, nsteps, fields):
        """make(**slab) -> configured Domain (rules, markers); init(d, x0, x1) imports rows [x0, x1); fields(d) -> arrays"""
        Xg = make.X
        x0, x1 = L.decompose_rows(Xg, world, rank)
        d = make(x0=x0, x1=x1, device=local, ring=True)
        init(d, x0, x1)
        d.step(nsteps)
        got = [ctx.gather_rows(a) for a in fields(d)]
        d.close()
        if rank == 0:
            mono = make(x0=0, x1=Xg, device=local, ring=False)
            init(mono, 0, Xg)
            mono.step(nsteps)
            out[name] = verdict(list(zip(got, fields(mono))))
            mono.close()
        ctx.barrier()

    class Make:
        """domain factory: create -> (ring only) lbm_comm_init -> rules -> lbm_comm_check"""

        def __init__(self, X, cfg, rules):
            self.X, self.cfg, self.rules = X, cfg, rules

        def __call__(self, x0, x1, device, ring):
            d = L.Domain(L.default_config(X=self.X, x0=x0, x1=x1, device=device, **self.cfg))
            if ring:
                join_ring(ctx, d)
            self.rules(d)
            if ring:
                d.comm_check()
            return d

    rng = np.random.default_rng(11)
    both = lambda d: (d.get_f(0), d.get_f(1))  # noqa: E731

    # ---- Poiseuille: pressure-periodic packets cross the ring (row 0 <- row X-2, row X-1 <- row 1)
    X, Y = 8 * world + 5, 33
    om, rho_in, rho_out = channel_constants(X, Y)
    f0 = W9 * (1.0 + 0.02 * rng.standard_normal((X, Y, 9)))
    run("poiseuille", Make(X, dict(model=L.MODEL_BGK, Y=Y, omega=om, equilibrium=L.EQ_INCOMPRESSIBLE), lambda d: d.preset_poiseuille(rho_in, rho_out)),
        lambda d, a, b: d.set_f(f0[a:b]), 37, lambda d: (d.get_f(),))

    # ---- cylinder: an immersed body whose ROI rows cross every cut of the ring; ABB rows at the two global ends
    X, Y = 12 * world + 9, 77
    r = 0.5 * (X - 14)
    th = 2.0 * np.pi * np.arange(max(16, int(round(2 * np.pi * r)))) / max(16, int(round(2 * np.pi * r)))
    xs, ys = 0.5 * X + 0.31 + r * np.cos(th), 0.5 * Y + 0.17 + min(r, 30.0) * np.sin(th)
    fc = W9 * (1.0 + 3.0 * CX9 * u_lb) * (1.0 + 0.01 * rng.standard_normal((X, Y, 9)))

    def cyl_rules(d):
        d.preset_free_stream(u_lb, 0.0)
        d.ibm_set_markers(xs, ys)  # every rank gets the list: co-owners of the ROI rows share the solve

    run("cylinder_ibm_across_cuts", Make(X, dict(model=L.MODEL_BGK, Y=Y, omega=omega, equilibrium=L.EQ_COMPRESSIBLE, force=L.FORCE_IBM), cyl_rules),
        lambda d, a, b: d.set_f(fc[a:b]), 40, lambda d: (d.get_f(),))

    # ---- sedimentation: fluid + advection-diffusion lattice, rectangle walls, inlet column
    X, Y = 16 * world + 6, 64
    R23, C28, C38, C_w = sedimentation_geometry(X, Y)
    R23, C28, C38 = -max(3, X // 4), 20, 26
    fs = np.broadcast_to((1.0 + 3.0 * CY9 * u_lb) * W9, (X, Y, 9)).copy()
    cu = CY9 * u_lb
    gs = np.zeros((X, Y, 9))
    gs[:, 0, :] = C_w[:, None] * (W9 * (1.0 + 3.0 * cu + 4.5 * cu * cu - 1.5 * u_lb ** 2))[None, :]

    def sed_init(d, a, b):
        d.set_f(fs[a:b], 0)
        d.set_f(gs[a:b], 1)

    run("sedimentation_ade", Make(X, dict(model=L.MODEL_BGK_ADE, Y=Y, omega=omega, omega_g=omega, equilibrium=L.EQ_COMPRESSIBLE, w_s=3e-3),
                                  lambda d: d.preset_sedimentation(u_lb, C_w, R23, C28, C38)), sed_init, 30, both)

    # ---- KBC double shear layer, fully periodic (all nine populations wrap around the ring)
    X, Y = 8 * world + 4, 40
    rr_, cc_ = np.arange(X)[:, None] + 0.0 * np.arange(Y)[None, :], np.arange(Y)[None, :] + 0.0 * np.arange(X)[:, None]
    uk = np.zeros((X, Y, 2))
    uk[..., 0] = 0.02 * np.tanh(80.0 * (0.25 * X - np.abs(cc_ - 0.5 * X)) / X * 8.0)
    uk[..., 1] = 0.02 * 0.05 * np.sin(6.2832 * (rr_ + 0.25 * X) / X)
    ones = np.ones((X, Y, 1))

    def kbc_init(d, a, b):
        d.init_equilibrium(ones[a:b], uk[a:b], L.EQ_KBC_FRESH)
        d.set_moments(ones[a:b], uk[a:b])

    run("kbc_periodic", Make(X, dict(model=L.MODEL_KBC, Y=Y, omega=1.0 / (0.5 + 3.0 * 1.70766666e-4)), lambda d: d.preset_periodic()),
        kbc_init, 30, lambda d: (d.get_f(),))

    # ---- two-phase models: population ghost rows + two-row halos of the moment planes (CSF: and of the normal field)
    R, C = 16 * world + 6, 40
    rt = rt_densities(R, C, 0, R)
    u0 = np.zeros((R, C, 2))
    tp_init = lambda d, a, b: d.init_two_phase(rt[0][a:b], rt[1][a:b], u0[a:b])  # noqa: E731
    tp_cfg = dict(Y=C, red=RED, blue=BLUE, sigma=0.1, delta=0.1, Fg=RT_FG, add_force=1)
    run("mrtcg", Make(R, dict(model=L.MODEL_MRTCG, **tp_cfg), lambda d: d.preset_mrtcg()), tp_init, 12, both)

    def with_band_rows(rows, *case):
        """a case with LBM_TP_OVERLAP=1 and slabs that march in bands of `rows` rows (LBM_TP_RPB; both read at lbm_create): every
        slab then has edge and interior bands and lbm_step sends both halo exchanges of a two-phase step behind the interior
        bands (tp_steps_ring).  That path is off by default (over NCCL it measured slower than the in-line exchange, DESIGN
        3.3); the ring keeps it honest on every multi-GPU run"""
        keep = os.environ.get("LBM_TP_RPB")
        os.environ["LBM_TP_RPB"] = str(rows)
        os.environ["LBM_TP_OVERLAP"] = "1"
        ctx.barrier()
        run(*case)
        os.environ.pop("LBM_TP_OVERLAP", None)
        if keep is None:
            os.environ.pop("LBM_TP_RPB", None)
        else:
            os.environ["LBM_TP_RPB"] = keep
        ctx.barrier()

    with_band_rows(4, "mrtcg_halos_behind_interior_bands", Make(R, dict(model=L.MODEL_MRTCG, **tp_cfg), lambda d: d.preset_mrtcg()), tp_init, 12, both)
    csf_fields = lambda d: both(d) + (d.get_interfacial_tension(),)  # noqa: E731
    keep = os.environ.get("LBM_CSF_FUSED")
    for tag, val in (("csf_single_pass", "1"), ("csf_three_pass", "0")):
        os.environ["LBM_CSF_FUSED"] = val
        run(tag, Make(R, dict(model=L.MODEL_MRT_CSF, **tp_cfg), lambda d: d.preset_mrtcg()), tp_init, 15, csf_fields)
    if keep is None:
        os.environ.pop("LBM_CSF_FUSED", None)
    else:
        os.environ["LBM_CSF_FUSED"] = keep

    Ln = 24 * world + 6
    dr = droplet_densities(Ln, Ln / 4.0, 0, Ln)
    ur = np.zeros((Ln, Ln, 2))
    rk_init = lambda d, a, b: d.init_two_phase(dr[0][a:b], dr[1][a:b], ur[a:b])  # noqa: E731
    rk_make = Make(Ln, dict(model=L.MODEL_RK, Y=Ln, red=RK_RED, blue=RK_BLUE, delta=0.98), lambda d: d.preset_rk())
    run("rk", rk_make, rk_init, 15, both)
    with_band_rows(7, "rk_halos_behind_interior_bands", rk_make, rk_init, 15, both)

    def rk_diag(d):
        """the RK driver's diagnostic fields after three steps: max|grad| is reduced over the ring (all-to-all of scalars),
        the normal planes swap halos"""
        g = d.rk_diagnostics(5e-3)
        return tuple(g[k] for k in ("phase", "grad", "norm", "n", "K", "Fs", "kappa", "omega1", "omega2"))

    run("rk_diagnostics_ring_max", rk_make, rk_init, 3, rk_diag)

    dog.cancel()
    if rank != 0:
        return None
    bad = {k: v for k, v in out.items() if v != "bit_exact" and not (isinstance(v, float) and v < 1e-12)}
    out.update({"ranks": world, "green": not bad, "criterion": "bit_exact, or relative error below 1e-12 against the monolithic run",
                "seconds": time.perf_counter() - t_start})
    return out


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def run_b200_arm(args):
    import torch

    import lbm_b200 as L

    if args.lib:
        L.LIB_PATH = os.path.abspath(args.lib)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = Ctx(L, torch, dist, rank, world, local)

    ring = None
    if world > 1 and not args.no_ring_parity:
        ring = ring_parity(ctx)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    head = measure(ctx, args.workload, args.X, args.Y, args.steps, args.warmup, pin=True, with_e2e=not args.no_e2e,
                   graph_mode=args.graph, sampler=sampler, cpu_sample=args.cpu_sample, dump_dir=args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None

    # ---- the other configs (device-resident value + roofline), only beside the default headline
    others = {}
    if args.workload == "cylinder" and not args.no_others:
        names = [w for w in args.others.split(",") if w] or (OTHERS_N1 if world == 1 else OTHERS_RING)
        for w in names:
            wl = WORKLOADS[w]
            t0 = time.perf_counter()
            r = measure(ctx, w, wl["X"], wl["Y"], args.steps, args.warmup, pin=False, with_e2e=False, graph_mode=args.graph)
            rf = r["roofline"]
            others[w] = {"value": r["value"], "unit": "MLUPS", "ms_per_step": r["ms_per_step"], "steps": r["steps"], "blocks": r["blocks"],
                         "grid_per_gpu": r["grid_per_gpu"], "global_grid": r["global_grid"], "cuda_graph": r["cuda_graph"],
                         "gpu_launches": r["gpu_launches"], "what": r["what"], "reference_driver": r["reference_driver"],
                         "roofline": {k: rf[k] for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "kernel", "bytes_per_node",
                                                         "kernel_ms_per_step", "launches_per_step", "whole_step_frac_per_gpu",
                                                         "frac_of_nominal_8TBs", "share_of_step", "timed_in")},
                         "setup_and_run_seconds": time.perf_counter() - t0}

    # every GPU is done: ranks other than 0 leave; the CPU baseline (N = 1 only) then runs with no GPU waiting on it
    if ctx.anchor is not None:
        ctx.anchor.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_leg(args.workload, args.cpu_sample)

    line = {
        "metric": "MLUPS", "value": head["value"], "unit": "MLUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(args, world),
        "roofline": head["roofline"], "cpu_baseline": cpu_baseline, "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
        "clocks": clocks,
        "timing": {"blocks": head["blocks"], "block_ms": head["block_ms"], "reported": "one block of exactly K steps after W warm-up steps (at least 4 with the CUDA graph)",
                   "cuda_graph": head["cuda_graph"]},
        "other_workloads": others or None, "ring_parity": ring,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
