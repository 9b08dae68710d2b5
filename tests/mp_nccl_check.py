"""Multi-process check of the NCCL slab ring (run under torchrun on >= 2 GPUs):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29517 tests/mp_nccl_check.py

Every rank owns one slab; the gathered result must equal the monolithic single-GPU run bit for bit
(single-phase cases) or to 1e-12 (two-phase), and the oracle for the cylinder case."""
import os
import sys

import functools

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "lattice-boltzmann-method_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
import lbm_b200 as L  # noqa: E402


print = functools.partial(print, flush=True)  # the launcher's pipe would hold the lines back until exit


class band_rows:
    """LBM_TP_RPB and LBM_TP_OVERLAP=1 (read when a domain is created) for the domains created inside; the ranks may be
    threads of one process"""

    def __init__(self, barrier, rows):
        self.barrier, self.rows = barrier, rows

    def __enter__(self):
        self.barrier()
        self.old = os.environ.get("LBM_TP_RPB")
        os.environ["LBM_TP_RPB"] = str(self.rows)
        os.environ["LBM_TP_OVERLAP"] = "1"  # (off by default: slower than the in-line exchange over NCCL, DESIGN 3.3)
        self.barrier()

    def __exit__(self, *exc):
        self.barrier()
        os.environ.pop("LBM_TP_OVERLAP", None)
        if self.old is None:
            os.environ.pop("LBM_TP_RPB", None)
        else:
            os.environ["LBM_TP_RPB"] = self.old
        self.barrier()


def run_checks(rank, world, local, fresh_id, gather, barrier, extra=False):
    """Every check of the ring on one rank.  fresh_id() hands all ranks one new communicator id, gather(a) returns the
    row-concatenation of every rank's array, barrier() joins the ranks — torch.distributed under torchrun (main below),
    threads of one process on the emulated device (tests/cpu_emu/ring_threads.py).  Returns rank 0's list of failures.
    extra: the checks whose collectives (an all-to-all group of small sends) have only run over the stand-in so far —
    lbm_comm_check and the RK diagnostics on a ring; LBM_RING_EXTRA=1 adds them under torchrun."""
    failures = []

    # ---- Poiseuille: pressure packets cross the ring (row 0 <- row X-2)
    X, Y = 8 * world + 5, 33
    omega, rho_in, rho_out = cases.channel_constants(X, Y, 0.1)
    kw = dict(model=L.MODEL_BGK, X=X, Y=Y, omega=omega, equilibrium=L.EQ_INCOMPRESSIBLE)
    rng = np.random.default_rng(5)
    w = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
    f0 = w * (1.0 + 0.02 * rng.standard_normal((X, Y, 9)))
    x0, x1 = L.decompose_rows(X, world, rank)
    d = L.Domain(L.default_config(x0=x0, x1=x1, device=local, **kw))
    d.comm_init(fresh_id(), world, rank)
    d.preset_poiseuille(rho_in, rho_out)
    d.set_f(f0[x0:x1])
    d.step(37)
    got = gather(d.get_f())
    if rank == 0:
        mono = L.Domain(L.default_config(device=local, **kw))
        mono.preset_poiseuille(rho_in, rho_out)
        mono.set_f(f0)
        mono.step(37)
        ok = np.array_equal(got, mono.get_f())
        print(f"poiseuille ring of {world}: bit-exact vs monolithic = {ok}")
        if not ok:
            failures.append("poiseuille")
    d.close()

    # ---- the statistics record on the ring: each rank accumulates its own rows, the pressure rows on the end ranks
    d = L.Domain(L.default_config(x0=x0, x1=x1, device=local, **kw))
    d.comm_init(fresh_id(), world, rank)
    d.preset_poiseuille(rho_in, rho_out)
    d.set_f(f0[x0:x1])
    d.stats_start(2)
    d.step(37)
    n, r, u, c = d.stats()
    got = [gather(a) for a in (r, u, c)]
    if rank == 0:
        mono = L.Domain(L.default_config(device=local, **kw))
        mono.preset_poiseuille(rho_in, rho_out)
        mono.set_f(f0)
        mono.stats_start(2)
        mono.step(37)
        want = mono.stats()
        ok = n == want[0] == 19 and all(np.array_equal(a, b) for a, b in zip(got, want[1:]))
        print(f"poiseuille statistics ring of {world}: bit-exact vs monolithic = {ok}")
        if not ok:
            failures.append("poiseuille-stats")
    d.close()

    # ---- MRT colour gradient: population ghost rows + 2-row moment halos
    from oracle_lib import MrtcgParams, Oracle

    R, C = 16 * world + 6, 40
    Fg = (6.25e-6, 0.0)
    orc = Oracle()
    p = MrtcgParams()
    p.R, p.C = R, C
    p.r_rho0, p.r_alpha, p.r_nu, p.r_beta = 3.0, 0.7, 0.04, 0.7
    p.b_rho0, p.b_alpha, p.b_nu, p.b_beta = 1.0, 0.1, 0.04, -0.7
    p.sigma, p.delta = 0.1, 0.1
    p.Fg[0], p.Fg[1] = Fg
    p.add_force = 1
    st = orc.mrtcg_init(p, "rt")
    st0 = {k: np.array(st[k], copy=True) for k in ("r_rho", "b_rho", "u")}
    x0, x1 = L.decompose_rows(R, world, rank)
    d = cases.mrtcg(R, C, Fg, 1, x0=x0, x1=x1, device=local)
    d.comm_init(fresh_id(), world, rank)
    d.init_two_phase(st["r_rho"][x0:x1], st["b_rho"][x0:x1], st["u"][x0:x1])
    d.step(12)
    fr, fb = gather(d.get_f(0)), gather(d.get_f(1))
    if rank == 0:
        for _ in range(12):
            orc.mrtcg_step(p, st)
        e = max(cases.relerr(fr, st["r_adv"]), cases.relerr(fb, st["b_adv"]))
        print(f"mrtcg ring of {world}: rel err vs oracle after 12 steps = {e:.2e}")
        if not e < 1e-12:
            failures.append("mrtcg")
    d.close()
    # the same run with LBM_TP_OVERLAP=1 and bands of four rows: every slab has edge and interior bands and lbm_step sends both
    # halo exchanges behind the interior bands (tp_steps_ring; off by default) — in three calls, so that the in-line
    # prologue and the join at the end of a call are crossed twice
    with band_rows(barrier, 4):
        d = cases.mrtcg(R, C, Fg, 1, x0=x0, x1=x1, device=local)
    d.comm_init(fresh_id(), world, rank)
    d.init_two_phase(st0["r_rho"][x0:x1], st0["b_rho"][x0:x1], st0["u"][x0:x1])
    for n in (5, 1, 6):
        d.step(n)
    ok = np.array_equal(gather(d.get_f(0)), fr) and np.array_equal(gather(d.get_f(1)), fb)
    if rank == 0:
        print(f"mrtcg halos behind the interior bands, ring of {world}: bit-exact vs the in-line exchange = {ok}")
        if not ok:
            failures.append("mrtcg-overlap")
    d.close()

    # ---- Rothman-Keller droplet: 1-row moment halo of the 3x3 differences, all-9 wrap rules
    from oracle_lib import RkParams

    Ln = 24 * world + 6
    rp = RkParams()
    rp.L, rp.radius = Ln, Ln / 4.0
    rp.r_rho0, rp.r_alpha, rp.r_A, rp.r_nu = 1.2, 1.0 / 3.0, 1e-4, 0.16
    rp.b_rho0, rp.b_alpha, rp.b_A, rp.b_nu = 1.0, 0.2, 1e-4, 0.14
    rp.delta = 0.98
    rst = orc.rk_init(rp)
    x0, x1 = L.decompose_rows(Ln, world, rank)
    d = cases.rk(Ln, x0=x0, x1=x1, device=local)
    d.comm_init(fresh_id(), world, rank)
    d.set_f(rst["r_adv"][x0:x1], 0)
    d.set_f(rst["b_adv"][x0:x1], 1)
    d.step(15)
    fr, fb = gather(d.get_f(0)), gather(d.get_f(1))
    d.close()
    with band_rows(barrier, 7):  # (24 or 25 rows in three bands and a rest of three or four: the last TWO bands / the last band are edge bands)
        d = cases.rk(Ln, x0=x0, x1=x1, device=local)
    d.comm_init(fresh_id(), world, rank)
    d.set_f(rst["r_adv"][x0:x1], 0)
    d.set_f(rst["b_adv"][x0:x1], 1)
    for n in (7, 8):
        d.step(n)
    ok = np.array_equal(gather(d.get_f(0)), fr) and np.array_equal(gather(d.get_f(1)), fb)
    d.close()
    if rank == 0:
        for _ in range(15):
            orc.rk_step(rp, rst)
        e = max(cases.relerr(fr, rst["r_adv"]), cases.relerr(fb, rst["b_adv"]))
        print(f"rk ring of {world}: rel err vs oracle after 15 steps = {e:.2e}")
        if not e < 1e-12:
            failures.append("rk")
        print(f"rk halos behind the interior bands, ring of {world}: bit-exact vs the in-line exchange = {ok}")
        if not ok:
            failures.append("rk-overlap")

    # ---- continuum-surface-force variant: halos of the moment planes and of the normal field across the ring
    R, Cc = 96, 40
    x0, x1 = L.decompose_rows(R, world, rank)
    import ctypes  # noqa: F401
    from oracle_lib import CsfParams, Oracle
    p = CsfParams()
    p.R, p.C = R, Cc
    p.r_rho0, p.r_alpha, p.r_nu, p.r_beta, p.r_A = 3.0, 0.7, 0.04, 0.7, 0.5
    p.b_rho0, p.b_alpha, p.b_nu, p.b_beta, p.b_A = 1.0, 0.1, 0.04, -0.7, 0.5
    p.sigma, p.delta = 0.1, 0.1
    p.Fg[0], p.Fg[1] = 6.25e-6, 0.0
    st = Oracle().csf_init(p)
    d = cases.csf(R, Cc, x0=x0, x1=x1, device=local)
    d.comm_init(fresh_id(), world, rank)
    d.init_two_phase(st["r_rho"][x0:x1], st["b_rho"][x0:x1], st["u"][x0:x1])
    d.step(15)
    got_r, got_b = gather(d.get_f(0)), gather(d.get_f(1))
    if rank == 0:
        mono = cases.csf(R, Cc, device=local)
        mono.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
        mono.step(15)
        ok = np.array_equal(got_r, mono.get_f(0)) and np.array_equal(got_b, mono.get_f(1))
        print(f"csf ring of {world}: bit-exact vs monolithic after 15 steps = {ok}")
        if not ok:
            failures.append("csf")
    d.close()

    # ---- cylinder: small IBM body near the inlet (inside rank 0's slab on 2 and 4 ranks), ABB rows at the two global ends, specular columns
    g = cases.golden("cylinder_99x77")
    X, Y = int(g["X"]), int(g["Y"])
    omega, u_lb = float(g["omega"]), float(g["u_lb"])
    xs = 14.3 + (g["marker_x"] - g["marker_x"].mean()) * 0.3
    ys = 38.6 + (g["marker_y"] - g["marker_y"].mean()) * 0.3
    kw = dict(model=L.MODEL_BGK, X=X, Y=Y, omega=omega, equilibrium=L.EQ_COMPRESSIBLE, force=L.FORCE_IBM)
    x0, x1 = L.decompose_rows(X, world, rank)
    d = L.Domain(L.default_config(x0=x0, x1=x1, device=local, **kw))
    d.comm_init(fresh_id(), world, rank)
    d.preset_free_stream(u_lb, 0.0)
    # EVERY rank gets the marker list: a rank that owns none of the ROI rows ignores it, and on rings where the ROI
    # (rows 6..23) crosses a cut (8 ranks: 12-13 rows each) the co-owners must all know about the body — handing it to
    # rank 0 alone would leave rank 0 waiting for a partner that never posts its half of the exchange
    d.ibm_set_markers(xs, ys)
    d.set_f(g["f0"][x0:x1])
    d.step(40)
    got = gather(d.get_f())
    if rank == 0:
        mono = L.Domain(L.default_config(device=local, **kw))
        mono.preset_free_stream(u_lb, 0.0)
        mono.ibm_set_markers(xs, ys)
        mono.set_f(g["f0"])
        mono.step(40)
        ok = np.array_equal(got, mono.get_f())
        print(f"cylinder ring of {world}: bit-exact vs monolithic = {ok}")
        if not ok:
            failures.append("cylinder")
    d.close()

    # ---- the same body as shipped: its ROI rows 28..73 cross every cut of a 2-, 4- or 8-rank ring; all ranks get the markers
    xs, ys = g["marker_x"], g["marker_y"]
    d = L.Domain(L.default_config(x0=x0, x1=x1, device=local, **kw))
    d.comm_init(fresh_id(), world, rank)
    d.preset_free_stream(u_lb, 0.0)
    d.ibm_set_markers(xs, ys)
    d.set_f(g["f0"][x0:x1])
    d.body_force_record(capacity=40)
    d.step(40)
    got = gather(d.get_f())
    part, first = d.body_force()
    parts = gather(part[None])
    if rank == 0:
        mono = L.Domain(L.default_config(device=local, **kw))
        mono.preset_free_stream(u_lb, 0.0)
        mono.ibm_set_markers(xs, ys)
        mono.set_f(g["f0"])
        mono.body_force_record(capacity=40)
        mono.step(40)
        ok = np.array_equal(got, mono.get_f())
        print(f"cylinder across the cuts, ring of {world}: bit-exact vs monolithic = {ok}")
        if not ok:
            failures.append("cylinder-straddling")
        # each rank sums the ROI nodes on its own rows: the parts add up to the whole in another order
        F = mono.body_force()[0]
        err = float(np.abs(parts.sum(axis=0) - F).max())
        ok = first == 0 and parts.shape == (world, 40, 2) and np.abs(F).max() > 0 and err <= 1e-13 * np.abs(F).max()
        print(f"cylinder body force across the cuts, ring of {world}: parts add up to the monolithic record = {ok} ({err:.1e})")
        if not ok:
            failures.append("cylinder-body-force")
    d.close()

    if extra:
        # ---- RK diagnostics on the ring: max|grad| reduced over the ranks, halos of the moment and normal planes
        x0, x1 = L.decompose_rows(Ln, world, rank)
        rst = orc.rk_init(rp)
        d = cases.rk(Ln, x0=x0, x1=x1, device=local)
        d.comm_init(fresh_id(), world, rank)
        d.set_f(rst["r_adv"][x0:x1], 0)
        d.set_f(rst["b_adv"][x0:x1], 1)
        d.comm_check()
        worst = 0.0
        for n in range(4):
            got = d.rk_diagnostics(5e-3)
            want = orc.rk_diagnostics(rp, rst)
            for k in ("phase", "grad", "norm", "n", "K", "Fs", "kappa", "rparams", "omega1", "omega2", "omega3"):
                worst = max(worst, float(np.abs(got[k] - want[k][x0:x1]).max()) / max(float(np.abs(want[k]).max()), 1e-3))
            orc.rk_step(rp, rst)
            d.step(1)
        worst = float(gather(np.array([worst])).max())
        if rank == 0:
            print(f"rk diagnostics ring of {world}: worst scaled err vs oracle over 4 steps = {worst:.2e}")
            if not worst < 1e-12:
                failures.append("rk-diagnostics")
        d.close()

    barrier()
    return failures


def main():
    import torch
    import torch.distributed as dist

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def fresh_id():
        """one NCCL unique id per communicator: rank 0 creates it, everyone receives it"""
        ident = [L.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ident, src=0)
        return ident[0]

    def gather(a):
        out = [None] * world
        dist.all_gather_object(out, a)
        return np.concatenate(out, axis=0)

    failures = run_checks(rank, world, local, fresh_id, gather, dist.barrier, extra=os.environ.get("LBM_RING_EXTRA") == "1")
    flag = [len(failures)]
    dist.broadcast_object_list(flag, src=0)
    dist.destroy_process_group()
    sys.exit(1 if flag[0] else 0)


if __name__ == "__main__":
    main()
