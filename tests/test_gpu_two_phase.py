"""GPU parity of the colour-gradient models (MRT colour gradient, Rothman-Keller) against the CPU
oracle and the reference's golden snapshots."""
import os
import subprocess

import numpy as np
import pytest
import torch

import cases
import lbm_b200 as L
from oracle_lib import MrtcgParams, Oracle, RkParams

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def orc():
    return Oracle()


def mrtcg_params(R, C, Fg, add_force):
    p = MrtcgParams()
    p.R, p.C = R, C
    p.r_rho0, p.r_alpha, p.r_nu, p.r_beta = 3.0, 0.7, 0.04, 0.7
    p.b_rho0, p.b_alpha, p.b_nu, p.b_beta = 1.0, 0.1, 0.04, -0.7
    p.sigma, p.delta = 0.1, 0.1
    p.Fg[0], p.Fg[1] = Fg
    p.add_force = add_force
    return p


def rk_params(Ln):
    p = RkParams()
    p.L, p.radius = Ln, 25.0
    p.r_rho0, p.r_alpha, p.r_A, p.r_nu = 1.2, 1.0 / 3.0, 1e-4, 0.16
    p.b_rho0, p.b_alpha, p.b_A, p.b_nu = 1.0, 0.2, 1e-4, 0.14
    p.delta = 0.98
    return p


def check_mrtcg_against_oracle(orc, d, p, st, steps, checkpoints, tol_f, tol_m):
    d.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
    assert cases.relerr(d.get_f(0), st["r_adv"]) < 1e-15 and cases.relerr(d.get_f(1), st["b_adv"]) < 1e-15
    for n in range(1, steps + 1):
        orc.mrtcg_step(p, st)
        d.step(1)
        if n in checkpoints:
            assert cases.relerr(d.get_f(0), st["r_adv"]) < tol_f, n
            assert cases.relerr(d.get_f(1), st["b_adv"]) < tol_f, n
            rho, u = d.get_moments()
            ph, rr, rb = d.get_phase()
            assert np.abs(rho - st["rho"]).max() < tol_m and np.abs(u - st["u"]).max() < tol_m, n
            assert np.abs(rr - st["r_rho"][..., 0]).max() < tol_m and np.abs(rb - st["b_rho"][..., 0]).max() < tol_m, n


@pytest.mark.parametrize("R,C", [(64, 48), (37, 71), (16, 9)])
def test_mrtcg_rayleigh_taylor_vs_oracle(orc, R, C):
    Fg = (6.25e-6, 0.0)
    p = mrtcg_params(R, C, Fg, 1)
    st = orc.mrtcg_init(p, "rt")
    d = cases.mrtcg(R, C, Fg, 1)
    check_mrtcg_against_oracle(orc, d, p, st, 30, {1, 2, 10, 30}, 1e-12, 1e-12)


def test_mrtcg_rayleigh_taylor_golden(orc):
    """config 3 at the reference's small size: snapshots written by test/mrtcg_rayleigh_taylor.cpp"""
    g = cases.golden("mrtcg_rt_64x48")
    Fg = (6.25e-6, 0.0)
    p = mrtcg_params(64, 48, Fg, 1)
    st = orc.mrtcg_init(p, "rt")
    d = cases.mrtcg(64, 48, Fg, 1)
    d.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
    t = 0
    for k, s in enumerate(int(s) for s in g["steps"]):
        d.step(s - t)
        t = s
        rho, u = d.get_moments()
        assert np.abs(rho[..., 0] - g["rhos"][k]).max() < 1e-12, s
        assert np.abs(u[..., 0] - g["uxs"][k]).max() < 1e-12 and np.abs(u[..., 1] - g["uys"][k]).max() < 1e-12, s
        if s + 1 < g["steps"].max():
            pass
    # phase saved in snapshot s is the phase field of iteration s-1, i.e. of the state after s-1 steps
    d2 = cases.mrtcg(64, 48, Fg, 1)
    d2.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
    d2.step(9)
    ph, _, _ = d2.get_phase()
    k10 = list(g["steps"]).index(10)
    assert np.abs(ph - g["phases"][k10]).max() < 1e-12


def test_mrtcg_static_droplet_vs_oracle_and_golden(orc):
    Fg = (0.0, -6.25e-6)
    g = cases.golden("mrtcg_droplet_72x72")
    p = mrtcg_params(72, 72, Fg, 0)
    st = orc.mrtcg_init(p, "droplet")
    d = cases.mrtcg(72, 72, Fg, 0)
    # 1e-10 on fields: the recolouring term uses the DIRECTION of a noise-level gradient at the droplet
    # centre (see tests/golden/make_golden.py), so the minority density there depends on summation order
    check_mrtcg_against_oracle(orc, d, p, st, 30, {1, 2, 10, 30}, 1e-10, 1e-10)
    d = cases.mrtcg(72, 72, Fg, 0)
    st = orc.mrtcg_init(p, "droplet")
    d.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
    t = 0
    for k, s in enumerate(int(s) for s in g["steps"]):
        d.step(s - t)
        t = s
        rho, u = d.get_moments()
        assert np.abs(rho[..., 0] - g["rhos"][k]).max() < 1e-10, s
        assert np.abs(u[..., 0] - g["uxs"][k]).max() < 1e-10, s


def test_mrtcg_colour_masses_follow_the_oracle(orc):
    """The reference's own rules (same-row copy on the side columns + bounce-back rows) do not conserve
    the colour masses exactly; the drift itself must match the oracle's."""
    R, C = 96, 64
    Fg = (6.25e-6, 0.0)
    p = mrtcg_params(R, C, Fg, 1)
    st = orc.mrtcg_init(p, "rt")
    d = cases.mrtcg(R, C, Fg, 1)
    d.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
    for _ in range(40):
        orc.mrtcg_step(p, st)
    d.step(40)
    _, rr, rb = d.get_phase()
    assert abs(rr.sum() - st["r_rho"].sum()) / st["r_rho"].sum() < 1e-13
    assert abs(rb.sum() - st["b_rho"].sum()) / st["b_rho"].sum() < 1e-13


def test_rk_droplet_vs_oracle_and_golden(orc):
    """config 4 at the reference's size (L = 101)."""
    g = cases.golden("rk_droplet_101")
    p = rk_params(101)
    st = orc.rk_init(p)
    d = cases.rk(101)
    # the driver initialises from its sigmoid densities; the oracle's rk_init returns rho_k = sum(adv_k),
    # and k_tp_init rebuilds the same populations from the raw densities
    L0 = 101
    r = np.arange(L0)[:, None] - L0 / 2.0
    c = np.arange(L0)[None, :] - L0 / 2.0
    s = np.sqrt(r * r + c * c)
    sig = 1.0 / (1.0 + np.exp(-(2.0 * (s - 25.0))))
    d.init_two_phase(1.2 * (1.0 - sig), 1.0 * sig, np.zeros((L0, L0, 2)))
    assert cases.relerr(d.get_f(0), st["r_adv"]) < 1e-14 and cases.relerr(d.get_f(1), st["b_adv"]) < 1e-14
    steps = [int(v) for v in g["steps"]]
    n = 0
    for k, sstep in enumerate(steps):
        while n < sstep + 1:  # entry s of the driver's arrays is the state after iteration s
            orc.rk_step(p, st)
            d.step(1)
            n += 1
        fr, fb = d.get_f(0), d.get_f(1)
        assert cases.relerr(fr, st["r_adv"]) < 1e-12 and cases.relerr(fb, st["b_adv"]) < 1e-12, sstep
        rows = g["rows"]  # the reference driver's fields are stored on every 10th row
        assert np.abs(fr[rows] - g["r_fs"][k]).max() < 1e-12 and np.abs(fb[rows] - g["b_fs"][k]).max() < 1e-12, sstep
        rho, u = d.get_moments()
        assert np.abs(rho[rows, :, 0] - g["rho"][k]).max() < 1e-12, sstep
        assert np.abs(u[rows, :, 0] - g["ux"][k]).max() < 1e-12 and np.abs(u[rows, :, 1] - g["uy"][k]).max() < 1e-12, sstep


def test_rk_long_run_stays_on_the_oracle(orc):
    """static droplet, 1500 steps: <= 1e-9 on density / velocity / phase (north-star long-run tolerance)"""
    Ln = 64
    p = rk_params(Ln)
    p.radius = 14.0
    st = orc.rk_init(p)
    d = cases.rk(Ln)
    d.set_f(st["r_adv"], 0)
    d.set_f(st["b_adv"], 1)
    for _ in range(1500):
        orc.rk_step(p, st)
    d.step(1500)
    rho, u = d.get_moments()
    ph, rr, rb = d.get_phase()
    assert np.abs(rho[..., 0] - st["rho"]).max() < 1e-9 and np.abs(u - st["u"]).max() < 1e-9
    # oracle's phase lags one step (it is the phase used by the last collision); compare densities instead
    assert np.abs(rr - st["r_rho"]).max() < 1e-9 and np.abs(rb - st["b_rho"]).max() < 1e-9


@pytest.mark.parametrize("R,C", [(300, 400), (131, 253), (40, 127)])
def test_mrtcg_fused_kernel_many_strips_and_bands(orc, R, C):
    """sizes that give the fused kernel several column strips (124 useful columns each) and row bands"""
    Fg = (6.25e-6, 0.0)
    p = mrtcg_params(R, C, Fg, 1)
    st = orc.mrtcg_init(p, "rt")
    d = cases.mrtcg(R, C, Fg, 1)
    d.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
    for _ in range(6):
        orc.mrtcg_step(p, st)
    d.step(6)
    assert cases.relerr(d.get_f(0), st["r_adv"]) < 1e-12 and cases.relerr(d.get_f(1), st["b_adv"]) < 1e-12
    rho, u = d.get_moments()
    assert np.abs(rho - st["rho"]).max() < 1e-12 and np.abs(u - st["u"]).max() < 1e-12
    # diagnostics in the middle of a run must not disturb it
    d.step(3)
    for _ in range(3):
        orc.mrtcg_step(p, st)
    assert cases.relerr(d.get_f(0), st["r_adv"]) < 1e-12 and cases.relerr(d.get_f(1), st["b_adv"]) < 1e-12


@pytest.mark.parametrize("Ln", [260, 127])
def test_rk_fused_kernel_many_strips_and_bands(orc, Ln):
    p = rk_params(Ln)
    p.radius = Ln / 4.0
    st = orc.rk_init(p)
    d = cases.rk(Ln)
    d.set_f(st["r_adv"], 0)
    d.set_f(st["b_adv"], 1)
    for _ in range(8):
        orc.rk_step(p, st)
    d.step(8)
    assert cases.relerr(d.get_f(0), st["r_adv"]) < 1e-12 and cases.relerr(d.get_f(1), st["b_adv"]) < 1e-12
    rho, u = d.get_moments()
    assert np.abs(rho[..., 0] - st["rho"]).max() < 1e-12 and np.abs(u - st["u"]).max() < 1e-12


@pytest.mark.parametrize("R,C", [(5, 5), (6, 7), (7, 130), (9, 126), (131, 6)])
def test_mrtcg_ragged_and_tiny_grids(orc, R, C):
    """grids smaller than a band / narrower than a strip, strip edges at the domain edge, odd sizes"""
    Fg = (6.25e-6, 0.0)
    p = mrtcg_params(R, C, Fg, 1)
    st = orc.mrtcg_init(p, "rt")
    d = cases.mrtcg(R, C, Fg, 1)
    d.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
    for _ in range(7):
        orc.mrtcg_step(p, st)
    d.step(7)
    assert cases.relerr(d.get_f(0), st["r_adv"]) < 1e-12 and cases.relerr(d.get_f(1), st["b_adv"]) < 1e-12


@pytest.mark.parametrize("Ln", [5, 8, 33, 129])
def test_rk_ragged_and_tiny_grids(orc, Ln):
    p = rk_params(Ln)
    p.radius = max(1.5, Ln / 4.0)
    st = orc.rk_init(p)
    d = cases.rk(Ln)
    d.set_f(st["r_adv"], 0)
    d.set_f(st["b_adv"], 1)
    for _ in range(6):
        orc.rk_step(p, st)
    d.step(6)
    assert cases.relerr(d.get_f(0), st["r_adv"]) < 1e-12 and cases.relerr(d.get_f(1), st["b_adv"]) < 1e-12


def test_rk_diagnostic_fields_vs_oracle_and_golden(orc):
    """lbm_rk_diagnostics: the fields driver 17 snapshots at the top of every iteration (normal with the 0.1 max|grad|
    cut, curvature, interfacial tension, eta, kappa, 1/tau, the red colour's omega1/2/3), against the oracle at every
    step and against the reference driver's own nx / ny / ks / norms / fx / fy / kappas / omegas1 / omegas2 files"""
    from test_oracle_golden import rk_diag_fields

    g = cases.golden("rk_droplet_101")
    p = rk_params(101)
    st = orc.rk_init(p)
    d = cases.rk(101)
    d.set_f(st["r_adv"], 0)
    d.set_f(st["b_adv"], 1)
    steps = [int(v) for v in g["steps"]]
    for n in range(steps[-2] + 1):
        want = orc.rk_diagnostics(p, st)
        got = d.rk_diagnostics(5e-3)
        scale = {k: max(float(np.abs(v).max()), 1e-30) for k, v in want.items()}
        for k in ("phase", "grad", "norm", "n", "K", "Fs", "eta", "kappa", "rparams", "omega1", "omega2", "omega3"):
            # absolute 1e-12 on O(1) fields, relative on the small ones (Fs ~ 1e-5, omega2 ~ 1e-6)
            assert np.abs(got[k] - want[k]).max() < 1e-12 * max(scale[k], 1e-3), (n, k)
        if n in steps:
            for name, a in rk_diag_fields(got).items():
                assert np.abs(a[g["rows"]] - g[name][steps.index(n)]).max() < 1e-12, (n, name)
        orc.rk_step(p, st)
        d.step(1)
    assert cases.relerr(d.get_f(0), st["r_adv"]) < 1e-12  # asking for diagnostics between steps does not disturb the state


def test_rk_diagnostics_error_behaviour():
    d = cases.mrtcg(16, 16, (0.0, 0.0), 0)
    with pytest.raises(L.LbmError, match="LBM_MODEL_RK"):
        d.rk_diagnostics()
    slab = cases.rk(32, x0=0, x1=16)
    slab.init_two_phase(np.ones((16, 32)), np.ones((16, 32)), np.zeros((16, 32, 2)))
    with pytest.raises(L.LbmError, match="monolithic domains or the ranks"):
        slab.rk_diagnostics()  # a slab outside a ring: no way to reduce max|grad| or to swap the normal's halo


def test_rk_driver_writes_all_nineteen_reference_files(tmp_path):
    """drivers/rk_static_droplet mirrors test/rk_static_droplet_test.cpp:617-635 file for file; the diagnostic stacks
    (normal, curvature, interfacial tension, kappa, omega1/2/3) equal the reference driver's own output"""
    exe = os.path.join(ROOT, "drivers", "bin", "rk_static_droplet")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "drivers")], stdout=subprocess.DEVNULL)
    r = subprocess.run([exe, "101", "12"], cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    g = cases.golden("rk_droplet_101")
    names = {"r-fs": "r_fs", "b-fs": "b_fs", "ux": "ux", "uy": "uy", "nx": "nx", "ny": "ny", "rho": "rho", "rhon": "rhon", "ks": "ks",
             "norms": "norms", "fx": "fx", "fy": "fy", "gradx": "gradx", "grady": "grady", "rparams": "rparams", "kappas": "kappas",
             "omegas1": "omegas1", "omegas2": "omegas2", "omegas3": None}
    got = {}
    for fname, key in names.items():
        path = tmp_path / f"rk-static-droplet-{fname}.pt"
        assert path.exists(), fname
        a = list(torch.jit.load(str(path)).parameters())[0].numpy()
        assert a.shape[:2] == (101, 101) and a.shape[-1] == 12, (fname, a.shape)
        got[fname] = a
        if key is not None:
            for k, s in enumerate(int(s) for s in g["steps"]):
                if s < 12:
                    assert np.abs(a[g["rows"]][..., s] - g[key][k]).max() < 1e-12, (fname, s)
    assert np.abs(got["omegas3"] - (got["omegas1"] + got["omegas2"])).max() < 1e-15
