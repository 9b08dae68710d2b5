"""CPU: the oracle and the product's host-side parameter code against the unmodified reference library.

Where the fixtures under tests/golden hold what the reference computed (make_golden.py stored it from oracle/_ref), the
comparison runs everywhere against them; where oracle/_ref is built (make -C oracle ref REF=<checkout of the original
sources>, or build() with LBM_REFERENCE_DIR set) the same tests also compare live through oracle/ref_harness.cpp, and the
tests without stored outputs run only there."""
import os
import tomllib

import numpy as np
import pytest

import cases
import lbm_b200 as L
from oracle_lib import Oracle, Ref, have_ref

needs_ref = pytest.mark.skipif(not have_ref(), reason="oracle/_ref not built (needs the original sources)")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARAMS = os.path.join(ROOT, "configs", "parameters.toml")
TWO_PHASE = os.path.join(ROOT, "configs", "mrtcg-rayleigh-taylor-gamma3.toml")


@pytest.fixture(scope="module")
def libs():
    return Oracle(), Ref()


@pytest.mark.ref
@needs_ref
def test_granular_ops(libs):
    o, r = libs
    rng = np.random.default_rng(0)
    for X, Y in [(1, 1), (2, 3), (13, 17), (64, 40)]:
        f = rng.random((X, Y, 9)) + 0.1
        assert [np.array_equal(a, b) for a, b in zip(o.constants(), r.constants())] == [True, True]
        rho = r.calc_rho(f)
        assert np.abs(o.calc_rho(f) - rho).max() < 1e-14
        u = r.calc_u(f, rho)
        assert np.abs(o.calc_u(f, rho) - u).max() < 1e-14
        assert np.abs(o.calc_incomp_u(f) - r.calc_incomp_u(f)).max() < 1e-14
        assert np.abs(o.equilibrium(u, rho) - r.equilibrium(u, rho)).max() < 1e-14
        assert np.abs(o.incomp_equilibrium(u, rho) - r.incomp_equilibrium(u, rho)).max() < 1e-14
        fe = r.equilibrium(u, rho)
        assert np.abs(o.collision(f, fe, 1.3) - r.collision(f, fe, 1.3)).max() < 1e-14
        if X > 1 and Y > 1:
            assert np.array_equal(o.advect(f), r.advect(f))


@pytest.mark.ref
@needs_ref
def test_differential_incl_replicate_padding(libs):
    o, r = libs
    rng = np.random.default_rng(1)
    for R, C in [(5, 5), (6, 9), (31, 18)]:
        psi = rng.random((R, C))
        for a, b in zip(o.diff5(psi), r.differential(psi)):
            assert np.abs(a - b).max() < 1e-14
    # linear fields: interior derivative exactly 1 along the differentiated axis
    i, j = np.meshgrid(np.arange(12.0), np.arange(9.0), indexing="ij")
    dx, dy = o.diff5(np.ascontiguousarray(i))
    assert np.abs(dx[2:-2, :] - 1.0).max() < 1e-13 and np.abs(dy).max() < 1e-13
    dx, dy = o.diff5(np.ascontiguousarray(j))
    assert np.abs(dy[:, 2:-2] - 1.0).max() < 1e-13 and np.abs(dx).max() < 1e-13


def test_params_bit_exact(tmp_path):
    """params::lattice of the product against the reference's: omega, u and the grid the reference derived from the TOML
    files of three fixtures (make_golden.py stored them), and with oracle/_ref every field for configs/parameters.toml"""
    o = Oracle()
    for name in ("free_stream_33x22", "cylinder_99x77", "sedimentation_176x264"):
        g = cases.golden(name)
        path = tmp_path / f"{name}.toml"
        path.write_text(str(g["toml"]))
        mine = L.params_from_toml(str(path), True)
        assert (mine.X, mine.Y) == (int(g["X"]), int(g["Y"])) and mine.omega == float(g["omega"]), name
        assert "u_lb" not in g or mine.u == float(g["u_lb"]), name
        la = tomllib.loads(str(g["toml"]))["lattice"]
        op = o.params_lattice(mine.flow_rho_0, mine.flow_nu, mine.flow_u, mine.flow_l, mine.tau, mine.dx, la["x_multiplier"],
                              la["y_multiplier"])
        assert (op["X"], op["Y"]) == (mine.X, mine.Y) and op["omega"] == mine.omega and op["u"] == mine.u, name
    if not have_ref():
        return
    ref = Ref().params(PARAMS, True)
    mine = L.params_from_toml(PARAMS, True)
    for k_ref, k in [("fp_nu", "flow_nu"), ("fp_u", "flow_u"), ("fp_l", "flow_l"), ("fp_rho_0", "flow_rho_0"),
                     ("fp_Re", "flow_Re"), ("tau", "tau"), ("omega", "omega"), ("Re", "Re"), ("nu", "nu"), ("l", "l"),
                     ("dx", "dx"), ("dt", "dt"), ("T", "T"), ("u", "u"), ("X", "X"), ("Y", "Y"),
                     ("stop_time", "stop_time"), ("snapshot_period", "snapshot_period"), ("total_steps", "total_steps"),
                     ("snapshot_steps", "snapshot_steps"), ("total_snapshots", "total_snapshots")]:
        assert float(getattr(mine, k)) == float(ref[k_ref]), k
    assert (mine.X, mine.Y) == (2700, 2100)
    op = o.params_lattice(mine.flow_rho_0, mine.flow_nu, mine.flow_u, mine.flow_l, mine.tau, mine.dx, 9, 7)
    assert (op["X"], op["Y"], op["l"], op["T"]) == (mine.X, mine.Y, mine.l, mine.T)
    assert op["u"] == mine.u and op["dt"] == mine.dt and op["omega"] == mine.omega


@pytest.mark.ref
@needs_ref
def test_colour_bit_exact(libs):
    o, r = libs
    for table in ("red", "blue"):
        ref = r.colour(TWO_PHASE, table)
        mine = L.colour_from_toml(TWO_PHASE, table)
        for k in ("rho_0", "alpha", "A", "nu", "mu", "beta", "cs2", "ics2", "rlx"):
            assert float(getattr(mine, k)) == float(ref[k]), k
        assert np.array_equal(np.array(mine.phi), ref["phi"]) and np.array_equal(np.array(mine.eta), ref["eta"])
        oc = o.colour_params(mine.rho_0, mine.alpha, mine.nu)
        assert oc["cs2"] == mine.cs2 and oc["rlx"] == mine.rlx and np.array_equal(oc["phi"], ref["phi"])
        assert np.array_equal(oc["eta"], ref["eta"])


@pytest.mark.ref
@needs_ref
def test_domain_shapes(libs):
    _, r = libs
    assert r.domain_shapes(21, 33) == [(21, 33, 9)] * 3 + [(21, 33, 1), (21, 33, 2)]


def test_ibm_force(tmp_path):
    """the reference's ibm class on a seeded field around the cylinder fixture's markers (make_golden.py stored its
    force), and with oracle/_ref live on a second body"""
    o = Oracle()
    g = cases.golden("cylinder_99x77")
    path = tmp_path / "cylinder.toml"
    path.write_text("[cylinder-a]\nx = [" + ", ".join(repr(float(v)) for v in g["marker_x"]) + "]\ny = [" +
                    ", ".join(repr(float(v)) for v in g["marker_y"]) + "]\n")
    mx, my = L.markers_from_toml(str(path), "cylinder-a")
    assert np.array_equal(mx, g["marker_x"]) and np.array_equal(my, g["marker_y"])
    ib = o.ibm_create(mx, my)
    assert o.ibm_roi(ib) == tuple(int(v) for v in g["roi"])
    assert cases.relerr(o.ibm_force(ib, g["ibm_u"], g["ibm_rho"]), g["ibm_F"]) < 1e-14
    o.ibm_destroy(ib)
    if not have_ref():
        return
    r = Ref()
    th = 2 * np.pi * np.arange(57) / 57
    xs, ys = 20.3 + 7.7 * np.cos(th), 17.9 + 6.1 * np.sin(th)
    path = tmp_path / "b.toml"
    path.write_text("[body]\nx = [" + ", ".join(repr(float(v)) for v in xs) + "]\ny = [" +
                    ", ".join(repr(float(v)) for v in ys) + "]\n")
    mx, my = L.markers_from_toml(str(path), "body")
    assert np.array_equal(mx, xs) and np.array_equal(my, ys)
    rng = np.random.default_rng(5)
    X, Y = 40, 36
    u = 0.05 * rng.standard_normal((X, Y, 2)); rho = 1.0 + 0.01 * rng.standard_normal((X, Y, 1))
    roi, F = r.ibm_force(str(path), "body", u, rho)
    ib = o.ibm_create(xs, ys)
    assert o.ibm_roi(ib) == roi
    assert cases.relerr(o.ibm_force(ib, u, rho), F) < 1e-14
    o.ibm_destroy(ib)


@pytest.mark.ref
@needs_ref
def test_kbc_class_and_driver_loops(libs):
    """ulbm::d2q9::kbc (src/ulbm.cpp) through ref_kbc_run: both drivers' loop bodies, warm and cold starts"""
    o, r = libs
    R, Cc = 28, 36
    m0, u = cases.double_shear_fields(R, Cc)
    s2 = 1.0 / (0.5 + 3.0 * 1.70766666e-4)
    f_fresh = o.kbc_equilibrium(m0, u, fresh_object=True)
    assert np.array_equal(f_fresh, r.kbc_equilibrium(m0, u))  # the driver's initial state, stale ux2 / uy2 included
    for bc, pr in ((0, (1.0, 1.0)), (1, (1.0004, 1.0))):
        fo, ao, bo = f_fresh.copy(), m0.copy(), u.copy()
        fr, ar, br = f_fresh.copy(), m0.copy(), u.copy()
        for n in (1, 1, 10, 150):
            for _ in range(n):
                o.kbc_step(fo, ao, bo, s2, bc, *pr)
            r.kbc_run(fr, ar, br, s2, n, bc, *pr)
            assert cases.relerr(fo, fr) < 1e-12 and np.abs(bo - br).max() < 1e-13 and np.abs(ao - ar).max() < 1e-13, (bc, n)
    # test/ulbm_poiseuille.cpp starts from adve_f = 0 with m0 = 1, m1 = 0
    fo = np.zeros((R, Cc, 9)); ao = np.ones((R, Cc)); bo = np.zeros((R, Cc, 2))
    fr, ar, br = fo.copy(), ao.copy(), bo.copy()
    for n in (1, 4, 60):
        for _ in range(n):
            o.kbc_step(fo, ao, bo, s2, 1, 1.0004, 1.0)
        r.kbc_run(fr, ar, br, s2, n, 1, 1.0004, 1.0)
        assert np.abs(fo - fr).max() < 1e-12, n


def test_poiseuille_loop_of_the_reference_matches_the_port():
    """the C port's step lands where the reference's Poiseuille loop does: the checksum of the populations after 100 steps of
    the reference driver (the poiseuille fixture), and with oracle/_ref after 60 steps of the timed loop bench.py uses as the
    CPU arm of the poiseuille workload (oracle/ref_harness.cpp: the reference's own operators in the order of
    test/horizontal_poiseuille_test.cpp:100-153)"""
    orc = Oracle()
    H, W = 21, 21
    omega, rho_in, rho_out = cases.channel_constants(H, W, 1.030985714e-1)
    g = cases.golden("poiseuille_21x21")
    k = [int(s) for s in g["steps"]].index(100)
    f = g["f"][0].copy(); u = np.zeros((H, W, 2)); rho = np.ones((H, W, 1))
    for _ in range(100):
        orc.poiseuille_step(f, u, rho, omega, rho_in, rho_out)
    assert abs(g["f"][k].sum() - f.sum()) < 1e-11 * abs(f.sum())
    if not have_ref():
        return
    steps = 60
    _, chk = Ref().poiseuille_loop(H, W, omega, rho_in, rho_out, 0, steps)
    u = np.zeros((H, W, 2)); rho = np.ones((H, W, 1))
    f = orc.incomp_equilibrium(u, rho)
    for _ in range(steps):
        orc.poiseuille_step(f, u, rho, omega, rho_in, rho_out)
    assert abs(chk - f.sum()) < 1e-11 * abs(f.sum())
