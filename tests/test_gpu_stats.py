"""lbm_stats_start / _read / _stop: time-averaged rho, u and the velocity covariance, accumulated inside the step kernels.

Every sampled step folds the moments its collision uses — what lbm_get_moments returns for the state the step starts from —
into per-node Welford accumulators.  Checked against NumPy's Welford over lbm_get_moments taken before each sampled step,
bit for bit where nothing may contract (the -fmad=false build, the emulated device), for decomposition and schedule
invariance, and for the absence of side effects on the step."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

import cases
import lbm_b200 as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.environ.get("LBM_EMU") == "1"  # tests/cpu_emu: no stream capture there, and no contraction either
# set by test_bit_exact_without_contraction for the run through liblbm_b200_nofma.so
EXACT = EMU or os.environ.get("LBM_STATS_EXACT") == "1"
gpu = pytest.mark.gpu

W9 = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
CX = np.array([0, 1, 0, -1, 0, 1, -1, -1, 1])
CY = np.array([0, 0, 1, 0, -1, 1, 1, -1, -1])


class Welford:
    """the device's update, restated: d = v - mean; mean += d * (1 / n); M_ab += d_a * (v_b - mean_b)"""

    def __init__(self):
        self.n = 0

    def add(self, rho, u):
        v = [rho[..., 0], u[..., 0], u[..., 1]]
        if self.n == 0:
            self.m = [np.zeros_like(v[0]) for _ in range(3)]
            self.M = [np.zeros_like(v[0]) for _ in range(3)]
        self.n += 1
        inv = 1.0 / self.n
        d = [v[k] - self.m[k] for k in range(3)]
        self.m = [self.m[k] + d[k] * inv for k in range(3)]
        self.M[0] = self.M[0] + d[1] * (v[1] - self.m[1])
        self.M[1] = self.M[1] + d[2] * (v[2] - self.m[2])
        self.M[2] = self.M[2] + d[1] * (v[2] - self.m[2])

    def result(self):
        return (self.n, self.m[0][..., None], np.stack(self.m[1:], axis=-1), np.stack([M / self.n for M in self.M], axis=-1))


def near_equilibrium(X, Y, seed, ux=0.0):
    rng = np.random.default_rng(seed)
    rho = 1.0 + 0.05 * rng.standard_normal((X, Y, 1))
    return rho * W9 * (1.0 + 3.0 * CX * ux) * (1.0 + 0.05 * rng.standard_normal((X, Y, 9)))


def disc(X, Y, cx, cy, r):
    return ((np.arange(X)[:, None] - cx) ** 2 + (np.arange(Y)[None, :] - cy) ** 2 <= r * r).astype(np.uint8)


# ---- the cases: make(**slab) -> domain with its state imported; `given` = the KBC moments of lbm_set_moments
def bgk(equilibrium, omega, seed):
    def make(X=40, **slab):
        Y = 36
        d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=omega, equilibrium=equilibrium, **slab))
        d.preset_periodic()
        d.set_f(near_equilibrium(X, Y, seed)[slab.get("x0", 0):slab.get("x1", X)])
        return d
    return make


def uniform_force(**slab):
    d, _ = cases.gravity(21, 21, Fg=(-3e-4, 2e-4))
    d.set_f(near_equilibrium(21, 21, 4))
    return d


def cylinder_ibm(**slab):
    g = cases.golden("cylinder_99x77")
    d = cases.cylinder(int(g["X"]), int(g["Y"]), float(g["omega"]), float(g["u_lb"]), g["marker_x"], g["marker_y"])
    d.set_f(g["f0"])
    return d


def region_force(**slab):
    X, Y = 40, 36
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=1.4, equilibrium=L.EQ_COMPRESSIBLE, force=L.FORCE_IBM))
    d.preset_periodic()
    d.set_force_region(8, 20, 5, 30, 2e-3, -1e-3)
    d.set_f(near_equilibrium(X, Y, 5))
    return d


def bb_solid(X, Y):
    return disc(X, Y, X / 2 - 0.4, Y / 2 + 0.3, min(X, Y) / 5)


def cylinder_bb(X=48, **slab):
    """cylinder_bb's rules: free stream, and a staircase body whose listed nodes sit in interior columns"""
    Y = 40
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=1.6, equilibrium=L.EQ_COMPRESSIBLE, **slab))
    d.preset_free_stream(0.05, 0.0)
    d.bc_add_solid(bb_solid(X, Y))
    d.bc_commit()
    d.set_f(near_equilibrium(X, Y, 6, ux=0.05)[slab.get("x0", 0):slab.get("x1", X)])
    return d


def poiseuille(X=21, **slab):
    d, _ = cases.poiseuille(X, 21, **slab)
    d.set_f(near_equilibrium(X, 21, 8)[slab.get("x0", 0):slab.get("x1", X)])
    return d


def kbc(**slab):
    X, Y = 32, 28
    d = cases.kbc(X, Y, 1.9)
    rho, u = cases.double_shear_fields(X, Y)
    rho = rho[..., None]
    d.init_equilibrium(rho, u, L.EQ_KBC_FRESH)
    given = (rho * 1.001, u * 0.98)  # differ from the populations' own moments: the first sample must take these
    d.set_moments(*given)
    d.given = given
    return d


def sedimentation(**slab):
    """the sedimentation rules: every row is an early row, so the early launch runs on the side stream"""
    g = cases.golden("sedimentation_176x264")
    X, Y, u_lb = int(g["X"]), int(g["Y"]), float(g["u_lb"])
    d = cases.sedimentation(X, Y, float(g["omega"]), u_lb, float(g["w_s"]), g["C_w"], g["walls"])
    f = np.broadcast_to((1.0 + 3.0 * CY * u_lb) * W9, (X, Y, 9)) * (1.0 + 0.01 * np.random.default_rng(9).standard_normal((X, Y, 9)))
    cu = CY * u_lb
    geq = W9 * (1.0 + 3.0 * cu + 4.5 * cu * cu - 1.5 * u_lb ** 2)
    gg = np.zeros((X, Y, 9))
    gg[:, 0, :] = g["C_w"][:, None] * geq[None, :]
    d.set_f(f, 0)
    d.set_f(gg, 1)
    return d


CASES = {
    "bgk-comp": bgk(L.EQ_COMPRESSIBLE, 1.7, 1),
    "bgk-incomp": bgk(L.EQ_INCOMPRESSIBLE, 1.3, 2),
    "uniform-force": uniform_force,
    "cylinder-ibm": cylinder_ibm,
    "region-force": region_force,
    "cylinder_bb": cylinder_bb,
    "poiseuille": poiseuille,
    "kbc": kbc,
    "bgk-ade": sedimentation,
}
# KBC's collision takes rho, u from its own pair sums (csrc/lbm_device.cuh, kbc_collide), in another order than
# lbm_get_moments: equal to rounding, not bit for bit
NOT_EXACT = {"kbc"}


def run_sampled(d, steps, every):
    """step `steps` times with a record of `every`, the NumPy Welford over get_moments before each sampled step"""
    ref = Welford()
    d.stats_start(every)
    for t in range(steps):
        if t % every == 0:
            given = getattr(d, "given", None)
            ref.add(*(given if (t == 0 and given is not None) else d.get_moments(0)))
        d.step(1)
    return ref.result(), d.stats()


@gpu
@pytest.mark.parametrize("every", [1, 3])
@pytest.mark.parametrize("case", list(CASES))
def test_matches_numpy_welford(case, every):
    """means within 1e-13 of max |value|, covariances within 1e-12 of max u^2; bit for bit where nothing contracts"""
    d = CASES[case]()
    steps = 10
    (n_ref, r_ref, u_ref, c_ref), (n, r, u, c) = run_sampled(d, steps, every)
    assert n == n_ref == len(range(0, steps, every))
    assert r.shape == (d.Xl, d.Y, 1) and u.shape == (d.Xl, d.Y, 2) and c.shape == (d.Xl, d.Y, 3)
    if EXACT and case not in NOT_EXACT:
        for got, want in ((r, r_ref), (u, u_ref), (c, c_ref)):
            assert np.array_equal(got, want), np.abs(got - want).max()
        return
    assert np.abs(r - r_ref).max() <= 1e-13 * np.abs(r_ref).max()
    assert np.abs(u - u_ref).max() <= 1e-13 * np.abs(u_ref).max()
    assert np.abs(c - c_ref).max() <= 1e-12 * (u_ref ** 2).max()
    assert np.abs(c_ref).max() > 0  # the flows do fluctuate


@gpu
@pytest.mark.skipif(EMU or os.environ.get("LBM_STATS_EXACT") == "1", reason="the emulated device is exact already; no recursion")
def test_bit_exact_without_contraction():
    """the cases above through liblbm_b200_nofma.so (-fmad=false), where the device's Welford must equal NumPy's exactly"""
    lib = os.path.join(L.PKG_DIR, "liblbm_b200_nofma.so")
    if not os.path.exists(lib):
        pytest.skip("liblbm_b200_nofma.so not built (python __graft_entry__.py)")
    env = dict(os.environ, LBM_TEST_LIB=lib, LBM_STATS_EXACT="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "gpu", "-p", "no:cacheprovider",
                        os.path.abspath(__file__) + "::test_matches_numpy_welford"], cwd=ROOT, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert f"{2 * len(CASES)} passed" in r.stdout, r.stdout[-2000:]


def slabs(make, X, P):
    ds = []
    for k in range(P):
        x0, x1 = L.decompose_rows(X, P, k)
        ds.append(make(X=X, x0=x0, x1=x1))
    if P > 1:
        for k, d in enumerate(ds):
            d.link(ds[(k - 1) % P], ds[(k + 1) % P])
    return ds


@gpu
@pytest.mark.parametrize("make,X", [(cylinder_bb, 48), (poiseuille, 21)], ids=["cylinder_bb", "poiseuille"])
def test_slabs_stack_to_the_monolithic_fields(make, X):
    """1, 2 and 3 linked slabs (the body and the pressure rows across the cuts), stacked along axis 0: bit for bit"""
    out = {}
    for P in (1, 2, 3):
        ds = slabs(make, X, P)
        for d in ds:
            d.stats_start(3)
        for _ in range(4):
            if P > 1:
                L.step_group(ds, 2)
            else:
                ds[0].step(2)
        parts = [d.stats() for d in ds]
        assert all(p[0] == 3 for p in parts)
        out[P] = [np.concatenate([p[k] for p in parts], axis=0) for k in (1, 2, 3)]
    for P in (2, 3):
        for got, want in zip(out[P], out[1]):
            assert np.array_equal(got, want)


def accumulate(make, plan, every=3, graph=False, record=True):
    d = make()
    if graph:
        d.use_graph(True)
    if record:
        d.stats_start(every)
    for n in plan:
        d.step(n)
    launches = d.kernel_launches()
    return (d.stats() if record else None), d.get_f(), launches


@gpu
@pytest.mark.parametrize("make", [cylinder_bb, cylinder_ibm, sedimentation], ids=["cylinder_bb", "cylinder_ibm", "sedimentation"])
def test_schedule_invariance_and_no_side_effects(make):
    """lbm_step(n), n x lbm_step(1) and CUDA graph replays give identical accumulators; the populations do not see the
    record; one launch a step while it runs and none once it stops"""
    if make is sedimentation:
        assert make().row_split()[1] == 0  # every row early: the early launch runs on the side stream
    s1, f1, n1 = accumulate(make, [17])
    s2, f2, _ = accumulate(make, [1] * 17)
    _, f_off, n_off = accumulate(make, [17], record=False)
    assert s1[0] == 6
    for a, b in zip(s1[1:], s2[1:]):
        assert np.array_equal(a, b)
    assert np.array_equal(f1, f_off) and np.array_equal(f2, f_off)
    assert n1 - n_off == 17
    if not EMU:  # the emulated device has no stream capture
        sg, fg, _ = accumulate(make, [6, 7, 4], graph=True)  # pairs replayed from a graph, odd remainders plain
        for a, b in zip(s1[1:], sg[1:]):
            assert np.array_equal(a, b)
        assert np.array_equal(fg, f_off)
    d, d0 = make(), make()
    d.stats_start(1)
    d.step(3)
    d.stats_stop()
    d0.step(3)
    n, n0 = d.kernel_launches(), d0.kernel_launches()
    d.step(5)
    d0.step(5)
    assert d.kernel_launches() - n == d0.kernel_launches() - n0
    assert np.array_equal(d.get_f(), d0.get_f())


@gpu
def test_restart_and_commit_during_a_record():
    """stats_start mid-run restarts from n = 0; an lbm_bc_commit that adds a body mid-record keeps counting, the new listed
    nodes sampled under the new rules"""
    d = cylinder_bb()
    d.stats_start(2)
    d.step(5)
    assert d.stats()[0] == 3
    d.stats_start(2)
    ref_d = cylinder_bb()
    ref_d.step(5)
    ref_d.stats_start(2)
    d.step(4)
    ref_d.step(4)
    a, b = d.stats(), ref_d.stats()
    assert a[0] == b[0] == 2
    for x, y in zip(a[1:], b[1:]):
        assert np.array_equal(x, y)

    X, Y = 48, 40
    d = cylinder_bb()
    ref = Welford()
    d.stats_start(1)
    for t in range(8):
        if t == 4:
            d.bc_add_solid(disc(X, Y, 10.2, 30.6, 4.5))
            d.bc_commit()
        ref.add(*d.get_moments(0))
        d.step(1)
    n_ref, r_ref, u_ref, c_ref = ref.result()
    n, r, u, c = d.stats()
    assert n == n_ref == 8
    assert np.abs(r - r_ref).max() <= 1e-13 * np.abs(r_ref).max()
    assert np.abs(u - u_ref).max() <= 1e-13 * np.abs(u_ref).max()
    assert np.abs(c - c_ref).max() <= 1e-12 * (u_ref ** 2).max()


def expect(status, fn, *args):
    with pytest.raises(L.LbmError) as e:
        fn(*args)
    assert e.value.status == status and e.value.message, e.value
    return e.value.message


@gpu
def test_errors():
    lib = L.load()
    d = bgk(L.EQ_COMPRESSIBLE, 1.7, 1)()
    expect(L.ERR_INVALID, d.stats_start, 0)
    expect(L.ERR_INVALID, d.stats_start, -3)
    assert "lbm_stats_start" in expect(L.ERR_INVALID, d.stats)
    expect(L.ERR_INVALID, d.stats_stop)
    d.stats_start(2)
    sentinel = np.full((d.Xl, d.Y, 3), 7.0)
    n = L.C.c_longlong(-1)
    p = sentinel.ctypes.data_as(L.dp)
    assert lib.lbm_stats_read(d.h, p, p, p, L.C.byref(n)) == 0 and n.value == 0  # before any sample
    assert np.all(sentinel == 7.0)
    assert lib.lbm_stats_read(d.h, None, None, None, None) == L.ERR_INVALID
    d.step(1)
    assert lib.lbm_stats_read(d.h, None, None, None, L.C.byref(n)) == 0 and n.value == 1
    d.stats_stop()
    expect(L.ERR_INVALID, d.stats)
    expect(L.ERR_INVALID, d.stats_stop)
    assert lib.lbm_stats_start(None, 1) == L.ERR_INVALID
    tp = cases.mrtcg(16, 16, (0.0, 0.0), 0)
    expect(L.ERR_UNSUPPORTED, tp.stats_start, 1)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
@pytest.mark.parametrize("lib", ["liblbm_b200.so", "liblbm_b200_nofma.so"])
def test_stats_kernels_do_not_spill(lib):
    """no local memory in any STATS instantiation.  The interior kernels (the step's bulk) have no stack frame either.  A
    listed-node kernel may keep the small frame that the fp64 division's slow-path calls already cost the listed-node
    kernels without a record (16 bytes at most)."""
    path = os.path.join(ROOT, "lattice-boltzmann-method_b200", lib)
    if not os.path.exists(path):
        pytest.skip(f"{lib} not built (python __graft_entry__.py)")
    out = subprocess.run(["cuobjdump", "-res-usage", path], capture_output=True, text=True, check=True).stdout
    found, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function (\S+?):", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", line)
        if m and name:
            found[name] = (int(m.group(1)), int(m.group(2)), int(m.group(3)))
            name = None
    stats = {k: v for k, v in found.items() if re.search(r"k_bgk_(interior|boundary)_statsI", k)}
    plain_boundary = [v[1] for k, v in found.items() if re.search(r"k_bgk_boundaryI", k)]
    assert len(stats) == 44, sorted(stats)  # (8 BGK + KBC + 2 ADE) x (MODE_LOCAL, MODE_PULL) x (interior, listed)
    for k, (reg, stack, local) in stats.items():
        assert local == 0, (k, reg, stack, local)
        if "k_bgk_interior_stats" in k:
            assert stack == 0, (k, reg, stack)
        else:
            assert stack <= max(plain_boundary) <= 16, (k, reg, stack)
    for k in ("k_stats_tick", "k_stats_read"):
        hit = [v for n, v in found.items() if k in n]
        assert hit and hit[0][1] == 0 and hit[0][2] == 0, (k, hit)
