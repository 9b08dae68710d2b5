"""lbm_body_force_record / _read / _stop: the force on one body, summed on the device once per step into a ring.

Bounce-back body (momentum exchange over the links of lbm_bc_add_solid) and immersed body (-sum of the Eulerian force field),
each slab recording the fluid on its own rows.  Checked against the momentum balance of the fluid (exact in the
discretisation), a NumPy evaluation of the definition, the immersed boundary's own force field, and for determinism and for
the absence of side effects on the step."""
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import cases
import lbm_b200 as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.environ.get("LBM_EMU") == "1"  # tests/cpu_emu: no stream capture there
gpu = pytest.mark.gpu

W9 = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
CX = np.array([0, 1, 0, -1, 0, 1, -1, -1, 1])
CY = np.array([0, 0, 1, 0, -1, 1, 1, -1, -1])


def disc(X, Y, cx, cy, r):
    return ((np.arange(X)[:, None] - cx) ** 2 + (np.arange(Y)[None, :] - cy) ** 2 <= r * r).astype(np.uint8)


def body(X, Y):
    """a disc across the middle row plus an off-grid rectangle that wraps around the periodic column edge"""
    solid = disc(X, Y, X / 2 - 0.4, Y / 3 + 0.3, min(X, Y) / 5)
    r = np.arange(X)[:, None] + 0.0 * np.arange(Y)[None, :]
    c = np.arange(Y)[None, :] + 0.0 * np.arange(X)[:, None]
    solid |= ((np.abs(r - (X / 3 + 0.35)) <= 4.2) & (np.minimum(np.abs(c - (Y - 0.6)), np.abs(c + 0.6)) <= 5.3)).astype(np.uint8)
    return solid


def near_equilibrium(X, Y, seed, ux=0.0):
    rng = np.random.default_rng(seed)
    rho = 1.0 + 0.05 * rng.standard_normal((X, Y, 1))
    return rho * W9 * (1.0 + 3.0 * CX * ux) * (1.0 + 0.05 * rng.standard_normal((X, Y, 9)))


def slabs_of(X, P, kw, setup):
    ds = []
    for r in range(P):
        x0, x1 = L.decompose_rows(X, P, r)
        d = L.Domain(L.default_config(X=X, x0=x0, x1=x1, **kw))
        setup(d)
        ds.append(d)
    if P > 1:
        for r, d in enumerate(ds):
            d.link(ds[(r - 1) % P], ds[(r + 1) % P])
    return ds


def step(ds, n=1):
    if len(ds) > 1:
        L.step_group(ds, n)
    else:
        ds[0].step(n)


def gather(ds):
    return np.concatenate([d.get_f() for d in ds], axis=0)


def links(solid):
    """counted links (n, q): n fluid, n - c_q solid (periodic), as index arrays per q"""
    fluid = solid == 0
    return {q: np.nonzero(fluid & (np.roll(solid, (CX[q], CY[q]), axis=(0, 1)) != 0)) for q in range(1, 9)}


def momentum_exchange(f_next, lk):
    """sum of 2 c_opp(q) f_adve(t+1)[n, q] over the links (bounce-back wrote f_coll(t)[n, opp q] there), and the sum of the
    magnitudes; math.fsum: exactly rounded"""
    fx, fy, mag = [], [], []
    for q, (i, j) in lk.items():
        v = 2.0 * f_next[i, j, q]
        fx.append(-CX[q] * v); fy.append(-CY[q] * v); mag.append(np.abs(v))
    cat = np.concatenate
    return np.array([math.fsum(cat(fx)), math.fsum(cat(fy))]), math.fsum(cat(mag))


MODELS = {
    "bgk-comp": dict(model=L.MODEL_BGK, equilibrium=L.EQ_COMPRESSIBLE, omega=1.7),
    "bgk-incomp": dict(model=L.MODEL_BGK, equilibrium=L.EQ_INCOMPRESSIBLE, omega=1.3),
    "kbc": dict(model=L.MODEL_KBC, omega=1.9),
}


@gpu
@pytest.mark.parametrize("slabs", [1, 2, 3])
@pytest.mark.parametrize("model", list(MODELS))
def test_momentum_balance_is_exact(model, slabs):
    """periodic box, no forcing: what the fluid loses in a step is the force on the body,
    P_fluid(t+1) - P_fluid(t) = -F(t), to 1e-12 of sum |c_q| f; the body crosses every slab cut"""
    X, Y, steps = 48, 40, 12
    solid = body(X, Y)
    ds = slabs_of(X, slabs, dict(Y=Y, **MODELS[model]), lambda d: (d.bc_clear(), d.bc_add_solid(solid), d.bc_commit()))
    f = near_equilibrium(X, Y, 3)
    for d in ds:
        d.set_f(f[d.cfg.x0:d.cfg.x1])
        d.body_force_record(solid, capacity=steps)
    fluid = solid == 0

    def momentum(g):
        g = g[fluid]
        return np.array([math.fsum((g * CX).ravel()), math.fsum((g * CY).ravel())]), math.fsum((g * (np.abs(CX) + np.abs(CY))).ravel())

    P, _ = momentum(f)
    for t in range(steps):
        step(ds)
        P1, scale = momentum(gather(ds))
        F, first = L.body_force_group(ds, 1)
        assert first == t and F.shape == (1, 2)
        assert np.all(np.abs(P1 - P + F[0]) <= 1e-12 * scale), (t, P1 - P, F[0])
        P = P1
    F, first = L.body_force_group(ds)
    assert first == 0 and len(F) == steps and np.abs(F).max() > 1e-3  # the body does take a force


@gpu
@pytest.mark.parametrize("rules", ["periodic", "cylinder_bb"])
def test_record_matches_numpy_momentum_exchange(rules):
    """1024^2 with 64 discs (125 blocks of links): every step's record equals the definition evaluated by NumPy on the
    exported state to 1e-13 of the summed magnitudes; with cylinder_bb's inlet, outlet and specular rules present too"""
    X = Y = 1024
    steps = 20
    solid = np.zeros((X, Y), dtype=np.uint8)
    for i in range(8):
        for j in range(8):
            solid |= disc(X, Y, 64 + 128 * i + 0.3, 64 + 128 * j + 0.7, 20.5 + i + 0.5 * j)
    d = L.Domain(L.default_config(X=X, Y=Y, model=L.MODEL_BGK, equilibrium=L.EQ_COMPRESSIBLE, omega=1.6))
    if rules == "periodic":
        d.preset_periodic()
    else:
        d.preset_free_stream(0.05, 0.0)
    d.bc_add_solid(solid)
    d.bc_commit()
    d.set_f(near_equilibrium(X, Y, 5, ux=0.05))
    d.body_force_record(solid, capacity=steps)
    lk = links(solid)
    assert sum(len(i) for i, _ in lk.values()) > 100 * 256
    for t in range(steps):
        d.step(1)
        want, scale = momentum_exchange(d.get_f(), lk)
        F, first = d.body_force(1)
        assert first == t
        assert np.all(np.abs(F[0] - want) <= 1e-13 * scale), (t, F[0], want)


def cylinder_case():
    g = cases.golden("cylinder_99x77")
    X, Y = int(g["X"]), int(g["Y"])
    kw = dict(model=L.MODEL_BGK, Y=Y, omega=float(g["omega"]), equilibrium=L.EQ_COMPRESSIBLE, force=L.FORCE_IBM)
    return g, X, Y, kw


@gpu
@pytest.mark.parametrize("P", [2, 3])
def test_immersed_body_record(P):
    """the record is -(sum of lbm_ibm_get_force) at every step to 1e-14 of sum |F_euler|; slabs that share the ROI across
    the cuts record parts that add up to the monolithic record within 1e-13"""
    g, X, Y, kw = cylinder_case()
    u_lb = float(g["u_lb"])
    xs, ys = g["marker_x"], g["marker_y"]
    mono = L.Domain(L.default_config(X=X, **kw))
    mono.preset_free_stream(u_lb, 0.0)
    mono.ibm_set_markers(xs, ys)
    roi = mono.ibm_roi()
    ds = slabs_of(X, P, kw, lambda d: (d.preset_free_stream(u_lb, 0.0), d.ibm_set_markers(xs, ys)))
    assert sum(1 for d in ds if d.cfg.x0 < roi[1] and roi[0] < d.cfg.x1) >= 2, "the body must cross a cut"
    mono.set_f(g["f0"])
    for d in ds:
        d.set_f(g["f0"][d.cfg.x0:d.cfg.x1])
    steps = 8
    for d in [mono] + ds:
        d.body_force_record(capacity=steps)
    scales = []
    for t in range(steps):
        mono.step(1)
        step(ds)
        Fe = mono.ibm_get_force()
        want = -np.array([math.fsum(Fe[..., 0].ravel()), math.fsum(Fe[..., 1].ravel())])
        scale = math.fsum(np.abs(Fe).ravel())
        scales.append(scale)
        F, first = mono.body_force(1)
        assert first == t and np.all(np.abs(F[0] - want) <= 1e-14 * scale), (t, F[0], want)
    mono_F, _ = mono.body_force()
    group_F, first = L.body_force_group(ds)
    assert first == 0 and np.abs(mono_F).max() > 0
    assert np.all(np.abs(group_F - mono_F) <= 1e-13 * np.array(scales)[:, None]), np.abs(group_F - mono_F).max()


def bb_domain(X=40, Y=36):
    solid = body(X, Y)
    d = L.Domain(L.default_config(X=X, Y=Y, **MODELS["bgk-comp"]))
    d.preset_free_stream(0.04, 0.0)
    d.bc_add_solid(np.pad(solid[3:-3, 4:-4], ((3, 3), (4, 4))))  # clear of the inlet / outlet / side rules
    d.bc_commit()
    d.set_f(near_equilibrium(X, Y, 7, ux=0.04))
    return d, np.pad(solid[3:-3, 4:-4], ((3, 3), (4, 4)))


def ibm_domain():
    g, X, Y, kw = cylinder_case()
    d = cases.cylinder(X, Y, kw["omega"], float(g["u_lb"]), g["marker_x"], g["marker_y"])
    d.set_f(g["f0"])
    return d, None


def run(make, plan, record=True, graph=False):
    d, solid = make()
    if graph:
        d.use_graph(True)
    if record:
        d.body_force_record(solid, capacity=64)
    for n in plan:
        d.step(n)
    F = d.body_force()[0] if record else None
    return F, d.get_f(), d.kernel_launches()


@gpu
@pytest.mark.parametrize("make", [bb_domain, ibm_domain], ids=["bounce_back", "immersed"])
def test_record_is_deterministic_and_changes_nothing(make):
    F1, f1, n1 = run(make, [20])
    F2, f2, n2 = run(make, [20])
    assert np.array_equal(F1, F2) and len(F1) == 20
    F3, f3, _ = run(make, [1] * 20)
    assert np.array_equal(F1, F3)
    _, f_off, n_off = run(make, [20], record=False)
    assert np.array_equal(f1, f_off) and np.array_equal(f3, f_off)  # the populations do not see the record
    assert n1 - n_off == 20 * 2  # two launches a step while recording ...
    d, solid = make()
    d.body_force_record(solid, capacity=4)
    d.step(3)
    d.body_force_stop()
    d0, _ = make()
    d0.step(3)
    n, n0 = d.kernel_launches(), d0.kernel_launches()
    d.step(20)
    d0.step(20)
    assert d.kernel_launches() - n == d0.kernel_launches() - n0  # ... and none once it is stopped
    assert np.array_equal(d.get_f(), d0.get_f())
    if EMU:
        return  # the emulated device has no stream capture
    Fg, fg, _ = run(make, [6, 7, 7], graph=True)  # step pairs replayed from a CUDA graph, odd remainders plain
    assert np.array_equal(Fg, F1) and np.array_equal(fg, f_off)


@gpu
def test_ring_buffer():
    d, solid = bb_domain()
    d.body_force_record(solid, capacity=30)
    d.step(12)
    full, first = d.body_force()
    assert first == 0 and len(full) == 12
    d.body_force_record(solid, capacity=5)  # a new record restarts the count
    d2, _ = bb_domain()
    d2.step(12)
    d2.body_force_record(solid, capacity=5)
    d.step(12); d2.step(12)
    F, first = d.body_force()
    assert first == 7 and len(F) == 5
    assert np.array_equal(F, d2.body_force()[0])
    F3, first3 = d.body_force(max_steps=3)
    assert first3 == 9 and np.array_equal(F3, F[2:])
    F0, first0 = d.body_force(max_steps=0)
    assert len(F0) == 0 and first0 == 12
    d.body_force_stop()
    with pytest.raises(L.LbmError) as e:
        d.body_force()
    assert e.value.status == L.ERR_INVALID and "record" in e.value.message
    d.body_force_record(solid, capacity=5)
    d.step(2)
    F, first = d.body_force()
    assert first == 0 and len(F) == 2
    ref, _ = bb_domain()
    ref.step(24)
    ref.body_force_record(solid, capacity=5)
    ref.step(2)
    assert np.array_equal(F, ref.body_force()[0])


def expect(status, fn, *args, **kw):
    with pytest.raises(L.LbmError) as e:
        fn(*args, **kw)
    assert e.value.status == status and e.value.message, e.value
    return e.value.message


@gpu
def test_errors():
    X, Y = 40, 36
    solid = body(X, Y)
    lib = L.load()
    d = L.Domain(L.default_config(X=X, Y=Y, **MODELS["bgk-comp"]))
    d.bc_clear()
    d.bc_add_solid(solid)
    assert "lbm_bc_commit" in expect(L.ERR_INVALID, d.body_force_record, solid)  # before the rules are compiled
    d.bc_commit()
    m = np.ascontiguousarray(solid)
    p = m.ctypes.data_as(L.C.POINTER(L.C.c_ubyte))
    assert lib.lbm_body_force_record(d.h, p, X - 1, Y, 8) == L.ERR_INVALID and b"global" in lib.lbm_last_error()
    assert lib.lbm_body_force_record(d.h, p, X, Y, 0) == L.ERR_INVALID
    assert "immersed" in expect(L.ERR_INVALID, d.body_force_record, None)  # no markers
    d.body_force_record(solid)
    d.bc_commit()  # recompiling the rules ends the record
    expect(L.ERR_INVALID, d.body_force)
    # a link whose population a later rule overwrites is not a bounce-back link any more
    i, j = np.argwhere((solid == 0) & (np.roll(solid, 1, axis=0) != 0))[0]
    d.bc_add(kind=L.BC_LINEAR, x_begin=int(i), x_end=int(i) + 1, y_begin=int(j), y_end=int(j) + 1, dst_q=1, src_q=3, coef=1.0, cst=1e-3)
    d.bc_commit()
    assert f"({i}, {j}, q = 1)" in expect(L.ERR_INVALID, d.body_force_record, solid)
    tp = cases.mrtcg(16, 16, (0.0, 0.0), 0)
    expect(L.ERR_UNSUPPORTED, tp.body_force_record, np.zeros((16, 16), dtype=np.uint8))
    # region force: no markers either
    r = L.Domain(L.default_config(X=X, Y=Y, force=L.FORCE_IBM, **MODELS["bgk-comp"]))
    r.preset_periodic()
    r.set_force_region(2, 6, 3, 9, 1e-3, 0.0)
    expect(L.ERR_INVALID, r.body_force_record, None)


NEW_KERNELS = ("k_body_force_links", "k_body_force_roi", "k_body_force_finish")


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")
@pytest.mark.parametrize("lib", ["liblbm_b200.so", "liblbm_b200_nofma.so"])
def test_new_kernels_do_not_spill(lib):
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
            for k in NEW_KERNELS:
                if k in name:
                    found[k] = (int(m.group(1)), int(m.group(2)), int(m.group(3)))
            name = None
    for k in NEW_KERNELS:
        assert k in found, f"{k} not in {lib}"
        reg, stack, local = found[k]
        assert stack == 0 and local == 0 and reg <= 64, (k, found[k])
