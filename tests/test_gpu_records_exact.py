"""The statistics record (lbm_stats_*) and the body-force record (lbm_body_force_*) against their definitions, evaluated
exactly from the ORACLE's moments — no device getter is involved on the reference side.

Reference.  At every sampled step the oracle's step (granular calc_rho / calc_u / calc_incomp_u on its own state, or the
u, rho its driver step computes for the collision) gives the moments the collision uses.  Per node, mean = fsum(v) / n and
the population covariance cov_ab = fsum((v_a - mean_a)(v_b - mean_b)) / n, two passes, math.fsum (exactly rounded).

Tolerance (`bounds`), derived from the device's arithmetic, u = 2^-53, n samples, per quantity M = max |v|, D = the span
max v - min v over samples and nodes (it bounds every |v - mean| the recurrences meet):
  means: the device runs m_j = m_{j-1} + (v_j - m_{j-1}) * fl(1/j).  An error e_{j-1} in m_{j-1} enters m_j multiplied by
         (1 - 1/j), and step j adds at most u|m_j| + 3u|v_j - m_{j-1}|/j (the difference, the rounded 1/j, the product; a
         fused multiply-add only removes a rounding).  Unrolled, step j's error reaches m_n with weight j/n, so
         E = |m_n - mean| <= u (M (n + 1) / 2 + 3 D).
  covariances: M_ab += d_a (v_b - m_b) telescopes to the exact sum when the means are exact.  Step j adds the rounding of
         the update, u |M_j| + 2u D_a D_b <= u D_a D_b (j + 2), and the means' errors, D_a E_b + D_b E_a; over n steps and
         divided by n: u D_a D_b ((n + 1) / 2 + 3) + D_a E_b + D_b E_a (the last u for M / n).
  samples: the device's state is the oracle's up to rounding, and its collision may sum the moments in another order
         (KBC).  delta = the moments of the device's exported populations against the oracle's, measured at every sample
         (or, where the grid is too large to export every step, the project's bar for the populations, 1e-12 of max |f|),
         plus 16 u max rho / min rho for the order of the moment sums.  A mean moves by at most delta, a covariance by at
         most 2 delta_a D_b + 2 delta_b D_a + 4 delta_a delta_b.
  reference: its own roundings (the division by n, the deviations and their products), u M and 4u D_a D_b.
Each check prints the largest error next to its bound.

Body force: the device sums the links in blocks of 256 (a tree of depth 8), the finisher adds the partials with a stride of
256 and a tree of depth 8 again, so each term passes through at most 17 + ceil(nblk / 256) additions: |error| <=
(17 + ceil(nblk / 256)) u sum |terms|.

Cases: every model family the statistics record supports (test_gpu_stats.CASES' families, plus a staircase body whose
listed nodes sit at y >= 96 of a 160+-column grid, so that the early launch reads mask words past word 1 on many rows), a
4096-sample record, both records on one domain, and the records at the benched sizes (the 128 x 128 tile method of
test_gpu_bench_scale.py)."""
import math
import os

import numpy as np
import pytest

import cases
import lbm_b200 as L
from oracle_lib import Oracle
from test_gpu_bench_scale import T, assert_tiles_identical, full, tile_fields, tiled
from test_gpu_bgk import bounce_back_step
from test_gpu_body_force import links, momentum_exchange

EMU = os.environ.get("LBM_EMU") == "1"  # tests/cpu_emu: no stream capture there
U = 2.0 ** -53
STEP_BAR = 1e-12  # populations against the oracle (test_gpu_bgk, test_gpu_bench_scale)
gpu = pytest.mark.gpu

W9 = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
CX = np.array([0, 1, 0, -1, 0, 1, -1, -1, 1.0])
CY = np.array([0, 0, 1, 0, -1, 1, 1, -1, -1.0])


@pytest.fixture(scope="module")
def orc():
    return Oracle()


def disc(X, Y, cx, cy, r):
    return ((np.arange(X)[:, None] - cx) ** 2 + (np.arange(Y)[None, :] - cy) ** 2 <= r * r).astype(np.uint8)


def near_equilibrium(X, Y, seed, ux=0.0):
    rng = np.random.default_rng(seed)
    rho = 1.0 + 0.05 * rng.standard_normal((X, Y, 1))
    return rho * W9 * (1.0 + 3.0 * CX * ux) * (1.0 + 0.05 * rng.standard_normal((X, Y, 9)))


# ---- the exact reference and its bound
def exact_stats(samples):
    """samples: [(rho {X,Y}, ux {X,Y}, uy {X,Y})] -> (mean {X,Y,3}, cov {X,Y,3}: <u'u'>, <v'v'>, <u'v'>), math.fsum per node"""
    n = len(samples)
    V = np.stack([np.stack(s, axis=-1) for s in samples], axis=-1)  # {X,Y,3,n}
    shape = V.shape[:2]
    rows = V.reshape(-1, n)
    mean = (np.array([math.fsum(r) for r in rows.tolist()]) / n).reshape(shape + (3,))
    dev = V - mean[..., None]
    cov = np.empty(shape + (3,))
    for k, (a, b) in enumerate(((1, 1), (2, 2), (1, 2))):
        prod = (dev[:, :, a] * dev[:, :, b]).reshape(-1, n)
        cov[..., k] = (np.array([math.fsum(r) for r in prod.tolist()]) / n).reshape(shape)
    return mean, cov


def bounds(samples, delta):
    """the module docstring's bounds: (bound on the three means, bound on the three covariances); delta[k] = bound on
    |device moment - oracle moment| of quantity k (rho, ux, uy)"""
    n = len(samples)
    V = np.stack([np.stack(s, axis=-1) for s in samples], axis=0)  # {n,X,Y,3}
    M = np.abs(V).max(axis=(0, 1, 2))
    D = V.max(axis=0).reshape(-1, 3) - V.min(axis=0).reshape(-1, 3)
    D = D.max(axis=0)
    E = U * (M * (n + 1) / 2 + 3 * D)
    bm = E + delta + U * M
    bc = []
    for a, b in ((1, 1), (2, 2), (1, 2)):
        welford = U * D[a] * D[b] * ((n + 1) / 2 + 3) + D[a] * E[b] + D[b] * E[a] + U * D[a] * D[b]
        drift = 2 * delta[a] * D[b] + 2 * delta[b] * D[a] + 4 * delta[a] * delta[b]
        bc.append(welford + drift + 4 * U * D[a] * D[b])
    return bm, np.array(bc)


def moment_delta(f_dev, sample, comp=True, orc=None):
    """|moments of the device's populations - the oracle's sample| per quantity, plus the moment sums' own rounding"""
    rho = orc.calc_rho(np.ascontiguousarray(f_dev))
    u = orc.calc_u(np.ascontiguousarray(f_dev), rho) if comp else orc.calc_incomp_u(np.ascontiguousarray(f_dev))
    got = (rho[..., 0], u[..., 0], u[..., 1])
    order = 16 * U * sample[0].max() / sample[0].min()
    return np.array([np.abs(g - s).max() for g, s in zip(got, sample)]) + order


def check(what, stats, samples, delta):
    """the record (n, rho_mean, u_mean, u_cov) against the exact reference within its bound; prints both"""
    n, r, u, c = stats
    assert n == len(samples), (n, len(samples))
    mean, cov = exact_stats(samples)
    got = np.concatenate([r, u], axis=-1)
    bm, bc = bounds(samples, delta)
    em = np.abs(got - mean).reshape(-1, 3).max(axis=0)
    ec = np.abs(c - cov).reshape(-1, 3).max(axis=0)
    print(f"{what}: n = {n}; means max err {em.max():.2e} (bound {bm.min():.2e} .. {bm.max():.2e}); covariances max err "
          f"{ec.max():.2e} (bound {bc.min():.2e} .. {bc.max():.2e}); max |cov| {np.abs(cov).max():.2e}")
    assert np.all(em <= bm), (what, em, bm)
    assert np.all(ec <= bc), (what, ec, bc)
    assert np.abs(cov).max() > 0  # the flow does fluctuate


# ---- the families: each builder returns (domain, oracle step), the step advancing the oracle's own state by one step and
# returning the moments (rho, ux, uy) its collision used, plus whether the model's u is j / rho
def periodic_bgk(orc, eq, omega, seed, X=40, Y=36, ux=0.0):
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=omega, equilibrium=eq))
    d.preset_periodic()
    f = near_equilibrium(X, Y, seed, ux)
    d.set_f(f)
    st = {"f": f}
    comp = eq == L.EQ_COMPRESSIBLE

    def step():
        f = st["f"]
        rho = orc.calc_rho(f)
        u = orc.calc_u(f, rho) if comp else orc.calc_incomp_u(f)
        feq = orc.equilibrium(u, rho) if comp else orc.incomp_equilibrium(u, rho)
        st["f"] = orc.advect(orc.collision(f, feq, omega))
        return rho[..., 0], u[..., 0], u[..., 1]
    return d, step, comp


def uniform_force(orc):
    d, omega = cases.gravity(21, 21, Fg=(-3e-4, 2e-4))
    f = near_equilibrium(21, 21, 4)
    d.set_f(f)
    u, rho = np.zeros((21, 21, 2)), np.ones((21, 21, 1))
    Fg = np.array([-3e-4, 2e-4])

    def step():
        orc.gravity_step(f, u, rho, omega, 1.0, 1.0, Fg)  # u: the collision's u, the += Fg shift of gravity_test.cpp:143 included
        return rho[..., 0].copy(), u[..., 0].copy(), u[..., 1].copy()
    # the recorded u carries + Fg, the populations' own moments do not: the delta check adds it back
    step.shift = Fg
    return d, step, False


def cylinder_ibm(orc, request):
    """the immersed body's collision takes the plain moments of the populations: the half-force shift of the IBM's
    multi-direct forcing (lbm_ibm.cu, orc_ibm_force) only feeds the force iteration, and orc_cylinder_step leaves u, rho
    as its collision used them"""
    g = cases.golden("cylinder_99x77")
    X, Y, omega, u_lb = int(g["X"]), int(g["Y"]), float(g["omega"]), float(g["u_lb"])
    d = cases.cylinder(X, Y, omega, u_lb, g["marker_x"], g["marker_y"])
    f = g["f0"].copy()
    d.set_f(f)
    ib = orc.ibm_create(g["marker_x"], g["marker_y"])
    request.addfinalizer(lambda: orc.ibm_destroy(ib))
    u, rho = np.zeros((X, Y, 2)), np.ones((X, Y, 1))

    def step():
        orc.cylinder_step(f, u, rho, omega, u_lb, ib)
        return rho[..., 0].copy(), u[..., 0].copy(), u[..., 1].copy()
    return d, step, True


REGION = (8, 20, 5, 30, 2e-3, -1e-3)


def region_force(orc):
    """set_force_region: the Guo source with the region's constants ics2 = 3, ics4 = 9 (decompose_domain_loop.cpp:68-69),
    composed from the oracle's granular operators the way blocks_oracle.step forces block A"""
    X, Y, omega = 40, 36, 1.4
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=omega, equilibrium=L.EQ_COMPRESSIBLE, force=L.FORCE_IBM))
    d.preset_periodic()
    d.set_force_region(*REGION)
    x0, x1, y0, y1, Fx, Fy = REGION
    f = near_equilibrium(X, Y, 5)
    d.set_f(f)
    st = {"f": f}

    def step():
        f = st["f"]
        rho = orc.calc_rho(f)
        u = orc.calc_u(f, rho)
        c = f + (-omega * (f - orc.equilibrium(u, rho)))
        ur = u[x0:x1, y0:y1]
        cu = ur[..., 0:1] * CX + ur[..., 1:2] * CY
        cF = Fx * CX + Fy * CY
        uF = ur[..., 0:1] * Fx + ur[..., 1:2] * Fy
        c[x0:x1, y0:y1] += ((1.0 - 0.5 * omega) * ((3.0 + 9.0 * cu) * cF - 3.0 * uF)) * W9
        st["f"] = orc.advect(np.ascontiguousarray(c))
        return rho[..., 0], u[..., 0], u[..., 1]
    return d, step, True


def kbc(orc):
    """the first step takes the moments of lbm_set_moments (here 0.1 % / 2 % off the populations' own), every later one
    the moments orc_kbc_step leaves for the next collision"""
    X, Y, s2 = 32, 28, 1.9
    d = cases.kbc(X, Y, s2)
    rho, u = cases.double_shear_fields(X, Y)
    d.init_equilibrium(rho[..., None], u, L.EQ_KBC_FRESH)
    m0, m1 = np.ascontiguousarray(rho * 1.001), np.ascontiguousarray(u * 0.98)
    d.set_moments(m0[..., None], m1)
    f = d.get_f()  # the imported populations are the oracle's initial state too

    def step():
        sample = (m0.copy(), m1[..., 0].copy(), m1[..., 1].copy())
        orc.kbc_step(f, m0, m1, s2)
        return sample
    step.given_first = True  # the first sample is lbm_set_moments' input on both sides, not the populations' moments
    return d, step, True


def bgk_ade(orc):
    """the fluid lattice of the sedimentation driver: orc_sedimentation_step collides with the u, rho it carries from the end
    of the previous step (calc_rho / calc_u of the boundary-completed populations); the first ones are computed here"""
    g = cases.golden("sedimentation_176x264")
    X, Y, u_lb, omega, w_s = int(g["X"]), int(g["Y"]), float(g["u_lb"]), float(g["omega"]), float(g["w_s"])
    C_w, walls = g["C_w"], [int(v) for v in g["walls"]]
    d = cases.sedimentation(X, Y, omega, u_lb, w_s, C_w, walls)
    f = np.ascontiguousarray(np.broadcast_to((1.0 + 3.0 * CY * u_lb) * W9, (X, Y, 9))
                             * (1.0 + 0.01 * np.random.default_rng(9).standard_normal((X, Y, 9))))
    cu = CY * u_lb
    gg = np.zeros((X, Y, 9))
    gg[:, 0, :] = C_w[:, None] * (W9 * (1.0 + 3.0 * cu + 4.5 * cu * cu - 1.5 * u_lb ** 2))[None, :]
    d.set_f(f, 0)
    d.set_f(gg, 1)
    rho = orc.calc_rho(f)
    u = orc.calc_u(f, rho)
    Cc = orc.calc_rho(gg)

    def step():
        sample = (rho[..., 0].copy(), u[..., 0].copy(), u[..., 1].copy())
        orc.sedimentation_step(f, gg, u, rho, Cc, omega, u_lb, w_s, C_w, *walls)
        return sample
    return d, step, True


def poiseuille(orc):
    d, (omega, rho_in, rho_out) = cases.poiseuille(21, 21)
    f = near_equilibrium(21, 21, 8)
    d.set_f(f)
    u, rho = np.zeros((21, 21, 2)), np.ones((21, 21, 1))

    def step():
        orc.poiseuille_step(f, u, rho, omega, rho_in, rho_out)  # u, rho: the collision's (incompressible) moments
        return rho[..., 0].copy(), u[..., 0].copy(), u[..., 1].copy()
    return d, step, False


STAIR_X, STAIR_Y, STAIR_OMEGA = 64, 192, 1.7


def stair_solid(X=STAIR_X, Y=STAIR_Y):
    """listed nodes on 40+ rows at 96 <= y < 185: mask words 3 .. 5 of a 6-word row"""
    return disc(X, Y, 32.3, 130.6, 20.2) | disc(X, Y, 12.2, 102.4, 5.5) | disc(X, Y, 50.7, 172.1, 8.6)


def staircase(orc):
    """a staircase body under plain periodic rules, stepped by test_gpu_bgk.bounce_back_step"""
    X, Y = STAIR_X, STAIR_Y
    solid = stair_solid()
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=STAIR_OMEGA, equilibrium=L.EQ_COMPRESSIBLE))
    d.bc_clear()
    d.bc_add_solid(solid)
    d.bc_commit()
    f = near_equilibrium(X, Y, 12, ux=0.04)
    d.set_f(f)
    st = {"f": f}

    def step():
        f = st["f"]
        rho = orc.calc_rho(f)
        u = orc.calc_u(f, rho)
        st["f"] = bounce_back_step(orc, f, solid, STAIR_OMEGA)
        return rho[..., 0], u[..., 0], u[..., 1]
    return d, step, True


FAMILIES = {
    "bgk-comp": lambda orc, rq: periodic_bgk(orc, L.EQ_COMPRESSIBLE, 1.7, 1),
    "bgk-incomp": lambda orc, rq: periodic_bgk(orc, L.EQ_INCOMPRESSIBLE, 1.3, 2),
    "uniform-force": lambda orc, rq: uniform_force(orc),
    "cylinder-ibm": cylinder_ibm,
    "region-force": lambda orc, rq: region_force(orc),
    "kbc": lambda orc, rq: kbc(orc),
    "bgk-ade": lambda orc, rq: bgk_ade(orc),
    "poiseuille": lambda orc, rq: poiseuille(orc),
    "staircase": lambda orc, rq: staircase(orc),
}


def sampled_run(orc, d, step, comp, steps, every):
    """steps device steps under a record of `every`; the oracle's moments at each sampled step and delta measured there"""
    d.stats_start(every)
    samples, delta = [], np.zeros(3)
    shift = getattr(step, "shift", None)
    for t in range(steps):
        s = step()
        if t % every == 0:
            samples.append(s)
            if t > 0 or not getattr(step, "given_first", False):
                dm = s if shift is None else (s[0], s[1] - shift[0], s[2] - shift[1])
                delta = np.maximum(delta, moment_delta(d.get_f(0), dm, comp, orc))
        d.step(1)
    return samples, delta


@gpu
@pytest.mark.parametrize("every", [1, 3])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_statistics_match_the_exact_definition(orc, request, family, every):
    d, step, comp = FAMILIES[family](orc, request)
    if family == "staircase":
        assert d.row_split()[1] > 0 and STAIR_Y >= 160  # bulk rows exist: the listed rows are early rows, read through the mask
    samples, delta = sampled_run(orc, d, step, comp, 12, every)
    check(f"{family} every {every}", d.stats(), samples, delta)


@gpu
def test_a_long_record_stays_within_its_bound(orc):
    """4096 samples, every = 1, a small periodic BGK grid: Welford with a rounded 1 / n against the exact mean and covariance"""
    d, step, comp = periodic_bgk(orc, L.EQ_COMPRESSIBLE, 1.2, 21, X=16, Y=12, ux=0.05)
    samples, delta = sampled_run(orc, d, step, comp, 4096, 1)
    check("long record, 4096 samples", d.stats(), samples, delta)


# ---- both records on one domain
def stair_domain():
    X, Y = STAIR_X, STAIR_Y
    solid = stair_solid()
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=STAIR_OMEGA, equilibrium=L.EQ_COMPRESSIBLE))
    d.bc_clear()
    d.bc_add_solid(solid)
    d.bc_commit()
    d.set_f(near_equilibrium(X, Y, 12, ux=0.04))
    return d, solid


def run_records(plan, force, stats, graph=False):
    d, solid = stair_domain()
    if graph:
        d.use_graph(True)
    if force:
        d.body_force_record(solid, capacity=64)
    if stats:
        d.stats_start(3)
    for n in plan:
        d.step(n)
    launches = d.kernel_launches()  # before the reads (lbm_stats_read launches its own kernel)
    return (d.body_force()[0] if force else None), (d.stats() if stats else None), d.get_f(), launches


@gpu
def test_both_records_on_one_domain():
    """body force and statistics together (both add work to the side chain; k_stats_tick waits on ev_side after the
    body-force kernels): each record bit-identical to itself alone, the populations to a run with neither, the launch
    counts adding up; the same under CUDA graph replays"""
    plan = [17]
    F_b, S_b, f_b, n_b = run_records(plan, True, True)
    F_f, _, f_f, n_f = run_records(plan, True, False)
    _, S_s, f_s, n_s = run_records(plan, False, True)
    _, _, f_0, n_0 = run_records(plan, False, False)
    assert np.array_equal(F_b, F_f) and len(F_b) == 17 and np.abs(F_b).max() > 0
    assert S_b[0] == S_s[0] == 6 and all(np.array_equal(a, b) for a, b in zip(S_b[1:], S_s[1:]))
    for f in (f_b, f_f, f_s):
        assert np.array_equal(f, f_0)
    assert n_b - n_0 == (n_f - n_0) + (n_s - n_0) == 17 * 2 + 17
    if EMU:
        return  # the emulated device has no stream capture
    F_g, S_g, f_g, _ = run_records([6, 7, 4], True, True, graph=True)  # pairs replayed from a graph, odd remainders plain
    assert np.array_equal(F_g, F_b) and np.array_equal(f_g, f_0)
    assert S_g[0] == 6 and all(np.array_equal(a, b) for a, b in zip(S_g[1:], S_b[1:]))


# ---- the records at the benched sizes (4 x 4 tiles on the emulated device)
def bar_delta(f_max, rho_min, u_max):
    """delta from the populations' bar (STEP_BAR of max |f|, held by test_gpu_bench_scale at these sizes)"""
    e = STEP_BAR * f_max
    d_rho = 9 * e
    d_u = (6 * e + u_max * d_rho) / rho_min
    return np.array([d_rho, d_u, d_u]) + 16 * U / rho_min


def assert_stats_tiles(stats, margin, what):
    n, r, u, c = stats
    return n, tuple(assert_tiles_identical(a, margin, f"{what} {name}").copy() for a, name in ((r, "rho_mean"), (u, "u_mean"), (c, "u_cov")))


@gpu
def test_cylinder_statistics_at_8192(orc):
    """k_bgk_interior_stats<PULL,COMP,IBM> at the benched size: the free-stream rules, a small immersed body in the first tile,
    50 steps; every tile one tile from the edges equal to every other in all six fields, the middle one to the exact
    reference over the oracle's 3 x 3-tile run"""
    X = Y = full(8192)
    omega, u_lb, steps = 1.0 / 0.55, 0.03, 50
    rho_t, u_t = tile_fields()
    f_t = orc.equilibrium(u_t, rho_t)
    th = 2 * np.pi * np.arange(40) / 40
    xs, ys = 40.3 + 9.0 * np.cos(th), 50.2 + 9.0 * np.sin(th)
    d = cases.cylinder(X, Y, omega, u_lb, xs, ys)
    d.set_f(tiled(f_t, X // T, Y // T))
    d.stats_start(1)
    d.step(steps)
    n, tile = assert_stats_tiles(d.stats(), 1, "cylinder statistics")
    d.close()
    f = tiled(f_t, 3, 3)
    u = np.zeros((3 * T, 3 * T, 2)); rho = np.ones((3 * T, 3 * T, 1))
    ib = orc.ibm_create(xs, ys)
    samples, fmax = [], np.abs(f).max()
    for _ in range(steps):
        orc.cylinder_step(f, u, rho, omega, u_lb, ib)
        mid = (slice(T, 2 * T), slice(T, 2 * T))
        samples.append((rho[mid][..., 0].copy(), u[mid][..., 0].copy(), u[mid][..., 1].copy()))
        fmax = max(fmax, np.abs(f[mid]).max())
    orc.ibm_destroy(ib)
    delta = bar_delta(fmax, min(s[0].min() for s in samples), max(np.abs(s[1:]).max() for s in samples))
    check("cylinder at 8192^2, middle tile", (n,) + tile, samples, delta)


@gpu
def test_kbc_statistics_at_8192(orc):
    """KBC's MODE_PULL statistics kernel at size on a fully periodic field: every tile, the edge tiles included, equal to the
    exact reference over the oracle's 128 x 128 run (the first sample: the moments of lbm_set_moments)"""
    X = Y = full(8192)
    s2, steps = 1.0 / (0.5 + 3.0 * 1.70766666e-4), 40
    rho_t, u_t = tile_fields()
    m0 = np.ascontiguousarray(rho_t[..., 0])
    f_t = orc.kbc_equilibrium(m0, u_t)
    d = cases.kbc(X, Y, s2)
    d.set_f(tiled(f_t, X // T, Y // T))
    d.set_moments(tiled(rho_t, X // T, Y // T), tiled(u_t, X // T, Y // T))
    d.stats_start(1)
    d.step(steps)
    n, tile = assert_stats_tiles(d.stats(), 0, "kbc statistics")
    d.close()
    f, m, u = f_t.copy(), m0.copy(), u_t.copy()
    samples, fmax = [], np.abs(f).max()
    for _ in range(steps):
        samples.append((m.copy(), u[..., 0].copy(), u[..., 1].copy()))
        orc.kbc_step(f, m, u, s2)
        fmax = max(fmax, np.abs(f).max())
    delta = bar_delta(fmax, min(s[0].min() for s in samples), max(np.abs(s[1:]).max() for s in samples))
    check("kbc at 8192^2, every tile", (n,) + tile, samples, delta)


def tile_solid():
    """one disc per tile spanning columns 14 .. 114: across a row of tiles its listed nodes fall in every mask word"""
    return disc(T, T, 63.7, 64.4, 50.2)


@gpu
def test_staircase_bodies_both_records_at_8192(orc):
    """one staircase disc per 128 x 128 tile of a periodic 8192^2 grid (listed nodes in interior columns on every tile row,
    across all 256 mask words), statistics and body force recorded together, 30 steps:
    - the statistics of every tile bit-identical, and equal to the exact reference over the oracle's periodic tile;
    - every step's force = ntiles x the tile's momentum exchange in the oracle's run, within the summation bound plus the
      links' share of the populations' bar;
    - the last step's force = the NumPy definition on the exported final state, to 1e-13 of the summed magnitudes;
    - more than 256 x 256 links: the finisher's strided loop runs more than once per thread"""
    X = Y = full(8192)
    steps, omega = 30, STAIR_OMEGA
    ntiles = (X // T) * (Y // T)
    rho_t, u_t = tile_fields()
    f_t = orc.equilibrium(u_t, rho_t)
    solid_t = tile_solid()
    solid = tiled(solid_t, X // T, Y // T)
    d = L.Domain(L.default_config(model=L.MODEL_BGK, X=X, Y=Y, omega=omega, equilibrium=L.EQ_COMPRESSIBLE))
    d.bc_clear()
    d.bc_add_solid(solid)
    d.bc_commit()
    d.set_f(tiled(f_t, X // T, Y // T))
    d.body_force_record(solid, capacity=steps)
    d.stats_start(1)
    d.step(steps)
    F, first = d.body_force()
    n, tile = assert_stats_tiles(d.stats(), 0, "staircase statistics")
    lk_t = links(solid_t)
    n_links = ntiles * sum(len(i) for i, _ in lk_t.values())
    nblk = -(-n_links // 256)
    if not EMU:
        assert n_links > 256 * 256, n_links
    # the definition on the exported final state
    f_end = d.get_f()
    d.close()
    want, scale = momentum_exchange(f_end, links(solid))
    del f_end
    err_last = np.abs(F[-1] - want).max()
    print(f"staircase at {X}^2: {n_links} links, {nblk} blocks; last step vs NumPy on the state: {err_last:.2e} "
          f"(bound {1e-13 * scale:.2e})")
    assert first == 0 and len(F) == steps
    assert np.all(np.abs(F[-1] - want) <= 1e-13 * scale), (F[-1], want)
    # the oracle's tile
    f = f_t.copy()
    samples, worst, fmax = [], 0.0, np.abs(f).max()
    depth = 17 + -(-nblk // 256)
    for t in range(steps):
        rho = orc.calc_rho(f)
        u = orc.calc_u(f, rho)
        samples.append((rho[..., 0], u[..., 0], u[..., 1]))
        f = bounce_back_step(orc, f, solid_t, omega)
        Ft, mag = momentum_exchange(f, lk_t)
        fmax = max(fmax, np.abs(f).max())
        bound = ntiles * (depth * U * mag + 2 * STEP_BAR * fmax * sum(len(i) for i, _ in lk_t.values()))
        err = np.abs(F[t] - ntiles * Ft).max()
        worst = max(worst, err / bound)
        assert np.all(np.abs(F[t] - ntiles * Ft) <= bound), (t, F[t], ntiles * Ft, bound)
    print(f"staircase at {X}^2: per-step force vs {ntiles} x the oracle's tile: worst err / bound = {worst:.2e}")
    delta = bar_delta(fmax, min(s[0].min() for s in samples), max(np.abs(s[1:]).max() for s in samples))
    check(f"staircase at {X}^2, every tile", (n,) + tile, samples, delta)
