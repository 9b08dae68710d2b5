"""GPU parity of the multi-block path (SURVEY §8(f) rank 4, test/decompose_domain_loop.cpp): blocks with their own
coordinates and wall rules, bound across column faces (lbm_link_face), a body force on part of one block
(lbm_set_force_region), advanced in lock step (lbm_step_group)."""
import os
import sys

import numpy as np
import pytest

import cases
import lbm_b200 as L
from oracle_lib import Oracle

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import blocks_oracle as BO  # noqa: E402

pytestmark = pytest.mark.gpu

OMEGA = 1.0 / (np.sqrt(3.0 / 16.0) + 0.5)   # decompose_domain_loop.cpp:49-50


def face_mask_from_bindings(Ln):
    """(block -> bool {R,C,9}) of the populations the driver's binding lines assign"""
    m = {k: np.zeros(s + (9,), dtype=bool) for k, s in BO.shapes(Ln).items()}
    for dst, drows, dcol, q, _, _, _ in BO.bindings(Ln):
        m[dst][drows, dcol, q] = True
    return m


@pytest.mark.parametrize("Ln", [64, 128])
def test_loop_blocks_vs_oracle(Ln):
    """random populations on all four blocks, 40 iterations: every step's populations at 1e-12, and the compiled masks of
    the bound populations equal to the driver's assignment lists bit for bit"""
    orc = Oracle()
    dom = cases.loop_blocks(Ln, OMEGA)
    st = BO.init(orc, Ln)
    rng = np.random.default_rng(5)
    want = face_mask_from_bindings(Ln)
    for k, b in st.items():
        b["f"] = b["f"] * (1.0 + 0.05 * rng.standard_normal(b["f"].shape))
        dom[k].set_f(b["f"])
        n_ops = 6 + (6 if k in "AC" else 0)
        assert np.array_equal(dom[k].bc_mask() > n_ops, want[k]), k
    order = [dom[k] for k in "ABCD"]
    for n in range(1, 41):
        BO.step(orc, st, Ln, OMEGA)
        L.step_group(order, 1)
        if n in (1, 2, 3, 17, 40):
            for k in "ABCD":
                assert cases.relerr(dom[k].get_f(), st[k]["f"]) < 1e-12, (n, k)
    # many steps in one call, then moments
    for _ in range(25):
        BO.step(orc, st, Ln, OMEGA)
    L.step_group(order, 25)
    for k in "ABCD":
        assert cases.relerr(dom[k].get_f(), st[k]["f"]) < 1e-12, k
        rho, u = dom[k].get_moments()
        r = orc.calc_rho(st[k]["f"])
        assert np.abs(rho - r).max() < 1e-12 and np.abs(u - orc.calc_u(st[k]["f"], r)).max() < 1e-12


def test_loop_blocks_statistics_vs_exact_definition():
    """a statistics record on the four bound blocks (their face columns are listed nodes in edge columns, the walls of A and
    C listed rows): each block's record against the exact mean and covariance over the moments of blocks_oracle's run, within
    test_gpu_records_exact's bound; the region force on block A samples the plain moments its collision uses"""
    from test_gpu_records_exact import check, moment_delta

    Ln, steps, every = 64, 30, 2
    orc = Oracle()
    dom = cases.loop_blocks(Ln, OMEGA)
    st = BO.init(orc, Ln)
    rng = np.random.default_rng(7)
    for k, b in st.items():
        b["f"] = b["f"] * (1.0 + 0.05 * rng.standard_normal(b["f"].shape))
        dom[k].set_f(b["f"])
        dom[k].stats_start(every)
    order = [dom[k] for k in "ABCD"]
    samples = {k: [] for k in "ABCD"}
    delta = {k: np.zeros(3) for k in "ABCD"}
    for t in range(steps):
        BO.step(orc, st, Ln, OMEGA)  # leaves rho, u: the moments its collision used
        if t % every == 0:
            for k in "ABCD":
                s = (st[k]["rho"][..., 0], st[k]["u"][..., 0], st[k]["u"][..., 1])
                samples[k].append(s)
                delta[k] = np.maximum(delta[k], moment_delta(dom[k].get_f(), s, True, orc))
        L.step_group(order, 1)
    for k in "ABCD":
        check(f"loop block {k}", dom[k].stats(), samples[k], delta[k])


def test_loop_blocks_reference_driver_golden():
    """snapshots of the reference's own binary (L = 128, 400 iterations; make_golden.py:case_loop_blocks): the flow the
    body force drives round the channel, m_1 and m_0 of every block"""
    g = cases.golden("loop_blocks_128")
    Ln = int(g["L"])
    dom = cases.loop_blocks(Ln, float(g["omega"]))
    orc = Oracle()
    st = BO.init(orc, Ln)
    for k in "ABCD":
        dom[k].set_f(st[k]["f"])
    order = [dom[k] for k in "ABCD"]
    t = 0
    for i, s in enumerate(int(s) for s in g["steps"]):
        if s == 0:
            continue
        # snapshot s holds the m_0, m_1 computed in iteration s - 1, i.e. the moments of the state after s - 1 iterations
        L.step_group(order, (s - 1) - t)
        t = s - 1
        for k in "ABCD":
            rho, u = dom[k].get_moments()
            want_u = np.stack([g[k + "_ux"][i], g[k + "_uy"][i]], axis=-1)
            if k == "A":   # the driver adds F to m_1 on the forced rows before it takes the snapshot (:116)
                want_u = want_u.copy()
                want_u[BO.force_rows(Ln), :, 0] -= 3e-3
            assert np.abs(rho[..., 0] - g[k + "_rho"][i]).max() < 1e-12, (s, k)
            assert np.abs(u - want_u).max() < 1e-12, (s, k)


def test_face_link_errors():
    a = L.Domain(L.default_config(model=L.MODEL_BGK, X=16, Y=8, omega=1.0))
    b = L.Domain(L.default_config(model=L.MODEL_BGK, X=8, Y=8, omega=1.0))
    with pytest.raises(L.LbmError):
        a.link_face(0, 10, 8, b, 0)        # rows outside block a
    a.link_face(0, 8, 8, b, 0)
    with pytest.raises(L.LbmError):
        a.link_face(0, 12, 4, b, 0)        # rows already bound
    a.preset_periodic()
    a.set_f(np.ones((16, 8, 9)))
    with pytest.raises(L.LbmError):
        a.step(1)                          # bound blocks advance with the group
    with pytest.raises(L.LbmError):
        L.step_group([a], 1)               # ... and the group must contain the other block


def test_loop_driver_writes_the_reference_files(tmp_path):
    """drivers/decompose_domain_loop (L = 128, T = 400) against the snapshots of the reference's binary: same file names,
    same {R, C, T/50} stacks, 1e-12"""
    import subprocess

    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "drivers", "bin", "decompose_domain_loop")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(root, "drivers")], stdout=subprocess.DEVNULL)
    r = subprocess.run([exe, "128", "400"], cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    g = cases.golden("loop_blocks_128")
    idx = [int(s) // 50 for s in g["steps"]]
    for k in "ABCD":
        for f in ("ux", "uy", "rho"):
            a = list(torch.jit.load(str(tmp_path / f"{k}-domain-decomp-hpt-{f}.pt")).parameters())[0].numpy()
            assert a.shape == BO.shapes(128)[k] + (8,)
            for i, ts in enumerate(idx):
                assert np.abs(a[..., ts] - g[f"{k}_{f}"][i]).max() < 1e-12, (k, f, ts)
