"""Every kernel instantiation the two-phase step can launch (tp_launch_fused, DESIGN §7d), held to the oracle and to each other.

MRT colour gradient (H = 2) and Rothman-Keller (H = 1) each run one of eight / nine kernels, chosen when the domain is created
from LBM_TP_STAGED, LBM_TP_STASH, LBM_TP_NS and LBM_TP_PIPE; LBM_TP_RPB sets the band height.  They differ where only hardware
can be wrong: tensor-memory columns per resident block, bulk-copy / mbarrier slot reuse at 2 to 6 slots and their prefetch
distance, register allocation.  Shapes sit around the strip width (USEFUL = 128 - 2H columns: 124 MRTCG, 126 RK) and the band
heights leave a last band of a single row, shorter than the 2H warm-up rows.

Bounds.  Oracle: populations relative, rho / u / rho_r / rho_b absolute, after 2 and 7 steps: TOL_ORACLE = 1e-13 for every
instantiation.  Measured on a B200 (1000 W power limit) over these shapes and band heights: the default kernels at most 4.9e-15
(MRTCG) and 1.1e-15 (RK), every other instantiation the same; the emulated device 4.0e-15 and 4.4e-16.  Instantiations against
k_tp_fused<MODEL, false>: TOL_AGREE = 1e-14 in the product build, where nvcc picks per kernel which multiply-adds it fuses
(measured on the same B200 after 7 steps: at most 2.2e-15 for MRTCG, 2.2e-18 for RK); bit for bit in the -fmad=false build
(tp_variant_check.py) and on the emulated device.  One instantiation against itself (run twice, other band heights): bit for
bit everywhere.  Record of the B200 run: profiles/r03_pytest_tp_variants.txt."""
import contextlib
import functools
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import cases
import lbm_b200 as L
from oracle_lib import Oracle
from test_gpu_two_phase import mrtcg_params, rk_params

pytestmark = pytest.mark.gpu

EMU = os.environ.get("LBM_EMU") == "1"
TOL_ORACLE = 1e-13
TOL_AGREE = 1e-14
SWITCHES = ("LBM_TP_STAGED", "LBM_TP_STASH", "LBM_TP_NS", "LBM_TP_PIPE", "LBM_TP_RPB")


def _staged(stash, ns):
    return {"LBM_TP_STAGED": "1", "LBM_TP_STASH": str(int(stash)), "LBM_TP_NS": str(ns)}


FUSED = {"LBM_TP_STAGED": "0", "LBM_TP_PIPE": "0"}
FUSED_PIPE = {"LBM_TP_STAGED": "0", "LBM_TP_PIPE": "1"}

# name -> (model, switches, the kernel tp_launch_fused launches with them)
VARIANTS = {
    "mrtcg-stash2": ("mrtcg", _staged(1, 2), "k_tp_staged<0, 2, 4, true>"),
    "mrtcg-stash3": ("mrtcg", _staged(1, 3), "k_tp_staged<0, 3, 3, true>"),
    "mrtcg-stash4": ("mrtcg", _staged(1, 4), "k_tp_staged<0, 4, 2, true>"),
    "mrtcg-slots4": ("mrtcg", _staged(0, 4), "k_tp_staged<0, 4, 2, false>"),
    "mrtcg-slots5": ("mrtcg", _staged(0, 5), "k_tp_staged<0, 5, 2, false>"),
    "mrtcg-slots6": ("mrtcg", _staged(0, 6), "k_tp_staged<0, 6, 2, false>"),
    "mrtcg-fused-pipe": ("mrtcg", FUSED_PIPE, "k_tp_fused<0, true>"),
    "mrtcg-fused": ("mrtcg", FUSED, "k_tp_fused<0, false>"),
    "rk-stash2": ("rk", _staged(1, 2), "k_tp_staged<1, 2, 4, true>"),
    "rk-stash3": ("rk", _staged(1, 3), "k_tp_staged<1, 3, 3, true>"),
    "rk-stash4": ("rk", _staged(1, 4), "k_tp_staged<1, 4, 2, true>"),
    "rk-slots3": ("rk", _staged(0, 3), "k_tp_staged<1, 3, 3, false>"),
    "rk-slots4": ("rk", _staged(0, 4), "k_tp_staged<1, 4, 2, false>"),
    "rk-slots5": ("rk", _staged(0, 5), "k_tp_staged<1, 5, 2, false>"),
    "rk-slots6": ("rk", _staged(0, 6), "k_tp_staged<1, 6, 2, false>"),
    "rk-fused-pipe": ("rk", FUSED_PIPE, "k_tp_fused<1, true>"),
    "rk-fused": ("rk", FUSED, "k_tp_fused<1, false>"),
}
DEFAULT = {"mrtcg": "mrtcg-stash3", "rk": "rk-slots5"}  # what runs with no switch set
REFERENCE = {"mrtcg": "mrtcg-fused", "rk": "rk-fused"}  # two pulls through registers, no staging: what the others must equal


def names_of(model):
    return [n for n, v in VARIANTS.items() if v[0] == model]


# MRTCG (R, C): 5 interior columns; exactly one strip of 124; a second strip of one column; a last strip of three.
# RK (L,): 3 interior columns, 31, exactly one strip of 126, a second strip of one column
SHAPES = {"mrtcg": [(9, 7), (25, 126), (31, 127), (13, 253)], "rk": [(5,), (33,), (128,), (129,)]}
# band heights: 1 < H for MRTCG, 2 and 3 < the 2H warm-up rows, 2H + 1, the least height pick_band_rows chooses; 121 rows
# leave a last band of one row at every one of them
RPBS = [0, 1, 2, 3, 5, 24]
BAND_SHAPES = {"mrtcg": (121, 127), "rk": (121,)}
SCHEDULE = (2, 5)  # the getters between steps 2 and 3 leave the moment planes full for the third step


@contextlib.contextmanager
def switches(env, rpb=0):
    """the LBM_TP_* variables as `env` (+ LBM_TP_RPB) while the domain is created, the caller's afterwards"""
    old = {k: os.environ.get(k) for k in SWITCHES}
    for k in SWITCHES:
        os.environ.pop(k, None)
    os.environ.update(env)
    if rpb:
        os.environ["LBM_TP_RPB"] = str(rpb)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@functools.lru_cache(maxsize=None)
def oracle():
    return Oracle()


def initial(model, shape):
    if model == "mrtcg":
        p = mrtcg_params(*shape, (6.25e-6, 0.0), 1)
        return p, oracle().mrtcg_init(p, "rt")
    p = rk_params(shape[0])
    p.radius = max(1.5, shape[0] / 4.0)
    return p, oracle().rk_init(p)


def fields(f_r, f_b, rho, u, rho_r, rho_b):
    return tuple(np.array(a, dtype=np.float64).reshape(-1) for a in (f_r, f_b, rho, u, rho_r, rho_b))


@functools.lru_cache(maxsize=None)
def oracle_run(model, shape):
    p, st = initial(model, shape)
    step = oracle().mrtcg_step if model == "mrtcg" else oracle().rk_step
    out = []
    for n in SCHEDULE:
        for _ in range(n):
            step(p, st)
        out.append(fields(st["r_adv"], st["b_adv"], st["rho"], st["u"], st["r_rho"], st["b_rho"]))
    return out


def device_run(model, env, shape, rpb=0):
    """[(f_red, f_blue, rho, u, rho_r, rho_b)] after each entry of SCHEDULE, the domain created under the switches `env`"""
    _, st = initial(model, shape)
    with switches(env, rpb):
        d = cases.mrtcg(*shape, (6.25e-6, 0.0), 1) if model == "mrtcg" else cases.rk(shape[0])
    try:
        if model == "mrtcg":
            d.init_two_phase(st["r_rho"], st["b_rho"], st["u"])
        else:
            d.set_f(st["r_adv"], 0)
            d.set_f(st["b_adv"], 1)
        out = []
        for n in SCHEDULE:
            d.step(n)
            rho, u = d.get_moments()
            _, rho_r, rho_b = d.get_phase()
            out.append(fields(d.get_f(0), d.get_f(1), rho, u, rho_r, rho_b))
    finally:
        d.close()
    return out


def run(name, shape, rpb=0):
    return device_run(VARIANTS[name][0], VARIANTS[name][1], shape, rpb)


cached_run = functools.lru_cache(maxsize=None)(run)  # shared by the tests below: each variant x shape runs once


def distance(A, B):
    """populations relative to the largest one, the O(1) moments absolute; the worst over every snapshot"""
    w = 0.0
    for a, b in zip(A, B):
        for k, (x, y) in enumerate(zip(a, b)):
            assert x.shape == y.shape, k
            w = max(w, float(np.abs(x - y).max()) / (float(np.abs(y).max()) if k < 2 else 1.0))
    return w


def first_difference(A, B):
    """None when every field of every snapshot is bit-identical, else where the first difference is"""
    for n, (a, b) in enumerate(zip(A, B)):
        for name, x, y in zip(("f_red", "f_blue", "rho", "u", "rho_r", "rho_b"), a, b):
            if not np.array_equal(x, y):
                return f"snapshot {n}, {name}: {int((x != y).sum())} entries differ, max |delta| {np.abs(x - y).max():.3e}"
    return None


def variant_shapes(shapes):
    return [pytest.param(n, s, id=f"{n}-{'x'.join(map(str, s))}") for n, v in VARIANTS.items() for s in shapes[v[0]]]


@pytest.mark.parametrize("name,shape", variant_shapes(SHAPES))
def test_variant_vs_oracle(name, shape):
    model = VARIANTS[name][0]
    got = cached_run(name, shape)
    assert distance(got, oracle_run(model, shape)) < TOL_ORACLE, distance(got, oracle_run(model, shape))


@pytest.mark.parametrize("rpb", RPBS)
@pytest.mark.parametrize("name", list(VARIANTS))
def test_variant_vs_oracle_at_band_height(name, rpb):
    model = VARIANTS[name][0]
    shape = BAND_SHAPES[model]
    got = cached_run(name, shape, rpb)
    assert distance(got, oracle_run(model, shape)) < TOL_ORACLE, distance(got, oracle_run(model, shape))


@pytest.mark.parametrize("name", list(VARIANTS))
def test_variant_is_one_function_of_its_input(name):
    """the same kernel run twice and at band heights 1, 3 and 16: bit for bit (the arithmetic of a node does not depend on the
    band; a stage slot refilled early, a wrong slot or parity, a ring row rotated wrongly shows here)"""
    shape = {"mrtcg": (49, 253), "rk": (129,)}[VARIANTS[name][0]]
    base = cached_run(name, shape)
    for what, rpb in (("again", 0), ("1-row bands", 1), ("3-row bands", 3), ("16-row bands", 16)):
        diff = first_difference(run(name, shape, rpb), base)
        assert diff is None, (what, diff)


@pytest.mark.parametrize("model", ["mrtcg", "rk"])
def test_variants_agree(model):
    """every instantiation within TOL_AGREE of the plain k_tp_fused; bit for bit on the emulated device, which never contracts"""
    for shape in SHAPES[model]:
        ref = cached_run(REFERENCE[model], shape)
        for name in names_of(model):
            if EMU:
                assert first_difference(cached_run(name, shape), ref) is None, (name, shape, first_difference(cached_run(name, shape), ref))
            else:
                assert distance(cached_run(name, shape), ref) < TOL_AGREE, (name, shape, distance(cached_run(name, shape), ref))


@pytest.mark.parametrize("model,shape", [("mrtcg", (31, 127)), ("mrtcg", (13, 253)), ("rk", (33,)), ("rk", (129,))])
def test_variants_bit_identical_without_contraction(model, shape):
    """the same sources compiled with -fmad=false (liblbm_b200_nofma.so, built by __graft_entry__.build()): every instantiation
    of the model bit for bit equal to the plain k_tp_fused.  On the emulated device the loaded library itself is held to it."""
    if EMU:
        ref = cached_run(REFERENCE[model], shape)
        for name in names_of(model):
            assert first_difference(cached_run(name, shape), ref) is None, name
        return
    lib = os.path.join(L.PKG_DIR, "liblbm_b200_nofma.so")
    assert os.path.exists(lib), f"{lib} is missing: make -C lattice-boltzmann-method_b200 NOFMA=1"
    r = subprocess.run([sys.executable, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tp_variant_check.py"), "--lib", lib,
                        model] + [str(s) for s in shape], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def mangled(kernel):
    """k_tp_staged<0, 3, 3, true> -> k_tp_stagedILi0ELi3ELi3ELb1E (the Itanium spelling of the same instantiation)"""
    name, args = kernel[:-1].split("<")
    return name + "I" + "".join(f"Lb{int(a == 'true')}E" if a in ("true", "false") else f"Li{a}E" for a in args.split(", ")) + "E"


@pytest.mark.parametrize("name", list(VARIANTS) + ["mrtcg-default", "rk-default"])
def test_switch_reaches_the_kernel(name):
    """one step under torch.profiler: the instantiation VARIANTS names (the default one with no switch set) is the only
    row-marching kernel that ran"""
    if EMU:
        pytest.skip("kernel names come from the device's profiler")
    import torch
    from torch.profiler import ProfilerActivity, profile

    if name.endswith("-default"):
        model, env, kernel = name.split("-")[0], {}, VARIANTS[DEFAULT[name.split("-")[0]]][2]
    else:
        model, env, kernel = VARIANTS[name]
    with switches(env):
        d = cases.mrtcg(31, 127, (6.25e-6, 0.0), 1) if model == "mrtcg" else cases.rk(33)
    try:
        d.init_two_phase(np.ones((d.Xl, d.Y)), np.ones((d.Xl, d.Y)), np.zeros((d.Xl, d.Y, 2)))
        d.step(1)
        d.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            d.step(1)
            d.synchronize()
            torch.cuda.synchronize()
    finally:
        d.close()
    ran = {m for e in prof.events() for m in re.findall(r"k_tp_(?:staged|fused)(?:<[^>]*>|I(?:L[ib]\d+E)+E)", e.name)}
    assert ran in ({kernel}, {mangled(kernel)}), (kernel, sorted(ran), sorted({e.name for e in prof.events()})[:40])


# LBM_TP_NS out of range -> the instantiation the clamp of tp_launch_fused selects
CLAMPED = {("mrtcg", 1): {"0": "mrtcg-stash3", "1": "mrtcg-stash2", "7": "mrtcg-stash4", "99": "mrtcg-stash4", "-3": "mrtcg-stash3"},
           ("mrtcg", 0): {"0": "mrtcg-slots5", "1": "mrtcg-slots4", "7": "mrtcg-slots6", "99": "mrtcg-slots6", "-3": "mrtcg-slots5"},
           ("rk", 1): {"0": "rk-stash4", "1": "rk-stash2", "7": "rk-stash4", "99": "rk-stash4", "-3": "rk-stash4"},
           ("rk", 0): {"0": "rk-slots5", "1": "rk-slots3", "7": "rk-slots6", "99": "rk-slots6", "-3": "rk-slots5"}}


@pytest.mark.parametrize("ns", ["0", "1", "7", "99", "-3"])
@pytest.mark.parametrize("stash", [1, 0])
@pytest.mark.parametrize("model", ["mrtcg", "rk"])
def test_out_of_range_stage_count(model, stash, ns):
    """runs the instantiation the clamp selects (bit for bit the same result) and holds the oracle bound"""
    shape = SHAPES[model][2]
    got = device_run(model, {"LBM_TP_STAGED": "1", "LBM_TP_STASH": str(stash), "LBM_TP_NS": ns}, shape)
    assert first_difference(got, cached_run(CLAMPED[(model, stash)][ns], shape)) is None, CLAMPED[(model, stash)][ns]
    assert distance(got, oracle_run(model, shape)) < TOL_ORACLE


# ---- the other step paths with two instantiations besides the defaults: linked slabs (lbm_step_group) and stream capture
OTHER = ["stash2", "fused"]


@pytest.mark.parametrize("kind", OTHER)
@pytest.mark.parametrize("model,P", [("mrtcg", 2), ("mrtcg", 3), ("rk", 2), ("rk", 3)])
def test_two_phase_slabs_equal_monolithic_with_variant(monkeypatch, model, P, kind):
    import test_gpu_slabs

    for k, v in VARIANTS[f"{model}-{kind}"][1].items():
        monkeypatch.setenv(k, v)
    test_gpu_slabs.test_two_phase_slabs_equal_monolithic(model, P)


@pytest.mark.parametrize("kind", OTHER)
@pytest.mark.parametrize("model", ["mrtcg", "rk"])
def test_two_phase_graph_equals_plain_with_variant(monkeypatch, model, kind):
    if EMU:
        pytest.skip("needs a real device (CUDA graphs): not emulated")
    import test_gpu_graph

    for k, v in VARIANTS[f"{model}-{kind}"][1].items():
        monkeypatch.setenv(k, v)
    test_gpu_graph.test_two_phase_graph_equals_plain(model)
