import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "lattice-boltzmann-method_b200", "python"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "ref: needs oracle/_ref (the compiled reference; built only from a checkout of the original sources, see oracle/Makefile)")


# TEST INFRASTRUCTURE: LBM_EMU=1 points the binding at tests/cpu_emu/_build/liblbm_b200_emu.so — the library's own CUDA
# sources compiled for host cores by the SIMT emulator of tests/cpu_emu/ — so that the `-m gpu` parity tests can
# exercise the kernels' logic in a container without a GPU (tests/test_emu.py does exactly that in a subprocess).
# The product never takes this route: lbm_b200.load() knows one path only and raises when liblbm_b200.so is missing.
if os.environ.get("LBM_EMU") == "1":
    import lbm_b200

    # LBM_EMU_ASAN=1: the AddressSanitizer build (make -C tests/cpu_emu SAN=1; run python with libasan preloaded)
    _emu_build = os.path.join(ROOT, "tests", "cpu_emu", "_build_asan" if os.environ.get("LBM_EMU_ASAN") == "1" else "_build")
    lbm_b200.LIB_PATH = os.path.join(_emu_build, "liblbm_b200_emu.so")
    # the drivers' binaries (RUNPATH to liblbm_b200.so) resolve the same soname to the emulated build first
    os.environ["LD_LIBRARY_PATH"] = os.path.join(_emu_build, "drv") + ":" + os.environ.get("LD_LIBRARY_PATH", "")


# TEST INFRASTRUCTURE: LBM_TEST_LIB=<path> runs the suite against another BUILD of the same library (an experiment variant of
# lattice-boltzmann-method_b200/Makefile: NOFMA=1, X4=1, HINTS=n) — still the CUDA path, still through the C ABI
if os.environ.get("LBM_TEST_LIB"):
    import lbm_b200

    lbm_b200.LIB_PATH = os.path.abspath(os.environ["LBM_TEST_LIB"])


# what the emulated runtime does not provide: stream capture (CUDA graphs)
EMU_SKIPS = ("test_gpu_graph.py", "slabs_and_graph")


def pytest_collection_modifyitems(config, items):
    if os.environ.get("LBM_EMU") != "1":
        return
    skip = pytest.mark.skip(reason="needs a real device (CUDA graphs): not emulated")
    for item in items:
        if any(k in item.nodeid for k in EMU_SKIPS):
            item.add_marker(skip)
