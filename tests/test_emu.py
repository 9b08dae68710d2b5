"""The `-m gpu` parity tests, run on host cores against the library's own CUDA sources compiled by the SIMT emulator of
tests/cpu_emu/ (fibers for the threads of a block, typed waits for __syncthreads and the warp shuffles, an
immediately-executing CUDA runtime whose fresh allocations are NaN-filled).  TEST INFRASTRUCTURE: it checks the kernels'
indexing, shared-memory rings, barriers, boundary tables and the host-side step schedule where there is no GPU; it says
nothing about speed, and rounding differs from the device's (no FMA contraction), so it is no substitute for the
`-m gpu` run on the B200.  The product never loads the emulated library (tests/conftest.py, LBM_EMU=1 only).

The default CPU suite runs every GPU test except the 10^4-step ones and two long golden runs;
`LBM_EMU=1 python -m pytest tests -m gpu` runs all of them (about ten minutes on eight cores)."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "cpu_emu")
SLOW = [
    "tests/test_gpu_long_horizon.py",
    "tests/test_gpu_kbc.py::test_double_shear_flow_reference_driver_golden",
    "tests/test_gpu_bgk.py::test_poiseuille_golden_and_l2",
]


@pytest.fixture(scope="module")
def emu_lib():
    if sys.platform != "linux":
        pytest.skip("the emulated build is set up for Linux")
    r = subprocess.run(["make", "-C", EMU_DIR, "-j8"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    path = os.path.join(EMU_DIR, "_build", "liblbm_b200_emu.so")
    assert os.path.exists(path)
    return path


def run_emulated(args, timeout, order="forward"):
    env = dict(os.environ, LBM_EMU="1", OMP_WAIT_POLICY="passive", EMU_ORDER=order)
    cmd = [sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider"] + args
    return subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)


def test_gpu_parity_tests_pass_on_the_emulated_device(emu_lib):
    args = ["tests"]
    for s in SLOW:
        args += ["--deselect", s]
    r = run_emulated(args, 1500)
    tail = r.stdout[-4000:]
    assert r.returncode == 0, tail
    last = r.stdout.strip().splitlines()[-1]
    assert " passed" in last and "failed" not in last, tail
    assert int(last.split(" passed")[0].split()[-1]) >= 80, last  # the emulated run really ran the parity tests


@pytest.mark.parametrize("order", ["reverse", "shuffle:3"])
def test_shared_memory_ring_kernels_do_not_depend_on_thread_order(emu_lib, order):
    """The threads of a block start and resume in reversed / shuffled order.  A missing barrier around the shared-memory
    rings of k_tp_fused / k_csf_collide_ring makes these runs fail (checked by deleting the ring's __syncthreads).  Every
    instantiation of the two-phase step runs here too (test_gpu_tp_variants.py: stage slots, mbarrier parities, ring rows),
    and both records' kernels (test_gpu_records_exact.py: the body-force block reductions, the statistics planes)."""
    r = run_emulated(["tests/test_gpu_two_phase.py", "tests/test_gpu_csf.py", "tests/test_gpu_tp_variants.py",
                      "tests/test_gpu_records_exact.py"], 1500, order)
    assert r.returncode == 0, r.stdout[-4000:]


def test_kernels_under_address_sanitizer():
    """Device buffers are heap blocks of the emulated runtime: an out-of-bounds load or store of a kernel (or of the host
    code around it) is an AddressSanitizer report.  The two-phase and CSF tests here (ragged and tiny grids included, every
    two-phase kernel instantiation at one-row bands) and the records' tests; `make -C tests/cpu_emu SAN=1` + LBM_EMU_ASAN=1 runs any of the others the same way."""
    asan = subprocess.run(["/usr/bin/gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("no libasan next to the system gcc")
    r = subprocess.run(["make", "-C", EMU_DIR, "-j8", "SAN=1"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    env = dict(os.environ, LBM_EMU="1", LBM_EMU_ASAN="1", OMP_WAIT_POLICY="passive", LD_PRELOAD=asan,
               ASAN_OPTIONS="detect_leaks=0:abort_on_error=1:verify_asan_link_order=0")
    cmd = [sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider",
           "tests/test_gpu_two_phase.py", "tests/test_gpu_csf.py", "tests/test_gpu_tp_variants.py", "tests/test_gpu_records_exact.py"]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0 and "AddressSanitizer" not in r.stdout + r.stderr, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.parametrize("world", [2, 3, 5, 8])
def test_slab_ring_over_the_nccl_stand_in(emu_lib, world, csf_fused="0"):
    """tests/mp_nccl_check.py's own checks (the GPU box runs them under torchrun over real NCCL) with one thread per rank on
    the emulated device: Poiseuille pressure packets across the ring, MRTCG / RK / CSF halos, an immersed body inside one
    slab and across every cut — bit-exact against the monolithic run at ring sizes the GPU budget never reached (8)."""
    env = dict(os.environ, OMP_WAIT_POLICY="passive", OMP_NUM_THREADS="2", FAKE_NCCL_TIMEOUT_S="120", LBM_CSF_FUSED=csf_fused)
    r = subprocess.run([sys.executable, os.path.join(EMU_DIR, "ring_threads.py"), str(world)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "failures: []" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    # six checks, the two overlapped two-phase runs, the RK diagnostics, the statistics and body-force records
    assert r.stdout.count(f"ring of {world}") == 11, r.stdout


@pytest.mark.parametrize("world", [2, 8])
def test_comm_check_turns_the_missing_marker_list_into_an_error(emu_lib, world):
    """lbm_comm_check on a ring of threads: a body across a cut handed to rank 0 only is LBM_ERR_COMM on every rank (it
    hung an eight-GPU run once); both correct usages pass"""
    env = dict(os.environ, OMP_NUM_THREADS="1", FAKE_NCCL_TIMEOUT_S="60")
    r = subprocess.run([sys.executable, os.path.join(EMU_DIR, "ring_check_misuse.py"), str(world)], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and f"misuse reported on all {world} ranks" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


@pytest.mark.parametrize("world", [2, 8])
def test_bench_ring_parity_leg_over_the_nccl_stand_in(emu_lib, world):
    """bench.py's ring_parity (what every multi-GPU bench run checks before its timed region: each model family over the ring
    against the monolithic run, lbm_comm_check, the ring-wide max of the RK diagnostics) on emulated rings"""
    env = dict(os.environ, OMP_WAIT_POLICY="passive", OMP_NUM_THREADS="1", FAKE_NCCL_TIMEOUT_S="120")
    r = subprocess.run([sys.executable, os.path.join(EMU_DIR, "bench_ring_threads.py"), str(world)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "'green': True" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("bit_exact") >= 11, r.stdout


def test_blocks_bound_across_ranks_over_the_nccl_stand_in(emu_lib):
    """test/decompose_domain_loop.cpp's four blocks, one per rank (lbm_comm_init_blocks, lbm_link_face_rank,
    lbm_comm_faces_commit, plain lbm_step), a statistics record on each: bit-identical to the blocks linked inside one process"""
    env = dict(os.environ, OMP_WAIT_POLICY="passive", OMP_NUM_THREADS="1", FAKE_NCCL_TIMEOUT_S="60")
    r = subprocess.run([sys.executable, os.path.join(EMU_DIR, "blocks_ring_threads.py")], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "bit-exact vs linked blocks = True" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
    assert "statistics record bit-exact vs linked blocks = True" in r.stdout, r.stdout[-2000:]


def test_two_phase_halos_behind_the_interior_bands_over_random_rings(emu_lib):
    """LBM_TP_OVERLAP=1 (tp_steps_ring: edge bands, then both halo exchanges on the side stream under the interior bands) over
    random ring sizes, slab heights, band heights and lbm_step call patterns: bit-identical to the monolithic run"""
    env = dict(os.environ, OMP_WAIT_POLICY="passive", OMP_NUM_THREADS="1", FAKE_NCCL_TIMEOUT_S="60")
    r = subprocess.run([sys.executable, os.path.join(EMU_DIR, "ring_overlap_fuzz.py"), "7", "10"], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "10 of 10 cases bit-exact" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_single_pass_csf_step_on_the_ring(emu_lib):
    """LBM_CSF_FUSED=1 on the slabs of a ring (two 2-row halos between the pre-pass stages): bit-identical to the monolithic run"""
    test_slab_ring_over_the_nccl_stand_in(emu_lib, 3, csf_fused="1")


def test_every_bench_workload_sets_up_and_steps_on_the_emulated_device(emu_lib):
    env = dict(os.environ, OMP_WAIT_POLICY="passive")
    r = subprocess.run([sys.executable, os.path.join(EMU_DIR, "bench_cases.py")], cwd=ROOT, env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count(" ok") >= 9, r.stdout


def test_the_product_binding_does_not_know_the_emulated_library():
    src = open(os.path.join(ROOT, "lattice-boltzmann-method_b200", "python", "lbm_b200", "__init__.py")).read()
    assert "emu" not in src.lower() and "LBM_EMU" not in src
    for name in ("bench.py", "__graft_entry__.py"):
        assert "cpu_emu" not in open(os.path.join(ROOT, name)).read()
