"""TEST INFRASTRUCTURE (see cuda_emu.hpp): test/decompose_domain_loop.cpp's four blocks with ONE block per rank — column faces
bound across ranks (lbm_comm_init_blocks, lbm_link_face_rank, lbm_comm_faces_commit), one thread per rank on the emulated
device over the in-process NCCL stand-in — against the same four blocks linked inside one process (lbm_link_face +
lbm_step_group), which tests/test_gpu_blocks.py ties to the oracle and to the reference binary: bit for bit."""
import os
import sys
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(ROOT, "lattice-boltzmann-method_b200", "python"), os.path.join(ROOT, "tests")]
BUILD = os.path.join(HERE, "_build_asan" if os.environ.get("LBM_EMU_ASAN") == "1" else "_build")
os.environ["LBM_NCCL_LIB"] = os.path.join(BUILD, "libnccl_emu.so")

import numpy as np  # noqa: E402

import lbm_b200 as L  # noqa: E402

L.LIB_PATH = os.path.join(BUILD, "liblbm_b200_emu.so")
import cases  # noqa: E402


def main(Ln=64, steps=45):
    L.load()
    omega = 1.0 / 0.8
    rng = np.random.default_rng(3)
    w = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
    shapes = {"A": (Ln, Ln // 4), "B": (Ln // 4, Ln // 2), "C": (Ln, Ln // 4), "D": (Ln // 4, Ln // 2)}
    f0 = {k: w * (1.0 + 0.05 * rng.standard_normal(shapes[k] + (9,))) for k in cases.LOOP_BLOCKS}
    # one process: linked blocks
    dom = cases.loop_blocks(Ln, omega)
    for k in cases.LOOP_BLOCKS:
        dom[k].set_f(f0[k])
        dom[k].stats_start(3)
    L.step_group([dom[k] for k in cases.LOOP_BLOCKS], steps)
    want = {k: dom[k].get_f() for k in cases.LOOP_BLOCKS}
    want_stats = {k: dom[k].stats() for k in cases.LOOP_BLOCKS}
    for d in dom.values():
        d.close()
    # four "processes"
    sync = threading.Barrier(4)
    shared = {"id": None}
    got, got_stats, errors = {}, {}, []

    def worker(rank):
        try:
            if rank == 0:
                shared["id"] = L.comm_unique_id()
            sync.wait()
            d = cases.loop_block_on_rank(Ln, omega, rank, shared["id"])
            d.comm_faces_commit()
            d.bc_commit()
            k = cases.LOOP_BLOCKS[rank]
            d.set_f(f0[k])
            d.stats_start(3)  # each rank accumulates its own block
            d.step(steps // 2)
            mid = d.get_f()          # an export in the middle: the next step re-prepares the state (face tails of the current buffers)
            d.step(steps - steps // 2)
            got[k] = d.get_f()
            got_stats[k] = d.stats()
            assert np.isfinite(mid).all()
            sync.wait()
            d.close()
        except BaseException as e:  # noqa: BLE001
            errors.append(f"rank {rank}: {type(e).__name__}: {e}")
            sync.abort()

    threads = [threading.Thread(target=worker, args=(r,)) for r in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    ok = not errors and all(np.array_equal(got[k], want[k]) for k in cases.LOOP_BLOCKS)
    print("errors:", errors)
    print("blocks across ranks: bit-exact vs linked blocks =", ok)
    ok_stats = not errors and all(got_stats[k][0] == want_stats[k][0] == 15 and
                                  all(np.array_equal(a, b) for a, b in zip(got_stats[k][1:], want_stats[k][1:])) for k in cases.LOOP_BLOCKS)
    print("blocks across ranks: statistics record bit-exact vs linked blocks =", ok_stats)
    return 0 if ok and ok_stats else 1


if __name__ == "__main__":
    sys.exit(main())
