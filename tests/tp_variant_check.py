"""Every two-phase kernel instantiation of a model against the plain k_tp_fused, bit for bit — helper of
tests/test_gpu_tp_variants.py for builds other than the one the suite loads.

With floating-point contraction off (liblbm_b200_nofma.so, `make NOFMA=1`) the eight (MRTCG) / nine (RK) instantiations of
tp_launch_fused are the same arithmetic in differently staged kernels and agree bit for bit; in the product build nvcc fuses
different multiply-adds in each and they part in the last bits.

As a script:  python tests/tp_variant_check.py --lib <path or suffix> mrtcg R C | rk L   -> exit 0 iff all bit-identical
TEST INFRASTRUCTURE."""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "lattice-boltzmann-method_b200", "python"))


def check(model, shape):
    """[(variant, first difference or None)] of every instantiation of `model` against the plain k_tp_fused"""
    import test_gpu_tp_variants as T

    ref = T.run(T.REFERENCE[model], shape)
    return [(name, T.first_difference(T.run(name, shape), ref)) for name in T.names_of(model) if name != T.REFERENCE[model]]


if __name__ == "__main__":
    import lbm_b200 as L

    argv = sys.argv[1:]
    if argv[:1] == ["--lib"]:
        L.LIB_PATH = argv[1] if "/" in argv[1] else os.path.join(L.PKG_DIR, f"liblbm_b200_{argv[1]}.so")
        argv = argv[2:]
    model, shape = argv[0], tuple(int(v) for v in argv[1:])
    bad = 0
    for name, diff in check(model, shape):
        print(f"{os.path.basename(L.LIB_PATH)} {name} {'x'.join(map(str, shape))}: " + (diff or "== k_tp_fused, bit for bit"))
        bad += diff is not None
    sys.exit(1 if bad else 0)
