"""CPU: the JSON line of `bench.py --impl reference` (the only arm that runs without a GPU) carries every key of the
measurement contract, for the default workload and for the others; and the B200 arm refuses to run without a device
instead of falling back to anything."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "cpu_baseline", "e2e", "impl"}


def run(args, timeout=600):
    return subprocess.run([sys.executable, "bench.py"] + args, cwd=ROOT, capture_output=True, text=True, timeout=timeout)


@pytest.mark.parametrize("workload", [None, "cylinder_bb", "poiseuille", "kbc_shear", "csf_rt"])
def test_reference_arm_line(workload):
    args = ["--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-sample", "64"]
    if workload:
        args += ["--workload", workload]
    r = run(args)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["impl"] == "reference" and d["metric"] == "MLUPS" and d["unit"] == "MLUPS" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


@pytest.mark.gpu
def test_dump_outputs_hold_the_state_after_exactly_warmup_plus_steps(tmp_path):
    """--dump-outputs writes the headline's state after the timed block: two runs with the same number of warm-up + timed
    steps write the same arrays, one more timed step changes them (warm-ups of at least 4: this grid replays a CUDA graph)"""
    import numpy as np

    if os.environ.get("LBM_EMU") == "1":
        pytest.skip("bench.py's B200 arm needs a real device")
    X, Y = 96, 64
    dumps = []
    for warmup, steps in ((6, 3), (5, 4), (5, 5)):
        out = tmp_path / f"w{warmup}_k{steps}"
        r = run(["--steps", str(steps), "--warmup", str(warmup), "--X", str(X), "--Y", str(Y), "--no-others", "--no-cpu-baseline",
                 "--no-e2e", "--dump-outputs", str(out)])
        assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
        d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert d["steps"] == steps and d["timing"]["blocks"] == 1
        dumps.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    shapes = {"f0": (X * Y, 9), "rho": (X * Y, 1), "u": (X * Y, 2)}
    assert {k: v.shape for k, v in dumps[0].items()} == shapes and all(v.dtype == np.float64 for v in dumps[0].values())
    relerr = lambda a, b: float(np.abs(a - b).max() / np.abs(b).max())  # noqa: E731
    assert all(relerr(dumps[1][k], dumps[0][k]) < 1e-12 for k in shapes)
    assert relerr(dumps[2]["u"], dumps[0]["u"]) > 1e-9


def test_b200_arm_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = run(["--steps", "1", "--warmup", "1"], timeout=300)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stdout + r.stderr)
