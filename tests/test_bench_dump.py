"""bench.py writes nothing into the source tree (where it runs the tree may be read-only), and --dump-outputs writes the
last timed step's outputs as float64 .npy files that repeat bit for bit from run to run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--particles", "3000", "--beams", "90", "--grid", "300", "--steps", "2", "--warmup", "1"]


def run_bench(extra, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def tree_state():
    state = {}
    for d, dirs, files in os.walk(ROOT):
        dirs[:] = [x for x in dirs if x != ".git"]
        for f in files:
            st = os.lstat(os.path.join(d, f))
            state[os.path.relpath(os.path.join(d, f), ROOT)] = (st.st_size, st.st_mtime_ns)
    return state


def test_reference_arm_writes_nothing_into_the_tree():
    before = tree_state()
    out = run_bench(["--impl", "reference", *SMALL])
    assert out.returncode == 0, out.stderr[-2000:]
    assert tree_state() == before


@pytest.mark.parametrize("extra", [["--impl", "reference", "--dump-outputs", "unused"], ["--steps", "0"]])
def test_bad_arguments_are_refused(extra):
    out = run_bench([*SMALL, *extra])
    assert out.returncode == 2 and "error" in out.stderr
    assert not out.stdout.strip() and not os.path.exists(os.path.join(ROOT, "unused"))


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    before = tree_state()
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        out = run_bench([*SMALL, "--no-cpu-baseline", "--dump-outputs", str(d)])
        assert out.returncode == 0, out.stderr[-4000:]
        line = json.loads([s for s in out.stdout.splitlines() if s.startswith("{")][-1])
        assert line["steps"] == 2 and line["value"] > 0
        dumps.append(d)
    assert tree_state() == before
    shapes = {"estimate_mean": (4,), "estimate_cov": (3, 3), "weight_sum": (1,), "particle_states": (3000, 4), "particle_weights": (3000,)}
    assert sorted(os.listdir(dumps[0])) == sorted(name + ".npy" for name in shapes)
    for name, shape in shapes.items():
        a, b = (np.load(d / (name + ".npy")) for d in dumps)
        assert a.dtype == np.float64 and a.shape == shape, name
        assert np.array_equal(a, b), name
    states = np.load(dumps[0] / "particle_states.npy")
    assert np.allclose(np.hypot(states[:, 0], states[:, 1]), 1.0)  # (cos, sin, x, y) rows
