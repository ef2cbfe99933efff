"""bench.py --dump-outputs: the last timed frame's outputs are written as small float arrays, and a second run with the same
arguments writes the same arrays bit for bit (so two builds can be compared output for output)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--workload", "tiny", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-parity", "--no-device-animation"]


def _bench(out_dir):
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *ARGS, "--dump-outputs", str(out_dir)], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout)


@pytest.mark.timeout(1300)
def test_dump_outputs_are_small_float_arrays_that_repeat_exactly(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    line = _bench(a)
    _bench(b)
    assert line["steps"] == 2
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    assert {"global_matrices.npy", "world_aabbs.npy", "visible.npy", "visible_counts.npy", "palettes.npy", "skinned_positions.npy",
            "skinned_normals.npy"} <= set(names)
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype in (np.float32, np.float64), n
        assert x.shape == y.shape and x.tobytes() == y.tobytes(), n
    assert sum(os.path.getsize(a / n) for n in names) <= 64 << 20
    counts, vis = np.load(a / "visible_counts.npy"), np.load(a / "visible.npy")
    assert counts.shape == (6,) and (counts > 0).all() and vis.shape[1] == 6 and 0 < vis.mean() < 1
