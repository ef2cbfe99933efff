"""bench.py's reference arm runs without a GPU: check the one-JSON-line contract and the keys the driver reads."""
import json
import os
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_exactly_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "nodes+verts/s"
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    mc = d["cpu_multicore"]  # the best-effort all-cores variant, reported next to the reference-shaped number
    assert mc["kind"] == "port-openmp" and mc["cores"] >= 1 and mc["value"] > 0


def test_c1_runs_whole_on_the_cpu():
    """BASELINE.json configs[0] (100k static nodes, 1 frustum, CPU only) is not sampled down."""
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--workload", "C1", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout)
    assert d["config"]["sample"].startswith("100000 nodes, 0 skinned meshes") and d["value"] > 0


def test_arguments_that_cannot_be_honoured_are_refused():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--workload", "tiny", *extra], capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and out.stdout.strip() == "", extra


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "tiny"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
