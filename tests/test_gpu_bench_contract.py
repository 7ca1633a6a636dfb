"""GPU: bench.py prints ONE JSON line with every key of the measurement contract (both arms)."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", "6", "--warmup", "3",
                          "--e2e-steps", "4", "--cpu-seconds", "1", "--prime", "5", *extra],
                         cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_own_arm_line_has_every_contract_key():
    d = _run()
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 6 and d["warmup"] == 3 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["value"] > 0 and d["gpu_launches"] > 0 and "workload" in d["config"]
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} and d["e2e"]["h2d_bytes_per_step"] > 0
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
    assert set(d["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"} and d["cpu_baseline"]["kind"] == "port"
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs: the same arguments give the same arrays; one more timed step gives another state."""
    import numpy as np

    dumps = {}
    for name, steps in (("a", "6"), ("b", "6"), ("c", "7")):
        d = _run("--dump-outputs", str(tmp_path / name), "--steps", steps, "--no-cpu-baseline")
        assert d["steps"] == int(steps)
        files = sorted(os.listdir(tmp_path / name))
        dumps[name] = {f[:-4]: np.load(tmp_path / name / f) for f in files}
        assert sum(os.path.getsize(tmp_path / name / f) for f in files) <= 64 * 10 ** 6
    a, b, c = dumps["a"], dumps["b"], dumps["c"]
    assert sorted(a) == ["action", "done", "human_human_edge_rnn", "human_node_rnn", "reward", "robot_node", "spatial_edges",
                         "temporal_edges", "value"]
    assert all(v.dtype == np.float32 and v.shape[0] == 16 for v in a.values())
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert not np.array_equal(a["robot_node"], c["robot_node"])


def test_reference_arm_line():
    d = _run("--impl", "reference")
    assert d["impl"] == "reference" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
