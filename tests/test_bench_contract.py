"""bench.py's contract: the reference arm (CPU, the oracle port) prints ONE JSON line with the keys a reader of the result
expects, both arms describe a workload with the same `config` object, and (GPU) the b200 arm times --steps steps and
dumps the outputs of its last one reproducibly."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "ttt2",
                          "--steps", "3", "--warmup", "3"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 3 and d["warmup"] == 3 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@pytest.mark.gpu
def test_steps_are_the_timed_steps_and_dumped_outputs_repeat(tmp_path):
    """Every measured leg times exactly --steps steps, and two runs with the same arguments dump the same outputs of
    the last timed step (float32 / float64, 64 MB at most) for every workload."""
    dumps = [tmp_path / "a", tmp_path / "b"]
    for d in dumps:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "7", "--warmup", "3", "--no-cpu",
                              "--dump-outputs", str(d)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout)
        for name, w in [("tron", line)] + list(line["workloads"].items()):
            assert w["steps"] == w["timed_steps"] == w["e2e"]["steps"] == 7
            assert (w["e2e"].get("copy_engine") or {"steps": 7})["steps"] == 7
            if name != "ttt2":                   # the step kernels' own count of the env-steps of the timed region
                assert w["env_steps_counted"] == w["n_gpus"] * w["config"]["batch_per_gpu"] * 7, name
    names = sorted(os.listdir(dumps[0]))
    assert names == sorted(os.listdir(dumps[1]))
    assert {n.split("_")[0] for n in names} == {"tron", "blokus", "ttt4", "ttt2"}
    assert sum(os.path.getsize(dumps[0] / n) for n in names) <= 64 << 20
    for n in names:
        a, b = np.load(dumps[0] / n), np.load(dumps[1] / n)
        assert a.dtype in (np.float32, np.float64) and a.shape == b.shape and np.array_equal(a, b), n


def test_both_arms_share_the_config_object():
    sys.path.insert(0, ROOT)
    import bench
    for name, wl in bench.WORKLOADS.items():
        cfg = bench.config_of(name, wl["B"])
        assert set(cfg) == {"workload", "batch_per_gpu", "policy"} and cfg["workload"] == wl["desc"]
    # BASELINE.json's configurations are all present: configs[0..3] as workloads, configs[4] = the same under torchrun
    assert bench.ORDER == ["tron", "blokus", "ttt4", "ttt2"]
