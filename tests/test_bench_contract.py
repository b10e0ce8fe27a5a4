"""bench.py's reference arm runs on the CPU: check the JSON line it prints against the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--trees", "300", "--lights", "32"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "entities/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"].startswith("config#3 forest 300x255")
    assert d["config"]["entities_total"] == 300 * 255 + 32 and d["config"]["scaling"] == "strong"
    assert d["steps"] == 2 and d["warmup"] == 1                      # the arm honours --steps / --warmup exactly
    # both arms print the same `config` object: it is a function of the command line only
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--print-config", "--trees", "300", "--lights", "32"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert res.returncode == 0 and json.loads(res.stdout) == d["config"]
    for k in ("ms_per_step_median", "ms_per_step_min", "ms_per_step_max"):
        assert d["cpu_baseline"][k] > 0
    # ranks other than 0 print nothing and exit 0
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], env=env,
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert res.returncode == 0 and res.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_same_on_every_run(tmp_path):
    """--dump-outputs: the last timed step's results as float32 / float64 .npy files, under 64 MB, bit for bit the same on
    two runs with the same arguments; --steps sets the number of timed steps."""
    n = 300 * 255 + 32
    dumps = []
    for run in range(2):
        out = tmp_path / f"run{run}"
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "7", "--warmup", "3", "--trees", "300",
                              "--lights", "32", "--no-cpu-baseline", "--no-next-rows", "--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-3000:]
        d = json.loads(res.stdout.strip().splitlines()[-1])
        assert d["steps"] == 7 and d["parity_checked"] is True
        files = {p.stem: np.load(p) for p in sorted(out.glob("*.npy"))}
        assert all(a.dtype in (np.float32, np.float64) for a in files.values())
        assert sum(a.nbytes for a in files.values()) <= 64 << 20
        dumps.append(files)
    a, b = dumps
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].shape == b[k].shape and a[k].tobytes() == b[k].tobytes(), k
    assert np.array_equal(a["rows"], np.arange(n)) and a["global_transform"].shape == (n, 12)
    assert a["view_visibility"].any() and a["visible_count"].sum() > 0
    for v in range(4):
        assert len(a[f"visible_rows_view{v}"]) == a["visible_count"][v]
        assert a[f"cluster_offsets_view{v}"][-1] == a["cluster_index_count"][v] == len(a[f"cluster_indices_view{v}"])


def test_reference_arm_refuses_dump_outputs(tmp_path):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert res.returncode != 0 and "--dump-outputs" in res.stderr and not any(tmp_path.iterdir())


def test_b200_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True,
                         text=True, timeout=300, cwd=ROOT)
    assert res.returncode != 0 and "no CPU fallback" in (res.stderr + res.stdout)
