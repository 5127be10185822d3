"""bench.py contract checks: the reference arm's JSON line, the static structure of our arm's line and --dump-outputs (its last
check runs our arm on the GPU)."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_json_line():
    env = dict(os.environ, PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--workload", "cartpole_rn"], env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "se_env_steps_per_s" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    # the unmodified reference when it is staged (oracle/make_ref.py -> oracle/_ref/pyref) with the C port as a second figure,
    # else the port alone
    assert cb["kind"] in ("reference", "port") and 1 <= cb["cores"] <= (os.cpu_count() or 1) and cb["value"] == d["value"] and "sample" in cb
    if cb["kind"] == "reference":
        assert cb["port"]["kind"] == "port" and cb["port"]["value"] > 0 and d["nes_generations_per_hour"] > 0 and d["nes_population"] == 16
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_nonzero_ranks():
    env = dict(os.environ, PYTHONPATH=ROOT, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], env=env, cwd=ROOT,
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_our_arm_line_carries_every_contract_key():
    """Static check of bench.py's source: the keys of the JSON line our arm prints (needs a GPU to run)."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    body = src[src.index("def measure_nes("):]
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert re.search(r'"%s":' % key, body) or re.search(r'res\["%s"\] =' % key, body), key
    assert 'line["cpu_baseline"] =' in body
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert re.search(r'"%s":' % key, body[body.index('"roofline"'):]), key
    assert "no CPU fallback" in src           # our arm refuses to run without a CUDA device


def test_dump_outputs_writes_float_arrays_within_the_size_limit(tmp_path, monkeypatch):
    """--dump-outputs: float32 kept, other dtypes as float64, the directory within DUMP_BYTES, and an array that does not fit cut
    to the same seeded row sample every time."""
    import bench
    import numpy as np
    monkeypatch.setattr(bench, "DUMP_BYTES", 16 << 10)
    big = np.arange(8192, dtype=np.float32).reshape(-1, 16)                   # 32 KB, twice the budget
    arrays = {"lane_train_steps": np.arange(5, dtype=np.int64), "score": np.linspace(0, 1, 5), "big": big}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    a, b = tmp_path / "a", tmp_path / "b"
    assert sorted(p.name for p in a.iterdir()) == ["big.npy", "big_rows.npy", "lane_train_steps.npy", "score.npy"]
    steps = np.load(a / "lane_train_steps.npy")
    assert steps.dtype == np.float64 and steps.tolist() == [0, 1, 2, 3, 4]
    assert np.load(a / "score.npy").dtype == np.float64
    sample, rows = np.load(a / "big.npy"), np.load(a / "big_rows.npy").astype(np.int64)
    assert sample.dtype == np.float32 and sample.shape[0] > 100 and np.array_equal(sample, big[rows])
    assert np.array_equal(rows, np.load(b / "big_rows.npy")) and np.array_equal(sample, np.load(b / "big.npy"))
    assert sum(p.stat().st_size for p in a.iterdir()) <= bench.DUMP_BYTES


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], cwd=ROOT, capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_step_and_repeat_exactly(tmp_path):
    """With one timed step the dumped lane results are that step's: their train steps are the JSON line's value x time.  A second
    run with the same arguments writes the same arrays bit for bit."""
    import numpy as np
    lines = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cartpole_se_pop16", "--steps", "1", "--warmup",
                              "1", "--extras", "none", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run)], cwd=ROOT,
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        lines.append(json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1]))
    d, a, b = lines[0], tmp_path / "a", tmp_path / "b"
    steps = np.load(a / "lane_train_steps.npy")
    assert steps.shape == (48,) and steps.dtype == np.float64 and steps.min() > 0
    assert abs(steps.sum() - d["value"] * d["ms_per_step"] * 1e-3) <= 1e-6 * steps.sum()
    theta = np.load(a / "env_theta.npy")
    assert theta.dtype == np.float32 and theta.shape[0] == 48 and np.isfinite(theta).all()
    assert np.allclose(theta[1] + theta[2], 2 * theta[0], atol=1e-6)          # member 0: theta, theta + eps, theta - eps
    names = sorted(p.name for p in a.iterdir())
    assert names == sorted(p.name for p in b.iterdir()) and len(names) >= 11
    for n in names:
        assert np.array_equal(np.load(a / n), np.load(b / n)), n
