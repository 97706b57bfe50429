"""bench.py's reference arm on CPU (the only arm that runs without a GPU): one JSON line with the contract's
keys; non-zero ranks stay silent and exit 0.  Uses the single-prompt workload so that it takes seconds."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1prompt",
                           "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "motions/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "motions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["cpu_sample_motions"] >= 1


def test_reference_arm_other_ranks_are_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_output_is_a_fixed_sample_within_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT", 200_000)
    x = torch.arange(64 * 100 * 66, dtype=torch.float32).reshape(64, 100, 22, 3)        # 1.7 MB of motions
    for d in ("a", "b"):
        bench.dump_output(str(tmp_path / d), "joints", x, 0)
    a, b = np.load(tmp_path / "a" / "joints.npy"), np.load(tmp_path / "b" / "joints.npy")
    assert os.path.getsize(tmp_path / "a" / "joints.npy") <= 200_000 and np.array_equal(a, b)
    assert a.dtype == np.float32 and a.shape[1:] == (100, 22, 3) and 0 < a.shape[0] < 64
    rows = a[:, 0, 0, 0] / (100 * 66)                                                     # whole motions, in order
    assert (np.diff(rows) > 0).all() and np.array_equal(a, x.numpy()[rows.astype(int)])
    bench.dump_output(str(tmp_path / "c"), "motion", x[:2], 0)                         # small: written whole
    assert np.array_equal(np.load(tmp_path / "c" / "motion.npy"), x[:2].numpy())


def test_bad_arguments_are_refused():
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                           timeout=60, cwd=ROOT)
        assert r.returncode == 2 and r.stdout == "", r.stderr[-500:]
