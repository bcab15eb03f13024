"""CPU: the reference arm of bench.py (`--impl reference`) prints ONE JSON line with the contract's
keys; under torchrun ranks other than 0 print nothing and exit 0."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--ref-seconds", "1"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                         text=True, env=env, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    return res.stdout.strip()


def test_reference_arm_line():
    out = _run({"RANK": "0", "WORLD_SIZE": "2"})
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 2 and d["steps"] == 1 and d["warmup"] == 0 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["metric"].startswith("STFT frames/sec (nfft=2048,hop=512,npks=50)")
    for k in ("workload", "sr", "nfft", "hop", "npks"):
        assert k in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None


def test_reference_arm_other_ranks_are_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2"}) == ""


def test_dump_outputs_sampled_within_budget(tmp_path):
    """--dump-outputs: float64 files, a fixed seeded row sample of arrays over their share of the budget,
    identical from call to call."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    tab = torch.arange(5000 * 4, dtype=torch.float64).reshape(5000, 4)
    arrays = {"tab": tab, "ids": tab.to(torch.int32), "small": torch.arange(10, dtype=torch.float32)}
    budget = 3 * 8 * 4 * 1000                            # 1000 rows of [*, 4] per array
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget)
    a = {k: np.load(str(tmp_path / "a" / (k + ".npy"))) for k in arrays}
    assert all(v.dtype == np.float64 for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= budget
    assert a["tab"].shape == (1000, 4) and np.array_equal(a["tab"], a["ids"])
    rows = a["tab"][:, 0] / 4
    assert np.all(np.diff(rows) > 0) and np.array_equal(a["tab"], tab.numpy()[rows.astype(int)])
    assert np.array_equal(a["small"], np.arange(10))
    for k in arrays:
        assert np.array_equal(np.load(str(tmp_path / "b" / (k + ".npy"))), a[k])


def test_bench_rejects_zero_steps_and_unsupported_dumps(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)],
                  ["--workload", "cfg3", "--dump-outputs", str(tmp_path)]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, stdout=subprocess.PIPE,
                             stderr=subprocess.PIPE, text=True, timeout=120)
        assert res.returncode == 2 and res.stdout == "", (extra, res.stderr)
