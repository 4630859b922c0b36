"""bench.py contract checks that need no GPU: the reference arm prints exactly ONE JSON line with the agreed keys, and
non-zero ranks of a multi-rank reference launch exit quietly."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None):
    env = dict(os.environ, **(extra_env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "aligner_train_tokens_per_sec" and d["unit"] == "tokens/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["din"] == 3584 and d["config"]["d"] == 4096


def test_reference_arm_nonzero_rank_is_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_is_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr and r.stdout.strip() == ""


def test_dump_outputs_writes_float32_and_the_same_sample_of_a_large_array_every_time(tmp_path):
    import importlib.util

    import numpy as np
    import torch

    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = bench.DUMP_SAMPLE + 1000
    arrays = {"loss": torch.tensor(1.25), "mask": torch.ones(3, 5, dtype=torch.int64), "big": torch.arange(n, dtype=torch.float64),
              "w": torch.randn(7, 9).to(torch.bfloat16)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {d: {k: np.load(tmp_path / d / f"{k}.npy") for k in arrays} for d in ("a", "b")}
    assert sorted(p.name for p in (tmp_path / "a").iterdir()) == ["big.npy", "loss.npy", "mask.npy", "w.npy"]
    for k in arrays:
        assert got["a"][k].dtype == np.float32 and np.array_equal(got["a"][k], got["b"][k])
    assert got["a"]["loss"].shape == () and got["a"]["loss"] == 1.25
    assert got["a"]["mask"].shape == (3, 5) and (got["a"]["mask"] == 1).all()
    assert np.array_equal(got["a"]["w"], arrays["w"].float().numpy())
    big = got["a"]["big"]  # the values are their own flat indices: a sorted sample without repeats
    assert big.shape == (bench.DUMP_SAMPLE,) and (np.diff(big) > 0).all() and big[0] >= 0 and big[-1] < n
    large = torch.zeros(bench.DUMP_SAMPLE)
    too_many = {f"a{i}": large for i in range(bench.DUMP_LIMIT // (4 * bench.DUMP_SAMPLE) + 1)}
    with pytest.raises(ValueError, match="exceed the limit"):
        bench.dump_outputs(str(tmp_path / "c"), too_many)
    assert not (tmp_path / "c").exists()


def test_reference_arm_times_the_steps_asked_for_and_dumps_its_outputs(tmp_path):
    import numpy as np

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "9", "--warmup", "1",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    assert d["steps"] == 9 and d["warmup"] == 1 and "9 steps after 1 warm-up" in d["cpu_baseline"]["sample"]
    names = sorted(p.name for p in tmp_path.iterdir())
    assert names == ["loss.npy", "param.0.bias.npy", "param.0.weight.npy", "param.2.bias.npy", "param.2.weight.npy", "param.3.weight.npy"]
    loss = np.load(tmp_path / "loss.npy")
    assert loss.dtype == np.float32 and loss.shape == () and np.isfinite(loss) and loss > 0
    assert np.load(tmp_path / "param.0.bias.npy").shape == (4096,) and np.load(tmp_path / "param.0.weight.npy").shape == (1 << 22,)


def test_watchdog_aborts_a_run_that_does_not_finish():
    """bench.py arms a timer before any work (a hung peer wait or collective has no timeout of its own): when it fires the process
    says so on stderr and exits with status 4 instead of sitting there until the launcher's limit. Disabled with 0."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, TD_BENCH_WATCHDOG_S="0.5")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "8", "--warmup", "2"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 4 and "bench.py watchdog" in r.stderr and r.stdout.strip() == ""
