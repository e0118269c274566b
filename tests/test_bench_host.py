"""Host-side contract of bench.py (no GPU): sharding rule, the config object both arms print, and the reference arm end to end
(the oracle port timed on the host cores, one bounded step)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    sys.path.insert(1, ROOT)
    import bench
    return bench


def test_strong_and_weak_shards():
    b = _bench()
    for world in (1, 2, 3, 8):
        parts = [b.shard(200, r, world, "strong") for r in range(world)]
        assert sorted(k for p in parts for k in p) == list(range(200))                       # the sweep's 200 episodes, each exactly once
        assert max(map(len, parts)) - min(map(len, parts)) <= 1
        assert parts[0][:3] == [0, world, 2 * world]                                          # k = r mod W, the rule of driver.shard
        weak = [b.shard(200, r, world, "weak") for r in range(world)]
        assert all(len(p) == 200 for p in weak) and len({k for p in weak for k in p}) == 200 * world


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference`: ONE JSON line, same metric / unit / config object as the native arm, cpu_baseline describing the run, e2e with no copies"""
    b = _bench()
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == b.METRIC and d["unit"] == "solves/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["scaling"] == "strong" and d["vs_baseline"] is None
    assert d["config"] == b.line_config("strong")                                             # identical to the native arm's config object
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_writes_float32_and_samples_rows_above_the_cap(tmp_path):
    """--dump-outputs: one float32 .npy per array; above the byte cap every array keeps the same seeded rows, listed in rows.npy"""
    import numpy as np
    b = _bench()
    rng = np.random.default_rng(1)
    arrays = {"cvar_cx": rng.normal(size=(200, 11)).astype(np.float32), "cvar_cost_obs": rng.normal(size=200).astype(np.float32)}
    assert b.write_outputs(str(tmp_path / "all"), arrays) == ["cvar_cost_obs", "cvar_cx"]
    for k, v in arrays.items():
        got = np.load(tmp_path / "all" / (k + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, v)
    cap = 2000
    names = [b.write_outputs(str(tmp_path / d), arrays, cap=cap) for d in ("a", "b")]
    assert names[0] == names[1] == ["cvar_cost_obs", "cvar_cx", "rows"]
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    assert sum((tmp_path / "a" / (k + ".npy")).stat().st_size - 128 for k in names[0]) <= cap
    r = rows.astype(int)
    assert len(r) > 0 and np.all(np.diff(r) > 0)
    for k, v in arrays.items():
        assert np.array_equal(np.load(tmp_path / "a" / (k + ".npy")), v[r])


def test_bad_arguments_are_refused():
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and out.stdout.strip() == "", (argv, out.stderr[-500:])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
