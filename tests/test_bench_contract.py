"""CPU: the reference arm of bench.py (`--impl reference`: the oracle port of the reference's CPU path on the host cores) runs
without a GPU and prints exactly ONE JSON line on stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-rows", "400000"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "rows/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"].startswith("rows/sec windowed group-agg") and d["config"]["workload"].startswith("cfg2")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1


def test_non_zero_ranks_of_the_reference_arm_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == "", (out.stdout, out.stderr[-1000:])


def test_e2e_step_plan_fits_the_device():
    """bench.py runs every e2e step through its own operator (~9 GB each for cfg 2): the number of steps follows the free device
    memory, with the driver's --steps 20 --warmup 5 as the case that used to need 26 operators."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
    assert b.plan_e2e_steps(11, 5, 20, 1) == (3, 7)          # 11 operators fit: 3 warm-ups + 7 timed + the parity pass
    assert b.plan_e2e_steps(40, 5, 20, 1) == (3, 20)
    assert b.plan_e2e_steps(9, 3, 5, 1) == (3, 5)
    assert b.plan_e2e_steps(3, 5, 20, 1) == (1, 1)
    for fit in range(3, 30):
        for par in (0, 1):
            w, s = b.plan_e2e_steps(fit, 5, 20, par)
            assert w >= 1 and s >= 1 and w + s + par <= max(fit, 2 + par)


def test_dump_outputs_is_independent_of_emission_order(tmp_path):
    """bench.py --dump-outputs: the same rows emitted in a different order and split into different polls write the same files,
    sorted by (window start, key), with NULL keys and NULL aggregates kept apart; above DUMP_ROWS rows a fixed sample is written."""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
    assert 7 * 8 * b.DUMP_ROWS <= 64 << 20
    rng = np.random.default_rng(5)
    rows = [(ws, key, int(rng.integers(1, 9)), float(rng.normal()), float(rng.normal()), float(rng.normal()))
            for ws in (3000, 1000, 2000) for key in (b"sensor_9", b"sensor_10", None, b"k")]
    rows[5] = rows[5][:2] + (0, None, None, None)

    def parts(order, splits):
        out = []
        for chunk in np.array_split(np.array(order), splits):
            rs = [rows[i] for i in chunk]
            kb = b"pad" + b"".join(r[1] or b"" for r in rs)
            off = np.cumsum([3] + [len(r[1] or b"") for r in rs]).astype(np.int32)
            out.append({"key_off": off, "key_bytes": np.frombuffer(kb, np.uint8), "key_valid": np.array([r[1] is not None for r in rs], np.uint8),
                        "count": np.array([r[2] for r in rs], np.int64), "min": np.array([r[3] or 0.0 for r in rs]),
                        "max": np.array([r[4] or 0.0 for r in rs]), "avg": np.array([r[5] or 0.0 for r in rs]),
                        "agg_valid": np.array([r[3] is not None for r in rs], np.uint8),
                        "window_start": np.array([r[0] for r in rs], np.int64), "window_end": np.array([r[0] + 1000 for r in rs], np.int64)})
        return out
    n = len(rows)
    assert b.dump_outputs(str(tmp_path / "a"), parts(range(n), 3)) == (n, n)
    assert b.dump_outputs(str(tmp_path / "b"), parts(rng.permutation(n), 5)) == (n, n)
    names = ["window_start_ms", "window_end_ms", "key_id", "count", "min", "max", "avg"]
    got = {c: np.load(tmp_path / "a" / f"{c}.npy") for c in names}
    for c in names:
        assert got[c].dtype == np.float64 and np.array_equal(got[c], np.load(tmp_path / "b" / f"{c}.npy"), equal_nan=True), c
    assert list(got["window_start_ms"]) == [1000.0] * 4 + [2000.0] * 4 + [3000.0] * 4
    assert list(got["key_id"][:4]) == [0.0, 1.0, 2.0, -1.0]          # b"k" < b"sensor_10" < b"sensor_9", NULL last
    null_row = (got["window_start_ms"] == 1000.0) & (got["key_id"] == 1.0)         # rows[5]: window 1000, b"sensor_10"
    assert got["count"][null_row] == 0 and np.isnan(got["min"][null_row]).all()
    b.DUMP_ROWS = 5
    assert b.dump_outputs(str(tmp_path / "c"), parts(range(n), 2)) == (n, 5)
    assert b.dump_outputs(str(tmp_path / "d"), parts(rng.permutation(n), 4)) == (n, 5)
    for c in names:
        assert np.array_equal(np.load(tmp_path / "c" / f"{c}.npy"), np.load(tmp_path / "d" / f"{c}.npy"), equal_nan=True), c
