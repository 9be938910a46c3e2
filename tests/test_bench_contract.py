"""bench.py's JSON contract, checked on CPU through the reference arm (the oracle port timed on host cores)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=e, timeout=300)


def test_reference_arm_prints_one_contract_line():
    r = run("--impl", "reference", "--steps", "2", "--warmup", "1", "--rows", "8000000")
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "rows_per_s" and d["unit"] == "rows/s" and d["dtype"] == "u64"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "numbers_mt" in d["config"]["workload"]
    assert d["value"] > 0 and abs(d["ms_per_step"] * 1e-3 * d["value"] - 8_000_000) < 1e-3 * 8_000_000


def test_reference_arm_dumps_its_last_result(tmp_path):
    import numpy as np
    r = run("--impl", "reference", "--steps", "1", "--warmup", "0", "--rows", "8000000", "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 0, r.stderr
    res = np.load(tmp_path / "out" / "result.npy")
    assert res.dtype == np.float64 and res.tolist() == [3999999, 7999999, 0]


def test_steps_below_one_are_refused():
    r = run("--impl", "reference", "--steps", "0", "--rows", "8000000")
    assert r.returncode != 0 and "--steps" in r.stderr and r.stdout == ""


@pytest.mark.gpu
def test_timed_path_dumps_what_its_last_step_computed(tmp_path):
    """--dump-outputs: the query's row, the merged leaf states as exact u64 halves and the row count, after exactly --steps steps."""
    import numpy as np
    rows = 80_000_000
    r = run("--steps", "3", "--warmup", "1", "--rows", str(rows), "--no-query-table", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 3 and d["gpu_launches"] >= 3
    out = {n: np.load(tmp_path / "out" / f"{n}.npy") for n in ("result", "leaf_states_hi_lo", "rows")}
    assert all(a.dtype == np.float64 for a in out.values())
    s = (rows * (rows - 1) // 2) % (1 << 64)
    assert out["result"].tolist() == [s // rows, rows - 1, 0]
    assert [int(h) << 32 | int(l) for h, l in out["leaf_states_hi_lo"].tolist()] == [s, rows, rows - 1, 0]
    assert out["rows"].tolist() == [rows]


def test_reference_arm_is_silent_on_other_ranks():
    r = run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_committed_bench_lines_carry_the_contract_and_verified_results():
    """profiles/r02_bench_n{1,2,4,8}.json are the lines `bench.py --gpus N` printed on the GPU boxes (kept as evidence and as
    the source of the tables in DESIGN.md / BASELINE.md): every one parses, carries the contract's keys, and every per-query,
    GROUP BY and ORDER BY entry was asserted against its closed form inside the run (`verified`)."""
    import pytest
    seen = 0
    for n in (1, 2, 4, 8):
        p = os.path.join(ROOT, "profiles", f"r02_bench_n{n}.json")
        if not os.path.exists(p):
            continue
        lines = [l for l in open(p) if l.startswith("{")]
        assert len(lines) == 1, p
        d = json.loads(lines[0])
        seen += 1
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                  "data", "config", "roofline", "e2e", "gpu_launches", "clocks", "per_query", "group_by"):
            assert k in d, (n, k)
        assert d["n_gpus"] == n and d["metric"] == "rows_per_s" and d["dtype"] == "u64" and d["gpu_launches"] > 0
        assert d["config"]["rows_total"] == 10_000_000_000
        assert abs(d["value"] - d["config"]["rows_total"] / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
        r = d["roofline"]
        assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0.5 < r["frac"] < 1.2
        e = d["e2e"]
        assert e["h2d_bytes_per_step"] == 8 * e["rows_per_step"] and e["d2h_bytes_per_step"] > 0 and e["roofline"]["bound"] == "pcie"
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        for name, modes in d["per_query"].items():
            for mode, q in modes.items():
                assert q["verified"] is True and q["n_gpus"] == n, (n, name, mode)
        for name, g in d["group_by"].items():
            assert g["verified"] is True, (n, name)
        if n == 1:
            assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
            for name, o in d["order_by"].items():
                assert o["verified"] is True and o["sort_ms"] > o["limit_10_ms"] > 0, name
    if not seen:
        pytest.skip("no committed bench lines")
