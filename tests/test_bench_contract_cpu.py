"""bench.py's contract, as far as it can be checked without a GPU: the reference arm (`--impl reference`) runs on host cores
only, prints exactly ONE JSON line on stdout and carries the keys the driver reads; under a 2-rank launch only rank 0 speaks."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
        "data", "config", "cpu_baseline", "e2e")


def _run(extra_env=None, gpus=1):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    env.update(extra_env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", str(gpus), "--steps", "2",
                        "--warmup", "1", "--ref-corridors", "8"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-800:]
    return [ln for ln in p.stdout.splitlines() if ln.strip()]


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = _run()
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in BASE:
        assert k in d, k
    assert d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert "cfg4" in d["config"]["workload"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["unit"] == d["unit"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] / 1e3 - 8 * 1024) < 1e-6 * 8 * 1024      # 8 corridors x 1024 pairs per step


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, gpus=2) == []


def test_dump_outputs_writes_float_arrays_within_the_budget(tmp_path, monkeypatch):
    """--dump-outputs: flags as float32, the rest as float64, one file per array; above the budget every array keeps the same
    seeded sample of its rows, identical from run to run."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(1)
    arrays = {"feasible": rng.integers(0, 2, 1000).astype(np.uint8), "cost": rng.normal(size=1000),
              "index": np.arange(1000, dtype=np.int32), "R": rng.normal(size=(1000, 9))}
    bench.dump_outputs(str(tmp_path / "full"), arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / "full" / (k + ".npy"))
        assert got.dtype == (np.float32 if k == "feasible" else np.float64) and np.array_equal(got, v)
    monkeypatch.setattr(bench, "DUMP_BYTES", 20000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    out = {k: np.load(tmp_path / "a" / (k + ".npy")) for k in arrays}
    assert sum(v.nbytes for v in out.values()) <= 20000 and len(out["cost"]) > 100
    rows = out["index"].astype(int)
    assert np.all(np.diff(rows) > 0) and np.array_equal(out["cost"], arrays["cost"][rows]) and np.array_equal(out["R"], arrays["R"][rows])
    assert all(np.array_equal(out[k], np.load(tmp_path / "b" / (k + ".npy"))) for k in arrays)
    arrays["cost"][7] = np.inf
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path / "c"), arrays)


def test_pair_outputs_write_no_result_entries_as_zero(tmp_path):
    """Costs of infeasible candidates (+inf), cost and dt of a sweep without a winner (+inf, nan), R without a whole winner
    (nan): 0 in the dump, every other entry as the library returned it."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from faster_b200 import capi
    feas = np.array([1, 0, 1, 0], np.uint8)
    cost = np.array([2.5, np.inf, 3.5, np.inf])
    res = np.zeros(2, capi.PAIR_RESULT_DTYPE)
    res["whole_dt_index"], res["safe_dt_index"] = [1, -1], [-1, -1]
    res["whole_cost"], res["whole_dt"], res["safe_cost"], res["safe_dt"] = [4.0, np.inf], [0.3, np.nan], np.inf, np.nan
    res["R"][0], res["R"][1], res["safe_dt_base"] = 1.5, np.nan, [0.2, np.nan]

    class Batch:
        out = {"feasible_whole": torch.from_numpy(feas), "cost_whole": torch.from_numpy(cost),
               "feasible_safe": torch.from_numpy(feas[::-1].copy()), "cost_safe": torch.from_numpy(cost[::-1].copy())}

        def results(self, capi):
            return res
    out = bench.pair_outputs([Batch()], capi)
    assert np.array_equal(out["cost_whole"], [2.5, 0, 3.5, 0]) and np.array_equal(out["cost_safe"], [0, 3.5, 0, 2.5])
    assert np.array_equal(out["result_whole_cost"], [4.0, 0]) and np.array_equal(out["result_whole_dt"], [0.3, 0])
    assert not out["result_safe_cost"].any() and not out["result_safe_dt"].any()
    assert np.array_equal(out["result_R"], [[1.5] * 9, [0] * 9]) and np.array_equal(out["result_safe_dt_base"], [0.2, 0])
    bench.dump_outputs(str(tmp_path), out)
    assert all(np.isfinite(np.load(tmp_path / (k + ".npy"))).all() for k in out)


def test_bad_arguments_are_refused():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=600,
                           env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), cwd=ROOT)
        assert p.returncode == 2 and p.stdout.strip() == "", p.stderr


def test_gpu_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: without a CUDA device the product arm exits non-zero and says why; nothing is printed on stdout."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                       timeout=600, env=env, cwd=ROOT)
    assert p.returncode != 0 and "CUDA" in p.stderr and p.stdout.strip() == ""
