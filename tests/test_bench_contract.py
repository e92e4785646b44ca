"""The driver's contract with bench.py, as far as it can be held without a GPU: the reference arm (`--impl reference`: the
CPU oracle timed on the host cores) prints exactly one JSON line on stdout with the keys the driver reads, on the same
workload description as the GPU arm, and the `--models` knob shows in it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1", "--steps", "2",
                          "--warmup", "1", *extra], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                      # stdout carries the result line and nothing else
    return json.loads(lines[0])


def test_reference_arm_line_has_the_contract_keys():
    d = _run()
    assert d["impl"] == "reference" and d["metric"] == "task_x_worker_cost_evaluations_per_sec" and d["unit"] == "evals/s"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["data"].startswith("synthetic") and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("cfg1") and d["config"]["n_asks"] == 1000 and d["config"]["n_workers"] == 10000
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert cb["cores"] == cb["host_cpus"]["threads"] <= cb["host_cpus"]["affinity"]      # the threads it really ran on
    assert d["gpu_launches"] == 0


def test_models_knob_shows_in_the_workload():
    d = _run("--models", "200")
    assert "200 distinct worker model strings" in d["config"]["workload"]


def _dumped(out_dir):
    got = {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}
    assert all(v.dtype == np.float64 and v.ndim == 1 for v in got.values())
    return got


def test_reference_arm_dumps_what_its_last_step_computed(tmp_path):
    """--dump-outputs on the reference arm: the oracle's all-pairs statistics of the timed sample (cfg1: every ask)."""
    from oracle import pm_oracle as orc

    _run("--dump-outputs", str(tmp_path))
    got = _dumped(tmp_path)
    assert sorted(got) == ["ask_best_cost", "ask_best_worker", "ask_count", "worker_first_ask"]
    w, a, (bits, npat, nmod, words), (T, W, Wg, desc) = bench.make_tables("cfg1", 1)
    ev = orc.soa_eval_matrix(w.a, w.b, a.asks, a.opts, bits, words, 0, T, 0, W, threads=4)
    packed = got["ask_best_cost"].astype(np.int64) * (1 << 32) + got["ask_best_worker"].astype(np.int64)
    assert np.array_equal(packed, ev["row_best"])
    assert np.array_equal(got["ask_count"], ev["row_count"]) and np.array_equal(got["worker_first_ask"], ev["col_first"])


def test_dump_keeps_the_same_seeded_sample_within_budget(tmp_path):
    """Outputs larger than the budget: every long array keeps the same positions each run, and its positions are written."""
    big = np.arange(50_000, dtype=np.uint32)[::-1].copy()
    arrays = {"big": big, "none": np.full(3, 0xFFFFFFFF, dtype=np.uint32), **bench.split_best(np.array([-1, (5 << 32) | 7]))}
    budget = 60_000
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, budget=budget)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= budget
    a, b = _dumped(tmp_path / "a"), _dumped(tmp_path / "b")
    assert sorted(a) == sorted(b) == ["ask_best_cost", "ask_best_worker", "big", "big_index", "none"]
    assert all(np.array_equal(a[k], b[k]) for k in a)
    idx = a["big_index"].astype(np.int64)
    assert 0 < len(idx) < len(big) and np.all(np.diff(idx) > 0) and np.array_equal(a["big"], big[idx])
    assert np.array_equal(a["none"], [0xFFFFFFFF] * 3)                           # PM_NONE survives exactly
    assert np.array_equal(a["ask_best_cost"], [-1, 5]) and np.array_equal(a["ask_best_worker"], [0xFFFFFFFF, 7])


@pytest.mark.gpu
def test_gpu_arm_dumps_the_result_of_its_last_timed_pass(tmp_path):
    """--dump-outputs on the CUDA arm: the arrays Engine.fetch() returns after the timed passes, on the seeded cfg1 tables."""
    from protocol_b200 import abi
    from protocol_b200.engine import Engine

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", "2", "--warmup", "3",
                          "--no-cpu", "--no-extras", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    got = _dumped(tmp_path)
    w, a, (bits, npat, nmod, words), _ = bench.make_tables("cfg1", 1)
    eng = Engine()
    eng.set_asks(a.asks, a.opts)
    eng.set_model_table(bits, npat, nmod, words)
    eng.set_workers(w.a, w.b)
    eng.match(abi.PM_MODE_FIRST_FIT | abi.PM_PATH_MATERIALIZED)
    r = eng.fetch()
    eng.close()
    want = {"worker_group": r.worker_group, "worker_ask": r.worker_ask, "group_ask": r.group_ask, "group_off": r.group_off,
            "group_members": r.group_members, **bench.split_best(r.ask_best), "ask_count": r.ask_count}
    assert sorted(got) == sorted(want)
    for k, v in want.items():
        assert np.array_equal(got[k], v), k
