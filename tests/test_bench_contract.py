"""The driver-facing contract of bench.py.  CPU: the reference arm prints ONE JSON line with the required keys,
and under a multi-rank launch only rank 0 speaks.  GPU: --steps and --dump-outputs."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def test_reference_arm_json_line():
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                                   "--warmup", "1", "--scale", "0.05"], text=True, timeout=600)
    lines = [ln for ln in out.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert REQUIRED <= set(d)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and "workload" in d["config"]
    # both arms print the SAME config object (the driver compares them): built by one function
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(0.05)
    assert d["cpu_baseline_1thread"]["cores"] == 1 and d["cpu_baseline"]["cores"] == bench.usable_threads()
    assert d["sample_pods_per_step"] == d["config"]["pods_per_gpu"]   # the whole snapshot per step


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_round(tmp_path, oracle):
    # --steps sets the timed step count exactly; --dump-outputs writes the last round, which must be the oracle's round
    # of the same seeded snapshot
    scale = 0.05
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1",
                                   "--scale", str(scale), "--no-cpu-baseline", "--no-replay", "--no-objects",
                                   "--dump-outputs", str(tmp_path)], text=True, timeout=600)
    d = json.loads([ln for ln in out.splitlines() if ln.strip()][-1])
    assert d["steps"] == 3 and d["steps_requested"] == 3
    got = {f[:-4]: np.load(os.path.join(str(tmp_path), f)) for f in os.listdir(str(tmp_path))}
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    sys.path.insert(0, ROOT)
    import bench
    snap = importlib.import_module("batch-scheduler_b200.snapshot").config(bench.WORKLOAD_CFG, scale)
    ref = oracle.round(snap, want_bitmap=True, want_score=True)
    for k in ("prefilter", "feasible_count", "best_node", "best_score", "admit", "admit_bitmap", "new_denied", "order",
              "rank"):
        np.testing.assert_array_equal(got[k], getattr(ref, k).astype(np.float64), err_msg=k)
    assert got["max_group"][0] == ref.max_group and got["max_finished"][0] == ref.max_finished
    rows = got["pod_sample"].astype(np.int64)
    assert len(rows) == min(snap.pods.n, bench.DUMP_SAMPLE_PODS)
    np.testing.assert_array_equal(got["score_rows"], ref.score[rows].astype(np.float64))
    np.testing.assert_array_equal(got["fit_bitmap_rows"], ref.fit_bitmap[rows].astype(np.float64))


def test_reference_arm_other_ranks_are_silent():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                                   "--steps", "1", "--warmup", "0"], text=True, timeout=120, env=env)
    assert out.strip() == ""
