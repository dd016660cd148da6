"""CPU: bench.py's reference arm runs without a GPU and prints the JSON contract the driver parses."""
import json
import os
import subprocess
import sys

from helpers import ROOT


def test_reference_arm_json_contract():
    env = dict(os.environ, OMP_NUM_THREADS="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--passages", "3000",
                          "--steps", "1", "--warmup", "0", "--cpu-seconds", "1"],
                         capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"].split(" ")[0] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["sample_queries"] >= 2 and 0 < line["cpu_baseline"]["sample_fraction"] <= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]
    # both arms describe the workload with the SAME config object (one function builds it)
    sys.path.insert(0, ROOT)
    import types

    import bench
    args = types.SimpleNamespace(passages=3000, nd=180, nq=320, batch=16, k=5)
    assert line["config"] == bench.workload_config(args, 1)


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_plaid_cpu_baseline_leg_runs_on_a_small_sample():
    """bench.py's PLAID leg (restated IndexScorer.rank over the reference's compiled kernels where they were
    built, else over their restatements), CPU build."""
    import types

    sys.path.insert(0, ROOT)
    import bench
    from oracle import plaid_search as P
    args = types.SimpleNamespace(plaid_passages=1000, nd=60, nq=64, k=5, plaid_ndocs=16)
    out = bench.cpu_plaid_rate(args, "cpu", target_seconds=1.0)
    assert out["kind"] == ("reference" if P.have_reference_kernels() else "port")
    assert out["value"] > 0 and out["cores"] >= 1
    assert out["recall_at_5"] >= 0.9          # clustered data: PLAID finds the planted passage
    assert min(out["candidates_per_query"]) >= 16 and "NOT extrapolated" in out["sample"]
