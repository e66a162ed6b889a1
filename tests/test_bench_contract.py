"""CPU: the reference arm of bench.py runs without a GPU and prints one JSON line with the contract's keys."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENV = dict(os.environ, PVB_BENCH_REF_BUDGET_S="3")      # the driver's run uses the full budget; the CPU tier a short one


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600,
                         cwd=ROOT, env=ENV)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "sdf_grad_queries_per_s" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    # the default line is the C4 RobotSDF headline, with the SAME config object the GPU arm prints ...
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.c4_config() and d["scaling"] == "strong"
    assert d["config"]["n_cfg"] == 200 and d["config"]["n_pts"] == 100_000
    # ... and carries every other BASELINE config next to it
    assert set(d["workloads"]) == set(bench.OTHER_WORKLOADS)
    for name, w in d["workloads"].items():
        assert w["value"] > 0 and w["cpu_baseline"]["cores"] >= 1, (name, w)


def test_reference_arm_single_workload():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--workload", "c2"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                         text=True, timeout=600, cwd=ROOT, env=ENV)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and "C2" in d["config"]["workload"] and "workloads" not in d


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(ENV, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--gpus", "2"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                         timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_sample(tmp_path):
    """--dump-outputs: a result over the byte budget is sampled along the point axis at the same indices in every run;
    one within it is written whole; float32 on disk."""
    sys.path.insert(0, ROOT)
    import bench
    import torch
    g = torch.Generator().manual_seed(1)
    val = torch.randn(200, 100_000, generator=g)
    grad = torch.randn(200, 100_000, 3, generator=g)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs((val, grad), str(d))
    v, gr = np.load(tmp_path / "a" / "value.npy"), np.load(tmp_path / "a" / "gradient.npy")
    assert v.dtype == np.float32 and gr.dtype == np.float32
    assert v.nbytes + gr.nbytes <= bench.DUMP_MAX_BYTES <= 64 << 20
    k = v.shape[1]
    assert v.shape == (200, k) and gr.shape == (200, k, 3) and k > 10_000
    assert np.array_equal(np.load(tmp_path / "b" / "value.npy"), v)
    assert np.array_equal(np.load(tmp_path / "b" / "gradient.npy"), gr)
    # the sample is one set of point columns: each column of the dump is a column of the result, in index order
    cols = [int(np.flatnonzero((val[0].numpy() == v[0, j]))[0]) for j in (0, k // 2, k - 1)]
    assert cols == sorted(cols)
    for j, c in zip((0, k // 2, k - 1), cols):
        assert np.array_equal(v[:, j], val[:, c].numpy()) and np.array_equal(gr[:, j], grad[:, c].numpy())
    small = torch.arange(12, dtype=torch.float64)
    bench.dump_outputs(small, str(tmp_path / "c"))
    assert np.array_equal(np.load(tmp_path / "c" / "value.npy"), small.numpy())
    assert not (tmp_path / "c" / "gradient.npy").exists()


def test_committed_ncu_side_files_cover_every_workload():
    """roofline.traffic / roofline.ncu are read from committed ncu extracts: every bench workload has an entry, the
    summaries they cite exist, and the numbers are sane (bytes > 0, percentages in (0, 100])."""
    sys.path.insert(0, ROOT)
    import bench
    names = {bench.HEADLINE, *bench.OTHER_WORKLOADS}
    traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    limits = json.load(open(os.path.join(ROOT, "profiles", "ncu_limits.json")))
    assert names <= set(traffic) and names <= set(limits)
    for n in names:
        assert traffic[n] > 0 and bench.ncu_traffic(n) == traffic[n]
        lim = bench.ncu_limits(n)
        assert os.path.exists(os.path.join(ROOT, lim["source"])), lim["source"]
        for k in ("issue_slots_pct", "l1_data_pipe_pct", "dram_pct", "warps_active_pct"):
            assert 0.0 < lim[k] <= 100.0, (n, k, lim[k])
