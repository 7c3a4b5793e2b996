"""bench.py prints exactly one JSON line with the keys the driver relies on (both arms)."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _run(*args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], capture_output=True, text=True,
                         timeout=timeout, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = out.stdout.strip().splitlines()          # nothing but the JSON line may reach stdout (library banners go to stderr)
    assert len(lines) == 1 and lines[0].startswith("{"), out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line_small_workload():
    """--impl reference runs without a GPU (oracle port on the host cores)."""
    d = _run("--impl", "reference", "--workload", "small", "--steps", "2", "--warmup", "1")
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["unit"] == "queries/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "workload" in d["config"]


def test_step_counts_and_dump_option_are_checked():
    for args, why in ((("--steps", "0"), "must be >= 1"), (("--warmup", "-1"), "must be >= 0"),
                      (("--dump-outputs", "out"), "--impl reference has none to write")):
        out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--workload", "small",
                              *args], capture_output=True, text=True, timeout=120, cwd=REPO)
        assert out.returncode == 2 and why in out.stderr, (args, out.stderr[-2000:])


def test_dump_outputs_types_sample_and_limit(tmp_path, monkeypatch):
    """bench.dump_outputs: float32 / float64 files, integers exact, packed keys and status left out, a seeded row
    sample (the same rows every time) once there are more queries than DUMP_QUERIES, and the size limit."""
    import numpy as np
    import torch
    sys.path.insert(0, REPO)
    import bench
    n = 40
    res = {"top_idx": torch.arange(n * 3, dtype=torch.int64).reshape(n, 3) + 2 ** 40,
           "top_scores": torch.linspace(-1, 1, n * 3).reshape(n, 3), "pred_vote": torch.arange(n, dtype=torch.int32),
           "hit_counts": torch.tensor([[5, 7]]), "keys": torch.zeros(n, 3, dtype=torch.int64),
           "status": torch.zeros(4, dtype=torch.int32), "precision": "rescore"}
    bench.dump_outputs(str(tmp_path / "all"), res, n)
    assert sorted(os.listdir(tmp_path / "all")) == ["hit_counts.npy", "pred_vote.npy", "top_idx.npy", "top_scores.npy"]
    got = {f[:-4]: np.load(tmp_path / "all" / f) for f in os.listdir(tmp_path / "all")}
    assert got["top_scores"].dtype == np.float32 and np.array_equal(got["top_scores"], res["top_scores"].numpy())
    for name in ("top_idx", "pred_vote", "hit_counts"):
        assert got[name].dtype == np.float64 and np.array_equal(got[name].astype(np.int64), res[name].numpy())
    monkeypatch.setattr(bench, "DUMP_QUERIES", 16)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), res, n)
    rows = np.load(tmp_path / "s1" / "query_rows.npy")
    assert rows.shape == (16,) and np.all(np.diff(rows) > 0)
    assert np.array_equal(rows, np.load(tmp_path / "s2" / "query_rows.npy"))
    r = rows.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "s1" / "top_idx.npy").astype(np.int64), res["top_idx"].numpy()[r])
    assert np.array_equal(np.load(tmp_path / "s1" / "hit_counts.npy"), [[5, 7]])
    monkeypatch.setattr(bench, "DUMP_BYTES", 100)
    with pytest.raises(RuntimeError, match="limit"):
        bench.dump_outputs(str(tmp_path / "big"), res, n)
    assert not os.path.exists(tmp_path / "big")


@pytest.mark.gpu
def test_b200_arm_line_small_workload(tmp_path):
    import numpy as np
    dump = tmp_path / "outputs"
    d = _run("--workload", "small", "--steps", "3", "--warmup", "3", "--cpu-sample", "8", "--dump-outputs", str(dump))
    assert BASE_KEYS | {"roofline", "clocks"} <= set(d)
    assert d["n_gpus"] == 1 and d["value"] > 0 and d["gpu_launches"] > 0 and d["data"] == "synthetic"
    assert d["steps"] == 3
    out = {f[:-4]: np.load(dump / f) for f in os.listdir(dump)}
    assert {"top_idx", "top_scores", "top_labels", "pred_vote", "pred_weighted", "hit_counts"} <= set(out)
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    assert out["top_idx"].shape == (2048, 10) and out["top_idx"].min() >= 0 and out["top_idx"].max() < 100_000
    assert np.all(np.diff(out["top_scores"], axis=1) <= 0)
    assert out["hit_counts"][0, 0] / 2048 == d["accuracy"]["top1"]
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 100_000_000 and e["d2h_bytes_per_step"] > 0
    assert e["value"] < d["value"]                      # the host-buffer path includes the copies
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["value"] > 0 and c["parity_on_sample"]["topk_rows_identical"] == 1.0
    assert c["parity_on_sample"]["vote_identical"] == 1.0


def test_roofline_denominator_rule():
    """Burst peak for short runs, sustained peak once the GPU has been under load for 1.5 s (bench.tensor_peak)."""
    sys.path.insert(0, REPO)
    import bench
    pk = {"tflops": 1382.1, "tflops_burst": 1657.8, "hbm_gbs": 6549.4, "src": "measured"}
    assert bench.tensor_peak(pk, 0.2)[0] == 1657.8 and "burst" in bench.tensor_peak(pk, 0.2)[1]
    assert bench.tensor_peak(pk, 1.9)[0] == 1382.1 and "sustained" in bench.tensor_peak(pk, 1.9)[1]
    got = bench.peaks()
    assert got["tflops_burst"] >= got["tflops"] > 0 and got["hbm_gbs"] > 0


def test_ncu_summary_tool(tmp_path, capsys):
    sys.path.insert(0, os.path.join(REPO, "tools"))
    import ncu_summary
    path = tmp_path / "launches.csv"
    rows = ['"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"']
    for i, (name, ns) in enumerate([("void emr2a::normalize_fuse_vec_kernel<float, 8, 0, 1>(NfParams)", 1700000), ("void emr2a::normalize_fuse_vec_kernel<float, 8, 0, 1>(NfParams)", 19000),
                                    ("void emr2a::tc2_topk_kernel<1, 16, 0>(CUtensorMap_st)", 13000000), ("emr2a::topk_merge_pway_kernel(const unsigned long *)", 60000),
                                    ("void at::native::vectorized_elementwise_kernel<4>(int)", 5000), ("void emr2a::vote_metrics_kernel<16>(VoteParams)", 15000)] * 2):
        rows.append(f'"{i}","1","python","box","{name}","1","7","(256, 1, 1)","(148, 1, 1)","0","10.0","Command line profiler metrics","gpu__time_duration.sum","ns","{ns}"')
    path.write_text("\n".join(rows) + "\n")
    ncu_summary.launches(str(path))
    out = capsys.readouterr().out
    assert "tc2_topk_kernel<1, 16, 0>" in out and "vectorized_elementwise" not in out
    assert "| 4 |" in out and "| 5 |" not in out            # the last step only: 5 of our launches
    assert "87.87%" in out and "= 88.3% of the step" in out   # tc2 share; filter + merge share
