"""The bench.py contract the driver relies on, checked without a GPU: the reference arm (`--impl reference`) runs on the
host cores and prints ONE JSON line with the agreed keys; the workload description is identical for both arms."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ)
    env.pop("RANK", None)
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                           "--cpu-sample-rows", "8192", "--gpus", "1"], capture_output=True, text=True, timeout=600, env=env,
                          cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines  # everything else (library banners, warnings) goes to stderr
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "queries/s"
    assert d["metric"].startswith("QPS, exact IP top-100 over 21000000x1024")
    assert d["config"]["rows"] == 21_000_000 and d["config"]["batch"] == 4096 and d["config"]["k"] == 100
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and "sample" in cb and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # a step of this arm is one pass over the bounded sample: steps * ms_per_step is what the run really took
    assert 0 < d["ms_per_step"] < 120_000 and d["ms_per_full_step_extrapolated"] > d["ms_per_step"]
    assert d["vs_baseline"] is None and d["gpu_launches"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                           "--cpu-sample-rows", "4096", "--gpus", "2"], capture_output=True, text=True, timeout=300, env=env,
                          cwd=ROOT)
    assert proc.returncode == 0 and proc.stdout.strip() == ""


def test_reference_arm_dumps_its_last_step_the_same_every_run(tmp_path):
    import numpy as np

    env = dict(os.environ)
    env.pop("RANK", None)
    for run in ("a", "b"):
        proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                               "--warmup", "0", "--cpu-sample-rows", "4096", "--batch", "64", "--k", "10",
                               "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=300,
                              env=env, cwd=ROOT)
        assert proc.returncode == 0, proc.stderr[-2000:]
        assert sorted(os.listdir(tmp_path / run)) == ["ids.npy", "scores.npy"]
    D, I = np.load(tmp_path / "a" / "scores.npy"), np.load(tmp_path / "a" / "ids.npy")
    assert D.shape == I.shape == (64, 10) and D.dtype == np.float32 and I.dtype == np.float64
    assert np.all(I == np.round(I))
    # the search the arm ran: its seeded inputs rebuilt here (bench.cpu_baseline), answers against fp64 ground truth
    import torch

    from tests.helpers import assert_topk_parity

    xb = torch.nn.functional.normalize(torch.randn(4096, 1024, generator=torch.Generator().manual_seed(1234)), dim=1)
    xq = torch.nn.functional.normalize(torch.randn(64, 1024, generator=torch.Generator().manual_seed(4321)), dim=1)
    assert_topk_parity(D, I.astype(np.int64), xb.numpy(), xq.numpy(), 10, what="dumped reference-arm step")
    assert np.array_equal(D, np.load(tmp_path / "b" / "scores.npy"))
    assert np.array_equal(I, np.load(tmp_path / "b" / "ids.npy"))


def test_dump_outputs_keeps_a_fixed_sample_of_rows_above_the_limit(tmp_path, monkeypatch):
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench

    D = np.arange(3000, dtype=np.float32).reshape(1000, 3)
    I = np.arange(3000, dtype=np.int64).reshape(1000, 3)
    bench.dump_outputs(str(tmp_path / "all"), {"scores": D, "ids": I})
    assert np.array_equal(np.load(tmp_path / "all" / "ids.npy"), I.astype(np.float64))
    assert not os.path.exists(tmp_path / "all" / "rows.npy")
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 20_000)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"scores": D, "ids": I})
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy")) and 0 < len(rows) < 1000
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 20_000
    r = rows.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "scores.npy"), D[r])
    assert np.array_equal(np.load(tmp_path / "a" / "ids.npy"), I[r].astype(np.float64))


def test_steps_below_one_are_rejected():
    for steps in ("0", "-1"):
        proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", steps],
                              capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert proc.returncode == 2 and "--steps" in proc.stderr and proc.stdout.strip() == ""


def test_both_arms_describe_the_same_workload():
    sys.path.insert(0, ROOT)
    import bench

    c = bench.workload_config(21_000_000, 4096, 100)
    assert set(c) == {"workload", "rows", "dim", "batch", "k", "l2"} and "configs[3]" in c["workload"]
    p = bench.load_peaks()
    assert p["hbm_gbs"] > 0 and p["bf16_tflops"] >= p["bf16_tflops_sustained"] > 0 and p["source"] in ("measured", "fallback")
