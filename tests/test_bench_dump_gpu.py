"""bench.py --dump-outputs on the GPU arm: the dumped scores and ids are the answer to the benchmark's own seeded
corpus and queries (rebuilt here the way bench.build_shard and run_ours generate them), checked against fp64."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.helpers import assert_topk_parity

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROWS, BATCH, K, CHUNK, DIM = 50_000, 64, 10, 1 << 20, 1024


def test_gpu_arm_dumps_the_answer_of_its_last_timed_step(tmp_path):
    import torch

    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                           "--rows", str(ROWS), "--batch", str(BATCH), "--k", str(K), "--sweep=", "--no-extras",
                           "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                          capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-3000:]
    assert sorted(os.listdir(tmp_path)) == ["ids.npy", "scores.npy"]
    D, I = np.load(tmp_path / "scores.npy"), np.load(tmp_path / "ids.npy")
    assert D.shape == I.shape == (BATCH, K) and D.dtype == np.float32 and I.dtype == np.float64
    assert np.all(I == np.round(I))
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev)
    g.manual_seed(1234)  # chunk 0 of the corpus
    xb = torch.nn.functional.normalize(torch.randn(CHUNK, DIM, generator=g, device=dev), dim=1)[:ROWS].cpu().numpy()
    g.manual_seed(4321)  # the queries
    xq = torch.nn.functional.normalize(torch.randn(BATCH, DIM, generator=g, device=dev), dim=1).cpu().numpy()
    assert_topk_parity(D, I.astype(np.int64), xb, xq, K, what="dumped GPU-arm step")
