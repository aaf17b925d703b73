"""bench.py on the GPU: --steps sets the timed steps, --dump-outputs writes what the timed search returned."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def test_bench_steps_and_dumped_outputs(mm, tmp_path):
    rows, dim, batch, k = 300_000, 768, 16, 100
    lines = {}
    for steps in (3, 6):
        cmd = [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--rows", str(rows), "--dim", str(dim),
               "--batch", str(batch), "--k", str(k), "--steps", str(steps), "--warmup", "1", "--legs", "none",
               "--no-cpu", "--dump-outputs", str(tmp_path / f"steps{steps}")]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines[steps] = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert lines[steps]["steps"] == steps
    # the timed region holds exactly --steps searches: twice the steps, twice the kernel launches
    assert lines[6]["gpu_launches"] == 2 * lines[3]["gpu_launches"] > 0
    # same arguments but --steps: same inputs, so the same lists
    dumped = {}
    for name in ("topk_values", "topk_indices"):
        a, b = np.load(tmp_path / "steps3" / f"{name}.npy"), np.load(tmp_path / "steps6" / f"{name}.npy")
        assert a.shape == (batch, k)
        np.testing.assert_array_equal(a, b)
        dumped[name] = a
    # and they are what a caller of the timed search receives on the bench's seeded gallery and queries
    # (device_gallery_shard with shard_id = rank * 64 + world, query generator seed 1)
    from bench import device_gallery_shard
    g = device_gallery_shard(torch, rows, dim, seed=0, shard_id=1, device=torch.device("cuda", 0))
    q = torch.randn((batch, dim), generator=torch.Generator().manual_seed(1))
    v, i = mm.search_topk(q.cuda(), mm.DeviceGallery(g), k)
    np.testing.assert_array_equal(dumped["topk_values"], v.cpu().numpy())
    np.testing.assert_array_equal(dumped["topk_indices"], i.cpu().numpy().astype(np.float64))
    del g
    torch.cuda.empty_cache()
