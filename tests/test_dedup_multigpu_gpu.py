"""Deduplication on a sharded gallery: self-spawns torchrun over the visible GPUs (2 are enough) and runs
tools/multigpu_dedup_check.py -- ShardedGallery.deduplicate against the single-GPU deduplicate on every rank.
Skipped on a one-GPU box."""
import os
import socket
import subprocess
import sys
from pathlib import Path

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_sharded_deduplicate_on_all_visible_gpus():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"{n} GPU visible: the sharded path needs at least 2")
    world = 2 if n < 4 else (4 if n < 8 else 8)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           str(ROOT / "tools" / "multigpu_dedup_check.py")]
    env = dict(os.environ, MMRS_GATHER_TIMEOUT_MS="60000", OMP_NUM_THREADS="4")
    res = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    tail = (res.stdout + res.stderr)[-3000:]
    assert res.returncode == 0, tail
    assert f"multigpu dedup ok: world={world}" in res.stdout, tail
