"""torchrun --nproc-per-node N tools/multigpu_threshold_check.py : per-class threshold tuning on a sharded gallery
(N >= 2 GPUs).  ShardedGallery.best_thresholds must equal the single-GPU best_thresholds over the full gallery
bit for bit on every rank, with `path` pinned: classes absent from shard 0 or from the whole gallery, a row
filter leaving shard 0 without rows, several chunks, host and device queries.  Rank 0 prints
'multigpu thresholds ok'.  Run by tests/test_thresholds_multigpu_gpu.py (self-spawned, skipped on a one-GPU box)."""
import os, sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch, torch.distributed as dist
import mmrs_b200
from oracle import oracle

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
n, d = 300_001, 256
g = oracle.synthetic_gallery(n, d, seed=0, dtype=torch.bfloat16)
sg = mmrs_b200.ShardedGallery.from_full(g, device=dev)
full = mmrs_b200.DeviceGallery(g, device=dev)         # the single-GPU reference: the whole gallery on this GPU
bounds = mmrs_b200.shard_bounds(n, world)
rng = np.random.default_rng(3)                        # same seed on every rank: the same labels everywhere
lab = rng.integers(0, 10, n).astype(np.int32)
lab[:bounds[0][1]][lab[:bounds[0][1]] == 4] = 0      # class 4 is absent from shard 0
L = mmrs_b200.RowLabels(lab, device=dev)
mask = np.ones(n, bool)
mask[:bounds[0][1]] = False                           # shard 0 has no allowed row
mask[rng.random(n) < 0.5] = False
filt = mmrs_b200.RowFilter(mask, device=dev)
checked = 0
for path in ("mma", "gemv"):
    for nq, max_bytes, f in ((10, 4 << 30, None), (13, 4 * bounds[0][1] * 4, None), (7, 4 << 30, filt)):
        q = oracle.synthetic_queries(nq, d, seed=nq)
        ql = torch.from_numpy(rng.choice(np.array([0, 3, 4, 11], dtype=np.int32), nq))   # 11: no row has it
        kw = dict(path=path, row_filter=f, max_score_bytes=max_bytes)
        want = mmrs_b200.best_thresholds(q, full, L, ql, **kw)
        for qq in (q, q.to(dev)):
            got = sg.best_thresholds(qq, L, ql, **kw)
            for a, b in zip(got, want):
                assert np.array_equal(a, b, equal_nan=True), (rank, path, nq, f is not None)
            checked += nq
gathered = [None] * world
dist.all_gather_object(gathered, got)
assert all(all(np.array_equal(a, b, equal_nan=True) for a, b in zip(x, gathered[0])) for x in gathered)
dist.barrier()
if rank == 0:
    print(f"multigpu thresholds ok: world={world} ({checked} prototypes equal the single-GPU best_thresholds)")
dist.destroy_process_group()
