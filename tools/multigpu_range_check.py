"""torchrun --nproc-per-node N tools/multigpu_range_check.py : range search on a sharded gallery (N >= 2 GPUs).
ShardedGallery.search_range must equal the single-GPU search_range over the full gallery bit for bit on every
rank, with `path` pinned: mixed selectivity, a row filter leaving shard 0 without rows, labels, several row
windows, host and device queries.  Rank 0 prints 'multigpu range ok'.  Run by tests/test_range_multigpu_gpu.py
(self-spawned, skipped on a one-GPU box)."""
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
rng = np.random.default_rng(3)                        # same seed on every rank: the same filter and labels everywhere
lab = rng.integers(0, 10, n).astype(np.int32)
L = mmrs_b200.RowLabels(lab, device=dev)
mask = np.ones(n, bool)
mask[:bounds[0][1]] = False                           # shard 0 has no allowed row
mask[rng.random(n) < 0.5] = False
filt = mmrs_b200.RowFilter(mask, device=dev)
checked = 0
for path in ("mma", "gemv"):
    for nq, max_bytes, f, labeled in ((10, 4 << 30, None, False), (13, 13 * 8 * 40_064, None, False),
                                      (7, 4 << 30, filt, False), (9, 4 << 30, None, True)):
        q = oracle.synthetic_queries(nq, d, seed=nq).to(dev)
        srt = mmrs_b200.full_scores(q, full, path=path).sort(1, descending=True).values
        thr = torch.stack([srt[j, [30, n // 10, 0, 5][j % 4]] for j in range(nq)])
        thr[2::4] = float("-inf")
        kw = dict(path=path, row_filter=f, max_candidate_bytes=max_bytes)
        if labeled:
            kw.update(row_labels=L, query_labels=torch.from_numpy(rng.integers(-1, 11, nq)), label_match="same")
        want = mmrs_b200.search_range(q, full, thr, **kw)
        for qq in (q, q.cpu()):
            got = sg.search_range(qq, thr, **kw)
            for a, b in zip(got, want):
                assert torch.equal(a.cpu(), b.cpu()), (rank, path, nq, f is not None, labeled)
            checked += nq
gathered = [None] * world
dist.all_gather_object(gathered, [x.cpu() for x in got])
assert all(all(torch.equal(a, b) for a, b in zip(x, gathered[0])) for x in gathered)
dist.barrier()
if rank == 0:
    print(f"multigpu range ok: world={world} ({checked} queries equal the single-GPU search_range)")
dist.destroy_process_group()
