"""torchrun --nproc-per-node N tools/multigpu_filter_check.py : row-filtered sharded search on N >= 2 GPUs.
The fused NVLink gather, the NCCL keys variant and the general path must equal the single-GPU filtered
search over the full gallery bit for bit (every row's score comes from the same kernel either way),
including a shard without any allowed row, all allowed rows in one shard with fewer than k elsewhere,
and a k above the allowed rows, which must raise on every rank without a hang.  Rank 0 prints
'multigpu filter ok'.  Run by tests/test_filter_multigpu_gpu.py (self-spawned, skipped on a one-GPU box)."""
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
n, d, k = 400_000, 512, 100
g = oracle.synthetic_gallery(n, d, seed=0, dtype=torch.bfloat16)
g[17] = g[n - 5]                                  # a tie across the first and last shard
sg = mmrs_b200.ShardedGallery.from_full(g, device=dev)
sg_nccl = mmrs_b200.ShardedGallery(sg.local, n, fused=False)
full = mmrs_b200.DeviceGallery(g, device=dev)      # the single-GPU reference: the whole gallery on this GPU
bounds = mmrs_b200.shard_bounds(n, world)
rng = np.random.default_rng(3)                     # same seed on every rank: the same masks everywhere

masks = {"p10": rng.random(n) < 0.1}
m = np.zeros(n, dtype=bool); m[bounds[1][0]:] = True
masks["shard0_empty"] = m                          # rank 0 holds no allowed row
m = np.zeros(n, dtype=bool); lo, hi = bounds[world - 1]; m[lo:hi] = True
for r in range(world - 1):                         # every other shard: fewer than k allowed rows
    m[rng.choice(np.arange(*bounds[r]), 20, replace=False)] = True
m[17] = m[n - 5] = True
masks["one_shard"] = m
masks["p01"] = rng.random(n) < 0.001               # ~50 per shard at world 8: short everywhere

for name, mask in masks.items():
    f = mmrs_b200.RowFilter(mask, device=dev)
    for nq in (3, 24, 130):
        q = oracle.synthetic_queries(nq, d, seed=nq).to(dev)
        wv, wi = mmrs_b200.search_topk(q, full, k, row_filter=f)
        v, i = sg.search_topk(q, k, row_filter=f)
        vb, ib = sg_nccl.search_topk(q, k, row_filter=f)
        vg, ig = sg.search_topk_general(q, k, row_filter=f)
        for a, b, what in ((v, i, "fused"), (vb, ib, "nccl"), (vg, ig, "general")):
            assert torch.equal(b, wi) and torch.equal(a, wv), (rank, name, nq, what, int((b != wi).sum()))
        assert bool(torch.from_numpy(mask)[i.cpu()].all())
    # per-call bool mask and host queries give the same lists
    qh = oracle.synthetic_queries(5, d, seed=9)
    hv, hi = sg.search_topk(qh, k, row_filter=mask)
    wv, wi = mmrs_b200.search_topk(qh, full, k, row_filter=f)
    assert not hv.is_cuda and torch.equal(hi, wi) and torch.equal(hv, wv), (rank, name)
assert sg.fused_active and not sg_nccl.fused_active, "the fused NVLink gather was not used"

# k above the allowed rows: every rank raises from the same filter, nobody enters a collective
few = np.zeros(n, dtype=bool); few[rng.choice(n, 50, replace=False)] = True
f = mmrs_b200.RowFilter(few, device=dev)
q = oracle.synthetic_queries(4, d, seed=2).to(dev)
for s in (sg, sg_nccl):
    try:
        s.search_topk(q, k, row_filter=f)
        raise SystemExit("k > allowed rows was accepted")
    except RuntimeError as e:
        assert "out of range" in str(e)
v, i = sg.search_topk(q, 50, row_filter=f)          # and the slot still works: k == allowed rows
wv, wi = mmrs_b200.search_topk(q, full, 50, row_filter=f)
assert torch.equal(i, wi) and torch.equal(v, wv)
dist.barrier()
if rank == 0:
    print(f"multigpu filter ok: world={world} (fused NVLink gather, NCCL variant and general path equal the single-GPU "
          "filtered search; empty shard; one shard holding the allowed rows; k > allowed raises on every rank)")
dist.destroy_process_group()
