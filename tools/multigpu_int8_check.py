"""torchrun --nproc-per-node N tools/multigpu_int8_check.py : int8 galleries sharded over N >= 2 GPUs.
Quantisation is per row, so every rank's shard holds exactly the rows of the single-GPU int8 gallery, and the
fused NVLink gather, the NCCL keys variant and the general path must all return the single-GPU int8 search bit
for bit -- short shards included.  Rank 0 prints 'multigpu int8 ok'.  Run by tests/test_int8_multigpu_gpu.py
(self-spawned, skipped on a one-GPU box)."""
import os, sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch, torch.distributed as dist
import mmrs_b200

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)


def unit_rows(n, d, seed):
    x = torch.from_numpy(np.random.default_rng(seed).standard_normal((n, d)).astype(np.float32))
    return x / x.norm(dim=1, keepdim=True)


def same(a, b, what):
    assert torch.equal(a[1].cpu(), b[1].cpu()) and torch.equal(a[0].cpu().view(torch.int32), b[0].cpu().view(torch.int32)), \
        (rank, what)


checked = 0
n, d, k = 300_001, 768, 100
g = unit_rows(n, d, seed=0)
g[17] = g[n - 5]                                      # a tie across the first and the last shard
full = mmrs_b200.DeviceGallery(g, mode="int8", device=dev)
sg = mmrs_b200.ShardedGallery.from_full(g, mode="int8", device=dev)
lo, hi = mmrs_b200.shard_bounds(n, world)[rank]
assert torch.equal(sg.local.data.cpu(), full.data[lo:hi].cpu()), "a shard's rows differ from the full gallery's"
sg_nccl = mmrs_b200.ShardedGallery(sg.local, n, fused=False)
sg_gen = mmrs_b200.ShardedGallery(sg.local, n, local_search=mmrs_b200.search_topk)
for nq in (1, 3, 24, 130, 600):
    q = unit_rows(nq, d, seed=nq).to(dev)
    want = mmrs_b200.search_topk(q, full, k)
    for h, what in ((sg, "fused"), (sg_nccl, "nccl"), (sg_gen, "general")):
        same(h.search_topk(q, k), want, (what, nq))
        checked += nq
assert sg.fused_active and not sg_nccl.fused_active, "the fused NVLink gather was not used"
# short shards: the last one just long enough for k (fused), and too short for it (NCCL variant pads)
for last_rows, want_fused in ((110, True), (50, False), (10, False)):
    n_short = 128 * (world - 1) + last_rows
    gs = unit_rows(n_short, 64, seed=7)
    fs = mmrs_b200.DeviceGallery(gs, mode="int8", device=dev)
    sgs = mmrs_b200.ShardedGallery.from_full(gs, mode="int8", device=dev)
    qq = unit_rows(4, 64, seed=3).to(dev)
    same(sgs.search_topk(qq, k), mmrs_b200.search_topk(qq, fs, k), ("short", last_rows))
    assert sgs.fused_active == want_fused, (n_short, sgs.fused_active, want_fused)
    checked += 4
dist.barrier()
if rank == 0:
    print(f"multigpu int8 ok: world={world} ({checked} query searches equal the single-GPU int8 search bit for bit)")
dist.destroy_process_group()
