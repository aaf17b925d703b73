"""torchrun --nproc-per-node N tools/multigpu_label_check.py : label-conditioned sharded search on N >= 2 GPUs.
The fused NVLink gather, the NCCL keys variant and the general path must equal the single-GPU labeled
search over the full gallery bit for bit, -inf / -1 padding included: a class absent from shard 0, a
class with fewer than k rows over all shards, a label absent from the gallery, unlabeled queries, and
"same" and "other".  Rank 0 prints 'multigpu labels ok'.  Run by tests/test_labels_multigpu_gpu.py
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
n, d, k = 400_000, 512, 100
g = oracle.synthetic_gallery(n, d, seed=0, dtype=torch.bfloat16)
g[17] = g[n - 5]                                  # a tie across the first and last shard
sg = mmrs_b200.ShardedGallery.from_full(g, device=dev)
sg_nccl = mmrs_b200.ShardedGallery(sg.local, n, fused=False)
full = mmrs_b200.DeviceGallery(g, device=dev)      # the single-GPU reference: the whole gallery on this GPU
bounds = mmrs_b200.shard_bounds(n, world)
rng = np.random.default_rng(3)                     # same seed on every rank: the same labels everywhere

lab = rng.integers(0, 10, n).astype(np.int32)                 # 10 random classes
lab[:bounds[0][1]][lab[:bounds[0][1]] == 4] = 0              # class 4 is absent from shard 0
lab[rng.choice(n, 30, replace=False)] = 11                    # class 11: 30 rows over all shards, fewer than k
lab[17] = lab[n - 5] = 3
L = mmrs_b200.RowLabels(lab, device=dev)
n_padded = 0
for match in ("same", "other"):
    for nq in (3, 24, 130):
        ql = torch.from_numpy(rng.choice(np.array([0, 3, 4, 11, 12, -1], dtype=np.int32), nq))   # 12: no row has it
        ql[0] = 11
        q = oracle.synthetic_queries(nq, d, seed=nq).to(dev)
        kw = dict(row_labels=L, query_labels=ql, label_match=match)
        wv, wi = mmrs_b200.search_topk(q, full, k, **kw)
        v, i = sg.search_topk(q, k, **kw)
        vb, ib = sg_nccl.search_topk(q, k, **kw)
        vg, ig = sg.search_topk_general(q, k, **kw)
        for a, b, what in ((v, i, "fused"), (vb, ib, "nccl"), (vg, ig, "general")):
            assert torch.equal(b, wi) and torch.equal(a, wv), (rank, match, nq, what, int((b != wi).sum()))
        n_padded += int((wi == -1).sum())
    # host queries and host labels give the same lists
    qh = oracle.synthetic_queries(5, d, seed=9)
    qlh = torch.tensor([11, 4, -1, 12, 0], dtype=torch.int32)
    hv, hi = sg.search_topk(qh, k, row_labels=L, query_labels=qlh, label_match=match)
    wv, wi = mmrs_b200.search_topk(qh, full, k, row_labels=L, query_labels=qlh, label_match=match)
    assert not hv.is_cuda and torch.equal(hi, wi) and torch.equal(hv, wv), (rank, match)
assert n_padded > 0, "no padded position was exercised"
assert sg.fused_active and not sg_nccl.fused_active, "the fused NVLink gather was not used"
dist.barrier()
if rank == 0:
    print(f"multigpu labels ok: world={world} (fused NVLink gather, NCCL variant and general path equal the single-GPU "
          f"labeled search, {n_padded} padded positions included)")
dist.destroy_process_group()
