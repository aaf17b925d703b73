"""torchrun --nproc-per-node N tools/multigpu_refine_check.py : refined search on an int8 gallery sharded over N >= 2
GPUs, each rank refining its shard's candidates against its own fp32 store (host memory on even ranks, device
memory on odd ones).  Expected result, computed on every rank with one GPU: the top-k of the union over shards of
each shard's refined top-k, where a shard's candidates are the unrefined int8 search of that shard alone -- a
superset of the one-GPU candidate set, so it may differ from the one-GPU refined result.  Where every shard's
candidates contain that shard's exact fp32 top-k, the result must also equal the sharded exact fp32 search.
Rank 0 prints 'multigpu refine ok'.  Run by tests/test_refine_multigpu_gpu.py (self-spawned, skipped on a one-GPU
box)."""
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


def bits(v):
    return v.cpu().contiguous().view(torch.int32)


checked = contained = 0
for n, d, k, refine_k in ((200_003, 768, 100, 400), (128 * (world - 1) + 50, 64, 80, 120)):   # 2nd: a short shard
    g = unit_rows(n, d, seed=n)
    g[17] = g[n - 5]                                                   # a tie across the first and the last shard
    bounds = mmrs_b200.shard_bounds(n, world)
    lo, hi = bounds[rank]
    sg = mmrs_b200.ShardedGallery.from_full(g, mode="int8", device=dev)
    store = mmrs_b200.RefineStore(g[lo:hi], mode="fp32", memory="host" if rank % 2 == 0 else "device", device=dev)
    sg32 = mmrs_b200.ShardedGallery.from_full(g, mode="fp32", device=dev, local_search=mmrs_b200.search_topk)
    for nq in (1, 7, 130):
        q = unit_rows(nq, d, seed=nq + 1).to(dev)
        v, i = sg.search_topk(q, k, refine=store, refine_k=refine_k)
        # the expectation on this GPU alone: every shard searched and refined separately, then merged
        vs, is_ = [], []
        for r_lo, r_hi in bounds:
            shard8 = mmrs_b200.DeviceGallery(g[r_lo:r_hi], mode="int8", device=dev, row_offset=r_lo)
            st = mmrs_b200.RefineStore(g[r_lo:r_hi], mode="fp32", memory="device", device=dev)
            kl = min(k, r_hi - r_lo)
            sv, si = mmrs_b200.search_topk(q, shard8, kl, refine=st, refine_k=refine_k)
            pad = k - kl
            vs.append(torch.cat([sv, torch.full((nq, pad), float("-inf"), device=dev)], 1))
            is_.append(torch.cat([si, torch.full((nq, pad), 2 ** 32 - 1, dtype=torch.int64, device=dev)], 1))
            st.close()
        wv, wi = mmrs_b200.sharded._merge_cuda(torch.stack(vs), torch.stack(is_), k)
        assert torch.equal(i.cpu(), wi.cpu()) and torch.equal(bits(v), bits(wv)), (rank, n, nq)
        # containment: every shard's candidates hold its exact fp32 top-k -> the sharded exact fp32 search
        ev, ei = sg32.search_topk(q, k, path="gemv")
        held = True
        for r_lo, r_hi in bounds:
            shard8 = mmrs_b200.DeviceGallery(g[r_lo:r_hi], mode="int8", device=dev, row_offset=r_lo)
            shard32 = mmrs_b200.DeviceGallery(g[r_lo:r_hi], mode="fp32", device=dev, row_offset=r_lo)
            kl = min(k, r_hi - r_lo)
            cand = mmrs_b200.search_topk(q, shard8, mmrs_b200.refine.candidate_k(kl, refine_k, r_hi - r_lo))[1].cpu()
            ex = mmrs_b200.search_topk(q, shard32, kl, path="gemv")[1].cpu()
            held &= all(set(ex[j].tolist()) <= set(cand[j].tolist()) for j in range(nq))
        if held:
            contained += 1
            assert torch.equal(i.cpu(), ei.cpu()) and torch.equal(bits(v), bits(ev)), (rank, n, nq, "containment")
        checked += nq
    store.close()
assert contained > 0, "containment never held: the comparison with the exact sharded search did not run"
dist.barrier()
if rank == 0:
    print(f"multigpu refine ok: world={world} ({checked} queries equal the union-of-shards expectation, "
          f"{contained} batches the sharded exact fp32 search)")
dist.destroy_process_group()
