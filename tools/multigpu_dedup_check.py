"""torchrun --nproc-per-node N tools/multigpu_dedup_check.py : deduplication on N >= 2 GPUs.
ShardedGallery.deduplicate must equal the single-GPU deduplicate on every rank: the tensor-core join dealt over
the ranks and the exact join split by row ranges (raw_join), the identity order, a permutation and a subset
order.  Rank 0 prints 'multigpu dedup ok'.  Run by tests/test_dedup_multigpu_gpu.py (self-spawned, skipped on a
one-GPU box)."""
import os, sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch, torch.distributed as dist
import mmrs_b200
from mmrs_b200.dedup import selfjoin_raw

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)

# bases plus 1-4 noisy copies each at cosine 0.955-0.995 (same seed on every rank): clusters that are not cliques
gen = torch.Generator().manual_seed(0)
n_base, d = 12_000, 128
base = torch.nn.functional.normalize(torch.randn(n_base, d, generator=gen), dim=1)
rows = [base]
for k in range(4):
    b = base[torch.rand(n_base, generator=gen) < 0.6 / (k + 1)]
    c = 0.955 + 0.04 * torch.rand(b.shape[0], 1, generator=gen)
    r = torch.randn(b.shape, generator=gen)
    r = torch.nn.functional.normalize(r - (r * b).sum(1, keepdim=True) * b, dim=1)
    rows.append(c * b + (1 - c * c).sqrt() * r)
x = torch.cat(rows)
x = x[torch.randperm(x.shape[0], generator=gen)].contiguous().to(dev)
n = x.shape[0]
sg = mmrs_b200.ShardedGallery.from_full(x, mode="fp32", device=dev)
perm = torch.randperm(n, generator=gen)
checked = 0
for order in (None, perm, perm[: n // 2].to(dev)):
    want = mmrs_b200.deduplicate(x, 0.95, order=order)
    got = sg.deduplicate(x, 0.95, order=order)
    assert torch.equal(got, want), (rank, "tc", int((got != want).sum()))
    want = mmrs_b200.deduplicate(x, 0.95, order=order, method="fp32")
    got = sg.deduplicate(x, 0.95, order=order, raw_join=selfjoin_raw)
    assert torch.equal(got, want), (rank, "fp32", int((got != want).sum()))
    checked += 2
keep = int((got == torch.arange(n, device=dev)).sum())
assert keep < n
gathered = [None] * world
dist.all_gather_object(gathered, got.cpu())
assert all(torch.equal(g, gathered[0]) for g in gathered)
dist.barrier()
if rank == 0:
    print(f"multigpu dedup ok: world={world} ({checked} calls equal the single-GPU deduplicate, {n - keep} of {n} rows removed)")
dist.destroy_process_group()
