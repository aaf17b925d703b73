"""torchrun --nproc-per-node N tools/multigpu_stored_join_check.py : the stored-format self-join on N >= 2 GPUs.
ShardedGallery.find_duplicate_pairs / deduplicate with method="stored" on a bf16 and an int8 gallery replicated on
every rank must equal the single-GPU calls, on every rank, for the identity order and a permutation.  Rank 0 prints
'multigpu stored join ok'.  Run by tests/test_stored_join_multigpu_gpu.py (self-spawned, skipped on a one-GPU box)."""
import os, sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch, torch.distributed as dist
import mmrs_b200

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)

# bases plus noisy copies at cosine 0.955-0.995 (same seed on every rank); 20 K rows: ten 2048-row panels
gen = torch.Generator().manual_seed(0)
n_base, d = 12_000, 256
base = torch.nn.functional.normalize(torch.randn(n_base, d, generator=gen), dim=1)
rows = [base]
for k in range(3):
    b = base[torch.rand(n_base, generator=gen) < 0.5 / (k + 1)]
    c = 0.955 + 0.04 * torch.rand(b.shape[0], 1, generator=gen)
    r = torch.randn(b.shape, generator=gen)
    r = torch.nn.functional.normalize(r - (r * b).sum(1, keepdim=True) * b, dim=1)
    rows.append(c * b + (1 - c * c).sqrt() * r)
x = torch.cat(rows)
x = x[torch.randperm(x.shape[0], generator=gen)].contiguous().to(dev)
n = x.shape[0]
sg = mmrs_b200.ShardedGallery.from_full(x, mode="bf16", device=dev)
perm = torch.randperm(n, generator=gen)
checked = 0
for mode in ("bf16", "int8"):
    gal = mmrs_b200.DeviceGallery(x, mode=mode, device=dev)      # every row on every rank
    want = mmrs_b200.find_duplicate_pairs(gal, 0.95, method="stored")
    got = sg.find_duplicate_pairs(gal, 0.95, method="stored")
    assert want.shape[0] > 1000 and torch.equal(got, want), (rank, mode, got.shape, want.shape)
    for order in (None, perm):
        want = mmrs_b200.deduplicate(gal, 0.95, order=order, method="stored")
        got = sg.deduplicate(gal, 0.95, order=order, method="stored")
        assert torch.equal(got, want), (rank, mode, int((got != want).sum()))
        checked += 1
    gathered = [None] * world
    dist.all_gather_object(gathered, got.cpu())
    assert all(torch.equal(g, gathered[0]) for g in gathered)
dist.barrier()
if rank == 0:
    print(f"multigpu stored join ok: world={world} ({checked} deduplicate calls and 2 pair lists equal the single-GPU ones)")
dist.destroy_process_group()
