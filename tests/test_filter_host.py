"""Row filters on the host: bitmap layout, shard slices and their allowed counts, and the sharded
filtered-search protocol at world 2 over gloo (the CUDA search replaced by the oracle on the allowed
rows through ShardedGallery's injection points)."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent


def host_filter(mm, mask):
    """RowFilter over host words packed with numpy (the layout mmrs_pack_row_filter writes on the GPU)."""
    from mmrs_b200.row_filter import filter_words
    n = mask.shape[0]
    padded = np.zeros(filter_words(n) * 32, dtype=bool)
    padded[:n] = mask
    words = torch.from_numpy(np.packbits(padded, bitorder="little")).view(torch.int32)
    return mm.RowFilter._wrap(words, n, int(mask.sum()))


def allowed_rows(f, n_rows):
    """Bool mask of a (possibly shard-view) host RowFilter's first n_rows rows."""
    bits = np.unpackbits(f.words.contiguous().view(torch.uint8).numpy(), bitorder="little")
    return bits[:n_rows].astype(bool)


def test_bitmap_layout_and_padding(mm):
    from mmrs_b200.row_filter import count_allowed, filter_words
    assert filter_words(1) == 4 and filter_words(128) == 4 and filter_words(129) == 8
    mask = np.zeros(300, dtype=bool)
    mask[[0, 31, 32, 200, 299]] = True
    f = host_filter(mm, mask)
    w = f.words.numpy().view(np.uint32)
    assert w.shape == (12,)
    assert w[0] == (1 | 1 << 31) and w[1] == 1 and w[6] == 1 << 8 and w[9] == 1 << 11
    assert (w[10:] == 0).all()                                           # whole-tile padding is zero
    assert count_allowed(f.words, 0, 300) == 5 == f.n_allowed
    assert count_allowed(f.words, 32, 299) == 2 and count_allowed(f.words, 32, 300) == 3 and count_allowed(f.words, 0, 0) == 0


@pytest.mark.parametrize("n_rows,world", [(1000, 2), (1000, 3), (70_001, 8), (130, 4)])
def test_shard_slices_and_counts(mm, n_rows, world):
    rng = np.random.default_rng(n_rows + world)
    mask = rng.random(n_rows) < 0.3
    f = host_filter(mm, mask)
    total = 0
    for lo, hi in mm.shard_bounds(n_rows, world):
        s = f.shard(lo, hi)
        assert s.n_rows == hi - lo and s.n_allowed == int(mask[lo:hi].sum())
        # the slice is a pointer offset of lo / 32 words into the same bitmap ...
        assert s.words.data_ptr() == f.words.data_ptr() + lo // 32 * 4
        # ... that still covers the shard's own whole tiles
        assert s.words.numel() >= 4 * ((hi - lo + 127) // 128)
        assert (allowed_rows(s, hi - lo) == mask[lo:hi]).all()
        assert f.shard(lo, hi) is s                                      # cached per range
        total += s.n_allowed
    assert total == f.n_allowed
    with pytest.raises(ValueError):
        f.shard(64, n_rows)                                              # not on a 128-row tile


class _HostShard:
    """Stand-in for DeviceGallery on CPU (tests only)."""
    def __init__(self, data, row_offset):
        self.data, self.row_offset = data, row_offset
    def __len__(self):
        return self.data.shape[0]


def _worker(rank, world, port, case, out_dir):
    sys.path.insert(0, str(ROOT))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import mmrs_b200
    from oracle import oracle
    n_rows, k = 1000, 10
    g = oracle.synthetic_gallery(n_rows, 32, seed=4, dtype=torch.float32)
    g[700] = g[5]                                     # an exact tie across the two shards
    q = oracle.synthetic_queries(6, 32)
    lo, hi = mmrs_b200.shard_bounds(n_rows, world)[rank]
    mask = np.zeros(n_rows, dtype=bool)
    if case == "empty_shard0":                        # rank 0 holds no allowed row
        mask[mmrs_b200.shard_bounds(n_rows, world)[1][0]:] = True
    elif case == "short_shard":                       # rank 0 holds fewer than k allowed rows
        mask[[5, 17, 200]] = True
        mask[512:] = True
    else:                                             # sparse everywhere
        mask[::7] = True
        mask[700] = True
    searched = []

    def local_search(queries, shard, kk, *, normalize_queries, scale, path, row_filter=None):
        keep = allowed_rows(row_filter, len(shard)) if row_filter is not None else np.ones(len(shard), bool)
        assert row_filter is None or row_filter.n_allowed == int(keep.sum()) >= kk
        rows = torch.from_numpy(np.nonzero(keep)[0])
        v, i = oracle.search_topk(queries, shard.data[rows], kk, normalize_queries=normalize_queries, scale=scale)
        searched.append(kk)
        return v, rows[i] + shard.row_offset

    sg = mmrs_b200.ShardedGallery(_HostShard(g[lo:hi], lo), n_rows, local_search=local_search,
                                  merge=oracle.merge_topk)
    f = host_filter(mmrs_b200, mask)
    v, i = sg.search_topk(q, k, row_filter=f)
    sub = torch.from_numpy(np.nonzero(mask)[0])
    want_v, want_i = oracle.search_topk(q, g[sub], k)
    assert torch.equal(i, sub[want_i]), (rank, i, sub[want_i])
    assert torch.equal(v, want_v)
    n_here = int(mask[lo:hi].sum())
    assert searched == ([min(k, n_here)] if n_here else [])     # a shard without allowed rows skips its search
    # k above the allowed rows: the same error on every rank, no collective entered
    with pytest.raises(RuntimeError, match="out of range"):
        sg.search_topk(q, int(mask.sum()) + 1, row_filter=f)
    with pytest.raises(ValueError):
        sg.search_topk(q, k, row_filter=host_filter(mmrs_b200, mask[:-1]))
    dist.barrier()
    Path(out_dir, f"ok{rank}").write_text("ok")
    dist.destroy_process_group()


@pytest.mark.parametrize("case", ["empty_shard0", "short_shard", "sparse"])
def test_filtered_sharded_protocol_world2(tmp_path, case):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(2, port, case, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
