"""Label-conditioned search on the host: RowLabels layout, padding, validation and shard views, the
argument checks of search_topk (refused before any device work), and the sharded labeled protocol at
world 2 over gloo (the CUDA search replaced by a torch fp32 masked top-k through ShardedGallery's
injection points)."""
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
CPU = torch.device("cpu")


def test_layout_and_padding(mm):
    from mmrs_b200.row_labels import label_elements
    assert label_elements(1) == 128 and label_elements(128) == 128 and label_elements(129) == 256
    lab = np.arange(300, dtype=np.int64) % 7
    L = mm.RowLabels(lab, device=CPU)
    assert L.n_rows == 300 and len(L) == 300 and L.labels.dtype == torch.int32
    assert L.labels.numel() == 384                                        # whole 128-row tiles
    assert (L.labels[:300].numpy() == lab).all() and (L.labels[300:] == 0).all()
    for dt in (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8):
        assert torch.equal(mm.RowLabels(torch.tensor([0, 1, 2], dtype=dt), device=CPU).labels[:3],
                           torch.tensor([0, 1, 2], dtype=torch.int32))
    assert mm.RowLabels([2 ** 31 - 2], device=CPU).labels[0] == 2 ** 31 - 2


@pytest.mark.parametrize("bad", [np.array([0, -1, 2]), np.array([2 ** 31 - 1]), np.array([2 ** 40]),
                                 np.array([0.5, 1.0]), np.array([True, False]), np.zeros((2, 2), np.int32),
                                 np.zeros(0, np.int32)])
def test_validation_at_construction(mm, bad):
    with pytest.raises(ValueError):
        mm.RowLabels(bad, device=CPU)


@pytest.mark.parametrize("n_rows,world", [(1000, 2), (1000, 3), (70_001, 8), (130, 4)])
def test_shard_views(mm, n_rows, world):
    lab = np.random.default_rng(n_rows + world).integers(0, 50, n_rows)
    L = mm.RowLabels(lab, device=CPU)
    for lo, hi in mm.shard_bounds(n_rows, world):
        s = L.shard(lo, hi)
        assert s.n_rows == hi - lo
        assert s.labels.data_ptr() == L.labels.data_ptr() + lo * 4          # a view at element lo
        assert s.labels.numel() >= 128 * ((hi - lo + 127) // 128)           # still whole tiles of the shard
        assert (s.labels[:hi - lo].numpy() == lab[lo:hi]).all()
        assert L.shard(lo, hi) is s                                         # cached per range
    with pytest.raises(ValueError):
        L.shard(64, n_rows)                                                 # not on a 128-row tile


class _FakeGallery:
    """What search_topk's argument checks read of a DeviceGallery (no device work happens before them)."""
    def __init__(self, n_rows, dim, device):
        self.n_rows, self.dim, self.padded_dim, self.device, self.mode = n_rows, dim, dim, device, "bf16"


def test_search_arguments_refused_before_device_work(mm, monkeypatch):
    from mmrs_b200 import search
    gal = _FakeGallery(300, 8, CPU)
    monkeypatch.setattr(search, "_as_gallery", lambda g, mode: g)
    monkeypatch.setattr(search, "_cabi", None)              # any device work would raise AttributeError
    q = torch.randn(4, 8)
    L = mm.RowLabels(np.arange(300) % 5, device=CPU)
    ql = torch.zeros(4, dtype=torch.int32)
    cases = [
        dict(row_labels=L),                                                  # labels come in pairs
        dict(query_labels=ql),
        dict(row_labels=L, query_labels=ql, label_match="different"),        # only "same" / "other"
        dict(label_match="SAME"),
        dict(row_labels=np.arange(300) % 5, query_labels=ql),                # not a RowLabels
        dict(row_labels=mm.RowLabels(np.arange(299) % 5, device=CPU), query_labels=ql),   # row count
        dict(row_labels=L, query_labels=torch.zeros(3, dtype=torch.int32)),  # shape
        dict(row_labels=L, query_labels=torch.zeros((4, 1), dtype=torch.int32)),
        dict(row_labels=L, query_labels=torch.zeros(4)),                     # dtype
        dict(row_labels=L, query_labels=torch.zeros(4, dtype=torch.bool)),
        dict(row_labels=L, query_labels=torch.tensor([0, 1, 2, 2 ** 31 - 1])),   # not < 2^31 - 1
        dict(row_labels=L, query_labels=torch.tensor([0, 1, 2, 2 ** 40])),
    ]
    for kw in cases:
        with pytest.raises(ValueError):
            search.search_topk(q, gal, 3, **kw)
    # another device than the gallery's
    gal_meta = _FakeGallery(300, 8, torch.device("meta"))
    with pytest.raises(ValueError):
        search.search_topk(q, gal_meta, 3, row_labels=L, query_labels=ql)


def masked_topk(oracle, q, shard, kk, row_labels, query_labels, label_match, normalize_queries, scale):
    """Torch fp32 reference of a labeled local search: per query the masked scores' stable top-k, padded
    with -inf / -1 like the library."""
    n = len(shard)
    lab = row_labels.labels[:n].numpy()
    ql = np.asarray(query_labels)
    vs, is_ = [], []
    for r in range(q.shape[0]):
        c = int(ql[r])
        keep = np.ones(n, bool) if c < 0 else ((lab == c) if label_match == "same" else (lab != c))
        rows = torch.from_numpy(np.nonzero(keep)[0])
        m = min(kk, rows.numel())
        v = torch.full((kk,), float("-inf"))
        i = torch.full((kk,), -1, dtype=torch.int64)
        if m:
            sv, si = oracle.search_topk(q[r:r + 1], shard.data[rows], m, normalize_queries=normalize_queries, scale=scale)
            v[:m], i[:m] = sv[0], rows[si[0]] + shard.row_offset
        vs.append(v); is_.append(i)
    return torch.stack(vs), torch.stack(is_)


class _HostShard:
    """Stand-in for DeviceGallery on CPU (tests only)."""
    def __init__(self, data, row_offset):
        self.data, self.row_offset = data, row_offset
    def __len__(self):
        return self.data.shape[0]


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import mmrs_b200
    from oracle import oracle
    n_rows, k = 1000, 10
    g = oracle.synthetic_gallery(n_rows, 32, seed=4, dtype=torch.float32)
    g[700] = g[5]                                     # an exact tie across the two shards
    q = oracle.synthetic_queries(8, 32)
    lo, hi = mmrs_b200.shard_bounds(n_rows, world)[rank]
    lab = np.arange(n_rows) % 4                       # classes 0..3 everywhere
    lab[:512] = np.where(lab[:512] == 2, 0, lab[:512])   # class 2 is absent from shard 0 (rows < 512)
    lab[[3, 600, 901]] = 5                            # class 5: 3 rows over both shards, fewer than k
    L = mmrs_b200.RowLabels(lab, device=CPU)
    ql = torch.tensor([2, 5, -1, 0, 7, 1, 5, 2], dtype=torch.int32)   # 7: absent from the gallery
    searched = []

    def local_search(queries, shard, kk, *, normalize_queries, scale, path, row_labels=None, query_labels=None,
                     label_match="same", row_filter=None):
        assert row_filter is None and row_labels is not None and row_labels.n_rows == len(shard)
        searched.append(kk)
        return masked_topk(oracle, queries, shard, kk, row_labels, query_labels, label_match, normalize_queries, scale)

    sg = mmrs_b200.ShardedGallery(_HostShard(g[lo:hi], lo), n_rows, local_search=local_search, merge=oracle.merge_topk)
    for match in ("same", "other"):
        v, i = sg.search_topk(q, k, row_labels=L, query_labels=ql, label_match=match)
        want_v, want_i = masked_topk(oracle, q, _HostShard(g, 0), k, L, ql, match, True, 1.0)
        assert torch.equal(i, want_i), (rank, match, i, want_i)
        assert torch.equal(v, want_v)
        if match == "same":
            assert (i[1, 3:] == -1).all() and (v[1, 3:] == float("-inf")).all()   # 3 rows of class 5, then padding
            assert (i[4] == -1).all()                                             # class 7: padding only
        gathered = [None, None]
        dist.all_gather_object(gathered, (v, i))
        assert torch.equal(gathered[0][1], gathered[1][1]) and torch.equal(gathered[0][0], gathered[1][0])
    assert searched == [min(k, hi - lo)] * 2
    # wrong arguments: the same error on every rank, before any collective
    with pytest.raises(ValueError):
        sg.search_topk(q, k, row_labels=mmrs_b200.RowLabels(lab[:-1], device=CPU), query_labels=ql)
    with pytest.raises(ValueError):
        sg.search_topk(q, k, row_labels=L)
    with pytest.raises(ValueError):
        sg.search_topk(q, k, row_labels=L, query_labels=ql[:-1])
    with pytest.raises(ValueError):
        sg.search_topk(q, k, row_labels=L, query_labels=ql, label_match="all")
    dist.barrier()
    Path(out_dir, f"ok{rank}").write_text("ok")
    dist.destroy_process_group()


def test_labeled_sharded_protocol_world2(tmp_path):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
