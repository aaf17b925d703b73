"""best_thresholds on the host: argument checks (refused before any device work), chunk sizing, and the
sharded protocol at world 2 over gloo -- the device steps replaced by numpy stand-ins through
ShardedGallery's local_range / local_counts injection points, on integer-valued data (exact fp32 scores
whatever the summation order)."""
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


def host_filter(mm, mask):
    """RowFilter over host words packed with numpy (the layout mmrs_pack_row_filter writes on the GPU)."""
    from mmrs_b200.row_filter import filter_words
    n = mask.shape[0]
    padded = np.zeros(filter_words(n) * 32, dtype=bool)
    padded[:n] = mask
    words = torch.from_numpy(np.packbits(padded, bitorder="little")).view(torch.int32)
    return mm.RowFilter._wrap(words, n, int(mask.sum()))


def allowed_rows(f, n_rows):
    if f is None:
        return np.ones(n_rows, bool)
    bits = np.unpackbits(f.words.contiguous().view(torch.uint8).numpy(), bitorder="little")
    return bits[:n_rows].astype(bool)


def test_chunk_sizing(mm):
    from mmrs_b200.thresholds import chunk_queries
    assert chunk_queries(100_000_000, 4 << 30) == 10            # 4.0 GB of scores at N = 100 M
    assert chunk_queries(12_500_000, 4 << 30) == 85
    assert chunk_queries(1_000_000_000, 4 << 30) == 1           # never below one query
    assert chunk_queries(1000, 4000) == 1 and chunk_queries(1000, 12_000) == 3
    # the sharded call sizes chunks from the longest shard, which every rank computes alike
    bounds = mm.shard_bounds(1000, 2)
    assert bounds == [(0, 512), (512, 1000)]
    assert chunk_queries(max(h - l for l, h in bounds), 4 * 488 * 5) == 4 != chunk_queries(488, 4 * 488 * 5)


class _FakeGallery:
    """What best_thresholds' argument checks read of a DeviceGallery."""
    def __init__(self, n_rows, dim, device):
        self.n_rows, self.dim, self.padded_dim, self.device, self.mode = n_rows, dim, dim, device, "bf16"


def test_arguments_refused_before_device_work(mm, monkeypatch):
    from mmrs_b200 import thresholds
    gal = _FakeGallery(300, 8, CPU)
    monkeypatch.setattr(thresholds, "_as_gallery", lambda g, mode: g)
    monkeypatch.setattr(thresholds, "DeviceSweep", None)        # any device work would raise TypeError
    q = torch.randn(4, 8)
    L = mm.RowLabels(np.arange(300) % 5, device=CPU)
    ql = torch.tensor([0, 1, 2, 3])
    cases = [
        (q, L, torch.tensor([0, -1, 2, 3]), {}),                         # negative label
        (q, L, torch.tensor([0, 1, 2, 2 ** 31 - 1]), {}),                # out of range
        (q, L, torch.tensor([0, 1, 2, 2 ** 40]), {}),
        (q, L, ql[:3], {}),                                              # one label per query
        (q, L, ql.float(), {}),
        (q, mm.RowLabels(np.arange(299) % 5, device=CPU), ql, {}),       # RowLabels length
        (q, np.arange(300) % 5, ql, {}),                                 # not a RowLabels
        (q, L, ql, dict(n_points=0)),
        (q, L, ql, dict(n_points=4097)),
        (q, L, ql, dict(row_filter=host_filter(mm, np.zeros(300, bool)))),   # allows no row
        (q, L, ql, dict(row_filter=host_filter(mm, np.ones(299, bool)))),    # row count
        (torch.randn(4, 7), L, ql, {}),                                  # width
    ]
    for qq, lab, qlab, kw in cases:
        with pytest.raises(ValueError):
            thresholds.best_thresholds(qq, gal, lab, qlab, **kw)
    out = thresholds.best_thresholds(q[:0], gal, L, ql[:0], n_points=7)  # C = 0: empty arrays
    assert [a.shape for a in out] == [(0,), (0,), (0,), (0,), (0, 7), (0, 7)]
    assert all(a.dtype == np.float64 for a in out)


# ---- numpy stand-ins of the two device steps ----------------------------------------------------------------
def _keys(s):
    b = (s + np.float32(0.0)).view(np.uint32).astype(np.int64)
    return np.where(b & 0x80000000, ~b & 0xffffffff, b | 0x80000000)


def _from_key(k):
    k = np.uint32(k)
    return (k & np.uint32(0x7fffffff) if k & np.uint32(0x80000000) else ~k).view(np.float32)


def _scores(oracle, q, shard, normalize_queries, scale):
    return oracle.full_scores(q, shard.data, normalize_queries=normalize_queries, scale=scale).numpy()


def make_steps(oracle, calls):
    def local_range(q, shard, *, normalize_queries, scale, path, row_filter):
        calls.append(int(q.shape[0]))
        s = _scores(oracle, q, shard, normalize_queries, scale)[:, allowed_rows(row_filter, len(shard))]
        if s.shape[1] == 0:
            return torch.tensor([[0xffffffff, 0]] * q.shape[0], dtype=torch.int64)
        k = _keys(s)
        return torch.from_numpy(np.stack([k.min(1), k.max(1)], 1))

    def local_counts(q, shard, rng, *, row_labels, query_labels, n_points, row_filter, grid_f32, normalize_queries,
                     scale, path):
        allowed = allowed_rows(row_filter, len(shard))
        s = _scores(oracle, q, shard, normalize_queries, scale)
        lab = row_labels.labels[:len(shard)].numpy()
        nq = q.shape[0]
        thr = np.zeros((nq, n_points))
        counts = np.zeros((nq, n_points, 2), np.int64)
        n_pos = np.zeros(nq, np.int64)
        for j in range(nq):
            lo, hi = _from_key(int(rng[j, 0])), _from_key(int(rng[j, 1]))
            thr[j] = np.linspace(lo, hi, n_points) if grid_f32 else np.linspace(np.float64(lo), np.float64(hi), n_points)
            pos = allowed & (lab == int(query_labels[j]))
            neg = allowed & (lab != int(query_labels[j]))
            counts[j, :, 0] = (s[j, pos][None, :] >= thr[j][:, None]).sum(1)
            counts[j, :, 1] = (s[j, neg][None, :] >= thr[j][:, None]).sum(1)
            n_pos[j] = pos.sum()
        return torch.from_numpy(thr), torch.from_numpy(counts), torch.from_numpy(n_pos)

    return local_range, local_counts


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
    from mmrs_b200.search import grid_f32
    from mmrs_b200.thresholds import run_chunks
    from oracle import oracle
    n_rows, d, n_points = 1000, 16, 200
    gen = torch.Generator().manual_seed(7)
    g = torch.randint(-3, 4, (n_rows, d), generator=gen).float()          # integer scores: exact in any order
    q = torch.randint(-2, 3, (7, d), generator=gen).float()
    lo, hi = mmrs_b200.shard_bounds(n_rows, world)[rank]                  # [0, 512) and [512, 1000): unequal
    lab = np.arange(n_rows) % 4
    lab[512:][lab[512:] == 3] = 0                                         # class 3 only on shard 0
    L = mmrs_b200.RowLabels(lab, device=CPU)
    ql = torch.tensor([3, 0, 1, 9, 2, 3, 1])                              # 9: no row has it
    calls = []
    local_range, local_counts = make_steps(oracle, calls)
    sg = mmrs_b200.ShardedGallery(_HostShard(g[lo:hi], lo), n_rows, local_range=local_range, local_counts=local_counts)
    full = _HostShard(g, 0)
    block0 = np.zeros(n_rows, bool)
    block0[:300] = True                                                   # shard 1 has no allowed row
    for mask in (None, block0):
        f = host_filter(mmrs_b200, mask) if mask is not None else None
        for scale, norm in ((100.0, False), (1.0, True)):
            calls.clear()
            got = sg.best_thresholds(q, L, ql, n_points=n_points, scale=scale, normalize_queries=norm, row_filter=f,
                                     max_score_bytes=4 * 488 * 5)
            assert calls == [4, 3], calls                                  # the longest shard sizes the chunks
            kw = dict(normalize_queries=norm, scale=scale, path="auto")
            want = run_chunks(q, ql, 7, n_points, lambda qq: local_range(qq, full, row_filter=f, **kw),
                              lambda qq, l, r: local_counts(qq, full, r, row_labels=L, query_labels=l, n_points=n_points,
                                                            row_filter=f, grid_f32=grid_f32(), **kw))
            for a, b in zip(got, want):
                np.testing.assert_array_equal(a, b)
            gathered = [None, None]
            dist.all_gather_object(gathered, got)
            for a, b in zip(*gathered):
                np.testing.assert_array_equal(a, b)
            assert np.isnan(got[5][3]).all() and got[0][3] == 0.0         # the absent class
            # the reference's arithmetic on the host split of the full scores
            s = _scores(oracle, q, full, norm, scale)
            allowed = mask if mask is not None else np.ones(n_rows, bool)
            for j in (0, 1, 4):
                sj, cj = s[j, allowed], lab[allowed] == int(ql[j])
                ref = oracle.find_thresholds(sj[cj], sj[~cj], n_points)
                np.testing.assert_array_equal(got[4][j], ref[4])
                np.testing.assert_array_equal(got[5][j], ref[5])
                assert (got[0][j], got[1][j], got[2][j], got[3][j]) == tuple(float(x) for x in ref[:4])
    with pytest.raises(ValueError):                                       # the same refusal on every rank
        sg.best_thresholds(q, L, ql, row_filter=host_filter(mmrs_b200, np.zeros(n_rows, bool)))
    with pytest.raises(ValueError):
        sg.best_thresholds(q, mmrs_b200.RowLabels(lab[:-1], device=CPU), ql)
    dist.barrier()
    Path(out_dir, f"ok{rank}").write_text("ok")
    dist.destroy_process_group()


def test_sharded_protocol_world2(tmp_path):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
