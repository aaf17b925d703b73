"""Refined search on the host: argument checks, the candidate count k_c, the store's row layout, the refine
workspace size, and the sharded refined protocol at world 2 over gloo (the CUDA search replaced by a torch
fp32 masked top-k through ShardedGallery's injection points).  No GPU needed."""
import os
import socket
import sys
import types
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parent.parent
CPU = torch.device("cpu")


def test_store_arguments_refused_before_device_work(mm):
    x = torch.randn(10, 8)
    with pytest.raises(ValueError, match="int8"):
        mm.RefineStore(x, mode="int8")
    with pytest.raises(ValueError, match="mode"):
        mm.RefineStore(x, mode="fp16")
    with pytest.raises(ValueError, match="memory"):
        mm.RefineStore(x, memory="disk")
    with pytest.raises(TypeError):
        mm.RefineStore(torch.randn(10))


def test_candidate_count(mm):
    from mmrs_b200.refine import MAX_CANDIDATES, candidate_k, default_refine_k
    assert default_refine_k(10) == 20 and default_refine_k(512) == 1024 and default_refine_k(1000) == 1024
    assert default_refine_k(1024) == 1024
    assert candidate_k(10, None, 1_000_000) == 20
    assert candidate_k(10, 25, 1_000_000) == 25
    assert candidate_k(10, 400, 120) == 120                       # capped by N
    assert candidate_k(10, 400, 1_000_000, n_allowed=57) == 57    # and by a RowFilter's allowed rows
    assert candidate_k(10, 10, 1_000_000) == 10
    with pytest.raises(ValueError, match="refine_k"):
        candidate_k(10, 9, 1_000_000)
    with pytest.raises(ValueError, match=str(MAX_CANDIDATES)):
        candidate_k(10, MAX_CANDIDATES + 1, 1_000_000)
    assert candidate_k(10, 5000, 700) == 700                      # N <= 1024: refine_k = N is allowed


def _bare_store(mm, n, d, device=None):
    s = object.__new__(mm.RefineStore)
    s.n_rows, s.dim, s.device, s.ptr = n, d, device, 1
    return s


def test_store_must_match_the_gallery(mm):
    gal = types.SimpleNamespace(n_rows=100, dim=64, device=torch.device("cuda", 0))
    _bare_store(mm, 100, 64).check_matches(gal)                    # host store: any device
    _bare_store(mm, 100, 64, torch.device("cuda", 0)).check_matches(gal)
    for bad in (_bare_store(mm, 99, 64), _bare_store(mm, 100, 63), _bare_store(mm, 100, 64, torch.device("cuda", 1))):
        with pytest.raises(ValueError, match="refine store"):
            bad.check_matches(gal)
    closed = _bare_store(mm, 100, 64)
    closed.ptr = 0
    with pytest.raises(ValueError, match="closed"):
        closed.check_matches(gal)


@pytest.mark.parametrize("d", [1, 7, 8, 100, 768])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_store_row_layout(mm, d, mode):
    """DeviceGallery's layout: [N, round_up(D, 8)] of the mode's dtype, zero columns past D."""
    from mmrs_b200.refine import store_rows
    n = 37
    x = torch.randn(n, d, dtype=torch.float64)
    dt = torch.bfloat16 if mode == "bf16" else torch.float32
    dp = (d + 7) // 8 * 8
    out = store_rows(x, mode, torch.full((n, dp), 7.0, dtype=dt))
    want = torch.zeros((n, dp), dtype=dt)
    want[:, :d] = x.to(dt)
    assert torch.equal(out.view(torch.int16 if mode == "bf16" else torch.int32),
                       want.view(torch.int16 if mode == "bf16" else torch.int32))
    assert out.stride(0) * out.element_size() % 16 == 0
    with pytest.raises(ValueError):
        store_rows(x, mode, torch.zeros((n, dp + 8), dtype=dt))


def test_page_aligned_host_buffer(mm):
    from mmrs_b200.refine import _page_aligned_host
    for nbytes in (1, 4096, 4097, 123_456):
        buf, pages = _page_aligned_host(nbytes)
        assert pages.data_ptr() % 4096 == 0 and pages.numel() % 4096 == 0 and pages.numel() >= nbytes
        assert buf.data_ptr() <= pages.data_ptr() and pages.data_ptr() + pages.numel() <= buf.data_ptr() + buf.numel()


def _align(x):
    return (x + 255) // 256 * 256


@pytest.mark.parametrize("dim,nq,kc", [(8, 1, 1), (768, 16, 400), (768, 1024, 1024), (1040, 300, 40), (100, 7, 13)])
def test_refine_workspace_bytes(mm, dim, nq, kc):
    """flags, fused-gather scratch, fp32 queries and three bf16 query planes (the search's carve), then one
    8-byte key per (query, candidate); every piece on a 256-byte boundary."""
    ldq, qp = (dim + 7) // 8 * 8, (nq + 15) // 16 * 16
    want = _align(32) + _align(512) + _align(qp * ldq * 4) + _align(3 * qp * ldq * 2) + _align(nq * kc * 8)
    assert mm._cabi.lib.mmrs_refine_workspace_bytes(dim, nq, kc) == want
    assert mm._cabi.lib.mmrs_refine_workspace_bytes(0, nq, kc) == 0
    assert mm._cabi.lib.mmrs_refine_workspace_bytes(dim, 0, kc) == 0
    assert mm._cabi.lib.mmrs_refine_workspace_bytes(dim, nq, 0) == 0


def masked_topk(oracle, q, shard, kk, row_labels, query_labels, label_match, normalize_queries, scale):
    """Exact top-kk of each query over its eligible rows, padded with -inf / -1 (as the library's labeled search)."""
    n = len(shard)
    lab = row_labels.labels[:n].numpy() if row_labels is not None else np.zeros(n, np.int32)
    ql = query_labels if query_labels is not None else torch.full((q.shape[0],), -1, dtype=torch.int32)
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
    seen = []

    def local_search(queries, shard, kk, *, normalize_queries, scale, path, row_labels=None, query_labels=None,
                     label_match="same", refine=None, refine_k=None):
        # the fake refined search is exact: what is tested is that every rank's own store and refine_k arrive
        seen.append((kk, refine, refine_k))
        return masked_topk(oracle, queries, shard, kk, row_labels, query_labels, label_match, normalize_queries, scale)

    store = f"store of rank {rank}"           # stands in for the rank's RefineStore: handed through untouched
    # a shard shorter than k (200 rows, k = 150: shard 1 holds 72), unlabeled and labeled
    for n_rows, k in ((1000, 10), (200, 150)):
        # small integers, unnormalised: every dot product is exact in fp32 whatever the summation order, so the
        # shard-by-shard reference and the merged result agree on every machine (and tie often)
        gen = torch.Generator().manual_seed(n_rows)
        g = torch.randint(-3, 4, (n_rows, 32), generator=gen).float()
        g[n_rows - 3] = g[5]                                  # an exact tie across the two shards
        q = torch.randint(-3, 4, (6, 32), generator=gen).float()
        lo, hi = mmrs_b200.shard_bounds(n_rows, world)[rank]
        sg = mmrs_b200.ShardedGallery(_HostShard(g[lo:hi], lo), n_rows, local_search=local_search,
                                      merge=oracle.merge_topk)
        seen.clear()
        v, i = sg.search_topk(q, k, normalize_queries=False, refine=store, refine_k=4 * k)
        want_v, want_i = masked_topk(oracle, q, _HostShard(g, 0), k, None, None, "same", False, 1.0)
        assert torch.equal(i, want_i) and torch.equal(v, want_v), (rank, n_rows)
        assert seen == [(min(k, hi - lo), store, 4 * k)], seen
        seen.clear()
        sg.search_topk(q, k, normalize_queries=False, refine=store)   # the default is decided from the global k
        assert seen == [(min(k, hi - lo), store, mmrs_b200.refine.default_refine_k(k))], seen
        pend = sg.search_topk(q, k, normalize_queries=False, refine=store, sync=False)
        assert torch.equal(pend.wait()[1], want_i)
        # labeled: class 5 has 3 rows over both shards, class 7 none -> padded positions merge to -inf / -1
        lab = np.arange(n_rows) % 4
        lab[[3, n_rows - 10, n_rows - 20]] = 5
        L = mmrs_b200.RowLabels(lab, device=CPU)
        ql = torch.tensor([5, 7, -1, 0, 1, 5], dtype=torch.int32)
        v, i = sg.search_topk(q, k, normalize_queries=False, refine=store, refine_k=k, row_labels=L, query_labels=ql)
        want_v, want_i = masked_topk(oracle, q, _HostShard(g, 0), k, L, ql, "same", False, 1.0)
        assert torch.equal(i, want_i) and torch.equal(v, want_v), (rank, n_rows, "labeled")
        assert (i[0, 3:] == -1).all() and (i[1] == -1).all()
        # refine_k < k: the same error on every rank, before any collective
        with pytest.raises(ValueError, match="refine_k"):
            sg.search_topk(q, k, refine=store, refine_k=k - 1)
    dist.barrier()
    Path(out_dir, f"ok{rank}").write_text("ok")
    dist.destroy_process_group()


def test_refined_sharded_protocol_world2(tmp_path):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
