"""search_range on the host: the float64 -> float32 threshold conversion against numpy, window planning, the
per-query join of CSR pieces, and the sharded protocol at world 2 over gloo -- the local step replaced by a
numpy stand-in through ShardedGallery's local_range_search injection point, on integer-valued data (exact
fp32 scores whatever the summation order)."""
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
FMAX = np.finfo(np.float32).max


def round_up_ref(t64):
    """The smallest float32 >= t, by numpy."""
    with np.errstate(over="ignore"):
        t32 = t64.astype(np.float32)
        return np.where(t32.astype(np.float64) < t64, np.nextafter(t32, np.float32(np.inf)), t32)


def test_threshold_round_up_matches_numpy(mm):
    from mmrs_b200.range_search import thresholds_f32
    rng = np.random.default_rng(0)
    f32 = rng.standard_normal(200).astype(np.float32)
    tiny = np.float64(np.finfo(np.float32).smallest_subnormal)
    t64 = np.concatenate([
        rng.standard_normal(500) * 10.0 ** rng.integers(-40, 39, 500),     # random, down to the subnormals
        f32.astype(np.float64),                                             # exactly representable
        f32.astype(np.float64) + np.abs(f32.astype(np.float64)) * 1e-9,     # just above one
        np.array([tiny, tiny * 0.5, tiny * 1.5, -tiny * 0.5, 1e-45, -1e-45, 0.0, -0.0]),
        np.array([FMAX, -FMAX, FMAX * (1 + 2 ** -30), -FMAX * (1 + 2 ** -30), 1e300, -1e300, np.inf, -np.inf]),
    ])
    got = thresholds_f32(torch.from_numpy(t64), t64.size).numpy()
    want = round_up_ref(t64)
    np.testing.assert_array_equal(got.view(np.uint32) & 0x7fffffff, want.view(np.uint32) & 0x7fffffff)
    assert np.array_equal(got, want)
    # the claim the conversion rests on: s >= t32 exactly when float64(s) >= t, for every float32 s
    fin = got[np.isfinite(got) & (got != -FMAX)]
    s = np.concatenate([f32, fin, np.nextafter(fin, np.float32(-np.inf)), np.array([np.inf, -np.inf, FMAX, -FMAX], np.float32)])
    for t, t32 in zip(t64[::7], got[::7]):
        assert np.array_equal(s >= t32, s.astype(np.float64) >= t)
    # Python floats and ints are float64; float32 passes unchanged; scalars broadcast
    assert thresholds_f32(0.1, 3).tolist() == [round_up_ref(np.array([0.1]))[0]] * 3
    assert thresholds_f32(np.float32(0.1), 2).numpy().tolist() == [np.float32(0.1)] * 2
    assert thresholds_f32(torch.tensor([1, 2]), 2).tolist() == [1.0, 2.0]
    for bad in (float("nan"), torch.tensor([0.0, float("nan")]), np.zeros(3), np.zeros((2, 1)), torch.tensor([True, False])):
        with pytest.raises(ValueError):
            thresholds_f32(bad, 2)


def test_window_planning(mm):
    from mmrs_b200.range_search import window_rows
    assert -(-100_000_000 // window_rows(16, 100_000_000, 4 << 30)) == 3
    assert -(-1_000_000 // window_rows(1024, 1_000_000, 4 << 30)) == 2
    rng = np.random.default_rng(1)
    for _ in range(300):
        nq, n = int(rng.integers(1, 2000)), int(rng.integers(1, 10 ** int(rng.integers(1, 9))))
        budget = int(rng.integers(8 * 128 * nq, 8 * 128 * nq * 64))
        w = window_rows(nq, n, budget)
        assert w % 128 == 0 and w >= 128 and nq * w * 8 <= budget
        starts = list(range(0, n, w))
        covered = np.zeros(n, np.int64)
        for r0 in starts:
            assert min(r0 + w, n) - r0 >= 1
            covered[r0:r0 + w] += 1
        assert (covered == 1).all()
    with pytest.raises(ValueError):
        window_rows(4, 1000, 8 * 128 * 4 - 1)


def test_concat_per_query(mm):
    from mmrs_b200.range_search import concat_per_query
    rng = np.random.default_rng(2)
    nq, n_pieces = 5, 4
    want_v = [[] for _ in range(nq)]
    pieces = []
    for p in range(n_pieces):
        counts = rng.integers(0, 4, nq)
        counts[p % nq] = 0                                  # empty segments in every piece
        off = np.concatenate([[0], np.cumsum(counts)])
        vals = rng.standard_normal(int(off[-1])).astype(np.float32)
        for q in range(nq):
            want_v[q] += vals[off[q]:off[q + 1]].tolist()
        pieces.append((torch.from_numpy(off), torch.from_numpy(vals), torch.arange(int(off[-1])) + 1000 * p))
    off, v, i = concat_per_query(pieces)
    assert off.tolist() == [0] + np.cumsum([len(x) for x in want_v]).tolist()
    for q in range(nq):
        assert v[off[q]:off[q + 1]].tolist() == want_v[q]
        assert (np.diff(i[off[q]:off[q + 1]].numpy() // 1000) >= 0).all()      # piece order inside a query
    one = pieces[0]
    assert concat_per_query([one]) is one
    empty = (torch.zeros(nq + 1, dtype=torch.int64), torch.empty(0), torch.empty(0, dtype=torch.int64))
    off, v, i = concat_per_query([empty, empty])
    assert off.tolist() == [0] * (nq + 1) and v.numel() == 0


# ---- the sharded protocol over gloo ---------------------------------------------------------------------------
def host_filter(mm, mask):
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


class _HostShard:
    def __init__(self, data, row_offset):
        self.data, self.row_offset = data, row_offset

    def __len__(self):
        return self.data.shape[0]


def numpy_range_search(oracle):
    """The contract on the host: mask = S >= t (and the filter / labels), CSR in row order, global indices."""
    def local(q, shard, thr, *, normalize_queries, scale, path, max_candidate_bytes, row_filter=None,
              row_labels=None, query_labels=None, label_match="same"):
        s = oracle.full_scores(q, shard.data, normalize_queries=normalize_queries, scale=scale).numpy()
        mask = (s >= thr.numpy()[:, None]) & allowed_rows(row_filter, len(shard))[None, :]
        if row_labels is not None:
            lab = row_labels.labels[:len(shard)].numpy()[None, :]
            ql = np.asarray(query_labels)[:, None]
            same = lab == ql
            mask &= (ql < 0) | (same if label_match == "same" else ~same)
        off = np.concatenate([[0], np.cumsum(mask.sum(1))])
        idx = np.nonzero(mask)[1] + shard.row_offset
        return torch.from_numpy(off), torch.from_numpy(s[mask] + np.float32(0)), torch.from_numpy(idx)
    return local


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, str(ROOT))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import mmrs_b200
    from oracle import oracle
    n_rows, d = 1000, 16
    gen = torch.Generator().manual_seed(11)
    g = torch.randint(-3, 4, (n_rows, d), generator=gen).float()
    q = torch.randint(-2, 3, (6, d), generator=gen).float()
    g[512:] = -g[512:].abs()                                              # query 5 matches no row of shard 1
    q[5] = q[5].abs() + 1
    thr = torch.tensor([0.0, 5.0, float("-inf"), 1.0, 3.0, 1.0])
    lo, hi = mmrs_b200.shard_bounds(n_rows, world)[rank]                  # [0, 512) and [512, 1000)
    local = numpy_range_search(oracle)
    sg = mmrs_b200.ShardedGallery(_HostShard(g[lo:hi], lo), n_rows, local_range_search=local)
    full = _HostShard(g, 0)
    lab = np.arange(n_rows) % 3
    L = mmrs_b200.RowLabels(lab, device=CPU)
    ql = torch.tensor([0, 1, -1, 2, 0, 1])
    block0 = np.zeros(n_rows, bool)
    block0[:300] = True                                                   # rank 1's shard: no allowed row
    for mask in (None, block0):
        f = host_filter(mmrs_b200, mask) if mask is not None else None
        for lab_kw in ({}, dict(row_labels=L, query_labels=ql, label_match="same"),
                       dict(row_labels=L, query_labels=ql, label_match="other")):
            kw = dict(normalize_queries=False, scale=1.0, path="auto", max_candidate_bytes=4 << 30)
            got = sg.search_range(q, thr, row_filter=f, **lab_kw, **kw)
            want = local(q, full, thr, row_filter=f, **lab_kw, **kw)
            for a, b in zip(got, want):
                assert torch.equal(a, b), (rank, mask is not None, lab_kw.get("label_match"))
            if mask is None and not lab_kw:
                five = got[2][got[0][5]:got[0][6]]
                assert five.numel() > 0 and int(five.max()) < 512
                assert got[0][3] - got[0][2] == n_rows                    # -inf: every row
            gathered = [None, None]
            dist.all_gather_object(gathered, [x.tolist() for x in got])
            assert gathered[0] == gathered[1]
    got = sg.search_range(q[:0], torch.zeros(0), normalize_queries=False)
    assert got[0].tolist() == [0] and got[1].numel() == 0
    with pytest.raises(ValueError):                                       # the same refusal on every rank
        sg.search_range(q, float("nan"))
    dist.barrier()
    Path(out_dir, f"ok{rank}").write_text("ok")
    dist.destroy_process_group()


def test_sharded_protocol_world2(tmp_path):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
