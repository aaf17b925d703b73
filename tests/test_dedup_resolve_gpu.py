"""resolve_duplicates / deduplicate on the GPU: the representative tensor must give exactly the walk of the
host `greedy_first_keeper` (representatives and duplicates, in walk order), -1 for rows outside the order,
on random graphs, the recorded reference walk, adversarial shapes and the self-join's own pairs."""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def walk_of(rep, order):
    """(representatives, duplicates) read off a representative tensor in walk order."""
    rep = rep.tolist()
    reps = [v for v in order if rep[v] == v]
    dups = [(v, rep[v]) for v in order if rep[v] not in (v, -1)]
    return reps, dups


def check(mm, n, pairs, order=None, device=True):
    """resolve_duplicates against greedy_first_keeper on one input; returns the (host) result."""
    pairs = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    walk = list(range(n)) if order is None else [int(v) for v in order]
    want_reps, want_dups = mm.greedy_first_keeper(n, pairs, walk)
    p = torch.from_numpy(pairs)
    o = None if order is None else torch.tensor(walk, dtype=torch.int64)
    if device:
        p = p.cuda()
        o = None if o is None else o.cuda()
    rep = mm.resolve_duplicates(p, n, order=o)
    assert rep.dtype == torch.int64 and rep.shape == (n,) and rep.is_cuda == device
    rep = rep.cpu()
    reps, dups = walk_of(rep, walk)
    assert reps == want_reps
    assert dups == [tuple(d) for d in want_dups]
    outside = np.setdiff1d(np.arange(n), np.asarray(walk, dtype=np.int64))
    assert (rep[torch.from_numpy(outside)] == -1).all()
    return rep


def orders(rng, n):
    yield "identity", None
    yield "random", rng.permutation(n)
    yield "subset", rng.permutation(n)[: n // 2]


@pytest.mark.parametrize("n,m", [(10, 12), (200, 300), (1000, 5000)])
def test_random_graphs_match_host_walk(mm, oracle, n, m):
    rng = np.random.default_rng(n)
    pairs = rng.integers(0, n, size=(m, 2))
    pairs = np.unique(np.sort(pairs[pairs[:, 0] != pairs[:, 1]], axis=1), axis=0)
    for _, order in orders(rng, n):
        for device in (True, False):
            rep = check(mm, n, pairs, order, device=device)
        walk = list(range(n)) if order is None else order.tolist()
        reps, dups = walk_of(rep, walk)
        want_reps, want_dups = oracle.greedy_keep_first(n, pairs.tolist(), walk)
        assert reps == want_reps and dups == [tuple(d) for d in want_dups]


def clustered_pairs(rng, n, frac=0.1):
    """Clusters of 2-8 rows over `frac` of the rows: half cliques, half sparser (a random spanning tree plus a
    few extra edges), in random orientation and order."""
    rows = rng.permutation(n)
    out, i = [], 0
    while i < int(n * frac):
        s = int(rng.integers(2, 9))
        c = rows[i:i + s]
        i += s
        if rng.random() < 0.5:
            a, b = np.triu_indices(len(c), 1)
            out.append(np.stack([c[a], c[b]], 1))
        else:
            e = [(c[k], c[int(rng.integers(0, k))]) for k in range(1, len(c))]
            e += [tuple(rng.choice(c, 2, replace=False)) for _ in range(len(c) // 2)]
            out.append(np.array(e, dtype=np.int64).reshape(-1, 2))
    p = np.concatenate(out).astype(np.int64)
    flip = rng.random(len(p)) < 0.5
    p[flip] = p[flip][:, ::-1]
    return p[rng.permutation(len(p))]


def test_clustered_100k_rows(mm):
    rng = np.random.default_rng(5)
    n = 100_000
    pairs = clustered_pairs(rng, n)
    for _, order in orders(rng, n):
        check(mm, n, pairs, order)


def test_reference_walk_golden(mm, tmp_path):
    """The result tuple recorded from tool/find_repeated_in_same_folder.py:56-106 (stub hashes): file-size
    order with two unreadable files skipped, i.e. a subset order."""
    from conftest import GOLDEN
    from golden_inputs import greedy_inputs
    gold = json.loads((GOLDEN / "same_folder_golden.json").read_text())
    folder, ids, similar, unreadable = greedy_inputs(str(tmp_path))
    paths = sorted(ids, key=lambda p: os.path.getsize(p), reverse=True)
    order = [ids[p] for p in paths if ids[p] not in unreadable]
    pairs = sorted(tuple(sorted(s)) for s in similar)
    n = len(ids)
    for device in (True, False):
        rep = mm.resolve_duplicates(torch.tensor(pairs, dtype=torch.int64, device="cuda" if device else "cpu"), n,
                                    order=order)
        reps, dups = walk_of(rep.cpu(), order)
        assert reps == gold["representatives"]
        assert [list(d) for d in dups] == gold["deleted"]
        assert all(rep[v] == -1 for v in unreadable)


def test_degenerate_inputs(mm):
    none = np.zeros((0, 2), dtype=np.int64)
    rep = check(mm, 5, none)
    assert rep.tolist() == [0, 1, 2, 3, 4]
    assert check(mm, 1, none).tolist() == [0]
    assert check(mm, 1, [[0, 0]]).tolist() == [0]
    assert check(mm, 6, [[0, 1], [2, 3]], order=[]).tolist() == [-1] * 6
    assert mm.resolve_duplicates(torch.zeros((0, 2), dtype=torch.int64, device="cuda"), 0).shape == (0,)


def test_clique_of_300(mm):
    rng = np.random.default_rng(3)
    n = 1000
    c = rng.choice(n, 300, replace=False)
    a, b = np.triu_indices(300, 1)
    pairs = np.stack([c[a], c[b]], 1)
    order = rng.permutation(n)
    rep = check(mm, n, pairs, order)
    first = [v for v in order if v in set(c.tolist())][0]
    assert (rep[torch.from_numpy(c)] == first).all()


@pytest.mark.parametrize("centre_first", [True, False])
def test_star(mm, centre_first):
    n, centre = 50_000, 12_345
    leaves = np.setdiff1d(np.arange(n), [centre])
    pairs = np.stack([np.full(n - 1, centre), leaves], 1)
    rng = np.random.default_rng(1)
    rest = rng.permutation(leaves)
    order = np.concatenate([[centre], rest]) if centre_first else np.concatenate([rest, [centre]])
    rep = check(mm, n, pairs, order)
    if centre_first:
        assert (rep == centre).all()
    else:
        assert rep[centre] == rest[0] and (rep[torch.from_numpy(leaves)] == torch.from_numpy(leaves)).all()


@pytest.mark.parametrize("reverse", [False, True])
def test_long_path_takes_the_tail(mm, reverse):
    """A 200 K-row path walked end to end: every rank depends on the one before it, so the rounds decide
    almost nothing and the single-warp tail finishes the walk."""
    from mmrs_b200.dedup import _resolve
    n = 200_000
    pairs = np.stack([np.arange(n - 1), np.arange(1, n)], 1)
    order = np.arange(n)[::-1].copy() if reverse else None
    check(mm, n, pairs, order)
    o = None if order is None else torch.from_numpy(order).cuda()
    rep, rounds, tail = _resolve(torch.from_numpy(pairs).cuda(), n, o)
    assert tail > n // 2 and rounds >= 1
    walk = np.arange(n) if order is None else order
    assert (rep.cpu()[torch.from_numpy(walk[0::2])] == torch.from_numpy(walk[0::2])).all()     # every other row kept


def test_messy_pair_lists(mm):
    """Self-pairs, repeated pairs, both orientations, and pairs touching rows outside the order."""
    rng = np.random.default_rng(9)
    n = 5000
    base = clustered_pairs(rng, n, frac=0.4)
    extra = [np.stack([np.arange(0, n, 7), np.arange(0, n, 7)], 1),          # self-pairs
             base[: len(base) // 3], base[: len(base) // 4][:, ::-1]]          # repeats, reversed
    pairs = np.concatenate([base] + extra)
    pairs = pairs[rng.permutation(len(pairs))]
    order = rng.permutation(n)[: 3 * n // 4]                                   # a quarter of the rows outside
    check(mm, n, pairs, order)
    check(mm, n, pairs, order, device=False)
    check(mm, n, pairs)


def test_errors_and_determinism(mm):
    pairs = torch.tensor([[0, 1], [1, 2], [3, 4]], dtype=torch.int64, device="cuda")
    with pytest.raises(ValueError, match="more than once"):
        mm.resolve_duplicates(pairs, 5, order=[0, 1, 2, 1])
    for bad in ([0, 5], [-1, 2]):
        with pytest.raises(ValueError, match="order id"):
            mm.resolve_duplicates(pairs, 5, order=bad)
    for bad in ([[0, 5]], [[-1, 2]]):
        with pytest.raises(ValueError, match="pair id"):
            mm.resolve_duplicates(torch.tensor(bad, dtype=torch.int64, device="cuda"), 5)
    with pytest.raises(ValueError, match="2\\^31"):
        mm.resolve_duplicates(pairs, 2 ** 31)
    rng = np.random.default_rng(4)
    p = torch.from_numpy(clustered_pairs(rng, 20_000, frac=0.5)).cuda()
    order = torch.from_numpy(rng.permutation(20_000)).cuda()
    a = mm.resolve_duplicates(p, 20_000, order=order)
    b = mm.resolve_duplicates(p, 20_000, order=order)
    assert torch.equal(a, b)


def near_copies(n_base, d, seed):
    """Unit rows: bases and 1-4 copies of each at cosines 0.955-0.995 to their base with independent noise, so
    two copies of a base meet at about the product of their cosines -- above 0.95 or not.  The clusters are not
    cliques and the walk order decides which rows survive."""
    gen = torch.Generator().manual_seed(seed)
    base = torch.nn.functional.normalize(torch.randn(n_base, d, generator=gen), dim=1)
    rows = [base]
    for k in range(4):
        take = torch.rand(n_base, generator=gen) < 0.6 / (k + 1)
        b = base[take]
        c = 0.955 + 0.04 * torch.rand(b.shape[0], 1, generator=gen)
        r = torch.randn(b.shape, generator=gen)
        r = torch.nn.functional.normalize(r - (r * b).sum(1, keepdim=True) * b, dim=1)
        rows.append(c * b + (1 - c * c).sqrt() * r)
    x = torch.cat(rows)
    return x[torch.randperm(x.shape[0], generator=gen)].contiguous()


@pytest.mark.parametrize("method", ["fp32", "tc"])
def test_deduplicate_equals_pairs_then_host_walk(mm, method):
    x = near_copies(2500, 128, seed=2)
    n = x.shape[0]
    pairs = mm.find_duplicate_pairs(x, 0.95, method=method)
    assert pairs.shape[0] > 500
    rng = np.random.default_rng(0)
    outcomes = set()
    for order in (None, rng.permutation(n), rng.permutation(n)):
        walk = list(range(n)) if order is None else order.tolist()
        want = mm.greedy_first_keeper(n, pairs, walk)
        outcomes.add(len(want[0]))
        for inp in (x, x.cuda()):
            rep = mm.deduplicate(inp, 0.95, order=order, method=method)
            assert rep.is_cuda == inp.is_cuda
            reps, dups = walk_of(rep.cpu(), walk)
            assert reps == want[0] and dups == [tuple(d) for d in want[1]]
    assert len(outcomes) > 1            # the order changes how many rows survive: the clusters are not cliques


def test_keep_mask_feeds_the_row_filter(mm, oracle):
    """RowFilter(rep == arange) searches exactly the gallery without its duplicates."""
    x = near_copies(3000, 128, seed=6)
    n = x.shape[0]
    rep = mm.deduplicate(x.cuda(), 0.95)
    keep = rep == torch.arange(n, device=rep.device)
    assert 3000 <= int(keep.sum()) < n
    g16 = x.to(torch.bfloat16)
    q = oracle.synthetic_queries(16, 128, seed=1)
    v, i = mm.search_topk(q, mm.DeviceGallery(g16), 10, row_filter=mm.RowFilter(keep))
    rows = keep.nonzero()[:, 0]
    sv, si = mm.search_topk(q, mm.DeviceGallery(g16[rows.cpu()]), 10)
    assert torch.equal(i, rows[si.to(rows.device)].to(i.device)) and torch.equal(v, sv)
