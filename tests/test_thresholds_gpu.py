"""best_thresholds on a B200: every row equals best_threshold_on_device of its row of one full_scores matrix,
bit for bit (grid, F1 curve with its NaN positions, best tuple), and the reference's find_thresholds on the
host split of those scores; chunking, row filters and arguments."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def gallery(oracle, n, d, mode, seed=0):
    g = oracle.synthetic_gallery(n, d, seed=seed, dtype=torch.bfloat16 if mode == "bf16" else torch.float32)
    return g


def labels(n, n_classes, sorted_, seed=0):
    if sorted_:
        return (np.arange(n) * n_classes // n).astype(np.int64)
    return np.random.default_rng(seed).integers(0, n_classes, n).astype(np.int64)


def assert_row(got, j, want):
    np.testing.assert_array_equal(got[4][j], want[4])                     # the grid
    np.testing.assert_array_equal(got[5][j], want[5])                     # F1 curve, NaN where it is NaN
    assert (got[0][j], got[1][j], got[2][j], got[3][j]) == tuple(float(x) for x in want[:4])


def check_contract(mm, q, gal, targets, ql, *, n_points=200, path="auto", normalize_queries=False, scale=100.0,
                   rows=None, **kw):
    L = mm.RowLabels(targets)
    got = mm.best_thresholds(q, gal, L, ql, n_points=n_points, path=path, normalize_queries=normalize_queries,
                             scale=scale, **kw)
    S = mm.full_scores(q.cuda(), gal, normalize_queries=normalize_queries, scale=scale, path=path)
    t = torch.from_numpy(targets).cuda()
    for j in (range(q.shape[0]) if rows is None else rows):
        assert_row(got, j, mm.best_threshold_on_device(S[j], t, int(ql[j]), n_points))
    return got, S


@pytest.mark.parametrize("mode,nq,path", [("bf16", 1, "auto"), ("bf16", 2, "auto"), ("bf16", 10, "auto"),
                                          ("bf16", 10, "gemv"), ("fp32", 3, "auto"), ("fp32", 12, "auto")])
def test_contract_per_kernel(mm, oracle, mode, nq, path):
    n, d = 20_001, 100                                                    # ragged N, D not a multiple of 8
    g = gallery(oracle, n, d, mode, seed=nq)
    gal = mm.DeviceGallery(g, mode=mode)
    targets = labels(n, 10, False, seed=nq)
    ql = np.arange(nq) % 10
    q = oracle.synthetic_queries(nq, d, seed=nq)
    got, S = check_contract(mm, q, gal, targets, ql, path=path)
    s = S.cpu().numpy()
    for j in range(min(nq, 3)):                                           # the reference's own arithmetic
        pos, neg = s[j][targets == ql[j]], s[j][targets != ql[j]]
        assert_row(got, j, oracle.find_thresholds(pos, neg))


@pytest.mark.parametrize("n_classes", [2, 10, 1000])
@pytest.mark.parametrize("sorted_", [False, True])
def test_contract_class_counts(mm, oracle, n_classes, sorted_):
    n, d = 30_000, 64
    g = gallery(oracle, n, d, "bf16", seed=n_classes)
    gal = mm.DeviceGallery(g)
    targets = labels(n, n_classes, sorted_, seed=n_classes)
    ql = np.arange(n_classes)
    q = oracle.synthetic_queries(n_classes, d, seed=3)
    rows = range(n_classes) if n_classes <= 10 else list(range(0, n_classes, 37)) + [n_classes - 1]
    check_contract(mm, q, gal, targets, ql, path="mma", rows=rows)


@pytest.mark.parametrize("n_points", [1, 2, 200, 4096])
def test_edge_classes_and_grid_sizes(mm, oracle, n_points):
    n, d = 5_000, 32
    g = gallery(oracle, n, d, "bf16", seed=5)
    gal = mm.DeviceGallery(g)
    targets = labels(n, 4, False, seed=5)
    targets[17] = 6                                                       # a one-row class
    ql = np.array([5, 6, 0, 1])                                           # 5: no row has it
    q = oracle.synthetic_queries(4, d, seed=5)
    got, _ = check_contract(mm, q, gal, targets, ql, n_points=n_points)
    assert np.isnan(got[5][0]).all() and (got[0][0], got[1][0], got[2][0], got[3][0]) == (0, 0, 0, 0)
    everyone = np.full(n, 2, np.int64)                                    # every row in one class: no negatives
    got, _ = check_contract(mm, q[:2], gal, everyone, np.array([2, 3]), n_points=n_points)


@pytest.mark.parametrize("mode,path", [("bf16", "mma"), ("bf16", "gemv"), ("fp32", "gemv")])
def test_chunking_does_not_change_results(mm, oracle, mode, path):
    n, d, nq = 10_000, 64, 7
    gal = mm.DeviceGallery(gallery(oracle, n, d, mode, seed=11), mode=mode)
    L = mm.RowLabels(labels(n, 5, False, seed=11))
    ql = np.arange(nq) % 5
    q = oracle.synthetic_queries(nq, d, seed=11)
    one = mm.best_thresholds(q, gal, L, ql, path=path)
    for per_chunk in (1, 3):
        got = mm.best_thresholds(q, gal, L, ql, path=path, max_score_bytes=4 * n * per_chunk)
        for a, b in zip(got, one):
            np.testing.assert_array_equal(a, b)


def test_row_filter_equals_subset_gallery(mm, oracle):
    n, d, nq = 20_001, 64, 6
    g = gallery(oracle, n, d, "bf16", seed=13)
    targets = labels(n, 3, False, seed=13)
    mask = np.random.default_rng(13).random(n) < 0.3
    ql = np.arange(nq) % 4                                                # 3: absent
    q = oracle.synthetic_queries(nq, d, seed=13)
    gal = mm.DeviceGallery(g)
    for filt in (mm.RowFilter(mask), torch.from_numpy(mask)):
        got = mm.best_thresholds(q, gal, mm.RowLabels(targets), ql, path="mma", row_filter=filt)
        sub = mm.DeviceGallery(g[torch.from_numpy(mask)])
        want = mm.best_thresholds(q, sub, mm.RowLabels(targets[mask]), ql, path="mma")
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b)
    with pytest.raises(ValueError):
        mm.best_thresholds(q, gal, mm.RowLabels(targets), ql, row_filter=mm.RowFilter(np.zeros(n, bool)))


def test_scores_planted_on_grid_points(mm, oracle):
    """fp32 gallery scored by e_0: each score is the row's first value exactly, so rows can sit on grid
    points and one ulp either side of them."""
    grid = np.linspace(np.float32(-1), np.float32(1), 200)
    pts = np.asarray(grid, dtype=np.float32)[::7]
    vals = np.concatenate([[-1, 1], pts, np.nextafter(pts, np.float32(2)), np.nextafter(pts, np.float32(-2)),
                           np.zeros(50)]).astype(np.float32)
    vals = np.clip(vals, -1, 1)
    n = vals.size * 3
    g = torch.zeros((n, 8))
    g[:, 0] = torch.from_numpy(np.tile(vals, 3))
    targets = (np.arange(n) % 3).astype(np.int64)
    mask = np.ones(n, bool)
    mask[5::11] = False
    q = torch.zeros((3, 8))
    q[:, 0] = 1.0
    gal = mm.DeviceGallery(g, mode="fp32")
    ql = np.arange(3)
    kw = dict(normalize_queries=False, scale=1.0, path="gemv")
    got, S = check_contract(mm, q, gal, targets, ql, **kw)
    s = S.cpu().numpy()
    assert np.isin(grid.astype(np.float64), s[0].astype(np.float64)).sum() > 20   # scores exactly on grid points
    for j in range(3):
        assert_row(got, j, oracle.find_thresholds(s[j][targets == j], s[j][targets != j]))
    fgot = mm.best_thresholds(q, gal, mm.RowLabels(targets), ql, row_filter=mm.RowFilter(mask), **kw)
    fwant = mm.best_thresholds(q, mm.DeviceGallery(g[torch.from_numpy(mask)], mode="fp32"),
                               mm.RowLabels(targets[mask]), ql, **kw)
    for a, b in zip(fgot, fwant):
        np.testing.assert_array_equal(a, b)


def test_arguments_and_inputs(mm, oracle):
    n, d = 4_000, 40
    g = gallery(oracle, n, d, "bf16", seed=17)
    gal = mm.DeviceGallery(g)
    targets = labels(n, 4, False, seed=17)
    L = mm.RowLabels(targets)
    q = oracle.synthetic_queries(5, d, seed=17)
    ql = np.array([0, 1, 2, 3, 0])
    host = mm.best_thresholds(q, gal, L, ql)
    for qq, ll in ((q.cuda(), torch.from_numpy(ql).cuda()), (q.numpy(), torch.from_numpy(ql).int()), (q, ql.tolist())):
        for a, b in zip(mm.best_thresholds(qq, gal, L, ll), host):
            np.testing.assert_array_equal(a, b)
    check_contract(mm, q, gal, targets, ql, normalize_queries=True, scale=1.0)
    out = mm.best_thresholds(q[:0], gal, L, ql[:0])
    assert [a.shape for a in out] == [(0,), (0,), (0,), (0,), (0, 200), (0, 200)]
    for bad in (dict(query_labels=np.array([0, -1, 2, 3, 0])), dict(query_labels=np.array([0, 1, 2, 3, 2 ** 31 - 1])),
                dict(row_labels=mm.RowLabels(targets[:-1])), dict(n_points=0), dict(n_points=4097)):
        kw = dict(row_labels=L, query_labels=ql)
        kw.update(bad)
        with pytest.raises(ValueError):
            mm.best_thresholds(q, gal, **kw)
