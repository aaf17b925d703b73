"""search_range on a B200: the result equals `S >= t` of full_scores of the same batch (same pinned path), bit for
bit -- offsets, indices in row order, values (with -0.0 as +0.0) -- over every scan kernel, threshold edges,
row windows, row filters and labels, NaN and signed-zero scores, and the chain best_thresholds -> search_range."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N, D = 20_001, 100                 # ragged N, D not a multiple of 8


def make_gallery(mm, oracle, mode, n=N, d=D, seed=0):
    g = oracle.synthetic_gallery(n, d, seed=seed, dtype=torch.bfloat16 if mode == "bf16" else torch.float32)
    return mm.DeviceGallery(g, mode=mode)


def expected(S, thr32, allowed=None):
    """The contract: mask = S >= t (and `allowed` [Q, N] or [N]), CSR in row order, -0.0 as +0.0."""
    mask = S >= thr32.to(S.device)[:, None]
    if allowed is not None:
        mask &= allowed.to(S.device)
    off = torch.zeros(S.shape[0] + 1, dtype=torch.int64, device=S.device)
    torch.cumsum(mask.sum(1), 0, out=off[1:])
    return off, S[mask] + 0.0, mask.nonzero()[:, 1]


def assert_same(got, want):
    assert torch.equal(got[0].cpu(), want[0].cpu())
    assert torch.equal(got[2].cpu(), want[2].cpu())
    assert torch.equal(got[1].cpu().view(torch.int32), want[1].cpu().view(torch.int32))


def mixed_thresholds(S):
    """Per query, in turn: about 0.1 % of the rows, about 10 %, -inf (every row), above the maximum (none);
    the first two planted exactly on a score."""
    srt = S.sort(1, descending=True).values
    n = S.shape[1]
    t = torch.empty(S.shape[0], dtype=torch.float32, device=S.device)
    for j in range(S.shape[0]):
        kind = j % 4
        t[j] = (srt[j, n // 1000] if kind == 0 else srt[j, n // 10] if kind == 1 else
                float("-inf") if kind == 2 else srt[j, 0] + 1.0)
    return t


def run(mm, q, gal, thr, path="auto", normalize_queries=True, scale=1.0, allowed=None, **kw):
    got = mm.search_range(q, gal, thr, path=path, normalize_queries=normalize_queries, scale=scale, **kw)
    S = mm.full_scores(q, gal, path=path, normalize_queries=normalize_queries, scale=scale)
    from mmrs_b200.range_search import thresholds_f32
    assert_same(got, expected(S, thresholds_f32(thr, S.shape[0]), allowed))
    return got, S


# bf16: K1 (1, 2), K2 single (16), pair (100, 200), multi-chunk (600); fp32: K1 (5), bf16x3 single (20) and pair (100)
@pytest.mark.parametrize("mode,nq", [("bf16", 1), ("bf16", 2), ("bf16", 16), ("bf16", 100), ("bf16", 200),
                                     ("bf16", 600), ("fp32", 5), ("fp32", 20), ("fp32", 100)])
def test_contract_every_kernel(mm, oracle, mode, nq):
    gal = make_gallery(mm, oracle, mode, seed=nq)
    q = oracle.synthetic_queries(nq, D, seed=nq).cuda()
    thr = mixed_thresholds(mm.full_scores(q, gal))
    got, _ = run(mm, q, gal, thr)
    counts = (got[0][1:] - got[0][:-1]).cpu()
    assert counts[0] >= N // 1000 and (nq < 3 or counts[2] == N)
    if nq >= 4:
        assert counts[3] == 0 and counts[1] >= N // 10


def test_threshold_edges(mm, oracle):
    gal = make_gallery(mm, oracle, "bf16", seed=3)
    q = oracle.synthetic_queries(4, D, seed=3).cuda()
    S = mm.full_scores(q, gal)
    s0 = S[:, 1234].clone()                                              # a score of every query
    inf = torch.full_like(s0, float("inf"))
    for t in (s0, torch.nextafter(s0, inf), torch.nextafter(s0, -inf)):  # on a score, one ulp either side
        got, _ = run(mm, q, gal, t)
        row = got[2][got[0][0]:got[0][1]].cpu()
        assert (1234 in row.tolist()) == bool((t[0] <= s0[0]).item())
    # float64 thresholds strictly between two float32 values: float64(score) >= t, as numpy compares
    lo = s0.double().cpu()
    hi = torch.nextafter(s0, inf).double().cpu()
    t64 = (lo + hi) / 2
    assert ((t64 > lo) & (t64 < hi)).all()
    off, vals, idx = mm.search_range(q, gal, t64)
    Sn = S.cpu().numpy()
    mask = Sn.astype(np.float64) >= t64.numpy()[:, None]
    assert off.cpu().tolist() == [0] + np.cumsum(mask.sum(1)).tolist()
    assert np.array_equal(idx.cpu().numpy(), np.nonzero(mask)[1])
    assert 1234 not in idx[off[0]:off[1]].tolist()
    got_scalar = mm.search_range(q, gal, float(t64[0]))                  # a Python float applies to every query
    assert_same(got_scalar, expected(S, torch.nextafter(s0[0:1], inf[0:1]).expand(4)))
    for bad in (float("nan"), torch.tensor([0.0, 0.1, float("nan"), 0.2])):
        with pytest.raises(ValueError):
            mm.search_range(q, gal, bad)


@pytest.mark.parametrize("mode,nq", [("bf16", 16), ("fp32", 5), ("fp32", 20)])
def test_windows_equal_one_window(mm, oracle, mode, nq):
    gal = make_gallery(mm, oracle, mode, seed=7)
    q = oracle.synthetic_queries(nq, D, seed=7).cuda()
    thr = mixed_thresholds(mm.full_scores(q, gal))
    from mmrs_b200.range_search import window_rows
    small = nq * 8 * 7040
    assert -(-N // window_rows(nq, N, small)) >= 3
    one, _ = run(mm, q, gal, thr)
    many, _ = run(mm, q, gal, thr, max_candidate_bytes=small)
    for a, b in zip(one, many):
        assert torch.equal(a, b)


def test_row_filter_and_labels(mm, oracle):
    gal = make_gallery(mm, oracle, "bf16", seed=9)
    nq = 16
    q = oracle.synthetic_queries(nq, D, seed=9).cuda()
    thr = mixed_thresholds(mm.full_scores(q, gal))
    rng = np.random.default_rng(9)
    mask = torch.from_numpy(rng.random(N) < 0.3)
    f = mm.RowFilter(mask)
    for rf in (f, mask, mask.cuda()):
        run(mm, q, gal, thr, row_filter=rf, allowed=mask[None, :])
    lab = rng.integers(0, 5, N)
    L = mm.RowLabels(lab)
    ql = torch.from_numpy(rng.integers(-1, 6, nq))                        # -1: unrestricted; 5: no row has it
    ql[0] = -1
    labt = torch.from_numpy(lab)
    for match in ("same", "other"):
        same = labt[None, :] == ql[:, None]
        allowed = (ql[:, None] < 0) | (same if match == "same" else ~same)
        run(mm, q, gal, thr, row_labels=L, query_labels=ql, label_match=match, allowed=allowed)
        run(mm, q, gal, thr, row_labels=L, query_labels=ql.cuda(), label_match=match, row_filter=f,
            allowed=allowed & mask[None, :])
    none = mm.RowFilter(torch.zeros(N, dtype=torch.bool))
    off, vals, idx = mm.search_range(q, gal, thr, row_filter=none)
    assert off.tolist() == [0] * (nq + 1) and vals.numel() == 0 and idx.numel() == 0 and off.is_cuda


# fp32 K1 (3), bf16x3 (12) and bf16 K2 (20): K2 also appends a NaN row to its padded query columns, which
# must not reach the result
@pytest.mark.parametrize("mode,nq", [("fp32", 3), ("fp32", 12), ("bf16", 20)])
def test_nan_and_signed_zero(mm, oracle, mode, nq):
    g = oracle.synthetic_gallery(N, D, seed=11, dtype=torch.float32)
    g[7, 5] = float("nan")                                               # row 7 scores NaN for every query
    g[9] = 0.0                                                           # row 9 scores 0; with scale < 0 it is -0.0
    gal = mm.DeviceGallery(g.to(torch.bfloat16) if mode == "bf16" else g, mode=mode)
    q = oracle.synthetic_queries(nq, D, seed=11).cuda()
    got, S = run(mm, q, gal, float("-inf"))
    assert torch.isnan(S[:, 7]).all()
    counts = (got[0][1:] - got[0][:-1]).cpu()
    assert (counts == N - 1).all() and 7 not in got[2].tolist()
    got, S = run(mm, q, gal, 0.0, scale=-1.0)
    assert (S[:, 9].cpu().view(torch.int32) == -2 ** 31).all()          # full_scores has -0.0 there
    for j in range(nq):
        seg = got[2][got[0][j]:got[0][j + 1]]
        k = int((seg == 9).nonzero()[0, 0])
        assert got[1][got[0][j] + k].cpu().view(torch.int32).item() == 0     # returned as +0.0


@pytest.mark.parametrize("path", ["mma", "gemv"])
def test_chain_best_thresholds(mm, oracle, path):
    n_classes = 10
    gal = make_gallery(mm, oracle, "bf16", seed=13)
    lab = np.random.default_rng(13).integers(0, n_classes, N)
    L = mm.RowLabels(lab)
    classes = np.arange(n_classes)
    protos = oracle.synthetic_queries(n_classes, D, seed=13)
    protos = protos + 3.0 * torch.from_numpy(np.stack([(lab == c).astype(np.float32) for c in classes])) @ \
        oracle.synthetic_gallery(N, D, seed=13, dtype=torch.float32) / N            # a little class signal
    best_f1, best_thr, best_p, best_r, _, _ = mm.best_thresholds(protos, gal, L, classes, path=path)
    off, vals, idx = mm.search_range(protos, gal, best_thr, scale=100., normalize_queries=False, path=path)
    checked = 0
    for c in classes:
        if not best_f1[c] > 0:
            continue
        rows = idx[off[c]:off[c + 1]].cpu().numpy()
        tp = np.int64((lab[rows] == c).sum())
        fp = np.int64(rows.size) - tp
        n_pos = np.int64((lab == c).sum())
        assert tp / (tp + fp) == best_p[c] and tp / n_pos == best_r[c], c
        checked += 1
    assert checked >= n_classes // 2


def test_other_cases(mm, oracle):
    gal = make_gallery(mm, oracle, "bf16", seed=17)
    q = oracle.synthetic_queries(100, D, seed=17)
    thr = mixed_thresholds(mm.full_scores(q.cuda(), gal))
    on_dev = mm.search_range(q.cuda(), gal, thr)
    on_host = mm.search_range(q, gal, thr.cpu())
    assert all(x.is_cuda for x in on_dev) and not any(x.is_cuda for x in on_host)
    for a, b in zip(on_dev, on_host):
        assert torch.equal(a.cpu(), b)
    again = mm.search_range(q.cuda(), gal, thr)                          # atomic append order does not show
    for a, b in zip(on_dev, again):
        assert torch.equal(a, b)
    off, vals, idx = mm.search_range(q[:0], gal, thr[:0])
    assert off.tolist() == [0] and vals.numel() == 0 and idx.numel() == 0
    z = q[:3].clone()
    z[1] = 0.0
    with pytest.raises(RuntimeError):
        mm.search_range(z, gal, 0.0)
    with pytest.raises(ValueError):
        mm.search_range(torch.randn(2, D + 1), gal, 0.0)
    with pytest.raises(ValueError):
        mm.search_range(q, gal, thr[:5])
    with pytest.raises(ValueError):
        mm.search_range(q, gal, thr, row_filter=torch.ones(N - 1, dtype=torch.bool))


def test_row_offset_is_added(mm, oracle):
    g = oracle.synthetic_gallery(N, D, seed=19)
    gal = mm.DeviceGallery(g, row_offset=1_000_000)
    q = oracle.synthetic_queries(16, D, seed=19).cuda()
    thr = mixed_thresholds(mm.full_scores(q, gal))
    off, vals, idx = mm.search_range(q, gal, thr)
    ref = mm.search_range(q, mm.DeviceGallery(g), thr)
    assert torch.equal(off, ref[0]) and torch.equal(vals, ref[1]) and torch.equal(idx, ref[2] + 1_000_000)
