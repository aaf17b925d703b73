"""Row-filtered search_topk on the GPU: the result must be the unfiltered search of the subset
gallery `g[mask]` with its indices mapped back through `nonzero(mask)` -- identical values and
indices, since every row's score depends only on that row and the query (same kernel, same
arithmetic), plus the edge cases, the overflow fallback and the graph cache."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N, D = 200_003, 200          # ragged rows (1563 tiles, a multi-phase plan), D not a multiple of 64
SEED_STRIDE = 32             # every plan of this N samples tiles t % 32 == 0 (or a subset of them) first


def make_masks():
    rng = np.random.default_rng(7)
    tiles = np.arange(N) // 128
    masks = {"all": np.ones(N, dtype=bool)}
    for name, p in (("p50", 0.5), ("p10", 0.1), ("p1", 0.01), ("p01", 0.001)):
        masks[name] = rng.random(N) < p
    # a class-sorted gallery (10 classes of N / 10 rows, as the reference's caches are built) and one class
    block = np.zeros(N, dtype=bool)
    block[3 * (N // 10):4 * (N // 10)] = True
    masks["class_block"] = block
    # no row of any seed tile: the seed select sees no allowed row (thr = -inf, every later row appended);
    # sparse elsewhere so that the appends stay within the candidate lists (overflow is tested below)
    masks["no_seed"] = (tiles % SEED_STRIDE != 0) & (rng.random(N) < 0.01)
    return masks


@pytest.fixture(scope="module")
def data(mm, oracle):
    g32 = oracle.synthetic_gallery(N, D, seed=11, dtype=torch.float32)
    g16 = g32.to(torch.bfloat16)
    masks = make_masks()
    dev = torch.device("cuda", 0)
    gals = {"fp32": mm.DeviceGallery(g32, mode="fp32"), "bf16": mm.DeviceGallery(g16, mode="bf16")}
    filters = {name: mm.RowFilter(torch.from_numpy(m), device=dev) for name, m in masks.items()}
    return {"g": {"fp32": g32, "bf16": g16}, "gal": gals, "masks": masks, "filters": filters, "subsets": {}}


def subset(mm, data, mode, name):
    key = (mode, name)
    if key not in data["subsets"]:
        rows = torch.from_numpy(np.nonzero(data["masks"][name])[0])
        data["subsets"][key] = (mm.DeviceGallery(data["g"][mode][rows], mode=mode), rows.cuda())
    return data["subsets"][key]


def assert_subset_equal(mm, data, mode, name, q, k, **kw):
    gal, f = data["gal"][mode], data["filters"][name]
    v, i = mm.search_topk(q, gal, k, row_filter=f, **kw)
    sub_gal, rows = subset(mm, data, mode, name)
    sv, si = mm.search_topk(q, sub_gal, k, **kw)
    assert torch.equal(i, rows[si]), (mode, name, k, int((i != rows[si]).sum()))
    assert torch.equal(v, sv), (mode, name, k, (v - sv).abs().max().item())
    return v, i


@pytest.mark.parametrize("mode,nq", [("fp32", 3), ("fp32", 12), ("fp32", 60),
                                     ("bf16", 1), ("bf16", 2), ("bf16", 16), ("bf16", 100), ("bf16", 600)])
@pytest.mark.parametrize("name", ["all", "p50", "p10", "p1", "p01", "class_block", "no_seed"])
def test_filtered_equals_subset_gallery(mm, oracle, data, mode, nq, name):
    q = oracle.synthetic_queries(nq, D, seed=nq).cuda()
    n_allowed = data["filters"][name].n_allowed
    for k in (1, 10, 100, 1024):
        if k > n_allowed:
            with pytest.raises(RuntimeError, match="out of range"):
                mm.search_topk(q, data["gal"][mode], k, row_filter=data["filters"][name])
            continue
        v, i = assert_subset_equal(mm, data, mode, name, q, k)
        if name == "all":     # the all-true filter is the unfiltered search, bit for bit
            uv, ui = mm.search_topk(q, data["gal"][mode], k)
            assert torch.equal(v, uv) and torch.equal(i, ui)


def test_filtered_matches_torch_oracle(mm, oracle, data):
    mask = data["masks"]["p10"]
    q = oracle.synthetic_queries(5, D, seed=3)
    rows = torch.from_numpy(np.nonzero(mask)[0])
    want_v, want_i = oracle.search_topk(q, data["g"]["fp32"][rows], 10, mode="fp32")
    v, i = mm.search_topk(q, data["gal"]["fp32"], 10, row_filter=data["filters"]["p10"])
    np.testing.assert_allclose(v.numpy(), want_v.numpy(), atol=1e-5, rtol=0)
    assert int((i != rows[want_i]).sum()) <= 1
    assert mask[i.numpy()].all()


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_overflow_takes_the_filtered_exhaustive_path(mm, oracle, data, monkeypatch, mode):
    """Every seed tile excluded and every other row allowed: after the seed select thr = -inf, so the
    next phase appends every row of its tiles and outgrows the candidate lists -> MMRS_ERR_RETRY -> the
    filtered exhaustive path, which must still give the subset's exact top-k (one query: the exhaustive
    path's per-query K1 pass is the very kernel the subset search runs)."""
    from mmrs_b200 import search
    calls = []
    real = search._search_exhaustive
    monkeypatch.setattr(search, "_search_exhaustive", lambda *a, **kw: (calls.append(kw), real(*a, **kw))[1])
    tiles = np.arange(N) // 128
    mask = tiles % SEED_STRIDE != 0
    f = mm.RowFilter(torch.from_numpy(mask), device=data["gal"][mode].device)
    rows = torch.from_numpy(np.nonzero(mask)[0]).cuda()
    sub = mm.DeviceGallery(data["g"][mode][rows.cpu()], mode=mode)
    q = oracle.synthetic_queries(1, D, seed=5).cuda()
    for k in (10, 100):
        v, i = mm.search_topk(q, data["gal"][mode], k, row_filter=f)
        sv, si = mm.search_topk(q, sub, k)
        assert torch.equal(i, rows[si]) and torch.equal(v, sv)
    assert len(calls) == 2, "the candidate lists did not overflow: the retry path was not exercised"
    # several queries: the retry re-scores on K1 one query at a time while the batch ran on K2 (bf16) --
    # the arithmetic of the unfiltered retry too: same rows, values within the fp32 summation-order noise
    q = oracle.synthetic_queries(16, D, seed=6).cuda()
    v, i = mm.search_topk(q, data["gal"][mode], 100, row_filter=f)
    sv, si = mm.search_topk(q, sub, 100)
    assert len(calls) == 3
    assert (v - sv).abs().max().item() < 1e-5
    assert int((i != rows[si]).sum()) <= 2


def test_edge_cases(mm, oracle, data):
    gal = data["gal"]["bf16"]
    q = oracle.synthetic_queries(4, D, seed=8).cuda()
    # k == n_allowed: every allowed row, sorted
    mask = np.zeros(N, dtype=bool)
    mask[np.random.default_rng(1).choice(N, 37, replace=False)] = True
    f = mm.RowFilter(mask, device=gal.device)
    v, i = mm.search_topk(q, gal, 37, row_filter=f)
    rows = torch.from_numpy(np.nonzero(mask)[0]).cuda()
    sv, si = mm.search_topk(q, mm.DeviceGallery(data["g"]["bf16"][rows.cpu()]), 37)
    assert torch.equal(i, rows[si]) and torch.equal(v, sv)
    assert torch.equal(torch.sort(i, dim=1).values, rows.expand(4, -1))
    for bad_k in (38, 1024):
        with pytest.raises(RuntimeError, match="out of range"):
            mm.search_topk(q, gal, bad_k, row_filter=f)
        with pytest.raises(RuntimeError, match="out of range"):
            mm.search_topk(q, gal, bad_k, row_filter=torch.from_numpy(mask))
    with pytest.raises(RuntimeError, match="out of range"):                 # all-false
        mm.search_topk(q, gal, 1, row_filter=mm.RowFilter(np.zeros(N, dtype=bool), device=gal.device))
    with pytest.raises(ValueError):                                           # wrong length
        mm.search_topk(q, gal, 5, row_filter=mm.RowFilter(mask[:-1], device=gal.device))
    with pytest.raises(ValueError):
        mm.search_topk(q, gal, 5, row_filter=torch.from_numpy(mask[1:]))
    with pytest.raises(ValueError):                                           # not a bool mask
        mm.search_topk(q, gal, 5, row_filter=torch.from_numpy(mask).to(torch.uint8))
    with pytest.raises(ValueError):                                           # another device
        mm.search_topk(q, gal, 5, row_filter=mm.RowFilter._wrap(f.words.cpu(), N, f.n_allowed))
    # a per-call bool mask (host numpy or device tensor) equals the packed RowFilter
    mp = data["masks"]["p1"]
    fv, fi = mm.search_topk(q, gal, 100, row_filter=data["filters"]["p1"])
    for m in (mp, torch.from_numpy(mp).cuda()):
        mv, mi = mm.search_topk(q, gal, 100, row_filter=m)
        assert torch.equal(mi, fi) and torch.equal(mv, fv)
    # host queries -> host results, identical; out= tensors; scale
    hv, hi = mm.search_topk(q.cpu(), gal, 100, row_filter=data["filters"]["p1"])
    assert not hv.is_cuda and torch.equal(hi, fi.cpu()) and torch.equal(hv, fv.cpu())
    ov = torch.empty((4, 100), dtype=torch.float32, device="cuda"); oi = torch.empty((4, 100), dtype=torch.int64, device="cuda")
    rv, ri = mm.search_topk(q, gal, 100, row_filter=data["filters"]["p1"], out=(ov, oi))
    assert rv is ov and ri is oi and torch.equal(oi, fi) and torch.equal(ov, fv)
    for scale in (100.0, -1.0):
        for mode, nq in (("bf16", 2), ("bf16", 16), ("fp32", 3), ("fp32", 12)):
            assert_subset_equal(mm, data, mode, "p10", q[:1].repeat(nq, 1) + 0.01 * torch.arange(nq, device="cuda")[:, None],
                                50, scale=scale)


def test_async_two_streams_two_filters(mm, oracle, data):
    gal = data["gal"]["bf16"]
    qs = [oracle.synthetic_queries(24, D, seed=30 + t).cuda() for t in range(4)]
    names = ["p10", "class_block", "p1", "p50"]
    want = [assert_subset_equal(mm, data, "bf16", names[t], qs[t], 100) for t in range(4)]
    streams = [torch.cuda.Stream() for _ in range(2)]
    torch.cuda.synchronize()
    pends = []
    for t in range(4):
        with torch.cuda.stream(streams[t % 2]):
            f = data["filters"][names[t]] if t < 2 else torch.from_numpy(data["masks"][names[t]]).cuda()
            pends.append(mm.search_topk(qs[t], gal, 100, row_filter=f, sync=False))
    for t, p in enumerate(pends):
        v, i = p.wait()
        assert torch.equal(i, want[t][1]) and torch.equal(v, want[t][0]), t


def test_graph_cache_bounded_captures(mm, oracle, data):
    """1000 calls on one shape alternating two RowFilters, per-call bool masks and unfiltered calls:
    correct every time, at most one capture per (slot, filter pointer): the two filters and the slot's
    own mask bitmap; unfiltered calls keep replaying their graph."""
    lib = mm._cabi.lib
    gal = data["gal"]["bf16"]
    q = oracle.synthetic_queries(8, D, seed=50).cuda()
    fa, fb = data["filters"]["p10"], data["filters"]["class_block"]
    ma, mb = (torch.from_numpy(data["masks"][n]).cuda() for n in ("p1", "p50"))
    want = {"u": mm.search_topk(q, gal, 100)}
    for key, f in (("a", fa), ("b", fb), ("ma", ma), ("mb", mb)):
        want[key] = mm.search_topk(q, gal, 100, row_filter=f)
    stats0 = ctypes_stats(lib)
    seq = [("a", fa), ("ma", ma), ("u", None), ("b", fb), ("mb", mb)]
    for t in range(1000):
        key, f = seq[t % len(seq)]
        v, i = mm.search_topk(q, gal, 100, row_filter=f)
        assert torch.equal(i, want[key][1]) and torch.equal(v, want[key][0]), (t, key)
    stats1 = ctypes_stats(lib)
    assert stats1[0] - stats0[0] == 0, "a warmed-up filter or the unfiltered call was captured again"
    # from cold: a new slot (another k) whose unfiltered graph exists captures at most three more graphs --
    # the two filters and the slot's mask bitmap -- however the calls interleave
    mm.search_topk(q, gal, 99)
    c0 = ctypes_stats(lib)[0]
    for t in range(50):
        key, f = seq[t % len(seq)]
        mm.search_topk(q, gal, 99, row_filter=f)
    assert ctypes_stats(lib)[0] - c0 <= 3


def ctypes_stats(lib):
    import ctypes
    out = (ctypes.c_int64 * 4)()
    assert lib.mmrs_graph_stats(out) == 0
    return list(out)
