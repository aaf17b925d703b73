"""Label-conditioned search_topk on the GPU.  For a query with label c the result must be, bit for bit,
that query's row of a row-filtered search of the SAME batch with the mask `L == c` (`L != c` for
"other"): the same kernel path runs, and every row's score depends only on the row and the query.
Plus the unlabeled identity, a torch oracle, the -inf / -1 padding, the combination with a row filter,
the labeled exhaustive retry, the asynchronous forms and the graph cache."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

N, D = 200_003, 200          # ragged rows (1563 tiles, a multi-phase plan), D not a multiple of 64
SEED_STRIDE = 32             # every plan of this N samples tiles t % 32 == 0 (or a subset of them) first


def make_labels():
    rng = np.random.default_rng(17)
    out = {}
    for n_cls in (2, 10, 1000):
        out[f"c{n_cls}_random"] = rng.integers(0, n_cls, N).astype(np.int32)
        out[f"c{n_cls}_sorted"] = (np.arange(N) * n_cls // N).astype(np.int32)   # class by class, like the reference's caches
    return out


@pytest.fixture(scope="module")
def data(mm, oracle):
    g32 = oracle.synthetic_gallery(N, D, seed=11, dtype=torch.float32)
    g16 = g32.to(torch.bfloat16)
    dev = torch.device("cuda", 0)
    labels = make_labels()
    return {"g": {"fp32": g32, "bf16": g16},
            "gal": {"fp32": mm.DeviceGallery(g32, mode="fp32"), "bf16": mm.DeviceGallery(g16, mode="bf16")},
            "labels": labels, "L": {name: mm.RowLabels(torch.from_numpy(l), device=dev) for name, l in labels.items()},
            "filters": {}}


def label_filter(mm, data, name, c, match):
    key = (name, c, match)
    if key not in data["filters"]:
        lab = data["labels"][name]
        data["filters"][key] = mm.RowFilter(torch.from_numpy(lab == c if match == "same" else lab != c),
                                            device=torch.device("cuda", 0))
    return data["filters"][key]


def query_labels_for(data, name, nq, seed):
    """At most four distinct labels per batch (each costs one filtered reference search) plus a few -1."""
    rng = np.random.default_rng(seed)
    present = np.unique(data["labels"][name])
    pool = rng.choice(present, min(4, present.size), replace=False)
    ql = rng.choice(pool, nq).astype(np.int32)
    if nq >= 3:
        ql[rng.choice(nq, max(1, nq // 8), replace=False)] = -1
    return ql


def assert_matches_filtered(mm, data, mode, name, q, ql, k, match, **kw):
    gal = data["gal"][mode]
    v, i = mm.search_topk(q, gal, k, row_labels=data["L"][name], query_labels=torch.from_numpy(ql).cuda(),
                          label_match=match, **kw)
    for c in np.unique(ql):
        rows = torch.from_numpy(np.nonzero(ql == c)[0]).cuda()
        if c < 0:
            fv, fi = mm.search_topk(q, gal, k, **kw)
        else:
            fv, fi = mm.search_topk(q, gal, k, row_filter=label_filter(mm, data, name, int(c), match), **kw)
        assert torch.equal(i[rows], fi[rows]), (mode, name, match, k, int(c), int((i[rows] != fi[rows]).sum()))
        assert torch.equal(v[rows], fv[rows]), (mode, name, match, k, int(c))
    return v, i


@pytest.mark.parametrize("mode,nq", [("bf16", 1), ("bf16", 2), ("fp32", 3), ("fp32", 12),
                                     ("bf16", 16), ("bf16", 100), ("bf16", 600), ("fp32", 60)])
@pytest.mark.parametrize("name", ["c2_random", "c10_random", "c10_sorted", "c1000_random", "c1000_sorted"])
@pytest.mark.parametrize("match", ["same", "other"])
def test_labeled_equals_row_filter_per_label(mm, oracle, data, mode, nq, name, match):
    q = oracle.synthetic_queries(nq, D, seed=nq).cuda()
    ql = query_labels_for(data, name, nq, seed=nq * 7 + len(name))
    for k in (1, 10, 100):
        assert_matches_filtered(mm, data, mode, name, q, ql, k, match)


@pytest.mark.parametrize("mode,nq", [("bf16", 1), ("fp32", 3), ("bf16", 16), ("bf16", 100), ("bf16", 600), ("fp32", 60)])
def test_unlabeled_queries_are_the_unlabeled_search(mm, oracle, data, mode, nq):
    gal, L = data["gal"][mode], data["L"]["c10_random"]
    q = oracle.synthetic_queries(nq, D, seed=100 + nq).cuda()
    uv, ui = mm.search_topk(q, gal, 100)
    for match in ("same", "other"):
        v, i = mm.search_topk(q, gal, 100, row_labels=L, query_labels=torch.full((nq,), -1, dtype=torch.int32),
                              label_match=match)
        assert torch.equal(v, uv) and torch.equal(i, ui)
    ql = np.full(nq, 3, dtype=np.int32)
    ql[::2] = -1
    v, i = mm.search_topk(q, gal, 100, row_labels=L, query_labels=torch.from_numpy(ql))
    rows = torch.from_numpy(np.nonzero(ql < 0)[0]).cuda()
    assert torch.equal(v[rows], uv[rows]) and torch.equal(i[rows], ui[rows])


def test_labeled_matches_torch_oracle(mm, oracle, data):
    lab = data["labels"]["c10_random"]
    q = oracle.synthetic_queries(5, D, seed=3)
    ql = np.array([0, 3, 3, 9, 5], dtype=np.int32)
    for match in ("same", "other"):
        v, i = mm.search_topk(q, data["gal"]["fp32"], 10, row_labels=data["L"]["c10_random"],
                              query_labels=torch.from_numpy(ql), label_match=match)
        for r, c in enumerate(ql):
            rows = torch.from_numpy(np.nonzero(lab == c if match == "same" else lab != c)[0])
            # masked scores, stable index-ascending top-k
            want_v, want_i = oracle.search_topk(q[r:r + 1], data["g"]["fp32"][rows], 10, mode="fp32")
            np.testing.assert_allclose(v[r].numpy(), want_v[0].numpy(), atol=1e-5, rtol=0)
            assert int((i[r] != rows[want_i[0]]).sum()) <= 1
            assert ((lab[i[r].numpy()] == c) == (match == "same")).all()


@pytest.mark.parametrize("mode,nq", [("bf16", 1), ("fp32", 3), ("bf16", 16), ("bf16", 100), ("fp32", 60)])
def test_padding_when_fewer_than_k_eligible(mm, oracle, data, mode, nq):
    gal = data["gal"][mode]
    dev = torch.device("cuda", 0)
    lab = np.zeros(N, dtype=np.int32)
    small = np.random.default_rng(2).choice(N, 5, replace=False)
    lab[small] = 7                                           # a class of 5 rows
    L = mm.RowLabels(lab, device=dev)
    q = oracle.synthetic_queries(nq, D, seed=40 + nq).cuda()
    ninf = float("-inf")
    # a class smaller than k: its 5 rows, then -inf / -1
    v, i = mm.search_topk(q, gal, 10, row_labels=L, query_labels=torch.full((nq,), 7, dtype=torch.int32))
    fv, fi = mm.search_topk(q, gal, 5, row_filter=mm.RowFilter(lab == 7, device=dev))
    assert torch.equal(i[:, :5], fi) and torch.equal(v[:, :5], fv)
    assert (i[:, 5:] == -1).all() and (v[:, 5:] == ninf).all()
    # a label absent from the gallery: every position padded
    v, i = mm.search_topk(q, gal, 10, row_labels=L, query_labels=torch.full((nq,), 12345, dtype=torch.int32))
    assert (i == -1).all() and (v == ninf).all()
    # "other" over a single-class gallery: nothing eligible
    L0 = mm.RowLabels(np.zeros(N, dtype=np.int32), device=dev)
    v, i = mm.search_topk(q, gal, 100, row_labels=L0, query_labels=torch.zeros(nq, dtype=torch.int32),
                          label_match="other")
    assert (i == -1).all() and (v == ninf).all()
    # "same" over it with a mixed batch: the whole gallery, i.e. the unlabeled search
    ql = torch.zeros(nq, dtype=torch.int32)
    ql[::2] = -1
    v, i = mm.search_topk(q, gal, 100, row_labels=L0, query_labels=ql)
    uv, ui = mm.search_topk(q, gal, 100)
    assert torch.equal(v, uv) and torch.equal(i, ui)


@pytest.mark.parametrize("mode,nq", [("bf16", 2), ("fp32", 12), ("bf16", 100)])
def test_labels_combined_with_row_filter(mm, oracle, data, mode, nq):
    gal, name = data["gal"][mode], "c10_sorted"
    lab = data["labels"][name]
    dev = torch.device("cuda", 0)
    allowed = np.random.default_rng(5).random(N) < 0.3
    f = mm.RowFilter(allowed, device=dev)
    q = oracle.synthetic_queries(nq, D, seed=60 + nq).cuda()
    ql = query_labels_for(data, name, nq, seed=61)
    for match in ("same", "other"):
        v, i = mm.search_topk(q, gal, 50, row_filter=f, row_labels=data["L"][name], query_labels=ql, label_match=match)
        for c in np.unique(ql):
            rows = torch.from_numpy(np.nonzero(ql == c)[0]).cuda()
            m = allowed if c < 0 else allowed & ((lab == c) if match == "same" else (lab != c))
            fv, fi = mm.search_topk(q, gal, 50, row_filter=mm.RowFilter(m, device=dev))
            assert torch.equal(i[rows], fi[rows]) and torch.equal(v[rows], fv[rows]), (match, int(c))


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_overflow_takes_the_labeled_exhaustive_path(mm, oracle, data, monkeypatch, mode):
    """Label 1 on every non-seed row, label 0 on every seed row: a label-1 query sees no eligible row in
    the seed sample (thr = -inf), the next phase appends every row of its tiles and outgrows the candidate
    lists -> MMRS_ERR_RETRY -> the labeled exhaustive path, one query at a time with its own label."""
    from mmrs_b200 import search
    calls = []
    real = search._search_exhaustive
    monkeypatch.setattr(search, "_search_exhaustive",
                        lambda *a, **kw: (calls.append(len(a) > 9 and a[9] is not None), real(*a, **kw))[1])
    tiles = np.arange(N) // 128
    lab = (tiles % SEED_STRIDE != 0).astype(np.int32)
    dev = torch.device("cuda", 0)
    L = mm.RowLabels(lab, device=dev)
    rows = torch.from_numpy(np.nonzero(lab == 1)[0]).cuda()
    sub = mm.DeviceGallery(data["g"][mode][rows.cpu()], mode=mode)
    q = oracle.synthetic_queries(1, D, seed=5).cuda()
    for k in (10, 100):
        v, i = mm.search_topk(q, data["gal"][mode], k, row_labels=L, query_labels=torch.ones(1, dtype=torch.int32))
        sv, si = mm.search_topk(q, sub, k)
        assert torch.equal(i, rows[si]) and torch.equal(v, sv)
    assert calls == [True, True], "the candidate lists did not overflow: the labeled retry did not run"
    # a mixed batch: label-1 queries, label-0 queries and unlabeled ones, each retried with its own label
    q = oracle.synthetic_queries(16, D, seed=6).cuda()
    ql = torch.tensor([1, 0, -1, 1] * 4, dtype=torch.int32)
    v, i = mm.search_topk(q, data["gal"][mode], 100, row_labels=L, query_labels=ql)
    assert calls == [True, True, True]
    for c in (1, 0, -1):
        r = (ql == c).nonzero().view(-1).cuda()
        ref = mm.search_topk(q, data["gal"][mode], 100) if c < 0 else \
            mm.search_topk(q, mm.DeviceGallery(data["g"][mode][torch.from_numpy(np.nonzero(lab == c)[0])], mode=mode), 100)
        ref_i = ref[1] if c < 0 else torch.from_numpy(np.nonzero(lab == c)[0]).cuda()[ref[1]]
        # the retry re-scores on K1 one query at a time while the batch ran on K2 (bf16): the same rows,
        # values within the fp32 summation-order noise
        assert (v[r] - ref[0][r]).abs().max().item() < 1e-5
        assert int((i[r] != ref_i[r]).sum()) <= 2


def test_host_async_out_and_two_streams(mm, oracle, data):
    gal, name = data["gal"]["bf16"], "c10_random"
    L = data["L"][name]
    q = oracle.synthetic_queries(24, D, seed=70).cuda()
    ql = query_labels_for(data, name, 24, seed=71)
    want = assert_matches_filtered(mm, data, "bf16", name, q, ql, 100, "same")
    # host queries + host labels -> host results
    hv, hi = mm.search_topk(q.cpu(), gal, 100, row_labels=L, query_labels=torch.from_numpy(ql))
    assert not hv.is_cuda and torch.equal(hi, want[1].cpu()) and torch.equal(hv, want[0].cpu())
    # numpy labels, device queries, out=, sync=False
    ov = torch.empty((24, 100), dtype=torch.float32, device="cuda"); oi = torch.empty((24, 100), dtype=torch.int64, device="cuda")
    p = mm.search_topk(q, gal, 100, row_labels=L, query_labels=ql, out=(ov, oi), sync=False)
    rv, ri = p.wait()
    assert rv is ov and ri is oi and torch.equal(oi, want[1]) and torch.equal(ov, want[0])
    # two streams, four batches in flight with different labels and matches (host labels for two of them)
    qls = [query_labels_for(data, name, 24, seed=80 + t) for t in range(4)]
    matches = ["same", "other", "same", "other"]
    wants = [assert_matches_filtered(mm, data, "bf16", name, q, qls[t], 100, matches[t]) for t in range(4)]
    streams = [torch.cuda.Stream() for _ in range(2)]
    torch.cuda.synchronize()
    pends = []
    for t in range(4):
        with torch.cuda.stream(streams[t % 2]):
            lt = torch.from_numpy(qls[t])
            pends.append(mm.search_topk(q, gal, 100, row_labels=L, query_labels=lt if t >= 2 else lt.cuda(),
                                        label_match=matches[t], sync=False))
    for t, p in enumerate(pends):
        v, i = p.wait()
        assert torch.equal(i, wants[t][1]) and torch.equal(v, wants[t][0]), t


def test_graph_cache_one_capture_for_changing_labels(mm, oracle, data):
    """Query labels go into a buffer of the slot: 300 calls with a different label batch each replay ONE
    graph per (slot, row labels, label_match)."""
    lib = mm._cabi.lib
    gal, name = data["gal"]["bf16"], "c1000_random"
    L = data["L"][name]
    q = oracle.synthetic_queries(8, D, seed=90).cuda()
    rng = np.random.default_rng(91)
    batches = [rng.integers(-1, 1000, 8).astype(np.int32) for _ in range(6)]
    want = [mm.search_topk(q, gal, 77, row_labels=L, query_labels=b) for b in batches]
    c0 = ctypes_stats(lib)[0]
    for t in range(300):
        b = batches[t % len(batches)]
        v, i = mm.search_topk(q, gal, 77, row_labels=L, query_labels=torch.from_numpy(b).cuda() if t % 2 else b)
        assert torch.equal(i, want[t % len(batches)][1]) and torch.equal(v, want[t % len(batches)][0]), t
    assert ctypes_stats(lib)[0] - c0 == 0, "changing query labels caused a new capture"
    # from cold: another k -> exactly one capture for all the label batches
    mm.search_topk(q, gal, 76, row_labels=L, query_labels=batches[0])
    c1 = ctypes_stats(lib)[0]
    for b in batches:
        mm.search_topk(q, gal, 76, row_labels=L, query_labels=b)
    assert ctypes_stats(lib)[0] - c1 == 0


def test_argument_errors_on_device(mm, oracle, data):
    gal = data["gal"]["bf16"]
    q = oracle.synthetic_queries(4, D, seed=8).cuda()
    L = data["L"]["c10_random"]
    with pytest.raises(RuntimeError, match="out of range"):                  # k > N still raises
        mm.search_topk(q, gal, N + 1, row_labels=L, query_labels=np.zeros(4, np.int32))
    with pytest.raises(ValueError):
        mm.search_topk(q, gal, 5, row_labels=mm.RowLabels(np.zeros(N - 1, np.int32)), query_labels=np.zeros(4, np.int32))
    with pytest.raises(ValueError):
        mm.search_topk(q, gal, 5, row_labels=mm.RowLabels._wrap(L.labels.cpu(), N), query_labels=np.zeros(4, np.int32))


def ctypes_stats(lib):
    import ctypes
    out = (ctypes.c_int64 * 4)()
    assert lib.mmrs_graph_stats(out) == 0
    return list(out)
