"""Refined top-k search on a B200 (search_topk(..., refine=RefineStore)), bit for bit:
  scores     every returned value equals full_scores(DeviceGallery(F, store.mode), path="gemv") at its row;
  selection  the output is a stable host sort (score descending, row ascending) of those scores over C_q, the
             indices of the unrefined call with k_c = min(refine_k, N, allowed rows), ties included;
  containment  when C_q holds the store's exact top-k, the result is that gallery's search_topk(path="gemv");
plus row filters, labels (padding), the overflow retry in both sync modes, streams, host queries, out=, the
store's layout and the C ABI's out-of-range candidate check."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def unit_rows(n, d, seed):
    x = np.random.default_rng(seed).standard_normal((n, d)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def bits(v):
    return v.detach().cpu().contiguous().view(torch.int32)


def expected(S, C, k):
    """Stable host sort of S [Q, N] over the candidate rows C [Q, k_c] (-1 = none): the k best as (values, rows),
    -0.0 returned as +0.0, short lists padded with -inf / -1."""
    S, C = S.cpu().numpy(), C.cpu().numpy()
    vals = np.full((C.shape[0], k), -np.inf, dtype=np.float32)
    rows = np.full((C.shape[0], k), -1, dtype=np.int64)
    for q in range(C.shape[0]):
        r = C[q][C[q] >= 0]
        s = S[q, r] + np.float32(0.0)
        order = np.lexsort((r, -s))[:k]
        vals[q, :order.size], rows[q, :order.size] = s[order], r[order]
    return torch.from_numpy(vals), torch.from_numpy(rows)


def check_refined(mm, q, gal, F, store, k, refine_k, **kw):
    """One refined call against the contract; returns the number of queries whose containment case held."""
    v, i = mm.search_topk(q, gal, k, refine=store, refine_k=refine_k, **kw)
    allowed = None
    if kw.get("row_filter") is not None:
        f = kw["row_filter"]
        allowed = f.n_allowed if isinstance(f, mm.RowFilter) else int(f.sum())
    k_c = mm.refine.candidate_k(k, refine_k, gal.n_rows, allowed)
    C = mm.search_topk(q, gal, k_c, **kw)[1]                                   # C_q: the unrefined call with k_c
    ref = mm.DeviceGallery(F, mode=store.mode)
    score_kw = {a: kw[a] for a in ("normalize_queries", "scale") if a in kw}
    S = mm.full_scores(q, ref, path="gemv", **score_kw)
    wv, wi = expected(S, C, k)
    assert torch.equal(i.cpu(), wi), "refined indices differ from a stable sort of the store's scores over C_q"
    assert torch.equal(bits(v), bits(wv)), "refined values differ from full_scores(path='gemv')"
    # containment: where C_q holds the exact top-k, the store gallery's own search_topk(path="gemv")
    ev, ei = mm.search_topk(q, ref, k, path="gemv", **kw)
    ei, Cc = ei.cpu(), C.cpu()
    held = 0
    for r in range(ei.shape[0]):
        want = set(ei[r][ei[r] >= 0].tolist())
        if want <= set(Cc[r].tolist()):
            held += 1
            assert torch.equal(i[r].cpu(), ei[r]) and torch.equal(bits(v[r]), bits(ev[r])), r
    return held


STORES = [("fp32", "host"), ("fp32", "device"), ("bf16", "host"), ("bf16", "device")]
SCORE_ARGS = [dict(), dict(normalize_queries=False), dict(normalize_queries=False, scale=100.0),
              dict(normalize_queries=True, scale=-1.0)]


@pytest.mark.parametrize("d", [8, 100, 512, 768, 1040])
def test_scores_selection_and_containment(mm, d):
    n = 3000 + 7 * d + 13                               # ragged: not whole 128-row tiles
    F = unit_rows(n, d, seed=d)
    F[n - 2] = F[1]                                     # planted exact ties: identical rows score alike everywhere
    F[777] = F[40]
    Ft = torch.from_numpy(F)
    stores = [mm.RefineStore(Ft, mode=m, memory=mem) for m, mem in STORES]
    for s, (m, mem) in zip(stores, STORES):            # the store's rows are DeviceGallery's rows
        assert torch.equal(s.data.cpu().view(torch.int16 if m == "bf16" else torch.int32),
                           mm.DeviceGallery(Ft, mode=m).data.cpu().view(torch.int16 if m == "bf16" else torch.int32))
    held = 0
    case = 0
    for gmode in ("int8", "bf16", "fp32"):
        gal = mm.DeviceGallery(Ft, mode=gmode)
        for store in stores:
            nq = (1, 7, 300)[case % 3]
            q = unit_rows(nq, d, seed=100 + case)
            q[:min(nq, 3)] = F[[1, 40, 1]][:min(nq, 3)] + 0.01 * q[:min(nq, 3)]   # near the tied rows
            qt = torch.from_numpy(q).cuda()
            held += check_refined(mm, qt, gal, Ft, store, 10, 40, **SCORE_ARGS[case % 4])
            case += 1
    assert held > 0, "no query had its exact top-k among the candidates: containment was not exercised"
    for s in stores:
        s.close()


@pytest.mark.parametrize("gmode", ["int8", "bf16"])
@pytest.mark.parametrize("smode", ["fp32", "bf16"])
def test_refine_k_equal_n_is_exact(mm, gmode, smode):
    n, d, k = 700, 96, 25
    F = torch.from_numpy(unit_rows(n, d, seed=3))
    gal = mm.DeviceGallery(F, mode=gmode)
    store = mm.RefineStore(F, mode=smode, memory="host")
    q = torch.from_numpy(unit_rows(40, d, seed=4)).cuda()
    v, i = mm.search_topk(q, gal, k, refine=store, refine_k=n)
    ev, ei = mm.search_topk(q, mm.DeviceGallery(F, mode=smode), k, path="gemv")
    assert torch.equal(i, ei) and torch.equal(bits(v), bits(ev))


def test_row_filter_and_labels(mm):
    n, d, k = 5000 + 33, 128, 10
    F = torch.from_numpy(unit_rows(n, d, seed=7))
    gal = mm.DeviceGallery(F, mode="int8")
    store = mm.RefineStore(F, mode="fp32", memory="device")
    rng = np.random.default_rng(0)
    mask = torch.from_numpy(rng.random(n) < 0.3)
    q = torch.from_numpy(unit_rows(9, d, seed=8)).cuda()
    check_refined(mm, q, gal, F, store, k, 40, row_filter=mask.cuda())
    check_refined(mm, q, gal, F, store, k, 40, row_filter=mm.RowFilter(mask.cuda()))
    few = torch.zeros(n, dtype=torch.bool)
    few[rng.choice(n, 25, replace=False)] = True                 # k_c capped by the 25 allowed rows
    assert mm.refine.candidate_k(k, 40, n, 25) == 25
    check_refined(mm, q, gal, F, store, k, 40, row_filter=mm.RowFilter(few.cuda()))
    lab = rng.integers(0, 5, n).astype(np.int32)
    lab[rng.choice(n, 4, replace=False)] = 9                     # class 9: 4 rows, fewer than k
    L = mm.RowLabels(lab)
    ql = torch.tensor([9, 0, -1, 3, 11, 9, 2, 1, 4], dtype=torch.int32)   # 11: absent from the gallery
    for match in ("same", "other"):
        check_refined(mm, q, gal, F, store, k, 40, row_labels=L, query_labels=ql, label_match=match)
        check_refined(mm, q, gal, F, store, k, 40, row_labels=L, query_labels=ql, label_match=match,
                      row_filter=mm.RowFilter(mask.cuda()))
    v, i = mm.search_topk(q, gal, k, refine=store, row_labels=L, query_labels=ql)
    assert (i[0, 4:] == -1).all() and torch.isinf(v[0, 4:]).all() and (i[4] == -1).all()


@pytest.mark.parametrize("sync", [True, False])
def test_overflow_is_refined_from_the_exhaustive_candidates(mm, monkeypatch, sync):
    """test_int8_gpu.py's tile-stride construction: every tile outside the seed sample beats it, the candidate list
    overflows, and the candidates that are refined must be those of the exhaustive repeat."""
    n, d, k = 70_000, 32, 10
    g = unit_rows(n, d, seed=5)
    q = unit_rows(2, d, seed=9)
    outside = (np.arange(n) // 128) % 16 != 0
    h = g[outside] + 2.0 * q[0]
    g[outside] = h / np.linalg.norm(h, axis=1, keepdims=True)
    F = torch.from_numpy(g)
    gal = mm.DeviceGallery(F, mode="int8")
    store = mm.RefineStore(F, mode="fp32", memory="host")
    import mmrs_b200.search as search_mod
    calls = []
    real = search_mod._search_exhaustive
    monkeypatch.setattr(search_mod, "_search_exhaustive", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    qt = torch.from_numpy(q).cuda()
    res = mm.search_topk(qt, gal, k, refine=store, refine_k=k, sync=sync)
    v, i = res if sync else res.wait()
    assert calls, "the candidate list did not overflow: the exhaustive path was not exercised"
    C = mm.search_topk(qt, gal, k)[1]                 # the unrefined call, itself repeated exhaustively
    wv, wi = expected(mm.full_scores(qt, mm.DeviceGallery(F, mode="fp32"), path="gemv"), C, k)
    assert torch.equal(i.cpu(), wi) and torch.equal(bits(v), bits(wv))


def test_streams_host_queries_and_out(mm):
    n, d, k = 20_000 + 5, 256, 16
    F = torch.from_numpy(unit_rows(n, d, seed=11))
    gal = mm.DeviceGallery(F, mode="int8")
    store = mm.RefineStore(F, mode="bf16", memory="host")
    qa = torch.from_numpy(unit_rows(33, d, seed=12))
    qb = torch.from_numpy(unit_rows(5, d, seed=13))
    want_a = mm.search_topk(qa.cuda(), gal, k, refine=store)
    want_b = mm.search_topk(qb.cuda(), gal, k, refine=store)
    # host queries give host results, equal to the device call
    hv, hi = mm.search_topk(qa, gal, k, refine=store)
    assert not hi.is_cuda and torch.equal(hi, want_a[1].cpu()) and torch.equal(bits(hv), bits(want_a[0]))
    # out= on the host and on the device
    ov, oi = torch.empty((33, k), pin_memory=True), torch.empty((33, k), dtype=torch.int64, pin_memory=True)
    r = mm.search_topk(qa, gal, k, refine=store, out=(ov, oi))
    assert r[0] is ov and torch.equal(oi, want_a[1].cpu())
    dv, di = torch.empty((5, k), device="cuda"), torch.empty((5, k), dtype=torch.int64, device="cuda")
    mm.search_topk(qb.cuda(), gal, k, refine=store, out=(dv, di))
    assert torch.equal(di, want_b[1]) and torch.equal(bits(dv), bits(want_b[0]))
    # two streams in flight, asynchronous, several rounds
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(3):
        with torch.cuda.stream(s1):
            pa = mm.search_topk(qa.cuda(), gal, k, refine=store, sync=False)
        with torch.cuda.stream(s2):
            pb = mm.search_topk(qb, gal, k, refine=store, sync=False)
        assert torch.equal(pa.wait()[1], want_a[1]) and torch.equal(pb.wait()[1], want_b[1].cpu())
    torch.cuda.synchronize()


def test_arguments(mm):
    n, d = 1000, 64
    F = torch.from_numpy(unit_rows(n, d, seed=1))
    gal = mm.DeviceGallery(F, mode="int8")
    store = mm.RefineStore(F, mode="fp32", memory="device")
    q = torch.from_numpy(unit_rows(3, d, seed=2)).cuda()
    with pytest.raises(ValueError, match="refine_k"):
        mm.search_topk(q, gal, 10, refine=store, refine_k=9)
    with pytest.raises(ValueError):
        mm.search_topk(q, gal, 10, refine=mm.RefineStore(F[:-1], mode="fp32", memory="device"))
    with pytest.raises(ValueError):
        mm.search_topk(q, gal, 10, refine=mm.RefineStore(F[:, :-1], mode="fp32", memory="device"))
    with pytest.raises(ValueError):
        mm.search_topk(q, gal, 10, refine=F)
    with pytest.raises(ValueError, match="int8"):
        mm.RefineStore(F, mode="int8")
    host = mm.RefineStore(F, mode="fp32", memory="host")
    host.close()
    with pytest.raises(ValueError, match="closed"):
        mm.search_topk(q, gal, 10, refine=host)


def test_abi_rejects_out_of_range_candidates(mm):
    """mmrs_refine_topk takes candidate lists from outside: a row outside [-1, n_rows) is caught on the device and
    returned as MMRS_ERR_ARG without being read; -1 entries pad."""
    lib, cabi = mm._cabi.lib, mm._cabi
    n, d, nq, kc, k = 300, 64, 2, 8, 4
    F = torch.from_numpy(unit_rows(n, d, seed=21))
    store = mm.RefineStore(F, mode="fp32", memory="device")
    q = torch.from_numpy(unit_rows(nq, d, seed=22)).cuda()
    ws_bytes = lib.mmrs_refine_workspace_bytes(d, nq, kc)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device="cuda")
    v = torch.empty((nq, k), device="cuda")
    i = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def call(cand):
        c = torch.tensor(cand, dtype=torch.int64, device="cuda")
        return lib.mmrs_refine_topk(store.ptr, cabi.DTYPE_F32, n, d, d, q.data_ptr(), nq, d, 1, 1.0, c.data_ptr(), kc,
                                    1000, k, v.data_ptr(), i.data_ptr(), mm.DeviceGallery.aligned_ptr(ws), ws_bytes,
                                    None, stream)

    ok = [[5, 9, 2, -1, -1, -1, -1, -1], [0, 1, 2, 3, 4, 5, 6, 299]]
    assert call(ok) == cabi.OK
    S = mm.full_scores(q, mm.DeviceGallery(F, mode="fp32"), path="gemv")
    wv, wi = expected(S, torch.tensor(ok), k)
    wi = torch.where(wi >= 0, wi + 1000, wi)                     # index_offset
    assert torch.equal(i.cpu(), wi) and torch.equal(bits(v), bits(wv))
    for bad in ([[5, 9, 2, 300, -1, -1, -1, -1], ok[1]], [ok[0], [0, 1, -2, 3, 4, 5, 6, 7]],
                [ok[0], [0, 1, 2, 3, 4, 5, 6, 1 << 40]]):
        assert call(bad) == cabi.ERR_ARG, bad
        assert "candidate" in cabi.last_error()
    assert call(ok) == cabi.OK                                   # the workspace's status word starts clean again
    status = torch.zeros(1, dtype=torch.int32).pin_memory()      # asynchronous form
    c = torch.tensor([[5, 9, 2, 300, -1, -1, -1, -1], ok[1]], dtype=torch.int64, device="cuda")
    assert lib.mmrs_refine_topk(store.ptr, cabi.DTYPE_F32, n, d, d, q.data_ptr(), nq, d, 1, 1.0, c.data_ptr(), kc, 0, k,
                                v.data_ptr(), i.data_ptr(), mm.DeviceGallery.aligned_ptr(ws), ws_bytes,
                                status.data_ptr(), stream) == cabi.OK
    torch.cuda.synchronize()
    assert lib.mmrs_search_status(status.data_ptr()) == cabi.ERR_ARG
    # an int8 store dtype and k > k_cand are refused
    assert lib.mmrs_refine_topk(store.ptr, cabi.DTYPE_I8, n, d, d + 16, q.data_ptr(), nq, d, 1, 1.0, c.data_ptr(), kc,
                                0, k, v.data_ptr(), i.data_ptr(), mm.DeviceGallery.aligned_ptr(ws), ws_bytes, None,
                                stream) == cabi.ERR_ARG
    assert lib.mmrs_refine_topk(store.ptr, cabi.DTYPE_F32, n, d, d, q.data_ptr(), nq, d, 1, 1.0, c.data_ptr(), kc,
                                0, kc + 1, v.data_ptr(), i.data_ptr(), mm.DeviceGallery.aligned_ptr(ws), ws_bytes,
                                None, stream) == cabi.ERR_ARG


def test_host_store_registration(mm):
    """A host store is page-locked host memory read through the device pointer mmrs_host_register returned: its
    pages cannot be registered a second time, and the refused registration leaves no error behind."""
    n, d = 2000, 100
    F = torch.from_numpy(unit_rows(n, d, seed=31))
    store = mm.RefineStore(F, mode="bf16", memory="host")
    assert not store.data.is_cuda and store.data.data_ptr() % 4096 == 0 and store.ptr != 0
    dptr = ctypes.c_void_p()
    assert mm._cabi.lib.mmrs_host_register(store.data.data_ptr(), 4096, ctypes.byref(dptr)) == mm._cabi.ERR_CUDA
    q = torch.from_numpy(unit_rows(3, d, seed=32)).cuda()
    gal = mm.DeviceGallery(F, mode="int8")
    v, i = mm.search_topk(q, gal, 5, refine=store, refine_k=n // 2)
    ev, ei = mm.search_topk(q, mm.DeviceGallery(F, mode="bf16"), 5, path="gemv")
    assert torch.equal(i, ei)
    store.close()
    buf = torch.empty(3 * 4096, dtype=torch.uint8)
    p = (buf.data_ptr() + 4095) // 4096 * 4096
    assert mm._cabi.lib.mmrs_host_register(p, 8192, ctypes.byref(dptr)) == mm._cabi.OK and dptr.value
    assert mm._cabi.lib.mmrs_host_unregister(p) == mm._cabi.OK
