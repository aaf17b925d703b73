"""int8 mode on a B200, bit for bit against the numpy mirror of test_int8_host.py.

The oracle takes the gallery's codes and scales as the device stored them (read back; they are themselves
checked against the mirror's quantisation) and the queries quantised by the mirror.  Queries are passed
already normalised with normalize_queries=False, so that their codes are the mirror's exactly; the normalised
form is checked by path agreement.  Every search path (K1 at 1-2 queries, K2 single CTA up to 64, CTA pairs
65-256, several query chunks from 512) must return the stable descending sort of the oracle's scores."""
import numpy as np
import pytest
import torch

from test_int8_host import quantize_rows, scores, topk

pytestmark = pytest.mark.gpu


def unit_rows(n, d, seed):
    x = np.random.default_rng(seed).standard_normal((n, d)).astype(np.float32)
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def device_codes(gal):
    c, s = gal.int8_codes_scales()
    return c.cpu().numpy(), s.cpu().numpy()


def oracle_scores(gal, q, scale=1.0):
    gc, gs = device_codes(gal)
    qc, qs = quantize_rows(q)
    return scores(qc, qs, gc, gs, scale)


def assert_topk(mm, q, gal, k, S, **kw):
    v, i = mm.search_topk(torch.from_numpy(q).cuda(), gal, k, normalize_queries=False, **kw)
    wv, wi = topk(S, k)
    np.testing.assert_array_equal(i.cpu().numpy(), wi)
    np.testing.assert_array_equal(v.cpu().numpy().view(np.uint32), wv.view(np.uint32))


@pytest.mark.parametrize("src_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("d", [1, 15, 16, 100, 768])
def test_quantizer_matches_mirror(mm, src_dtype, d):
    n = 1_000
    x = unit_rows(n, d, seed=d) * 3.0
    x[1] = 0.0                                                           # zero row
    x[2, :] = 0.0
    x[2, 0] = 127.0
    x[2, 1:min(d, 6)] = [0.5, 1.5, 2.5, -0.5, -2.5][:min(d, 6) - 1]     # exact .5 code boundaries: half to even
    x[3] = np.linspace(-1e3, 1e3, d, dtype=np.float32)                  # wide range
    xt = torch.from_numpy(x).to(src_dtype)
    gal = mm.DeviceGallery(xt.cuda(), mode="int8")
    assert gal.data.dtype == torch.int8 and gal.data.shape == (n, (d + 15) // 16 * 16 + 16)
    assert gal.dtype_code == mm._cabi.DTYPE_I8 and gal.nbytes == n * gal.data.shape[1]
    c, s = device_codes(gal)
    wc, ws = quantize_rows(xt.float().numpy())
    np.testing.assert_array_equal(c, wc)
    np.testing.assert_array_equal(s.view(np.uint32), ws.view(np.uint32))
    if d >= 6:
        assert c[2, :6].tolist() == [127, 0, 2, 2, 0, -2]
    pad = gal.data[:, d:gal.padded_dim].cpu()                            # zero codes up to the padded width
    assert (pad == 0).all()
    # host input goes through the chunked upload and gives the same rows
    assert torch.equal(mm.DeviceGallery(xt, mode="int8").data, gal.data)


@pytest.mark.parametrize("src_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("bad", [float("nan"), float("inf"), float("-inf")])
def test_quantizer_refuses_non_finite(mm, src_dtype, bad):
    x = torch.from_numpy(unit_rows(300, 64, seed=1))
    x[217, 5] = bad
    with pytest.raises(ValueError, match="NaN or an infinity"):
        mm.DeviceGallery(x.to(src_dtype).cuda(), mode="int8")


@pytest.mark.parametrize("d", [1, 15, 16, 100, 512, 768, 1040, 1100])
def test_every_path_bit_exact(mm, d):
    n = 4_000 + 77                                                       # ragged: not a multiple of 128
    g = unit_rows(n, d, seed=d)
    g[100] = g[3000]                                                     # planted exact ties
    g[101] = g[3000]
    g[4050] = g[7]
    gal = mm.DeviceGallery(torch.from_numpy(g), mode="int8")
    for nq in (1, 2, 16, 64, 65, 256, 600):
        q = unit_rows(nq, d, seed=1000 + nq)
        q[nq // 2] = g[3000]                                             # a query that ties rows 100, 101, 3000
        S = oracle_scores(gal, q)
        for k in (1, 10, 100, 1000):
            assert_topk(mm, q, gal, k, S)


def test_full_scores_bit_exact_and_paths_agree(mm):
    n, d = 3_000 + 5, 768
    gal = mm.DeviceGallery(torch.from_numpy(unit_rows(n, d, seed=2)), mode="int8")
    for nq in (1, 3, 16, 100, 300):
        q = unit_rows(nq, d, seed=nq)
        S = oracle_scores(gal, q, scale=100.0)
        qd = torch.from_numpy(q).cuda()
        a = mm.full_scores(qd, gal, normalize_queries=False, scale=100.0, path="gemv")
        b = mm.full_scores(qd, gal, normalize_queries=False, scale=100.0, path="mma")
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        np.testing.assert_array_equal(a.cpu().numpy().view(np.uint32), S.view(np.uint32))
        # normalised queries: the device's own quantisation, the same on both kernels
        qr = qd * 3.0
        a = mm.full_scores(qr, gal, path="gemv")
        b = mm.full_scores(qr, gal, path="mma")
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        v, i = mm.search_topk(qr, gal, 50)
        wv, wi = b.topk(50, dim=1)
        assert torch.equal(v, wv)


def test_negative_scale_ties_and_zero(mm):
    n, d = 2_000, 64
    g = unit_rows(n, d, seed=4)
    g[10:20] = 0.0                                                       # zero rows score +0.0 under any scale
    gal = mm.DeviceGallery(torch.from_numpy(g), mode="int8")
    q = unit_rows(20, d, seed=5)
    S = oracle_scores(gal, q, scale=-3.0)
    for path in ("gemv", "mma"):
        assert_topk(mm, q, gal, 100, S, scale=-3.0, path=path)
        got = mm.full_scores(torch.from_numpy(q).cuda(), gal, normalize_queries=False, scale=-3.0, path=path)
        assert not torch.signbit(got[:, 10:20]).any()


def test_edges_k_above_n_empty_batch_and_bad_queries(mm):
    gal = mm.DeviceGallery(torch.from_numpy(unit_rows(500, 32, seed=6)), mode="int8")
    with pytest.raises(RuntimeError, match="out of range"):
        mm.search_topk(torch.randn(2, 32).cuda(), gal, 501)
    v, i = mm.search_topk(torch.empty(0, 32).cuda(), gal, 10)
    assert v.shape == (0, 10) and i.shape == (0, 10)
    q = torch.randn(3, 32).cuda()
    q[1] = 0.0
    with pytest.raises(mm._cabi.MmrsError) as e:                         # normalize_queries: zero norm as ever
        mm.search_topk(q, gal, 5)
    assert e.value.code == mm._cabi.ERR_ZERO_NORM
    q[1, 3] = float("nan")
    for path in ("gemv", "mma"):
        with pytest.raises(ValueError, match="NaN or an infinity"):
            mm.search_topk(q, gal, 5, normalize_queries=False, path=path)
    with pytest.raises(ValueError, match="NaN or an infinity"):
        mm.full_scores(q, gal, normalize_queries=False)


def test_overflow_takes_the_int8_exhaustive_path(mm, monkeypatch):
    """Scores correlated with the tile-stride pattern (test_search_gpu.py's construction): every tile outside
    the seed sample beats it, the candidate list overflows, and the exhaustive path must be exact."""
    n, d = 70_000, 32
    g = unit_rows(n, d, seed=5)
    q = unit_rows(2, d, seed=9)
    outside = (np.arange(n) // 128) % 16 != 0
    h = g[outside] + 2.0 * q[0]
    g[outside] = h / np.linalg.norm(h, axis=1, keepdims=True)
    gal = mm.DeviceGallery(torch.from_numpy(g), mode="int8")
    import mmrs_b200.search as search_mod
    calls = []
    real = search_mod._search_exhaustive
    monkeypatch.setattr(search_mod, "_search_exhaustive", lambda *a, **kw: calls.append(1) or real(*a, **kw))
    S = oracle_scores(gal, q)
    assert_topk(mm, q, gal, 10, S)
    assert calls, "the candidate list did not overflow: the exhaustive path was not exercised"


def test_row_filter_and_labels(mm):
    n, d = 6_000 + 33, 128
    g = unit_rows(n, d, seed=7)
    gal = mm.DeviceGallery(torch.from_numpy(g), mode="int8")
    rng = np.random.default_rng(0)
    mask = rng.random(n) < 0.3
    lab = rng.integers(0, 5, n).astype(np.int32)
    nq = 70
    q = unit_rows(nq, d, seed=8)
    ql = rng.integers(-1, 7, nq)                                         # -1: unrestricted, 5 and 6: absent labels
    S = oracle_scores(gal, q)
    L = mm.RowLabels(lab)
    for path in ("gemv", "mma"):
        for nqq in (1, 2, nq):
            qq = torch.from_numpy(q[:nqq]).cuda()
            v, i = mm.search_topk(qq, gal, 40, normalize_queries=False, path=path, row_filter=mm.RowFilter(mask))
            wv, wi = topk(np.where(mask[None, :], S[:nqq], -np.inf).astype(np.float32), 40)
            np.testing.assert_array_equal(i.cpu().numpy(), wi)
            np.testing.assert_array_equal(v.cpu().numpy(), wv)
            for match in ("same", "other"):
                v, i = mm.search_topk(qq, gal, 40, normalize_queries=False, path=path, row_labels=L,
                                      query_labels=ql[:nqq], label_match=match)
                for j in range(nqq):
                    ok = np.ones(n, bool) if ql[j] < 0 else ((lab == ql[j]) if match == "same" else (lab != ql[j]))
                    idx = np.flatnonzero(ok)
                    order = idx[np.argsort(-S[j, idx], kind="stable")][:40]
                    m = len(order)
                    np.testing.assert_array_equal(i[j, :m].cpu().numpy(), order)
                    np.testing.assert_array_equal(v[j, :m].cpu().numpy(), S[j, order])
                    assert (i[j, m:] == -1).all() and torch.isinf(v[j, m:]).all()


def test_search_range_and_best_thresholds(mm):
    n, d = 9_000 + 3, 256
    gal = mm.DeviceGallery(torch.from_numpy(unit_rows(n, d, seed=11)), mode="int8")
    nq = 12
    q = torch.from_numpy(unit_rows(nq, d, seed=12)).cuda()
    for path in ("gemv", "mma"):
        S = mm.full_scores(q, gal, path=path)
        t = S.sort(1, descending=True).values[:, 37]
        off, val, idx = mm.search_range(q, gal, t, path=path)
        for j in range(nq):
            want = torch.nonzero(S[j] >= t[j]).flatten()
            assert torch.equal(idx[off[j]:off[j + 1]].cpu(), want.cpu())
            assert torch.equal(val[off[j]:off[j + 1]], S[j, want])
    targets = np.random.default_rng(1).integers(0, 4, n).astype(np.int64)
    ql = np.arange(nq) % 4
    for path in ("gemv", "mma"):
        got = mm.best_thresholds(q, gal, mm.RowLabels(targets), ql, path=path, normalize_queries=False)
        S = mm.full_scores(q, gal, normalize_queries=False, scale=100.0, path=path)
        tt = torch.from_numpy(targets).cuda()
        for j in range(nq):
            want = mm.best_threshold_on_device(S[j], tt, int(ql[j]), 200)
            np.testing.assert_array_equal(got[4][j], want[4])
            np.testing.assert_array_equal(got[5][j], want[5])
            assert (got[0][j], got[1][j], got[2][j], got[3][j]) == tuple(float(x) for x in want[:4])


def test_async_out_and_capture_once(mm):
    n, d = 20_000, 768
    g = unit_rows(n, d, seed=13)
    gal = mm.DeviceGallery(torch.from_numpy(g), mode="int8")
    base = torch.from_numpy(unit_rows(200 * 16, d, seed=14)).cuda().view(200, 16, d)
    mm.search_topk(base[0], gal, 10)
    s0 = np.zeros(4, np.int64)
    mm._cabi.lib.mmrs_graph_stats(s0.ctypes.data)
    kept = [mm.search_topk(base[t], gal, 10, sync=False) for t in range(200)]
    res = [p.wait() for p in kept]
    s1 = np.zeros(4, np.int64)
    mm._cabi.lib.mmrs_graph_stats(s1.ctypes.data)
    assert s1[0] == s0[0] and s1[3] == s0[3] and s1[1] - s0[1] == 200
    for t in (0, 77, 199):
        S = mm.full_scores(base[t], gal)
        wv, wi = S.topk(10, dim=1)
        assert torch.equal(res[t][0], wv)
    v = torch.empty((16, 10), device="cuda"); i = torch.empty((16, 10), dtype=torch.int64, device="cuda")
    rv, ri = mm.search_topk(base[5], gal, 10, out=(v, i))
    assert rv is v and torch.equal(i, res[5][1])
    hv, hi = mm.search_topk(base[5].cpu(), gal, 10)
    assert torch.equal(hi, res[5][1].cpu())


def test_selfjoin_refuses_int8(mm):
    gal = mm.DeviceGallery(torch.from_numpy(unit_rows(300, 32, seed=1)), mode="int8")
    with pytest.raises(ValueError):
        mm.find_duplicate_pairs(gal, 0.9)
    lib = mm._cabi.lib
    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    st = lib.mmrs_selfjoin_pairs(gal.data.data_ptr(), 300, gal.padded_dim, gal.data.stride(0), mm._cabi.DTYPE_I8,
                                 0.9, 0, 300, 0, 0, cnt.data_ptr(), 0, 0, 0)
    assert st == mm._cabi.ERR_ARG
