"""The self-join on bf16 and int8 galleries in their stored format (method="stored"), bit for bit.

bf16: the pair set must be the exact fp32 join's on the stored values widened to fp32,
`find_duplicate_pairs(gal.data.float(), tau, method="fp32")`.  The tensor-core pass multiplies the stored values
exactly, so its margin covers only the fp32 accumulations; families planted tens of fp32 ulps apart around tau (tau is
an attained score of the fp32 chain, emulated in numpy) and rows whose products all have one sign put pairs where
that margin is tight.
int8: the pair set must be every i < j whose int8 score, with the lower row as the query at scale 1, reaches tau:
the numpy mirror of test_int8_host.py on the gallery's own codes and scales."""
import numpy as np
import pytest
import torch

from test_int8_host import scores

pytestmark = pytest.mark.gpu

SHAPES_N = [1, 2, 127, 128, 129, 255, 256, 257, 2047, 2048, 2049, 4225]


def unit_rows(n, d, rng, positive=False):
    x = rng.standard_normal((n, d))
    if positive:
        x = np.abs(x)
    return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)


def to_bf16(x):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).float().numpy()


def fp32_chain(a, b):
    """The exact join's fmaf chain, k ascending, for pairs of bf16-valued rows a[m], b[m]: each bf16 product is exact in
    float64, and so is its sum with the fp32 accumulator, so rounding that sum to float32 is one fmaf."""
    acc = np.zeros(a.shape[0], np.float32)
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    for k in range(a.shape[1]):
        acc = (a64[:, k] * b64[:, k] + acc).astype(np.float32)
    return acc


def bf16_family(n, d, seed, scale_pow=0, positive=False, m=400):
    """n bf16-valued rows scaled by 2^scale_pow: random unit rows, plus one base row and up to m rows at cosine
    0.95 +- 2e-4 from it (tens of fp32 ulps apart).  tau = the fp32-chain score of the family's median pair (an
    attained score).  Returns (rows float32, tau, family scores)."""
    rng = np.random.default_rng(seed)
    x = unit_rows(n, d, rng, positive)
    m = min(m, n - 1)
    if m >= 1:
        a = x[0]
        r = unit_rows(m, d, rng, positive)
        r = r - np.outer(r @ a, a)
        r /= np.linalg.norm(r, axis=1, keepdims=True)
        c = 0.95 + rng.uniform(-2e-4, 2e-4, size=(m, 1))
        b = c * a + np.sqrt(1 - c * c) * r
        if positive:
            b = np.abs(b)
        x[1:m + 1] = b / np.linalg.norm(b, axis=1, keepdims=True)
    x = to_bf16(x) * np.float32(2.0 ** scale_pow)
    if m < 1:
        return x, float(np.float32(0.95 * 4.0 ** scale_pow)), np.zeros(0, np.float32)
    fam = fp32_chain(np.repeat(x[:1], m, 0), x[1:m + 1])
    return x, float(np.sort(fam)[m // 2]), fam


def bf16_gallery(mm, x):
    gal = mm.DeviceGallery(torch.from_numpy(x), mode="bf16")
    assert torch.equal(gal.data[:, :x.shape[1]].float().cpu(), torch.from_numpy(x))   # x is bf16-valued
    return gal


def fp32_reference(mm, gal, tau):
    return mm.find_duplicate_pairs(gal.data.float(), tau, method="fp32")


def stored(mm, gal, tau):
    return mm.find_duplicate_pairs(gal, tau, method="stored")


def panels(gal, tau, world):
    from mmrs_b200.dedup import selfjoin_stored_raw, sort_pairs
    parts = torch.cat([selfjoin_stored_raw(gal, tau, r, world) for r in range(world)])
    return parts.shape[0], sort_pairs(parts, gal.n_rows)


# ---- bf16 --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pair", ["0", "1"], ids=["single_cta", "cta_pair"])
@pytest.mark.parametrize("d", [8, 64, 100, 512, 768])
@pytest.mark.parametrize("n", SHAPES_N + [16_385])
def test_bf16_equals_the_fp32_join_at_every_shape(mm, monkeypatch, n, d, pair):
    monkeypatch.setenv("MMRS_SJ_PAIR", pair)
    x, tau, fam = bf16_family(n, d, seed=n * 7 + d)
    gal = bf16_gallery(mm, x)
    want = fp32_reference(mm, gal, tau)
    got = stored(mm, gal, tau)
    assert torch.equal(got, want)
    if fam.size >= 64:
        assert ((fam >= tau).sum() >= 1) and ((fam < tau).sum() >= 1)
    if n >= 2049:
        for world in (2, 3):
            cnt, merged = panels(gal, tau, world)
            assert cnt == want.shape[0] and torch.equal(merged, want)


@pytest.mark.parametrize("positive", [False, True], ids=["mixed_signs", "one_sign"])
@pytest.mark.parametrize("scale_pow", [0, 3])
@pytest.mark.parametrize("d", [64, 512, 768])
def test_bf16_at_attained_scores_norms_and_signs(mm, d, scale_pow, positive):
    """tau an attained fp32-chain score, and the next float32 on either side; rows of norm 1 and 8; rows whose
    products all have one sign (the accumulation error is largest)."""
    n = 2100
    x, tau, fam = bf16_family(n, d, seed=d + scale_pow, scale_pow=scale_pow, positive=positive)
    gal = bf16_gallery(mm, x)
    sets = []
    for t in (float(np.nextafter(np.float32(tau), np.float32(-np.inf))), tau,
              float(np.nextafter(np.float32(tau), np.float32(np.inf)))):
        want = fp32_reference(mm, gal, t)
        assert torch.equal(stored(mm, gal, t), want), t
        sets.append(set(map(tuple, want.tolist())))
    assert sets[0] >= sets[1] > sets[2]        # the family's median pair scores exactly tau
    assert (0, 1 + int(np.argsort(fam)[fam.size // 2])) in sets[1] - sets[2]


def test_bf16_capacity_regrows(mm):
    from mmrs_b200.dedup import selfjoin_stored_raw, sort_pairs
    x, tau, _ = bf16_family(2500, 64, seed=5)
    gal = bf16_gallery(mm, x)
    want = fp32_reference(mm, gal, tau)
    assert want.shape[0] > 8
    assert torch.equal(sort_pairs(selfjoin_stored_raw(gal, tau, capacity=1), gal.n_rows), want)
    low = float(np.float32(0.2))                    # many candidates and pairs: both buffers regrow
    assert torch.equal(stored(mm, gal, low), fp32_reference(mm, gal, low))


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), float("-inf")], ids=["nan", "inf", "-inf"])
def test_bf16_non_finite_rows_raise(mm, bad):
    x, tau, _ = bf16_family(300, 64, seed=9)
    x[77, 3] = bad
    gal = mm.DeviceGallery(torch.from_numpy(x), mode="bf16")
    with pytest.raises(ValueError, match="non-finite"):
        mm.find_duplicate_pairs(gal, tau, method="stored")
    with pytest.raises(ValueError, match="non-finite"):
        mm.deduplicate(gal, tau, method="stored")


# ---- int8 --------------------------------------------------------------------------------------------------
def int8_gallery(mm, n, d, seed, zero_rows=0):
    """Random unit rows with about n/8 near-copies (cosine 0.9-1.0), some rows zero."""
    rng = np.random.default_rng(seed)
    x = unit_rows(n, d, rng)
    k = n // 8
    if k:
        src, dst = rng.permutation(n)[:2 * k].reshape(2, k)
        x[dst] = x[src] + rng.uniform(0.0, 0.5, (k, 1)) * unit_rows(k, d, rng)
    if zero_rows:
        x[rng.permutation(n)[:zero_rows]] = 0
    return mm.DeviceGallery(torch.from_numpy(x), mode="int8")


def int8_scores(gal):
    """scores(c, s, c, s) of the gallery's own codes and scales: [i, j] is row i as the query."""
    c, s = gal.int8_codes_scales()
    c, s = c.cpu().numpy(), s.cpu().numpy()
    return scores(c, s, c, s)


def mirror_pairs(S, tau):
    """All i < j with S[i, j] >= tau, lexicographic."""
    return torch.from_numpy(np.argwhere(np.triu(S >= np.float32(tau), 1)).astype(np.int64)).reshape(-1, 2)


def attained_tau(S, rank=40):
    """An upper-triangle score with about `rank` scores above it."""
    u = np.sort(S[np.triu_indices(S.shape[0], 1)])[::-1]
    return float(u[min(rank, u.size - 1)]) if u.size else 0.5


@pytest.mark.parametrize("pair", ["0", "1"], ids=["single_cta", "cta_pair"])
@pytest.mark.parametrize("d", [16, 100, 512, 768, 1040, 1100])
@pytest.mark.parametrize("n", SHAPES_N)
def test_int8_equals_the_mirror_at_every_shape(mm, monkeypatch, n, d, pair):
    """tau an attained score (its pairs kept) and the next float32 above it (they go).  At D = 1100, float(dot)
    rounds for large dots."""
    monkeypatch.setenv("MMRS_SJ_PAIR", pair)
    gal = int8_gallery(mm, n, d, seed=n * 3 + d)
    S = int8_scores(gal)
    tau = attained_tau(S)
    at, above = mirror_pairs(S, tau), mirror_pairs(S, np.nextafter(np.float32(tau), np.float32(np.inf)))
    assert torch.equal(stored(mm, gal, tau).cpu(), at)
    assert torch.equal(stored(mm, gal, float(np.nextafter(np.float32(tau), np.float32(np.inf)))).cpu(), above)
    if n >= 2:
        assert at.shape[0] > above.shape[0]
    if n >= 2049:
        want = at
        for world in (2, 3):
            cnt, merged = panels(gal, tau, world)
            assert cnt == want.shape[0] and torch.equal(merged.cpu(), want)


@pytest.mark.parametrize("tau", [0.3, 0.0, -0.05], ids=["positive", "zero", "negative"])
def test_int8_zero_rows_and_low_thresholds(mm, tau):
    """Zero rows (scale 0, every score 0) pair with every row when tau <= 0 and with none above; a negative tau
    keeps tens of thousands of pairs, past the first pair buffer."""
    gal = int8_gallery(mm, 700, 64, seed=4, zero_rows=9)
    want = mirror_pairs(int8_scores(gal), tau)
    if tau < 0:
        assert want.shape[0] > 4096 * 4
    assert torch.equal(stored(mm, gal, tau).cpu(), want)


def test_int8_capacity_regrows(mm):
    from mmrs_b200.dedup import selfjoin_stored_raw, sort_pairs
    gal = int8_gallery(mm, 3000, 128, seed=8)
    S = int8_scores(gal)
    tau = attained_tau(S, 500)
    want = mirror_pairs(S, tau)
    assert torch.equal(sort_pairs(selfjoin_stored_raw(gal, tau, capacity=3), gal.n_rows).cpu(), want)


# ---- C3's generator: both stored joins give the fp32 join's pairs -----------------------------------------
def test_c3_stored_joins_equal_the_fp32_join(mm):
    """20 K x 512 rows of C3's generator.  The int8 score of a pair differs from <x_i, x_j> by at most
    B = sqrt(D)/2 (s_i |x_j| + s_j |s_i c_i|) plus float32 rounding (3 2^-24 of the score), which is at most the
    bound below from the actual scales.  No fp32 score lies within B of tau (the fp32 joins at tau - B and tau + B
    agree), so every predicate within B of the exact one -- int8, and bf16 whose operand rounding moves a score by
    at most (2^-7 + 2^-16) |a| |b| < B -- selects the same pairs."""
    import sys
    from pathlib import Path
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
    from bench_dedup import c3_data
    tau = float(np.float32(0.95))
    x = c3_data(20_000)
    want = mm.find_duplicate_pairs(x, tau, method="fp32")
    assert want.shape[0] >= 150
    g8 = mm.DeviceGallery(x, mode="int8")
    c, s = g8.int8_codes_scales()
    c64, s64 = c.double(), s.double()
    d = x.shape[1]
    xn = x.double().norm(dim=1)
    qn = (c64 * s64[:, None]).norm(dim=1)
    bound = float((d ** 0.5 / 2) * (s64.max() * xn.max() + s64.max() * qn.max())) + 3 * 2.0 ** -24 * 1.01
    assert 2.0 ** -7 + 2.0 ** -16 < bound < 0.05
    assert torch.equal(mm.find_duplicate_pairs(x, tau - bound, method="fp32"),
                       mm.find_duplicate_pairs(x, tau + bound, method="fp32"))      # the guard band is empty
    assert torch.equal(mm.find_duplicate_pairs(g8, tau, method="stored"), want)
    g16 = mm.DeviceGallery(x, mode="bf16")
    assert torch.equal(mm.find_duplicate_pairs(g16, tau, method="stored"), want)


# ---- deduplicate and argument errors -----------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["bf16", "int8"])
@pytest.mark.parametrize("order", ["identity", "random"])
def test_deduplicate_stored_is_the_greedy_walk(mm, mode, order):
    n = 3000
    if mode == "bf16":
        x, tau, _ = bf16_family(n, 128, seed=2)
        gal = bf16_gallery(mm, x)
    else:
        gal = int8_gallery(mm, n, 128, seed=2)
        tau = attained_tau(int8_scores(gal), 300)
    pairs = mm.find_duplicate_pairs(gal, tau, method="stored")
    walk = list(range(n)) if order == "identity" else np.random.default_rng(1).permutation(n).tolist()
    o = None if order == "identity" else torch.tensor(walk, dtype=torch.int64)
    _, dups = mm.greedy_first_keeper(n, pairs, walk)
    want = torch.arange(n)
    for v, r in dups:
        want[v] = r
    assert len(dups) >= 1      # (a random walk may keep a family member first: the base row is then its only duplicate)
    assert torch.equal(mm.deduplicate(gal, tau, method="stored", order=o).cpu(), want)


def test_argument_errors(mm):
    x = unit_rows(300, 32, np.random.default_rng(0))
    g32 = mm.DeviceGallery(torch.from_numpy(x), mode="fp32")
    g16 = mm.DeviceGallery(torch.from_numpy(x), mode="bf16")
    g8 = mm.DeviceGallery(torch.from_numpy(x), mode="int8")
    for emb in (g32, torch.from_numpy(x), torch.from_numpy(x).cuda()):
        with pytest.raises(ValueError, match="stored"):
            mm.find_duplicate_pairs(emb, 0.9, method="stored")
        with pytest.raises(ValueError, match="stored"):
            mm.deduplicate(emb, 0.9, method="stored")
    for gal in (g16, g8):
        with pytest.raises(ValueError):
            mm.find_duplicate_pairs(gal, 0.9)           # without "stored" they are refused as before
        with pytest.raises(ValueError, match="method must be"):
            mm.find_duplicate_pairs(gal, 0.9, method="int8")
    lib, C = mm._cabi.lib, mm._cabi
    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    out = torch.empty((16, 2), dtype=torch.int64, device="cuda")
    ws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    wp = mm.DeviceGallery.aligned_ptr(ws)

    def call(gal, dtype, margin=0.0):
        return lib.mmrs_selfjoin_pairs_stored(gal.data.data_ptr(), dtype, gal.data.stride(0), 300, gal.padded_dim,
                                              0.9, margin, 0, 1, out.data_ptr(), 16, cnt.data_ptr(), 16, wp,
                                              (1 << 20) - 256, 0)
    assert call(g32, C.DTYPE_F32) == C.ERR_ARG
    assert call(g16, C.DTYPE_BF16X3) == C.ERR_ARG
    assert call(g8, C.DTYPE_I8, margin=0.01) == C.ERR_ARG
    assert call(g8, C.DTYPE_I8) == C.OK and call(g16, C.DTYPE_BF16, margin=0.01) == C.OK
