"""Both CUDA self-joins against a float64 reference, on data at the edges of bf16 and fp32 rounding.

The reference scores the fp32 rows in float64.  An fp32 dot product of d terms is within
delta = d 2^-24 / (1 - d 2^-24) |a| |b| of it, so every pair scoring >= tau + delta must be emitted, none
scoring < tau - delta may be, and inside that band the tensor-core join (bf16 prefilter + fp32 recheck) must
take the exact mode's decision, whose arithmetic its recheck repeats.  The data plants pairs whose every
entry rounds to bf16 in the same direction, so the prefilter's score moves by nearly the most it can:
"shrinking" pairs just above tau score far below it in bf16, "growing" pairs just below tau score above it,
and "at threshold" pairs sit within a few fp32 ulps of tau.  Each family checks on the CPU that its case is
present."""
import functools

import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

TAU = float(np.float32(0.95))      # the kernels compare in fp32; the reference uses this exact value
OLD_MARGIN = 0.0045                # the unit-row margin this join used before it covered bf16's 2^-8 roundoff


def _families(n: int, d: int, seed: int, k: int, at_threshold: bool, n_fam: int = 48):
    """n rows scaled by 2^k: random unit rows, with up to n_fam pairs of each family planted at random rows
    (shrinking and growing pairs keep 2^-12 from tau, beyond the fp32 band).  Returns (rows [n, d] float32
    numpy, tau scaled by 4^k (an fp32 value), planted {family: [(i, j)]})."""
    rng = np.random.default_rng(seed)
    x = O.l2_normalize(torch.randn(n, d, generator=torch.Generator().manual_seed(seed))).numpy()
    m = min(n_fam, n // 6)
    fams = {"shrinking": O.bf16_edge_pairs(m, d, TAU + 2.0 ** -12, TAU + 0.008, False, seed)[0],
            "growing": O.bf16_edge_pairs(m, d, TAU - 0.008, TAU - 2.0 ** -12, True, seed + 1)[0]}
    if at_threshold:
        fams["at_threshold"] = O.threshold_pairs(m, d, TAU, seed + 2)
    slots = rng.permutation(n)[: 2 * len(fams) * m].reshape(len(fams), m, 2)
    planted = {}
    for (name, rows), s in zip(fams.items(), slots):
        x[s.reshape(-1)] = rows
        planted[name] = [(int(min(a, b)), int(max(a, b))) for a, b in s]
    return x * np.float32(2.0 ** k), float(np.float32(TAU * 4.0 ** k)), planted


@functools.lru_cache(maxsize=16)
def _data(n, d, seed, k=0, at_threshold=True):
    """_families plus the float64 reference (must, may) of dedup_pairs_fp32_band."""
    x, tau, planted = _families(n, d, seed, k, at_threshold)
    must, may = O.dedup_pairs_fp32_band(x, tau)
    return x, tau, planted, must, may


def _keys(pairs, n):
    p = pairs.cpu().to(torch.int64)
    return p[:, 0] * n + p[:, 1]


def _check_reference(got, must, may, n):
    """must <= got <= may as pair sets, and got free of repeats (got sorted)."""
    g, mu, ma = _keys(got, n), _keys(must, n), _keys(may, n)
    assert torch.unique(g).numel() == g.numel(), "a pair is emitted twice"
    missing = mu[~torch.isin(mu, g)]
    extra = g[~torch.isin(g, ma)]
    assert missing.numel() == 0, f"{missing.numel()} pairs above tau + delta were dropped, e.g. {divmod(int(missing[0]), n)}"
    assert extra.numel() == 0, f"{extra.numel()} pairs below tau - delta were emitted, e.g. {divmod(int(extra[0]), n)}"


def _bf16_dots(x, pairs):
    b = O.to_bf16_f64(x)
    i, j = np.asarray(pairs).T
    return (b[i] * b[j]).sum(1)


def _exact_dots(x, pairs):
    x64 = x.astype(np.float64)
    i, j = np.asarray(pairs).T
    return (x64[i] * x64[j]).sum(1)


def _tc(xd, tau, rank=0, world=1):
    from mmrs_b200.dedup import selfjoin_tc_raw
    return selfjoin_tc_raw(xd, tau, rank, world)


def _sorted(pairs, n):
    from mmrs_b200.dedup import sort_pairs
    return sort_pairs(pairs, n).cpu()


# ---- every shape, both tensor-core schedules, rank panels --------------------------------------------------
@pytest.mark.parametrize("pair", ["0", "1"], ids=["single_cta", "cta_pair"])
@pytest.mark.parametrize("d", [8, 72, 200, 512, 768])
@pytest.mark.parametrize("n", [1, 2, 127, 129, 255, 257, 2047, 2049, 4225, 16_385])
def test_tc_join_follows_the_reference_at_every_shape(mm, monkeypatch, n, d, pair):
    """method="tc" forced at every size: around the 128-row i-blocks, the 256-row j-blocks, the 2048-row
    switch of "auto", 33 i-blocks + 1 row and one row past 8 panels.  Rank panels for 2, 3 and 8 ranks (more
    ranks than panels below 6145 rows) must cover the single-rank result with no pair twice."""
    from mmrs_b200.dedup import _device_f32
    monkeypatch.setenv("MMRS_SJ_PAIR", pair)
    x, tau, planted, must, may = _data(n, d, seed=n + d)
    xd = _device_f32(torch.from_numpy(x))
    got = _sorted(_tc(xd, tau), n)
    _check_reference(got, must, may, n)
    assert torch.equal(got, mm.find_duplicate_pairs(x, tau, method="fp32"))
    if n >= 2049:
        assert len(planted["shrinking"]) == 48 and set(planted["shrinking"]) <= set(map(tuple, must.tolist()))
    for world in (2, 3, 8):
        parts = torch.cat([_tc(xd, tau, r, world) for r in range(world)])
        assert parts.shape[0] == got.shape[0]
        assert torch.equal(_sorted(parts, n), got)


# ---- the families, at unit and power-of-two scales ---------------------------------------------------------
@pytest.mark.parametrize("k", [-1, 0, 1, 2])
@pytest.mark.parametrize("d", [72, 512, 768])
def test_families_at_bf16_edges(mm, d, k):
    """Rows and tau scaled by 2^k and 4^k (the margin scales with the largest squared row norm).  Shrinking
    pairs the bf16 pass scores below tau - 0.0045 |a| |b| must survive the prefilter; growing pairs it
    scores at or above tau must be rejected by the recheck; at-threshold pairs must take the exact decision."""
    from mmrs_b200.dedup import _device_f32
    n = 4225
    x, tau, planted, must, may = _data(n, d, seed=d, k=k)
    s2 = 4.0 ** k
    shrink, grow, at = planted["shrinking"], planted["growing"], planted["at_threshold"]
    # the interesting cases are present (checked in float64 on the CPU)
    exact_s = _exact_dots(x, shrink)
    assert (exact_s >= tau).all()
    if k >= 0:    # (below unit norm the margin is not scaled down, and the old one sufficed)
        assert (_bf16_dots(x, shrink) < tau - OLD_MARGIN * s2).sum() >= 8
    assert ((_bf16_dots(x, grow) >= tau) & (_exact_dots(x, grow) < tau)).sum() >= 8
    gamma = d * 2.0 ** -24 / (1 - d * 2.0 ** -24)
    x64 = x.astype(np.float64)
    norms = np.sqrt(np.square(x64).sum(1))
    i, j = np.asarray(at).T
    assert (np.abs(_exact_dots(x, at) - tau) < gamma * norms[i] * norms[j]).sum() > 0   # the ambiguous band
    # the pair sets
    got = _sorted(_tc(_device_f32(torch.from_numpy(x)), tau), n)
    _check_reference(got, must, may, n)
    assert torch.equal(got, mm.find_duplicate_pairs(x, tau, method="fp32"))
    assert torch.equal(got, mm.find_duplicate_pairs(x, tau))                       # "auto": tensor cores here
    emitted = set(map(tuple, got.tolist()))
    assert set(shrink) <= emitted and not set(grow) & emitted


# ---- end to end -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ["identity", "random"])
def test_deduplicate_tc_equals_fp32_and_the_host_walk(mm, order):
    n, d = 4225, 512
    x, tau, planted, must, may = _data(n, d, seed=d, at_threshold=False)
    assert torch.equal(must, may)                   # no pair in the ambiguous band: one right answer
    assert len(must) >= len(planted["shrinking"]) == 48
    walk = list(range(n)) if order == "identity" else np.random.default_rng(1).permutation(n).tolist()
    o = None if order == "identity" else torch.tensor(walk, dtype=torch.int64)
    reps, dups = mm.greedy_first_keeper(n, must, walk)
    want = torch.arange(n)
    for v, r in dups:
        want[v] = r
    for method in ("tc", "fp32", "auto"):
        assert torch.equal(mm.deduplicate(x, tau, method=method, order=o), want), method


@pytest.mark.parametrize("n", [2047, 2048, 2049])
def test_auto_is_the_same_join_on_both_sides_of_2048_rows(mm, n):
    x, tau, planted, must, may = _data(n, 512, seed=3)
    got = mm.find_duplicate_pairs(x, tau)
    _check_reference(got, must, may, n)
    assert torch.equal(got, mm.find_duplicate_pairs(x, tau, method="fp32"))
    assert torch.equal(got, mm.find_duplicate_pairs(x, tau, method="tc"))


# ---- row ranges of the exact join ------------------------------------------------------------------------
def test_row_ranges_are_exact(mm):
    """selfjoin_raw(x, tau, lo, hi) returns exactly the pairs with lo <= i < hi, for bounds inside 128-row
    blocks too, and ranges that meet cover the join once."""
    from mmrs_b200.dedup import selfjoin_raw, _device_f32
    from mmrs_b200.sharded import triangle_bounds
    n, d = 1000, 72
    x, tau, planted, must, may = _data(n, d, seed=11)
    xd = _device_f32(torch.from_numpy(x))
    full = _sorted(selfjoin_raw(xd, tau), n)
    _check_reference(full, must, may, n)
    i0 = int(full[full[:, 0] % 128 > 0][0, 0])      # a row with pairs, inside a 128-row block
    for lo, hi in [(0, 100), (0, 1), (100, 257), (128, 300), (999, 1000), (0, 1000), (500, 500), (37, 38),
                   (i0 - i0 % 128, i0), (0, i0), (i0, i0 + 1), (i0, n)]:
        got = _sorted(selfjoin_raw(xd, tau, lo, hi), n)
        assert torch.equal(got, full[(full[:, 0] >= lo) & (full[:, 0] < hi)]), (lo, hi)
    for bounds in ([0, 100, 350, 777, 1000], [0, 1, 2, 999, 1000], [0, 129, 255, 1000],
                   [b for b, _ in triangle_bounds(n, 3)] + [n]):
        parts = torch.cat([selfjoin_raw(xd, tau, a, b) for a, b in zip(bounds[:-1], bounds[1:])])
        assert parts.shape[0] == full.shape[0] and torch.equal(_sorted(parts, n), full), bounds


# ---- non-finite rows ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", [float("nan"), float("inf"), float("-inf")], ids=["nan", "inf", "-inf"])
@pytest.mark.parametrize("n", [300, 2500])
def test_non_finite_rows_are_refused_by_every_method(mm, oracle, n, bad):
    x, _ = oracle.synthetic_dedup(n, 64, dup_frac=0.05, seed=n)
    x[n // 3, 5] = bad
    for method in ("auto", "fp32", "tc"):
        with pytest.raises(ValueError, match="non-finite"):
            mm.find_duplicate_pairs(x, 0.95, method=method)
        with pytest.raises(ValueError, match="non-finite"):
            mm.deduplicate(x, 0.95, method=method)
