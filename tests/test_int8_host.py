"""The numpy mirror of int8 mode (include/mmrs_b200.h, "int8 galleries"), checked on hand-built rows.

The GPU tests (test_int8_gpu.py, tools/multigpu_int8_check.py) use these functions as their oracle: row
quantisation `s = fl(m / 127)`, `c = clamp(rint(x / s), -127, 127)` and the score
`fl(fl(float(dot) * a_q) * s_r)` with `a_q = fl(s_q * scale)` and the exact integer dot."""
import numpy as np
import pytest


def quantize_rows(x):
    """(codes int8 [N, D], scales float32 [N]) of float32 rows: IEEE float32 division, half to even."""
    x = np.asarray(x, dtype=np.float32)
    if not np.isfinite(x).all():
        raise ValueError("a row holds a NaN or an infinity")
    s = (np.abs(x).max(axis=1, initial=np.float32(0)) / np.float32(127)).astype(np.float32)
    safe = np.where(s > 0, s, np.float32(1)).astype(np.float32)
    c = np.clip(np.rint(x / safe[:, None]), -127, 127)
    c[s == 0] = 0
    return c.astype(np.int8), s


def scores(q_codes, q_scales, g_codes, g_scales, scale=1.0):
    """[Q, N] float32 scores of int8 mode: the exact dot (float64 products of int8 codes are exact below 2^53),
    converted to float32 once, times a_q, times s_r, -0.0 as +0.0."""
    dot = np.asarray(q_codes, np.float64) @ np.asarray(g_codes, np.float64).T
    a_q = (np.asarray(q_scales, np.float32) * np.float32(scale)).astype(np.float32)
    s = (dot.astype(np.int64).astype(np.float32) * a_q[:, None]).astype(np.float32)
    s = (s * np.asarray(g_scales, np.float32)[None, :]).astype(np.float32)
    return s + np.float32(0)


def topk(s, k):
    """Stable descending sort of each row: values desc, equal values by ascending index (torch.topk's order here)."""
    idx = np.argsort(-s, axis=1, kind="stable")[:, :k]
    return np.take_along_axis(s, idx, axis=1), idx


def test_half_to_even_and_clamp():
    # m = 127 -> s = 1: codes are rint of the values themselves, ties to even
    row = np.array([[127.0, 0.5, 1.5, 2.5, -0.5, -1.5, -2.5, 126.5, -127.0]], np.float32)
    c, s = quantize_rows(row)
    assert s[0] == np.float32(1)
    assert c.tolist() == [[127, 0, 2, 2, 0, -2, -2, 126, -127]]


def test_scale_is_float32_division():
    row = np.array([[0.3, -0.1, 0.0]], np.float32)
    c, s = quantize_rows(row)
    assert s[0] == np.float32(np.float32(0.3) / np.float32(127))
    assert c[0, 0] == 127 and c[0, 2] == 0
    assert c[0, 1] == np.rint(np.float32(-0.1) / s[0])


def test_zero_row_and_non_finite():
    c, s = quantize_rows(np.zeros((2, 5), np.float32))
    assert (c == 0).all() and (s == 0).all()
    for bad in (np.nan, np.inf, -np.inf):
        row = np.ones((1, 4), np.float32)
        row[0, 2] = bad
        with pytest.raises(ValueError):
            quantize_rows(row)


def test_scores_formula_and_negative_zero():
    gc = np.array([[1, -2, 0], [0, 0, 0], [127, 127, 127]], np.int8)
    gs = np.array([0.5, 0.25, 2.0], np.float32)
    qc = np.array([[3, 1, -1]], np.int8)
    qs = np.array([0.1], np.float32)
    got = scores(qc, qs, gc, gs, scale=-2.0)
    a_q = np.float32(np.float32(0.1) * np.float32(-2.0))
    assert got[0, 0] == np.float32(np.float32(np.float32(1) * a_q) * np.float32(0.5))
    assert got[0, 1] == 0 and not np.signbit(got[0, 1])          # 0 * negative a_q is -0.0 before canonicalising
    assert got[0, 2] == np.float32(np.float32(np.float32(127 * 3) * a_q) * np.float32(2.0))


def test_topk_ties_by_index():
    s = np.array([[1.0, 3.0, 3.0, 2.0, 3.0]], np.float32)
    v, i = topk(s, 4)
    assert i.tolist() == [[1, 2, 4, 3]] and v.tolist() == [[3.0, 3.0, 3.0, 2.0]]
