"""The tensor-core self-join keeps a pair when its bf16 score reaches threshold - margin and then re-scores it in
fp32; the pair set equals the exact mode's only if the margin bounds how far bf16 rounding (and both fp32
accumulations) can move a dot product.  Rows whose entries all round the same way move it by nearly the
first-order bound 2^-7 |a| |b|; this checks the margin the join passes to the kernel against such rows, in
float64, without a GPU."""
import numpy as np
import pytest


def _gaps(x: np.ndarray):
    """|<a, b> - <bf16(a), bf16(b)>| over every pair of rows of `x` (diagonal included: a row and its exact
    copy), and the largest row norm, all in float64."""
    from oracle.oracle import to_bf16_f64
    x64 = x.astype(np.float64)
    b16 = to_bf16_f64(x)
    return np.abs(x64 @ x64.T - b16 @ b16.T), float(np.sqrt(np.square(x64).sum(1)).max())


@pytest.mark.parametrize("round_up", [False, True], ids=["shrinking", "growing"])
@pytest.mark.parametrize("k", [-1, 0, 1, 2])
@pytest.mark.parametrize("d", [8, 64, 512, 768, 1024, 4096])
def test_margin_bounds_the_rounding_of_aligned_rows(mm, oracle, d, k, round_up):
    from mmrs_b200.dedup import tc_margin
    rows, _ = oracle.bf16_edge_pairs(12, d, 0.90, 1.0, round_up, seed=d + 7 * k)
    x = rows * np.float32(2.0 ** k)                  # a power of two keeps every entry's rounding
    gap, max_norm = _gaps(x)
    first_order = 2.0 ** -7 * max_norm ** 2
    # the rows are adversarial: bf16 moves their dot products by most of the first-order bound, far more
    # than random rows do (~2^-8 / sqrt(d) |a| |b|) and more than the 0.0045 |a| |b| this join once assumed
    assert gap.max() > 0.85 * first_order
    # the margin covers the operand rounding plus both fp32 dot products rounded to nearest
    fp32_dots = 2 * d * 2.0 ** -24 / (1 - d * 2.0 ** -24) * max_norm ** 2
    device_norm = float(np.float32(max_norm))        # what mmrs_row_norm_range reports, to fp32 rounding
    assert tc_margin(d, device_norm) >= gap.max() + fp32_dots


def test_margin_scales_with_the_largest_squared_norm(mm):
    from mmrs_b200.dedup import BF16_MARGIN, tc_margin
    assert BF16_MARGIN == 2.0 ** -7 + 2.0 ** -16
    assert tc_margin(512, 1.0) == pytest.approx(2.0 ** -7 + 2.0 ** -16 + 512 * 2.0 ** -22, rel=2e-4)
    assert tc_margin(512, 0.25) == tc_margin(512, 0.0) == 2.0 ** -7 + 2.0 ** -16 + 512 * 2.0 ** -22   # never below unit
    assert tc_margin(512, 3.0) == pytest.approx(9.0 * tc_margin(512, 1.0), rel=1e-9)
