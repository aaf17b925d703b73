"""Host-side argument checks of resolve_duplicates / deduplicate: they raise before any device work, so they
hold without a GPU."""
import numpy as np
import pytest
import torch


@pytest.mark.parametrize("n", [-1, 2 ** 31, 2 ** 40, 3.0, True, "10"])
def test_row_count_is_checked(mm, n):
    with pytest.raises(ValueError, match="n"):
        mm.resolve_duplicates(torch.zeros((0, 2), dtype=torch.int64), n)


@pytest.mark.parametrize("pairs", [torch.zeros((3, 2), dtype=torch.int32), torch.zeros((3, 2), dtype=torch.float64),
                                   torch.zeros((3, 3), dtype=torch.int64), torch.zeros(6, dtype=torch.int64),
                                   [[0, 1]]])
def test_pairs_must_be_int64_p_by_2(mm, pairs):
    with pytest.raises(ValueError, match="pairs"):
        mm.resolve_duplicates(pairs, 10)


@pytest.mark.parametrize("order", [torch.arange(4, dtype=torch.int32), np.arange(4, dtype=np.float32),
                                   torch.zeros((2, 2), dtype=torch.int64)])
def test_order_must_be_int64_ids(mm, order):
    with pytest.raises(ValueError, match="order"):
        mm.resolve_duplicates(torch.zeros((0, 2), dtype=torch.int64), 10, order=order)


def test_deduplicate_checks_method_first(mm):
    with pytest.raises(ValueError, match="method"):
        mm.deduplicate(torch.randn(16, 8), 0.9, method="fp16")


def test_workspace_query_is_host_arithmetic(mm):
    lib = mm._cabi.lib
    small = lib.mmrs_resolve_duplicates_workspace_bytes(1000, 1000, 100)
    assert small >= 1000 * 4 + 100 * 16 + 1001 * 8 + 1000 * (8 + 4 + 4 + 4)
    assert lib.mmrs_resolve_duplicates_workspace_bytes(10_000_000, 10_000_000, 100_000) > 10_000_000 * 24
    assert lib.mmrs_resolve_duplicates_workspace_bytes(-1, 0, 0) == 0


def test_valid_input_needs_the_gpu(mm):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU path"):
        mm.resolve_duplicates(torch.tensor([[0, 1]]), 2, order=[1, 0])
    with pytest.raises(RuntimeError, match="no CPU path"):
        mm.deduplicate(torch.randn(16, 8), 0.9)
