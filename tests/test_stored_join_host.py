"""The bf16 stored-format self-join re-scores its survivors from the stored rows, so its prefilter margin only has to
cover the two fp32 accumulations (tc_margin with unit_margin=0).  This checks that margin against the fp32 fmaf
chain of worst-case bf16 rows -- every product of one sign, so no rounding error cancels -- in float64, and that
`method` is validated before anything reaches a device.  No GPU needed."""
import numpy as np
import pytest
import torch


def _fmaf_chain(a, b):
    """The exact join's serial fmaf chain, k ascending, for bf16-valued rows (products and sums exact in float64)."""
    acc = np.zeros(a.shape[0], np.float32)
    for k in range(a.shape[1]):
        acc = (a[:, k].astype(np.float64) * b[:, k] + acc).astype(np.float32)
    return acc


@pytest.mark.parametrize("k", [0, 3])
@pytest.mark.parametrize("d", [8, 64, 512, 768, 4096])
def test_zero_rounding_margin_bounds_the_accumulation(mm, d, k):
    from mmrs_b200.dedup import tc_margin
    rng = np.random.default_rng(d + k)
    # positive rows whose entries span eight binades: the partial sums need more than fp32's 24 bits, so the chain
    # rounds, and with every product of one sign no rounding error cancels another
    x = np.abs(rng.standard_normal((64, d))) * 2.0 ** rng.integers(-8, 1, size=(64, d))
    x = torch.from_numpy(x / np.linalg.norm(x, axis=1, keepdims=True)).to(torch.bfloat16).float().numpy()
    x = x * np.float32(2.0 ** k)
    i, j = np.triu_indices(x.shape[0], 1)
    x64 = x.astype(np.float64)
    exact = (x64[i] * x64[j]).sum(1)
    chain = _fmaf_chain(x[i], x[j]).astype(np.float64)
    norms = np.sqrt(np.square(x64).sum(1))
    ab = norms[i] * norms[j]
    gamma = d * 2.0 ** -24 / (1 - d * 2.0 ** -24)
    err = np.abs(chain - exact)
    assert (err <= gamma * ab).all()                  # the bound the margin is built from
    if d >= 64:
        assert err.max() > 0                          # and the rows do exercise it
    device_norm = float(np.float32(norms.max()))
    margin = tc_margin(d, device_norm, unit_margin=0.0)
    # the recheck's chain and the tensor cores' sum (same bound, order undocumented) may each be off by gamma |a||b|
    assert margin >= (err + gamma * ab).max()
    assert margin == pytest.approx(d * 2.0 ** -22 * max(1.0, device_norm ** 2 * 1.0001), rel=1e-12)
    assert margin < tc_margin(d, device_norm) / 40 if d <= 768 else True


def test_method_is_checked_before_any_device_work(mm):
    x = torch.randn(16, 8)
    for fn in (mm.find_duplicate_pairs, mm.deduplicate):
        with pytest.raises(ValueError, match="method must be"):
            fn(x, 0.9, method="int8")
        with pytest.raises(ValueError, match="stored"):
            fn(x, 0.9, method="stored")               # a plain tensor has no stored format
        with pytest.raises(ValueError, match="stored"):
            fn(x.numpy(), 0.9, method="stored")
