"""Row labels: one class id per gallery row, for label-conditioned search.

A `RowLabels` is the device array the scan kernels read (csrc/common.cuh, ScanParams::row_labels):
int32 [128 * ceil(N / 128)], the label of row `r` at element `r`, padded to whole 128-row tiles -- the
padding contract of the row-filter bitmap -- so that a kernel reads the label of any row of a visited
tile without a bounds check (padding values are never compared: rows past N fail the kernels' row
test first).  100 M rows take 400 MB.

`search_topk(q, gal, k, row_labels=L, query_labels=ql, label_match="same")` restricts query q to the
rows with `L[r] == ql[q]` ("other": `L[r] != ql[q]`, the hard negatives); `ql[q] < 0` leaves that query
unrestricted.  A query with fewer than k eligible rows is padded with value -inf, index -1 (a
`RowFilter` with fewer than k allowed rows raises instead: a small class is a normal condition, and
counting every query's eligible rows would cost a host sync per call).
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _cabi

TILE_ROWS = 128
MAX_LABEL = 2 ** 31 - 2          # labels are in [0, 2^31 - 1)


def label_elements(n_rows: int) -> int:
    """Elements of the label array of an `n_rows`-row gallery (whole 128-row tiles)."""
    return (int(n_rows) + TILE_ROWS - 1) // TILE_ROWS * TILE_ROWS


class RowLabels:
    """Immutable class ids of the rows of one gallery: `RowLabels(labels)` with an integer array [N]
    (torch or numpy, host or device), every value in [0, 2^31 - 1), copied to the gallery's GPU once.
    Attributes: `labels` (device int32 [128 * ceil(N / 128)]), `n_rows` (N).  Pass it as
    `search_topk(..., row_labels=L, query_labels=ql)`; reusing it across calls costs nothing per call."""

    def __init__(self, labels, device: Optional[torch.device] = None):
        t = labels if isinstance(labels, torch.Tensor) else torch.from_numpy(np.asarray(labels))
        if t.dim() != 1 or t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError(f"row labels are a 1-D integer array, got {t.dtype} {tuple(t.shape)}")
        if t.numel() < 1:
            raise ValueError("row labels need at least one row")
        lo, hi = int(t.min().item()), int(t.max().item())
        if lo < 0 or hi > MAX_LABEL:
            raise ValueError(f"row labels must be in [0, 2^31 - 1), got values in [{lo}, {hi}]")
        if device is None:
            device = t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device()
                                                            if torch.cuda.is_available() else 0)
        device = torch.device(device)
        if device.type == "cuda":
            _cabi.require_b200(device.index if device.index is not None else 0)
        self.n_rows = int(t.numel())
        self.labels = torch.zeros(label_elements(self.n_rows), dtype=torch.int32, device=device)
        self.labels[:self.n_rows].copy_(t.to(torch.int32))
        self._shards: dict = {}

    @classmethod
    def _wrap(cls, labels: torch.Tensor, n_rows: int) -> "RowLabels":
        r = cls.__new__(cls)
        r.labels, r.n_rows, r._shards = labels, int(n_rows), {}
        return r

    @property
    def device(self) -> torch.device:
        return self.labels.device

    def shard(self, lo: int, hi: int) -> "RowLabels":
        """The labels of rows [lo, hi) as labels over a shard's local rows (lo a multiple of 128, as
        `shard_bounds` makes them): a view of the same tensor at element lo, which still covers the
        shard's own whole tiles.  Cached per range."""
        if (lo % TILE_ROWS and lo != self.n_rows) or not 0 <= lo <= hi <= self.n_rows:
            raise ValueError(f"shard [{lo}, {hi}) must start on a {TILE_ROWS}-row tile inside the {self.n_rows} rows")
        hit = self._shards.get((lo, hi))
        if hit is None:
            hit = self._shards[(lo, hi)] = RowLabels._wrap(self.labels[lo:], hi - lo)
        return hit

    def __len__(self) -> int:
        return self.n_rows

    def __repr__(self) -> str:
        return f"RowLabels(rows={self.n_rows}, device={self.device})"


def query_labels_arg(query_labels, n_queries: int, device: Optional[torch.device]) -> torch.Tensor:
    """`query_labels` checked: an integer tensor / array [n_queries] on the host or on `device`
    (None: any).  Returned as given (converted to a tensor); values < 0 mean "no restriction"."""
    t = query_labels if isinstance(query_labels, torch.Tensor) else torch.from_numpy(np.asarray(query_labels))
    if t.dim() != 1 or t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
        raise ValueError(f"query_labels must be a 1-D integer tensor, got {t.dtype} {tuple(t.shape)}")
    if t.numel() != n_queries:
        raise ValueError(f"query_labels has {t.numel()} entries for {n_queries} queries")
    if t.is_cuda and device is not None and t.device != device:
        raise ValueError(f"query_labels is on {t.device}, the gallery on {device}")
    if t.dtype != torch.int32 and t.numel():
        lo, hi = int(t.min().item()), int(t.max().item())
        if lo < -2 ** 31 or hi > MAX_LABEL:
            raise ValueError(f"query labels must fit int32 and be < 2^31 - 1, got values in [{lo}, {hi}]")
    return t


LABEL_MATCHES = ("same", "other")


def label_match_arg(label_match) -> int:
    if label_match not in LABEL_MATCHES:
        raise ValueError(f"label_match must be 'same' or 'other', got {label_match!r}")
    return _cabi.LABEL_MATCH[label_match]
