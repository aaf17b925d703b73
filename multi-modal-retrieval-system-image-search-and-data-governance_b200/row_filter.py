"""Row filters: per-call allow-lists over the rows of a resident gallery.

A `RowFilter` is the device bitmap the scan kernels read (csrc/common.cuh, ScanParams::row_filter):
uint32 words, bit `r & 31` of word `r >> 5` set when row `r` may be returned, zero-padded to whole
128-row tiles (4 words per tile) so that a kernel reads the word of any row of a visited tile
without a bounds check.  100 M rows take 12.5 MB -- against 153.6 GB to re-upload a 100 M x 768 bf16
gallery without the rows dedup removed or a split / class leaves out.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _cabi

TILE_ROWS = 128
WORDS_PER_TILE = TILE_ROWS // 32

# popcount of every byte value: counts of bitmap ranges without unpacking them
_POPCOUNT8 = torch.tensor([bin(b).count("1") for b in range(256)], dtype=torch.int64)


def filter_words(n_rows: int) -> int:
    """Words of the bitmap of an `n_rows`-row gallery (whole 128-row tiles)."""
    return (int(n_rows) + TILE_ROWS - 1) // TILE_ROWS * WORDS_PER_TILE


def count_allowed(words: torch.Tensor, lo: int, hi: int) -> int:
    """Allowed rows in [lo, hi) of a bitmap (any device); lo must be a multiple of 32."""
    if hi <= lo:
        return 0
    if lo % 32:
        raise ValueError("lo must be a multiple of 32")
    w = words[lo // 32:(hi + 31) // 32]
    if hi % 32:
        w = w.clone()
        w[-1] = w[-1] & ((1 << (hi % 32)) - 1)
    lut = _POPCOUNT8.to(w.device)
    return int(lut[w.contiguous().view(torch.uint8).long()].sum().item())


class RowFilter:
    """Immutable allow-list over the rows of one gallery: `RowFilter(mask)` with a bool mask [N]
    (torch or numpy, host or device) packs it on the gallery's GPU once.  Attributes: `words`
    (device int32 [4 * ceil(N / 128)], the bitmap), `n_rows` (N), `n_allowed` (rows set).
    Pass it as `search_topk(..., row_filter=f)`; a filter reused across calls costs nothing per call
    (a bool mask passed directly is packed again every call)."""

    def __init__(self, mask, device: Optional[torch.device] = None):
        m = torch.from_numpy(np.asarray(mask)) if not isinstance(mask, torch.Tensor) else mask
        if m.dim() != 1 or m.dtype != torch.bool:
            raise ValueError(f"a row filter is built from a 1-D bool mask, got {m.dtype} {tuple(m.shape)}")
        if m.numel() < 1:
            raise ValueError("a row filter needs at least one row")
        if device is None:
            device = m.device if m.is_cuda else torch.device("cuda", torch.cuda.current_device()
                                                            if torch.cuda.is_available() else 0)
        device = torch.device(device)
        _cabi.require_b200(device.index if device.index is not None else 0)
        self.n_rows = int(m.numel())
        self.words = torch.empty(filter_words(self.n_rows), dtype=torch.int32, device=device)
        count = pack_mask(m, self.words)
        self.n_allowed = int(count.item())
        self._shards: dict = {}

    @classmethod
    def _wrap(cls, words: torch.Tensor, n_rows: int, n_allowed: int) -> "RowFilter":
        f = cls.__new__(cls)
        f.words, f.n_rows, f.n_allowed, f._shards = words, int(n_rows), int(n_allowed), {}
        return f

    @property
    def device(self) -> torch.device:
        return self.words.device

    def shard(self, lo: int, hi: int) -> "RowFilter":
        """The filter of rows [lo, hi) as a filter over a shard's local rows (lo a multiple of 128, as
        `shard_bounds` makes them): a view of the same words starting at word lo / 32 -- the tail bits
        past hi belong to the next shard and are ignored by the kernels.  Cached per range."""
        if (lo % TILE_ROWS and lo != self.n_rows) or not 0 <= lo <= hi <= self.n_rows:
            raise ValueError(f"shard [{lo}, {hi}) must start on a {TILE_ROWS}-row tile inside the {self.n_rows} rows")
        hit = self._shards.get((lo, hi))
        if hit is None:
            hit = self._shards[(lo, hi)] = RowFilter._wrap(self.words[lo // 32:], hi - lo,
                                                           count_allowed(self.words, lo, hi))
        return hit

    def __len__(self) -> int:
        return self.n_rows

    def __repr__(self) -> str:
        return f"RowFilter(rows={self.n_rows}, allowed={self.n_allowed}, device={self.device})"


def pack_mask(mask: torch.Tensor, words: torch.Tensor) -> torch.Tensor:
    """Pack a bool mask into `words` (device int32, >= filter_words(len(mask))) with the library's
    ballot kernel on the current stream; returns the device int64 [1] count of allowed rows."""
    dev = words.device
    with torch.cuda.device(dev):
        m = mask.to(dev, non_blocking=True).contiguous()
        count = torch.empty(1, dtype=torch.int64, device=dev)
        _cabi.check(_cabi.lib.mmrs_pack_row_filter(m.data_ptr(), m.numel(), words.data_ptr(), words.numel(),
                                                   count.data_ptr(), int(torch.cuda.current_stream(dev).cuda_stream)))
    return count
