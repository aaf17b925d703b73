"""Per-class threshold tuning of a batch of class prototypes (code/search_image.py:382-389).

The reference's main workflow loops over the classes: build the prototype `q_c`, score every gallery row
(`get_similarity`, :105-117, `100. * G @ q_c.t()`), split the scores by `targets == c` and sweep a 200-point
`np.linspace(min, max)` grid for the best F1 (`find_thresholds`, :58-79).  `best_thresholds` does that for
every prototype of a batch: one gallery pass per chunk of queries, nothing of size N crossing to the host.

Per chunk of `Qc = max(1, max_score_bytes // (4 N))` queries:
  1. `mmrs_full_scores` of the chunk into one [Qc, N] fp32 buffer reused across chunks (the kernels and
     arithmetic of `full_scores`, so each score is the one `full_scores` gives);
  2. `mmrs_score_range_batched`: each query's order-preserving (min, max) over the allowed rows;
  3. `mmrs_threshold_sweep_batched`: each query's linspace grid from its range, histograms of its positives
     (row label == the query's label) and negatives, suffix counts [Qc, T, 2] and its positives n_pos;
  4. on the host, the F1 curve and the first strict maximum (`search.best_from_counts`, shared with
     `best_threshold_on_device`).
A sharded gallery runs the same steps on every rank's shard with two collectives per chunk: MIN / MAX of
the ranges before the sweep, SUM of the counts after it (`ShardedGallery.best_thresholds`).
"""
from __future__ import annotations

from typing import Callable, Optional

import numpy as np
import torch

from . import _cabi
from .gallery import DeviceGallery
from .row_filter import RowFilter
from .row_labels import RowLabels, query_labels_arg
from .search import (GalleryLike, _as_gallery, _filter_arg, _prep_queries, _scores_into, _stream_handle,
                     best_from_counts, grid_f32)

MAX_POINTS = 4096                  # kSweepMaxT of csrc/selfjoin.cu: one query's grid and histograms in shared memory


def chunk_queries(n_rows: int, max_score_bytes: int) -> int:
    """Queries per chunk: as many fp32 score rows of `n_rows` as fit `max_score_bytes`, at least one."""
    return max(1, int(max_score_bytes) // (4 * max(1, int(n_rows))))


def check_arguments(n_queries: int, query_labels, n_points: int, device) -> torch.Tensor:
    """`query_labels` as an integer tensor [n_queries] with every value >= 0; `n_points` in [1, MAX_POINTS]."""
    n_points = int(n_points)
    if not 1 <= n_points <= MAX_POINTS:
        raise ValueError(f"n_points must be in [1, {MAX_POINTS}], got {n_points}")
    ql = query_labels_arg(query_labels, n_queries, device)
    if ql.numel() and int(ql.min().item()) < 0:
        raise ValueError("query labels must be >= 0 (a class id of the gallery's RowLabels)")
    return ql


def check_row_labels(row_labels, n_rows: int, device) -> None:
    if not isinstance(row_labels, RowLabels):
        raise ValueError(f"row_labels must be a RowLabels, got {type(row_labels).__name__}")
    if row_labels.n_rows != n_rows:
        raise ValueError(f"row_labels covers {row_labels.n_rows} rows, the gallery has {n_rows}")
    if device is not None and row_labels.device != device:
        raise ValueError(f"row_labels is on {row_labels.device}, the gallery on {device}")


def run_chunks(queries: torch.Tensor, query_labels: torch.Tensor, qc: int, n_points: int,
               range_step: Callable, count_step: Callable,
               reduce_range: Optional[Callable] = None, reduce_counts: Optional[Callable] = None):
    """Drive the chunks: range_step(q) -> int64 [nq, 2] keys; reduce_range (ranks: MIN / MAX); count_step(q,
    labels, range) -> (thresholds [nq, T] fp64, counts [nq, T, 2] int64, n_pos [nq] int64); reduce_counts
    (ranks: SUM); the F1 tail on the host.  -> the six arrays of `best_thresholds`."""
    c = int(queries.shape[0])
    best = np.zeros((4, c), dtype=np.float64)
    thresholds = np.zeros((c, n_points), dtype=np.float64)
    f1_scores = np.zeros((c, n_points), dtype=np.float64)
    for lo in range(0, c, qc):
        q, lab = queries[lo:lo + qc], query_labels[lo:lo + qc]
        rng = range_step(q)
        if reduce_range is not None:
            rng = reduce_range(rng)
        thr, counts, n_pos = count_step(q, lab, rng)
        if reduce_counts is not None:
            counts, n_pos = reduce_counts(counts, n_pos)
        thr, counts, n_pos = thr.cpu().numpy(), counts.cpu().numpy(), n_pos.cpu().numpy()
        for j in range(thr.shape[0]):
            b_f1, b_thr, b_p, b_r, f1s = best_from_counts(thr[j], counts[j], int(n_pos[j]))
            best[:, lo + j] = (b_f1, b_thr, b_p, b_r)
            thresholds[lo + j] = thr[j]
            f1_scores[lo + j] = f1s
    return best[0], best[1], best[2], best[3], thresholds, f1_scores


def _bits32(rng: torch.Tensor) -> torch.Tensor:
    """int64 keys in [0, 2^32) -> int32 tensor with the same bits (the kernels' uint32)."""
    return torch.where(rng >= 2 ** 31, rng - 2 ** 32, rng).to(torch.int32).contiguous()


class DeviceSweep:
    """The device steps of `best_thresholds` over one gallery (or one shard): `range(q)` scores a chunk into
    the [qc, N] buffer and returns its (min, max) keys, `counts(labels, range)` sweeps those same scores.
    The buffer and the sweep's workspace live as long as this object, across chunks."""

    def __init__(self, gal: DeviceGallery, qc: int, n_points: int, normalize_queries: bool, scale: float, path: str,
                 row_labels: RowLabels, row_filter: Optional[RowFilter], grid_f32: int):
        self.gal, self.n_points, self.grid_f32 = gal, int(n_points), int(grid_f32)
        self.normalize_queries, self.scale, self.path = bool(normalize_queries), float(scale), path
        self.labels_ptr = row_labels.labels.data_ptr()
        self.filt_ptr = row_filter.words.data_ptr() if row_filter is not None else 0
        dev = gal.device
        self.scores = torch.empty((qc, gal.n_rows), dtype=torch.float32, device=dev)
        self.ws_bytes = int(_cabi.lib.mmrs_threshold_sweep_batched_workspace_bytes(qc, self.n_points))
        self.ws = torch.empty(self.ws_bytes + 256, dtype=torch.uint8, device=dev)

    def range(self, queries: torch.Tensor) -> torch.Tensor:
        gal = self.gal
        q, _ = _prep_queries(queries, gal)
        nq = int(q.shape[0])
        with torch.cuda.device(gal.device):
            _scores_into(gal, q.to(gal.device), self.scores, self.normalize_queries, self.scale, self.path)
        return self.range_keys(nq)

    def range_keys(self, nq: int) -> torch.Tensor:
        """int64 [nq, 2] (min, max) keys of the first nq rows of the scores buffer, over the allowed rows."""
        gal = self.gal
        with torch.cuda.device(gal.device):
            # (0xffffffff, 0): the neutral element of MIN / MAX, kept by a query that sees no allowed row
            rng = torch.tensor([[-1, 0]], dtype=torch.int32, device=gal.device).repeat(nq, 1)
            _cabi.check(_cabi.lib.mmrs_score_range_batched(self.scores.data_ptr(), self.scores.stride(0), nq, gal.n_rows,
                                                           self.filt_ptr, rng.data_ptr(), _stream_handle(gal.device)))
        return rng.to(torch.int64) & 0xffffffff

    def counts(self, query_labels: torch.Tensor, rng: torch.Tensor):
        gal, t = self.gal, self.n_points
        nq = int(rng.shape[0])
        dev = gal.device
        with torch.cuda.device(dev):
            rng32 = _bits32(rng.to(dev))
            ql = query_labels.to(device=dev, dtype=torch.int32).contiguous()
            thr = torch.empty((nq, t), dtype=torch.float64, device=dev)
            counts = torch.empty((nq, t, 2), dtype=torch.int64, device=dev)
            n_pos = torch.empty(nq, dtype=torch.int64, device=dev)
            _cabi.check(_cabi.lib.mmrs_threshold_sweep_batched(
                self.scores.data_ptr(), self.scores.stride(0), nq, gal.n_rows, self.labels_ptr, ql.data_ptr(),
                self.filt_ptr, rng32.data_ptr(), t, self.grid_f32, thr.data_ptr(), counts.data_ptr(), n_pos.data_ptr(),
                DeviceGallery.aligned_ptr(self.ws), self.ws_bytes, _stream_handle(dev)))
        return thr, counts, n_pos


def empty_result(n_points: int):
    z = np.zeros(0, dtype=np.float64)
    return z, z.copy(), z.copy(), z.copy(), np.zeros((0, n_points)), np.zeros((0, n_points))


def best_thresholds(queries, gallery: GalleryLike, row_labels, query_labels, *, n_points: int = 200, scale: float = 100.0,
                    normalize_queries: bool = False, row_filter=None, mode: Optional[str] = None, path: str = "auto",
                    max_score_bytes: int = 4 << 30):
    """The best-F1 threshold of every class prototype over a labelled gallery: the reference's per-class loop
    `find_thresholds(*get_similarity(features, targets, c, q_c), c)` (code/search_image.py:382-389) for a
    whole batch, with the scores kept on the device.

    queries [C, D] (host or device) are the prototypes, `query_labels` [C] (integer, host or device, every
    value >= 0) their classes, `row_labels` the RowLabels of the gallery (the reference's `targets`).  Row q
    is scored as `full_scores` scores it (`scale * q @ G.T`, by default get_similarity's `100. * G @ q.t()`
    without normalising q); the rows of class `query_labels[q]` are its positives, every other row its
    negatives; `row_filter` (a RowFilter or a bool mask [N]) leaves rows out of both.  Returns host float64
    arrays `(best_f1 [C], best_threshold [C], best_precision [C], best_recall [C], thresholds [C, n_points],
    f1_scores [C, n_points])`; row q equals `best_threshold_on_device(S[q], targets, c, n_points)` bit for bit,
    where S is `full_scores` of the chunk holding q over the allowed rows.  A class without rows has an all-NaN
    curve and best tuple (0, 0, 0, 0), as there.

    The queries go in chunks of `max(1, max_score_bytes // (4 N))` (one [chunk, N] fp32 score buffer, one
    gallery pass each; 10 queries at N = 100 M with the default 4 GB).  With `path="auto"` each chunk's kernel
    is chosen for its own size, as `full_scores` chooses it (bf16: K1 up to 2 queries, K2 above; fp32: K1 up
    to 8, the bf16x3 tensor-core path from 9), so a short last chunk may be scored by another kernel than the
    others; pin `path="gemv"` or `"mma"` for results that do not depend on the chunking."""
    gal = _as_gallery(gallery, mode)
    if isinstance(queries, np.ndarray):
        queries = torch.from_numpy(queries)
    if queries.dim() == 1:
        queries = queries.unsqueeze(0)
    c = int(queries.shape[0])
    check_row_labels(row_labels, gal.n_rows, gal.device)
    ql = check_arguments(c, query_labels, n_points, gal.device)
    filt = _filter_arg(row_filter, gal)
    if filt is not None and not isinstance(filt, RowFilter):
        filt = RowFilter(filt, device=gal.device)
    if filt is not None and filt.n_allowed == 0:
        raise ValueError("row_filter allows no row")
    _prep_queries(queries[:0], gal)                  # the width, before any device work
    if c == 0:
        return empty_result(int(n_points))
    qc = min(c, chunk_queries(gal.n_rows, max_score_bytes))
    sweep = DeviceSweep(gal, qc, n_points, normalize_queries, scale, path, row_labels, filt, grid_f32())
    return run_chunks(queries, ql, qc, int(n_points), sweep.range, lambda q, lab, rng: sweep.counts(lab, rng))
