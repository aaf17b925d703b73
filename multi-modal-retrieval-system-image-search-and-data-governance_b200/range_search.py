"""Range search: every gallery row scoring at or above a per-query threshold.

The third step of the reference's workflow: score the gallery against a class prototype, tune a threshold
(`best_thresholds`), then accept every image at or above it -- `preds = similarity >= threshold`
(code/merge_dataset.py:259-284), `union_clip_by_threshold` with its frozen per-class thresholds
(code/union_clip_llava2.py:134, :153-162), and the A x B leakage join of tool/delete repeated.py (every
train image within tau of a test image).  `search_range` returns the passing rows in CSR form without
materialising the [Q, N] score matrix, in one pass over the gallery.

The rows go in windows of W rows (a multiple of 128, with Q * W * 8 bytes of candidate keys within
`max_candidate_bytes`).  Per window, `mmrs_range_search_window` runs the filter-mode scan of `search_topk`
over the window (every key with score >= t, capacity W per query, so no list can overflow), then sorts
each query's keys into row order with a bitmap counting sort and returns the per-query counts; the host
sizes the window's output and `mmrs_range_search_scatter` fills it.  The pieces of the windows (and, in
`ShardedGallery.search_range`, of the ranks) are joined per query by `concat_per_query`.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _cabi
from .gallery import DeviceGallery
from .row_filter import RowFilter
from .search import GalleryLike, _as_gallery, _filter_arg, _labels_arg, _operand, _prep_queries, _stream_handle

TILE_ROWS = 128
MAX_WINDOW_ROWS = 2 ** 31 - TILE_ROWS     # the scan's int32 list capacity
MAX_QUERIES = 65535                       # one CUDA grid row per query in the finalize kernels


def thresholds_f32(thresholds, n_queries: int) -> torch.Tensor:
    """Per-query thresholds as a host float32 tensor [n_queries] that the scan compares in float32 with the
    meaning numpy gives `scores >= thresholds`: float32 (and narrower float) thresholds compare as they are;
    float64 thresholds -- Python floats and integers included -- mean `float64(score) >= t`, which for a
    float32 score is `score >= t32` with t32 the smallest float32 >= t (above FLT_MAX: +inf).  A scalar
    applies to every query.  A NaN threshold raises ValueError."""
    t = thresholds if isinstance(thresholds, torch.Tensor) else torch.from_numpy(np.asarray(thresholds))
    t = t.detach().cpu()
    if t.dtype == torch.bool or t.dtype.is_complex:
        raise ValueError(f"thresholds must be real numbers, got {t.dtype}")
    if t.dim() == 0:
        t = t.reshape(1).expand(n_queries)
    elif t.dim() != 1 or t.numel() != n_queries:
        raise ValueError(f"thresholds must be a scalar or [{n_queries}], got {tuple(t.shape)}")
    if t.dtype in (torch.float32, torch.float16, torch.bfloat16):
        t32 = t.to(torch.float32)
    else:
        t64 = t.to(torch.float64)
        t32 = t64.to(torch.float32)
        below = t32.to(torch.float64) < t64                       # rounded down: the next float32 up
        t32 = torch.where(below, torch.nextafter(t32, torch.full_like(t32, float("inf"))), t32)
    if torch.isnan(t32).any():
        raise ValueError("a threshold is NaN")
    return t32.contiguous()


def window_rows(n_queries: int, n_rows: int, max_candidate_bytes: int) -> int:
    """Rows per window: the fewest windows whose keys (8 bytes per query and row) fit `max_candidate_bytes`,
    balanced, rounded up to whole 128-row tiles.  Windows are [r0, min(r0 + W, n_rows)) for r0 in
    range(0, n_rows, W): every row once, each window at least one row."""
    most = min(int(max_candidate_bytes) // (8 * max(1, int(n_queries))) // TILE_ROWS * TILE_ROWS, MAX_WINDOW_ROWS)
    if most < TILE_ROWS:
        raise ValueError(f"max_candidate_bytes = {max_candidate_bytes} holds less than one 128-row window of "
                         f"{n_queries} queries ({8 * TILE_ROWS * n_queries} bytes)")
    n = max(1, int(n_rows))
    n_windows = -(-n // most)
    per = -(-n // n_windows)
    return -(-per // TILE_ROWS) * TILE_ROWS


def concat_per_query(pieces):
    """Join CSR pieces `(offsets [Q+1] int64, values [M_i], indices [M_i])` (all on one device) query by
    query: query q's segment is its segment of piece 0, then of piece 1, ...  Row windows and row shards
    are ascending row blocks, so joining their pieces in order keeps every query's rows ascending."""
    if len(pieces) == 1:
        return pieces[0]
    offs = torch.stack([p[0] for p in pieces])                                    # [P, Q+1]
    counts = offs[:, 1:] - offs[:, :-1]                                           # [P, Q]
    out_off = torch.zeros_like(offs[0])
    torch.cumsum(counts.sum(0), 0, out=out_off[1:])
    before = torch.cumsum(counts, 0) - counts                                     # earlier pieces' matches of q
    m = int(out_off[-1].item())
    dev = offs.device
    values = torch.empty(m, dtype=pieces[0][1].dtype, device=dev)
    indices = torch.empty(m, dtype=pieces[0][2].dtype, device=dev)
    for k, (off, v, i) in enumerate(pieces):
        if v.numel() == 0:
            continue
        shift = out_off[:-1] + before[k] - off[:-1]
        dst = torch.repeat_interleave(shift, counts[k], output_size=v.numel()) + torch.arange(v.numel(), device=dev)
        values[dst] = v
        indices[dst] = i
    return out_off, values, indices


def empty_result(n_queries: int, device=None):
    return (torch.zeros(n_queries + 1, dtype=torch.int64, device=device),
            torch.empty(0, dtype=torch.float32, device=device), torch.empty(0, dtype=torch.int64, device=device))


def search_range(queries, gallery: GalleryLike, thresholds, *, normalize_queries: bool = True, scale: float = 1.0,
                 mode: Optional[str] = None, path: str = "auto", row_filter=None, row_labels=None, query_labels=None,
                 label_match: str = "same", max_candidate_bytes: int = 4 << 30):
    """Every gallery row r with `scale * q @ G[r] >= thresholds[q]`, for each query q, in one pass over the gallery.

    Returns CSR `(offsets [Q+1] int64, values [M] fp32, indices [M] int64)`: the matches of query q are
    `values[offsets[q]:offsets[q+1]]` / `indices[...]` in ascending row order, with global indices
    (`gallery.row_offset` added).  Host queries give host results, device queries device results.
    With S = `full_scores(queries, gallery, normalize_queries=, scale=, path=)` of the same batch, the result
    equals `mask = S >= t[:, None]` (ANDed with the filter and label predicates):
    `indices = mask.nonzero()[:, 1]`, `values = S[mask]`, `offsets = [0] + cumsum(mask.sum(1))`, bit for bit,
    except that a -0.0 score is returned as +0.0.  A NaN score never matches.

    `thresholds`: a scalar or [Q] (host or device).  As in numpy, float32 thresholds compare in float32
    and float64 thresholds (Python floats too) mean `float64(score) >= t` exactly, so the `best_threshold`
    of `best_thresholds` returns exactly the rows it counted as predicted positive.  NaN raises ValueError;
    -inf returns every allowed row, +inf only +inf scores.
    `row_filter`, `row_labels`, `query_labels`, `label_match`: as in `search_topk`; a filter allowing no row
    gives an empty result.  The rows go in windows of W rows with Q * W * 8 <= `max_candidate_bytes`
    (16 queries at 100 M rows: 3 windows); the gallery is still read once.  The call blocks: the size of
    the result is known only once the matches are counted."""
    gal = _as_gallery(gallery, mode)
    q, on_host = _prep_queries(queries, gal)
    nq = int(q.shape[0])
    thr = thresholds_f32(thresholds, nq)
    filt = _filter_arg(row_filter, gal)
    labels = _labels_arg(row_labels, query_labels, label_match, gal, nq)
    if nq > MAX_QUERIES:
        raise ValueError(f"at most {MAX_QUERIES} queries per call, got {nq}")
    dev = gal.device
    w = window_rows(nq, gal.n_rows, max_candidate_bytes)
    out_dev = None if on_host else dev
    if nq == 0:
        return empty_result(0, out_dev)
    lib = _cabi.lib
    with torch.cuda.device(dev):
        if filt is not None and not isinstance(filt, RowFilter):
            filt = RowFilter(filt, device=dev)
        if filt is not None and filt.n_allowed == 0:
            return empty_result(nq, out_dev)
        filt_ptr = filt.words.data_ptr() if filt is not None else 0
        lab_ptr, ql_ptr, match = 0, 0, 0
        if labels is not None:
            ql = labels[1].to(device=dev, dtype=torch.int32).contiguous()
            lab_ptr, ql_ptr, match = labels[0].labels.data_ptr(), ql.data_ptr(), labels[2]
        qd = q.to(dev)
        thr_d = thr.to(dev)
        g_ptr, g_ld, g_dtype = _operand(gal, nq, path)
        ws_bytes = int(lib.mmrs_range_search_workspace_bytes(w, gal.padded_dim, nq))
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        ws_ptr = DeviceGallery.aligned_ptr(ws)
        stream = _stream_handle(dev)
        counts = np.empty(nq, dtype=np.int64)
        pieces = []
        for r0 in range(0, gal.n_rows, w):
            _cabi.check(lib.mmrs_range_search_window(
                g_ptr, gal.n_rows, gal.padded_dim, g_ld, g_dtype, qd.data_ptr(), nq, qd.stride(0),
                int(bool(normalize_queries)), float(scale), _cabi.PATHS[path], thr_d.data_ptr(), r0, w, filt_ptr,
                lab_ptr, ql_ptr, match, counts.ctypes.data, ws_ptr, ws_bytes, stream))
            off = np.zeros(nq + 1, dtype=np.int64)
            np.cumsum(counts, out=off[1:])
            off_d = torch.from_numpy(off).to(dev)
            values = torch.empty(int(off[-1]), dtype=torch.float32, device=dev)
            indices = torch.empty(int(off[-1]), dtype=torch.int64, device=dev)
            if values.numel():
                _cabi.check(lib.mmrs_range_search_scatter(nq, w, gal.padded_dim, off_d.data_ptr(), gal.row_offset + r0,
                                                          values.data_ptr(), indices.data_ptr(), ws_ptr, ws_bytes,
                                                          stream))
            pieces.append((off_d, values, indices))
        out = concat_per_query(pieces)
    return tuple(x.cpu() for x in out) if on_host else out
