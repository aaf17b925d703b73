"""Search hot path: the reference's scoring functions on top of the CUDA library.

Mirrors (same names, positional order, return tuples) of code/search_image.py:
    get_similarity   :105-117     construct_dataset :167-182
    eval_threshold   :39-56       find_thresholds   :58-103
and the tensor-level calls they sit on (`search_topk` returns like
`output.topk(k, 1, True, True)`, code/utils.py:17).
"""
from __future__ import annotations

import os
from typing import Optional, Union

import numpy as np
import torch

from . import _cabi
from .gallery import DeviceGallery, _pad_dim
from .row_filter import RowFilter, filter_words, pack_mask
from .row_labels import RowLabels, label_match_arg, query_labels_arg

# module-level configuration with the reference's names (code/search_image.py:14-38); scripts
# that `from search_image import *` and set these keep working
class_names = ["T-shirt", "badminton-racket", "baozi", "guitar", "lychee", "cherry", "tennis-racket",
               "violin", "mantou", "dress-shirt"]
class_to_idx = {name: i for i, name in enumerate(class_names)}
dataset_path = "data/search"

GalleryLike = Union[DeviceGallery, torch.Tensor, np.ndarray]


def _as_gallery(gallery: GalleryLike, mode: Optional[str]) -> DeviceGallery:
    if isinstance(gallery, DeviceGallery):
        if mode is not None and mode != gallery.mode:
            raise ValueError(f"gallery is resident in {gallery.mode} mode, asked for {mode}")
        return gallery
    return DeviceGallery(gallery, mode=mode)


def _stream_handle(device: torch.device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


def _prep_queries(queries, gal: DeviceGallery):
    """-> (fp32 contiguous [Q, padded_dim] tensor, on_host: bool)."""
    if isinstance(queries, np.ndarray):
        queries = torch.from_numpy(queries)
    if queries.dim() == 1:
        queries = queries.unsqueeze(0)
    if queries.dim() != 2 or queries.shape[1] != gal.dim:
        raise ValueError(f"queries must be [Q, {gal.dim}], got {tuple(queries.shape)}")
    q = queries.detach()
    if q.dtype != torch.float32:
        q = q.to(torch.float32)
    if gal.padded_dim != gal.dim:
        q = torch.nn.functional.pad(q, (0, gal.padded_dim - gal.dim))
    if not q.is_contiguous():
        q = q.contiguous()
    if q.is_cuda and q.device != gal.device:
        q = q.to(gal.device)
    return q, not q.is_cuda


FP32_TC_MIN_QUERIES = 9     # fp32 galleries: K1 (CUDA cores) up to 8 queries, bf16x3 tensor-core path beyond


def _operand(gal: DeviceGallery, nq: int, path: str):
    """(pointer, row stride, dtype code) of the gallery operand the library should scan."""
    if gal.mode == "fp32" and path != "gemv" and (nq >= FP32_TC_MIN_QUERIES or path == "mma"):
        planes = gal.split3()
        return planes.data_ptr(), planes.stride(1), _cabi.DTYPE_BF16X3
    return gal.data.data_ptr(), gal.data.stride(0), gal.dtype_code


class PendingSearch:
    """Handle of an asynchronous search (`search_topk(..., sync=False)`): `values` / `indices` are
    filled once the work enqueued on the stream has run; `wait()` blocks until then, checks the
    batch's status word and returns `(values, indices)` (repeating the batch on the exhaustive path
    in the rare case a candidate list overflowed)."""

    def __init__(self, values, indices, slot, ticket, status, event, redo):
        self.values, self.indices = values, indices
        self._slot, self._ticket, self._status, self._event, self._redo = slot, ticket, status, event, redo
        self._done = slot is None
        self.retried = False       # True once wait() has repeated the batch on the exhaustive path

    def wait(self):
        if not self._done:
            self._event.synchronize()
            st = _cabi.lib.mmrs_search_status(self._status.data_ptr())
            self._slot.release(self._ticket)      # only now may the status word serve another batch
            self._done = True
            if st == _cabi.ERR_RETRY:
                self.retried = True
                self._redo(self.values, self.indices)
            else:
                _cabi.check(st)
        return self.values, self.indices


def _search_exhaustive(gal: DeviceGallery, q: torch.Tensor, k: int, normalize_queries: bool, scale: float,
                       path: str, values: torch.Tensor, indices: torch.Tensor, row_filter_ptr: int = 0,
                       labels=None) -> None:
    """The exact fallback for a batch whose candidate lists overflowed (MMRS_ERR_RETRY): every row a
    key, one query at a time.  Its 8-bytes-per-row workspace lives only for this call.
    `row_filter_ptr`: device bitmap of the allowed rows (0 = all).  `labels`: None, or (RowLabels,
    device int32 query labels [Q], label_match code) -- each query is re-run with its own label."""
    lib = _cabi.lib
    dev = gal.device
    nq = int(q.shape[0])
    with torch.cuda.device(dev):
        qd = q.to(dev) if not q.is_cuda else q
        dv = values if values.is_cuda else torch.empty((nq, k), dtype=torch.float32, device=dev)
        di = indices if indices.is_cuda else torch.empty((nq, k), dtype=torch.int64, device=dev)
        g_ptr, g_ld, g_dtype = _operand(gal, nq, path)
        ws_bytes = lib.mmrs_search_exhaustive_workspace_bytes(gal.n_rows, gal.padded_dim, nq)
        ws = torch.empty(int(ws_bytes) + 256, dtype=torch.uint8, device=dev)
        args = (g_ptr, gal.n_rows, gal.padded_dim, g_ld, g_dtype, qd.data_ptr(), nq, qd.stride(0), k,
                int(bool(normalize_queries)), float(scale), gal.row_offset, dv.data_ptr(), di.data_ptr(),
                DeviceGallery.aligned_ptr(ws), ws_bytes)
        lab = (0, 0, 0) if labels is None else (labels[0].labels.data_ptr(), labels[1].data_ptr(), labels[2])
        _cabi.check(lib.mmrs_search_topk_exhaustive(*args, row_filter_ptr, *lab, _stream_handle(dev)))
        if dv is not values:
            values.copy_(dv)
            indices.copy_(di)
        del ws


def _filter_arg(row_filter, gal: DeviceGallery):
    """`row_filter` checked against the gallery: None, a RowFilter, or a 1-D bool mask tensor."""
    if row_filter is None:
        return None
    if isinstance(row_filter, RowFilter):
        n, dev = row_filter.n_rows, row_filter.device
    else:
        row_filter = row_filter if isinstance(row_filter, torch.Tensor) else torch.from_numpy(np.asarray(row_filter))
        if row_filter.dim() != 1 or row_filter.dtype != torch.bool:
            raise ValueError(f"row_filter must be a RowFilter or a 1-D bool mask, got {row_filter.dtype} "
                             f"{tuple(row_filter.shape)}")
        n, dev = int(row_filter.numel()), (row_filter.device if row_filter.is_cuda else None)
    if n != gal.n_rows:
        raise ValueError(f"row_filter covers {n} rows, the gallery has {gal.n_rows}")
    if dev is not None and dev != gal.device:
        raise ValueError(f"row_filter is on {dev}, the gallery on {gal.device}")
    return row_filter


def _labels_arg(row_labels, query_labels, label_match, gal: DeviceGallery, nq: int):
    """(RowLabels, query labels tensor as given, label_match code) checked against the gallery, or None."""
    if row_labels is None and query_labels is None:
        if label_match != "same":
            label_match_arg(label_match)         # a typo still raises
        return None
    if row_labels is None or query_labels is None:
        raise ValueError("row_labels and query_labels come together")
    match = label_match_arg(label_match)
    if not isinstance(row_labels, RowLabels):
        raise ValueError(f"row_labels must be a RowLabels, got {type(row_labels).__name__}")
    if row_labels.n_rows != gal.n_rows:
        raise ValueError(f"row_labels covers {row_labels.n_rows} rows, the gallery has {gal.n_rows}")
    if row_labels.device != gal.device:
        raise ValueError(f"row_labels is on {row_labels.device}, the gallery on {gal.device}")
    return row_labels, query_labels_arg(query_labels, nq, gal.device), match


def _stage_query_labels(slot, ql: torch.Tensor, dev: torch.device):
    """Copy this call's query labels into the slot's own device int32 buffer on the current stream (a
    stable pointer: the slot keeps replaying one graph while the labels change per call).  Host labels
    go through pinned memory with a plain asynchronous copy.  -> (slot buffer, copy source to keep alive)."""
    n = int(ql.numel())
    buf = slot.extra.get("query_labels")
    if buf is None or buf.numel() != n:
        buf = slot.extra["query_labels"] = torch.empty(n, dtype=torch.int32, device=dev)
    src = ql.to(torch.int32)
    if not src.is_cuda:
        src = src.contiguous().pin_memory()
    buf.copy_(src, non_blocking=True)
    return buf, src


def _result_tensors(out, nq: int, k: int, on_host: bool, dev: torch.device):
    """(values, indices) a search writes: `out` checked, or new tensors (pinned host tensors for host queries)."""
    if out is not None:
        values, indices = out
        if (tuple(values.shape) != (nq, k) or tuple(indices.shape) != (nq, k) or values.dtype != torch.float32
                or indices.dtype != torch.int64 or values.is_cuda == on_host or indices.is_cuda == on_host
                or not values.is_contiguous() or not indices.is_contiguous()):
            raise ValueError(f"out must be contiguous (float32 [{nq}, {k}], int64 [{nq}, {k}]) tensors on the "
                             f"{'host' if on_host else 'device'}")
        return values, indices
    if on_host:
        return (torch.empty((nq, k), dtype=torch.float32, pin_memory=True),
                torch.empty((nq, k), dtype=torch.int64, pin_memory=True))
    return (torch.empty((nq, k), dtype=torch.float32, device=dev),
            torch.empty((nq, k), dtype=torch.int64, device=dev))


def search_topk(queries, gallery: GalleryLike, k: int, *, normalize_queries: bool = True,
                scale: float = 1.0, mode: Optional[str] = None, path: str = "auto", sync: bool = True,
                out=None, row_filter=None, row_labels=None, query_labels=None, label_match: str = "same",
                refine=None, refine_k: Optional[int] = None):
    """Per-query top-k of `scale * q @ G.T` without materialising the score matrix.

    Returns `(values [Q, k] fp32 descending, indices [Q, k] int64)` exactly like
    `torch.topk(k, dim=1, largest=True, sorted=True)` (code/utils.py:17); equal scores are ordered
    by ascending row index; indices are global (`gallery.row_offset` added).
    Host queries (CPU tensor / numpy) give host results -- the reference's call shape
    (host in, `.cpu()` out, code/search_image.py:105-109) -- device queries give device results.
    `sync=False` enqueues the search on the current stream and returns a PendingSearch, so several
    batches can be in flight.  `out=(values, indices)` writes into caller-owned tensors (pinned host
    tensors for host queries) instead of allocating; either way the library replays ONE captured
    graph per (shape, stream) slot and only re-points its query / result nodes.
    `row_filter` (a RowFilter or a bool mask [N]) restricts the search to the allowed rows: the result
    is the top-k of `gallery[mask]` with indices of the full gallery; `k` may not exceed the allowed
    rows.  A RowFilter costs one graph capture per slot; a mask is packed into a buffer of the slot on
    every call (and its allowed count read back: one host sync).
    `row_labels` (a RowLabels over the gallery's rows) with `query_labels` (an integer tensor [Q], host or
    device) makes the search label-conditioned: query q with c = query_labels[q] >= 0 sees only the rows
    whose label equals c (`label_match="same"`) or differs from c (`"other"`: hard negatives); c < 0 is
    the unlabeled search of that query, bit for bit.  With a `row_filter` too, a row must pass both.
    Unlike `row_filter`'s `k > allowed` error, a query with fewer than k eligible rows (a small class, a
    label absent from the gallery) is padded: positions n_eligible .. k-1 hold value -inf, index -1.
    The labels are copied into a buffer of the slot on every call (no host sync, one graph per slot).
    `refine` (a RefineStore holding the gallery's rows in fp32 or bf16) makes the search two-stage: the search
    above with k_c = min(refine_k, N, rows a row_filter allows) candidates and every other argument as given
    (its exhaustive retry included), then each candidate rescored against the store and the k best kept.  A
    refined score is bit for bit `full_scores(queries, DeviceGallery(features, store.mode), path="gemv")` at
    that row; whenever the candidates contain the store's exact top-k under the same constraints the result is
    that gallery's `search_topk(..., path="gemv")`.  `refine_k` (default 2 k, at most 1024) must be >= k; the
    store must match the gallery's rows, width and (for a device store) device.  DESIGN.md section 4.
    """
    gal = _as_gallery(gallery, mode)
    if refine is not None or refine_k is not None:
        return _search_refined(queries, gal, k, refine, refine_k, normalize_queries, scale, path, sync, out,
                               row_filter, dict(row_labels=row_labels, query_labels=query_labels,
                                                label_match=label_match))
    q, on_host = _prep_queries(queries, gal)
    nq = int(q.shape[0])
    k = int(k)
    if k < 1:
        raise ValueError("k must be >= 1")
    if k > gal.n_rows:
        raise RuntimeError("selected index k out of range")  # torch.topk's message
    filt = _filter_arg(row_filter, gal)
    labels = _labels_arg(row_labels, query_labels, label_match, gal, nq)
    if isinstance(filt, RowFilter) and k > filt.n_allowed:
        raise RuntimeError("selected index k out of range")
    lib = _cabi.lib
    dev = gal.device
    if torch.cuda.current_device() != dev.index:
        torch.cuda.set_device(dev)
    stream = torch.cuda.current_stream(dev)
    values, indices = _result_tensors(out, nq, k, on_host, dev)
    if nq == 0:
        if filt is not None and not isinstance(filt, RowFilter) and k > int(filt.sum()):
            raise RuntimeError("selected index k out of range")
        return (values, indices) if sync else PendingSearch(values, indices, None, None, None, None, None)
    if on_host and not q.is_pinned():
        q = q.pin_memory()
    slot = gal.search_slot(nq, k, on_host, stream.cuda_stream)
    filt_ptr = 0
    if isinstance(filt, RowFilter):
        filt_ptr = filt.words.data_ptr()
    elif filt is not None:
        # a per-call mask goes into the slot's own bitmap: a stable pointer, so the slot keeps replaying
        # one graph; calls on the slot run in stream order, so the next pack cannot overtake this search
        words = slot.extra.get("row_filter")
        if words is None:
            words = slot.extra["row_filter"] = torch.empty(filter_words(gal.n_rows), dtype=torch.int32, device=dev)
        filt = filt.to(dev)
        if k > int(pack_mask(filt, words).item()):
            raise RuntimeError("selected index k out of range")
        filt_ptr = words.data_ptr()
    if labels is not None:
        # by the time a retry runs the slot buffer may hold a later call's labels: redo keeps its own copy
        staged, src = _stage_query_labels(slot, labels[1], dev)
        labels = (labels[0], staged, labels[2], labels[1], src)
    g_ptr, g_ld, g_dtype = _operand(gal, nq, path)
    args = (g_ptr, gal.n_rows, gal.padded_dim, g_ld, g_dtype,
            q.data_ptr(), nq, q.stride(0), k, int(bool(normalize_queries)), float(scale),
            gal.row_offset, _cabi.PATHS[path], values.data_ptr(), indices.data_ptr(), slot.ptr, slot.nbytes)

    def redo(v, i):
        lab = None
        if labels is not None:
            # this call's own labels (the slot buffer may hold a later call's by now)
            lab = (labels[0], labels[3].to(device=dev, dtype=torch.int32).contiguous(), labels[2])
        if filt is None:
            _search_exhaustive(gal, q, k, normalize_queries, scale, path, v, i, 0, lab)
        else:
            # by now the slot's bitmap may hold a later call's mask: repack this call's own
            f = filt if isinstance(filt, RowFilter) else RowFilter(filt)
            _search_exhaustive(gal, q, k, normalize_queries, scale, path, v, i, f.words.data_ptr(), lab)

    if sync and filt is None and labels is None:
        fn = lib.mmrs_search_topk_host if on_host else lib.mmrs_search_topk
        st = fn(*args, stream.cuda_stream)
        if st == _cabi.ERR_RETRY:
            redo(values, indices)
        else:
            _cabi.check(st)
        return values, indices
    ticket, status, event = slot.acquire()
    fn = lib.mmrs_search_topk_host_async if on_host else lib.mmrs_search_topk_async
    lab = (0, 0, 0) if labels is None else (labels[0].labels.data_ptr(), labels[1].data_ptr(), labels[2])
    st = fn(*args, status.data_ptr(), filt_ptr, *lab, stream.cuda_stream)
    if st != _cabi.OK:
        slot.release(ticket)
        _cabi.check(st)
    event.record(stream)
    pend = PendingSearch(values, indices, slot, ticket, status, event, redo)
    pend._keepalive = (q, filt, labels)        # the enqueued copies / kernels read them
    return pend.wait() if sync else pend


class _PendingRefined:
    """Handle of an asynchronous refined search: `wait()` finishes the candidate stage first; when that batch
    was repeated on the exhaustive path, its candidates are refined again before the result is returned."""

    def __init__(self, values, indices, cand, refine_again, status, event):
        self.values, self.indices = values, indices
        self._cand, self._again, self._status, self._event = cand, refine_again, status, event
        self._done = False

    def wait(self):
        if not self._done:
            self._event.synchronize()
            self._cand.wait()
            self._done = True
            if self._cand.retried:
                self._again()                    # the enqueued refine read the overflowed lists
            else:
                _cabi.check(_cabi.lib.mmrs_search_status(self._status.data_ptr()))
        return self.values, self.indices


def _search_refined(queries, gal: DeviceGallery, k, store, refine_k, normalize_queries, scale, path, sync, out,
                    row_filter, label_kw):
    """search_topk with a RefineStore: candidate stage, then mmrs_refine_topk on the same stream."""
    from .refine import RefineStore, candidate_k
    if not isinstance(store, RefineStore):
        raise ValueError(f"refine must be a RefineStore, got {type(store).__name__}")
    store.check_matches(gal)
    q, on_host = _prep_queries(queries, gal)
    nq = int(q.shape[0])
    k = int(k)
    if k < 1:
        raise ValueError("k must be >= 1")
    if k > gal.n_rows:
        raise RuntimeError("selected index k out of range")
    filt = _filter_arg(row_filter, gal)
    allowed = None
    if isinstance(filt, RowFilter):
        allowed = filt.n_allowed
    elif filt is not None:
        allowed = int(filt.sum())
    if allowed is not None and k > allowed:
        raise RuntimeError("selected index k out of range")
    k_c = candidate_k(k, refine_k, gal.n_rows, allowed)
    dev = gal.device
    if torch.cuda.current_device() != dev.index:
        torch.cuda.set_device(dev)
    stream = torch.cuda.current_stream(dev)
    values, indices = _result_tensors(out, nq, k, on_host, dev)
    if nq == 0:
        return (values, indices) if sync else PendingSearch(values, indices, None, None, None, None, None)
    qd = q.pin_memory().to(dev, non_blocking=True) if on_host else q      # [nq, gal.padded_dim] fp32
    cand = search_topk(qd[:, :gal.dim], gal, k_c, normalize_queries=normalize_queries, scale=scale, path=path,
                       sync=sync, row_filter=filt, **label_kw)
    cand_idx = cand[1] if sync else cand.indices
    dv, di = (torch.empty((nq, k), dtype=torch.float32, device=dev),
              torch.empty((nq, k), dtype=torch.int64, device=dev)) if on_host else (values, indices)
    lib = _cabi.lib
    ws_bytes = lib.mmrs_refine_workspace_bytes(store.padded_dim, nq, k_c)
    ws = gal.workspace(("refine", nq, k_c, stream.cuda_stream), ws_bytes)

    def run(status_ptr: int):
        local = cand_idx
        if gal.row_offset:                       # a shard's candidates carry global rows: the store is local
            local = torch.where(cand_idx >= 0, cand_idx - gal.row_offset, cand_idx)
        _cabi.check(lib.mmrs_refine_topk(store.ptr, store.dtype_code, store.n_rows, store.padded_dim, store.ld,
                                         qd.data_ptr(), nq, qd.stride(0), int(bool(normalize_queries)), float(scale),
                                         local.data_ptr(), k_c, gal.row_offset, k, dv.data_ptr(), di.data_ptr(),
                                         DeviceGallery.aligned_ptr(ws), ws_bytes, status_ptr, stream.cuda_stream))
        if on_host:
            values.copy_(dv, non_blocking=True)
            indices.copy_(di, non_blocking=True)
        return local

    if sync:
        run(0)
        if on_host:
            stream.synchronize()
        return values, indices
    status = torch.zeros(1, dtype=torch.int32).pin_memory()
    local = run(status.data_ptr())
    event = torch.cuda.Event()
    event.record(stream)

    def again():
        with torch.cuda.stream(stream):
            run(0)
        stream.synchronize()

    pend = _PendingRefined(values, indices, cand, again, status, event)
    pend._keepalive = (qd, local, ws)            # the enqueued kernels read them
    return pend


def full_scores(queries, gallery: GalleryLike, *, normalize_queries: bool = True, scale: float = 1.0,
                mode: Optional[str] = None, path: str = "auto") -> torch.Tensor:
    """[Q, N] fp32 scores `scale * q @ G.T` (the expression of code/search_image.py:107,
    CLIP/lab3.py:114 for all classes at once).  Host queries give a host result."""
    gal = _as_gallery(gallery, mode)
    q, on_host = _prep_queries(queries, gal)
    nq = int(q.shape[0])
    with torch.cuda.device(gal.device):
        if on_host:
            q = q.to(gal.device)
        out = torch.empty((nq, gal.n_rows), dtype=torch.float32, device=gal.device)
        _scores_into(gal, q, out, normalize_queries, scale, path)
    return out.cpu() if on_host else out


def _scores_into(gal: DeviceGallery, q: torch.Tensor, out: torch.Tensor, normalize_queries: bool, scale: float,
                 path: str) -> None:
    """mmrs_full_scores of prepared device queries `q` [nq, padded_dim] into `out` [>= nq, N] (row stride
    out.stride(0)); the kernel is chosen for nq queries."""
    nq = int(q.shape[0])
    if nq == 0:
        return
    lib = _cabi.lib
    ws_bytes = lib.mmrs_full_scores_workspace_bytes(gal.n_rows, gal.padded_dim, gal.dtype_code, nq)
    ws = gal.workspace(("scores", nq), ws_bytes)
    g_ptr, g_ld, g_dtype = _operand(gal, nq, path)
    _cabi.check(lib.mmrs_full_scores(g_ptr, gal.n_rows, gal.padded_dim,
                                     g_ld, g_dtype, q.data_ptr(), nq,
                                     q.stride(0), int(bool(normalize_queries)), float(scale),
                                     _cabi.PATHS[path], out.data_ptr(), out.stride(0),
                                     DeviceGallery.aligned_ptr(ws), ws_bytes,
                                     _stream_handle(gal.device)))


# one-entry upload cache: the reference re-uploads `features` on every call (:107); a script that
# passes the SAME host tensor object again (identity, same in-place version) reuses the resident copy.
# The entry holds a strong reference to that tensor, so its address cannot be recycled by a different
# tensor while the entry lives (a data_ptr key could: the allocator reuses freed blocks at once).
# numpy arrays have no version counter -- in-place edits are invisible -- and are uploaded every time;
# pass a DeviceGallery to keep a gallery resident explicitly.
_last_upload: dict = {}


def _resident(features, mode: Optional[str]) -> DeviceGallery:
    if isinstance(features, DeviceGallery):
        return features
    if isinstance(features, np.ndarray):
        return DeviceGallery(torch.from_numpy(features), mode=mode)
    hit = _last_upload.get("entry")
    if hit is not None and hit[0] is features and hit[1] == features._version and hit[2] == mode:
        return hit[3]
    gal = DeviceGallery(features, mode=mode)
    _last_upload["entry"] = (features, features._version, mode, gal)
    return gal


def get_similarity(features, targets, label, ref_feature, device="cuda"):
    """Drop-in for code/search_image.py:105-117.

    `similarity = 100. * features.cuda() @ ref_feature.t()`; scores copied to host and split by
    `targets == label` -> `(pos_res, neg_res)` numpy arrays.  `features` may be the host tensor
    the reference passes (uploaded once, see _resident) or a DeviceGallery."""
    del device  # the reference ignores its own argument too (hard-coded .cuda())
    gal = _resident(features, None)
    with torch.no_grad():
        q = ref_feature if isinstance(ref_feature, torch.Tensor) else torch.as_tensor(ref_feature)
        q = q.detach().reshape(1, -1).to(torch.float32)
        if not q.is_cuda:
            q = q.to(gal.device)
        scores = full_scores(q, gal, normalize_queries=False, scale=100.0)[0].cpu().numpy()
        targets = np.asarray(targets)
        pos_mask = (targets == label)
        neg_mask = (targets != label)
        return scores[pos_mask], scores[neg_mask]


def get_similarity_from_matrix(similarity, targets, label, device="cuda"):
    """Drop-in for the OTHER `get_similarity` of the reference, code/main_custom.py:93-105: the scores of
    class `label` are a column of an already computed [N, classes] similarity matrix (e.g.
    `full_scores(class_embeddings, gallery).T`); returns (pos_res, neg_res) split by `targets == label`."""
    scores = similarity[:, label]
    scores = scores.detach().cpu().numpy() if isinstance(scores, torch.Tensor) else np.asarray(scores)
    t = targets.detach().cpu().numpy() if isinstance(targets, torch.Tensor) else np.asarray(targets)
    return scores[t == label], scores[t != label]


def construct_dataset(feature_dict, sample_images, class_name):
    """Drop-in for code/search_image.py:167-182: gallery of every cached image except the
    `sample_images` of `class_name`; returns `(test_features [N, D] tensor, targets np.ndarray)`.
    Uses this module's `class_names`, `class_to_idx`, `dataset_path` like the reference's globals."""
    test_imgs = []
    targets = []
    for cls_name in class_names:
        listing = os.listdir(os.path.join(dataset_path, cls_name))
        if cls_name == class_name:
            listing = [p for p in listing if p not in sample_images]
        test_imgs.extend(cls_name + "/" + p for p in listing)
        targets.extend([class_to_idx[cls_name]] * len(listing))
    targets = np.array(targets)
    test_features = torch.tensor(np.array([feature_dict[img] for img in test_imgs]))
    return test_features, targets


# ---- query construction on cached features (SURVEY.md section 8 row a3) ---------------------------
def outlier_filter_features(image_features, keep_percentile: float = 95):
    """The arithmetic of `outlier_filter` (code/search_image.py:310-318) on already encoded,
    unit-norm sample features [S, D] (the CLIP forward of :296-309 is the caller's): mean of the
    samples whose cosine distance to the global mean is within the 95th percentile.  The result is
    NOT re-normalised, as in the reference (SURVEY.md M3).  S is ~10: host numpy, like the reference."""
    f = np.asarray(image_features.detach().cpu() if isinstance(image_features, torch.Tensor) else image_features)
    center = np.mean(f, axis=0)
    cos_distances = 1 - f @ center
    keep_mask = cos_distances <= np.percentile(cos_distances, keep_percentile)
    return torch.tensor(np.mean(f[keep_mask], axis=0))


def mix_image_text_query(image_prototype, text_embedding):
    """`(robust_features + class_embeddings[c]) / 2` (code/search_image.py:387): the query handed to
    get_similarity; un-normalised on purpose."""
    return (torch.as_tensor(image_prototype) + torch.as_tensor(text_embedding)) / 2


def image_text_prototypes(image_features, text_embedding):
    """The arithmetic of `get_image_text_features` (code/search_image.py:128-140) on already encoded
    sample features [S, D] (as they leave `encode_image`, not yet normalised) and the class's text
    embedding [D]: returns `(image_features, image_text_features)` --
      image_text_features = mean over samples of (unit image row + unit text row) / 2   (:135-136)
      image_features      = mean of the unit image rows, re-normalised                    (:137-139)
    S is the shot count (<= 50): host torch, like the reference's few-row tensors."""
    img = torch.as_tensor(image_features).detach().to(torch.float32).clone()
    txt = torch.as_tensor(text_embedding).detach().to(torch.float32).reshape(1, -1).repeat(img.shape[0], 1)
    txt /= txt.norm(dim=-1, keepdim=True)
    img /= img.norm(dim=-1, keepdim=True)
    image_text_features = ((img + txt) / 2.).mean(dim=0)
    image_mean = img.mean(dim=0)
    image_mean /= image_mean.norm()
    return image_mean, image_text_features


def _encode_samples(clip_model, preprocess, sample_images, class_name):
    """Load and encode the sample images exactly as the reference's query builders do
    (code/search_image.py:120-131, :187-196): `dataset_path/class_name/sample`, RGB, `preprocess`,
    stacked, `clip_model.encode_image`.  The encoder is the caller's (out of scope here)."""
    from PIL import Image
    images = []
    class_path = os.path.join(dataset_path, class_name)
    for sample_img in sample_images:
        with open(os.path.join(class_path, sample_img), "rb") as f:
            images.append(preprocess(Image.open(f).convert("RGB")))
    images = torch.stack(images, dim=0)
    try:
        images = images.to(next(clip_model.parameters()).device)
    except (AttributeError, StopIteration, TypeError):
        pass
    with torch.no_grad():
        return clip_model.encode_image(images)


def get_image_text_features(clip_model, preprocess, class_embeddings, sample_images, class_name):
    """Drop-in for code/search_image.py:119-140 -> (image_features [D], image_text_features [D])."""
    feats = _encode_samples(clip_model, preprocess, sample_images, class_name)
    return image_text_prototypes(feats.float().cpu(), torch.as_tensor(class_embeddings[class_to_idx[class_name]]).cpu())


def cluster_prototype(image_features, shots: int, *, random_state=None):
    """The arithmetic of `get_cluster_features` (code/search_image.py:197-232) on encoded sample
    features: unit-normalise, 2-means, then the mean of the `shots` samples nearest to the global
    centre (clusters of similar size, :210-213) or to the majority cluster's centre (:214-227).
    `random_state` seeds KMeans (the reference leaves it unseeded).  Returns a [D] fp32 tensor."""
    from collections import Counter
    from sklearn.cluster import KMeans
    f = torch.as_tensor(image_features).detach().to(torch.float32)
    f = (f / f.norm(dim=-1, keepdim=True)).cpu().numpy()
    kmeans = KMeans(n_clusters=2, random_state=random_state)
    kmeans.fit(f)
    cluster_labels = kmeans.labels_
    label_counts = Counter(cluster_labels)
    majority_label = max(label_counts, key=label_counts.get)
    if abs(label_counts[0] - label_counts[1]) / len(cluster_labels) < 0.2:
        distances = np.linalg.norm(f - kmeans.cluster_centers_.mean(axis=0), axis=1)
        nearest_indices = np.argsort(distances)[:shots]
    else:
        majority_mask = (cluster_labels == majority_label)
        distances = np.linalg.norm(f[majority_mask] - kmeans.cluster_centers_[majority_label], axis=1)
        nearest_indices = np.where(majority_mask)[0][np.argsort(distances)[:shots]]
    return torch.tensor(np.mean(f[nearest_indices], axis=0))


def get_cluster_features(clip_model, preprocess, sample_imgs, shots, class_name):
    """Drop-in for code/search_image.py:185-232 (host result; the reference moves it to the GPU)."""
    return cluster_prototype(_encode_samples(clip_model, preprocess, sample_imgs, class_name).float().cpu(), shots)


# ---- top-k over an existing score matrix; cls_acc (code/utils.py:15-39) --------------------------------
def topk_of_scores(scores, k: int):
    """`scores.topk(k, 1, True, True)` (code/utils.py:17) for a [N, C] score matrix that already
    exists (the Tip-Adapter logits of code/main_custom.py): one select CTA per row on packed
    (score, ~column) keys -- values descending, equal scores by ascending column.  C * 1 lists of
    length C: C may be anything, k <= min(C, 1024).  Host input gives a host result."""
    t = scores if isinstance(scores, torch.Tensor) else torch.as_tensor(np.asarray(scores))
    if t.dim() != 2:
        raise ValueError("scores must be [N, C]")
    n, c = int(t.shape[0]), int(t.shape[1])
    k = int(k)
    if k < 1:
        raise ValueError("k must be >= 1")
    if k > c:
        raise RuntimeError("selected index k out of range")
    on_host = not t.is_cuda
    dev = t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)
    _cabi.require_b200(dev.index or 0)
    lib = _cabi.lib
    with torch.cuda.device(dev):
        v_in = t.detach().to(device=dev, dtype=torch.float32).contiguous()
        i_in = torch.arange(c, dtype=torch.int64, device=dev).repeat(n, 1)
        out_v = torch.empty((n, k), dtype=torch.float32, device=dev)
        out_i = torch.empty((n, k), dtype=torch.int64, device=dev)
        if n:
            ws_bytes = lib.mmrs_topk_merge_workspace_bytes(1, n, c)
            ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
            _cabi.check(lib.mmrs_topk_merge(v_in.data_ptr(), i_in.data_ptr(), 1, n, c, k, out_v.data_ptr(),
                                            out_i.data_ptr(), DeviceGallery.aligned_ptr(ws), ws_bytes,
                                            _stream_handle(dev)))
    return (out_v.cpu(), out_i.cpu()) if on_host else (out_v, out_i)


def cls_acc(output, target, topk=1, exclude_class=None):
    """Drop-in for code/utils.py:15-39: percentage of rows whose `topk` best-scoring classes contain
    the target; rows with `target == exclude_class` are left out; 0.0 when nothing is left.  The
    top-k (:17) runs on the GPU select kernel (`topk_of_scores`)."""
    target = torch.as_tensor(target)
    pred = topk_of_scores(output, topk)[1].t().to(target.device)          # [topk, batch]
    correct = pred.eq(target.view(1, -1).expand_as(pred))
    mask = target.ne(exclude_class) if exclude_class is not None else torch.ones_like(target, dtype=torch.bool)
    correct = correct[:, mask]
    valid_num = mask.sum().item()
    if valid_num == 0:
        return 0.0
    acc = correct.any(dim=0).float().sum().item()
    return 100 * acc / valid_num


# ---- logit_scale * F.cosine_similarity (code/merge_dataset.py:275-278, :303) ------------------------------
def cosine_similarity_scores(image_features, text_features, logit_scale=1.0, eps: float = 1e-8):
    """`logit_scale * torch.nn.functional.cosine_similarity(image_features, text_features)` for image rows
    [B, D] against ONE text row ([1, D] or [D], the reference's use): each side is divided by
    max(||x||, eps) -- torch's clamp semantics, NOT the `x / x.norm()` idiom of search_image.py:157 (a zero
    row scores 0 here, NaN there) -- then the rows are scored by the gallery scan with scale = logit_scale.
    Returns [B] fp32 (host input -> host result)."""
    x = image_features if isinstance(image_features, torch.Tensor) else torch.as_tensor(np.asarray(image_features))
    t = text_features if isinstance(text_features, torch.Tensor) else torch.as_tensor(np.asarray(text_features))
    t = t.detach().to(torch.float32).reshape(-1, x.shape[-1])
    if x.dim() != 2 or t.shape[0] != 1:
        raise ValueError("image_features must be [B, D] and text_features one row ([1, D] or [D])")
    on_host = not x.is_cuda
    x = x.detach().to(torch.float32)
    xn = x / x.norm(dim=1, keepdim=True).clamp_min(eps)
    tn = (t / t.norm(dim=1, keepdim=True).clamp_min(eps)).to(x.device)
    scale = float(logit_scale.detach().float().item()) if isinstance(logit_scale, torch.Tensor) else float(logit_scale)
    out = full_scores(tn, DeviceGallery(xn, mode="fp32"), normalize_queries=False, scale=scale)[0]
    return out.cpu() if on_host else out


# ---- threshold sweep (SURVEY.md section 8 row f2) ---------------------------------------------------
def _is_f64(x) -> bool:
    if isinstance(x, torch.Tensor):
        return x.dtype == torch.float64
    a = np.asarray(x)
    return a.dtype == np.float64 or a.dtype.kind not in "f"      # python floats / ints compare as float64 in numpy


def threshold_sweep_counts(pos_res, neg_res, thresholds, device: Optional[torch.device] = None):
    """(tp [T], fp [T]) int64 numpy: tp[t] = #{pos >= thresholds[t]}, fp likewise, on the GPU.
    Thresholds must be ascending (np.linspace(min, max, T) is).  The comparison is numpy's: float32
    scores are promoted to float64 against the float64 grid; float64 scores (e.g. Python floats, a
    float64 similarity matrix) are compared as they are -- they are never rounded to float32."""
    thr = np.ascontiguousarray(np.asarray(thresholds, dtype=np.float64).reshape(-1))
    if thr.size > 1 and np.any(np.diff(thr) < 0):
        raise ValueError("thresholds must be ascending")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)
    _cabi.require_b200(dev.index or 0)
    f64 = _is_f64(pos_res) or _is_f64(neg_res)
    tdt, ndt = (torch.float64, np.float64) if f64 else (torch.float32, np.float32)

    def dev_scores(x):
        if isinstance(x, torch.Tensor):
            return x.detach().to(device=dev, dtype=tdt).contiguous().reshape(-1)
        return torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=ndt).reshape(-1))).to(dev)

    with torch.cuda.device(dev):
        p, n = dev_scores(pos_res), dev_scores(neg_res)
        t = torch.from_numpy(thr).to(dev)
        out = torch.empty((thr.size, 2), dtype=torch.int64, device=dev)
        ws_bytes = _cabi.lib.mmrs_threshold_sweep_workspace_bytes(thr.size)
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        fn = _cabi.lib.mmrs_threshold_sweep_f64 if f64 else _cabi.lib.mmrs_threshold_sweep
        _cabi.check(fn(p.data_ptr(), p.numel(), n.data_ptr(), n.numel(), t.data_ptr(), thr.size, out.data_ptr(),
                       DeviceGallery.aligned_ptr(ws), ws_bytes, _stream_handle(dev)))
        counts = out.cpu().numpy()
    return counts[:, 0].copy(), counts[:, 1].copy()


def _f1_from_counts(tp, fp, n_pos):
    # the reference's arithmetic (code/search_image.py:43-54): numpy int64 counts, float64 ratios,
    # 0/0 -> nan exactly as there
    fn = n_pos - tp
    with np.errstate(divide="ignore", invalid="ignore"):
        precision = tp / (tp + fp)
        recall = tp / (tp + fn)
        f1 = 2 * precision * recall / (precision + recall)
    return f1, precision, recall


def grid_f32() -> int:
    """1 when np.linspace of two float32 scalars is float32 (NEP 50, NumPy >= 2), 0 when float64 (NumPy 1.x):
    the device grid follows the installed numpy."""
    return int(np.linspace(np.float32(0), np.float32(1), 3).dtype == np.float32)


def best_from_counts(thresholds, counts, n_pos: int):
    """find_thresholds' tail (code/search_image.py:62-79) on the sweep's (tp, fp) counts [T, 2]:
    -> (best_f1, best_threshold, best_precision, best_recall, f1_scores); the first strict maximum wins."""
    f1s, ps, rs = _f1_from_counts(counts[:, 0], counts[:, 1], n_pos)
    best = (0., 0., 0., 0.)
    for th, f1, p, r in zip(thresholds, f1s, ps, rs):
        if f1 > best[0]:                      # first strict maximum wins (:74)
            best = (f1, th, p, r)
    return best[0], best[1], best[2], best[3], f1s


def best_threshold_on_device(scores: torch.Tensor, targets, label, n_points: int = 200):
    """find_thresholds (code/search_image.py:58-79) for scores that never leave the GPU: `scores` is a
    CUDA fp32 vector (e.g. one row of full_scores), `targets` the class ids.  Returns
    (best_f1, best_threshold, best_precision, best_recall, thresholds, f1_scores); only the
    n_points-sized grid and counts are copied to the host."""
    dev = scores.device
    _cabi.require_b200(dev.index or 0)
    s = scores.detach().to(torch.float32).contiguous().reshape(-1)
    t = torch.as_tensor(np.asarray(targets) if not isinstance(targets, torch.Tensor) else targets)
    t = t.to(device=dev, dtype=torch.int64).contiguous().reshape(-1)
    if t.numel() != s.numel():
        raise ValueError("scores and targets differ in length")
    lib = _cabi.lib
    with torch.cuda.device(dev):
        thr = torch.empty(n_points, dtype=torch.float64, device=dev)
        out = torch.empty((n_points, 2), dtype=torch.int64, device=dev)
        ws_bytes = lib.mmrs_threshold_sweep_workspace_bytes(n_points) + 256
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        _cabi.check(lib.mmrs_threshold_sweep_labeled(s.data_ptr(), t.data_ptr(), int(label), s.numel(), n_points,
                                                     grid_f32(), thr.data_ptr(), out.data_ptr(),
                                                     DeviceGallery.aligned_ptr(ws), ws_bytes, _stream_handle(dev)))
        n_pos = int((t == int(label)).sum().item())
        counts = out.cpu().numpy()
        thresholds = thr.cpu().numpy()
    best_f1, best_thr, best_p, best_r, f1s = best_from_counts(thresholds, counts, n_pos)
    return best_f1, best_thr, best_p, best_r, thresholds, f1s


def evaluate_thresholds(similarities, thresholds, positive_class, negative_class):
    """Drop-in for `evaluate_thresholds` of CLIP/lab3.py:39-65 (also CLIP-Chinese/lab_chinese.py,
    CLIP/union_dataset.py:46): `similarities` is the list of {"similarity", "true_label", ...} dicts the
    lab scripts build, only items of the two named classes count; returns one dict per threshold with
    threshold / precision / recall / f1 / TP / FP / TN / FN (0 where a denominator is 0).  The
    O(T * N) generator sums of :47-48 (1001 thresholds) run as one GPU histogram pass."""
    rel = [it for it in similarities if it["true_label"] in [positive_class, negative_class]]
    sim64 = np.array([it["similarity"] for it in rel], dtype=np.float64)
    sim32 = sim64.astype(np.float32)
    if not np.array_equal(sim32.astype(np.float64), sim64):
        sim32 = sim64      # not float32-representable: compared in float64, exactly as the reference's Python floats
    is_pos = np.array([it["true_label"] == positive_class for it in rel], dtype=bool)
    total_pos, total_neg = int(is_pos.sum()), int((~is_pos).sum())
    thr = np.asarray(thresholds, dtype=np.float64).reshape(-1)
    order = np.argsort(thr, kind="stable")
    tp_s, fp_s = threshold_sweep_counts(sim32[is_pos], sim32[~is_pos], thr[order])
    tp = np.empty_like(tp_s); fp = np.empty_like(fp_s)
    tp[order], fp[order] = tp_s, fp_s
    results = []
    for threshold, TP, FP in zip(thresholds, tp.tolist(), fp.tolist()):
        FN, TN = total_pos - TP, total_neg - FP
        precision = TP / (TP + FP) if (TP + FP) > 0 else 0
        recall = TP / (TP + FN) if (TP + FN) > 0 else 0
        f1 = 2 * precision * recall / (precision + recall) if (precision + recall) > 0 else 0
        results.append({"threshold": threshold, "precision": precision, "recall": recall, "f1": f1,
                        "TP": TP, "FP": FP, "TN": TN, "FN": FN})
    return results


def score_classes(image_features, text_features, classes, labels, paths, *, scorer=None):
    """The similarity loop of the lab pipelines as ONE scoring call: CLIP/lab3.py:108-117,
    CLIP/union_dataset.py:247-260 (`process_images`, D = 512) and CLIP-Chinese/lab_chinese.py:116-120
    (D = 768) normalise each image batch (`feats / feats.norm(dim=1, keepdim=True)`) and then, class by
    class, run `feats @ text_features[cls].t()` followed by a blocking `.cpu()` -- five GEMVs and five
    syncs per batch of 64.  Here all images of the run and all classes go through one `full_scores`
    call: the normalised image rows are the gallery (streamed once), the class embeddings the queries.

    image_features [N, D] (as they leave the image tower, NOT yet normalised), text_features
    {class: [1, D] or [D] unit vector} as built at lab3.py:84-90, `labels` / `paths` the N true labels
    and file paths.  Returns {class: [{"similarity": float, "true_label": ..., "file_path": ...}, ...]}
    in image order, items labelled "error" skipped (lab3.py:116) -- exactly what `evaluate_thresholds`
    and `calc_combined_metrics` consume.  `scorer` is a test hook with the signature of `full_scores`."""
    classes = list(classes)
    labels, paths = list(labels), list(paths)
    feats = image_features if isinstance(image_features, torch.Tensor) else torch.as_tensor(np.asarray(image_features))
    if feats.dim() != 2 or feats.shape[0] != len(labels) or len(labels) != len(paths):
        raise ValueError("image_features must be [N, D] with N labels and N paths")
    out = {cls: [] for cls in classes}
    if not classes or feats.shape[0] == 0:
        return out
    text = torch.stack([torch.as_tensor(text_features[cls]).detach().float().cpu().reshape(-1) for cls in classes])
    if text.shape[1] != feats.shape[1]:
        raise ValueError("text and image features differ in width")
    score = full_scores if scorer is None else scorer
    feats = feats.detach().float()
    feats = feats / feats.norm(dim=1, keepdim=True)      # lab3.py:112, at ingest like build_cache (search_image.py:157)
    sims = score(text, feats, normalize_queries=False, mode="fp32")        # [n_classes, N]; text rows are unit (lab3.py:90)
    sims = sims.cpu().numpy()
    keep = [i for i, lab in enumerate(labels) if lab != "error"]
    for c, cls in enumerate(classes):
        col = sims[c]
        out[cls] = [{"similarity": float(col[i]), "true_label": labels[i], "file_path": paths[i]} for i in keep]
    return out


def calc_combined_metrics(en_sims, cn_sims, en_threshs, cn_threshs, en_pos, en_neg, cn_pos, cn_neg, verbose=False):
    """Drop-in for `calc_combined_metrics` of CLIP/union_dataset.py:133-231: per class pair, an image
    (keyed by file basename) counts as detected when the English OR the Chinese model scores it at or
    above that model's threshold; TP over the union of both models' positive-class images, FP over
    the union of the negative-class images.  Same argument order and result dicts; the reference's
    debug prints are behind `verbose`.  Basenames repeated inside one model's list: the last item
    wins, as the reference's dict assignments do."""
    results = []
    for i, en_pos_cls in enumerate(en_pos):
        cn_pos_cls, en_neg_cls, cn_neg_cls = cn_pos[i], en_neg[i], cn_neg[i]
        en_thresh, cn_thresh = en_threshs[i], cn_threshs[i]

        def flags(items, label, thresh):
            return {os.path.basename(it["file_path"]): it["similarity"] >= thresh
                    for it in items if it["true_label"] == label}

        en_p, en_n = flags(en_sims[en_pos_cls], en_pos_cls, en_thresh), flags(en_sims[en_pos_cls], en_neg_cls, en_thresh)
        cn_p, cn_n = flags(cn_sims[cn_pos_cls], cn_pos_cls, cn_thresh), flags(cn_sims[cn_pos_cls], cn_neg_cls, cn_thresh)
        pos_names, neg_names = en_p.keys() | cn_p.keys(), en_n.keys() | cn_n.keys()
        tp = sum(1 for b in pos_names if en_p.get(b, False) or cn_p.get(b, False))
        fp = sum(1 for b in neg_names if en_n.get(b, False) or cn_n.get(b, False))
        total_pos, total_neg = len(pos_names), len(neg_names)
        fn = total_pos - tp
        prec = tp / (tp + fp) if (tp + fp) > 0 else 0
        rec = tp / (tp + fn) if (tp + fn) > 0 else 0
        f1 = 2 * prec * rec / (prec + rec) if (prec + rec) > 0 else 0
        if verbose:
            print(f"{en_pos_cls} vs {en_neg_cls}: unique pos {total_pos}, unique neg {total_neg}, "
                  f"TP {tp}, FP {fp}, FN {fn}, precision {prec:.3f}, recall {rec:.3f}, F1 {f1:.3f}")
        results.append({"en_positive_class": en_pos_cls, "en_negative_class": en_neg_cls,
                        "cn_positive_class": cn_pos_cls, "cn_negative_class": cn_neg_cls,
                        "en_threshold": en_thresh, "cn_threshold": cn_thresh,
                        "combined_f1": f1, "combined_precision": prec, "combined_recall": rec,
                        "TP": tp, "FP": fp, "FN": fn,
                        "total_unique_pos": total_pos, "total_unique_neg": total_neg})
    return results


def eval_threshold(pos_res, neg_res, threshold):
    """Drop-in for code/search_image.py:39-56 -> (f1_score, precision, recall)."""
    tp, fp = threshold_sweep_counts(pos_res, neg_res, [threshold])
    f1, p, r = _f1_from_counts(tp, fp, int(np.asarray(pos_res).size))
    return f1[0], p[0], r[0]


def find_thresholds(pos_res, neg_res, target_class, verbose=False, grid="full"):
    """Drop-in for code/search_image.py:58-103: 200-point linspace over [min, max] of all scores,
    F1 per threshold, FIRST strict maximum wins (:74); returns best_f1_score.  The O(200 * N)
    interpreted `sum(pos_res >= threshold)` loops run as one histogram pass on the GPU.
    grid="overlap" is the variant of code/main_custom.py:46-50: the grid spans only the range where
    positive and negative scores overlap, [max(min pos, min neg), min(max pos, max neg)], with
    int(10 * width) points (none at all when the classes overlap over less than 0.1)."""
    pos_np = np.asarray(pos_res)
    neg_np = np.asarray(neg_res)
    if grid == "full":
        min_val = min(pos_np.min(), neg_np.min())
        max_val = max(pos_np.max(), neg_np.max())
        thresholds = np.linspace(min_val, max_val, 200)
    elif grid == "overlap":
        min_val = max(pos_np.min(), neg_np.min())
        max_val = min(pos_np.max(), neg_np.max())
        thresholds = np.linspace(min_val, max_val, int((max_val - min_val) * 10))
    else:
        raise ValueError("grid must be 'full' (search_image.py) or 'overlap' (main_custom.py)")
    if thresholds.size:
        tp, fp = threshold_sweep_counts(pos_np, neg_np, thresholds)
        f1s, ps, rs = _f1_from_counts(tp, fp, int(pos_np.size))
    else:
        f1s = ps = rs = np.zeros(0)

    best_threshold = 0.
    best_f1_score = 0.
    best_precision = 0.
    best_recall = 0.
    for t, f1, p, r in zip(thresholds, f1s, ps, rs):
        if f1 > best_f1_score:
            best_threshold, best_f1_score, best_precision, best_recall = t, f1, p, r

    if verbose:
        print(f"{target_class}_best_threshold", best_threshold)
        print(f"{target_class}_best_f1_score", best_f1_score)
        print(f"{target_class}_best_precision", best_precision)
        print(f"{target_class}_best_recall", best_recall)
        try:  # the reference plots the curve (:81-100); matplotlib is optional here
            import matplotlib
            matplotlib.use("Agg")
            import matplotlib.pyplot as plt
            plt.figure(figsize=(9, 9))
            plt.plot(thresholds, f1s)
            plt.scatter(x=best_threshold, y=best_f1_score)
            plt.annotate(f"threshold:{best_threshold:.5f}/f1:{best_f1_score:.5f}", xy=(best_threshold, best_f1_score))
            plt.xlabel('threshold')
            plt.ylabel('f1_score')
            plt.title(f'{target_class}_precision:{best_precision:.4f}_recall:{best_recall:.4f}')
            plt.savefig(f'result_{target_class}_all.jpg')
        except ImportError:
            print("(matplotlib not installed: F1 curve not plotted)")
        print('done')
    return best_f1_score
