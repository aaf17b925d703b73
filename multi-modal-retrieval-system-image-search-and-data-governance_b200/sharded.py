"""Row-sharded gallery over the GPUs of one box (SURVEY.md section 8e).

One process per GPU (`torch.distributed`, backend "nccl" over NVLink 5 / NVSwitch).  The gallery is
split into contiguous row blocks, queries are replicated, every rank runs the fused local top-k
on its shard with global row ids, ONE all-gather moves the `[Q, k]` (value, index) lists --
Q*k*12 bytes per rank -- and every rank merges the `world * k` candidates per query with the same
order rule (score desc, index asc).  There is no other exchange: the scan itself is embarrassingly
parallel, so scaling is weak in the gallery and the collective is latency-sized.

The reference has no distributed code at all (SURVEY.md section 2); this is new.
"""
from __future__ import annotations

import math
from typing import Callable, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _cabi
from .gallery import DeviceGallery
from .row_filter import RowFilter
from .row_labels import RowLabels, label_match_arg, query_labels_arg


def shard_bounds(n_rows: int, world: int, align: int = 128) -> list[tuple[int, int]]:
    """Contiguous [lo, hi) row blocks, one per rank, block starts aligned to the 128-row tile
    (global index = lo + local index).  Earlier ranks hold lower indices, so "lower rank first"
    agrees with the index-ascending tie rule."""
    if world < 1:
        raise ValueError("world must be >= 1")
    per = math.ceil(n_rows / world / align) * align if n_rows > 0 else 0
    out = []
    for r in range(world):
        lo = min(n_rows, r * per)
        hi = min(n_rows, lo + per)
        out.append((lo, hi))
    return out


def triangle_bounds(n_rows: int, world: int, align: int = 128) -> list[tuple[int, int]]:
    """Row ranges of the i-side of the upper-triangular self-join with equal PAIR counts:
    rows [lo, hi) own pairs (i, j > i), i.e. area ~ integral of (n - i); boundary r solves
    1 - (1 - x)^2 = r / world."""
    bounds = [0]
    for r in range(1, world):
        x = 1.0 - math.sqrt(1.0 - r / world)
        b = int(round(x * n_rows / align)) * align
        bounds.append(min(max(b, bounds[-1]), n_rows))
    bounds.append(n_rows)
    return [(bounds[i], bounds[i + 1]) for i in range(world)]


def _all_gather(t: torch.Tensor, world: int, group) -> torch.Tensor:
    """[world, *t.shape] gathered copy of `t` (same shape on every rank); one collective."""
    t = t.contiguous()
    out = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
    if t.numel():
        dist.all_gather_into_tensor(out.view(-1), t.view(-1), group=group)
    return out


def _merge_cuda(values: torch.Tensor, indices: torch.Tensor, k: int):
    """values/indices [G, Q, k_in] on one device -> merged (values [Q, k], indices [Q, k])."""
    g, q, kin = values.shape
    dev = values.device
    lib = _cabi.lib
    out_v = torch.empty((q, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((q, k), dtype=torch.int64, device=dev)
    if q == 0:
        return out_v, out_i
    with torch.cuda.device(dev):
        ws_bytes = lib.mmrs_topk_merge_workspace_bytes(g, q, kin)
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        _cabi.check(lib.mmrs_topk_merge(values.contiguous().data_ptr(), indices.contiguous().data_ptr(),
                                        g, q, kin, k, out_v.data_ptr(), out_i.data_ptr(),
                                        DeviceGallery.aligned_ptr(ws), ws_bytes,
                                        int(torch.cuda.current_stream(dev).cuda_stream)))
    return out_v, out_i


class _PendingSharded:
    def __init__(self, finish, general):
        self._finish, self._general, self._out = finish, general, None

    def wait(self):
        if self._out is None:
            out = self._finish()
            self._out = out if out is not None else self._general()
        return self._out


class ShardedGallery:
    """This rank's shard of a row-sharded gallery plus the merge step.

    `local` is the rank's DeviceGallery with `row_offset` = first global row.  `local_search` and
    `merge` exist so the host-side protocol (gather layout, index offsets, tie rule) can be
    exercised on CPU with the gloo backend in tests; the product defaults are the CUDA kernels.
    `local_range` / `local_counts` do the same for `best_thresholds`' two local steps:
    `local_range(queries, shard, *, normalize_queries, scale, path, row_filter)` -> int64 [nq, 2] (min, max)
    score keys, and `local_counts(queries, shard, range, *, row_labels, query_labels, n_points, row_filter,
    normalize_queries, scale, path, grid_f32)` -> (thresholds [nq, T] float64, counts [nq, T, 2] int64, n_pos
    [nq] int64) of the shard; the product default is `thresholds.DeviceSweep`.
    `local_range_search(queries, shard, thresholds, **kw)` -> CSR (offsets, values, indices) of the shard with
    global indices is `search_range`'s local step (default: `range_search.search_range`).
    `fused=False` forces the NCCL all-gather variant (also: MMRS_NO_FUSED_GATHER=1).
    """

    def __init__(self, local, n_rows_global: int, group: Optional[dist.ProcessGroup] = None,
                 local_search: Optional[Callable] = None, merge: Optional[Callable] = None,
                 fused: Optional[bool] = None, local_range: Optional[Callable] = None,
                 local_counts: Optional[Callable] = None, local_range_search: Optional[Callable] = None):
        if (local_range is None) != (local_counts is None):
            raise ValueError("local_range and local_counts come together")
        self._local_range, self._local_counts = local_range, local_counts
        self._local_range_search = local_range_search
        self.local = local
        self.n_rows_global = int(n_rows_global)
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self._fast = local_search is None and merge is None   # product path: packed-key pipeline
        self._fused = {}
        import os
        self._fused_ok = os.environ.get("MMRS_NO_FUSED_GATHER", "0") != "1" if fused is None else bool(fused)
        self._fused_used = False
        if local_search is None:
            from .search import search_topk as local_search
        self._search = local_search
        self._merge = merge or _merge_cuda
        # The fused gather needs every rank to contribute exactly k keys per query (one buffer stride and one
        # merge shape for all ranks; a rank that contributed fewer than min(k, its rows) could drop rows of the
        # global top-k), so it is used only when the SHORTEST shard has at least k rows; otherwise the NCCL
        # variant pads short lists with key 0.  One small collective at construction.
        self.min_shard_rows = len(local)
        if self.world > 1:
            sizes = [None] * self.world
            dist.all_gather_object(sizes, len(local), group=group)
            self.min_shard_rows = int(min(sizes))

    @property
    def fused_active(self) -> bool:
        """True once a search of this handle has gone through the fused NVLink gather."""
        return self._fused_used and self._fused_ok

    @classmethod
    def from_full(cls, features: torch.Tensor, mode: Optional[str] = None, device=None,
                  group: Optional[dist.ProcessGroup] = None, **kw) -> "ShardedGallery":
        """Every rank is handed the full host matrix and keeps only its block."""
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        lo, hi = shard_bounds(features.shape[0], world)[rank]
        local = DeviceGallery(features[lo:hi], mode=mode, device=device, row_offset=lo)
        return cls(local, features.shape[0], group, **kw)

    # ---- per-slot buffers ---------------------------------------------------------------------------------
    def _stage_queries(self, slot, queries):
        """fp32 [Q, padded_dim] queries on the device, in a buffer the slot owns (so the library's graph
        of this slot keeps its query pointer); host queries are copied asynchronously."""
        from .search import _prep_queries
        gal = self.local
        q, on_host = _prep_queries(queries, gal)
        if not on_host:
            return q, False, None
        qd = slot.extra.get("q_dev")
        if qd is None or qd.shape != q.shape:
            qd = slot.extra["q_dev"] = torch.empty(q.shape, dtype=torch.float32, device=gal.device)
        if not q.is_pinned():
            q = q.pin_memory()
        qd.copy_(q, non_blocking=True)
        return qd, True, q

    @staticmethod
    def _results(slot, nq, k, dev, on_host, out):
        """(device result tensors the kernels write, host tensors handed back or None)."""
        if on_host:
            dv = slot.extra.get("out_v")
            if dv is None or dv.shape != (nq, k):
                dv = slot.extra["out_v"] = torch.empty((nq, k), dtype=torch.float32, device=dev)
                slot.extra["out_i"] = torch.empty((nq, k), dtype=torch.int64, device=dev)
            di = slot.extra["out_i"]
            if out is not None:
                hv, hi = out
            else:
                hv = torch.empty((nq, k), dtype=torch.float32, pin_memory=True)
                hi = torch.empty((nq, k), dtype=torch.int64, pin_memory=True)
            return dv, di, hv, hi
        if out is not None:
            return out[0], out[1], None, None
        return (torch.empty((nq, k), dtype=torch.float32, device=dev),
                torch.empty((nq, k), dtype=torch.int64, device=dev), None, None)

    def _search_topk_keys(self, queries, k: int, normalize_queries: bool, scale: float, path: str, out=None,
                          local_filter: Optional[RowFilter] = None, labels=None):
        """CUDA fast path: local top-k as packed 64-bit keys -> ONE all-gather (Q*k*8 bytes per rank)
        -> merge kernel reading the gathered buffer in place.  Nothing synchronises with the host
        until the final status check.  Shards shorter than k pad their lists with key 0, and so does a
        shard with fewer than k allowed rows (the library pads them)."""
        gal = self.local
        dev = gal.device
        lib = _cabi.lib
        if torch.cuda.current_device() != dev.index:
            torch.cuda.set_device(dev)
        stream = torch.cuda.current_stream(dev)
        nq = int(queries.shape[0]) if hasattr(queries, "shape") and len(queries.shape) == 2 else 1
        k_local = min(k, gal.n_rows)
        slot = gal.search_slot(nq, k_local, False, stream.cuda_stream)
        q, on_host, keep = self._stage_queries(slot, queries)
        n_keys = nq * k
        bufs = slot.extra.get(("keys", k))
        if bufs is None:
            bufs = slot.extra[("keys", k)] = (
                torch.zeros(n_keys + 1, dtype=torch.int64, device=dev),                # key 0 = "no entry"; [-1] = status
                torch.zeros(nq * k_local + 1, dtype=torch.int64, device=dev) if k_local != k else None,
                torch.empty((self.world, n_keys + 1), dtype=torch.int64, device=dev),
                torch.empty(1, dtype=torch.int32, device=dev))
        buf, short, gathered, d_status = bufs
        dv, di, hv, hi = self._results(slot, nq, k, dev, on_host, out)
        ticket, status, event = slot.acquire()
        shard_status = None
        staged = None
        if labels is not None:
            from .search import _stage_query_labels
            staged = _stage_query_labels(slot, labels[1], dev)
        if nq:
            dst = buf if short is None else short
            args = (gal.data.data_ptr(), gal.n_rows, gal.padded_dim, gal.data.stride(0), gal.dtype_code,
                    q.data_ptr(), nq, q.stride(0), k_local, int(bool(normalize_queries)), float(scale),
                    gal.row_offset, _cabi.PATHS[path], dst.data_ptr(), slot.ptr, slot.nbytes, status.data_ptr())
            filt_ptr = local_filter.words.data_ptr() if local_filter is not None else 0
            if labels is not None:   # a query with fewer than k eligible rows here: its list is padded with key 0
                st = lib.mmrs_search_topk_keys_async_labeled(*args, filt_ptr, labels[0].labels.data_ptr(),
                                                             staged[0].data_ptr(), labels[2], stream.cuda_stream)
            elif local_filter is None:
                st = lib.mmrs_search_topk_keys_async(*args, stream.cuda_stream)
            else:
                st = lib.mmrs_search_topk_keys_async_filtered(*args, local_filter.words.data_ptr(), stream.cuda_stream)
            if st != _cabi.OK:
                slot.release(ticket)
                _cabi.check(st)
            if short is not None:                       # a shard shorter than k: the rest of its lists stays key 0
                buf[:n_keys].view(nq, k)[:, :k_local] = short[:-1].view(nq, k_local)
                buf[-1] = short[-1]
        dist.all_gather_into_tensor(gathered.view(-1), buf, group=self.group)      # [world, nq*k + 1]
        if nq:
            # labeled: fewer than k eligible rows over all ranks is legitimate -> -inf / -1
            merge = lib.mmrs_topk_merge_keys_padded_async if labels is not None else lib.mmrs_topk_merge_keys_async
            _cabi.check(merge(gathered.data_ptr(), self.world, nq, k, n_keys + 1, k, dv.data_ptr(), di.data_ptr(),
                              d_status.data_ptr(), status[1:].data_ptr(), stream.cuda_stream))
            table = slot.extra.get("shard_status")          # one pinned row per status ticket of the slot
            if table is None or table.shape[0] <= ticket:
                table = slot.extra["shard_status"] = torch.zeros((max(ticket + 1, slot.N_STATUS), self.world),
                                                                 dtype=torch.int64).pin_memory()
            shard_status = table[ticket]
            shard_status.copy_(gathered[:, -1], non_blocking=True)
        if on_host:
            hv.copy_(dv, non_blocking=True)
            hi.copy_(di, non_blocking=True)
        event.record(stream)

        def finish():
            event.synchronize()
            res = (hv, hi) if on_host else (dv, di)
            if shard_status is None:
                slot.release(ticket)
                return res
            worst = int(shard_status.max().item())
            merge_rc = lib.mmrs_search_status(status[1:].data_ptr())
            if worst not in (0, 1):                  # e.g. a zero-norm query: same error as single-GPU
                status[0] = worst
            own_rc = lib.mmrs_search_status(status.data_ptr()) if worst not in (0, 1) else _cabi.OK
            slot.release(ticket)
            if worst == 1:
                return None                          # some rank overflowed: ALL ranks take the general path
            _cabi.check(own_rc)
            _cabi.check(merge_rc)
            return res

        finish._keepalive = (q, keep, local_filter, labels, staged)
        return finish

    # ---- search fused with its all-gather over NVLink peer memory -----------------------------------
    def _fused_state(self, slot, nq: int, k_local: int):
        """Symmetric (peer-mapped) gather buffer + flag array of one (shape, stream) slot; the
        rendezvous is collective and happens once per slot."""
        st = slot.extra.get("fused")
        if st is None:
            import torch.distributed._symmetric_memory as symm_mem
            dev = self.local.device
            stride = nq * k_local + 1                       # one list + the rank's status word
            total = self.world * stride + self.world         # + 2 * world uint32 flags
            t = symm_mem.empty(total, dtype=torch.int64, device=dev)
            t.zero_()
            hdl = symm_mem.rendezvous(t, self.group if self.group is not None else dist.group.WORLD)
            torch.cuda.synchronize(dev)
            dist.barrier(group=self.group)                   # everyone zeroed before anyone stores
            ptrs = [int(x) for x in hdl.buffer_ptrs]
            flag_off = self.world * stride * 8
            st = {"t": t, "hdl": hdl, "stride": stride,
                  "bufs": torch.tensor(ptrs, dtype=torch.int64, device=dev),
                  "flags": torch.tensor([x + flag_off for x in ptrs], dtype=torch.int64, device=dev),
                  "local_flags": t.data_ptr() + flag_off}
            slot.extra["fused"] = st
        return st

    def _search_topk_fused(self, queries, k: int, normalize_queries: bool, scale: float, path: str, out=None,
                           local_filter: Optional[RowFilter] = None, labels=None):
        """Local scan -> last select stores its keys into EVERY rank's buffer over NVLink and raises
        a ready flag -> a one-warp kernel waits for all flags -> merge select.  One library call, one
        graph replay, no NCCL, no host sync until the final status check; every buffer the call
        touches belongs to the (shape, stream) slot and was allocated once."""
        gal = self.local
        dev = gal.device
        lib = _cabi.lib
        if torch.cuda.current_device() != dev.index:
            torch.cuda.set_device(dev)
        stream = torch.cuda.current_stream(dev)
        nq = int(queries.shape[0])
        k_local = k                                      # every shard has >= k rows (checked by search_topk)
        slot = gal.search_slot(nq, k_local, False, stream.cuda_stream)
        st = self._fused_state(slot, nq, k_local)         # collective on first use of the slot
        q, on_host, keep = self._stage_queries(slot, queries)
        dv, di, hv, hi = self._results(slot, nq, k, dev, on_host, out)
        staged = None
        if labels is not None:
            from .search import _stage_query_labels
            staged = _stage_query_labels(slot, labels[1], dev)
        ticket, status, event = slot.acquire()
        args = (gal.data.data_ptr(), gal.n_rows, gal.padded_dim, gal.data.stride(0), gal.dtype_code,
                q.data_ptr(), nq, q.stride(0), k_local, k, int(bool(normalize_queries)), float(scale),
                gal.row_offset, _cabi.PATHS[path], st["bufs"].data_ptr(), st["flags"].data_ptr(),
                st["t"].data_ptr(), st["local_flags"], self.rank, self.world, st["stride"],
                dv.data_ptr(), di.data_ptr(), slot.ptr, slot.nbytes, status.data_ptr())
        if labels is not None:   # the merge select pads queries with fewer than k eligible rows with -inf / -1
            rc = lib.mmrs_search_topk_fused_gather_async_labeled(
                *args, local_filter.words.data_ptr() if local_filter is not None else 0, labels[0].labels.data_ptr(),
                staged[0].data_ptr(), labels[2], stream.cuda_stream)
        elif local_filter is None:
            rc = lib.mmrs_search_topk_fused_gather_async(*args, stream.cuda_stream)
        else:   # a shard with fewer than k allowed rows still stores k keys (padded with key 0)
            rc = lib.mmrs_search_topk_fused_gather_async_filtered(*args, local_filter.words.data_ptr(), stream.cuda_stream)
        if rc != _cabi.OK:
            slot.release(ticket)
            _cabi.check(rc)
        if on_host:
            hv.copy_(dv, non_blocking=True)
            hi.copy_(di, non_blocking=True)
        event.record(stream)
        self._fused_used = True

        def finish():
            event.synchronize()
            rc = lib.mmrs_gather_status(status.data_ptr(), self.world)
            slot.release(ticket)
            if rc == _cabi.ERR_RETRY:
                return None                  # the same verdict on every rank: all take the general path
            if rc == _cabi.ERR_TIMEOUT:
                self._fused_ok = False       # a peer is dead or diverged: later calls use NCCL (its own abort handling)
            _cabi.check(rc)
            return (hv, hi) if on_host else (dv, di)

        finish._keepalive = (q, keep, local_filter, labels, staged)
        return finish

    def _local_filter(self, row_filter):
        """(filter over the GLOBAL rows as a RowFilter -- a bool mask is packed here --, this rank's slice of it)."""
        dev = getattr(self.local, "device", None)
        f = row_filter if isinstance(row_filter, RowFilter) else RowFilter(row_filter, device=dev)
        if f.n_rows != self.n_rows_global:
            raise ValueError(f"row_filter covers {f.n_rows} rows, the sharded gallery has {self.n_rows_global}")
        if dev is not None and f.device != dev:
            raise ValueError(f"row_filter is on {f.device}, this rank's shard on {dev}")
        lo = self.local.row_offset
        return f, f.shard(lo, lo + len(self.local))

    def _local_labels(self, row_labels, query_labels, label_match, queries):
        """(RowLabels over this rank's rows -- a view of the global one --, query labels as given, label_match
        code), or None when unlabeled.  Checked alike on every rank, before any collective."""
        if row_labels is None and query_labels is None:
            label_match_arg(label_match)
            return None
        if row_labels is None or query_labels is None:
            raise ValueError("row_labels and query_labels come together")
        match = label_match_arg(label_match)
        if not isinstance(row_labels, RowLabels):
            raise ValueError(f"row_labels must be a RowLabels, got {type(row_labels).__name__}")
        if row_labels.n_rows != self.n_rows_global:
            raise ValueError(f"row_labels covers {row_labels.n_rows} rows, the sharded gallery has {self.n_rows_global}")
        dev = getattr(self.local, "device", None)
        if dev is not None and row_labels.device != dev:
            raise ValueError(f"row_labels is on {row_labels.device}, this rank's shard on {dev}")
        nq = 1 if len(queries.shape) == 1 else int(queries.shape[0])
        ql = query_labels_arg(query_labels, nq, dev)
        lo = self.local.row_offset
        return row_labels.shard(lo, lo + len(self.local)), ql, match

    def search_topk(self, queries: torch.Tensor, k: int, *, normalize_queries: bool = True,
                    scale: float = 1.0, path: str = "auto", sync: bool = True, out=None, row_filter=None,
                    row_labels=None, query_labels=None, label_match: str = "same"):
        """Global top-k, identical on every rank.  `queries` must be the same on all ranks.
        `sync=False` returns an object whose `.wait()` yields `(values, indices)`, so that several
        batches (and their all-gathers) can be in flight.  `out=(values, indices)`: caller-owned result
        tensors (pinned host tensors for host queries).  `row_filter`: a RowFilter (or bool mask) over the
        GLOBAL rows, the same on every rank like the queries; each rank searches its slice of it.
        `row_labels` (a RowLabels over the GLOBAL rows) / `query_labels` / `label_match`: label-conditioned
        search as in `search_topk`, the same on every rank (query labels replicated like the queries); a
        query with fewer than k eligible rows over all shards is padded with -inf / -1."""
        if k > self.n_rows_global:
            raise RuntimeError("selected index k out of range")
        if isinstance(queries, np.ndarray):
            queries = torch.from_numpy(queries)
        labels = self._local_labels(row_labels, query_labels, label_match, queries)
        lab_kw = dict(row_labels=row_labels, query_labels=query_labels, label_match=label_match)
        local_filter = None
        if row_filter is not None:
            row_filter, local_filter = self._local_filter(row_filter)
            if k > row_filter.n_allowed:      # every rank decides alike from the same filter: no collective
                raise RuntimeError("selected index k out of range")
        if self._fast and self.world > 1:
            if isinstance(queries, np.ndarray):
                queries = torch.from_numpy(queries)
            if queries.dim() == 1:
                queries = queries.unsqueeze(0)
            nq = int(queries.shape[0])
            if nq == 0:
                out_t = self.search_topk_general(queries, k, normalize_queries=normalize_queries, scale=scale, path=path,
                                                 row_filter=row_filter, **lab_kw)
                return out_t if sync else _PendingSharded(lambda: out_t, None)
            # fused NVLink gather: every rank contributes its full top-k (needs >= k rows in every shard)
            fused = self._fused_ok and 1 <= nq <= 1024 and self.min_shard_rows >= k
            finish = None
            if fused:
                try:
                    finish = self._search_topk_fused(queries, k, normalize_queries, scale, path, out, local_filter, labels)
                except (ImportError, AttributeError, RuntimeError) as e:   # no symmetric memory here
                    if isinstance(e, _cabi.MmrsError):
                        raise
                    self._fused_ok = False
            if finish is None:
                finish = self._search_topk_keys(queries, k, normalize_queries, scale, path, out, local_filter, labels)
            general = lambda: self.search_topk_general(queries, k, normalize_queries=normalize_queries,
                                                       scale=scale, path=path, row_filter=row_filter, **lab_kw)
            pend = _PendingSharded(finish, general)
            return pend.wait() if sync else pend
        out_t = self.search_topk_general(queries, k, normalize_queries=normalize_queries, scale=scale, path=path,
                                         row_filter=row_filter, **lab_kw)
        return out_t if sync else _PendingSharded(lambda: out_t, None)

    def search_topk_general(self, queries: torch.Tensor, k: int, *, normalize_queries: bool = True,
                            scale: float = 1.0, path: str = "auto", row_filter=None, row_labels=None,
                            query_labels=None, label_match: str = "same"):
        """(values, indices) lists, two all-gathers, merge -- also the path every rank takes together
        when some rank's candidate list overflowed (None from the fast path on EVERY rank alike: the
        shard statuses were gathered with the keys).  With a `row_filter` a rank searches for
        min(k, its allowed rows) and one without allowed rows skips its local search.  Labeled: positions
        that no rank could fill hold -inf / -1, as on one GPU."""
        if isinstance(queries, np.ndarray):
            queries = torch.from_numpy(queries)
        labels = self._local_labels(row_labels, query_labels, label_match, queries)
        n_local = len(self.local)
        k_local = min(k, n_local)
        local_filter = None
        if row_filter is not None:
            row_filter, local_filter = self._local_filter(row_filter)
            if k > row_filter.n_allowed:
                raise RuntimeError("selected index k out of range")
            k_local = min(k, local_filter.n_allowed)
        on_host = False
        if self._fast and self.world > 1 and not (isinstance(queries, torch.Tensor) and queries.is_cuda):
            on_host = True                    # NCCL gathers device tensors: search on the device, copy back
            queries = torch.as_tensor(queries).to(self.local.device)
        kw = {} if local_filter is None else {"row_filter": local_filter}
        if labels is not None:
            kw.update(row_labels=labels[0], query_labels=labels[1], label_match=label_match)
        if local_filter is None or k_local > 0:
            v, i = self._search(queries, self.local, k_local, normalize_queries=normalize_queries,
                                scale=scale, path=path, **kw)
        else:                                 # no allowed row here: contribute padding only
            nq = 1 if len(queries.shape) == 1 else int(queries.shape[0])
            dev = getattr(self.local, "device", torch.device("cpu"))
            v = torch.empty((nq, 0), dtype=torch.float32, device=dev)
            i = torch.empty((nq, 0), dtype=torch.int64, device=dev)
        if self.world == 1:
            return v, i
        if k_local < k:
            # a shard smaller than k: pad with -inf / sentinel so all ranks gather equal shapes
            pad = k - k_local
            v = torch.cat([v, torch.full((v.shape[0], pad), float("-inf"), dtype=v.dtype, device=v.device)], 1)
            i = torch.cat([i, torch.full((i.shape[0], pad), 2 ** 32 - 1, dtype=i.dtype, device=i.device)], 1)
        if labels is not None:
            # labeled, a query may have fewer than k eligible rows over ALL ranks, so padding can reach the
            # merged result: every padded position (the local search's -1, the sentinel above) gets its own
            # sentinel 2^32 - 1 - (rank * k + position), so that the merge sees unique keys, and the merged
            # -inf positions become the public -1
            pad = (i < 0) | (i == 2 ** 32 - 1)
            sentinel = 2 ** 32 - 1 - (self.rank * k + torch.arange(k, dtype=i.dtype, device=i.device))
            i = torch.where(pad, sentinel.expand_as(i), i)
        gv = _all_gather(v, self.world, self.group)
        gi = _all_gather(i, self.world, self.group)
        mv, mi = self._merge(gv, gi, k)
        if labels is not None:
            mi = torch.where(mv == float("-inf"), torch.full_like(mi, -1), mi)
        return (mv.cpu(), mi.cpu()) if on_host else (mv, mi)

    def best_thresholds(self, queries, row_labels, query_labels, *, n_points: int = 200, scale: float = 100.0,
                        normalize_queries: bool = False, row_filter=None, path: str = "auto",
                        max_score_bytes: int = 4 << 30):
        """`best_thresholds` over the sharded gallery, the same arrays on every rank.  `queries`, `query_labels`,
        `row_labels` and `row_filter` are the same on every rank, the last two over the GLOBAL rows.  Per chunk
        of queries each rank scores its shard and takes the range of its allowed rows; one all-reduce gives the
        global (min, max) of every query, so every rank builds the same grid; each rank counts its rows against
        it and one all-reduce sums the counts.  The chunk size comes from the longest shard of
        `shard_bounds(n_rows_global, world)`, which every rank knows: all ranks run the same collectives."""
        from .search import grid_f32
        from .thresholds import (DeviceSweep, check_arguments, check_row_labels, chunk_queries, empty_result,
                                 run_chunks)
        if isinstance(queries, np.ndarray):
            queries = torch.from_numpy(queries)
        if queries.dim() == 1:
            queries = queries.unsqueeze(0)
        c = int(queries.shape[0])
        dev = getattr(self.local, "device", None)
        check_row_labels(row_labels, self.n_rows_global, dev)
        ql = check_arguments(c, query_labels, n_points, dev)
        local_filter = None
        if row_filter is not None:
            row_filter, local_filter = self._local_filter(row_filter)
            if row_filter.n_allowed == 0:
                raise ValueError("row_filter allows no row")
        if c == 0:
            return empty_result(int(n_points))
        lo = self.local.row_offset
        local_labels = row_labels.shard(lo, lo + len(self.local))
        longest = max(hi - lo_ for lo_, hi in shard_bounds(self.n_rows_global, self.world))
        qc = min(c, chunk_queries(longest, max_score_bytes))
        n_points = int(n_points)
        kw = dict(normalize_queries=normalize_queries, scale=scale, path=path)
        if self._local_range is None:
            sweep = DeviceSweep(self.local, qc, n_points, normalize_queries, scale, path, local_labels, local_filter,
                                grid_f32())
            range_step = sweep.range
            count_step = lambda q, lab, rng: sweep.counts(lab, rng)
        else:
            range_step = lambda q: self._local_range(q, self.local, row_filter=local_filter, **kw)
            count_step = lambda q, lab, rng: self._local_counts(q, self.local, rng, row_labels=local_labels,
                                                                query_labels=lab, n_points=n_points,
                                                                row_filter=local_filter, grid_f32=grid_f32(), **kw)
        if self.world == 1:
            return run_chunks(queries, ql, qc, n_points, range_step, count_step)

        def reduce_range(rng):
            # MIN of the min keys and MAX of the max keys in ONE exact int64 all-reduce: MIN of the negated max keys
            t = torch.stack([rng[:, 0], -rng[:, 1]], 1).contiguous()
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.group)
            return torch.stack([t[:, 0], -t[:, 1]], 1)

        def reduce_counts(counts, n_pos):
            flat = torch.cat([counts.reshape(-1), n_pos.reshape(-1)])
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
            return flat[:counts.numel()].view(counts.shape), flat[counts.numel():]

        return run_chunks(queries, ql, qc, n_points, range_step, count_step, reduce_range, reduce_counts)

    def search_range(self, queries, thresholds, *, normalize_queries: bool = True, scale: float = 1.0,
                     path: str = "auto", row_filter=None, row_labels=None, query_labels=None, label_match: str = "same",
                     max_candidate_bytes: int = 4 << 30):
        """`search_range` over the sharded gallery: the same CSR (offsets, values, indices) on every rank, equal
        to the single-GPU call on the full gallery.  `queries`, `thresholds`, `query_labels`, `row_labels` and
        `row_filter` are the same on every rank, the last two over the GLOBAL rows.  Each rank range-searches
        its shard; one all-gather moves the per-query counts [world, Q], a second the values and indices
        (padded to the largest total); the pieces are joined per query in rank order, which is row order
        because shards are ascending row blocks."""
        from .range_search import concat_per_query, search_range, thresholds_f32
        if isinstance(queries, np.ndarray):
            queries = torch.from_numpy(queries)
        if queries.dim() == 1:
            queries = queries.unsqueeze(0)
        nq = int(queries.shape[0])
        thr = thresholds_f32(thresholds, nq)      # a NaN threshold raises on every rank alike
        labels = self._local_labels(row_labels, query_labels, label_match, queries)
        kw = dict(normalize_queries=normalize_queries, scale=scale, path=path, max_candidate_bytes=max_candidate_bytes)
        if row_filter is not None:
            kw["row_filter"] = self._local_filter(row_filter)[1]
        if labels is not None:
            kw.update(row_labels=labels[0], query_labels=labels[1], label_match=label_match)
        local = self._local_range_search or search_range
        on_host = not queries.is_cuda
        if self._local_range_search is None and self.world > 1 and on_host:
            queries = queries.to(self.local.device)       # NCCL gathers device tensors: search there, copy back
        off, v, i = local(queries, self.local, thr, **kw)
        if self.world == 1:
            return off, v, i
        counts = _all_gather(off[1:] - off[:-1], self.world, self.group)          # [world, Q]
        totals = counts.sum(1)
        m = max(1, int(totals.max().item()))
        bufs = []
        for x in (v, i):
            b = torch.zeros(m, dtype=x.dtype, device=x.device)
            b[:x.numel()] = x
            bufs.append(_all_gather(b, self.world, self.group))
        pieces = []
        for r in range(self.world):
            o = torch.zeros(nq + 1, dtype=torch.int64, device=counts.device)
            torch.cumsum(counts[r], 0, out=o[1:])
            n_r = int(totals[r].item())
            pieces.append((o, bufs[0][r, :n_r], bufs[1][r, :n_r]))
        out = concat_per_query(pieces)
        return tuple(x.cpu() for x in out) if on_host and self._local_range_search is None else out

    def find_duplicate_pairs(self, emb_full: torch.Tensor, threshold: float, raw_join: Optional[Callable] = None):
        """Self-join with the gallery replicated (10M x 512 fp32 = 20 GB fits every GPU) and the
        upper-triangular tile grid split by equal pair count; variable-length pair lists are
        gathered (counts first, then padded buffers) and sorted lexicographically."""
        from .dedup import selfjoin_tc_raw, sort_pairs
        n = int(emb_full.shape[0])
        if raw_join is None and emb_full.is_cuda and n >= 2048:
            # tensor-core path: column panels dealt round-robin to the ranks
            pairs = selfjoin_tc_raw(emb_full, threshold, self.rank, self.world)
        else:
            from .dedup import selfjoin_raw
            raw_join = raw_join or selfjoin_raw
            lo, hi = triangle_bounds(n, self.world)[self.rank]
            pairs = raw_join(emb_full, threshold, lo, hi) if hi > lo else emb_full.new_empty((0, 2), dtype=torch.int64)
        if self.world == 1:
            return sort_pairs(pairs, n)
        cnt = torch.tensor([pairs.shape[0]], dtype=torch.int64, device=pairs.device)
        cnts = _all_gather(cnt, self.world, self.group).view(-1)
        m = int(cnts.max().item())
        buf = torch.zeros((max(m, 1), 2), dtype=torch.int64, device=pairs.device)
        buf[:pairs.shape[0]] = pairs
        allbuf = _all_gather(buf, self.world, self.group)
        parts = [allbuf[r, :int(cnts[r].item())] for r in range(self.world)]
        return sort_pairs(torch.cat(parts, dim=0), n)

    def deduplicate(self, emb_full: torch.Tensor, threshold: float, *, order=None,
                    raw_join: Optional[Callable] = None) -> torch.Tensor:
        """`deduplicate` over the ranks: the pairs of `find_duplicate_pairs` (every rank holds the whole
        gathered list), then `resolve_duplicates` on each rank.  The resolve is deterministic, so every rank
        returns the same [n] representative tensor without another collective."""
        from .dedup import resolve_duplicates
        pairs = self.find_duplicate_pairs(emb_full, threshold, raw_join=raw_join)
        return resolve_duplicates(pairs, int(emb_full.shape[0]), order=order)
