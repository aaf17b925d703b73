"""Device-resident gallery (SURVEY.md section 8, row f1).

The reference keeps its gallery as a pickle `{relpath: float[D]}` (code/search_image.py:159-164),
rebuilds an `np.array` -> `torch.tensor [N, D]` per class (`construct_dataset`, :167-182) and
uploads the WHOLE matrix on every score call (`features.cuda()`, :107).  Here the matrix is
uploaded once into HBM, row-major, rows 16-byte aligned (D padded with zeros to a multiple of 8),
in fp32 (exact mode), bf16 (tensor-core mode) or per-row-scaled int8 (compact mode), and stays resident
across calls.
"""
from __future__ import annotations

import pickle
from typing import Optional, Sequence

import numpy as np
import torch

from . import _cabi


def _pad_dim(d: int) -> int:
    return (d + 7) // 8 * 8


def _pad_dim_i8(d: int) -> int:
    return (d + 15) // 16 * 16


class DeviceGallery:
    """[N, D] embedding matrix resident on one B200.

    mode "fp32": values kept as given (exact mode: scores within 1e-5 of the torch CPU path).
    mode "bf16": values rounded to bf16 -- that bf16 tensor IS the gallery (BASELINE.md section 5).
    mode "int8": each row quantised on the device to int8 codes with one fp32 scale (include/mmrs_b200.h,
    "int8 galleries"): `data` is int8 [N, padded_dim + 16], codes [padded_dim] (padded_dim = D rounded up to
    16) then the scale's 16-byte tail -- 784 bytes per row at D = 768 instead of 1536.  Scores are an exact
    function of the codes; a row holding a NaN or an infinity raises ValueError.  Never chosen by default.
    `row_offset` is the global index of row 0 when this is one shard of a larger gallery.
    """

    def __init__(self, features, mode: Optional[str] = None, device: Optional[torch.device] = None,
                 row_offset: int = 0, paths: Optional[Sequence[str]] = None):
        if isinstance(features, np.ndarray):
            features = torch.from_numpy(features)
        if not isinstance(features, torch.Tensor) or features.dim() != 2:
            raise TypeError("features must be a 2-D torch.Tensor / numpy array [N, D]")
        if mode is None:
            mode = "bf16" if features.dtype == torch.bfloat16 else "fp32"
        if mode not in ("fp32", "bf16", "int8"):
            raise ValueError("mode must be 'fp32', 'bf16' or 'int8'")
        if device is None:
            device = features.device if features.is_cuda else torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)
        device = torch.device(device)
        _cabi.require_b200(device.index if device.index is not None else 0)
        self.mode = mode
        self.device = device
        self.n_rows, self.dim = int(features.shape[0]), int(features.shape[1])
        if self.n_rows < 1 or self.dim < 1:
            raise ValueError("gallery must have at least one row and one column")
        self.row_offset = int(row_offset)
        self.paths = list(paths) if paths is not None else None
        self._workspaces: dict = {}
        self._split = None
        if mode == "int8":
            self.padded_dim = _pad_dim_i8(self.dim)
            self.data = self._quantize(features.detach(), device)
            return
        dt = torch.bfloat16 if mode == "bf16" else torch.float32
        dp = _pad_dim(self.dim)
        src = features.detach()
        if src.is_cuda and src.dtype == dt and dp == self.dim and src.is_contiguous():
            data = src  # adopt in place (no copy): e.g. a shard generated on the device
        else:
            data = torch.zeros((self.n_rows, dp), dtype=dt, device=device)
            # chunked upload keeps the pinned/pageable staging small for multi-GB galleries
            step = max(1, (256 << 20) // max(1, self.dim * 4))
            for lo in range(0, self.n_rows, step):
                blk = src[lo:lo + step]
                data[lo:lo + step, :self.dim] = blk.to(device=device, dtype=dt, non_blocking=False)
        self.data = data
        self.padded_dim = dp
        self._workspaces: dict = {}
        self._split = None

    def _quantize(self, src: torch.Tensor, device: torch.device) -> torch.Tensor:
        """int8 rows [N, padded_dim + 16] quantised on the device (mmrs_quantize_rows_i8); host input goes up
        in fp32 (bf16 input as bf16) chunks of at most 256 MB."""
        data = torch.empty((self.n_rows, self.padded_dim + 16), dtype=torch.int8, device=device)
        sdt = torch.bfloat16 if src.dtype == torch.bfloat16 else torch.float32
        code = _cabi.DTYPE_BF16 if sdt == torch.bfloat16 else _cabi.DTYPE_F32
        step = max(1, (256 << 20) // max(1, self.dim * 4))
        with torch.cuda.device(device):
            stream = int(torch.cuda.current_stream(device).cuda_stream)
            for lo in range(0, self.n_rows, step):
                blk = src[lo:lo + step].to(device=device, dtype=sdt)
                if blk.stride(1) != 1:
                    blk = blk.contiguous()
                _cabi.check(_cabi.lib.mmrs_quantize_rows_i8(blk.data_ptr(), code, blk.shape[0], self.dim, blk.stride(0),
                                                            data[lo].data_ptr(), data.stride(0), stream))
        return data

    # -- C-ABI views ---------------------------------------------------------------------------
    @property
    def dtype_code(self) -> int:
        if self.mode == "int8":
            return _cabi.DTYPE_I8
        return _cabi.DTYPE_BF16 if self.mode == "bf16" else _cabi.DTYPE_F32

    def int8_codes_scales(self):
        """int8 mode: (codes int8 [N, D], scales fp32 [N]) -- views of the resident rows."""
        if self.mode != "int8":
            raise ValueError("codes and scales exist for int8 galleries only")
        scales = self.data[:, self.padded_dim:self.padded_dim + 4].contiguous().view(torch.float32).reshape(-1)
        return self.data[:, :self.dim], scales

    @property
    def nbytes(self) -> int:
        return self.data.numel() * self.data.element_size()

    def workspace(self, key, nbytes: int) -> torch.Tensor:
        """Cached device scratch buffer (256-byte aligned) for repeated calls of one shape."""
        buf = self._workspaces.get(key)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(int(nbytes), 256) + 256, dtype=torch.uint8, device=self.device)
            self._workspaces[key] = buf
        return buf

    MAX_SEARCH_SLOTS = 32      # LRU cap on cached search slots (a service with ever-changing batch sizes)

    def search_slot(self, nq: int, k: int, host_io: bool, stream_id: int = 0) -> "SearchSlot":
        """The slot of one search shape on one stream: device workspace (sized by the library's own
        query, zero-filled once), pinned status words and events -- everything a steady-state call
        needs, so that it allocates nothing.  One per stream: searches in flight on different
        streams must not share candidate lists.  The library's CUDA-graph cache is keyed on the
        slot's workspace, so one slot == one captured graph.  At most MAX_SEARCH_SLOTS are kept
        (least recently used first out; the exhaustive fallback's 8-bytes-per-row buffer is NOT part
        of a slot, it is allocated for the rare call that needs it)."""
        key = ("search", nq, k, host_io, stream_id)
        slot = self._workspaces.pop(key, None)
        if slot is None:
            slots = [kk for kk in self._workspaces if isinstance(kk, tuple) and kk and kk[0] == "search"]
            if len(slots) >= self.MAX_SEARCH_SLOTS:
                torch.cuda.synchronize(self.device)       # the victim may still be in flight
                del self._workspaces[slots[0]]            # dicts keep insertion order: [0] is the LRU
            slot = SearchSlot(self, nq, k, host_io)
        self._workspaces[key] = slot                      # (re)insert as most recently used
        return slot

    def search_workspace(self, nq: int, k: int, host_io: bool, stream_id: int = 0):
        """(aligned device pointer, byte size) of the slot's workspace."""
        slot = self.search_slot(nq, k, host_io, stream_id)
        return slot.ptr, slot.nbytes

    @staticmethod
    def aligned_ptr(buf: torch.Tensor) -> int:
        p = buf.data_ptr()
        return (p + 255) // 256 * 256

    def split3(self) -> torch.Tensor:
        """fp32 mode only: the gallery as three bf16 planes [3, N, Dp] with x == hi + mid + lo, built
        once on first use (mmrs_split_bf16x3).  Larger fp32 batches are searched from these planes on
        the tensor cores (six bf16 MMAs per tile, fp32-grade scores) instead of K1's CUDA-core passes."""
        if self.mode != "fp32":
            raise ValueError("split planes exist for fp32 galleries only")
        if self._split is None:
            planes = torch.empty((3, self.n_rows, self.padded_dim), dtype=torch.bfloat16, device=self.device)
            with torch.cuda.device(self.device):
                _cabi.check(_cabi.lib.mmrs_split_bf16x3(self.data.data_ptr(), self.n_rows, self.padded_dim,
                                                        self.data.stride(0), planes.data_ptr(), self.padded_dim,
                                                        int(torch.cuda.current_stream(self.device).cuda_stream)))
            self._split = planes
        return self._split

    def lookup_paths(self, indices):
        """Relative paths (the keys of the reference's feature pickle, search_image.py:157) of the
        rows a search returned; `indices` are global ids (row_offset already added)."""
        if self.paths is None:
            raise ValueError("this gallery was built without a path table")
        idx = indices.detach().cpu().numpy() if isinstance(indices, torch.Tensor) else np.asarray(indices)
        flat = [self.paths[int(i) - self.row_offset] for i in idx.reshape(-1)]
        return np.array(flat, dtype=object).reshape(idx.shape).tolist()

    @classmethod
    def from_feature_cache(cls, path: str, mode: Optional[str] = None, device=None) -> "DeviceGallery":
        """Resident gallery straight from the reference's cache file (pickle dict or .pt tensor)."""
        feats, keys = load_feature_cache(path)
        return cls(feats, mode=mode, device=device, paths=keys)

    def __len__(self) -> int:
        return self.n_rows

    def __repr__(self) -> str:
        return (f"DeviceGallery(rows={self.n_rows}, dim={self.dim}, mode={self.mode}, "
                f"device={self.device}, row_offset={self.row_offset})")


class SearchSlot:
    """Buffers owned by one (gallery, n_queries, k, host_io, stream) search slot."""
    N_STATUS = 16          # status words handed out round-robin to the batches in flight on the slot
    STATUS_WORDS = 80      # int32 per status record (the fused gather reports world + 2 <= 66 words)

    def __init__(self, gal: "DeviceGallery", nq: int, k: int, host_io: bool):
        lib = _cabi.lib
        nbytes = lib.mmrs_search_workspace_bytes(gal.n_rows, gal.padded_dim, gal.dtype_code, max(nq, 1), k)
        if host_io:
            nbytes += lib.mmrs_search_host_staging_bytes(gal.padded_dim, max(nq, 1), k)
        self.buf = torch.zeros(int(nbytes) + 256, dtype=torch.uint8, device=gal.device)
        self.ptr = DeviceGallery.aligned_ptr(self.buf)
        self.nbytes = int(nbytes)
        self.device = gal.device
        self._status = torch.zeros((self.N_STATUS, self.STATUS_WORDS), dtype=torch.int32).pin_memory()
        self._events = [torch.cuda.Event() for _ in range(self.N_STATUS)]
        self._free = list(range(self.N_STATUS))
        self.extra: dict = {}      # callers' per-slot state (e.g. the sharded search's device staging)

    def acquire(self):
        """-> (ticket, pinned status tensor [STATUS_WORDS] int32, event) for one batch in flight."""
        if not self._free:         # every record is held by an unfinished (or dropped) handle: grow
            n = self._status.shape[0]
            self._status = torch.cat([self._status, torch.zeros_like(self._status)]).pin_memory()
            self._events += [torch.cuda.Event() for _ in range(n)]
            self._free = list(range(n, 2 * n))
            self._grown = True
        t = self._free.pop()
        return t, self._status[t], self._events[t]

    def release(self, ticket: int) -> None:
        self._free.append(ticket)


def load_feature_cache(path: str):
    """Read the reference's on-disk gallery formats.

    *.pkl : pickle `{relpath: np.ndarray[D]}` written by build_cache (code/search_image.py:159-160)
            -> (features [N, D] fp32 tensor, [relpath]) in the dict's insertion order
    *.pt  : `torch.save` of an [N, D] tensor (pre_load_features, code/utils.py:150-151) -> (tensor, None)
    """
    if path.endswith(".pt"):
        t = torch.load(path, map_location="cpu")
        return t.to(torch.float32), None
    with open(path, "rb") as f:
        d = pickle.load(f)
    keys = list(d.keys())
    feats = torch.from_numpy(np.stack([np.asarray(d[k], dtype=np.float32).reshape(-1) for k in keys]))
    return feats, keys
