"""Refined top-k search (DESIGN.md section 4, "Refined search").

A compact gallery (bf16, int8) gives approximate scores.  `search_topk(..., refine=store, refine_k=...)` scans it
for `refine_k` candidates per query and rescores only those against a full-precision copy of the rows, a
`RefineStore`, keeping the k best.  The store is read at `Q * refine_k` rows per call, so it can stay in host
memory: an fp32 copy of a gallery that fits no GPU still gives fp32-grade answers at the compact scan's speed.
"""
from __future__ import annotations

import ctypes
import weakref
from typing import Optional

import numpy as np
import torch

from . import _cabi
from .gallery import DeviceGallery, _pad_dim

MAX_CANDIDATES = 1024      # candidates per query: the largest k a candidate search returns
_PAGE = 4096


def default_refine_k(k: int) -> int:
    """The candidate count `search_topk` scans for when `refine_k` is not given: 2 k, at most MAX_CANDIDATES and
    never fewer than k.  On 1M x 768 unit-gaussian and clustered rows, int8 and bf16 galleries refined from 2 k
    candidates already reach the recall of 4 k and 8 k (DESIGN.md section 4, "Refined search"); 2 k reads half
    the store rows of 4 k."""
    return max(int(k), min(2 * int(k), MAX_CANDIDATES))


def candidate_k(k: int, refine_k: Optional[int], n_rows: int, n_allowed: Optional[int] = None) -> int:
    """k_c = min(refine_k, n_rows, rows a RowFilter allows): the candidate search's k.  refine_k None: the
    default; refine_k < k raises ValueError, and so does a k_c above MAX_CANDIDATES."""
    rk = default_refine_k(k) if refine_k is None else int(refine_k)
    if rk < k:
        raise ValueError(f"refine_k = {rk} must be >= k = {k}")
    k_c = min(rk, int(n_rows))
    if n_allowed is not None:
        k_c = min(k_c, int(n_allowed))
    if k_c > MAX_CANDIDATES:
        raise ValueError(f"refine: {k_c} candidates per query, at most {MAX_CANDIDATES} (lower refine_k)")
    return k_c


def store_rows(features: torch.Tensor, mode: str, out: torch.Tensor) -> torch.Tensor:
    """Fill `out` [N, Dp] (Dp = D rounded up to 8, the row layout of `DeviceGallery(features, mode)`) with the
    rows of `features` in the mode's dtype and zero padding, in chunks of at most 256 MB of fp32 input."""
    n, d = int(features.shape[0]), int(features.shape[1])
    dt = torch.bfloat16 if mode == "bf16" else torch.float32
    if out.dtype != dt or tuple(out.shape) != (n, _pad_dim(d)):
        raise ValueError(f"store rows must be {dt} [{n}, {_pad_dim(d)}]")
    if out.shape[1] > d:
        out[:, d:] = 0
    step = max(1, (256 << 20) // max(1, d * 4))
    for lo in range(0, n, step):
        out[lo:lo + step, :d] = features[lo:lo + step].detach().to(device=out.device, dtype=dt)
    return out


def _page_aligned_host(nbytes: int):
    """(backing uint8 buffer, page-aligned byte view of it covering whole pages >= nbytes): pages no other
    tensor shares, so registering them cannot overlap another registration."""
    span = (nbytes + _PAGE - 1) // _PAGE * _PAGE
    buf = torch.empty(span + _PAGE, dtype=torch.uint8)
    off = (-buf.data_ptr()) % _PAGE
    return buf, buf[off:off + span]


def _unregister(ptr: int, buf) -> None:
    del buf                          # held until here: the pages stay allocated while they are registered
    _cabi.lib.mmrs_host_unregister(ptr)


class RefineStore:
    """A full-precision copy of a gallery's rows for `search_topk(..., refine=store)`.

    mode "fp32" or "bf16": the rows exactly as `DeviceGallery(features, mode).data` holds them -- [N, Dp], Dp = D
    rounded up to 8, zero columns past D, rows 16-byte aligned.  int8 is refused: the store exists to be exact.
    memory "device": in HBM of `device` (default: the features' device, else the current one).
    memory "host": in ordinary host memory, page-locked with cudaHostRegister (mmrs_host_register) and read by
    the refine kernel over PCIe; it is not a `pin_memory()` tensor, whose allocator would round the block up to
    a power of two.  `close()` (or dropping the store) unregisters it.  Input is copied in bounded chunks.
    """

    def __init__(self, features, mode: str = "fp32", memory: str = "host", device: Optional[torch.device] = None):
        if mode == "int8":
            raise ValueError("a refine store is fp32 or bf16: int8 rows are what it refines")
        if mode not in ("fp32", "bf16"):
            raise ValueError("mode must be 'fp32' or 'bf16'")
        if memory not in ("host", "device"):
            raise ValueError("memory must be 'host' or 'device'")
        if isinstance(features, np.ndarray):
            features = torch.from_numpy(features)
        if not isinstance(features, torch.Tensor) or features.dim() != 2:
            raise TypeError("features must be a 2-D torch.Tensor / numpy array [N, D]")
        self.mode, self.memory = mode, memory
        self.n_rows, self.dim = int(features.shape[0]), int(features.shape[1])
        if self.n_rows < 1 or self.dim < 1:
            raise ValueError("a refine store must have at least one row and one column")
        self.padded_dim = _pad_dim(self.dim)
        self._finalizer = None
        if memory == "device":
            gal = DeviceGallery(features, mode=mode, device=device)
            self.device = gal.device
            self.data = gal.data
            self.ptr = self.data.data_ptr()
            return
        if device is None:
            device = features.device if features.is_cuda else torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)
        device = torch.device(device)
        _cabi.require_b200(device.index if device.index is not None else 0)
        self.device = None                       # registered as portable: any device of the process reads it
        dt = torch.bfloat16 if mode == "bf16" else torch.float32
        nbytes = self.n_rows * self.padded_dim * (2 if mode == "bf16" else 4)
        buf, pages = _page_aligned_host(nbytes)
        self.data = store_rows(features, mode, pages[:nbytes].view(dt).view(self.n_rows, self.padded_dim))
        dptr = ctypes.c_void_p()
        with torch.cuda.device(device):
            _cabi.check(_cabi.lib.mmrs_host_register(pages.data_ptr(), pages.numel(), ctypes.byref(dptr)))
        self.ptr = int(dptr.value)
        self._finalizer = weakref.finalize(self, _unregister, pages.data_ptr(), buf)

    @property
    def dtype_code(self) -> int:
        return _cabi.DTYPE_BF16 if self.mode == "bf16" else _cabi.DTYPE_F32

    @property
    def ld(self) -> int:
        return self.padded_dim

    @property
    def nbytes(self) -> int:
        return self.n_rows * self.padded_dim * (2 if self.mode == "bf16" else 4)

    def close(self) -> None:
        """Release the rows now (a host store is unregistered first); the store cannot be used afterwards."""
        if self._finalizer is not None:
            self._finalizer()
        self.data, self.ptr = None, 0

    def check_matches(self, gal) -> None:
        """ValueError unless this store holds the rows of `gal`: same row count and width, and for a device
        store the same device."""
        if self.ptr == 0:
            raise ValueError("this RefineStore was closed")
        if self.n_rows != gal.n_rows or self.dim != gal.dim:
            raise ValueError(f"refine store is [{self.n_rows}, {self.dim}], the gallery [{gal.n_rows}, {gal.dim}]")
        if self.device is not None and self.device != gal.device:
            raise ValueError(f"refine store is on {self.device}, the gallery on {gal.device}")

    def __len__(self) -> int:
        return self.n_rows

    def __repr__(self) -> str:
        return (f"RefineStore(rows={self.n_rows}, dim={self.dim}, mode={self.mode}, memory={self.memory}"
                f"{'' if self.device is None else f', device={self.device}'})")
