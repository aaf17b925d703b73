"""Near-duplicate join behind the reference's data-governance signatures.

Reference tools (paths relative to the reference checkout):
    tool/find_repeated.py                  cross-folder exact join (MD5 of RGB bytes), :35-71
    tool/find_repeated_in_same_folder.py   same-folder near join (pHash/dHash/wHash, Hamming), :56-106
    tool/delete repeated.py                train-vs-test join (dHash), :11-162
BASELINE.json replaces the hash predicates by `cos(e_i, e_j) >= tau` on unit-norm embeddings
(SURVEY.md M2); the call signatures and result tuples are kept.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Callable, Optional, Sequence

import numpy as np
import torch

from . import _cabi
from .gallery import DeviceGallery, _pad_dim
from .search import search_topk, _stream_handle


# ---- tensor level -------------------------------------------------------------------------------
def _device_f32(emb, device=None) -> torch.Tensor:
    if isinstance(emb, DeviceGallery):
        if emb.mode != "fp32":
            raise ValueError("exact self-join needs an fp32 gallery")
        return emb.data
    if isinstance(emb, np.ndarray):
        emb = torch.from_numpy(emb)
    if emb.dim() != 2:
        raise ValueError("embeddings must be [N, D]")
    dev = torch.device(device) if device is not None else (
        emb.device if emb.is_cuda else torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0))
    _cabi.require_b200(dev.index or 0)
    n, d = emb.shape
    dp = _pad_dim(d)
    x = emb.detach().to(device=dev, dtype=torch.float32)
    if dp != d:
        x = torch.nn.functional.pad(x, (0, dp - d))
    return x.contiguous()


def selfjoin_raw(x: torch.Tensor, threshold: float, row_begin: int = 0, row_end: Optional[int] = None,
                 capacity: Optional[int] = None) -> torch.Tensor:
    """Unsorted int64 [P, 2] pairs (i < j, row_begin <= i < row_end) from the CUDA kernel;
    grows the pair buffer and retries when the kernel reports more pairs than `capacity`."""
    n = int(x.shape[0])
    row_end = n if row_end is None else int(row_end)
    lib = _cabi.lib
    cap = int(capacity) if capacity is not None else max(4096, 2 * (row_end - row_begin))
    with torch.cuda.device(x.device):
        count = torch.zeros(1, dtype=torch.int64, device=x.device)
        while True:
            pairs = torch.empty((cap, 2), dtype=torch.int64, device=x.device)
            st = lib.mmrs_selfjoin_pairs(x.data_ptr(), n, int(x.shape[1]), x.stride(0), _cabi.DTYPE_F32,
                                         float(threshold), int(row_begin), row_end, pairs.data_ptr(),
                                         cap, count.data_ptr(), None, 0, _stream_handle(x.device))
            found = int(count.item())
            if st == _cabi.ERR_CAPACITY:
                cap = found  # exact size is known now
                continue
            _cabi.check(st)
            return pairs[:found]


BF16_MARGIN = 0.0045   # > 2 * 2^-9 * (1 + 2^-9): bound on the bf16 rounding of a unit-norm dot product


def row_norm_range(x32: torch.Tensor) -> "tuple[float, float]":
    """(min, max) L2 norm over the rows of a device fp32 matrix (mmrs_row_norm_range)."""
    with torch.cuda.device(x32.device):
        mm = torch.empty(2, dtype=torch.float32, device=x32.device)
        _cabi.check(_cabi.lib.mmrs_row_norm_range(x32.data_ptr(), int(x32.shape[0]), int(x32.shape[1]), x32.stride(0),
                                                  mm.data_ptr(), _stream_handle(x32.device)))
        lo, hi = mm.tolist()
    return float(lo), float(hi)


def selfjoin_tc_raw(x32: torch.Tensor, threshold: float, rank: int = 0, world: int = 1,
                    x16: Optional[torch.Tensor] = None, margin: float = BF16_MARGIN,
                    capacity: Optional[int] = None) -> torch.Tensor:
    """Unsorted int64 [P, 2] pairs of rank `rank`'s panels: tcgen05 bf16 prefilter at
    threshold - margin, exact fp32 recheck (mmrs_selfjoin_pairs_tc); buffers grow on demand.
    `margin` bounds the bf16 rounding error of a dot product of UNIT rows; it is scaled by the
    largest squared row norm found on the device (|<a,b> - <a16,b16>| <= ~2^-8 |a||b|), so rows that
    are not unit-norm (raw CLIP features) cannot lose true pairs before the exact recheck."""
    n, d = int(x32.shape[0]), int(x32.shape[1])
    lib = _cabi.lib
    dev = x32.device
    _, max_norm = row_norm_range(x32)
    if not (max_norm < float("inf")):
        raise ValueError("embeddings contain non-finite rows")
    margin = float(margin) * max(1.0, max_norm * max_norm * 1.0001)
    if x16 is None:
        x16 = x32.to(torch.bfloat16)
    cap = int(capacity) if capacity is not None else max(4096, n // 4)
    cand_cap = 2 * cap
    with torch.cuda.device(dev):
        counts = torch.zeros(2, dtype=torch.int64, device=dev)
        while True:
            pairs = torch.empty((cap, 2), dtype=torch.int64, device=dev)
            ws_bytes = lib.mmrs_selfjoin_tc_workspace_bytes(n, cand_cap)
            ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
            st = lib.mmrs_selfjoin_pairs_tc(x32.data_ptr(), x32.stride(0), x16.data_ptr(), x16.stride(0), n, d,
                                            float(threshold), float(margin), int(rank), int(world),
                                            pairs.data_ptr(), cap, counts.data_ptr(), cand_cap,
                                            DeviceGallery.aligned_ptr(ws), ws_bytes, _stream_handle(dev))
            found, n_cand = (int(v) for v in counts.tolist())
            if st == _cabi.ERR_CAPACITY:
                # counts are exact: candidates first (the recheck does not run past its capacity)
                cand_cap = max(cand_cap, n_cand)
                cap = max(cap, found, n_cand)
                continue
            _cabi.check(st)
            return pairs[:found]


def sort_pairs(pairs: torch.Tensor, n: int) -> torch.Tensor:
    """Lexicographic (i, j) order -- what `triu(S >= tau, 1).nonzero()` yields row-major.
    Device pair lists are sorted by the library's own bitonic sort on packed (i << 32 | j) keys
    (mmrs_sort_pairs); host lists (CPU tests of the sharded protocol) by numpy."""
    del n
    if pairs.numel() == 0:
        return pairs.reshape(0, 2)
    if not pairs.is_cuda:
        a = pairs.numpy()
        return torch.from_numpy(a[np.lexsort((a[:, 1], a[:, 0]))].copy())
    out = pairs.contiguous().clone()
    lib = _cabi.lib
    with torch.cuda.device(out.device):
        ws_bytes = lib.mmrs_sort_pairs_workspace_bytes(int(out.shape[0]))
        ws = torch.empty(int(ws_bytes) + 256, dtype=torch.uint8, device=out.device)
        _cabi.check(lib.mmrs_sort_pairs(out.data_ptr(), int(out.shape[0]), DeviceGallery.aligned_ptr(ws), ws_bytes,
                                        _stream_handle(out.device)))
    return out


def find_duplicate_pairs(emb, threshold: float, *, device=None, method: str = "auto") -> torch.Tensor:
    """All (i, j), i < j, with <e_i, e_j> >= threshold over unit-norm fp32 rows -> int64 [P, 2]
    sorted lexicographically.  Host input gives a host result.

    method "fp32": every pair in fp32 on the CUDA cores.  "tc": bf16 tensor-core prefilter with a
    safety margin + exact fp32 recheck of the survivors -- the same pair set (rows must be
    unit-norm for the margin to hold), ~20x the throughput.  "auto": "tc" from 2048 rows on."""
    on_host = not isinstance(emb, DeviceGallery) and not (isinstance(emb, torch.Tensor) and emb.is_cuda)
    x = _device_f32(emb, device)
    pairs = sort_pairs(_join_raw(x, threshold, method), int(x.shape[0]))
    return pairs.cpu() if on_host else pairs


def _join_raw(x: torch.Tensor, threshold: float, method: str) -> torch.Tensor:
    """The unsorted pair list of find_duplicate_pairs' `method` on a device fp32 matrix."""
    if method not in ("auto", "fp32", "tc"):
        raise ValueError("method must be 'auto', 'fp32' or 'tc'")
    use_tc = method == "tc" or (method == "auto" and x.shape[0] >= 2048)
    return selfjoin_tc_raw(x, threshold) if use_tc else selfjoin_raw(x, threshold)


def greedy_first_keeper(n: int, pairs, order: Sequence[int]):
    """The keep/delete decision of tool/find_repeated_in_same_folder.py:76-95 on a pair list:
    walk items in `order`; an item adjacent to an already kept representative is a duplicate of
    the EARLIEST-kept such representative (the reference's `for ... break` over
    reference_hashes), otherwise it becomes a representative.
    Returns (representatives, [(dup, original)]) as item ids."""
    pairs = np.asarray(pairs.cpu() if isinstance(pairs, torch.Tensor) else pairs, dtype=np.int64).reshape(-1, 2)
    # CSR adjacency of the undirected pair graph
    src = np.concatenate([pairs[:, 0], pairs[:, 1]])
    dst = np.concatenate([pairs[:, 1], pairs[:, 0]])
    o = np.argsort(src, kind="stable")
    src, dst = src[o], dst[o]
    start = np.searchsorted(src, np.arange(n + 1))
    keep_rank = np.full(n, -1, dtype=np.int64)   # position in the representative list, -1 = not kept
    reps, dups = [], []
    for item in order:
        nb = dst[start[item]:start[item + 1]]
        ranks = keep_rank[nb]
        ranks = ranks[ranks >= 0]
        if ranks.size:
            dups.append((int(item), reps[int(ranks.min())]))
        else:
            keep_rank[item] = len(reps)
            reps.append(int(item))
    return reps, dups


MAX_RESOLVE_ROWS = 2 ** 31 - 1     # ranks and row ids are 32-bit on the device


def _resolve_args(pairs, n, order):
    """Host-side checks of resolve_duplicates -> (pairs, n, order or None, device or None); raises ValueError."""
    if isinstance(n, bool) or not isinstance(n, (int, np.integer)):
        raise ValueError(f"n must be an integer row count, got {n!r}")
    n = int(n)
    if not 0 <= n <= MAX_RESOLVE_ROWS:
        raise ValueError(f"n = {n}: the resolve takes 0 <= n < 2^31 rows")
    if isinstance(pairs, np.ndarray):
        pairs = torch.from_numpy(np.ascontiguousarray(pairs))
    if not isinstance(pairs, torch.Tensor):
        raise ValueError(f"pairs must be an int64 [P, 2] tensor, got {type(pairs).__name__}")
    if pairs.dtype != torch.int64:
        raise ValueError(f"pairs must be int64, got {pairs.dtype}")
    if pairs.dim() != 2 or pairs.shape[1] != 2:
        raise ValueError(f"pairs must be [P, 2], got {tuple(pairs.shape)}")
    if order is not None:
        if isinstance(order, np.ndarray):
            order = torch.from_numpy(np.ascontiguousarray(order))
        elif not isinstance(order, torch.Tensor):
            order = torch.as_tensor(list(order), dtype=torch.int64)
        if order.dtype != torch.int64:
            raise ValueError(f"order must be int64 row ids, got {order.dtype}")
        if order.dim() != 1:
            raise ValueError(f"order must be 1-D, got {tuple(order.shape)}")
        if order.numel() > MAX_RESOLVE_ROWS:
            raise ValueError(f"order has {order.numel()} ids: at most 2^31 - 1")
    dev = pairs.device if pairs.is_cuda else (order.device if order is not None and order.is_cuda else None)
    return pairs, n, order, dev


def _resolve(pairs, n: int, order=None):
    """resolve_duplicates plus the schedule it took: (representative, rounds, rows decided by the tail)."""
    pairs, n, order, dev = _resolve_args(pairs, n, order)
    on_host = dev is None
    if on_host:
        dev = torch.device("cuda", torch.cuda.current_device() if torch.cuda.is_available() else 0)
    _cabi.require_b200(dev.index or 0)
    with torch.cuda.device(dev):
        p = pairs.to(dev).contiguous()
        o = order.to(dev).contiguous() if order is not None else None
        n_order = n if o is None else int(o.numel())
        rep = torch.empty(n, dtype=torch.int64, device=dev)
        lib = _cabi.lib
        ws_bytes = int(lib.mmrs_resolve_duplicates_workspace_bytes(n, n_order, int(p.shape[0])))
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        stats = (C.c_int64 * 2)()
        st = lib.mmrs_resolve_duplicates(p.data_ptr() if p.numel() else None, int(p.shape[0]),
                                         o.data_ptr() if o is not None and o.numel() else None,   # null: 0..n_order-1
                                         n_order, n, rep.data_ptr() if n else None, stats,
                                         DeviceGallery.aligned_ptr(ws), ws_bytes, _stream_handle(dev))
        if st == _cabi.ERR_ARG:
            raise ValueError(_cabi.last_error())
        _cabi.check(st)
    return (rep.cpu() if on_host else rep), int(stats[0]), int(stats[1])


def resolve_duplicates(pairs, n: int, *, order=None) -> torch.Tensor:
    """The decision of `greedy_first_keeper` on the device: int64 [n] with representative[v] =
        v                                        if v is kept,
        the kept neighbour of v first in order   if v is removed (v duplicates it),
        -1                                       if v is not in `order`.
    `pairs` is int64 [P, 2] with ids in [0, n), in any order and orientation (repeated and self-pairs
    allowed; a self-pair has no effect); `order` the walk order, distinct ids in [0, n) (default
    0..n-1; a subset is allowed -- the reference walks by file size, pass that permutation).  For such
    inputs `[v for v in order if rep[v] == v]` is greedy_first_keeper's representatives and
    `[(v, rep[v]) for v in order if rep[v] not in (v, -1)]` its duplicates.  A repeated or out-of-range
    order id, an out-of-range pair id and n >= 2^31 raise ValueError.  Device input gives a device
    result; host input runs on the current device and returns a host tensor.
    `rep == torch.arange(n, device=rep.device)` is the keep mask (RowFilter of the deduplicated gallery)."""
    return _resolve(pairs, n, order)[0]


def deduplicate(emb, threshold: float, *, order=None, method: str = "auto", device=None) -> torch.Tensor:
    """find_duplicate_pairs followed by resolve_duplicates, with the pair list kept on the device and
    unsorted (the resolve does not need the lexicographic order).  Same inputs and `method` as
    find_duplicate_pairs; returns the [n] representative tensor (host input gives a host result)."""
    on_host = not isinstance(emb, DeviceGallery) and not (isinstance(emb, torch.Tensor) and emb.is_cuda)
    if method not in ("auto", "fp32", "tc"):
        raise ValueError("method must be 'auto', 'fp32' or 'tc'")     # before the embeddings are uploaded
    x = _device_f32(emb, device)
    rep = resolve_duplicates(_join_raw(x, threshold, method), int(x.shape[0]), order=order)
    return rep.cpu() if on_host else rep


# ---- file level -------------------------------------------------------------------------------
IMAGE_EXTENSIONS = {'.jpg', '.jpeg', '.png', '.bmp', '.gif', '.tiff'}


def get_all_images(folder_path):
    """Drop-in for tool/find_repeated.py:21-33: recursive listing filtered by extension."""
    image_files = []
    for root, _, files in os.walk(folder_path):
        image_files.extend(os.path.join(root, f) for f in files
                           if os.path.splitext(f)[1].lower() in IMAGE_EXTENSIONS)
    return image_files


def pixel_embedding(paths: Sequence[str], size: int = 16):
    """Default embedder when no CLIP encoder is supplied (the encoders are third-party and out of
    scope, SURVEY.md L1): RGB pixels box-resized to size x size, mean-removed, unit-normalised.
    Pixel-identical images (the MD5 predicate of find_repeated.py:6-19) map to identical vectors.
    Returns (embeddings [n_ok, 3*size*size] fp32, ok_mask [len(paths)] bool); unreadable files
    are reported and skipped like the reference does (:17-19)."""
    from PIL import Image
    vecs, ok = [], []
    for p in paths:
        try:
            with Image.open(p) as img:
                a = np.asarray(img.convert("RGB").resize((size, size), Image.BOX), dtype=np.float32).reshape(-1)
            a = a - a.mean()
            nrm = np.linalg.norm(a)
            vecs.append(a / nrm if nrm > 0 else np.full_like(a, 1.0 / np.sqrt(a.size)))
            ok.append(True)
        except Exception as e:  # noqa: BLE001 -- mirror the reference's blanket handler
            print(f"Error processing {p}: {e}")
            ok.append(False)
    emb = torch.from_numpy(np.stack(vecs)) if vecs else torch.empty((0, 3 * size * size))
    return emb, np.array(ok, dtype=bool)


Embedder = Callable[[Sequence[str]], "tuple[torch.Tensor, np.ndarray]"]


def _remove(path: str, dry_run: bool) -> bool:
    if dry_run:
        return True
    try:
        os.remove(path)
        return True
    except Exception as e:  # noqa: BLE001
        print(f"Failed to delete {path}: {e}")
        return False


def calculate_image_hash(image_path):
    """Drop-in for tool/find_repeated.py:6-19: MD5 of the RGB pixel bytes (None for unreadable files)."""
    import hashlib
    from PIL import Image
    try:
        with Image.open(image_path) as img:
            return hashlib.md5(img.convert("RGB").tobytes()).hexdigest()
    except Exception as e:  # noqa: BLE001 -- mirror the reference's blanket handler
        print(f"Error processing {image_path}: {e}")
        return None


def _check_cosine_threshold(t, what: str) -> float:
    """Thresholds of the destructive wrappers must be cosines in (0.5, 1]."""
    if isinstance(t, bool) or not isinstance(t, (int, float, np.floating, np.integer)):
        raise TypeError(f"{what} must be a number in (0.5, 1], got {t!r}")
    t = float(t)
    if not (0.5 < t <= 1.0):
        raise ValueError(f"{what} = {t!r}: this build's predicate is cos(e_i, e_j) >= threshold on unit-norm "
                         "embeddings and accepts 0.5 < threshold <= 1 (higher = stricter); the reference's "
                         "`similarity_threshold` is a Hamming radius on perceptual hashes (0 = strictest, default 5) "
                         "and cannot be translated -- pass cosine_threshold=0.95 (or stricter) instead")
    return t


def _cross_folder(reference_folder, delete_folder, embed: Optional[Embedder], threshold: float, dry_run: bool,
                  confirm: str):
    reference_images = get_all_images(reference_folder)
    delete_images = get_all_images(delete_folder)
    print(f"Found {len(reference_images)} images in reference folder")
    print(f"Found {len(delete_images)} images in delete folder")
    deleted_files, kept_files = [], []
    embed_fn = embed or pixel_embedding
    ref_emb, ref_ok = embed_fn(reference_images)
    del_emb, del_ok = embed_fn(delete_images)
    ref_paths = [p for p, ok in zip(reference_images, ref_ok) if ok]
    match = {}
    if len(ref_paths) and del_emb.shape[0]:
        # probe side = queries, build side = gallery: top-1 per delete image, thresholded
        vals, idx = search_topk(del_emb, DeviceGallery(ref_emb, mode="fp32"), 1,
                                normalize_queries=False, scale=1.0)
        vals, idx = vals.cpu().numpy()[:, 0], idx.cpu().numpy()[:, 0]
        ok_pos = np.flatnonzero(del_ok)
        for row, (v, i) in enumerate(zip(vals, idx)):
            if v >= threshold:
                match[delete_images[ok_pos[row]]] = ref_paths[int(i)]
    if confirm == "exact" and match:
        # The reference's predicate is pixel identity (MD5 of the RGB bytes, find_repeated.py:6-19).  The
        # embedding search above is the prefilter (identical pixels -> identical vectors -> cos = 1, so it
        # has no false negatives); a candidate is only deleted when its hash equals a reference image's, and
        # the reported reference is the LAST one with that hash, as the reference's dict build leaves it (:50-52).
        reference_hashes = {}
        for p in reference_images:
            h = calculate_image_hash(p)
            if h:
                reference_hashes[h] = p
        confirmed = {}
        for p in match:
            h = calculate_image_hash(p)
            if h and h in reference_hashes:
                confirmed[p] = reference_hashes[h]
        match = confirmed
    for img_path in delete_images:
        if img_path in match:
            if _remove(img_path, dry_run):
                deleted_files.append((img_path, match[img_path]))
        else:
            kept_files.append(img_path)
    return deleted_files, kept_files, len(reference_images), len(delete_images)


def find_and_remove_near_duplicate_images(folder_path, cosine_threshold=0.95, *,
                                          embed: Optional[Embedder] = None, dry_run: bool = False):
    """Same-folder form, tool/find_repeated_in_same_folder.py:56-106: sort by file size descending
    (:73), keep the first of every group of similar images, delete the rest.
    Returns (deleted_files [(dup, original)], reference_images, total).
    The predicate is cos(e_i, e_j) >= `cosine_threshold` (0.5 < t <= 1) on the embeddings, where the
    reference uses a Hamming radius on perceptual hashes (SURVEY.md M2)."""
    cosine_threshold = _check_cosine_threshold(cosine_threshold, "cosine_threshold")
    embed = embed or pixel_embedding
    all_images = get_all_images(folder_path)
    print(f"在文件夹中找到 {len(all_images)} 个图像")
    all_images.sort(key=lambda x: os.path.getsize(x), reverse=True)
    emb, ok = embed(all_images)
    usable = [p for p, good in zip(all_images, ok) if good]   # unreadable files are skipped (:78)
    reference_images, duplicate_images = [], []
    if len(usable) >= 2:
        pairs = find_duplicate_pairs(emb, cosine_threshold)
        reps, dups = greedy_first_keeper(len(usable), pairs, range(len(usable)))
        reference_images = [usable[i] for i in reps]
        duplicate_images = [(usable[d], usable[o]) for d, o in dups]
    else:
        reference_images = list(usable)
    deleted_files = [(d, o) for d, o in duplicate_images if _remove(d, dry_run)]
    return deleted_files, reference_images, len(all_images)


def find_and_remove_duplicate_images(reference_folder, delete_folder=None, *, embed: Optional[Embedder] = None,
                                     threshold: float = 0.9999, cosine_threshold: float = 0.95,
                                     confirm: Optional[str] = None, dry_run: bool = False):
    """Drop-in for BOTH reference functions of this name.

    (reference_folder, delete_folder: path)  -> tool/find_repeated.py:35-71
        images of `delete_folder` that match an image of `reference_folder` are deleted;
        returns (deleted_files [(path, ref_path)], kept_files, n_ref, n_del).  The GPU top-1 search
        (cos >= `threshold`) finds the candidates; with the default embedder every candidate is then
        CONFIRMED with the reference's own predicate -- equal MD5 of the RGB bytes -- before it is
        deleted (`confirm="exact"`), so the deletion set and the reported reference paths are the
        reference's.  A caller who passes an encoder (`embed=`) asks for the embedding predicate and gets
        `confirm="none"` unless stated otherwise.
    (folder_path) -> tool/find_repeated_in_same_folder.py:56-106
        returns (deleted_files, reference_images, total); the predicate is cos >= `cosine_threshold`.
        The reference's second positional argument is a Hamming radius (0 = strictest, default 5): a number
        there is REFUSED with a ValueError -- it has no cosine equivalent, and guessing one on a function
        that deletes files is not acceptable.
    """
    if delete_folder is None:
        return find_and_remove_near_duplicate_images(reference_folder, cosine_threshold, embed=embed, dry_run=dry_run)
    if not isinstance(delete_folder, (str, bytes, os.PathLike)):
        raise ValueError(f"second argument {delete_folder!r}: a folder path selects the cross-folder form "
                         "(tool/find_repeated.py); the same-folder form's `similarity_threshold` is a Hamming "
                         "radius on perceptual hashes in the reference (0 = strictest, default 5), which this "
                         "embedding-based build cannot honour -- call find_and_remove_duplicate_images(folder, "
                         "cosine_threshold=0.95) with a cosine in (0.5, 1]")
    threshold = _check_cosine_threshold(threshold, "threshold")
    if confirm is None:
        confirm = "exact" if embed is None else "none"
    if confirm not in ("exact", "none"):
        raise ValueError("confirm must be 'exact' or 'none'")
    return _cross_folder(reference_folder, delete_folder, embed, threshold, dry_run, confirm)


CROSS_SET_EXTENSIONS = ['.jpg', '.jpeg', '.png', '.bmp', '.gif', '.webp']   # tool/delete repeated.py:35
last_cross_set_summary: dict = {}


def detect_and_remove_cross_set_duplicates(test_dir, train_dir, hash_size=8, similarity_threshold=0, *,
                                           embed: Optional[Embedder] = None, cosine_threshold: float = 0.9999,
                                           dry_run: bool = False):
    """Drop-in for `tool/delete repeated.py`:11-162 (train-vs-test leakage removal): every image of
    `train_dir` that matches an image of `test_dir` is deleted from `train_dir`; prints the same
    summary and returns None like the reference (the numbers are kept in `last_cross_set_summary`).
    `hash_size` / `similarity_threshold` are the reference's dHash parameters and are accepted for
    signature compatibility; the predicate here is cos(e_train, e_test) >= `cosine_threshold`
    (top-1 search of the train embeddings against the test gallery)."""
    del hash_size
    if similarity_threshold != 0:
        raise ValueError("similarity_threshold is the reference's dHash Hamming radius; only its default 0 (identical "
                         "hashes) is accepted here -- the predicate of this build is cos >= cosine_threshold")
    cosine_threshold = _check_cosine_threshold(cosine_threshold, "cosine_threshold")
    for d, name in ((test_dir, "测试集"), (train_dir, "训练集")):
        if not os.path.exists(d):
            print(f"错误: {name}目录 '{d}' 不存在。")
            return

    def listing(folder):
        out = []
        for root, _, files in os.walk(folder):
            out.extend(os.path.join(root, f) for f in files if os.path.splitext(f)[1].lower() in CROSS_SET_EXTENSIONS)
        return out

    embed = embed or pixel_embedding
    test_images, train_images = listing(test_dir), listing(train_dir)
    test_emb, test_ok = embed(test_images)
    train_emb, train_ok = embed(train_images)
    test_paths = [p for p, ok in zip(test_images, test_ok) if ok]
    duplicates_found = deleted_files = 0
    if len(test_paths) and train_emb.shape[0]:
        vals, idx = search_topk(train_emb, DeviceGallery(test_emb, mode="fp32"), 1, normalize_queries=False)
        ok_pos = np.flatnonzero(train_ok)
        for row, (v, i) in enumerate(zip(vals.cpu().numpy()[:, 0], idx.cpu().numpy()[:, 0])):
            if v >= cosine_threshold:
                duplicates_found += 1
                path = train_images[ok_pos[row]]
                print(f"\n发现重复图片 #{duplicates_found}:\n测试集: {test_paths[int(i)]}\n训练集: {path}")
                if _remove(path, dry_run):
                    deleted_files += 1
    last_cross_set_summary.clear()
    last_cross_set_summary.update(test_images=len(test_images), train_images=len(train_images),
                                  duplicates_found=duplicates_found, deleted_files=deleted_files)
    print("\n====== 操作摘要 ======")
    print(f"测试集图片数: {len(test_images)}")
    print(f"训练集图片数: {len(train_images)}")
    print(f"发现的重复图片数: {duplicates_found}")
    print(f"已删除的训练集重复图片: {deleted_files}")
    print("=====================")
