"""CPU oracle for the retrieval hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module; the product package never does (it has no CPU path at all).

The reference's arithmetic for this path lives in PyTorch (unpinned third-party dependency; this
container has torch 2.11.0 CPU/MKL).  Every function below is the reference's own expression
restated on CPU tensors, with the reference file:line it follows (paths relative to the
reference checkout).  Parity pinning: the reference ships no tests or golden vectors for this
path (SURVEY.md section 4); tests/golden/make_golden.py executes the reference's OWN function
bodies (get_similarity, eval_threshold, find_thresholds, cls_acc's topk, find_repeated.py)
in this container with `.cuda()` patched to a no-op, and tests/test_oracle.py checks this module
against those recorded outputs.
"""
from __future__ import annotations

import hashlib
import os
from typing import Iterable

import numpy as np
import torch


# --------------------------------------------------------------------------------------------
# normalisation idiom: code/search_image.py:130,133,139,157,336 ; code/utils.py:90,144
# --------------------------------------------------------------------------------------------
def l2_normalize(x: torch.Tensor) -> torch.Tensor:
    """`x /= x.norm(dim=-1, keepdim=True)` -- no epsilon (a zero row gives NaN)."""
    return x / x.norm(dim=-1, keepdim=True)


def prepare_queries(queries: torch.Tensor, normalize_queries: bool, mode: str) -> torch.Tensor:
    """fp32 query matrix as the scoring sees it.

    mode "bf16": the normalised query is rounded to bf16 (the value the tensor cores multiply);
    SURVEY.md H2: recall >= 0.999 is only meaningful when the oracle is fed the same bf16-valued
    gallery AND queries."""
    q = queries.detach().to(torch.float32).cpu()
    if normalize_queries:
        q = l2_normalize(q)
    if mode == "bf16":
        q = q.to(torch.bfloat16).to(torch.float32)
    elif mode != "fp32":
        raise ValueError(f"mode must be 'fp32' or 'bf16', got {mode!r}")
    return q


def _gallery_f32(gallery: torch.Tensor) -> torch.Tensor:
    # a bf16 gallery IS the dataset; the oracle upcasts those exact values (BASELINE.md section 5)
    return gallery.detach().cpu().to(torch.float32)


# --------------------------------------------------------------------------------------------
# scores: code/search_image.py:107  `100. * features.cuda() @ ref_feature.t()`
#         CLIP/lab3.py:114 (scale 1), code/merge_dataset.py:275-278 (scale logit_scale.exp())
# --------------------------------------------------------------------------------------------
def full_scores(queries: torch.Tensor, gallery: torch.Tensor, *, normalize_queries: bool = True,
                scale: float = 1.0, mode: str = "fp32") -> torch.Tensor:
    """[Q, N] fp32 scores = scale * q @ G.T (the reference computes G @ q.T for one q)."""
    q = prepare_queries(queries, normalize_queries, mode)
    g = _gallery_f32(gallery)
    s = q @ g.t()
    if scale != 1.0:
        s = torch.tensor(scale, dtype=torch.float32) * s
    return s


# --------------------------------------------------------------------------------------------
# top-k: code/utils.py:17  `output.topk(topk, 1, True, True)` -> (values, indices)
# --------------------------------------------------------------------------------------------
def topk_rows(scores: torch.Tensor, k: int) -> tuple[torch.Tensor, torch.Tensor]:
    """k largest per row, sorted descending, equal scores by ascending index.

    torch.topk does not promise an order among ties; a stable descending sort does, and is what
    the CUDA path's (score, ~row) keys reproduce (SURVEY.md H1)."""
    if k > scores.shape[1]:
        raise RuntimeError("selected index k out of range")  # torch.topk's own error
    vals, idx = torch.sort(scores, dim=1, descending=True, stable=True)
    return vals[:, :k].contiguous(), idx[:, :k].contiguous()


def search_topk(queries: torch.Tensor, gallery: torch.Tensor, k: int, *,
                normalize_queries: bool = True, scale: float = 1.0, mode: str = "fp32",
                block_rows: int = 1 << 18) -> tuple[torch.Tensor, torch.Tensor]:
    """search_image.py:107 followed by utils.py:17, blocked over gallery rows so the [Q, N]
    matrix of a 1M-row gallery need not be resident; the merge keeps the stable order."""
    q = prepare_queries(queries, normalize_queries, mode)
    n = gallery.shape[0]
    if k > n:
        raise RuntimeError("selected index k out of range")
    best_v = None
    best_i = None
    sc = torch.tensor(scale, dtype=torch.float32)
    for lo in range(0, n, block_rows):
        g = _gallery_f32(gallery[lo:lo + block_rows])
        s = q @ g.t()
        if scale != 1.0:
            s = sc * s
        kk = min(k, s.shape[1])
        v, i = torch.sort(s, dim=1, descending=True, stable=True)
        v, i = v[:, :kk], i[:, :kk] + lo
        if best_v is None:
            best_v, best_i = v, i
        else:
            cv = torch.cat([best_v, v], dim=1)
            ci = torch.cat([best_i, i], dim=1)
            # earlier blocks come first in the concatenation and hold lower indices, so a stable
            # sort keeps "index ascending among equal scores"
            o = torch.sort(cv, dim=1, descending=True, stable=True)[1][:, :k]
            best_v, best_i = torch.gather(cv, 1, o), torch.gather(ci, 1, o)
    return best_v.contiguous(), best_i.contiguous()


def merge_topk(values: torch.Tensor, indices: torch.Tensor, k: int) -> tuple[torch.Tensor, torch.Tensor]:
    """Merge [G, Q, k_in] per-shard results (global indices) -> [Q, k]; score desc, index asc."""
    g, q, kin = values.shape
    v = values.permute(1, 0, 2).reshape(q, g * kin)
    i = indices.permute(1, 0, 2).reshape(q, g * kin)
    # order by (score desc, index asc): sort by index first, then stable by score
    o1 = torch.sort(i, dim=1, stable=True)[1]
    v, i = torch.gather(v, 1, o1), torch.gather(i, 1, o1)
    o2 = torch.sort(v, dim=1, descending=True, stable=True)[1][:, :k]
    return torch.gather(v, 1, o2).contiguous(), torch.gather(i, 1, o2).contiguous()


# --------------------------------------------------------------------------------------------
# get_similarity: code/search_image.py:105-117
# --------------------------------------------------------------------------------------------
def get_similarity(features: torch.Tensor, targets: np.ndarray, label: int, ref_feature: torch.Tensor):
    """scores = 100 * features @ ref_feature.t(); split by targets == label."""
    with torch.no_grad():
        similarity = 100. * features.cpu() @ ref_feature.cpu().t()
        scores = similarity.numpy()
        pos_mask = (targets == label)
        neg_mask = (targets != label)
        return scores[pos_mask], scores[neg_mask]


# --------------------------------------------------------------------------------------------
# query construction arithmetic: code/search_image.py:310-318 (outlier_filter, after the CLIP
# forward) and :387 (mix with the text embedding)
# --------------------------------------------------------------------------------------------
def outlier_filter_features(image_features: np.ndarray) -> torch.Tensor:
    center = np.mean(image_features, axis=0)
    cos_distances = 1 - image_features @ center
    keep_mask = cos_distances <= np.percentile(cos_distances, 95)
    return torch.tensor(np.mean(image_features[keep_mask], axis=0))


# --------------------------------------------------------------------------------------------
# eval_threshold / find_thresholds: code/search_image.py:39-79 (plotting at :81-102 omitted)
# --------------------------------------------------------------------------------------------
def eval_threshold(pos_res, neg_res, threshold):
    pos_res = np.array(pos_res)
    neg_res = np.array(neg_res)
    tp = np.sum(pos_res >= threshold)   # reference uses the builtin sum over a bool array
    fp = np.sum(neg_res >= threshold)
    fn = np.sum(pos_res < threshold)
    with np.errstate(divide="ignore", invalid="ignore"):
        precision = tp / (tp + fp)
        recall = tp / (tp + fn)
        f1_score = 2 * precision * recall / (precision + recall)
    return f1_score, precision, recall


def find_thresholds(pos_res, neg_res, n_points: int = 200, grid: str = "full"):
    """Returns (best_f1, best_threshold, best_precision, best_recall, thresholds, f1_scores);
    the reference returns best_f1 only (:103) and prints the rest.  grid="overlap": the grid of
    code/main_custom.py:46-50 (overlap range of the two score sets, int(10 * width) points)."""
    if grid == "overlap":
        min_val = max(min(pos_res), min(neg_res))
        max_val = min(max(pos_res), max(neg_res))
        thresholds = np.linspace(min_val, max_val, int((max_val - min_val) * 10))
    else:
        min_val = min(min(pos_res), min(neg_res))
        max_val = max(max(pos_res), max(neg_res))
        thresholds = np.linspace(min_val, max_val, n_points)
    best = (0., 0., 0., 0.)
    f1s = []
    for t in thresholds:
        f1, p, r = eval_threshold(pos_res, neg_res, t)
        f1s.append(f1)
        if f1 > best[0]:          # first strict maximum wins (:74); NaN never wins
            best = (f1, t, p, r)
    return best[0], best[1], best[2], best[3], thresholds, np.array(f1s)


# --------------------------------------------------------------------------------------------
# evaluate_thresholds: CLIP/lab3.py:39-65 (same in CLIP-Chinese/lab_chinese.py, CLIP/union_dataset.py:46)
# --------------------------------------------------------------------------------------------
def lab_evaluate_thresholds(similarities, thresholds, positive_class, negative_class):
    rel = [it for it in similarities if it["true_label"] in [positive_class, negative_class]]
    sim = np.array([it["similarity"] for it in rel], dtype=np.float64)
    is_pos = np.array([it["true_label"] == positive_class for it in rel], dtype=bool)
    total_pos, total_neg = int(is_pos.sum()), int((~is_pos).sum())
    results = []
    for threshold in thresholds:
        TP = int(np.sum((sim >= threshold) & is_pos))
        FP = int(np.sum((sim >= threshold) & ~is_pos))
        FN, TN = total_pos - TP, total_neg - FP
        precision = TP / (TP + FP) if (TP + FP) > 0 else 0
        recall = TP / (TP + FN) if (TP + FN) > 0 else 0
        f1 = 2 * precision * recall / (precision + recall) if (precision + recall) > 0 else 0
        results.append({"threshold": threshold, "precision": precision, "recall": recall, "f1": f1,
                        "TP": TP, "FP": FP, "TN": TN, "FN": FN})
    return results


# --------------------------------------------------------------------------------------------
# near-duplicate self-join (BASELINE.json north_star; SURVEY.md M2, 8c):
#   triu((G @ G.T) >= tau, 1).nonzero()   -- row-major nonzero == lexicographic (i, j)
# --------------------------------------------------------------------------------------------
def lab_process_images(image_features: torch.Tensor, text_features: dict, classes, labels, paths, batch: int = 64):
    """The similarity loop of CLIP/union_dataset.py:247-260 (`process_images`; the same lines are
    CLIP/lab3.py:108-117 and CLIP-Chinese/lab_chinese.py:116-120) on features that have already left
    the image tower: per batch of `batch` images (lab3.py:73) normalise the rows
    (`feats / feats.norm(dim=1, keepdim=True)`), then class by class `feats @ text_features[cls].t()`;
    items whose label is "error" are skipped.  Same batching as the reference, so the fp32 CPU
    results are bit-identical to the recorded golden on the CPU it was recorded on."""
    out = {cls: [] for cls in classes}
    for lo in range(0, image_features.shape[0], batch):
        feats = image_features[lo:lo + batch].float()
        feats = feats / feats.norm(dim=1, keepdim=True)
        for cls in classes:
            sims = (feats @ text_features[cls].t()).squeeze().cpu().numpy()
            for s, lab, p in zip(np.atleast_1d(sims), labels[lo:lo + batch], paths[lo:lo + batch]):
                if lab != "error":
                    out[cls].append({"similarity": float(s), "true_label": lab, "file_path": p})
    return out


def dedup_pairs(emb: torch.Tensor, threshold: float, block: int = 4096) -> torch.Tensor:
    g = _gallery_f32(emb)
    n = g.shape[0]
    out = []
    for i0 in range(0, n, block):
        gi = g[i0:i0 + block]
        for j0 in range(i0, n, block):
            s = gi @ g[j0:j0 + block].t()
            hit = s >= threshold
            ii, jj = hit.nonzero(as_tuple=True)
            ii = ii + i0
            jj = jj + j0
            keep = ii < jj
            if keep.any():
                out.append(torch.stack([ii[keep], jj[keep]], dim=1))
    if not out:
        return torch.empty((0, 2), dtype=torch.int64)
    p = torch.cat(out, dim=0)
    key = p[:, 0] * n + p[:, 1]
    return p[torch.argsort(key)].contiguous()


def greedy_keep_first(n: int, pairs: Iterable[tuple[int, int]], order: list[int]):
    """Greedy first-keeper clustering of tool/find_repeated_in_same_folder.py:76-95: walk items in
    `order`; an item similar to an already kept representative is a duplicate of the FIRST such
    representative (in keeping order), otherwise it becomes a representative.
    Returns (representatives, [(dup, original)]) as item ids."""
    adj = [set() for _ in range(n)]
    for i, j in pairs:
        adj[int(i)].add(int(j))
        adj[int(j)].add(int(i))
    reps: list[int] = []
    dups: list[tuple[int, int]] = []
    for item in order:
        hit = None
        for r in reps:
            if r in adj[item]:
                hit = r
                break
        if hit is None:
            reps.append(item)
        else:
            dups.append((item, hit))
    return reps, dups


# --------------------------------------------------------------------------------------------
# exact-duplicate hash join: tool/find_repeated.py:6-19, 35-71
# --------------------------------------------------------------------------------------------
def image_md5(path: str):
    from PIL import Image
    try:
        with Image.open(path) as img:
            return hashlib.md5(img.convert("RGB").tobytes()).hexdigest()
    except Exception:
        return None


def get_all_images(folder_path: str) -> list[str]:
    """tool/find_repeated.py:21-33."""
    exts = {'.jpg', '.jpeg', '.png', '.bmp', '.gif', '.tiff'}
    found = []
    for root, _, files in os.walk(folder_path):
        for filename in files:
            if os.path.splitext(filename)[1].lower() in exts:
                found.append(os.path.join(root, filename))
    return found


def exact_duplicates(reference_folder: str, delete_folder: str):
    """The join of find_repeated.py:47-69 without the os.remove side effect:
    returns ([(dup_path, ref_path)], [kept], n_ref, n_del)."""
    ref_images = get_all_images(reference_folder)
    del_images = get_all_images(delete_folder)
    table = {}
    for p in ref_images:
        h = image_md5(p)
        if h:
            table[h] = p
    dup, kept = [], []
    for p in del_images:
        h = image_md5(p)
        if h and h in table:
            dup.append((p, table[h]))
        else:
            kept.append(p)
    return dup, kept, len(ref_images), len(del_images)


# --------------------------------------------------------------------------------------------
# synthetic data of the BASELINE configs (SURVEY.md section 8d) -- shared by tests and bench
# --------------------------------------------------------------------------------------------
def synthetic_gallery(n: int, d: int, seed: int = 0, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """randn rows, L2-normalised in fp32, cast to `dtype` (C2/C4: the bf16 tensor IS the gallery)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g, dtype=torch.float32)
    x = l2_normalize(x)
    return x.to(dtype)


def synthetic_queries(q: int, d: int, seed: int = 1) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return torch.randn(q, d, generator=g, dtype=torch.float32)


def synthetic_dedup(n: int, d: int, dup_frac: float = 0.01, noise: float = 0.1, seed: int = 0):
    """C3 data: randn base rows; a fraction re-planted as row_i + noise * randn / sqrt(d) * ...
    (cos ~ 0.995) so that nothing lies near tau = 0.95; rows unit-normalised fp32.
    Returns (embeddings [n, d] fp32, planted [(i, j)] with i < j)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g, dtype=torch.float32)
    n_dup = int(n * dup_frac)
    perm = torch.randperm(n, generator=g)
    src = perm[:n_dup]
    dst = perm[n_dup:2 * n_dup]
    x[dst] = x[src] + noise * torch.randn(n_dup, d, generator=g, dtype=torch.float32)
    x = l2_normalize(x)
    planted = sorted((min(int(a), int(b)), max(int(a), int(b))) for a, b in zip(src, dst))
    return x, planted
