"""B200-native retrieval hot path of
chy980959830/Multi-Modal-Retrieval-System-Image-Search-and-Data-Governance.

Import as `mmrs_b200` (see ../mmrs_b200.py).  The public names mirror the reference's module-level
functions for this path (same names, positional order and return tuples):

    code/search_image.py   get_similarity, construct_dataset, eval_threshold, find_thresholds,
                           get_image_text_features, get_cluster_features (+ their arithmetic on encoded
                           features: image_text_prototypes, cluster_prototype, outlier_filter_features)
    code/utils.py          cls_acc (top-k of an existing score matrix: topk_of_scores)
    code/merge_dataset.py  cosine_similarity_scores (logit_scale * F.cosine_similarity, :275-278)
    tool/find_repeated.py  get_all_images, find_and_remove_duplicate_images
    tool/find_repeated_in_same_folder.py
                           find_and_remove_duplicate_images (same-folder form)
    tool/delete repeated.py
                           detect_and_remove_cross_set_duplicates
    CLIP/lab3.py (and lab_chinese.py, union_dataset.py)
                           evaluate_thresholds, score_classes (the per-class similarity loop as one call)
    CLIP/union_dataset.py  calc_combined_metrics
    code/main_custom.py    find_thresholds(..., grid="overlap") (:46-91), get_similarity_from_matrix (:93-105)

plus the tensor-level entry points they sit on: search_topk, full_scores, find_duplicate_pairs,
DeviceGallery, ShardedGallery, RowFilter (row-filtered search_topk: leave rows out per call) and
RowLabels (label-conditioned search_topk: each query searches the rows of its own class, or of every other)
and best_thresholds (the best-F1 threshold of every class prototype of a batch, find_thresholds per class) and
search_range (every row at or above a per-query threshold, in CSR form) and resolve_duplicates / deduplicate
(greedy_first_keeper's keep / delete decision on the device: the representative of every row) and RefineStore
(refined search_topk: a compact gallery's candidates rescored against full-precision rows in host or device memory).  Everything computes through the C-ABI CUDA library
(include/mmrs_b200.h); there is no CPU path -- without a B200 the calls raise.
"""
from . import _cabi  # noqa: F401  (fails loudly when the CUDA library is missing)
from .gallery import DeviceGallery, load_feature_cache
from .refine import RefineStore
from .row_filter import RowFilter
from .row_labels import RowLabels
from .search import (best_threshold_on_device, calc_combined_metrics, cls_acc, cluster_prototype, construct_dataset,
                     cosine_similarity_scores, eval_threshold, evaluate_thresholds, find_thresholds, full_scores,
                     get_cluster_features, get_image_text_features, get_similarity, get_similarity_from_matrix,
                     image_text_prototypes, mix_image_text_query, outlier_filter_features, score_classes, search_topk,
                     threshold_sweep_counts, topk_of_scores)
from .dedup import (calculate_image_hash, deduplicate, detect_and_remove_cross_set_duplicates,
                    find_and_remove_duplicate_images, find_duplicate_pairs, find_and_remove_near_duplicate_images,
                    get_all_images, greedy_first_keeper, resolve_duplicates)
from .sharded import ShardedGallery, shard_bounds
from .range_search import search_range
from .thresholds import best_thresholds

__all__ = [
    "DeviceGallery", "RefineStore", "RowFilter", "RowLabels", "ShardedGallery", "best_threshold_on_device", "best_thresholds", "calc_combined_metrics", "calculate_image_hash", "cls_acc",
    "cluster_prototype", "construct_dataset", "cosine_similarity_scores", "deduplicate", "get_cluster_features", "get_image_text_features",
    "image_text_prototypes", "topk_of_scores",
    "detect_and_remove_cross_set_duplicates", "evaluate_thresholds", "eval_threshold", "find_thresholds",
    "find_and_remove_duplicate_images", "find_and_remove_near_duplicate_images",
    "find_duplicate_pairs", "full_scores", "get_all_images", "get_similarity", "get_similarity_from_matrix",
    "greedy_first_keeper", "load_feature_cache", "mix_image_text_query", "outlier_filter_features", "resolve_duplicates",
    "score_classes", "search_range", "search_topk", "shard_bounds",
    "threshold_sweep_counts",
]
