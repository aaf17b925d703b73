"""The oracle against outputs of the reference's OWN functions (tests/golden/make_golden.py ran
them in the build container; the reference checkout is not needed here)."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from golden_inputs import dedup_image_set, similarity_inputs, topk_inputs


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN / "search_image_golden.npz")


def assert_same_fp32_dot_products(got, want, dot_scale, ulps=8):
    """fp32 dot products of the same expression as the recorded reference output.  On the CPU the golden
    was recorded on they are bit-identical; another CPU's BLAS kernel sums the D products of a row in
    another order.  That rounding scales with the summed products, sum |x_i y_i| <= |x| |y| = `dot_scale`,
    not with the result, so the bound is `ulps` units in the last place of `dot_scale`.  Measured on these
    inputs, in ulps of dot_scale: an AMD EPYC and a second Xeon host <= 0.5, vectorised block orders
    (4 to 64 lanes) <= 1.5, a scalar loop over D in either direction <= 6.5.  8 ulps of the ~77 here is 6.1e-5, 16x tighter than
    the 1e-3 the CUDA path is held to against the same goldens."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.dtype == want.dtype == np.float32 and got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=0, atol=ulps * np.spacing(np.float32(dot_scale)))


@pytest.mark.parametrize("name", ["small", "clip512", "taiyi768"])
def test_get_similarity_matches_reference(oracle, gold, name):
    features, targets, label, ref = similarity_inputs()[name]
    pos, neg = oracle.get_similarity(features, targets, label, ref)
    # same library, same expression: equal up to the summation order of the CPU's BLAS
    dot_scale = 100.0 * float(features.norm(dim=1).max()) * float(ref.norm())
    assert_same_fp32_dot_products(pos, gold[f"{name}_pos"], dot_scale)
    assert_same_fp32_dot_products(neg, gold[f"{name}_neg"], dot_scale)
    # full_scores restates the same product as scale * (q @ G.T): within 1e-5 * scale
    s = oracle.full_scores(ref[None], features, normalize_queries=False, scale=100.0)[0].numpy()
    np.testing.assert_allclose(s[targets == label], gold[f"{name}_pos"], atol=1e-3, rtol=0)


@pytest.mark.parametrize("name", ["small", "clip512", "taiyi768"])
def test_threshold_functions_match_reference(oracle, gold, name):
    pos, neg = gold[f"{name}_pos"], gold[f"{name}_neg"]
    for t, want in zip(gold[f"{name}_probe"], gold[f"{name}_eval"]):
        got = np.array(oracle.eval_threshold(pos, neg, t), dtype=np.float64)
        np.testing.assert_array_equal(got, want)  # nan == nan positions included
    best = oracle.find_thresholds(pos, neg)[0]
    assert best == gold[f"{name}_best_f1"]


def test_topk_matches_reference_topk(oracle):
    g = np.load(GOLDEN / "utils_topk_golden.npz")
    for name, (logits, _t) in topk_inputs().items():
        for k in (1, 3):
            v, i = oracle.topk_rows(logits, k)
            np.testing.assert_array_equal(v.numpy(), g[f"{name}_topk{k}_values"])
            ref_i = g[f"{name}_topk{k}_indices"]
            if name == "random":           # no ties: indices identical
                np.testing.assert_array_equal(i.numpy(), ref_i)
            else:
                # torch.topk leaves the order among equal scores unspecified (recorded output
                # has e.g. indices [1, 5, 4] for three equal values); the oracle's rule is index
                # ascending.  Both must select equal VALUES position by position.
                np.testing.assert_array_equal(np.take_along_axis(logits.numpy(), ref_i, 1), v.numpy())
                assert np.all(np.take_along_axis(logits.numpy(), i.numpy(), 1) == v.numpy())
                # oracle order: among equal values indices ascend
                vi = v.numpy(); ii = i.numpy()
                same = vi[:, 1:] == vi[:, :-1]
                assert np.all(ii[:, 1:][same] > ii[:, :-1][same])


def test_search_topk_blocked_equals_unblocked(oracle):
    g = oracle.synthetic_gallery(5000, 64, seed=3, dtype=torch.float32)
    q = oracle.synthetic_queries(7, 64)
    v0, i0 = oracle.topk_rows(oracle.full_scores(q, g), 20)
    v1, i1 = oracle.search_topk(q, g, 20, block_rows=777)
    assert torch.equal(i0, i1) and torch.equal(v0, v1)


def test_hand_computed_case(oracle):
    # 4 gallery rows x 3 dims, hand-checkable: q = (3, 4, 0) -> unit (0.6, 0.8, 0)
    g = torch.tensor([[1., 0, 0], [0, 1, 0], [0.6, 0.8, 0], [0, 0, 1]])
    q = torch.tensor([[3., 4, 0]])
    s = oracle.full_scores(q, g)
    np.testing.assert_allclose(s.numpy(), [[0.6, 0.8, 1.0, 0.0]], atol=1e-7)
    v, i = oracle.search_topk(q, g, 3)
    assert i.tolist() == [[2, 1, 0]]
    # exact ties (duplicate rows) fall to the lower index
    g2 = torch.cat([g, g[2:3], g[1:2]])
    v, i = oracle.search_topk(q, g2, 4)
    assert i.tolist() == [[2, 4, 1, 5]]


def test_merge_topk(oracle):
    g = oracle.synthetic_gallery(4096, 32, seed=9, dtype=torch.float32)
    g[100] = g[3000]                                 # a tie across shards
    q = oracle.synthetic_queries(5, 32)
    want_v, want_i = oracle.search_topk(q, g, 10)
    vs, is_ = [], []
    for lo in range(0, 4096, 1024):
        v, i = oracle.search_topk(q, g[lo:lo + 1024], 10)
        vs.append(v); is_.append(i + lo)
    v, i = oracle.merge_topk(torch.stack(vs), torch.stack(is_), 10)
    assert torch.equal(i, want_i) and torch.equal(v, want_v)


def test_exact_duplicates_match_reference(oracle, tmp_path):
    gold = json.loads((GOLDEN / "find_repeated_golden.json").read_text())
    ref_dir, del_dir = dedup_image_set(str(tmp_path))
    rel = lambda p: os.path.relpath(p, tmp_path)
    hashes = {rel(p): oracle.image_md5(p) for p in oracle.get_all_images(str(tmp_path))}
    assert hashes == gold["hashes"]
    dup, kept, n_ref, n_del = oracle.exact_duplicates(ref_dir, del_dir)
    assert sorted([rel(a), rel(b)] for a, b in dup) == gold["deleted"]
    assert sorted(rel(p) for p in kept) == gold["kept"]
    assert (n_ref, n_del) == (gold["n_ref"], gold["n_del"])


def test_dedup_pairs_planted(oracle):
    x, planted = oracle.synthetic_dedup(2000, 64, dup_frac=0.05, seed=2)
    pairs = oracle.dedup_pairs(x, 0.95, block=512)
    assert [tuple(p) for p in pairs.tolist()] == planted
    # guard band: nothing within 0.02 of the threshold, so the set is accumulation-order proof
    s = x @ x.t()
    iu = torch.triu_indices(2000, 2000, 1)
    vals = s[iu[0], iu[1]]
    assert not ((vals > 0.93) & (vals < 0.97)).any()


def test_greedy_keep_first(oracle):
    # chain 0-1, 1-2: walking 0,1,2 keeps 0, drops 1 (dup of 0), keeps 2 (not adjacent to 0)
    reps, dups = oracle.greedy_keep_first(3, [(0, 1), (1, 2)], [0, 1, 2])
    assert reps == [0, 2] and dups == [(1, 0)]
    reps, dups = oracle.greedy_keep_first(4, [(0, 3), (1, 3)], [1, 0, 3, 2])
    assert reps == [1, 0, 2] and dups == [(3, 1)]


def test_lab3_evaluate_thresholds_matches_reference(oracle):
    from golden_inputs import lab3_inputs
    g = np.load(GOLDEN / "lab3_golden.npz")
    sims, thresholds, pos_cls, neg_cls = lab3_inputs()
    res = oracle.lab_evaluate_thresholds(sims, thresholds, pos_cls, neg_cls)
    for key in ("threshold", "precision", "recall", "f1", "TP", "FP", "TN", "FN"):
        np.testing.assert_array_equal(np.array([r[key] for r in res], dtype=np.float64), g[key])


def test_lab_process_images_matches_reference(oracle):
    """CLIP/union_dataset.py process_images, run by make_golden.py on seeded feature batches."""
    from golden_inputs import union_inputs
    gold = json.loads((GOLDEN / "union_golden.json").read_text())["sims"]
    u = union_inputs()
    for key, pos in (("en", u["en_pos"]), ("cn", u["cn_pos"])):
        feats, text, labels, paths = u[key]
        got = oracle.lab_process_images(feats, text, pos, labels, paths)
        for cls in pos:
            assert [[it["true_label"], it["file_path"]] for it in got[cls]] == [w[1:] for w in gold[key][cls]]
            # unit image rows (normalised in the loop) times a unit text feature: dot_scale 1
            assert_same_fp32_dot_products(np.array([it["similarity"] for it in got[cls]], dtype=np.float32),
                                          np.array([w[0] for w in gold[key][cls]], dtype=np.float32),
                                          float(text[cls].norm()))


def test_overlap_grid_find_thresholds_matches_reference(oracle):
    """code/main_custom.py:46-91: the grid spans only the overlap of the two score sets."""
    from golden_inputs import overlap_grid_inputs
    g = np.load(GOLDEN / "main_custom_golden.npz")
    for name, (pos, neg) in overlap_grid_inputs().items():
        if str(g[f"{name}_raises"]):
            with pytest.raises(ValueError):
                oracle.find_thresholds(pos, neg, grid="overlap")
        else:
            assert oracle.find_thresholds(pos, neg, grid="overlap")[0] == g[f"{name}_best_f1"]
