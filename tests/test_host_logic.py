"""Host-side logic that needs no GPU: phase schedule, sharding arithmetic, greedy clustering,
file listing, gallery-cache readers."""
import ctypes
import os
import pickle
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "multi-modal-retrieval-system-image-search-and-data-governance_b200"


@pytest.fixture(scope="module")
def plan_lib(tmp_path_factory):
    """plan.h compiled with g++ behind a tiny C shim."""
    d = tmp_path_factory.mktemp("plan")
    src = d / "shim.cpp"
    src.write_text(f'''
#include "{PKG / "csrc" / "plan.h"}"
extern "C" int plan(long long n, int k, int ratio, int dense, int* out) {{
  mmrs::SearchPlan p = mmrs::make_search_plan(n, k, 128, ratio, dense);
  out[0] = p.n_tiles; out[1] = p.n_phases; out[2] = p.dense_rows; out[3] = p.cap;
  for (int i = 0; i < p.n_phases; ++i) {{ out[4+3*i] = p.phase[i].inc; out[5+3*i] = p.phase[i].exc; out[6+3*i] = p.phase[i].n_sel; }}
  return 0;
}}
// the visited-tile / CTA-pair work-unit enumeration the scan kernel uses (plan.h)
extern "C" int visited(int inc, int exc, int n_sel, int* out_j) {{
  const int R = mmrs::plan_exclusion_ratio(inc, exc), n = mmrs::plan_n_visited(n_sel, R);
  for (int v = 0; v < n; ++v) out_j[v] = mmrs::plan_visited_to_j(v, R);
  return n;
}}
extern "C" int pair_units(int inc, int exc, int n_sel, int n_chunks, int rank, int* out) {{   // out: [u][j, chunk, valid]
  const int R = mmrs::plan_exclusion_ratio(inc, exc), n = mmrs::plan_n_visited(n_sel, R);
  const int units = mmrs::plan_pair_units(n, n_chunks);
  for (int u = 0; u < units; ++u) {{
    mmrs::PairUnit pu = mmrs::plan_pair_unit(u, rank, n_chunks, n, R);
    out[3*u] = pu.j; out[3*u+1] = pu.chunk; out[3*u+2] = pu.valid;
  }}
  return units;
}}''')
    so = d / "shim.so"
    subprocess.run(["g++", "-O1", "-shared", "-fPIC", str(src), "-o", str(so)], check=True)
    return ctypes.CDLL(str(so))


def get_plan(lib, n, k, ratio=3, dense=32):
    out = (ctypes.c_int * 64)()
    lib.plan(ctypes.c_longlong(n), k, ratio, dense, out)
    phases = [(out[4 + 3 * i], out[5 + 3 * i], out[6 + 3 * i]) for i in range(out[1])]
    return dict(n_tiles=out[0], dense_rows=out[2], cap=out[3], phases=phases)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 16384, 16385, 20000, 70000, 1_000_000, 12_500_000, 100_000_000])
@pytest.mark.parametrize("k", [1, 10, 100, 1024])
def test_plan_visits_every_tile_exactly_once(plan_lib, n, k):
    p = get_plan(plan_lib, n, k)
    T = p["n_tiles"]
    assert T == (n + 127) // 128
    seen = np.zeros(T, dtype=np.int32)
    for inc, exc, n_sel in p["phases"]:
        t = np.arange(n_sel, dtype=np.int64) * inc
        assert t.max() < T and n_sel == (T + inc - 1) // inc
        if exc:
            t = t[t % exc != 0]
        np.add.at(seen, t, 1)
    assert (seen == 1).all()
    # phase 0 is dense and unfiltered, holds >= k valid rows, and fits the list
    inc0, exc0, n0 = p["phases"][0]
    assert exc0 == 0 and p["dense_rows"] == n0 * 128 <= p["cap"]
    valid0 = sum(min(128, n - j * inc0 * 128) for j in range(n0))
    assert valid0 >= min(k, n)
    # later phases: expected appends k * ratio stay far below the capacity
    for (inc_prev, _, _), (inc, _, _) in zip(p["phases"], p["phases"][1:]):
        assert inc_prev % inc == 0 and 4 * (k + 32) * (inc_prev // inc) <= p["cap"]


@pytest.mark.parametrize("n", [129, 16385, 70_001, 1_000_000, 12_500_000])
def test_visited_tiles_and_cta_pair_units(plan_lib, n):
    """The dense enumeration of a phase's visited tiles, and the (tile pair, query chunk) work units
    of the CTA-pair scan: every (visited tile, chunk) is read by exactly one CTA."""
    for dense in (32, 64):
        p = get_plan(plan_lib, n, 100, dense=dense)
        for inc, exc, n_sel in p["phases"]:
            want = [j for j in range(n_sel) if not (exc and (j * inc) % exc == 0)]
            buf = (ctypes.c_int * max(1, n_sel))()
            got_n = plan_lib.visited(inc, exc, n_sel, buf)
            assert got_n == len(want) and list(buf[:got_n]) == want
            if n_sel > 20_000:
                continue                      # the unit check below is O(units) in Python
            for n_chunks in (1, 3, 4):
                units = (len(want) + 1) // 2 * n_chunks
                seen = {}
                for rank in (0, 1):
                    out = (ctypes.c_int * (3 * max(1, units)))()
                    assert plan_lib.pair_units(inc, exc, n_sel, n_chunks, rank, out) == units
                    for u in range(units):
                        j, chunk, valid = out[3 * u], out[3 * u + 1], out[3 * u + 2]
                        assert j in want and 0 <= chunk < n_chunks      # even an unread half tile is a real tile
                        if valid:
                            assert (j, chunk) not in seen
                            seen[(j, chunk)] = (u, rank)
                assert len(seen) == len(want) * n_chunks
                # the chunks of one tile pair are consecutive units: neighbouring pairs share the tile in L2
                for (j, chunk), (u, rank) in seen.items():
                    assert u % n_chunks == chunk and want[2 * (u // n_chunks) + rank] == j


def test_shard_bounds(mm):
    for n, w in [(1_000_000, 8), (100_000_000, 8), (1000, 3), (5, 4), (128, 2), (129, 2)]:
        b = mm.shard_bounds(n, w)
        assert len(b) == w and b[0][0] == 0 and b[-1][1] == n
        assert all(lo % 128 == 0 or lo == n for lo, _ in b)
        assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
    from mmrs_b200.sharded import triangle_bounds
    n = 1_000_000
    tb = triangle_bounds(n, 8)
    assert tb[0][0] == 0 and tb[-1][1] == n
    areas = [sum(n - i for i in (lo, hi - 1)) * (hi - lo) / 2 for lo, hi in tb]
    assert max(areas) / min(areas) < 1.02      # equal pair counts per rank


def test_greedy_first_keeper_matches_oracle(mm, oracle):
    rng = np.random.default_rng(0)
    for n, m in [(10, 12), (200, 300), (1000, 5000)]:
        pairs = rng.integers(0, n, size=(m, 2))
        pairs = np.unique(np.sort(pairs[pairs[:, 0] != pairs[:, 1]], axis=1), axis=0)
        order = rng.permutation(n).tolist()
        assert mm.greedy_first_keeper(n, pairs, order) == oracle.greedy_keep_first(n, pairs.tolist(), order)


def test_get_all_images_matches_oracle(mm, oracle, tmp_path):
    from golden_inputs import dedup_image_set
    dedup_image_set(str(tmp_path))
    assert mm.get_all_images(str(tmp_path)) == oracle.get_all_images(str(tmp_path))
    assert not any(p.endswith(".webp") for p in mm.get_all_images(str(tmp_path)))


def test_load_feature_cache(mm, tmp_path):
    d = {f"cls/{i}.jpg": np.random.default_rng(i).standard_normal(16).astype(np.float16) for i in range(5)}
    with open(tmp_path / "features.pkl", "wb") as f:
        pickle.dump(d, f)                              # the format of search_image.py:159-160
    feats, keys = mm.load_feature_cache(str(tmp_path / "features.pkl"))
    assert keys == list(d) and feats.shape == (5, 16) and feats.dtype == torch.float32
    np.testing.assert_array_equal(feats.numpy(), np.stack([d[k] for k in keys]).astype(np.float32))
    torch.save(torch.randn(7, 16), tmp_path / "test_f.pt")   # utils.py:150
    feats, keys = mm.load_feature_cache(str(tmp_path / "test_f.pt"))
    assert keys is None and feats.shape == (7, 16)


def test_construct_dataset_host_logic(mm, tmp_path, monkeypatch):
    import mmrs_b200.search as S
    names = ["a", "b"]
    for c in names:
        os.makedirs(tmp_path / c)
        for i in range(3):
            (tmp_path / c / f"{i}.jpg").write_bytes(b"x")
    monkeypatch.setattr(S, "class_names", names)
    monkeypatch.setattr(S, "class_to_idx", {"a": 0, "b": 1})
    monkeypatch.setattr(S, "dataset_path", str(tmp_path))
    fd = {f"{c}/{i}.jpg": np.full(4, ci * 10 + i, dtype=np.float32) for ci, c in enumerate(names) for i in range(3)}
    feats, targets = S.construct_dataset(fd, ["1.jpg"], "b")
    assert feats.shape == (5, 4) and targets.tolist().count(1) == 2 and targets.tolist().count(0) == 3
    assert 11.0 not in feats[:, 0].tolist()


def test_query_construction_helpers(mm, oracle):
    rng = np.random.default_rng(4)
    f = rng.standard_normal((10, 64)).astype(np.float32)
    f[3] = -f[0]                                   # an outlier: far from the mean direction
    f /= np.linalg.norm(f, axis=1, keepdims=True)
    want = oracle.outlier_filter_features(f)
    got = mm.outlier_filter_features(torch.from_numpy(f))
    assert torch.equal(got, want)
    assert abs(float(got.norm()) - 1.0) > 1e-3     # un-normalised, as in the reference (M3)
    text = torch.from_numpy(rng.standard_normal(64).astype(np.float32))
    assert torch.equal(mm.mix_image_text_query(got, text), (want + text) / 2)


def _union_gold():
    import json
    from conftest import GOLDEN
    g = json.loads((GOLDEN / "union_golden.json").read_text())
    sims = {k: {cls: [{"similarity": a, "true_label": b, "file_path": c} for a, b, c in v] for cls, v in d.items()}
            for k, d in g["sims"].items()}
    return sims, g["combined"]


def test_calc_combined_metrics_matches_reference(mm):
    """CLIP/union_dataset.py:133-231, golden recorded from the reference function."""
    from golden_inputs import union_inputs
    u = union_inputs()
    sims, want = _union_gold()
    got = mm.calc_combined_metrics(sims["en"], sims["cn"], u["en_threshs"], u["cn_threshs"],
                                   u["en_pos"], u["en_neg"], u["cn_pos"], u["cn_neg"])
    assert got == want
    assert all(r["TP"] > 0 and r["FN"] > 0 for r in want) and any(r["FP"] > 0 for r in want)   # a non-trivial fixture


def test_score_classes_host_logic(mm, oracle):
    """score_classes = the per-class loop of the lab scripts as one scoring call; here the scoring call
    is the oracle's, so this pins the normalisation, the class/row bookkeeping and the "error" filter."""
    from golden_inputs import union_inputs
    u = union_inputs()
    sims, _ = _union_gold()
    for key, pos in (("en", u["en_pos"]), ("cn", u["cn_pos"])):
        feats, text, labels, paths = u[key]
        got = mm.score_classes(feats, text, pos, labels, paths, scorer=lambda q, g, **kw: oracle.full_scores(q, g, **kw))
        assert list(got) == pos
        for cls in pos:
            want = sims[key][cls]
            assert [(it["true_label"], it["file_path"]) for it in got[cls]] == [(it["true_label"], it["file_path"]) for it in want]
            np.testing.assert_allclose([it["similarity"] for it in got[cls]], [it["similarity"] for it in want], atol=1e-6, rtol=0)
    assert mm.score_classes(torch.zeros(0, 8), {}, [], [], []) == {}


def test_get_similarity_from_matrix_matches_reference(mm):
    """code/main_custom.py:93-105 (column slice of a similarity matrix), golden from the reference function."""
    from conftest import GOLDEN
    from golden_inputs import similarity_inputs
    g = np.load(GOLDEN / "main_custom_golden.npz")
    feats, targets, label, _ = similarity_inputs()["small"]
    sim = 100.0 * feats @ feats[:7].t()
    pos, neg = mm.get_similarity_from_matrix(sim, torch.from_numpy(targets), label)
    np.testing.assert_array_equal(pos, g["sliced_pos"])
    np.testing.assert_array_equal(neg, g["sliced_neg"])
    pos2, neg2 = mm.get_similarity_from_matrix(sim.numpy(), targets, label)
    np.testing.assert_array_equal(pos2, pos) and np.testing.assert_array_equal(neg2, neg)


# ---- pinned against outputs of the reference's own function bodies (tests/golden/make_golden.py) ----------------
def _greedy_case(tmp_path):
    """The same-folder greedy loop's inputs as (n, pairs, order by file size desc, unreadable ids, golden)."""
    import json
    from conftest import GOLDEN
    from golden_inputs import greedy_inputs
    gold = json.loads((GOLDEN / "same_folder_golden.json").read_text())
    folder, ids, similar, unreadable = greedy_inputs(str(tmp_path))
    paths = sorted(ids, key=lambda p: os.path.getsize(p), reverse=True)      # find_repeated_in_same_folder.py:73
    order = [ids[p] for p in paths if ids[p] not in unreadable]                # hash None -> skipped (:78)
    pairs = sorted(tuple(sorted(s)) for s in similar)
    return len(ids), pairs, order, gold


def test_greedy_walk_matches_reference_same_folder_loop(mm, oracle, tmp_path):
    """greedy_first_keeper (product) and greedy_keep_first (oracle) against the result tuple recorded from
    tool/find_repeated_in_same_folder.py:56-106 run with stub hash functions."""
    n, pairs, order, gold = _greedy_case(tmp_path)
    for fn in (lambda: mm.greedy_first_keeper(n, np.array(pairs), order), lambda: oracle.greedy_keep_first(n, pairs, order)):
        reps, dups = fn()
        assert reps == gold["representatives"]
        assert [list(d) for d in dups] == gold["deleted"]
    assert gold["total"] == n


def test_same_folder_wrapper_matches_reference_loop(mm, tmp_path, monkeypatch):
    """The whole same-folder wrapper (listing, size sort, skip of unreadable files, greedy walk, deletion,
    result tuple) against the recorded reference run: the pair predicate is injected where the CUDA
    self-join sits, everything else is the product code."""
    import mmrs_b200.dedup as D
    from golden_inputs import greedy_inputs
    import json
    from conftest import GOLDEN
    gold = json.loads((GOLDEN / "same_folder_golden.json").read_text())
    folder, ids, similar, unreadable = greedy_inputs(str(tmp_path))

    def embed(paths):                                   # "embedding" = the id; unreadable files flagged
        ok = np.array([ids[p] not in unreadable for p in paths])
        return torch.tensor([[float(ids[p])] for p, good in zip(paths, ok) if good]), ok

    def fake_pairs(emb, threshold, **kw):               # stands in for the GPU self-join
        idv = [int(v) for v in emb[:, 0].tolist()]
        out = [(i, j) for i in range(len(idv)) for j in range(i + 1, len(idv)) if frozenset((idv[i], idv[j])) in similar]
        return torch.tensor(out, dtype=torch.int64).reshape(-1, 2)

    monkeypatch.setattr(D, "find_duplicate_pairs", fake_pairs)
    deleted, refs, total = D.find_and_remove_duplicate_images(folder, cosine_threshold=0.95, embed=embed)
    assert [[ids[a], ids[b]] for a, b in deleted] == gold["deleted"]
    assert [ids[p] for p in refs] == gold["representatives"] and total == gold["total"]
    assert sorted(ids[p] for p in D.get_all_images(folder)) == gold["remaining"]


def test_query_builders_match_reference(mm, oracle, tmp_path, monkeypatch):
    """get_image_text_features (:119-140), get_cluster_features (:185-232) and the outlier_filter arithmetic
    (:310-318) against outputs of the reference functions on the same on-disk samples and stand-in encoder."""
    import contextlib, io
    import mmrs_b200.search as S
    from conftest import GOLDEN
    from golden_inputs import query_builder_setup
    g = np.load(GOLDEN / "query_builders_golden.npz")
    dataset_path, tower, preprocess, class_embeddings, class_to_idx, samples = query_builder_setup(str(tmp_path))
    monkeypatch.setattr(S, "dataset_path", dataset_path)
    monkeypatch.setattr(S, "class_to_idx", class_to_idx)
    for cls in samples:
        img_f, img_txt_f = S.get_image_text_features(tower, preprocess, class_embeddings.clone(), samples[cls], cls)
        np.testing.assert_array_equal(img_f.numpy(), g[f"{cls}_image_features"])
        np.testing.assert_array_equal(img_txt_f.numpy(), g[f"{cls}_image_text_features"])
        feats = S._encode_samples(tower, preprocess, samples[cls], cls)
        unit = (feats / feats.norm(dim=-1, keepdim=True)).numpy()
        np.testing.assert_array_equal(S.outlier_filter_features(unit).numpy(), g[f"{cls}_outlier_filter"])
        np.testing.assert_array_equal(oracle.outlier_filter_features(unit).numpy(), g[f"{cls}_outlier_filter"])
    for cls, shots in (("alpha", 5), ("beta", 8)):
        np.random.seed(0)
        with contextlib.redirect_stdout(io.StringIO()):
            got = S.get_cluster_features(tower, preprocess, samples[cls], shots, cls)
        np.testing.assert_allclose(got.numpy(), g[f"{cls}_cluster_features"], atol=1e-7, rtol=0)


def test_destructive_wrappers_validate_thresholds_without_a_gpu(mm, tmp_path):
    """Argument checks run before anything touches the GPU or the files."""
    (tmp_path / "x.png").write_bytes(b"not an image")
    for bad in (0, 5, 0.5, 1.01, -1):
        with pytest.raises(ValueError):
            mm.find_and_remove_duplicate_images(str(tmp_path), bad)
        with pytest.raises(ValueError):
            mm.find_and_remove_duplicate_images(str(tmp_path), cosine_threshold=bad)
        with pytest.raises(ValueError):
            mm.find_and_remove_duplicate_images(str(tmp_path), str(tmp_path), threshold=bad)
    with pytest.raises(ValueError):
        mm.detect_and_remove_cross_set_duplicates(str(tmp_path), str(tmp_path), 8, 3)
    with pytest.raises(TypeError):
        mm.find_and_remove_duplicate_images(str(tmp_path), cosine_threshold="0.95")
    assert os.path.exists(tmp_path / "x.png")


def test_upload_cache_is_keyed_on_identity_not_address(mm, monkeypatch):
    """get_similarity's one-entry upload cache must not serve a stale gallery to a NEW tensor that happens
    to reuse a freed tensor's address (same shape, same dtype, _version 0)."""
    import mmrs_b200.search as S
    made = []

    class FakeGallery:
        def __init__(self, features, mode=None):
            made.append(features)

    monkeypatch.setattr(S, "DeviceGallery", FakeGallery)
    S._last_upload.clear()
    a = torch.randn(64, 8)
    g1 = S._resident(a, None)
    assert S._resident(a, None) is g1 and len(made) == 1           # same object, same version: reused
    a.add_(1.0)
    assert S._resident(a, None) is not g1 and len(made) == 2       # in-place edit: re-uploaded
    ptr = a.data_ptr()
    del a
    b = torch.randn(64, 8)                                         # may or may not land on the old address
    g3 = S._resident(b, None)
    assert made[-1] is b and len(made) == 3
    arr = np.zeros((4, 8), dtype=np.float32)
    S._resident(arr, None); S._resident(arr, None)
    assert len(made) == 5                                          # numpy inputs are never cached
    S._last_upload.clear()
    del ptr, g3


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): one JSON line with the contract's keys,
    the same workload description as our arm, honouring --steps / --warmup, no GPU needed."""
    import json
    import sys
    root = Path(__file__).resolve().parent.parent
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--rows", "30000", "--dim", "64",
                          "--batch", "4", "--k", "5", "--steps", "3", "--warmup", "2", "--gpus", "1"],
                         capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "top-k queries/sec" and d["unit"] == "queries/s"
    assert d["steps"] == 3 and d["warmup"] == 2 and d["n_gpus"] == 1 and d["higher_is_better"] is True
    assert d["scaling"] == "strong" and d["vs_baseline"] is None and d["value"] > 0
    assert d["config"]["global_rows"] == 30000 and d["config"]["queries_per_step"] == 4 and d["config"]["k"] == 5
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # ranks other than 0 print nothing and exit 0 (torchrun launches the arm on every rank)
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=root, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_rejects_zero_steps_and_dumps_of_the_reference_arm():
    import sys
    root = Path(__file__).resolve().parent.parent
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, str(root / "bench.py")] + extra, capture_output=True, text=True,
                             timeout=120, cwd=root)
        assert out.returncode == 2 and out.stdout == "", out.stderr[-2000:]


def test_bench_dump_outputs_full_and_sampled(tmp_path, monkeypatch):
    """dump_outputs keeps the lists whole below the size limit and a fixed, seeded row sample above it."""
    import bench
    gen = torch.Generator().manual_seed(0)
    v = torch.randn(300, 20, generator=gen)
    i = torch.randint(0, 1 << 40, (300, 20), generator=gen)
    bench.dump_outputs(tmp_path / "full", v, i)
    assert sorted(p.name for p in (tmp_path / "full").iterdir()) == ["topk_indices.npy", "topk_values.npy"]
    got_v, got_i = np.load(tmp_path / "full" / "topk_values.npy"), np.load(tmp_path / "full" / "topk_indices.npy")
    assert got_v.dtype == np.float32 and got_i.dtype == np.float64
    np.testing.assert_array_equal(got_v, v.numpy())
    np.testing.assert_array_equal(got_i.astype(np.int64), i.numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4096 + 100 * (20 * 12 + 8))
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, v, i)
        assert sum(p.stat().st_size for p in (tmp_path / d).iterdir()) <= bench.DUMP_LIMIT_BYTES
    rows = np.load(tmp_path / "a" / "query_rows.npy")
    assert rows.shape == (100,) and np.all(np.diff(rows) > 0)
    for name in ("query_rows", "topk_values", "topk_indices"):
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "topk_values.npy"), v.numpy()[rows.astype(np.int64)])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "topk_indices.npy").astype(np.int64),
                                  i.numpy()[rows.astype(np.int64)])


def test_bench_traffic_table_is_keyed_by_shape():
    import json
    root = Path(__file__).resolve().parent.parent
    table = json.loads((root / "profiles" / "traffic.json").read_text())
    keys = [k for k in table if not k.startswith("_")]
    assert keys and all("@" in k and "x" in k.split("@")[1] and "q" in k.split("@")[1] for k in keys)
    for k in keys:
        assert table[k]["dram_bytes_read"] > 0 and (root / table[k]["source"].split(" ")[0]).exists(), k


def test_calculate_image_hash_matches_reference(mm, tmp_path):
    """calculate_image_hash (the exact predicate that confirms deletions) against the MD5s recorded from the
    reference's tool/find_repeated.py:6-19 on the same generated image set; unreadable file -> None."""
    import json
    from conftest import GOLDEN
    from golden_inputs import dedup_image_set
    gold = json.loads((GOLDEN / "find_repeated_golden.json").read_text())
    dedup_image_set(str(tmp_path))
    got = {os.path.relpath(p, tmp_path): mm.calculate_image_hash(p) for p in sorted(mm.get_all_images(str(tmp_path)))}
    assert got == gold["hashes"]
    assert got["delete/broken.png"] is None
    assert got["reference/sub/c.png"] == got["reference/sub/c_again.png"] == got["delete/nested/c_copy.png"]
