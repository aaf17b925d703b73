"""Duplicate resolve on one GPU: resolve_duplicates against the host greedy_first_keeper on the same device pair
list (its device-to-host copy included), and deduplicate end to end against find_duplicate_pairs + the host walk.

Graphs (walk order = identity):
  c3_matching_10m   C3's planted matching: 10 M rows, 100 K pairs between two disjoint random row sets
  cliques_1m/_10m   cliques of 2-8 rows over 10 % of the rows (about 240 K / 2.4 M pairs)
  path_1m           a 1 M-row path walked in order (the tail's worst case: every row waits for the previous one)
End to end: 1 M x 512 from C3's generator (randn rows, 1 % re-planted as a copy plus 0.1 randn, unit rows).

Device times are a host clock around work that ends in a device synchronise, after a warm-up, median of
--repeats; the host walk runs once per graph (seconds each).  Every result is checked equal to the host walk
first.  The card's name and power limit are read in the same run.  One JSON line per measurement to --out."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import mmrs_b200  # noqa: E402
from mmrs_b200.dedup import _resolve, selfjoin_tc_raw  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}


def matching(n, rng):
    m = n // 100
    perm = rng.permutation(n)
    return np.stack([perm[:m], perm[m:2 * m]], 1)


def cliques(n, rng, frac=0.1):
    sizes = rng.integers(2, 9, size=int(n * frac) // 2)
    sizes = sizes[: np.searchsorted(np.cumsum(sizes), int(n * frac)) + 1]
    rows = rng.permutation(n)[: int(sizes.sum())]
    starts = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    out = []
    for s in range(2, 9):
        st = starts[sizes == s]
        members = rows[st[:, None] + np.arange(s)[None, :]]          # [k, s]
        a, b = np.triu_indices(s, 1)
        out.append(np.stack([members[:, a].ravel(), members[:, b].ravel()], 1))
    p = np.concatenate(out)
    return p[rng.permutation(len(p))]


def path(n, rng):
    del rng
    return np.stack([np.arange(n - 1), np.arange(1, n)], 1)


def timed(fn, repeats):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts, out


def check_equal(rep, walk):
    reps, dups = walk
    r = rep.cpu().numpy()
    order = np.arange(r.shape[0])
    kept = order[r == order]
    removed = order[(r != order) & (r >= 0)]
    assert kept.tolist() == reps, "representatives differ from the host walk"
    assert [(int(v), int(r[v])) for v in removed] == [tuple(d) for d in dups], "duplicates differ from the host walk"


def c3_data(n, d=512):
    """bench.py leg_c3's generator on the device."""
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn((n, d), generator=gen, device=dev)
    m = n // 100
    perm = torch.randperm(n, generator=gen, device=dev)
    src, dst = perm[:m], perm[m:2 * m]
    x[dst] = x[src] + 0.1 * torch.randn((m, d), generator=gen, device=dev)
    return x / x.norm(dim=-1, keepdim=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r07_bench_dedup.jsonl")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--graphs", default="c3_matching_10m,cliques_1m,cliques_10m,path_1m,e2e_c3_1m")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_dedup measures on a GPU"
    torch.cuda.set_device(0)
    info = card()
    rng = np.random.default_rng(0)
    graphs = {"c3_matching_10m": (matching, 10_000_000), "cliques_1m": (cliques, 1_000_000),
              "cliques_10m": (cliques, 10_000_000), "path_1m": (path, 1_000_000)}
    rows = []
    for name in args.graphs.split(","):
        if name == "e2e_c3_1m":
            n = 1_000_000
            x = c3_data(n)
            t_dev, ts_dev, rep = timed(lambda: mmrs_b200.deduplicate(x, 0.95), args.repeats)

            def host():
                pairs = mmrs_b200.find_duplicate_pairs(x, 0.95)
                return pairs, mmrs_b200.greedy_first_keeper(n, pairs, range(n))
            t0 = time.perf_counter()
            pairs, walk = host()
            t_host = time.perf_counter() - t0
            check_equal(rep, walk)
            t_join, _, _ = timed(lambda: selfjoin_tc_raw(x, 0.95), args.repeats)
            row = {"graph": name, "rows": n, "dim": 512, "pairs": int(pairs.shape[0]), "deduplicate_s": t_dev,
                   "deduplicate_all_s": ts_dev, "join_only_s": t_join,
                   "find_duplicate_pairs_plus_host_walk_s": t_host, **info}
        else:
            gen_fn, n = graphs[name]
            pairs = torch.from_numpy(gen_fn(n, rng).astype(np.int64)).cuda()
            t_dev, ts_dev, (rep, rounds, tail) = timed(lambda: _resolve(pairs, n), args.repeats)
            t0 = time.perf_counter()
            walk = mmrs_b200.greedy_first_keeper(n, pairs, range(n))
            t_host = time.perf_counter() - t0
            check_equal(rep, walk)
            row = {"graph": name, "rows": n, "pairs": int(pairs.shape[0]), "resolve_s": t_dev, "resolve_all_s": ts_dev,
                   "rounds": rounds, "tail_rows": tail, "host_walk_s": t_host, "kept": len(walk[0]), **info}
        print(json.dumps(row), flush=True)
        rows.append(row)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
