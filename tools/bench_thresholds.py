"""python tools/bench_thresholds.py [--out FILE] : per-class threshold tuning on one B200.

Shapes (bf16, D = 768): the 1M-row gallery and one 12.5M-row shard of C4 (100M / 8), with C = 10, 100 and
1 000 class prototypes over random row labels of C classes, n_points = 200, get_similarity's scale 100.
Arms, alternated round by round after a warm-up of each, each timed on the host around work that ends in
a device synchronise (median over rounds):
  reference  the reference's loop `find_thresholds(*get_similarity(gal, targets, c, q_c), c)` (C = 10 only:
             every class copies N scores to the host, splits them in numpy and uploads them again);
  per_class  `best_threshold_on_device(full_scores(q_c, gal)[0], targets, c)`: one gallery pass per class;
  batched    `best_thresholds(queries, gal, row_labels, labels)`.
For `batched` the line also splits one call into its scoring pass (`full_scores` of every chunk) and its
sweep kernels (range + histogram + suffix, on the scores already in place), each with CUDA events, and the
sweep's bytes from shapes (4 B score read for the range and 4 B for the histogram per (query, row), 4 B
label per row per chunk) over its time.  Prints one JSON line per shape with the card name and power
limit; --out FILE keeps a copy."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch
import mmrs_b200
from mmrs_b200 import search as _search
from mmrs_b200.thresholds import DeviceSweep, chunk_queries


def device_gallery(n, d, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    data = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    for lo in range(0, n, 1 << 20):
        x = torch.randn((min(1 << 20, n - lo), d), generator=gen, device="cuda")
        data[lo:lo + x.shape[0]] = (x / x.norm(dim=1, keepdim=True)).to(torch.bfloat16)
    return mmrs_b200.DeviceGallery(data)


def host_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def split_batched(gal, q, labels, row_labels, n_points):
    """(scoring ms, sweep ms, sweep bytes) of one best_thresholds call, chunk by chunk, with CUDA events."""
    c, n = q.shape[0], gal.n_rows
    qc = min(c, chunk_queries(n, 4 << 30))
    sweep = DeviceSweep(gal, qc, n_points, False, 100.0, "auto", row_labels, None, _search.grid_f32())
    score_ms = sweep_ms = 0.0
    chunks = 0
    for lo in range(0, c, qc):
        qq, lab = q[lo:lo + qc], labels[lo:lo + qc]
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        qp, _ = _search._prep_queries(qq, gal)
        e[0].record()
        _search._scores_into(gal, qp, sweep.scores, False, 100.0, "auto")
        e[1].record()
        rng = sweep.range_keys(qq.shape[0])
        sweep.counts(lab, rng)
        e[2].record()
        e[2].synchronize()
        score_ms += e[0].elapsed_time(e[1])
        sweep_ms += e[1].elapsed_time(e[2])
        chunks += 1
    return score_ms, sweep_ms, 8 * n * c + 4 * n * chunks


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else "unknown"
    n_points = 200
    lines = []
    for n, d in ((1_000_000, 768), (12_500_000, 768)):
        gal = device_gallery(n, d, seed=n)
        for c in (10, 100, 1000):
            rng = np.random.default_rng(c)
            targets_np = rng.integers(0, c, n).astype(np.int64)
            targets = torch.from_numpy(targets_np).cuda()
            row_labels = mmrs_b200.RowLabels(targets)
            labels = torch.arange(c, dtype=torch.int32).cuda()
            q = torch.randn((c, d), generator=torch.Generator().manual_seed(c)).cuda()
            arms = {
                "per_class": lambda: [mmrs_b200.best_threshold_on_device(
                    mmrs_b200.full_scores(q[j:j + 1], gal, normalize_queries=False, scale=100.0)[0], targets, j)
                    for j in range(c)],
                "batched": lambda: mmrs_b200.best_thresholds(q, gal, row_labels, labels),
            }
            if c == 10:
                arms["reference"] = lambda: [mmrs_b200.find_thresholds(
                    *mmrs_b200.get_similarity(gal, targets_np, j, q[j]), j) for j in range(c)]
            # the arms agree before anything is timed; with "auto" one query is scored by K1 and a chunk by K2,
            # so the check pins the kernel (the timed arms keep "auto")
            want = mmrs_b200.best_thresholds(q, gal, row_labels, labels, path="mma")
            for j in range(0, c, max(1, c // 5)):
                s = mmrs_b200.full_scores(q[j:j + 1], gal, normalize_queries=False, scale=100.0, path="mma")[0]
                got = mmrs_b200.best_threshold_on_device(s, targets, j)
                assert np.array_equal(got[5], want[5][j], equal_nan=True) and got[0] == want[0][j], (n, c, j)
            for fn in arms.values():                   # warm-up
                fn()
            times = {k: [] for k in arms}
            for _ in range(args.rounds):
                for k, fn in arms.items():
                    times[k].append(host_time(fn))
            med = {k: float(np.median(v)) for k, v in times.items()}
            splits = [split_batched(gal, q, labels, row_labels, n_points) for _ in range(args.rounds)]
            score_ms = float(np.median([s[0] for s in splits]))
            sweep_ms = float(np.median([s[1] for s in splits]))
            sweep_bytes = splits[0][2]
            line = {"rows": n, "dim": d, "classes": c, "n_points": n_points, "card": card,
                    "ms_median": {k: round(v, 3) for k, v in med.items()},
                    "spread_pct": {k: round(100 * (max(v) - min(v)) / med[k], 1) for k, v in times.items()},
                    "batched_split_ms": {"scoring": round(score_ms, 3), "sweep": round(sweep_ms, 3)},
                    "sweep_bytes": sweep_bytes, "sweep_tb_per_s": round(sweep_bytes / (sweep_ms * 1e-3) / 1e12, 3),
                    "speedup_vs_per_class": round(med["per_class"] / med["batched"], 2)}
            if "reference" in med:
                line["speedup_vs_reference"] = round(med["reference"] / med["batched"], 2)
            print(json.dumps(line), flush=True)
            lines.append(line)
            del row_labels, targets
        del gal
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
