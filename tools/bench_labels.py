"""python tools/bench_labels.py [--out FILE] : cost of label-conditioned search on one B200.

Shapes (bf16, D = 768, top-100): the 1M-row gallery at Q = 1, 16, 128, one 12.5M-row shard of C4
(100M / 8) at Q = 16, and a C5-shaped tensor-bound launch (1024 queries over 4M rows).  Row labels:
10, 100 and 1 000 classes, each random and class-sorted (the reference's caches are built class by
class).  Variants per label set: every query labelled with a random class and "same", the same with
"other", and a batch half of whose queries are unlabeled (-1).  Each cell is relative to the unlabeled
search of the same batch.  Each call is a complete, status-checked search (device queries, labels and
results); the variants are alternated round by round after a warm-up of every one, and each cell is the
median over rounds of the CUDA-event time of `--calls` back-to-back calls.  `retries` counts calls that
overflowed a candidate list and were repeated on the exhaustive path.  Prints one JSON line per shape
(with the card name and power limit); --out FILE keeps a copy."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch
import mmrs_b200
from mmrs_b200 import search as _search


def device_gallery(n, d, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    data = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    for lo in range(0, n, 1 << 20):
        x = torch.randn((min(1 << 20, n - lo), d), generator=gen, device="cuda")
        data[lo:lo + x.shape[0]] = (x / x.norm(dim=1, keepdim=True)).to(torch.bfloat16)
    return mmrs_b200.DeviceGallery(data)


def label_sets(n, dev):
    rng = np.random.default_rng(0)
    out = {}
    for c in (10, 100, 1000):
        out[f"c{c}_random"] = (c, mmrs_b200.RowLabels(torch.from_numpy(rng.integers(0, c, n).astype(np.int32)), device=dev))
        out[f"c{c}_sorted"] = (c, mmrs_b200.RowLabels(torch.from_numpy((np.arange(n) * c // n).astype(np.int32)), device=dev))
    return out


def time_calls(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else "unknown"
    retries = {}
    real = _search._search_exhaustive

    def counting(*a, **kw):
        retries[current[0]] = retries.get(current[0], 0) + 1
        return real(*a, **kw)
    _search._search_exhaustive = counting
    current = [None]
    lines = []
    for n, d, qs in ((1_000_000, 768, (1, 16, 128)), (12_500_000, 768, (16,)), (4_000_000, 768, (1024,))):
        gal = device_gallery(n, d, seed=n)
        sets = label_sets(n, gal.device)
        for nq in qs:
            q = torch.randn((nq, d), generator=torch.Generator().manual_seed(nq)).cuda()
            rng = np.random.default_rng(nq)
            fns = {"none": lambda: mmrs_b200.search_topk(q, gal, args.k)}
            for name, (c, L) in sets.items():
                ql = torch.from_numpy(rng.integers(0, c, nq).astype(np.int32)).cuda()
                half = ql.clone()
                half[::2] = -1
                for var, lab, match in (("same", ql, "same"), ("other", ql, "other"), ("half", half, "same")):
                    fns[f"{name}/{var}"] = (lambda L=L, lab=lab, match=match:
                                            mmrs_b200.search_topk(q, gal, args.k, row_labels=L, query_labels=lab,
                                                                  label_match=match))
            for name, fn in fns.items():      # warm-up: graph capture, module load, allocator
                current[0] = name
                for _ in range(2):
                    fn()
            retries.clear()
            times = {name: [] for name in fns}
            for _ in range(args.rounds):
                for name, fn in fns.items():
                    current[0] = name
                    times[name].append(time_calls(fn, args.calls))
            med = {name: float(np.median(t)) for name, t in times.items()}
            line = {"rows": n, "dim": d, "queries": nq, "k": args.k, "card": card,
                    "ms_per_call_median": {k: round(v, 4) for k, v in med.items()},
                    "spread_pct": {k: round(100 * (max(t) - min(t)) / med[k], 1) for k, t in times.items()},
                    "vs_none": {k: round(v / med["none"], 3) for k, v in med.items()},
                    "retries": dict(retries)}
            print(json.dumps(line), flush=True)
            lines.append(line)
        del gal, sets
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
