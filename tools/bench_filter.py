"""python tools/bench_filter.py [--out FILE] : cost of a row filter on one B200.

Shapes: the 1M x 768 bf16 gallery at Q = 1, 16, 128 and one 12.5M x 768 shard of C4 (100M / 8) at
Q = 16, all top-100.  Variants: no filter, the all-true filter, random 50 / 10 / 1 / 0.1 % of the rows
and a contiguous 10 % block (one class of a class-sorted gallery).  Each call is a complete,
status-checked search (device queries and results); the variants are alternated round by round after
a warm-up of every one, and each cell is the median over rounds of the CUDA-event time of `--calls`
back-to-back calls.  Galleries are generated on the device (unit rows) and are larger than L2.
Prints one JSON line per shape (with the card name and power limit); --out FILE keeps a copy."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch
import mmrs_b200


def device_gallery(n, d, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    data = torch.empty((n, d), dtype=torch.bfloat16, device="cuda")
    for lo in range(0, n, 1 << 20):
        x = torch.randn((min(1 << 20, n - lo), d), generator=gen, device="cuda")
        data[lo:lo + x.shape[0]] = (x / x.norm(dim=1, keepdim=True)).to(torch.bfloat16)
    return mmrs_b200.DeviceGallery(data)


def masks(n):
    rng = np.random.default_rng(0)
    out = {"none": None, "all": np.ones(n, dtype=bool)}
    for name, p in (("p50", 0.5), ("p10", 0.1), ("p1", 0.01), ("p0.1", 0.001)):
        out[name] = rng.random(n) < p
    block = np.zeros(n, dtype=bool)
    block[n * 4 // 10:n * 5 // 10] = True
    out["block10"] = block
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
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else "unknown"
    lines = []
    for n, d, qs in ((1_000_000, 768, (1, 16, 128)), (12_500_000, 768, (16,))):
        gal = device_gallery(n, d, seed=n)
        filters = {name: (mmrs_b200.RowFilter(m, device=gal.device) if m is not None else None)
                   for name, m in masks(n).items()}
        for nq in qs:
            q = torch.randn((nq, d), generator=torch.Generator().manual_seed(nq)).cuda()
            fns = {name: (lambda f=f: mmrs_b200.search_topk(q, gal, args.k, row_filter=f)) for name, f in filters.items()}
            for fn in fns.values():           # warm-up: graph capture, module load, allocator
                for _ in range(3):
                    fn()
            base = fns["none"]()
            same = fns["all"]()
            assert torch.equal(base[0], same[0]) and torch.equal(base[1], same[1])
            times = {name: [] for name in fns}
            for _ in range(args.rounds):
                for name, fn in fns.items():
                    times[name].append(time_calls(fn, args.calls))
            med = {name: float(np.median(t)) for name, t in times.items()}
            line = {"rows": n, "dim": d, "queries": nq, "k": args.k, "card": card,
                    "ms_per_call_median": {k: round(v, 4) for k, v in med.items()},
                    "spread_pct": {k: round(100 * (max(t) - min(t)) / med[k], 1) for k, t in times.items()},
                    "vs_none": {k: round(v / med["none"], 3) for k, v in med.items()},
                    "allowed": {k: (f.n_allowed if f is not None else n) for k, f in filters.items()}}
            print(json.dumps(line), flush=True)
            lines.append(line)
        del gal, filters
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
