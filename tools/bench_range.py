"""python tools/bench_range.py [--out FILE] : range search on one B200.

Shapes (bf16, D = 768): the 1M-row gallery and one 12.5M-row shard of C4 (100M / 8), with Q = 1, 16 and 128
queries.  Per query, the threshold is picked from its `full_scores` row before anything is timed (the score
of rank max(1, sel * N)), at selectivity sel = 1e-5, 1e-3, 1e-2 and 1e-1.  Arms, alternated round by round
after a warm-up of each, each timed on the host around work that ends in a device synchronise (median over
rounds):
  range        `search_range(q, gal, t)` (CSR, rows in order);
  materialise  `full_scores(q, gal)` and then `(S >= t).nonzero()` plus the values `S[mask]` -- the [Q, N]
               fp32 matrix written and read again (the whole batch in one matrix: it fits at these shapes);
  topk100      `search_topk(q, gal, 100)` of the same batch, as the reference point of a fixed-k search.
The range arm is checked against the materialised result (offsets, indices, values) before timing.  Prints
one JSON line per shape with the card name and power limit; --out FILE keeps a copy."""
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
from mmrs_b200.range_search import window_rows


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


def materialise(q, gal, thr):
    s = mmrs_b200.full_scores(q, gal)
    mask = s >= thr[:, None]
    off = torch.zeros(q.shape[0] + 1, dtype=torch.int64, device=s.device)
    torch.cumsum(mask.sum(1), 0, out=off[1:])
    return off, s[mask], mask.nonzero()[:, 1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else "unknown"
    lines = []
    for n, d in ((1_000_000, 768), (12_500_000, 768)):
        gal = device_gallery(n, d, seed=n)
        for nq in (1, 16, 128):
            q = torch.randn((nq, d), generator=torch.Generator().manual_seed(nq)).cuda()
            srt = mmrs_b200.full_scores(q, gal).sort(1, descending=True).values
            for sel in (1e-5, 1e-3, 1e-2, 1e-1):
                thr = srt[:, max(1, int(round(sel * n))) - 1].contiguous()
                got = mmrs_b200.search_range(q, gal, thr)
                want = materialise(q, gal, thr)
                assert torch.equal(got[0], want[0]) and torch.equal(got[2], want[2]), (n, nq, sel)
                assert torch.equal(got[1].view(torch.int32), (want[1] + 0.0).view(torch.int32)), (n, nq, sel)
                matches = int(got[0][-1])
                del got, want
                arms = {"range": lambda: mmrs_b200.search_range(q, gal, thr),
                        "materialise": lambda: materialise(q, gal, thr),
                        "topk100": lambda: mmrs_b200.search_topk(q, gal, 100)}
                for fn in arms.values():            # warm-up
                    fn()
                times = {k: [] for k in arms}
                for _ in range(args.rounds):
                    for k, fn in arms.items():
                        times[k].append(host_time(fn))
                med = {k: float(np.median(v)) for k, v in times.items()}
                line = {"rows": n, "dim": d, "queries": nq, "selectivity": sel, "matches": matches,
                        "windows": -(-n // window_rows(nq, n, 4 << 30)), "card": card,
                        "ms_median": {k: round(v, 3) for k, v in med.items()},
                        "spread_pct": {k: round(100 * (max(v) - min(v)) / med[k], 1) for k, v in times.items()},
                        "range_vs_materialise": round(med["materialise"] / med["range"], 2),
                        "range_vs_topk100": round(med["topk100"] / med["range"], 2)}
                print(json.dumps(line), flush=True)
                lines.append(line)
            del srt
            torch.cuda.empty_cache()
        del gal
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
