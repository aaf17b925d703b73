"""python tools/bench_int8.py [--out FILE] [--skip-100m | --only-100m] : int8 against bf16 galleries on one B200.

Shapes (D = 768), top-100, Q = 1, 16, 128 and 1024 unit queries on the device:
  12.5M rows  C4's per-GPU shard (100M / 8): the bf16 and the int8 gallery both resident, timed alternately;
  1M rows     likewise, plus recall@10 / @100 of each mode against the fp32 exact top-k (torch fp32 matmul of the
              unrounded rows) on unit-gaussian rows and on bench.py's clustered rows (1000 centroids + 0.5 noise,
              stored cluster by cluster, queries near centroids);
  100M rows   the int8 gallery alone on one GPU (78.4 GB), then freed, then the bf16 gallery (153.6 GB) in the
              same call.
Timing: after a warm-up of each arm, rounds alternate the arms; each sample is a host clock around one
`search_topk` that ends in a device synchronise; the median over rounds is reported with its spread.  Derived
from shapes: gallery bytes per call (bf16 2 D, int8 D + 16 per row) over the median time against the 7.7 TB/s
data-sheet HBM bandwidth, and at Q = 1024 the int8 tera-operations per second (2 N D Q / time) against the
4.5 POPS dense int8 data-sheet rate.  Galleries of 12.5M rows and more exceed the 126 MB L2.  Prints one JSON
line per (shape, Q) with the card name and power limit read in the same call; --out FILE keeps a copy."""
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

D, K = 768, 100
QS = (1, 16, 128, 1024)
HBM_TBS, I8_POPS = 7.7, 4.5


def unit_rows(n, gen, chunk=1 << 20):
    """fp32 unit-gaussian rows [n, D] produced chunk by chunk (yields (lo, rows))."""
    for lo in range(0, n, chunk):
        x = torch.randn((min(chunk, n - lo), D), generator=gen, device="cuda")
        yield lo, x / x.norm(dim=1, keepdim=True)


def galleries(n, seed, modes):
    """{mode: DeviceGallery} of the same unit-gaussian rows; the int8 rows are quantised from fp32."""
    out = {}
    for mode in modes:
        gen = torch.Generator(device="cuda").manual_seed(seed)
        if mode == "bf16":
            data = torch.empty((n, D), dtype=torch.bfloat16, device="cuda")
            for lo, x in unit_rows(n, gen):
                data[lo:lo + x.shape[0]] = x.to(torch.bfloat16)
            out[mode] = mmrs_b200.DeviceGallery(data)
        else:
            # the fp32 rows of a 100M gallery do not fit beside it: quantise chunk by chunk into one int8 buffer,
            # then hand that buffer to a gallery object of the same layout
            lib = mmrs_b200._cabi.lib
            data = torch.empty((n, D + 16), dtype=torch.int8, device="cuda")
            for lo, x in unit_rows(n, gen):
                mmrs_b200._cabi.check(lib.mmrs_quantize_rows_i8(x.data_ptr(), mmrs_b200._cabi.DTYPE_F32, x.shape[0], D,
                                                                 D, data[lo].data_ptr(), D + 16, 0))
            gal = mmrs_b200.DeviceGallery(torch.zeros((1, D)), mode="int8")
            gal.data, gal.n_rows = data, n
            out[mode] = gal
    return out


def host_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def queries(nq, seed):
    q = torch.randn((nq, D), generator=torch.Generator().manual_seed(seed)).cuda()
    return q / q.norm(dim=1, keepdim=True)


def gallery_bytes(gal):
    return gal.n_rows * (D + 16 if gal.mode == "int8" else 2 * D)


def time_arms(gals, nq, rounds, card, n):
    q = queries(nq, seed=nq)
    arms = {m: (lambda g=g: mmrs_b200.search_topk(q, g, K, normalize_queries=False)) for m, g in gals.items()}
    for fn in arms.values():
        fn()
        fn()
    times = {m: [] for m in arms}
    for _ in range(rounds):
        for m, fn in arms.items():
            times[m].append(host_time(fn))
    line = {"rows": n, "dim": D, "queries": nq, "k": K, "card": card}
    for m, t in times.items():
        med = float(np.median(t))
        line[m] = {"ms": round(med, 4), "spread_pct": round(100 * (max(t) - min(t)) / med, 1),
                   "hbm_frac": round(gallery_bytes(gals[m]) / (med * 1e-3) / (HBM_TBS * 1e12), 3)}
        if m == "int8" and nq == 1024:
            tops = 2.0 * n * D * nq / (med * 1e-3) / 1e12
            line[m]["tops"] = round(tops, 1)
            line[m]["frac_of_4500_tops"] = round(tops / (I8_POPS * 1e3), 3)
    if "bf16" in times and "int8" in times:
        line["speedup_int8_vs_bf16"] = round(line["bf16"]["ms"] / line["int8"]["ms"], 3)
    return line


def recall_lines(card):
    """recall@10 / @100 of bf16 and int8 mode against the fp32 exact top-k at 1M x 768, two distributions."""
    out = []
    n = 1_000_000
    for dist in ("gaussian", "clustered"):
        gen = torch.Generator(device="cuda").manual_seed(7)
        if dist == "gaussian":
            x = torch.cat([r for _, r in unit_rows(n, gen)])
            q = queries(1024, seed=5)
        else:
            cent = torch.randn((1000, D), generator=gen, device="cuda")
            lab = torch.arange(1000, device="cuda").repeat_interleave(1000)
            x = cent[lab] + 0.5 * torch.randn((n, D), generator=gen, device="cuda")
            x = x / x.norm(dim=1, keepdim=True)
            q = cent[torch.arange(1024, device="cuda") % 1000] + 0.3 * torch.randn((1024, D), generator=gen, device="cuda")
            q = q / q.norm(dim=1, keepdim=True)
        exact = torch.cat([(q[i:i + 128] @ x.T).topk(K, dim=1).indices for i in range(0, 1024, 128)])
        line = {"rows": n, "dim": D, "queries": 1024, "data": dist, "card": card}
        for mode in ("bf16", "int8"):
            gal = mmrs_b200.DeviceGallery(x.to(torch.bfloat16) if mode == "bf16" else x, mode=mode)
            _, idx = mmrs_b200.search_topk(q, gal, K, normalize_queries=False)
            for kk in (10, 100):
                hit = sum(len(set(a[:kk].tolist()) & set(b[:kk].tolist())) for a, b in zip(idx.cpu(), exact.cpu()))
                line[f"{mode}_recall@{kk}"] = round(hit / (1024 * kk), 4)
            del gal
        out.append(line)
        del x
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    ap.add_argument("--skip-100m", action="store_true")
    ap.add_argument("--only-100m", action="store_true", help="the 100M-row shape alone (it needs its own minutes)")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else "unknown"
    lines = []

    def emit(line):
        print(json.dumps(line), flush=True)
        lines.append(line)

    for n in (() if args.only_100m else (12_500_000, 1_000_000)):
        gals = galleries(n, seed=n, modes=("bf16", "int8"))
        for nq in QS:
            emit(time_arms(gals, nq, args.rounds, card, n))
        del gals
        torch.cuda.empty_cache()
    for line in ([] if args.only_100m else recall_lines(card)):
        emit(line)
    if not args.skip_100m:
        n = 100_000_000
        per_mode = {}
        for mode in ("int8", "bf16"):                          # one at a time: both do not fit one GPU
            gals = galleries(n, seed=1, modes=(mode,))
            per_mode[mode] = {nq: time_arms(gals, nq, args.rounds, card, n)[mode] for nq in QS}
            del gals
            torch.cuda.empty_cache()
        for nq in QS:
            emit({"rows": n, "dim": D, "queries": nq, "k": K, "card": card, "bf16": per_mode["bf16"][nq],
                  "int8": per_mode["int8"][nq],
                  "speedup_int8_vs_bf16": round(per_mode["bf16"][nq]["ms"] / per_mode["int8"][nq]["ms"], 3),
                  "note": "int8 and bf16 galleries resident one after the other, not alternated"})
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
