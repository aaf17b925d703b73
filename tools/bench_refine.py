"""python tools/bench_refine.py [--out FILE] [--rounds R] : refined top-k search on one B200.

Recall (1M x 768, 1024 unit queries, the unit-gaussian and clustered generators of tools/bench_int8.py): recall@10
and @100 against the fp32 exact top-k (torch fp32 matmul of the unrounded rows) of the int8 and bf16 galleries,
unrefined and refined against an fp32 store with refine_k = k, 2k, 4k, 8k.  This decides the refine_k default.

Time per call (D = 768, k = 100, refine_k = 4k = 400, Q = 1, 16, 128, 1024 unit queries on the device; 1M and 12.5M
rows, C4's per-GPU shard): unrefined int8; int8 + device fp32 store; int8 + host fp32 store; int8 + host bf16
store; unrefined bf16.  After a warm-up of every arm, rounds alternate the arms; each sample is a host clock
around one `search_topk` that ends in a device synchronise; the median over rounds is reported with its spread.
The refine stage's share of a refined call is (refined - unrefined int8) / refined, from those medians.  The
bytes the refine stage reads are computed from shapes (Q * k_c * Dp * element size).  A host store larger than
half of MemAvailable (/proc/meminfo) is skipped and its arm says so.  Galleries of 12.5M rows exceed the 126 MB
L2; a store's candidate rows are scattered.  Every host store is unregistered before exit.  Prints one JSON line
per measurement with the card name and power limit read in the same call; --out FILE keeps a copy."""
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


def mem_available_bytes():
    for line in Path("/proc/meminfo").read_text().splitlines():
        if line.startswith("MemAvailable:"):
            return int(line.split()[1]) * 1024
    return 0


def host_time(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def unit_gaussian(n, gen):
    x = torch.empty((n, D), device="cuda")
    for lo in range(0, n, 1 << 20):
        r = torch.randn((min(1 << 20, n - lo), D), generator=gen, device="cuda")
        x[lo:lo + r.shape[0]] = r / r.norm(dim=1, keepdim=True)
    return x


def data(dist, n, seed):
    """(rows [n, D] fp32 on the device, 1024 queries) of bench_int8.py's generators."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    if dist == "gaussian":
        x = unit_gaussian(n, gen)
        q = torch.randn((1024, D), generator=torch.Generator().manual_seed(5)).cuda()
        return x, q / q.norm(dim=1, keepdim=True)
    cent = torch.randn((1000, D), generator=gen, device="cuda")
    lab = torch.arange(1000, device="cuda").repeat_interleave(n // 1000)
    x = cent[lab] + 0.5 * torch.randn((n, D), generator=gen, device="cuda")
    x = x / x.norm(dim=1, keepdim=True)
    q = cent[torch.arange(1024, device="cuda") % 1000] + 0.3 * torch.randn((1024, D), generator=gen, device="cuda")
    return x, q / q.norm(dim=1, keepdim=True)


def recall(idx, exact, kk):
    hit = sum(len(set(a[:kk].tolist()) & set(b[:kk].tolist())) for a, b in zip(idx.cpu(), exact.cpu()))
    return round(hit / (idx.shape[0] * kk), 4)


def recall_lines(card, emit):
    n = 1_000_000
    for dist in ("gaussian", "clustered"):
        x, q = data(dist, n, seed=7)
        exact = torch.cat([(q[i:i + 128] @ x.T).topk(K, dim=1).indices for i in range(0, 1024, 128)])
        store = mmrs_b200.RefineStore(x, mode="fp32", memory="device")
        for mode in ("int8", "bf16"):
            gal = mmrs_b200.DeviceGallery(x.to(torch.bfloat16) if mode == "bf16" else x, mode=mode)
            line = {"kind": "recall", "rows": n, "dim": D, "queries": 1024, "data": dist, "gallery": mode,
                    "store": "fp32", "card": card}
            for kk in (10, 100):
                _, idx = mmrs_b200.search_topk(q, gal, kk, normalize_queries=False)
                line[f"unrefined_recall@{kk}"] = recall(idx, exact, kk)
                for mult in (1, 2, 4, 8):
                    _, idx = mmrs_b200.search_topk(q, gal, kk, normalize_queries=False, refine=store,
                                                   refine_k=mult * kk)
                    line[f"refine_k={mult}k_recall@{kk}"] = recall(idx, exact, kk)
            emit(line)
            del gal
        del x, store
        torch.cuda.empty_cache()


def time_group(g8, g16, stores, nq, rounds):
    """{arm: [ms per round]} of the unrefined int8 / bf16 searches and int8 refined by each store, alternated."""
    q = torch.randn((nq, D), generator=torch.Generator().manual_seed(nq)).cuda()
    q = q / q.norm(dim=1, keepdim=True)
    arms = {"int8": lambda: mmrs_b200.search_topk(q, g8, K, normalize_queries=False),
            "bf16": lambda: mmrs_b200.search_topk(q, g16, K, normalize_queries=False)}
    for name, s in stores.items():
        arms[f"int8+{name}"] = (lambda s=s: mmrs_b200.search_topk(q, g8, K, normalize_queries=False, refine=s,
                                                                  refine_k=4 * K))
    for fn in arms.values():
        fn()
        fn()
    times = {a: [] for a in arms}
    for _ in range(rounds):
        for a, fn in arms.items():
            times[a].append(host_time(fn))
    return times


def time_lines(n, card, rounds, emit):
    """Two groups, each alternated with the unrefined arms: the fp32 stores, then (the fp32 host store released
    first) the bf16 host store -- both host stores registered at once can exceed what the host lets one process
    page-lock."""
    gen = torch.Generator(device="cuda").manual_seed(n)
    x = unit_gaussian(n, gen)
    g8 = mmrs_b200.DeviceGallery(x, mode="int8")
    g16 = mmrs_b200.DeviceGallery(x.to(torch.bfloat16))
    k_c = 4 * K
    results = {nq: {} for nq in QS}
    skipped = {}
    groups = ((("fp32", "device"), ("fp32", "host")), (("bf16", "host"),))
    for gi, group in enumerate(groups):
        stores = {}
        try:
            for mode, mem in group:
                name = f"{mode}_{mem}"
                nbytes = n * D * (2 if mode == "bf16" else 4)
                free = mem_available_bytes()
                if mem == "host" and nbytes > free // 2:
                    skipped[name] = f"skipped: {nbytes / 1e9:.1f} GB store > half of MemAvailable {free / 1e9:.1f} GB"
                    continue
                try:
                    stores[name] = mmrs_b200.RefineStore(x, mode=mode, memory=mem)
                except mmrs_b200._cabi.MmrsError as e:
                    skipped[name] = f"skipped: the store could not be registered ({e})"
            for nq in QS:
                times = time_group(g8, g16, stores, nq, rounds)
                for a, t in times.items():
                    if gi > 0 and a in ("int8", "bf16"):
                        a = f"{a}_group{gi + 1}"      # the baseline this group was alternated with
                    med = float(np.median(t))
                    results[nq][a] = {"ms": round(med, 4), "spread_pct": round(100 * (max(t) - min(t)) / med, 1)}
                    base = results[nq]["int8" if gi == 0 else f"int8_group{gi + 1}"]["ms"]
                    if a.startswith("int8+"):
                        s = stores[a[5:]]
                        results[nq][a]["refine_share"] = round((med - base) / med, 3)
                        results[nq][a]["refine_read_mb"] = round(
                            nq * k_c * s.padded_dim * (2 if s.mode == "bf16" else 4) / 1e6, 2)
        finally:
            for s in stores.values():
                s.close()
    for nq in QS:
        line = {"kind": "time", "rows": n, "dim": D, "queries": nq, "k": K, "refine_k": k_c, "card": card,
                "rounds": rounds}
        line.update(results[nq])
        for name, why in skipped.items():
            line[f"int8+{name}"] = why
        emit(line)
    del g8, g16, x
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", help="also write the JSON lines to this file")
    ap.add_argument("--skip-recall", action="store_true")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    card = smi[0] if smi else "unknown"
    lines = []

    def emit(line):
        print(json.dumps(line), flush=True)
        lines.append(line)

    emit({"kind": "host", "card": card, "mem_available_gb": round(mem_available_bytes() / 1e9, 1)})
    if not args.skip_recall:
        recall_lines(card, emit)
    for n in (1_000_000, 12_500_000):
        time_lines(n, card, args.rounds, emit)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
