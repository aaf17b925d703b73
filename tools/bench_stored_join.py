"""The self-join on one GPU in three storage formats, on C3's generator (bench_dedup.c3_data: randn rows, 1 % re-planted
as a copy plus 0.1 randn, unit rows), tau = 0.95:
  tc           method="tc" on the fp32 rows: bf16 copy, tensor-core prefilter, fp32 recheck
  bf16_stored  method="stored" on a bf16 DeviceGallery: prefilter with the accumulation-only margin, bf16 recheck
  int8_stored  method="stored" on an int8 DeviceGallery: exact int8 decisions in the epilogue
Workloads: c3_1m (1 M x 512, the whole join) and c3_rank (10 M x 512, rank 0's panels of an 8-way dealing, as
tools/c3_one_rank.py).  Arms alternate inside every repeat.  Join time is a host clock around the join and a device
synchronise (the pair list, unsorted), median of --repeats after one warm-up call per arm.  Also reported: the
prefilter's candidate count, the pair set against the tc arm's (= the fp32 join's), the arm's resident rows and the
peak device memory the call allocates on top of them, and the card's name and power limit read in the same run.
One JSON line per (workload, arm) to --out."""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import mmrs_b200  # noqa: E402
from mmrs_b200 import _cabi  # noqa: E402
from mmrs_b200.dedup import selfjoin_stored_raw, selfjoin_tc_raw, sort_pairs, tc_margin, _max_row_norm  # noqa: E402
from bench_dedup import c3_data, card  # noqa: E402

TAU = 0.95


def candidates(arm, inp, rank, world):
    """The prefilter's candidate count (d_out_count[1]) of one call with ample buffers."""
    lib, dev = _cabi.lib, torch.device("cuda", 0)
    cap = cand_cap = 1 << 22
    counts = torch.zeros(2, dtype=torch.int64, device=dev)
    pairs = torch.empty((cap, 2), dtype=torch.int64, device=dev)
    if arm == "tc":
        x16 = inp.to(torch.bfloat16)
        n, d = inp.shape
        ws_bytes = lib.mmrs_selfjoin_tc_workspace_bytes(n, cand_cap)
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        st = lib.mmrs_selfjoin_pairs_tc(inp.data_ptr(), inp.stride(0), x16.data_ptr(), x16.stride(0), n, d, TAU,
                                        tc_margin(d, _max_row_norm(inp)), rank, world, pairs.data_ptr(), cap,
                                        counts.data_ptr(), cand_cap, mmrs_b200.DeviceGallery.aligned_ptr(ws), ws_bytes,
                                        0)
    else:
        i8 = inp.mode == "int8"
        margin = 0.0 if i8 else tc_margin(inp.padded_dim, _max_row_norm(inp.data))
        ws_bytes = lib.mmrs_selfjoin_stored_workspace_bytes(inp.n_rows, inp.dtype_code, cand_cap)
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        st = lib.mmrs_selfjoin_pairs_stored(inp.data.data_ptr(), inp.dtype_code, inp.data.stride(0), inp.n_rows,
                                            inp.padded_dim, TAU, margin, rank, world, pairs.data_ptr(), cap,
                                            counts.data_ptr(), cand_cap, mmrs_b200.DeviceGallery.aligned_ptr(ws),
                                            ws_bytes, 0)
    _cabi.check(st)
    return int(counts[1].item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r10_bench_stored_join.jsonl")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--workloads", default="c3_1m,c3_rank")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_stored_join measures on a GPU"
    torch.cuda.set_device(0)
    info = card()
    shapes = {"c3_1m": (1_000_000, 0, 1), "c3_rank": (10_000_000, 0, 8)}
    rows = []
    for wl in args.workloads.split(","):
        n, rank, world = shapes[wl]
        x = c3_data(n)
        inputs = {"tc": x, "bf16_stored": mmrs_b200.DeviceGallery(x, mode="bf16"),
                  "int8_stored": mmrs_b200.DeviceGallery(x, mode="int8")}
        joins = {"tc": lambda: selfjoin_tc_raw(x, TAU, rank, world),
                 "bf16_stored": lambda: selfjoin_stored_raw(inputs["bf16_stored"], TAU, rank, world),
                 "int8_stored": lambda: selfjoin_stored_raw(inputs["int8_stored"], TAU, rank, world)}
        times = {a: [] for a in joins}
        peak = {}
        result = {}
        for a, fn in joins.items():                 # warm-up, pair sets and peak memory, one arm at a time
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            result[a] = sort_pairs(fn(), n)
            torch.cuda.synchronize()
            peak[a] = torch.cuda.max_memory_allocated() - base
        for _ in range(args.repeats):
            for a, fn in joins.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                times[a].append(time.perf_counter() - t0)
        ref = result["tc"]
        for a in joins:
            inp = inputs[a]
            resident = inp.numel() * inp.element_size() if a == "tc" else inp.nbytes
            row = {"workload": wl, "rows": n, "dim": 512, "rank": rank, "world": world, "arm": a,
                   "join_s": float(np.median(times[a])), "join_all_s": times[a],
                   "candidates": candidates(a, inp, rank, world), "pairs": int(result[a].shape[0]),
                   "pairs_equal_fp32_join": bool(torch.equal(result[a], ref)),
                   "resident_rows_bytes": int(resident), "peak_extra_bytes": int(peak[a]), **info}
            print(json.dumps(row), flush=True)
            rows.append(row)
        del x, inputs, joins, result
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
