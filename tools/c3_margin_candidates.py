"""Candidates of the tensor-core self-join's bf16 prefilter on BASELINE config C3 (N x 512 unit rows, 1 % planted
pairs at cos ~ 0.995, tau = 0.95; the data of bench.py's C3 leg) at two prefilter margins: the bound
`dedup.tc_margin` passes to the kernel and the 0.0045 the join used before.  The margin is a kernel parameter,
so only the candidate count can move.  Prints one JSON line per margin with the join time (CUDA events), the
candidate count, the pair count and whether the pairs equal the planted set.
Usage: python tools/c3_margin_candidates.py [N] [repeats]"""
import json
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch

from mmrs_b200 import _cabi
from mmrs_b200.dedup import _max_row_norm, tc_margin, sort_pairs
from mmrs_b200.gallery import DeviceGallery
from mmrs_b200.search import _stream_handle

n = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 1
d, tau = 512, 0.95
dev = torch.device("cuda", 0)
gen = torch.Generator(device=dev).manual_seed(0)
x = torch.empty((n, d), dtype=torch.float32, device=dev)
step = 1 << 20
for lo in range(0, n, step):
    x[lo:lo + step] = torch.randn((min(step, n - lo), d), generator=gen, device=dev)
m = n // 100
perm = torch.randperm(n, generator=gen, device=dev)
src, dst = perm[:m], perm[m:2 * m]
for lo in range(0, m, step):
    x[dst[lo:lo + step]] = x[src[lo:lo + step]] + 0.1 * torch.randn((min(step, m - lo), d), generator=gen, device=dev)
for lo in range(0, n, step):
    blk = x[lo:lo + step]
    blk /= blk.norm(dim=-1, keepdim=True)
planted = sort_pairs(torch.stack([torch.minimum(src, dst), torch.maximum(src, dst)], 1), n)
x16 = x.to(torch.bfloat16)
max_norm = _max_row_norm(x)
scale = max(1.0, max_norm * max_norm * 1.0001)
margins = {"tc_margin": tc_margin(d, max_norm), "previous_0.0045": 0.0045 * scale}

cap = cand_cap = max(4096, 2 * m)
pairs = torch.empty((cap, 2), dtype=torch.int64, device=dev)
counts = torch.zeros(2, dtype=torch.int64, device=dev)
ws_bytes = _cabi.lib.mmrs_selfjoin_tc_workspace_bytes(n, cand_cap)
ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)


def join(margin, rows):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    st = _cabi.lib.mmrs_selfjoin_pairs_tc(x.data_ptr(), x.stride(0), x16.data_ptr(), x16.stride(0), rows, d, tau,
                                          margin, 0, 1, pairs.data_ptr(), cap, counts.data_ptr(), cand_cap,
                                          DeviceGallery.aligned_ptr(ws), ws_bytes, _stream_handle(dev))
    ev1.record()
    torch.cuda.synchronize()
    _cabi.check(st)
    return ev0.elapsed_time(ev1) / 1e3


join(margins["tc_margin"], 65536)                    # warm-up: module load
name = torch.cuda.get_device_name(dev)
for rep in range(repeats):
    for label, margin in (margins.items() if rep % 2 == 0 else reversed(list(margins.items()))):
        t = join(margin, n)
        found, n_cand = counts.tolist()
        got = sort_pairs(pairs[:found], n)
        print(json.dumps({"config": f"C3 {n} x {d}, tau {tau}, one GPU ({name})", "margin": label,
                          "margin_value": margin, "join_seconds": round(t, 3), "candidates": n_cand,
                          "pairs_found": found, "planted": m,
                          "pairs_equal_planted": bool(got.shape == planted.shape and torch.equal(got, planted))}),
              flush=True)
