#!/usr/bin/env python
"""bench.py -- top-k queries/sec of the B200 search path on BASELINE.json's metric workload.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
    python bench.py --impl reference ...                     (the reference's torch-CPU path)
    python bench.py ... --dump-outputs DIR                   (also save the last timed step's top-k lists)

Headline workload (config.workload = "C4", BASELINE.json configs[3], the shape `metric` is quoted on):
a 100 000 000 x 768 bf16 unit-norm synthetic gallery (153.6 GB -- fits ONE B200), 16 queries per step,
top-100, cosine.  The gallery is row-sharded over the N GPUs (100M / N rows each, generated on the
device, never on the host), queries are replicated, every rank scans its shard, the [Q, k] lists are
all-gathered over NVLink inside the select kernels and merged on every rank.  The global work per
step is the same at every N  ==>  "scaling": "strong"; value = queries / (max-over-ranks step time).

`value`  : device-resident queries and results, CUDA-event timed, max over ranks, 2 batches in flight.
`e2e`    : the same search through the public host API (pinned host queries -> H2D -> search ->
           D2H of values/indices), host clock around status-checked calls.
`roofline`: dominant kernel (the last-phase gallery scan) timed live by the library's CUDA-event
           hooks: algorithmic gallery bytes / duration vs the measured HBM peak.
`cpu_baseline`: the oracle (torch CPU restatement of search_image.py:107 + utils.py:17) on the
           host cores, on a bounded 1M-row slice of the same workload.
`parity_check`: after timing, every rank recomputes its shard's exact top-k with a torch fp32 matmul,
           the lists are all-gathered and merged with a stable sort and compared with what the
           product returned (fused NVLink gather and NCCL variant at N > 1).
Extra keys (never part of `value`):
  `gallery_1m`   N = 1: the 1M x 768 (and 1M x 512, BASELINE configs[1]) single-GPU shapes, Q = 16
                 pipelined + a sweep over Q = 1..256 (blocking and pipelined step times)
  `c5`           BASELINE configs[4]: 65 536 queries over the same sharded gallery (tensor-bound)
  `c3`           BASELINE configs[2]: 10M x 512 self-join, cos >= 0.95, panels dealt over the ranks
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

C4_ROWS = 100_000_000
C4_DIM = 768
TOPK = 100
Q_STEP = 16
C5_QUERIES = 65_536
C3_ROWS, C3_DIM, C3_TAU = 10_000_000, 512, 0.95
CPU_SLICE_ROWS = 1_000_000      # the CPU arm scans this many rows per step and scales linearly in rows


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=C4_ROWS, help="GLOBAL gallery rows (sharded over the GPUs)")
    ap.add_argument("--dim", type=int, default=C4_DIM)
    ap.add_argument("--k", type=int, default=TOPK)
    ap.add_argument("--batch", type=int, default=Q_STEP, help="queries per step (global)")
    ap.add_argument("--path", default="auto", choices=["auto", "gemv", "mma"])
    ap.add_argument("--legs", default="all",
                    help="comma list of extra legs: gallery_1m,c5,c3,parity  ('all', 'none')")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--one-stream", action="store_true", help="keep the batches in flight on ONE stream")
    ap.add_argument("--no-fused", action="store_true", help="N > 1: NCCL all-gather variant instead of the fused NVLink gather")
    ap.add_argument("--c3-rows", type=int, default=C3_ROWS)
    ap.add_argument("--c5-queries", type=int, default=C5_QUERIES)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the top-k lists of the last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the timed search of --impl ours")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, values, indices):
    """What the timed search returned in its last step, for comparing two builds output for output:
    DIR/topk_values.npy (float32 [Q, k]) and DIR/topk_indices.npy (float64 [Q, k], global row ids, exact
    below 2**53).  When the lists would exceed 64 MB, a fixed, seeded sample of query rows is written
    instead, and DIR/query_rows.npy (float64) names the rows kept."""
    import numpy as np
    v = values.cpu().numpy().astype(np.float32)
    i = indices.cpu().numpy().astype(np.float64)
    arrays = {"topk_values": v, "topk_indices": i}
    per_row = v.shape[1] * (v.itemsize + i.itemsize) + 8
    if v.shape[0] * per_row > DUMP_LIMIT_BYTES:
        keep = (DUMP_LIMIT_BYTES - 4096) // per_row          # 4096: room for the three .npy headers
        rows = np.sort(np.random.default_rng(0).choice(v.shape[0], size=keep, replace=False))
        arrays = {"topk_values": v[rows], "topk_indices": i[rows], "query_rows": rows.astype(np.float64)}
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a)


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm": d.get("hbm_gbs", 6650.0), "tc": d.get("bf16_tflops", 1590.0),
                "tc_sustained": d.get("bf16_tflops_sustained", 1400.0), "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tc": 1590.0, "tc_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock and throttle reasons sampled DURING a timed region, in-process through NVML (the
    nvidia-smi child of round 1 needed longer to start than a short region lasts): a thread samples
    every 20 ms (an NVML query is a driver round trip that can delay kernel launches -- per-step
    queries slowed 0.2 ms steps measurably, so the timing loop itself never calls NVML), plus one
    synchronous sample at the end of the region, so that every region has a record."""

    def __init__(self, torch, device):
        self.samples, self.reason_bits, self.max_mhz = [], 0, None
        self.h = self.nv = None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device).uuid)
            uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:   # noqa: BLE001
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device.index or 0)
            self.nv = pynvml
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:   # noqa: BLE001
            self.err = repr(e)

    def _one(self):
        try:
            self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
            self.reason_bits |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:   # noqa: BLE001
            pass

    def _loop(self):
        while not self._stop.wait(0.02):
            self._one()

    def __enter__(self):
        if self.h is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()
        return self

    def mark(self):
        """A synchronous sample taken by the timing thread while the GPU is busy."""
        if self.h is not None:
            self._one()

    def __exit__(self, *a):
        if self.h is not None:
            self._one()
            self._stop.set()
            self._t.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unsampled"], "samples": 0,
                    "error": getattr(self, "err", None)}
        nv = self.nv
        names = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                 ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                 ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
                 ("hw_power_brake_slowdown", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown)]
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz,
                "reasons": [n for n, bit in names if self.reason_bits & bit], "samples": len(sm),
                "how": "NVML in-process, 20 ms period + one sample at the end, during the timed region"}


def device_gallery_shard(torch, rows, dim, seed, shard_id, device):
    """randn rows generated on the device in chunks, unit-normalised in fp32, cast to bf16
    (SURVEY.md section 8d: C2/C4 galleries are never materialised on the host)."""
    gen = torch.Generator(device=device).manual_seed(1000 * seed + shard_id)
    out = torch.empty((rows, dim), dtype=torch.bfloat16, device=device)
    step = 1 << 18
    for lo in range(0, rows, step):
        n = min(step, rows - lo)
        x = torch.randn((n, dim), generator=gen, device=device, dtype=torch.float32)
        out[lo:lo + n] = (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16)
    return out


# ---- the reference's CPU path (oracle port), bounded sample ------------------------------------------------
def cpu_reference(torch, rows_global, dim, nq, k, steps, warmup, budget_s=None):
    """The reference's CPU path on this host: scores = q @ G.T (search_image.py:107, after the
    normalisation idiom :157), then output.topk(k, 1, True, True) (utils.py:17); all host threads.
    A step scans a slice of min(rows_global, 1M) rows; the time of a full step is that scaled
    linearly in rows (a GEMM + a row-wise top-k are both linear in the gallery rows)."""
    from oracle import oracle
    torch.set_num_threads(os.cpu_count() or 1)
    rows = min(rows_global, CPU_SLICE_ROWS)
    g = oracle.synthetic_gallery(rows, dim, seed=0, dtype=torch.bfloat16).to(torch.float32)
    q = oracle.synthetic_queries(nq, dim, seed=1)

    def step():
        s = oracle.l2_normalize(q) @ g.t()
        return s.topk(k, 1, True, True)

    for _ in range(warmup):
        step()
    times = []
    t_end = None if budget_s is None else time.perf_counter() + budget_s
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if t_end is not None and time.perf_counter() > t_end and len(times) >= 2:
            break
    scale = rows_global / rows
    per_step = sum(times) / len(times) * scale
    sample = (f"{len(times)} steps of {nq} queries x a {rows}x{dim} slice (bf16 gallery upcast to fp32), top-{k}"
              + (f"; step time scaled x{scale:g} (linear in rows) for the {rows_global}-row gallery" if scale != 1 else ""))
    return {"value": nq / per_step, "ms_per_step": per_step * 1e3, "steps": len(times),
            "cores": torch.get_num_threads(), "sample": sample}


def workload_config(args, world):
    if (args.rows, args.dim, args.batch, args.k) == (C4_ROWS, C4_DIM, Q_STEP, TOPK):
        name = "C4: 100M x 768 bf16 gallery, 16 queries per step, top-100 cosine (BASELINE.json configs[3])"
    else:
        name = f"{args.rows} x {args.dim} bf16 gallery, {args.batch} queries per step, top-{args.k} cosine"
    per = -(-args.rows // world)
    return {"workload": name, "global_rows": args.rows, "rows_per_gpu": per, "dim": args.dim, "k": args.k,
            "queries_per_step": args.batch, "sharding": f"rows x{world}" if world > 1 else "none",
            "l2": f"gallery shard {per * args.dim * 2 / 1e9:.3f} GB streamed per step > 126 MB L2 (no flush needed)"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port: the
    reference is a set of Python scripts that cannot be installed or imported, DESIGN.md section 3).
    Same config as our arm: the GLOBAL gallery does not depend on N (strong scaling)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    r = cpu_reference(torch, args.rows, args.dim, args.batch, args.k, max(1, args.steps), max(0, args.warmup))
    line = {
        "impl": "reference", "metric": "top-k queries/sec", "value": r["value"], "unit": "queries/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": max(0, args.warmup), "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": r["value"], "unit": "queries/s", "cores": r["cores"], "kind": "port",
                         "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---- our arm ----------------------------------------------------------------------------------------------------
class Bench:
    DEPTH = 2      # batches in flight: the host prepares step i+1 while the GPU runs step i

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import mmrs_b200
        from mmrs_b200 import _cabi
        self.torch, self.dist, self.mm, self.lib = torch, dist, mmrs_b200, _cabi.lib
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        torch.cuda.set_device(self.local_rank)
        self.device = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.device)
        self.peaks = measured_peaks()
        self.streams = None if args.one_stream else [torch.cuda.Stream(device=self.device) for _ in range(self.DEPTH)]
        self.t_start = time.perf_counter()

    # -- helpers --
    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], device=self.device, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def run_steps(self, fn, n, clocks=None):
        """n steps with up to DEPTH batches in flight, alternating over DEPTH streams (each with its
        own workspace slot) so that the short seed/mid kernels of one search overlap the long
        last-phase scan of the other; every batch is waited on and status-checked."""
        torch = self.torch
        inflight, out = [], None
        for i in range(n):
            if self.streams is not None:
                with torch.cuda.stream(self.streams[i % self.DEPTH]):
                    inflight.append(fn(sync=False))
            else:
                inflight.append(fn(sync=False))
            if len(inflight) >= self.DEPTH:
                out = inflight.pop(0).wait()
        for pnd in inflight:
            out = pnd.wait()
        return out

    def searcher(self, gal, sg, q, k):
        mm, path = self.mm, self.args.path
        if sg is not None:
            return lambda sync=True: sg.search_topk(q, k, path=path, sync=sync)
        return lambda sync=True: mm.search_topk(q, gal, k, path=path, sync=sync)

    def measure(self, gal, sg, q_host, k, steps, warmup, *, blocking=True, e2e=True, prof_steps=None,
                e2e_warmup=3):
        """One workload shape: device-timed pipelined steps (`value`), the kernel timeline from the
        library's event hooks, optionally the blocking-call latency and the host-API e2e leg."""
        torch, lib = self.torch, self.lib
        dev = self.device
        nq, dim = int(q_host.shape[0]), int(q_host.shape[1])
        rows_local = gal.n_rows
        q_dev = q_host.to(dev)
        search_dev = self.searcher(gal, sg, q_dev, k)
        search_host = self.searcher(gal, sg, q_host, k)
        warmup = max(warmup, 3)
        res = {"nq": nq, "steps": steps, "warmup": warmup}

        # ---- value: device-resident, CUDA events ----
        self.run_steps(search_dev, warmup)
        self.barrier()
        launches0 = lib.mmrs_launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(torch, dev) as clocks:
            self.barrier()
            ev0.record()
            if self.streams is not None:
                for st in self.streams:
                    st.wait_stream(torch.cuda.current_stream(dev))       # timed region starts at ev0
            out = self.run_steps(search_dev, steps, clocks)
            if self.streams is not None:
                for st in self.streams:
                    torch.cuda.current_stream(dev).wait_stream(st)       # ... and ends when both streams drain
            ev1.record()
            self.barrier()
        res["out"] = out
        ms_total = self.max_over_ranks(ev0.elapsed_time(ev1))
        res["launches"] = int(lib.mmrs_launch_count() - launches0)
        res["clocks"] = clocks.summary()
        res["ms_per_step"] = ms_total / steps
        res["value"] = nq * steps / (ms_total / 1e3)

        # ---- synchronous per-call latency (one batch in flight, host blocks on each) ----
        if blocking:
            for _ in range(3):
                search_dev()
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                search_dev()
            torch.cuda.synchronize()
            res["blocking_call_ms"] = (time.perf_counter() - t0) / steps * 1e3

        # ---- kernel timeline: the same steps with the library's CUDA-event hooks on (the hooks
        # bracket every launch on the launching stream; while they are on the library issues the
        # launches one by one instead of replaying its CUDA graph -- the kernels are the same) ----
        prof_steps = steps if prof_steps is None else prof_steps
        self.barrier()
        lib.mmrs_profile_enable(1)
        for _ in range(prof_steps):
            search_dev()
        torch.cuda.synchronize()
        lib.mmrs_profile_enable(0)
        import ctypes as C
        cap = (res["launches"] // max(steps, 1) + 4) * prof_steps + 64
        ms = (C.c_float * cap)(); kind = (C.c_int32 * cap)(); nbytes = (C.c_int64 * cap)(); flops = (C.c_int64 * cap)()
        nrec = lib.mmrs_profile_read(ms, kind, nbytes, flops, cap)
        recs = [(ms[i], kind[i], nbytes[i], flops[i]) for i in range(nrec) if ms[i] > 0]
        scans = [r for r in recs if r[1] in (1, 2)]
        per_step = nrec // max(prof_steps, 1)
        if per_step and nrec == per_step * prof_steps and per_step <= 64:
            names = {1: "scan_gemv", 2: "scan_mma", 3: "select", 4: "prep"}
            res["kernel_timeline_ms"] = [{"kernel": names.get(kind[j], "?"),
                                          "ms": sum(ms[s * per_step + j] for s in range(prof_steps)) / prof_steps}
                                         for j in range(per_step)]
        res["roofline"] = self.roofline(scans, nq, rows_local, dim, res["ms_per_step"], prof_steps)

        # ---- e2e: host API, host buffers ----
        if e2e:
            self.run_steps(search_host, e2e_warmup)
            self.barrier()
            t0 = time.perf_counter()
            self.run_steps(search_host, steps)
            torch.cuda.synchronize()
            dt = self.max_over_ranks(time.perf_counter() - t0)
            res["e2e"] = {"value": nq * steps / dt, "unit": "queries/s",
                          "h2d_bytes_per_step": nq * dim * 4, "d2h_bytes_per_step": nq * k * 12,
                          "ms_per_step": dt / steps * 1e3,
                          "mode": (f"host API search_topk(host queries, sync=False), {self.DEPTH} batches in flight, every batch waited on and status-checked"
                                   if sg is None else
                                   f"ShardedGallery.search_topk(host queries, sync=False), {self.DEPTH} batches in flight, every batch waited on and status-checked")}
            if blocking:
                for _ in range(3):
                    search_host()
                self.barrier()
                t0 = time.perf_counter()
                for _ in range(steps):
                    search_host()
                torch.cuda.synchronize()
                res["e2e"]["blocking_call_ms"] = (time.perf_counter() - t0) / steps * 1e3
        return res

    def roofline(self, scans, nq, rows_local, dim, ms_per_step, prof_steps):
        """Dominant kernel = the scan launches that stream the most gallery bytes (the last phase)."""
        if not scans:
            return None
        pk = self.peaks
        big = max(r[2] for r in scans)
        dom = [r for r in scans if r[2] == big]
        avg_ms = sum(r[0] for r in dom) / len(dom)
        gbs = big / (avg_ms / 1e3) / 1e9
        tfl = dom[0][3] / (avg_ms / 1e3) / 1e12
        scan_ms = sum(r[0] for r in scans) / max(prof_steps, 1)
        kname = "scan_mma_kernel<filter>" if dom[0][1] == 2 else "scan_gemv_kernel<filter>"
        how = ("CUDA events around every launch of the kernel, on the launching stream, "
               f"{prof_steps} steps re-run with the library's profiling hooks enabled")
        shape = f"{rows_local}x{dim}q{nq}"
        traffic, traffic_src = None, None
        tpath = ROOT / "profiles" / "traffic.json"       # dram bytes of ncu --set full captures, keyed kernel@shape
        if tpath.exists():
            for key, tj in json.loads(tpath.read_text()).items():
                if not key.startswith(kname + "@"):
                    continue
                r_, rest = key.split("@")[1].split("x")
                d_, q_ = rest.split("q")
                if int(d_) == dim and int(q_) == nq and abs(int(r_) - rows_local) <= 1e-3 * rows_local:
                    traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                    traffic_src = f"{tj['source']}, captured at {key.split('@')[1]}"
        if min(nq, 256) >= 224:     # past the ridge (SURVEY.md section 8d: Q* ~ 206-248): tensor-bound
            long_step = ms_per_step > 50.0
            tpk = pk["tc_sustained"] if long_step else pk["tc"]
            return {"bound": "tensor", "achieved": tfl, "peak": tpk, "unit": "TFLOP/s", "frac": tfl / tpk, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": f"{pk['src']} bf16_tflops{'_sustained (step > 50 ms: runs against the power cap)' if long_step else ' (burst)'}",
                    "kernel": kname, "shape": shape, "algorithmic_flops_per_launch": dom[0][3], "avg_launch_ms": avg_ms,
                    "launches_timed": len(dom), "hbm_gbs": gbs,
                    "whole_step_tflops_per_gpu": 2.0 * nq * rows_local * dim / (ms_per_step / 1e3) / 1e12,
                    "frac_of_burst": tfl / pk["tc"], "how": how}
        return {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": f"{pk['src']} hbm_gbs (burst copy)", "kernel": kname, "shape": shape,
                "algorithmic_bytes_per_launch": big, "avg_launch_ms": avg_ms, "launches_timed": len(dom), "tflops": tfl,
                "scan_kernels_ms_per_step": scan_ms, "share_of_step": scan_ms / ms_per_step,
                "whole_step_frac": (rows_local * dim * 2) / (ms_per_step / 1e3) / 1e9 / pk["hbm"],
                "whole_step_note": ("`frac` is the kernel timed one search at a time (profiling hooks): the clean roofline number. "
                                    "`whole_step_frac` divides one gallery pass by the PIPELINED step time; with two searches in flight "
                                    "their scans co-run on every SM and the second reader of a tile can hit L2, and a read-only "
                                    "stream beats the copy the peak was measured with -- so it can exceed 1 and is not a DRAM rate"),
                "how": how}

    # -- legs --
    def parity(self, gal, sg, shard, q_host, k, got):
        """Exact top-k of the same bf16 shard with torch: fp32 matmul of the bf16-rounded normalised
        queries (what bf16 mode scores), per-rank top-k, all-gather, stable sort merge; compared
        with the product's result (`got`), and at N > 1 also with the NCCL (non-fused) variant."""
        torch, dist = self.torch, self.dist
        dev = self.device
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            q = q_host.to(dev)
            qn = (q / q.norm(dim=-1, keepdim=True)).to(torch.bfloat16).to(torch.float32)
            kl = min(k, shard.shape[0])
            best_v = torch.full((q.shape[0], 0), 0.0, device=dev)
            best_i = torch.zeros((q.shape[0], 0), dtype=torch.int64, device=dev)
            step = 1 << 18
            for lo in range(0, shard.shape[0], step):
                blk = shard[lo:lo + step].to(torch.float32)
                s = qn @ blk.t()
                v, i = s.topk(min(kl, s.shape[1]), dim=1)
                best_v = torch.cat([best_v, v], 1)
                best_i = torch.cat([best_i, i + lo + gal.row_offset], 1)
                if best_v.shape[1] > 4 * kl:
                    o = torch.sort(best_v, dim=1, descending=True, stable=True).indices[:, :kl]
                    best_v, best_i = best_v.gather(1, o), best_i.gather(1, o)
            if self.world > 1:
                o = torch.sort(best_v, dim=1, descending=True, stable=True).indices[:, :kl]
                best_v, best_i = best_v.gather(1, o).contiguous(), best_i.gather(1, o).contiguous()
                gv = [torch.empty_like(best_v) for _ in range(self.world)]
                gi = [torch.empty_like(best_i) for _ in range(self.world)]
                dist.all_gather(gv, best_v)
                dist.all_gather(gi, best_i)
                best_v, best_i = torch.cat(gv, 1), torch.cat(gi, 1)
            # order: score desc, index asc (sort by index first, then stable by score)
            o = torch.sort(best_i, dim=1, stable=True).indices
            best_v, best_i = best_v.gather(1, o), best_i.gather(1, o)
            o = torch.sort(best_v, dim=1, descending=True, stable=True).indices[:, :k]
            want_v, want_i = best_v.gather(1, o), best_i.gather(1, o)

            def compare(v, i):
                v, i = v.to(dev), i.to(dev)
                diff = i != want_i
                # a differing position only counts when the two scores really differ: accumulation order
                # (tcgen05 vs cuBLAS fp32) moves scores by ~1e-7 and can swap near-ties
                hard = diff & ((v - want_v).abs() > 1e-5)
                return {"index_mismatches": int(diff.sum().item()), "mismatches": int(hard.sum().item()),
                        "max_abs_score_diff": float((v - want_v).abs().max().item())}

            out = {"checked_queries": int(q.shape[0]), "k": k, "reference": "torch fp32 matmul on the bf16 shard + stable sort merge"}
            out["product"] = compare(*got)
            ok = out["product"]["mismatches"] == 0 and out["product"]["max_abs_score_diff"] < 1e-4
            if sg is not None:
                sg_nccl = self.mm.ShardedGallery(gal, sg.n_rows_global, fused=False)
                out["nccl_variant"] = compare(*sg_nccl.search_topk(q, k))
                ok = ok and out["nccl_variant"]["mismatches"] == 0
                out["fused_gather_used"] = bool(sg.fused_active)
            out["mismatches"] = out["product"]["mismatches"] + (out.get("nccl_variant", {}).get("mismatches", 0))
            out["ok"] = bool(ok)
            return out
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev

    def leg_gallery_1m(self, shard768):
        """N = 1: BASELINE's single-GPU shapes, 1M x 768 (a slice of the resident gallery) and 1M x 512."""
        torch, mm = self.torch, self.mm
        out = {}
        for dim in (768, 512):
            if dim == 768:
                gal = mm.DeviceGallery(shard768[:1_000_000])
            else:
                gal = mm.DeviceGallery(device_gallery_shard(torch, 1_000_000, 512, seed=0, shard_id=0, device=self.device))
            q = torch.randn((Q_STEP, dim), generator=torch.Generator().manual_seed(1)).pin_memory()
            r = self.measure(gal, None, q, TOPK, steps=200, warmup=10)
            bytes_step = gal.n_rows * dim * 2
            entry = {"workload": f"1M x {dim} bf16 gallery, {Q_STEP} queries per step, top-{TOPK}", "value": r["value"],
                     "unit": "queries/s", "ms_per_step": r["ms_per_step"], "e2e": r["e2e"], "roofline": r["roofline"],
                     "blocking_call_ms": r["blocking_call_ms"], "clocks": r["clocks"],
                     "kernel_timeline_ms": r.get("kernel_timeline_ms")}
            sweep = []
            for b in (1, 2, 4, 8, 16, 32, 64, 128, 256):
                qd = torch.randn((b, dim), generator=torch.Generator().manual_seed(2)).to(self.device)
                fn = self.searcher(gal, None, qd, TOPK)
                for _ in range(3):
                    fn()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(20):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                blocking_ms = e0.elapsed_time(e1) / 20
                self.run_steps(fn, 4)
                torch.cuda.synchronize()
                e0.record()
                if self.streams is not None:
                    for st in self.streams:
                        st.wait_stream(torch.cuda.current_stream(self.device))
                self.run_steps(fn, 60)
                if self.streams is not None:
                    for st in self.streams:
                        torch.cuda.current_stream(self.device).wait_stream(st)
                e1.record()
                torch.cuda.synchronize()
                per = e0.elapsed_time(e1) / 60
                sweep.append({"batch": b, "ms_pipelined": per, "ms_blocking": blocking_ms, "qps": b / per * 1e3,
                              "hbm_frac": bytes_step / (per / 1e3) / 1e9 / self.peaks["hbm"],
                              "tflops": 2.0 * b * gal.n_rows * dim / (per / 1e3) / 1e12})
            entry["sweep"] = sweep
            entry["sweep_mode"] = ("ms_pipelined: 2 batches in flight on 2 streams, CUDA events over 60 steps; ms_blocking: one "
                                   "blocking call at a time; device-resident queries; hbm_frac = gallery bytes / ms_pipelined / measured peak "
                                   "(two searches in flight can share gallery reads through L2, so > 1 is possible)")
            out[f"1Mx{dim}"] = entry
            del gal
        # SURVEY.md section 8d: unit-gaussian rows are the best case for nobody in particular, but show it -- a
        # clustered gallery (1000 centroids + noise, queries drawn near centroids, stored cluster by cluster).
        # The thresholds come from a strided SAMPLE's order statistics, which are distribution-free, so the
        # appends per phase (k x ratio) and hence the step time should not move.
        gen = torch.Generator(device=self.device).manual_seed(7)
        cent = torch.randn((1000, 768), generator=gen, device=self.device)
        lab = torch.arange(1000, device=self.device).repeat_interleave(1000)
        g = torch.empty((1_000_000, 768), dtype=torch.bfloat16, device=self.device)
        for lo in range(0, 1_000_000, 1 << 18):
            x = cent[lab[lo:lo + (1 << 18)]] + 0.5 * torch.randn((min(1 << 18, 1_000_000 - lo), 768), generator=gen, device=self.device)
            g[lo:lo + (1 << 18)] = (x / x.norm(dim=-1, keepdim=True)).to(torch.bfloat16)
        gal = mm.DeviceGallery(g)
        q = (cent[torch.arange(0, 1000, 63, device=self.device)[:Q_STEP]] +
             0.3 * torch.randn((Q_STEP, 768), generator=gen, device=self.device)).cpu().pin_memory()
        r = self.measure(gal, None, q, TOPK, steps=200, warmup=10, e2e=False)
        out["1Mx768_clustered"] = {"workload": "1M x 768 bf16 gallery, 1000 clusters stored cluster by cluster, 16 queries near centroids, top-100",
                                   "value": r["value"], "unit": "queries/s", "ms_per_step": r["ms_per_step"], "roofline": r["roofline"],
                                   "blocking_call_ms": r["blocking_call_ms"],
                                   "parity_check": self.parity(gal, None, g, q, TOPK, r["out"])}
        del gal, g
        return out

    def leg_c5(self, gal, sg):
        """BASELINE configs[4]: 64K-query batch over the sharded 100M x 768 gallery (tensor-bound)."""
        torch = self.torch
        nq = self.args.c5_queries
        q = torch.randn((nq, self.args.dim), generator=torch.Generator().manual_seed(1)).pin_memory()
        r = self.measure(gal, sg, q, self.args.k, steps=2, warmup=3, blocking=False, e2e=True, prof_steps=1, e2e_warmup=1)
        flops = 2.0 * nq * self.args.rows * self.args.dim
        agg = flops / (r["ms_per_step"] / 1e3) / 1e12
        return {"workload": f"C5: {nq} queries over the {self.args.rows} x {self.args.dim} bf16 gallery, top-{self.args.k}, {self.world} GPU(s)",
                "value": r["value"], "unit": "queries/s", "ms_per_step": r["ms_per_step"], "steps": 2, "warmup": 3,
                "e2e": r["e2e"], "roofline": r["roofline"], "clocks": r["clocks"], "gpu_launches": r["launches"],
                "whole_step_tflops_aggregate": agg,
                "whole_step_frac_of_measured_burst": agg / (self.world * self.peaks["tc"]),
                "whole_step_frac_of_measured_sustained": agg / (self.world * self.peaks["tc_sustained"]),
                "target": "north_star: >= 60 % of bf16 tensor peak on 8 GPUs (<= 1.29 s per batch against the measured burst peak)"}

    def leg_c3(self):
        """BASELINE configs[2]: N x 512 near-duplicate self-join, cos >= 0.95; every rank holds the
        matrix (replicated, generated from one seed), joins its column panels, pair lists are gathered
        and compared with the planted set."""
        torch, dist = self.torch, self.dist
        from mmrs_b200.dedup import selfjoin_tc_raw, sort_pairs
        dev = self.device
        n, d = self.args.c3_rows, C3_DIM
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
        planted = torch.stack([torch.minimum(src, dst), torch.maximum(src, dst)], 1)
        planted = sort_pairs(planted, n)
        x16 = x.to(torch.bfloat16)
        selfjoin_tc_raw(x[:65536], C3_TAU, x16=x16[:65536])          # warm-up (module load, buffers)
        self.barrier()
        with ClockSampler(torch, dev) as clocks:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            mine = selfjoin_tc_raw(x, C3_TAU, self.rank, self.world, x16=x16, capacity=max(4096, 2 * m))
            ev1.record()
            torch.cuda.synchronize()
            clocks.mark()
        t_join = self.max_over_ranks(ev0.elapsed_time(ev1) / 1e3)
        # gather the variable-length pair lists (counts, then padded buffers) and sort
        t0 = time.perf_counter()
        if self.world > 1:
            cnt = torch.tensor([mine.shape[0]], dtype=torch.int64, device=dev)
            cnts = [torch.empty_like(cnt) for _ in range(self.world)]
            dist.all_gather(cnts, cnt)
            mx = int(max(int(c.item()) for c in cnts))
            buf = torch.zeros((max(mx, 1), 2), dtype=torch.int64, device=dev)
            buf[:mine.shape[0]] = mine
            bufs = [torch.empty_like(buf) for _ in range(self.world)]
            dist.all_gather(bufs, buf)
            mine = torch.cat([b[:int(c.item())] for b, c in zip(bufs, cnts)], 0)
        pairs = sort_pairs(mine, n)
        torch.cuda.synchronize()
        t_gather = self.max_over_ranks(time.perf_counter() - t0)
        ok = pairs.shape == planted.shape and bool(torch.equal(pairs, planted))
        total_pairs = n * (n - 1) / 2
        tf = 2 * d * total_pairs / t_join / 1e12
        return {"workload": f"C3: {n} x {d} self-join, cos >= {C3_TAU}, {self.world} GPU(s), tcgen05 prefilter + exact fp32 recheck",
                "join_seconds": t_join, "gather_sort_seconds": t_gather, "pairs_found": int(pairs.shape[0]), "planted": int(m),
                "pair_set_equals_planted": ok, "pair_dots_per_s": total_pairs / t_join, "tflops_aggregate": tf,
                "frac_of_measured_burst": tf / (self.world * self.peaks["tc"]),
                "frac_of_measured_sustained": tf / (self.world * self.peaks["tc_sustained"]),
                "timing": "one join, CUDA events on the launching stream, max over ranks (a one-shot job: no repeated steps)",
                "clocks": clocks.summary()}


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    b = Bench(args)
    torch, mm = b.torch, b.mm
    world, rank = b.world, b.rank
    legs = {"gallery_1m", "c5", "c3", "parity"} if args.legs == "all" else (
        set() if args.legs == "none" else set(args.legs.split(",")))

    from mmrs_b200.sharded import shard_bounds
    lo, hi = shard_bounds(args.rows, world)[rank]
    shard = device_gallery_shard(torch, hi - lo, args.dim, seed=0, shard_id=rank * 64 + world, device=b.device)
    gal = mm.DeviceGallery(shard, row_offset=lo)
    sg = mm.ShardedGallery(gal, args.rows, fused=False if args.no_fused else None) if world > 1 else None
    q_host = torch.randn((args.batch, args.dim), generator=torch.Generator().manual_seed(1)).pin_memory()
    t_setup = time.perf_counter() - b.t_start

    head = b.measure(gal, sg, q_host, args.k, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:          # every rank holds the merged lists
        dump_outputs(args.dump_outputs, *head["out"])
    gather_desc = None if sg is None else ("fused into the select kernels over NVLink peer memory" if sg.fused_active
                                           else "NCCL all_gather_into_tensor of packed keys + merge kernel")
    extra = {}

    def run_leg(name, fn):
        if name not in legs:
            return
        t0 = time.perf_counter()
        try:
            extra[name] = fn()
        except Exception as e:   # noqa: BLE001 -- a failed extra leg must not cost the headline line
            import traceback
            extra[name] = {"error": f"{type(e).__name__}: {e}", "trace": traceback.format_exc()[-600:]}
            if world > 1:
                raise            # ranks would diverge: fail loudly instead of hanging in a collective
        if isinstance(extra[name], dict):
            extra[name]["leg_seconds"] = round(time.perf_counter() - t0, 2)

    run_leg("parity", lambda: b.parity(gal, sg, shard, q_host, args.k, head["out"]))
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        r = cpu_reference(torch, args.rows, args.dim, args.batch, args.k, steps=200, warmup=1, budget_s=12.0)
        cpu = {"value": r["value"], "unit": "queries/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    if world == 1:
        run_leg("gallery_1m", lambda: b.leg_gallery_1m(shard))
    run_leg("c5", lambda: b.leg_c5(gal, sg))
    if "c3" in legs:
        del gal, sg, shard
        head.pop("out", None)
        torch.cuda.empty_cache()
        run_leg("c3", b.leg_c3)

    if rank == 0:
        line = {
            "metric": "top-k queries/sec", "value": head["value"], "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": head["warmup"], "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args, world), "clocks": head["clocks"], "e2e": head["e2e"],
            "gpu_launches": head["launches"], "roofline": head["roofline"], "cpu_baseline": cpu,
            "pipelining": f"{b.DEPTH} batches in flight" + ("" if args.one_stream else f" on {b.DEPTH} streams"),
            "gather": gather_desc,
            "blocking_call_ms": head.get("blocking_call_ms"),
            # one gallery pass per step / step time / (N x measured copy peak); see roofline.whole_step_note
            "aggregate_hbm_frac": (args.rows * args.dim * 2) / (head["ms_per_step"] / 1e3) / 1e9 / (world * b.peaks["hbm"]),
            "setup_seconds": round(t_setup, 2), "total_seconds": round(time.perf_counter() - b.t_start, 2),
        }
        if "kernel_timeline_ms" in head:
            line["kernel_timeline_ms"] = head["kernel_timeline_ms"]
        if "parity" in extra:
            line["parity_check"] = extra.pop("parity")
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        b.dist.destroy_process_group()


if __name__ == "__main__":
    main()
