"""Top-k selection on one GPU: spectral_topk_device against the single-pass floor (spectral_argmin_device) and against what a
user writes without it (a stable torch.sort of the costs, then the first k).

    python tools/topk_bench.py [--iters 200] [--json out.json]

Costs are seeded: uniform in [0, 50) rounded to 0.1 (many exact ties), 30 % failure sentinels (1e11).  Before timing, each
(B, k) checks topk_device against the stable sort bit for bit.  Times are CUDA-event averages over --iters back-to-back
calls after a warm-up, on an explicitly passed stream:
  "call"   through the Python API (what a caller pays; at small B the host launch path can dominate),
  "graph"  the same calls captured in a CUDA graph and replayed (device time without the Python/ctypes launch cost).
"GB/s" is the bytes the kernels must read over the graph time (topk: 6 radix passes + 1 compaction pass over the 8-byte
costs; argmin: one pass).  Prints the GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from spectral_b200 import api  # noqa: E402

L2_BYTES = 126 * 1024 * 1024
TOPK_PASSES_READ = 7   # k_topk_pass x 6 + k_topk_compact (k_topk_finish rereads only the blocks that hold needed ties)


def gpu_info(dev):
    import torch
    name = torch.cuda.get_device_name(dev)
    power = "unknown"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev)],
                           capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            power = r.stdout.strip()
    except Exception:
        pass
    return name, power


def costs(B, seed):
    rng = np.random.default_rng(seed)
    c = np.round(rng.uniform(0.0, 50.0, B), 1)
    c[rng.random(B) < 0.30] = api.FAIL_COST
    return c


def time_us(fn, iters, warmup=10):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def graph_us(fn, iters, per_graph=20):
    """fn(stream) captured `per_graph` times in one CUDA graph; mean device time per call over >= iters replayed calls."""
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):  # warm-up outside the capture (first-use allocations happen here)
        for _ in range(3):
            fn(side.cuda_stream)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cs = torch.cuda.current_stream().cuda_stream
        for _ in range(per_graph):
            fn(cs)
    reps = max(1, (iters + per_graph - 1) // per_graph)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * per_graph)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--sizes", type=str, default="65536,1048576,16777216")
    ap.add_argument("--ks", type=str, default="1,16,256,1024")
    ap.add_argument("--json", type=str, default=None, help="also write the rows to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("topk_bench: no CUDA device (the measurement has no CPU path)")
    dev = torch.device("cuda", 0)
    name, power = gpu_info(0)
    print("device: %s, power limit: %s" % (name, power))
    pl = api.SpectralPlanner(device=0, max_batch=1024, n_max=128, r_max=8, k_max=16)
    rows = []
    hdr = "%10s %5s %4s | %9s %9s %7s | %9s %9s %7s | %9s | %7s" % (
        "B", "k", "L2", "topk call", "graph", "GB/s", "argmin", "graph", "GB/s", "sort call", "speedup")
    print(hdr)
    print("-" * len(hdr))
    for B in [int(x) for x in args.sizes.split(",")]:
        c = torch.from_numpy(costs(B, seed=B)).to(dev)
        bc = torch.empty(1, dtype=torch.float64, device=dev)
        bi = torch.empty(1, dtype=torch.int64, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        t_arg = time_us(lambda: pl.argmin_device(c, 0, bc, bi, stream=st), args.iters)
        g_arg = graph_us(lambda s: pl.argmin_device(c, 0, bc, bi, stream=s), args.iters)
        fits = B * 8 <= L2_BYTES
        for k in [int(x) for x in args.ks.split(",")]:
            oc = torch.empty(k, dtype=torch.float64, device=dev)
            oi = torch.empty(k, dtype=torch.int64, device=dev)

            def topk(s=st):
                pl.topk_device(c, k, 0, oc, oi, stream=s)

            def baseline():
                v, i = torch.sort(c, stable=True)
                return v[:k], i[:k]

            topk()
            v, i = baseline()
            torch.cuda.synchronize()
            if not (torch.equal(oi, i) and torch.equal(oc.view(torch.int64), v.view(torch.int64))):
                raise SystemExit("topk_device differs from the stable sort at B=%d k=%d" % (B, k))
            t_topk = time_us(topk, args.iters)
            g_topk = graph_us(topk, args.iters)
            t_sort = time_us(baseline, args.iters)
            gbs = TOPK_PASSES_READ * 8.0 * B / (g_topk * 1e-6) / 1e9
            gbs_arg = 8.0 * B / (g_arg * 1e-6) / 1e9
            row = dict(B=B, k=k, fits_l2=fits, topk_call_us=t_topk, topk_graph_us=g_topk, topk_read_gbs=gbs, argmin_call_us=t_arg,
                       argmin_graph_us=g_arg, argmin_read_gbs=gbs_arg, stable_sort_us=t_sort, speedup_vs_sort=t_sort / t_topk)
            rows.append(row)
            print("%10d %5d %4s | %9.1f %9.1f %7.0f | %9.1f %9.1f %7.0f | %9.1f | %6.1fx" % (
                B, k, "yes" if fits else "no", t_topk, g_topk, gbs, t_arg, g_arg, gbs_arg, t_sort, t_sort / t_topk))
        del c
        torch.cuda.empty_cache()
    # one sweep_topk call on a single rank, D2H of the records and the payloads included (host clock: the call synchronises)
    B, k, km = 1 << 20, 1024, 16
    rng = np.random.default_rng(7)
    outs = dict(a_cost=torch.from_numpy(costs(B, seed=3)).to(dev),
                K=torch.from_numpy(rng.integers(1, km + 1, B).astype(np.int32)).to(dev),
                segs=torch.zeros(B, km * 112, dtype=torch.uint8, device=dev),
                ctrl=torch.from_numpy(rng.standard_normal((B, 12 * km))).to(dev))
    for _ in range(3):
        pl.sweep_topk(outs, 0, k)
    ts = []
    for _ in range(20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pl.sweep_topk(outs, 0, k)
        ts.append((time.perf_counter() - t0) * 1e6)
    sweep = dict(B=B, k=k, median_us=float(np.median(ts)), min_us=float(np.min(ts)))
    print("sweep_topk (1 rank, B=%d, k=%d, records + payloads to the host): median %.1f us, min %.1f us" % (
        B, k, sweep["median_us"], sweep["min_us"]))
    pl.close()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(device=name, power_limit=power, iters=args.iters, rows=rows, sweep_topk=sweep), f, indent=1)


if __name__ == "__main__":
    main()
