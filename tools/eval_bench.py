"""Trajectory evaluation on one GPU: spectral_eval_device against a device-to-device copy of the same number of bytes.

    python tools/eval_bench.py [--iters 50] [--json out.json]

Trajectories are seeded synthetic solves (tests/eval_ref.synthetic: K in [1, 32], durations 0.1 .. 1.0 s, tiled to B
scenarios).  Sizes: (B, T) = (65 536, 1) (the replan step), (65 536, 100), (65 536, 1000) with shared times and
(1024, 1000) with per-scenario times, each with and without jerk.  Times are CUDA-event averages over --iters calls after a
warm-up:
  "call"   through the Python API (output tensors allocated by the call),
  "graph"  the kernel alone, captured in a CUDA graph into preallocated outputs and replayed.
"bytes" is what one call must move: written states (48 B per point) and jerk (16 B), horizons (8 B per scenario), read
times and the scenarios' K, status, durations and control points once.  "GB/s" = bytes / graph time; "copy GB/s" is a
torch device-to-device copy of the same number of bytes measured in the same run.  Prints the GPU name and power limit.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from spectral_b200 import api  # noqa: E402

SIZES = ((65536, 1, 0), (65536, 100, 0), (65536, 1000, 0), (1024, 1000, 1))   # (B, T, times_stride)


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


def time_us(fn, iters, warmup=5):
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


def graph_us(fn, iters, per_graph=10):
    """fn(stream) captured `per_graph` times in one CUDA graph; mean device time per call over >= iters replayed calls."""
    import torch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
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
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--json", type=str, default=None, help="also write the rows to this file")
    args = ap.parse_args()
    import torch
    import eval_ref as R
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench: no CUDA device (the measurement has no CPU path)")
    dev = torch.device("cuda", 0)
    name, power = gpu_info(0)
    print("device: %s, power limit: %s" % (name, power))
    k_max = 32
    pl = api.SpectralPlanner(device=0, max_batch=1024, n_max=128, r_max=8, k_max=k_max)
    K, status, segs, ctrl = R.synthetic(1024, k_max, seed=2024)
    status[:] = api.SOLVED
    K[[6, 7]] = 3   # synthetic() marks a few scenarios invalid; here every scenario is evaluated
    base = dict(K=torch.from_numpy(K).to(dev), status=torch.from_numpy(status).to(dev),
                segs=torch.from_numpy(segs.view(np.uint8).reshape(1024, -1)).to(dev), ctrl=torch.from_numpy(np.nan_to_num(ctrl)).to(dev))
    rows = []
    hdr = "%7s %5s %5s %4s | %9s %9s %9s %8s | %8s" % ("B", "T", "times", "jerk", "call us", "graph us", "MB", "GB/s", "copy GB/s")
    print(hdr)
    print("-" * len(hdr))
    for B, T, stride in SIZES:
        idx = torch.arange(B, device=dev) % 1024
        outs = {n: v[idx].contiguous() for n, v in base.items()}
        H = float(np.max([R.horizon(segs[b]["t"], int(K[b])) for b in range(1024)]))
        if stride:
            times = torch.rand(B, T, dtype=torch.float64, device=dev, generator=torch.Generator(dev).manual_seed(1)) * H
        else:
            times = torch.linspace(0.0, H, T, dtype=torch.float64, device=dev) if T > 1 else torch.tensor([0.1], dtype=torch.float64, device=dev)
        Kd = outs["K"].cpu().numpy()
        read = times.numel() * 8 + B * 8 + int(Kd.sum()) * (8 + 12 * 8)
        for jerk in (False, True):
            written = B * T * (48 + (16 if jerk else 0)) + B * 8
            nbytes = written + read
            st = torch.empty(B, T, 6, dtype=torch.float64, device=dev)
            jk = torch.empty(B, T, 2, dtype=torch.float64, device=dev) if jerk else None
            hz = torch.empty(B, dtype=torch.float64, device=dev)
            o = api.SpectralOutputs()
            o.K = ctypes.cast(ctypes.c_void_p(outs["K"].data_ptr()), api._ip)
            o.status = ctypes.cast(ctypes.c_void_p(outs["status"].data_ptr()), api._ip)
            o.segs = outs["segs"].data_ptr()
            o.ctrl = ctypes.cast(ctypes.c_void_p(outs["ctrl"].data_ptr()), api._dp)

            def raw(s):
                rc = pl._lib.spectral_eval_device(pl._h, B, ctypes.byref(o), T, ctypes.c_void_p(times.data_ptr()), stride,
                                                  ctypes.c_void_p(st.data_ptr()), ctypes.c_void_p(jk.data_ptr()) if jk is not None else None,
                                                  ctypes.c_void_p(hz.data_ptr()), ctypes.c_void_p(s))
                if rc:
                    raise SystemExit("spectral_eval_device failed: %d" % rc)

            t_call = time_us(lambda: pl.eval_device(outs, times, jerk=jerk), args.iters)
            t_graph = graph_us(raw, args.iters)
            src = torch.empty(nbytes // 8, dtype=torch.float64, device=dev)
            dst = torch.empty_like(src)
            t_copy = time_us(lambda: dst.copy_(src), args.iters)
            del src, dst
            gbs, copy_gbs = nbytes / (t_graph * 1e-6) / 1e9, 2 * nbytes / (t_copy * 1e-6) / 1e9
            row = dict(B=B, T=T, per_scenario_times=bool(stride), jerk=jerk, call_us=t_call, graph_us=t_graph, bytes=nbytes,
                       gbs=gbs, copy_us=t_copy, copy_gbs=copy_gbs)
            rows.append(row)
            print("%7d %5d %5s %4s | %9.1f %9.1f %9.1f %8.0f | %8.0f" % (B, T, "B x T" if stride else "T", "yes" if jerk else "no",
                                                                         t_call, t_graph, nbytes / 1e6, gbs, copy_gbs))
            del st, jk, hz
        del outs, times
        torch.cuda.empty_cache()
    print("copy GB/s counts the copy's read and write (2 x bytes); eval GB/s counts the bytes one call must move once.")
    pl.close()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(device=name, power_limit=power, iters=args.iters, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
