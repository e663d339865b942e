"""Feasibility certificate on one GPU: time of spectral_certify_device next to the solve of the same batch, and what it finds.

    python tools/certify_bench.py [--iters 50] [--json out.json]

Time.  config-2 scenarios (cuboid, GOLDEN_W_CUB) solved once at B = 1024; inputs and outputs tiled on the device to
B = 1 024, 65 536 and 1 048 576.  "call" is certify_device through the Python API (outputs allocated by the call), "graph"
the kernel alone, captured in a CUDA graph into preallocated outputs and replayed (tools/eval_bench.py's timers).  "bytes" is
what one call must move: status, K, a_cost, init, scalars and the written viol / cost per scenario, the K segments (112 B)
and control points (96 B) per segment, the ds_bounds knots the segments span and the l-axis' 5 dl_bounds knots.  The solve
time is one spectral_solve_batch_device call on the tiled inputs (the solver's iteration counts are the tiles').

Findings.  config 2 (1024 cuboid scenarios) and config 4 (bench.py --config 4: mixed_batches(262 144), trp and cub) solved
at the default settings: per status class (verified = SOLVED or SOLVED INACCURATE with a KKT proof on both axes; SOLVED
without it; SOLVED INACCURATE without it) the quantiles of the largest violation per family (over both axes, in the QP's row units); the certified share
of the solved scenarios at tol in {1e-9, 1e-6, 1e-5, 1e-3}; and whether the sweep's arg-min moves once uncertified
scenarios are excluded.  Prints the GPU name and power limit.
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from spectral_b200 import api  # noqa: E402
from eval_bench import gpu_info, graph_us, time_us  # noqa: E402

SIZES = (1024, 65536, 1048576)
TOLS = (1e-9, 1e-6, 1e-5, 1e-3)
QUANTILES = (0.5, 0.9, 0.99, 1.0)
NAMES = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")


def device_inputs(batch, weights, dev):
    import torch
    inputs = {n: torch.from_numpy(np.ascontiguousarray(a)).to(dev) for n, a in zip(NAMES, batch.arrays())}
    inputs["weights"] = torch.tensor(weights, dtype=torch.float64, device=dev)
    return inputs


def call_bytes(K, status, segs, B):
    """Bytes one call moves for B scenarios tiled from the base scenarios (K, status [n], segs [n, k_max] CUBE_DTYPE)."""
    n = len(K)
    ok = status <= api.SOLVED_INACCURATE
    live = (np.arange(segs.shape[1])[None, :] < K[:, None]) & ok[:, None]
    knots = int(((segs["end_t"] - segs["beg_t"] + 1) * live).sum())
    per_scen = 4 + 4 + 8 + 2 * 4 * 8 + 8           # status, K, a_cost; viol and cost written
    per_ok = 48 + 80 + 5 * 16                       # init, scalars, the l-axis dl_bounds knots
    base = n * per_scen + int(ok.sum()) * per_ok + int(K[ok].sum()) * (112 + 96) + knots * 16
    return base * B // n


def summarize(viol, status, flags, a_cost, cost_by_tol):
    """viol [B, 2, 4] -> per class, per family quantiles of the max over the axes; certified shares; arg-min moves."""
    ok = status <= api.SOLVED_INACCURATE
    ver = ok & ((flags & api.FLAG_VERIFIED) == api.FLAG_VERIFIED)
    classes = {"verified": ver, "solved_not_verified": (status == api.SOLVED) & ~ver,
               "solved_inaccurate_not_verified": (status == api.SOLVED_INACCURATE) & ~ver}
    fam = np.full((len(status), viol.shape[2]), np.nan)
    fam[ok] = viol[ok].max(axis=1)   # [B, 4]: the larger of the two axes
    out = {"scenarios": int(len(status)), "solved": int(ok.sum())}
    for name, m in classes.items():
        q = {}
        for f, fname in enumerate(api.CERT_FAMILIES):
            q[fname] = [float(np.quantile(fam[m, f], p)) for p in QUANTILES] if m.any() else None
        out[name] = dict(count=int(m.sum()), quantiles=q)
    best = int(np.argmin(a_cost))
    out["argmin"] = best
    out["tol"] = {}
    for tol, cost in cost_by_tol.items():
        cert = cost < api.FAIL_COST
        nb = int(np.argmin(cost))
        out["tol"]["%g" % tol] = dict(certified=int(cert.sum()), share_of_solved=float(cert.sum() / max(1, ok.sum())),
                                      argmin=nb, argmin_moves=bool(nb != best and cost[nb] < api.FAIL_COST))
    return out


def findings(pl, dev, label, parts):
    """parts: list of (variant, batch, weights); solved and certified part by part, summarized as one sweep."""
    import torch
    acc = dict(viol=[], status=[], flags=[], a_cost=[], cost={t: [] for t in TOLS})
    for variant, batch, w in parts:
        B = batch.batch
        inputs = device_inputs(batch, w, dev)
        outs = pl.alloc_device_outputs(B)
        pl.solve_device(variant, batch.n_knots, batch.n_regions, batch.delta_t, inputs, outs)
        viol, _ = pl.certify_device(variant, batch.n_knots, inputs, outs, 0.0)
        for t in TOLS:
            acc["cost"][t].append(pl.certify_device(variant, batch.n_knots, inputs, outs, t)[1].cpu().numpy())
        torch.cuda.synchronize()
        acc["viol"].append(viol.cpu().numpy())
        for n in ("status", "flags", "a_cost"):
            acc[n].append(outs[n].cpu().numpy())
        del inputs, outs
    cat = {n: np.concatenate(v) for n, v in acc.items() if n != "cost"}
    res = summarize(cat["viol"], cat["status"], cat["flags"], cat["a_cost"], {t: np.concatenate(v) for t, v in acc["cost"].items()})
    print("\n%s: %d scenarios, %d solved" % (label, res["scenarios"], res["solved"]))
    for cls in ("verified", "solved_not_verified", "solved_inaccurate_not_verified"):
        c = res[cls]
        print("  %-30s %7d  " % (cls, c["count"]) + "  ".join(
            "%s q50/q90/q99/max %s" % (f[:3], "/".join("%.1e" % v for v in c["quantiles"][f]) if c["quantiles"][f] else "-")
            for f in api.CERT_FAMILIES))
    for t, r in res["tol"].items():
        print("  tol %-6s certified %7d (%.4f of solved), arg-min %s" % (t, r["certified"], r["share_of_solved"],
                                                                        "moves" if r["argmin_moves"] else "unchanged"))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--json", type=str, default=None, help="also write the results to this file")
    args = ap.parse_args()
    import torch
    from spectral_b200.scenarios import GOLDEN_W_CUB, config2, mixed_batches
    if not torch.cuda.is_available():
        raise SystemExit("certify_bench: no CUDA device (the measurement has no CPU path)")
    dev = torch.device("cuda", 0)
    name, power = gpu_info(0)
    print("device: %s, power limit: %s" % (name, power))
    pl = api.SpectralPlanner(device=0, max_batch=max(SIZES), n_max=128, r_max=8, k_max=32)
    base = config2(1024)
    N = base.n_knots
    inputs0 = device_inputs(base, GOLDEN_W_CUB, dev)
    outs0 = pl.alloc_device_outputs(1024)
    pl.solve_device("cub", N, base.n_regions, base.delta_t, inputs0, outs0)
    torch.cuda.synchronize()
    K0, st0 = outs0["K"].cpu().numpy(), outs0["status"].cpu().numpy()
    segs0 = outs0["segs"].cpu().numpy().view(api.CUBE_DTYPE)
    tol = np.full(4, 1e-6)
    rows = []
    hdr = "%8s | %9s %9s %8s %8s | %10s %9s" % ("B", "call us", "graph us", "MB", "GB/s", "solve us", "cert/solve")
    print(hdr)
    print("-" * len(hdr))
    for B in SIZES:
        idx = torch.arange(B, device=dev) % 1024
        inputs = {n: v[idx].contiguous() if v.dim() > 1 else v for n, v in inputs0.items()}
        outs = {n: v[idx].contiguous() for n, v in outs0.items()}
        viol = torch.empty(B, 2, 4, dtype=torch.float64, device=dev)
        cost = torch.empty(B, dtype=torch.float64, device=dev)
        inp = api.SpectralInputs()
        for n in ("ds_bounds", "dl_bounds", "init", "scalars"):
            setattr(inp, n, ctypes.cast(ctypes.c_void_p(inputs[n].data_ptr()), api._dp))
        o = api.SpectralOutputs()
        o.K = ctypes.cast(ctypes.c_void_p(outs["K"].data_ptr()), api._ip)
        o.status = ctypes.cast(ctypes.c_void_p(outs["status"].data_ptr()), api._ip)
        o.segs = outs["segs"].data_ptr()
        o.ctrl = ctypes.cast(ctypes.c_void_p(outs["ctrl"].data_ptr()), api._dp)
        o.a_cost = ctypes.cast(ctypes.c_void_p(outs["a_cost"].data_ptr()), api._dp)

        def raw(s):
            rc = pl._lib.spectral_certify_device(pl._h, api.CUB, B, N, ctypes.byref(inp), 1, ctypes.byref(o), api._d(tol),
                                                 ctypes.c_void_p(viol.data_ptr()), ctypes.c_void_p(cost.data_ptr()), ctypes.c_void_p(s))
            if rc:
                raise SystemExit("spectral_certify_device failed: %d" % rc)

        t_call = time_us(lambda: pl.certify_device("cub", N, inputs, outs, 1e-6), args.iters)
        t_graph = graph_us(raw, args.iters)
        # one solve of the same B (warmed at B = 1024 above); its outputs go to scratch tensors
        souts = pl.alloc_device_outputs(B)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pl.solve_device("cub", N, base.n_regions, base.delta_t, inputs, souts)
        e1.record()
        e1.synchronize()
        t_solve = e0.elapsed_time(e1) * 1e3
        nbytes = call_bytes(K0, st0, segs0, B)
        gbs = nbytes / (t_graph * 1e-6) / 1e9
        rows.append(dict(B=B, call_us=t_call, graph_us=t_graph, bytes=nbytes, gbs=gbs, solve_us=t_solve))
        print("%8d | %9.1f %9.1f %8.1f %8.0f | %10.0f %9.4f" % (B, t_call, t_graph, nbytes / 1e6, gbs, t_solve, t_graph / t_solve))
        del inputs, outs, souts, viol, cost
        torch.cuda.empty_cache()
    del inputs0, outs0
    res2 = findings(pl, dev, "config 2", [("cub", base, GOLDEN_W_CUB)])
    from spectral_b200.scenarios import WEIGHTS_FILE
    res4 = findings(pl, dev, "config 4", [(v, b, WEIGHTS_FILE) for v, b in mixed_batches(262144)])
    pl.close()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(device=name, power_limit=power, iters=args.iters, timing=rows, config2=res2, config4=res4), f, indent=1)


if __name__ == "__main__":
    main()
