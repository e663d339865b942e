#!/usr/bin/env python
"""bench.py -- corridor+QP trajectory solves/sec of the planning hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W              our arm (CUDA path through the C-ABI)
    python bench.py --impl reference --gpus N --steps K ...    the reference's own CPU code on the host cores

Workload (config.workload): BASELINE.json configs[1] -- scenario_1 (c1.txt), CUBOID corridors (libcub.so
path), a batch of 1024 obstacle-perturbed copies per step and per GPU (SURVEY.md 8d "Config 2", seed
20230531).  One step = one pass of the whole hot path (corridor generation/split/selection, QP assembly,
ADMM solve + polish, Bezier sampling, cost, local argmin) over one batch.  Weak scaling: every rank
processes its own 1024-scenario shards (scenario ids rank*POOL*1024 ...), the only exchange is the final
(cost, index) arg-min gather over NCCL.

value : whole-job solves/s with the inputs already resident in HBM (CUDA events, max over ranks).
        L2 hygiene: the step rotates through a pool of distinct batches whose inputs + outputs exceed the
        126 MB L2 ("inputs larger than L2").
e2e   : same metric through spectral_solve_batch() with HOST buffers (pinned), H2D + D2H inside the timed region.
roofline      : the dominant kernel (k_qpa / k_qpd, batched ADMM; k_qps4 with --config 3): algorithmic FP64 flops / its
                CUDA-event time vs the FP64 FMA peak measured on this device by the library's probe kernel, per solver
                class too; plus `roofline_corridor` (the corridor kernel) and `roofline_side_kernels` (k_bounds and the
                downstream kernels) against the HBM copy bandwidth of MEASURED_PEAKS.json.
cpu_baseline  : the reference's own sources (oracle/_ref, OSQP restated) on all host cores, bounded sample.
Other workloads (supplementary lines, same JSON shape): --config 3 (BASELINE configs[2]: 65 536 shared-KKT variants on the
FP64 tensor cores, --groups 1|8|64), --config 4 (configs[3]: 262 144 mixed trp + cub), --config 5 (configs[4]: the 1 M-scenario
sweep, strong scaling, NCCL arg-min through the C-ABI).
--dump-outputs DIR : after the timed steps, the outputs of the last timed step as DIR/<name>.npy (float64), so that two builds
        can be compared output for output on the same seeded inputs (see dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "corridor+QP trajectory solves/sec"
UNIT = "solves/s"
BATCH = 1024
SEED_NOTE = "config2: c1.txt base, cub, 1024 obstacle-perturbed copies/step/GPU, seed 20230531"


def workload(cfg, groups=8, shared=True):
    """The bench workloads (SURVEY.md 8d).  2 = BASELINE configs[1], the default and the metric's config; 3 = configs[2]."""
    from spectral_b200.scenarios import GOLDEN_W_CUB, WEIGHTS_FILE, config2, config3
    if cfg == 2:
        return dict(name=SEED_NOTE, batch=BATCH, variant="cub", weights=GOLDEN_W_CUB, make=lambda n, first: config2(n, first=first),
                    options={}, pool=16, streams=4)
    if cfg == 3:
        return dict(name="config3: c2.txt base, trp, 65536 synthetic obstacle/time-allocation variants per step and GPU in %d shared-KKT "
                         "groups, seed 20230601; %s" % (groups, "shared-KKT tiles of 8 on FP64 DMMA (SpectralOptions.shared_kkt = 1)" if shared
                                                        else "per-scenario kernels (shared_kkt = 0)"),
                    batch=65536, variant="trp", weights=WEIGHTS_FILE, make=lambda n, first: config3(n, groups=groups, first=first),
                    options=dict(shared_kkt=1) if shared else {}, pool=2, streams=2)
    raise SystemExit("bench.py: --config must be 2 or 3")


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_LIMIT = 64 << 20   # bytes --dump-outputs writes at most
DUMP_SEED = 20231020    # the scenario sample it writes when a step's outputs are larger
# Cube fields the path defines (the reference never initialises t_dif; count is bookkeeping of its push loop)
DUMP_SEG_FIELDS = ("beg_t", "end_t", "t", "beg_l", "end_l", "upp_skew", "upp_bias", "down_skew", "down_bias",
                   "l_upp_skew", "l_upp_bias", "l_down_skew", "l_down_bias", "merge", "split")


def dump_outputs(path, per_scenario, whole=None):
    """Writes one step's outputs as <path>/<name>.npy in float64 (the integer fields convert exactly).

    per_scenario: name -> array or CUDA tensor with one row per scenario (K, segs, ctrl, obj, a_cost, status, ...); `segs`
    (raw 112-byte Cube records or a Cube structured array) is written as one segs_<field>.npy per field.  whole: name ->
    small array written as is (the step's arg-min).  When the rows would take more than 64 MB, a fixed seeded sample of
    scenarios is written instead, in index order, with the sampled scenario indices as scenario_index.npy."""
    from spectral_b200.api import CUBE_DTYPE

    def structured(a):
        return getattr(a.dtype, "names", None) is not None

    def values_per_row(name, a):
        if name == "segs":
            cubes = a.shape[1] if structured(a) else a.shape[1] // CUBE_DTYPE.itemsize
            return cubes * len(DUMP_SEG_FIELDS)
        return int(np.prod(a.shape[1:]))

    n = len(per_scenario["K"])
    row_bytes = 8 * sum(values_per_row(name, a) for name, a in per_scenario.items())
    idx = None
    if n * row_bytes > DUMP_LIMIT:
        # (1 MB of the budget left for the .npy headers and `whole`; 8 bytes per row for scenario_index)
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, (DUMP_LIMIT - (1 << 20)) // (row_bytes + 8), replace=False))
    os.makedirs(path, exist_ok=True)

    def save(name, a):
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))

    for name, a in per_scenario.items():
        if hasattr(a, "cpu"):  # CUDA tensor: only the sampled rows leave the device
            import torch
            a = (a if idx is None else a.index_select(0, torch.from_numpy(idx).to(a.device))).cpu().numpy()
        elif idx is not None:
            a = a[idx]
        if name == "segs":
            cubes = a if structured(a) else np.ascontiguousarray(a).view(CUBE_DTYPE)
            for f in DUMP_SEG_FIELDS:
                save("segs_" + f, cubes[f])
        else:
            save(name, a)
    if idx is not None:
        save("scenario_index", idx)
    for name, a in (whole or {}).items():
        save(name, a.cpu().numpy() if hasattr(a, "cpu") else a)


def _dump_dir(path, rank, world):
    return path if world == 1 else os.path.join(path, "rank%d" % rank)


def _host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def _cpu_reference(batch, weights, n_scen, threads, variant="cub"):
    """The reference's CPU implementation of the path on `n_scen` scenarios: oracle/_ref (the reference's own
    sources + OSQP restatement) when present, else the plain-C port.  Returns (seconds, kind, result)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle as po
    kind = "reference" if po.have_reference() else "port"
    sub = batch.slice(0, n_scen)
    # all host threads, explicitly: torchrun exports OMP_NUM_THREADS=1, which an OpenMP default would obey
    threads = threads if threads > 0 else _host_threads()
    t0 = time.perf_counter()
    r = po.solve_batch(variant, sub, weights, mode=0, nthreads=threads, kind=kind)
    return time.perf_counter() - t0, kind, r


def run_reference(args):
    """--impl reference: the reference's own CPU code, all host threads, same config/metric."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = workload(args.config, args.groups, not args.no_shared)
    cores = _host_threads()
    sample = 256
    batch = wl["make"](sample, 0)
    times = []
    kind = "port"
    for i in range(args.warmup + args.steps):
        dt, kind, result = _cpu_reference(batch, wl["weights"], sample, 0, wl["variant"])
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result)
    total = sum(times)
    value = sample * len(times) / total
    line = {"metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["name"], "batch_per_gpu": wl["batch"], "variant": wl["variant"], "n_knots": batch.n_knots,
                       "n_regions": batch.n_regions},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": "first %d scenarios of the %d-scenario batch per step, OSQP settings of the "
                                       "reference (eps 1e-5, max_iter 5000), OpenMP over scenarios" % (sample, wl["batch"])},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from spectral_b200 import api
    wl = workload(args.config, args.groups, not args.no_shared)
    VAR, W_VEC = wl["variant"], wl["weights"]
    base_opt = api.default_options(**wl["options"]) if wl["options"] else None

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = wl["batch"]
    POOL = args.pool if args.pool > 0 else wl["pool"]
    k_max = 16
    # one handle (= one set of intermediates + one stream) per in-flight step: a 1024-scenario batch fills only part
    # of a B200 (2 CTAs/SM x 148 SMs = 296 scenarios in flight, 3.5 waves with a ragged tail), so consecutive steps
    # are enqueued round-robin on `streams` CUDA streams and overlap
    NS = max(1, args.streams if args.streams > 0 else wl["streams"])
    planners = [api.SpectralPlanner(device=local, max_batch=B, n_max=128, r_max=8, k_max=k_max) for _ in range(NS)]
    planner = planners[0]
    streams = [torch.cuda.Stream(device=dev) for _ in range(NS)]
    # ---- synthetic inputs: POOL distinct batches per rank, resident in HBM
    first = rank * POOL * B
    big = wl["make"](POOL * B, first)
    N, R, delta = big.n_knots, big.n_regions, big.delta_t
    names = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")
    host = {k: np.ascontiguousarray(a) for k, a in zip(names, big.arrays())}
    resident = {k: torch.from_numpy(a).to(dev) for k, a in host.items()}
    w_dev = torch.tensor(W_VEC, dtype=torch.float64, device=dev)
    outs = [planner.alloc_device_outputs(B) for _ in range(POOL)]
    best_cost = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(NS)]
    best_idx = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(NS)]
    in_bytes = sum(a.nbytes for a in host.values()) // POOL
    out_bytes = sum(t.numel() * t.element_size() for t in outs[0].values())
    pool_mb = POOL * (in_bytes + out_bytes) / 1e6

    def slot_inputs(i):
        d = {k: t[i * B:(i + 1) * B] for k, t in resident.items()}
        d["weights"] = w_dev
        return d

    slots = [slot_inputs(i) for i in range(POOL)]
    gather_buf = torch.zeros(world, 2, dtype=torch.float64, device=dev) if world > 1 else None

    def step(i, lane=None, options=None):
        """One pass of the hot path over one batch, enqueued on stream `lane` (round-robin by default)."""
        s = i % POOL
        j = (i % NS) if lane is None else lane
        with torch.cuda.stream(streams[j]):
            planners[j].solve_device(VAR, N, R, delta, slots[s], outs[s], options=options if options is not None else base_opt)
            planners[j].argmin_device(outs[s]["a_cost"], first + s * B, best_cost[j], best_idx[j])
            if world > 1:  # the path's only exchange: (cost, index) arg-min gather
                mine = torch.stack([best_cost[j][0], best_idx[j][0].to(torch.float64)])
                dist.all_gather_into_tensor(gather_buf.view(-1), mine)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, NS)):
        step(i)
    barrier()
    # ---- pass A (kernel accounting, untimed for `value`): a few steps on ONE stream with the per-kernel event ring on,
    #      so that kernel durations are not inflated by overlap with other steps
    planner.get_work(reset=True)
    planner.set_timing(True)
    na = min(args.steps, 8)
    for i in range(na):
        step(args.warmup + i, lane=0)
    barrier()
    kt = planner.get_timing()
    kt_cls = planner.get_class_timing()
    planner.set_timing(False)
    work_a = planner.get_work(reset=True)
    # ---- pass B (the timed region): exactly `steps` steps, round-robin over the streams
    for p in planners:
        p.get_work(reset=True)
    l0 = sum(p.launch_count() for p in planners)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    main = torch.cuda.current_stream()
    e0.record(main)
    for st in streams:
        st.wait_event(e0)
    for i in range(args.steps):
        step(args.warmup + i)
    for st in streams:
        ev = torch.cuda.Event()
        ev.record(st)
        main.wait_event(ev)
    e1.record(main)
    barrier()
    ms = e0.elapsed_time(e1)
    works = [p.get_work(reset=True) for p in planners]
    work = {k: sum(w[k] for w in works) for k in works[0]}
    launches = sum(p.launch_count() for p in planners) - l0
    clk = clocks.stop() if rank == 0 else None
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    value = world * B * args.steps / (ms_max * 1e-3)
    if args.dump_outputs:  # before the supplementary passes below overwrite the output buffers
        last = args.warmup + args.steps - 1
        whole = {"best_cost": best_cost[last % NS], "best_index": best_idx[last % NS]}
        if world > 1:  # what the exchange hands every rank: the arg-min over the ranks' (cost, index), ties -> lowest index
            g = gather_buf.cpu().numpy()
            k = np.lexsort((g[:, 1], g[:, 0]))[0]
            whole.update(global_best_cost=g[k:k + 1, 0], global_best_index=g[k:k + 1, 1])
        dump_outputs(_dump_dir(args.dump_outputs, rank, world), outs[last % POOL], whole)

    # ---- supplementary (not the headline): the same timed loop with one option changed
    def timed_variant(opts):
        for i in range(NS):
            step(i, options=opts)
        barrier()
        for p in planners:
            p.get_work(reset=True)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(main)
        for st in streams:
            st.wait_event(p0)
        for i in range(args.steps):
            step(args.warmup + i, options=opts)
        for st in streams:
            ev = torch.cuda.Event()
            ev.record(st)
            main.wait_event(ev)
        p1.record(main)
        barrier()
        v_ms = torch.tensor([p0.elapsed_time(p1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(v_ms, op=dist.ReduceOp.MAX)
        ws = [p.get_work(reset=True) for p in planners]
        return world * B * args.steps / (float(v_ms.item()) * 1e-3), {k: sum(w[k] for w in ws) for k in ws[0]}

    # (1) SpectralOptions.infeasibility_precheck = 1: provably empty corridors fail at once instead of burning up to max_iter
    #     ADMM iterations like the reference
    pre_value, pre_work = timed_variant(api.default_options(infeasibility_precheck=1, **wl["options"]))
    # (2) SpectralOptions.polish = 0, the reference's own setting (solve_3d.cc:1243): the output is OSQP's eps = 1e-5 iterate, no
    #     refinement to the exact optimum and no KKT proof -- what the polish (on by default) costs
    nopol_value, _nopol_work = timed_variant(api.default_options(polish=0, **wl["options"]))

    # ---- end to end: HOST buffers through the public host API (spectral_solve_batch_async / spectral_wait), the
    #      H2D copy of every step's inputs from page-locked memory, the kernels and the D2H copy of every step's outputs
    #      inside the timed region; NS planners (handle + stream each) are cycled so that the copies and the ragged tail
    #      of one step overlap the kernels of the next -- the way a sweep driver calls the library
    from spectral_b200.wire import ScenarioBatch

    def host_batch(i):
        s = i % POOL
        return ScenarioBatch(N, R, delta, *[host[k][s * B:(s + 1) * B] for k in names])

    hb = [host_batch(i) for i in range(POOL)]
    w_host = np.array(W_VEC)
    # every planner owns page-locked staging buffers; a step's inputs are copied into them (host memcpy, timed) and
    # from there to the device
    best = []
    for i in range(max(3, args.warmup, NS)):
        pl = planners[i % NS]
        if getattr(pl, "_pending", None) is not None:
            pl.wait()
        pl.solve_async(VAR, hb[i % POOL], w_host, options=base_opt)
    for pl in planners:
        if getattr(pl, "_pending", None) is not None:
            pl.wait()
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        pl = planners[i % NS]
        if getattr(pl, "_pending", None) is not None:
            res = pl.wait()
            best.append(float(res.a_cost.min()))  # the step's result is read on the host
        pl.solve_async(VAR, hb[(args.warmup + i) % POOL], w_host, options=base_opt)
    for pl in planners:
        if getattr(pl, "_pending", None) is not None:
            res = pl.wait()
            best.append(float(res.a_cost.min()))
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert len(best) == args.steps
    t_e = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(t_e.item())
    d2h = sum(getattr(res, f).nbytes for f in ("K", "segs", "ctrl", "obj", "a_cost", "status", "iters", "flags", "npts"))
    solved_frac = work["solved"] / max(work["scenarios"], 1.0)

    if rank == 0:
        peaks, peak_src = _peaks()
        fp64_peak = planner.measure_fp64_peak()
        calls = max(kt["calls"], 1)
        qp_ms = kt["qp"] / calls            # pass A: mean per step of the QP stage (the solver classes of one step, forked streams)
        cor_ms = kt["corridor"] / calls
        flops_per_step = work_a["admm_flops"] / max(na, 1)
        flops_var_per_step = work_a["admm_flops_variable"] / max(na, 1)
        iters_per_step = work["admm_iters"] / max(args.steps, 1)
        achieved_tf = flops_per_step / (qp_ms * 1e-3) / 1e12 if qp_ms > 0 else 0.0
        achieved_var_tf = flops_var_per_step / (qp_ms * 1e-3) / 1e12 if qp_ms > 0 else 0.0
        # corridor kernel: algorithmic bytes with the MEASURED segment counts (work counter sum_K), SURVEY.md 8d
        sum_k_step = work_a["sum_K"] / max(na, 1)
        cor_bytes = B * (8 * (4 * R * N + 2 * N) + 4) + 112 * sum_k_step
        cor_gbs = cor_bytes / (cor_ms * 1e-3) / 1e9 if cor_ms > 0 else 0.0
        # ncu-measured DRAM traffic per launch, if a committed profile of THIS build's kernels exists (tools/make_profiles.py)
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        except Exception:
            pass
        cls_names = ("K<=8", "K<=10", "K<=12", "K<=16", "K<=32")
        cls_kern = ("k_qps (shared-KKT DMMA)" if wl["options"].get("shared_kkt") else "k_qpa<8>", "k_qpa<10>", "k_qpd<12>", "k_qpd<16>", "k_qp<32,2>")
        per_class = []
        for c in range(5):
            ms_c = kt_cls[c] / calls
            fl_c = work_a["admm_flops_class%d" % c] / max(na, 1)
            if fl_c > 0 and ms_c > 0:
                per_class.append({"class": cls_names[c], "kernel": cls_kern[c], "ms_per_step": ms_c, "flops_per_step": fl_c,
                                  "achieved_tflops": fl_c / (ms_c * 1e-3) / 1e12, "frac": fl_c / (ms_c * 1e-3) / 1e12 / fp64_peak if fp64_peak else None})
        # CPU baseline: the full batch of one step (bounded: <= 1024 scenarios) on all host cores
        cpu_sample = min(B, 1024)
        dt, kind, _ = _cpu_reference(hb[0], w_host, cpu_sample, 0, VAR)
        ksum = max(sum(kt[k] for k in ("tables", "corridor", "classify", "qp", "finalize")), 1e-9)
        dmma = bool(wl["options"].get("shared_kkt"))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["name"], "batch_per_gpu": B, "variant": VAR, "n_knots": N, "n_regions": R,
                       "k_max": k_max, "streams": NS,
                       "l2": "inputs larger than L2: pool of %d distinct batches, %.0f MB in+out per rank" % (POOL, pool_mb),
                       "solved_fraction": solved_frac, "admm_iters_per_s": world * iters_per_step / (ms_max / args.steps * 1e-3),
                       "mean_axis_iters": iters_per_step / (2 * B),
                       "with_infeasibility_precheck": {
                           "note": "supplementary, NOT the headline: option infeasibility_precheck=1 (sound interval test, include/spectral.h) "
                                   "fails provably empty corridors before the ADMM loop; the reference has no such test",
                           "value": pre_value, "unit": UNIT, "solved_fraction": pre_work["solved"] / max(pre_work["scenarios"], 1.0),
                           "mean_axis_iters": pre_work["admm_iters"] / max(args.steps, 1) / (2 * B)},
                       "with_reference_polish_setting": {
                           "note": "supplementary, NOT the headline: polish = 0 like the reference (solve_3d.cc:1243): outputs are the raw ADMM "
                                   "iterate at eps 1e-5 instead of the polished, KKT-verified optimum the library returns by default",
                           "value": nopol_value, "unit": UNIT}},
            "roofline": {"kernel": ("k_qps (shared-KKT tiles, X~ = G [g1..g8] on mma.sync.m8n8k4.f64) + the per-scenario kernels of K > 8" if dmma else
                                    "k_qpa<8|10> + k_qpd<12|16> (batched dense-operator ADMM + polish; all solver classes of one step)"),
                         "bound": "tensor" if dmma else "fp64",
                         "achieved": achieved_tf, "peak": fp64_peak,
                         "unit": "TFLOP/s", "frac": achieved_tf / fp64_peak if fp64_peak else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per launch from the committed ncu
                         # capture of this build (profiles/r2_traffic.json, written by tools/make_profiles.py), else null
                         "traffic": traffic.get("k_qps" if dmma else "k_qpa<8>"),
                         "traffic_source": traffic.get("source"),
                         "peak_source": "FP64 FMA probe kernel measured in this run (MEASURED_PEAKS.json has no FP64 entry; the DMMA probe "
                                        "profiles/r1_dmma_probe.md measured 37.1 TFLOP/s on the tensor pipe vs 34.9 on the FMA pipe)",
                         "ms_per_launch_group": qp_ms, "flops_per_step": flops_per_step,
                         "count": "dense-operator count 72 K^2 + 208 K - 24 flops per axis-iteration (what the kernels execute)",
                         "variable_structure_count": {"flops_per_step": flops_var_per_step, "achieved": achieved_var_tf,
                                                      "frac": achieved_var_tf / fp64_peak if fp64_peak else None,
                                                      "note": "SURVEY.md 8d count 424 K - 168 per axis-iteration (block-tridiagonal solve): "
                                                              "the algorithmic minimum when no two scenarios share a KKT matrix"},
                         "per_class": per_class,
                         "note": "timed on one stream (pass A, %d steps) with CUDA events around the QP stage; the headline value overlaps %d steps; "
                                 "per_class times are events on each class' own stream (classes overlap)" % (na, NS)},
            "roofline_corridor": {"kernel": "k_corridor", "bound": "hbm", "achieved": cor_gbs, "peak": peaks.get("hbm_gbs"),
                                  "unit": "GB/s", "frac": cor_gbs / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None,
                                  "traffic": traffic.get("k_corridor"), "traffic_source": traffic.get("source"),
                                  "algorithmic_bytes_per_launch": cor_bytes, "mean_K": sum_k_step / max(B, 1),
                                  "peak_source": peak_src, "ms_per_launch": cor_ms,
                                  "note": "bound by the lane-0 replay of the sequential selection logic, not by HBM (profiles/r1_small_kernels.md)"},
            "roofline_side_kernels": _side_kernel_rooflines(planner, dev, peaks, peak_src),
            "kernel_ms_per_step": {k: kt[k] / calls for k in ("tables", "corridor", "classify", "qp", "finalize")},
            # every kernel of the step with the resource that bounds it; shares from the CUDA-event ring of pass A
            "kernels": [
                {"kernel": "QP stage (k_qps / k_qpa / k_qpd / k_qp)", "bound": "fp64 pipe / shared-memory pipe / latency", "share": kt["qp"] / ksum,
                 "frac_of_fp64_peak": achieved_tf / fp64_peak if fp64_peak else None},
                {"kernel": "k_corridor", "bound": "hbm", "share": kt["corridor"] / ksum,
                 "frac_of_hbm_peak": cor_gbs / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None},
                {"kernel": "k_finalize", "bound": "latency", "share": kt["finalize"] / ksum},
                {"kernel": "k_tables + k_classify", "bound": "launch latency (one CTA each)", "share": (kt["tables"] + kt["classify"]) / ksum}],
            "cpu_baseline": {"value": cpu_sample / dt, "unit": UNIT, "cores": _host_threads(), "kind": kind,
                             "sample": "first %d scenarios of one %d-scenario batch, reference OSQP settings" % (cpu_sample, B)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(in_bytes), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "clocks": clk,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_sweep5(args):
    """--config 5: BASELINE configs[4], the 1 M-scenario sweep (config-4 generator, seed 20230603) STRONG-scaled over the
    ranks, ending in the path's only exchange: spectral_sweep_argmin (NCCL all-gather of 16-byte records + winner broadcast
    inside the C-ABI).  One step = one pass over all scenarios + the exchange."""
    import torch
    import torch.distributed as dist
    from spectral_b200 import api, sweep_driver as sd
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    total = args.total if args.total > 0 else (262144 if args.config == 4 else 1048576)
    # --shared: the K <= 8 class of every chunk through structure-sorted shared-KKT tiles (k_qps4); default: per-scenario kernels
    sweep_opt = api.default_options(shared_kkt=1) if args.shared else None
    planner = api.SpectralPlanner(device=local, max_batch=sd.CHUNK, n_max=128, r_max=8, k_max=16)
    ident = [api.SpectralPlanner.comm_unique_id() if (rank == 0 and world > 1) else None]
    if world > 1:
        dist.broadcast_object_list(ident, src=0)
    planner.comm_init(world, rank, ident[0])
    t0 = time.perf_counter()
    shard = sd.upload_shard(total, rank, world, dev)
    gen_s = time.perf_counter() - t0
    n_local = (shard["g_hi"] - shard["g_lo"]) * sd.CHUNK
    outs = planner.alloc_device_outputs(max(n_local, 1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    winner = None
    for _ in range(max(1, args.warmup)):
        winner = sd.run_sweep(planner, shard, outs, options=sweep_opt)
    barrier()
    planner.get_work(reset=True)
    l0 = planner.launch_count()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        winner = sd.run_sweep(planner, shard, outs, options=sweep_opt)
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    work = planner.get_work(reset=True)
    launches = planner.launch_count() - l0
    clk = clocks.stop() if rank == 0 else None
    value = total * args.steps / (float(ms.item()) * 1e-3)
    if args.dump_outputs:
        dump_outputs(_dump_dir(args.dump_outputs, rank, world), {k: t[:n_local] for k, t in outs.items()},
                     {"winner_" + k: np.asarray(winner[k]) for k in ("cost", "index", "rank", "K", "ctrl")})
    # every rank must hold the same winner
    chk = torch.tensor([winner["cost"], float(winner["index"]), float(winner["rank"]), float(winner["K"])], dtype=torch.float64, device=dev)
    if world > 1:
        ref = chk.clone()
        dist.broadcast(ref, src=0)
        assert torch.equal(ref, chk), "ranks disagree on the winner"
    # end to end: a bounded sample of this rank's chunks from page-locked host memory through solve_batch_async
    names = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")
    ns = min(8, len(shard["chunks"]))
    from spectral_b200.wire import ScenarioBatch
    host = []
    for variant, N, R, delta, inp in shard["chunks"][:ns]:
        host.append((variant, ScenarioBatch(N, R, delta, *[inp[k].cpu().numpy() for k in names])))
    pls = [planner, api.SpectralPlanner(device=local, max_batch=sd.CHUNK, n_max=128, r_max=8, k_max=16)]
    w_host = np.array(sd.WEIGHTS_FILE)
    for rep in range(2):   # first repetition warms the staging buffers
        barrier()
        t0 = time.perf_counter()
        for i, (variant, hb) in enumerate(host):
            pl = pls[i % 2]
            if getattr(pl, "_pending", None) is not None:
                pl.wait()
            pl.solve_async(variant, hb, w_host)
        for pl in pls:
            if getattr(pl, "_pending", None) is not None:
                pl.wait()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    t_e = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * ns * sd.CHUNK / float(t_e.item()) if ns else 0.0
    in_bytes = sum(a.nbytes for a in host[0][1].arrays()) if host else 0
    if rank == 0:
        fp64_peak = planner.measure_fp64_peak()
        tf = work["admm_flops"] / (float(ms.item()) * 1e-3) / 1e12
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(1, args.warmup),
                "ms_per_step": float(ms.item()) / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": ("config4: mixed trp+cub batch of %d heterogeneous corridor sequences (K in [4,14], seed 20230603), variable-structure "
                                        "ADMM path, %d rank(s), arg-min of the batch at the end (spectral_sweep_argmin)" if args.config == 4 else
                                        "config5: %d-scenario sweep, config-4 generator (mixed trp+cub, K in [4,14], seed 20230603), contiguous "
                                        "global-index shards over %d rank(s), one NCCL argmin exchange per pass (spectral_sweep_argmin)") % (total, world),
                           "total_scenarios": total, "chunk": sd.CHUNK, "shared_kkt": bool(args.shared), "scenarios_this_rank": n_local,
                           "l2": "inputs larger than L2: %.1f GB resident per rank" % (n_local * 8.1e3 / 1e9),
                           "winner": {"cost": winner["cost"], "index": winner["index"], "rank": winner["rank"], "K": winner["K"]},
                           "solved_fraction": work["solved"] / max(work["scenarios"], 1.0), "generation_s_untimed": gen_s,
                           "mean_axis_iters": work["admm_iters"] / max(work["scenarios"], 1.0) / 2},
                "roofline": {"kernel": "QP stage of rank 0 (k_qpa<8|10> + k_qpd<12|16>)", "bound": "fp64", "achieved": tf, "peak": fp64_peak,
                             "unit": "TFLOP/s", "frac": tf / fp64_peak if fp64_peak else None, "traffic": None,
                             "note": "rank 0's algorithmic flops (dense-operator count) over the whole timed pass, exchange included"},
                "cpu_baseline": None,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(in_bytes) * ns, "d2h_bytes_per_step": None,
                        "sample": "the first %d chunks of every rank's shard from page-locked host buffers (spectral_solve_batch_async, 2 handles)" % ns},
                "gpu_launches": int(launches), "clocks": clk}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _side_kernel_rooflines(planner, dev, peaks, peak_src):
    """The element-wise kernels before / after the path (SURVEY.md 8f rows 1 and 3), each timed alone with CUDA events on the
    launching stream at a size larger than L2: algorithmic bytes / time against the measured HBM copy bandwidth."""
    import torch
    from spectral_b200.scenarios import random_obstacles
    out = []
    hbm = peaks.get("hbm_gbs")

    def timed(fn, reps=10):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    try:
        Bb, N, Rc = 65536, 71, 8
        obs, n_obs = random_obstacles(4096, max_obs=3, seed=20230607)
        d_obs = torch.from_numpy(np.tile(obs, (Bb // 4096, 1, 1))).to(dev)
        d_n = torch.from_numpy(np.tile(n_obs, Bb // 4096)).to(dev)
        ms = timed(lambda: planner.bounds_device(d_obs, N, Rc, n_obs=d_n))
        by = Bb * (3 * 48 + 4 + 2 * Rc * N * 16 + 4)
        out.append({"kernel": "k_bounds", "bound": "hbm", "units": "%d scenarios, <= 3 obstacles, %d lanes x %d knots out" % (Bb, Rc, N),
                    "algorithmic_bytes_per_launch": by, "ms_per_launch": ms, "achieved": by / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                    "frac": by / (ms * 1e-3) / 1e9 / hbm if hbm else None, "peak_source": peak_src})
        cap = 72
        smp = torch.rand(Bb, cap, 6, dtype=torch.float64, device=dev)
        npts = torch.full((Bb,), cap, dtype=torch.int32, device=dev)
        off = torch.zeros(Bb, dtype=torch.float64, device=dev)
        ms = timed(lambda: planner.ego_states_device(smp, npts, off))
        by = Bb * cap * (48 + 32)
        out.append({"kernel": "k_ego_states", "bound": "hbm", "units": "%d trajectories x %d samples" % (Bb, cap), "algorithmic_bytes_per_launch": by,
                    "ms_per_launch": ms, "achieved": by / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                    "frac": by / (ms * 1e-3) / 1e9 / hbm if hbm else None, "peak_source": peak_src,
                    "note": "includes the zero-fill of the output tensor by the Python wrapper"})
        n = Bb * cap
        ref = torch.rand(n, 6, dtype=torch.float64, device=dev)
        sc = torch.rand(n, 3, dtype=torch.float64, device=dev)
        dc = torch.rand(n, 3, dtype=torch.float64, device=dev) * 0.1
        ms = timed(lambda: planner.frenet_to_cartesian_device(ref, sc, dc))
        by = n * (96 + 48)
        out.append({"kernel": "k_frenet_to_cartesian", "bound": "hbm", "units": "%d points" % n, "algorithmic_bytes_per_launch": by,
                    "ms_per_launch": ms, "achieved": by / (ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                    "frac": by / (ms * 1e-3) / 1e9 / hbm if hbm else None, "peak_source": peak_src})
    except Exception as exc:  # a side measurement must never take the headline line down
        out.append({"error": repr(exc)})
    return out


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--pool", type=int, default=0, help="distinct batches resident per rank (0: the workload's default)")
    ap.add_argument("--streams", type=int, default=0, help="steps in flight (one handle + CUDA stream each; 0: the workload's default)")
    ap.add_argument("--config", type=int, default=2, help="2: BASELINE configs[1] (default, the metric's config); 3: configs[2] (shared-KKT, DMMA); 4: configs[3] (262 144 mixed trp+cub, variable structure); 5: configs[4] (1 M sweep, strong scaling)")
    ap.add_argument("--total", type=int, default=0, help="config 4 / 5: scenarios in the batch / sweep (multiple of 8192; default 262144 / 1048576)")
    ap.add_argument("--shared", action="store_true", help="config 4 / 5: route the K <= 8 class through the shared-KKT tile kernel (SpectralOptions.shared_kkt = 1)")
    ap.add_argument("--no-shared", action="store_true", help="config 3 through the per-scenario kernels (A/B of the shared-KKT path)")
    ap.add_argument("--groups", type=int, default=8, help="config 3: number of shared-KKT groups (1, 8, 64)")
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, at most 64 MB; with several ranks "
                         "one DIR/rank<r>/ per rank)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def main(args):
    if args.impl == "reference":
        run_reference(args)
    elif args.config in (4, 5):
        run_sweep5(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    args = parse_args()  # (outside the handler below: a usage error exits with argparse's code 2 and no traceback)
    try:
        main(args)
    except BaseException as exc:  # a rank that dies must not leave its peers waiting in a collective until the launcher's timeout
        if isinstance(exc, SystemExit) and exc.code in (0, None):
            raise
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        os._exit(1)
