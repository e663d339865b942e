"""Trajectory evaluation on the GPU (spectral_eval_device, eval.cuh): against the NumPy reference of tests/eval_ref.py on
synthetic trajectories, against the solver's own samples and constraints on real solves, in a receding-horizon loop
that never leaves the device, at sizes past 2^31 output elements, and on invalid arguments."""
import ctypes

import numpy as np
import pytest

import eval_ref as R
from spectral_b200 import api

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def planner():
    p = api.SpectralPlanner(device=0, max_batch=1024, n_max=128, r_max=8, k_max=32)
    yield p
    p.close()


def to_dev(K, status, segs, ctrl):
    import torch
    dev = torch.device("cuda", 0)
    return dict(K=torch.from_numpy(np.ascontiguousarray(K)).to(dev), status=torch.from_numpy(np.ascontiguousarray(status)).to(dev),
                segs=torch.from_numpy(np.ascontiguousarray(segs).view(np.uint8).reshape(len(K), -1)).to(dev),
                ctrl=torch.from_numpy(np.ascontiguousarray(ctrl)).to(dev))


def run(planner, outs, times, B=None, jerk=True, stream=None):
    import torch
    st, jk, hz = planner.eval_device(outs, torch.from_numpy(np.ascontiguousarray(times)).cuda(), B=B, jerk=jerk, stream=stream)
    torch.cuda.synchronize()
    return st.cpu().numpy(), (jk.cpu().numpy() if jk is not None else None), hz.cpu().numpy()


def probe_grid(K, segs, k_max):
    rows = [R.probe_times(segs[b]["t"], min(int(K[b]), k_max), 16, seed=b) for b in range(len(K))]
    T = max(len(r) for r in rows)
    return np.stack([np.pad(r, (0, T - len(r)), constant_values=0.5) for r in rows])


# ---------------------------------------------------------------- 3: synthetic trajectories vs NumPy
def test_eval_matches_numpy_shared_and_per_scenario_times(planner):
    K, status, segs, ctrl = R.synthetic(256, 32, seed=3)
    outs = to_dev(K, status, segs, ctrl)
    times = probe_grid(K, segs, 32)
    st, jk, hz = run(planner, outs, times)
    rst, rjk, rhz = R.ref_eval(K, status, segs, ctrl, 32, times)
    R.assert_close(st, rst, "states")
    R.assert_close(jk, rjk, "jerk")
    assert np.array_equal(hz, rhz, equal_nan=True)
    shared = times[0]
    a = run(planner, outs, shared)
    b = run(planner, outs, np.tile(shared, (len(K), 1)))
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    R.assert_close(a[0], R.ref_eval(K, status, segs, ctrl, 32, shared)[0], "shared")


# ---------------------------------------------------------------- 4: real solves
def reference_grid(K, segs_t, delta):
    out, T0 = [0.0], 0.0
    for k in range(K):
        t = float(segs_t[k])
        linter = int(t / delta)
        out += [T0 + (l / linter) * t for l in range(1, linter + 1)]
        T0 += t
    return out


def device_inputs(batch, weights):
    import torch
    dev = torch.device("cuda", 0)
    names = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")
    inputs = {n: torch.from_numpy(np.ascontiguousarray(a)).to(dev) for n, a in zip(names, batch.arrays())}
    inputs["weights"] = torch.tensor(weights, dtype=torch.float64, device=dev)
    return inputs


def test_eval_on_real_solves(planner):
    import torch
    from spectral_b200.scenarios import GOLDEN_W_CUB, config2
    B, cap = 1024, 200
    batch = config2(B)
    outs = planner.alloc_device_outputs(B, samples_cap=cap)
    planner.solve_device("cub", batch.n_knots, batch.n_regions, batch.delta_t, device_inputs(batch, GOLDEN_W_CUB), outs)
    torch.cuda.synchronize()
    K, status, flags, npts = (outs[k].cpu().numpy() for k in ("K", "status", "flags", "npts"))
    segs = outs["segs"].cpu().numpy().view(api.CUBE_DTYPE)
    ctrl, samples = outs["ctrl"].cpu().numpy(), outs["samples"].cpu().numpy()
    ok = status <= api.SOLVED_INACCURATE
    assert ok.sum() > B // 4
    # the reference sampler's grid: the samples, row for row
    grids = [reference_grid(int(K[b]), segs[b]["t"], batch.delta_t) if ok[b] else [0.0] for b in range(B)]
    T = max(len(g) for g in grids)
    times = np.stack([np.pad(g, (0, T - len(g)), constant_values=g[-1]) for g in grids])
    st, jk, hz = run(planner, outs, times)
    for b in np.nonzero(ok)[0]:
        n = int(npts[b])
        assert len(grids[b]) == n
        assert np.abs(st[b, 1:n] - samples[b, 1:n]).max() <= 1e-9, b
    assert np.isnan(st[~ok]).all() and np.isnan(hz[~ok]).all()
    # verified scenarios: tau = 0 is the initial state and the trajectory is continuous in (s, ds, dds) at every joint, both
    # to the row feasibility a verified polish guarantees (eval_ref.verified_row_bounds / state_tolerances)
    ver = np.nonzero(ok & ((flags & api.FLAG_VERIFIED) == api.FLAG_VERIFIED))[0]
    assert len(ver) > 50
    n_joints = 0
    for b in ver[:200]:
        Kb = int(K[b])
        t = segs[b]["t"][:Kb]
        rows = R.verified_row_bounds("cub", batch, b, GOLDEN_W_CUB, segs[b, :Kb], ctrl[b, :12 * Kb])
        init_tol, joint_tol = R.state_tolerances(rows, t, Kb)
        assert (np.abs(st[b, 0] - batch.init[b]) <= init_tol).all(), (b, st[b, 0] - batch.init[b], init_tol)
        ends = np.cumsum(t)
        jidx = [k for k in range(Kb - 1) if t[k] > R.MIN_T and t[k + 1] > R.MIN_T]
        if not jidx:
            continue
        left = np.array([ends[k] for k in jidx])
        right = np.nextafter(left, np.inf)   # the first time that belongs to segment k + 1
        sl = run(planner, {n: v[b:b + 1] for n, v in outs.items()}, np.concatenate([left, right]), jerk=False)[0][0]
        jump = np.abs(sl[:len(jidx)] - sl[len(jidx):])
        assert (jump <= joint_tol[jidx] + 1e-12 * (1 + np.abs(sl[:len(jidx)]))).all(), (b, jump, joint_tol[jidx])
        n_joints += len(jidx)
    assert n_joints > 100
    # jerk = d(dds)/dtau: central differences at segment midpoints; tolerance = truncation h^2/6 max|d4 s| (d4 s =
    # 120 sum D4c_i B1_i / t^3) plus the rounding of the two dds values over 2h.  dds = 20 sum D2c_i B3_i / t cancels
    # control points of size max|c| (positions / t), so each dds carries up to 64 ulp of 20 max|c| / t
    for b in ver[:100]:
        Kb = int(K[b])
        t = segs[b]["t"][:Kb]
        T0 = np.concatenate([[0.0], np.cumsum(t)[:-1]])
        ks = [k for k in range(Kb) if t[k] > 1e-3]
        h = np.array([1e-4 * t[k] for k in ks])
        mid = np.array([T0[k] + 0.5 * t[k] for k in ks])
        tt = np.concatenate([mid, mid - h, mid + h])
        s1, j1, _ = run(planner, {n: v[b:b + 1] for n, v in outs.items()}, tt)
        n = len(ks)
        for ax in range(2):
            dds_m, dds_p = s1[0, n:2 * n, 3 * ax + 2], s1[0, 2 * n:, 3 * ax + 2]
            fd = (dds_p - dds_m) / (2 * h)
            c = np.array([ctrl[b, 6 * Kb * ax + 6 * k:6 * Kb * ax + 6 * k + 6] for k in ks])
            d4 = np.abs(np.diff(c, 4, axis=1)).max(1) * 120.0 / t[ks] ** 3
            rnd = 64 * np.finfo(np.float64).eps * 20.0 * np.abs(c).max(1) / t[ks]
            tol = h ** 2 / 6 * d4 + 2 * rnd / (2 * h)
            assert (np.abs(j1[0, :n, ax] - fd) <= tol).all(), (b, ax, np.abs(j1[0, :n, ax] - fd), tol)


# ---------------------------------------------------------------- 5: receding horizon on the device
def test_receding_horizon_on_device(planner):
    import torch
    from spectral_b200.scenarios import GOLDEN_W_TRP, load_fixture, random_obstacles
    from spectral_b200.wire import ScenarioBatch
    dev = torch.device("cuda", 0)
    B, Rc = 512, 8
    base = load_fixture("c1")
    obs, n_obs = random_obstacles(B, max_obs=2, seed=5)
    sb, lb, nl = planner.bounds_device(torch.from_numpy(obs).to(dev), base.n_knots, Rc, n_obs=torch.from_numpy(n_obs).to(dev))
    tile = lambda a: torch.from_numpy(np.ascontiguousarray(np.broadcast_to(a, (B,) + np.shape(a)))).to(dev)  # noqa: E731
    init0 = tile(np.concatenate([base.init_s, base.init_l]))
    inputs = dict(s_bounds=sb, l_bounds=lb, ds_bounds=tile(base.ds_bounds), dl_bounds=tile(base.dl_bounds), s_ref=tile(base.s_ref),
                  l_ref=tile(base.l_ref), init=init0, scalars=tile(base.scalars),
                  weights=torch.tensor(GOLDEN_W_TRP, dtype=torch.float64, device=dev))
    outs1 = planner.alloc_device_outputs(B)
    planner.solve_device("trp", base.n_knots, Rc, base.delta_t, inputs, outs1)
    tau = torch.tensor([base.delta_t], dtype=torch.float64, device=dev)
    st, _, _ = planner.eval_device(outs1, tau)                       # [B, 1, 6]: the plan one step ahead
    nxt = torch.where(torch.isnan(st[:, 0]).any(1, keepdim=True), init0, st[:, 0]).contiguous()
    outs2 = planner.alloc_device_outputs(B)
    planner.solve_device("trp", base.n_knots, Rc, base.delta_t, dict(inputs, init=nxt), outs2)
    st2, _, _ = planner.eval_device(outs2, torch.zeros(1, dtype=torch.float64, device=dev))
    # the evaluated states feed the downstream kernel as samples with npts = T
    ego = planner.ego_states_device(st, torch.ones(B, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.float64, device=dev))
    torch.cuda.synchronize()
    ok1 = (outs1["status"] <= api.SOLVED_INACCURATE).cpu().numpy()
    assert ok1.sum() > B // 8 and not np.isnan(st.cpu().numpy()[ok1]).any()
    ego = ego.cpu().numpy()
    assert np.array_equal(ego[ok1, 0, :2], st.cpu().numpy()[ok1, 0][:, [0, 3]])
    flags, status, K = outs2["flags"].cpu().numpy(), outs2["status"].cpu().numpy(), outs2["K"].cpu().numpy()
    ver = np.nonzero((status <= api.SOLVED_INACCURATE) & ((flags & api.FLAG_VERIFIED) == api.FLAG_VERIFIED))[0]
    assert len(ver) > B // 16
    fed, got0 = nxt.cpu().numpy(), st2.cpu().numpy()[:, 0]
    segs = outs2["segs"].cpu().numpy().view(api.CUBE_DTYPE)
    ctrl = outs2["ctrl"].cpu().numpy()
    batch2 = ScenarioBatch(base.n_knots, Rc, base.delta_t, sb.cpu().numpy(), lb.cpu().numpy(), *[inputs[k].cpu().numpy() for k in
                           ("ds_bounds", "dl_bounds", "s_ref", "l_ref")], fed, inputs["scalars"].cpu().numpy())
    for b in ver[:100]:
        Kb = int(K[b])
        rows = R.verified_row_bounds("trp", batch2, b, GOLDEN_W_TRP, segs[b, :Kb], ctrl[b, :12 * Kb])
        init_tol, _ = R.state_tolerances(rows, segs[b]["t"], Kb)
        assert (np.abs(got0[b] - fed[b]) <= init_tol).all(), (b, got0[b] - fed[b], init_tol)


# ---------------------------------------------------------------- 6: determinism
def test_eval_deterministic_across_calls_and_streams(planner):
    import torch
    K, status, segs, ctrl = R.synthetic(4096, 32, seed=9)
    outs = to_dev(K, status, segs, ctrl)
    times = np.linspace(-0.1, 12.0, 777)
    a = run(planner, outs, times)
    b = run(planner, outs, times)
    s = torch.cuda.Stream()
    c = run(planner, outs, times, stream=s.cuda_stream)
    for x, y, z in zip(a, b, c):
        assert x.tobytes() == y.tobytes() == z.tobytes()


# ---------------------------------------------------------------- 7: sizes past 2^31 output elements
def _tiled(B, base=1024, seed=11):
    """B scenarios on the device, scenario b = synthetic scenario b % base (tiled on the device: the host holds `base`)."""
    import torch
    K, status, segs, ctrl = R.synthetic(base, 32, seed=seed)
    idx = np.arange(B) % base
    d_idx = torch.from_numpy(idx).cuda()
    outs = {n: v[d_idx].contiguous() for n, v in to_dev(K, status, segs, ctrl).items()}
    return (K, status, segs, ctrl), outs, idx


@pytest.mark.parametrize("B,T", [(65536, 6000), (1048583, 1)])
def test_eval_sizes_64bit_indexing(planner, B, T):
    import torch
    (K, status, segs, ctrl), outs, idx = _tiled(B)
    times = np.linspace(0.0, 9.0, T) if T > 1 else np.array([0.37])
    st, _, hz = planner.eval_device(outs, torch.from_numpy(times).cuda())
    torch.cuda.synchronize()
    assert st.shape == (B, T, 6)
    rng = np.random.default_rng(B)
    bs = np.concatenate([rng.integers(0, B, 64), [B - 1, B - 2]])
    js = np.concatenate([rng.integers(0, T, 64), [T - 1, max(T - 2, 0)]])
    got = st[torch.from_numpy(bs).cuda(), torch.from_numpy(js).cuda()].cpu().numpy()
    for i, (b, j) in enumerate(zip(bs, js)):
        ref = R.ref_eval_one(int(K[idx[b]]), int(status[idx[b]]), segs[idx[b]]["t"], ctrl[idx[b]], 32, times[j:j + 1])[0][0]
        R.assert_close(got[i], ref, (b, j))
    del st
    torch.cuda.empty_cache()


# ---------------------------------------------------------------- 8: invalid arguments
def test_eval_invalid_arguments(planner):
    import torch
    K, status, segs, ctrl = R.synthetic(8, 32, seed=1)
    outs = to_dev(K, status, segs, ctrl)
    t = torch.linspace(0.0, 1.0, 5, dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        planner.eval_device(outs, t.cpu())                                   # not on the GPU
    with pytest.raises(ValueError):
        planner.eval_device(outs, t.float())                                 # float32
    with pytest.raises(ValueError):
        planner.eval_device(outs, torch.zeros(5, 2, dtype=torch.float64, device="cuda")[:, 0])   # strided
    with pytest.raises(ValueError):
        planner.eval_device(outs, torch.zeros(0, dtype=torch.float64, device="cuda"))           # empty
    with pytest.raises(ValueError):
        planner.eval_device(outs, torch.zeros(4, 5, dtype=torch.float64, device="cuda"))        # [B', T] with B' < B
    with pytest.raises(ValueError):
        planner.eval_device(outs, t, B=9)                                    # more scenarios than the tensors hold
    with pytest.raises(ValueError):
        planner.eval_device(dict(outs, K=outs["K"].long()), t)
    with pytest.raises(ValueError):
        planner.eval_device(dict(outs, ctrl=outs["ctrl"][:, :12]), t)
    with pytest.raises(ValueError):
        planner.eval_device(dict(outs, segs=outs["segs"][:, :112].contiguous()), t)
    lib, h = planner._lib, planner._h
    P = lambda x: ctypes.c_void_p(x.data_ptr())  # noqa: E731
    out = api.SpectralOutputs()
    out.K = ctypes.cast(P(outs["K"]), api._ip)
    out.status = ctypes.cast(P(outs["status"]), api._ip)
    out.segs = outs["segs"].data_ptr()
    out.ctrl = ctypes.cast(P(outs["ctrl"]), api._dp)
    st = torch.zeros(8, 5, 6, dtype=torch.float64, device="cuda")
    INVALID = 1
    call = lambda hh=h, B=8, o=ctypes.byref(out), T=5, tm=P(t), ts=0, s=P(st): lib.spectral_eval_device(hh, B, o, T, tm, ts, s, None, None, None)  # noqa: E731,E501
    assert call(hh=None) == INVALID
    assert call(o=None) == INVALID
    assert call(tm=None) == INVALID
    assert call(s=None) == INVALID
    assert call(B=0) == INVALID
    assert call(T=0) == INVALID
    assert call(ts=2) == INVALID and b"times_stride" in lib.spectral_last_error(h)
    assert call(ts=-1) == INVALID
    for f in ("K", "status", "segs", "ctrl"):
        o2 = api.SpectralOutputs.from_buffer_copy(out)
        setattr(o2, f, None)
        assert call(o=ctypes.byref(o2)) == INVALID, f
    assert call() == 0
    torch.cuda.synchronize()
