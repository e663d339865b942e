"""The feasibility certificate on the GPU (spectral_certify_device, certify.cuh): against the rows of the QP the CPU oracle
assembles (tests/certify_ref.py) on real solves of every solver class and input layout, sound against the interval
pre-check, as the cost that selects the best feasible trajectories, and on invalid arguments."""
import ctypes

import numpy as np
import pytest

import certify_ref as C
from spectral_b200 import api

pytestmark = pytest.mark.gpu

NAMES = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")


@pytest.fixture(scope="module")
def planner():
    p = api.SpectralPlanner(device=0, max_batch=1024, n_max=256, r_max=8, k_max=32)
    yield p
    p.close()


def device_inputs(batch, weights):
    import torch
    dev = torch.device("cuda", 0)
    inputs = {n: torch.from_numpy(np.ascontiguousarray(a)).to(dev) for n, a in zip(NAMES, batch.arrays())}
    inputs["weights"] = torch.from_numpy(np.ascontiguousarray(weights, dtype=np.float64)).to(dev)
    return inputs


def solve(pl, variant, batch, w, **opts):
    inputs = device_inputs(batch, w)
    outs = pl.alloc_device_outputs(batch.batch)
    pl.solve_device(variant, batch.n_knots, batch.n_regions, batch.delta_t, inputs, outs,
                    options=api.default_options(**opts) if opts else None)
    return inputs, outs


def solve_weights(pl, variant, scenario, W):
    """spectral_solve_weights_device: one scenario, B weight vectors (outputs per weight vector, inputs shared)."""
    import torch
    inputs = device_inputs(scenario, W)
    outs = pl.alloc_device_outputs(len(W))
    dp = lambda t: ctypes.cast(ctypes.c_void_p(t.data_ptr()), api._dp)  # noqa: E731
    ip = lambda t: ctypes.cast(ctypes.c_void_p(t.data_ptr()), api._ip)  # noqa: E731
    inp = api.SpectralInputs(*[dp(inputs[n]) for n in NAMES], dp(inputs["weights"]), 1)
    out = api.SpectralOutputs(ip(outs["K"]), ctypes.c_void_p(outs["segs"].data_ptr()), dp(outs["ctrl"]), dp(outs["obj"]),
                              dp(outs["a_cost"]), ip(outs["status"]), ip(outs["iters"]), ip(outs["flags"]), ip(outs["npts"]),
                              None, 0, None)
    pl._check(pl._lib.spectral_solve_weights_device(pl._h, api.VARIANT_ID[variant], len(W), scenario.n_knots, scenario.n_regions,
                                                    float(scenario.delta_t), ctypes.byref(inp), None, ctypes.byref(out),
                                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return inputs, outs


class Host:
    def __init__(self, outs):
        self.K, self.status, self.iters = (outs[n].cpu().numpy() for n in ("K", "status", "iters"))
        self.segs = outs["segs"].cpu().numpy().view(api.CUBE_DTYPE)
        self.ctrl, self.a_cost = outs["ctrl"].cpu().numpy(), outs["a_cost"].cpu().numpy()

    def ok(self):
        return self.status <= api.SOLVED_INACCURATE


def certify(pl, variant, batch, inputs, outs, tol, shared=False):
    import torch
    viol, cost = pl.certify_device(variant, batch.n_knots, inputs, outs, tol, shared_inputs=shared)
    torch.cuda.synchronize()
    return viol.cpu().numpy(), cost.cpu().numpy()


def assert_parity(pl, variant, batch, inputs, outs, label, tol=1e-6, shared=False):
    """Every certifiable scenario within the bar of the oracle; every other one exactly NaN and FAIL_COST; the cost is a_cost
    where the entries are <= tol.  Returns (host outputs, kernel viol, kernel cost, oracle viol, oracle scale)."""
    viol, cost = certify(pl, variant, batch, inputs, outs, tol, shared)
    r = Host(outs)
    ok = r.ok()
    assert np.isnan(viol[~ok]).all() and (cost[~ok] == api.FAIL_COST).all(), label
    want, scale = np.full_like(viol, np.nan), np.full_like(viol, np.nan)
    for b in np.nonzero(ok)[0]:
        K = int(r.K[b])
        want[b], scale[b] = C.oracle_viol(variant, batch, 0 if shared else b, r.segs[b, :K], r.ctrl[b, :12 * K])
        err = np.abs(viol[b] - want[b])
        assert (err <= C.BAR * np.maximum(1.0, scale[b])).all(), (label, b, viol[b], want[b])
    cert = ok & (viol <= tol).all(axis=(1, 2))
    assert np.array_equal(cost, np.where(cert, r.a_cost, api.FAIL_COST)), label
    print("%s: B=%d certifiable=%d certified=%d max viol %.3e" % (label, len(ok), ok.sum(), cert.sum(),
                                                               np.nanmax(viol) if ok.any() else 0.0))
    return r, viol, cost, want, scale


# ---------------------------------------------------------------- 1: parity with the oracle
@pytest.mark.parametrize("variant", ("trp", "cub"))
def test_certify_config2_matches_oracle(planner, variant):
    from spectral_b200.scenarios import GOLDEN_W_CUB, GOLDEN_W_TRP, config2
    batch = config2()
    inputs, outs = solve(planner, variant, batch, GOLDEN_W_TRP if variant == "trp" else GOLDEN_W_CUB)
    r = assert_parity(planner, variant, batch, inputs, outs, "config2/" + variant)[0]
    assert r.ok().sum() > 256 and (~r.ok()).sum() > 0


@pytest.mark.parametrize("variant", ("trp", "cub"))
def test_certify_every_segment_count(planner, variant):
    """segment_ladder(K) for K = 1 .. 32: every solver class (k_qpa<8>, <10>, k_qpd<12>, <16>, k_qp<32, 2>)."""
    from spectral_b200.scenarios import GOLDEN_W_CUB, GOLDEN_W_TRP, segment_ladder
    w = GOLDEN_W_TRP if variant == "trp" else GOLDEN_W_CUB
    n_ok = 0
    for K in range(1, 33):
        batch = segment_ladder(K, 4)
        inputs, outs = solve(planner, variant, batch, w)
        r = assert_parity(planner, variant, batch, inputs, outs, "ladder/%s/K%d" % (variant, K))[0]
        assert (r.K == K).all()
        n_ok += int(r.ok().sum())
    assert n_ok >= 64


def test_certify_mixed_batches(planner):
    from spectral_b200.scenarios import WEIGHTS_FILE, mixed_batches
    for i, (variant, batch) in enumerate(mixed_batches(320)):
        inputs, outs = solve(planner, variant, batch, WEIGHTS_FILE)
        assert_parity(planner, variant, batch, inputs, outs, "mixed/%d/%s" % (i, variant))


def test_certify_weight_sweep_shared_inputs(planner):
    """spectral_solve_weights_device outputs (one scenario, B weight vectors) with inputs_stride 0, and the same scenario
    tiled B times with inputs_stride 1: identical bytes."""
    from spectral_b200.scenarios import load_fixture
    from spectral_b200.wire import ScenarioBatch
    scenario = ScenarioBatch.from_scenarios([load_fixture("c1")])
    W = np.random.default_rng(7).uniform(0.0, 50.0, (256, 10))
    inputs, outs = solve_weights(planner, "trp", scenario, W)
    r, viol, cost, _, _ = assert_parity(planner, "trp", scenario, inputs, outs, "weights/trp", shared=True)
    assert r.ok().sum() >= 16
    tiled = {n: t.expand(len(W), *t.shape[1:]).contiguous() for n, t in inputs.items() if n in NAMES}
    v2, c2 = certify(planner, "trp", scenario, tiled, outs, 1e-6)
    assert v2.tobytes() == viol.tobytes() and c2.tobytes() == cost.tobytes()


def test_certify_shared_kkt_config3(planner):
    from spectral_b200.scenarios import WEIGHTS_FILE, config3
    batch = config3(512, groups=8)
    inputs, outs = solve(planner, "trp", batch, WEIGHTS_FILE, shared_kkt=1)
    r = assert_parity(planner, "trp", batch, inputs, outs, "config3/shared_kkt")[0]
    assert r.ok().sum() > 128


def test_certify_non_finite_control_points_and_refusals_on_the_device(planner):
    """The NaN-keeping warp maximum the device runs (sp_warp_max_nonneg's bit-pattern reduction): a NaN or infinite control
    point makes exactly its axis' entries NaN and the cost FAIL_COST, at the first, a middle and the last segment; so do a
    failed status and a K outside [1, k_max] on a solved scenario.  Every other scenario keeps its bytes."""
    from spectral_b200.scenarios import GOLDEN_W_CUB, config2
    batch = config2()
    inputs, outs = solve(planner, "cub", batch, GOLDEN_W_CUB)
    base_viol, base_cost = certify(planner, "cub", batch, inputs, outs, 1.0)
    r = Host(outs)
    ok = np.nonzero(r.ok() & (r.K >= 3))[0]
    assert len(ok) >= 12
    ctrl = outs["ctrl"].clone()
    cases = {}
    for j, (ax, val) in enumerate([(0, np.nan), (1, np.nan), (0, np.inf), (1, -np.inf), (0, -np.nan), (1, np.inf)]):
        b = int(ok[j])
        K = int(r.K[b])
        k = (0, K // 2, K - 1)[j % 3]
        ctrl[b, 6 * K * ax + 6 * k + (j % 6)] = float(val)
        cases[b] = ax
    v, c = certify(planner, "cub", batch, inputs, dict(outs, ctrl=ctrl), 1.0)
    for b, ax in cases.items():
        assert np.isnan(v[b, ax]).all() and v[b, 1 - ax].tobytes() == base_viol[b, 1 - ax].tobytes(), (b, ax, v[b])
        assert c[b] == api.FAIL_COST
    rest = np.setdiff1d(np.arange(len(r.K)), list(cases))
    assert v[rest].tobytes() == base_viol[rest].tobytes() and c[rest].tobytes() == base_cost[rest].tobytes()
    assert np.isfinite(base_viol[ok]).all() and (base_cost[ok] < api.FAIL_COST).any()
    status, K = outs["status"].clone(), outs["K"].clone()
    refused = [int(b) for b in ok[6:12]]
    for b, (st, k) in zip(refused, [(api.FAIL_SOLVER, None), (api.FAIL_TOO_MANY, None), (None, 0), (None, -1), (None, 33),
                                    (api.FAIL_POINTS_CHECK, None)]):
        if st is not None:
            status[b] = st
        if k is not None:
            K[b] = k
    v, c = certify(planner, "cub", batch, inputs, dict(outs, status=status, K=K), 1.0)
    assert np.isnan(v[refused]).all() and (c[refused] == api.FAIL_COST).all()
    rest = np.setdiff1d(np.arange(len(r.K)), refused)
    assert v[rest].tobytes() == base_viol[rest].tobytes() and c[rest].tobytes() == base_cost[rest].tobytes()


# ---------------------------------------------------------------- 2: soundness against the interval pre-check
def test_certify_is_sound_against_the_precheck(planner):
    """Scenarios the pre-check proves infeasible (a position gap g > margin at a joint, or an initial state outside the first
    segment's rows) that OSQP nevertheless returns as solved: rows 5 of k-1, 0 of k and 18 of k cannot all hold within g/3
    for ANY x (g/2 for the initial state), so the certificate must report at least margin/3 and must not certify them at
    margin/4."""
    from spectral_b200.scenarios import GOLDEN_W_CUB, config2
    batch = config2()
    margin = api.default_options().precheck_margin
    _, pre = solve(planner, "cub", batch, GOLDEN_W_CUB, infeasibility_precheck=1)
    inputs, outs = solve(planner, "cub", batch, GOLDEN_W_CUB)
    rp, r = Host(pre), Host(outs)
    caught = (rp.status > api.SOLVED_INACCURATE) & (rp.iters == 0) & r.ok()
    print("precheck-infeasible scenarios returned as solved: %d (of which solved inaccurate: %d)" %
          (caught.sum(), (caught & (r.status == api.SOLVED_INACCURATE)).sum()))
    assert caught.sum() >= 10
    viol, cost = certify(planner, "cub", batch, inputs, outs, margin / 4)
    worst = viol[caught].max(axis=(1, 2))
    assert (worst >= margin / 3 * (1 - 1e-9)).all(), np.sort(worst)[:8]
    assert (cost[caught] == api.FAIL_COST).all()


# ---------------------------------------------------------------- 3: selection of the best feasible trajectories
def test_certified_cost_selects_the_best_feasible(planner):
    import torch
    from spectral_b200.scenarios import GOLDEN_W_CUB, config2
    batch = config2()
    inputs, outs = solve(planner, "cub", batch, GOLDEN_W_CUB)
    r, _, _, want, scale = assert_parity(planner, "cub", batch, inputs, outs, "selection", tol=1e-6)
    band = 2 * C.BAR * np.maximum(1.0, scale)
    for tol in (1e-6, 2e-6, 5e-6, 1e-5, 2e-5, 5e-5, 1e-4):
        if not (np.abs(want - tol) <= band).any():
            break
    assert not (np.abs(want - tol) <= band).any(), "every candidate tol has an oracle value inside its rounding band"
    ocert = r.ok() & (want <= tol).all(axis=(1, 2))
    viol_t, cost_t = planner.certify_device("cub", batch.n_knots, inputs, outs, tol)
    cost = cost_t.cpu().numpy()
    assert np.array_equal(cost != api.FAIL_COST, ocert), tol
    n_unc = int((r.ok() & ~ocert).sum())
    print("tol %.0e: solved %d, certified %d, solved but not certified %d" % (tol, r.ok().sum(), ocert.sum(), n_unc))
    assert ocert.sum() >= 16 and n_unc > 0
    idx = np.nonzero(ocert)[0]
    order = idx[np.lexsort((idx, r.a_cost[idx]))][:16]
    tc, ti = planner.topk_device(cost_t, 16)
    assert np.array_equal(ti.cpu().numpy(), order) and tc.cpu().numpy().tobytes() == r.a_cost[order].tobytes()
    oc = torch.empty(1, dtype=torch.float64, device="cuda")
    oi = torch.empty(1, dtype=torch.int64, device="cuda")
    planner.argmin_device(cost_t, 0, oc, oi)
    assert int(oi.item()) == order[0] and oc.item() == r.a_cost[order[0]]
    wins = planner.sweep_topk(dict(outs, a_cost=cost_t), 0, 16)
    assert [w["index"] for w in wins] == list(order)
    for w in wins:
        b = w["index"]
        K = int(r.K[b])
        assert w["cost"] == r.a_cost[b] and w["K"] == K and np.array_equal(w["ctrl"], r.ctrl[b, :12 * K])


# ---------------------------------------------------------------- 4: invalid arguments
def test_certify_invalid_arguments(planner):
    import torch
    from spectral_b200.scenarios import GOLDEN_W_CUB, config2
    batch = config2(8)
    inputs, outs = solve(planner, "cub", batch, GOLDEN_W_CUB)
    with pytest.raises(ValueError):
        planner.certify_device("cub", batch.n_knots, inputs, outs, -1.0)
    with pytest.raises(ValueError):
        planner.certify_device("cub", batch.n_knots, inputs, outs, [1e-6, 1e-6, np.nan, 1e-6])
    with pytest.raises(ValueError):
        planner.certify_device("cub", batch.n_knots, inputs, outs, [1e-6, 1e-6])
    with pytest.raises(ValueError):
        planner.certify_device("cub", batch.n_knots, inputs, outs, 1e-6, B=9)
    with pytest.raises(ValueError):
        planner.certify_device("cub", batch.n_knots, dict(inputs, init=inputs["init"][:4]), outs, 1e-6)
    with pytest.raises(ValueError):
        planner.certify_device("cub", batch.n_knots + 1, inputs, outs, 1e-6)   # ds_bounds rows of another N
    lib, h = planner._lib, planner._h
    dp = lambda t: ctypes.cast(ctypes.c_void_p(t.data_ptr()), api._dp)  # noqa: E731
    ip = lambda t: ctypes.cast(ctypes.c_void_p(t.data_ptr()), api._ip)  # noqa: E731
    inp = api.SpectralInputs()
    for n in ("ds_bounds", "dl_bounds", "init", "scalars"):
        setattr(inp, n, dp(inputs[n]))
    out = api.SpectralOutputs()
    out.K, out.status, out.segs, out.ctrl, out.a_cost = (ip(outs["K"]), ip(outs["status"]), outs["segs"].data_ptr(),
                                                         dp(outs["ctrl"]), dp(outs["a_cost"]))
    viol = torch.zeros(8, 2, 4, dtype=torch.float64, device="cuda")
    cost = torch.zeros(8, dtype=torch.float64, device="cuda")
    tol = np.full(4, 1e-6)
    N = batch.n_knots
    INVALID = 1

    def call(hh=h, variant=api.CUB, B=8, n=N, i=ctypes.byref(inp), s=1, o=ctypes.byref(out), t=api._d(tol),
             v=ctypes.c_void_p(viol.data_ptr()), c=ctypes.c_void_p(cost.data_ptr())):
        return lib.spectral_certify_device(hh, variant, B, n, i, s, o, t, v, c, None)

    before = planner.launch_count()
    assert call(hh=None) == INVALID
    assert call(variant=2) == INVALID
    assert call(i=None) == INVALID and call(o=None) == INVALID
    for f in ("ds_bounds", "dl_bounds", "init", "scalars"):
        i2 = api.SpectralInputs.from_buffer_copy(inp)
        setattr(i2, f, None)
        assert call(i=ctypes.byref(i2)) == INVALID, f
    for f in ("K", "status", "segs", "ctrl", "a_cost"):
        o2 = api.SpectralOutputs.from_buffer_copy(out)
        setattr(o2, f, None)
        assert call(o=ctypes.byref(o2)) == INVALID, f
    assert call(B=0) == INVALID and call(B=-3) == INVALID
    assert call(n=2) == INVALID and call(n=planner.n_max + 1) == INVALID
    assert call(s=2) == INVALID and call(s=-1) == INVALID
    assert call(t=None) == INVALID
    for bad in (-1e-9, np.nan, -np.inf):
        t2 = tol.copy()
        t2[3] = bad
        assert call(t=api._d(t2)) == INVALID, bad
    assert call(v=None, c=None) == INVALID
    assert b"certify" in lib.spectral_last_error(h)
    assert planner.launch_count() == before
    # a_cost is needed only for the cost output
    o2 = api.SpectralOutputs.from_buffer_copy(out)
    o2.a_cost = None
    assert call(o=ctypes.byref(o2), c=None) == 0
    assert call(v=None) == 0 and call() == 0
    assert planner.launch_count() == before + 3
    torch.cuda.synchronize()
