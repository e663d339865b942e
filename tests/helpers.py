"""Shared test helpers: golden loading, the kernel-logic emulator binding, parity comparisons."""
import ctypes
import os

import numpy as np

from spectral_b200 import api
from spectral_b200.scenarios import load_fixture
from spectral_b200.wire import ScenarioBatch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# north_star tolerance for the floating-point part of the path (control points, costs)
RTOL, ATOL = 1e-5, 1e-6

ALL_FIXTURES = ("c1", "c2", "c3", "c4", "c4_2", "c5", "c6", "c7", "c7_7", "c7_10", "c_road_s1", "c_road_s1_2",
                "c_road_s1_3", "bounds")
VARIANTS = ("trp", "cub")

_npz = {}


def golden(name):
    if name not in _npz:
        _npz[name] = np.load(os.path.join(GOLDEN, name + ".npz"))
    return _npz[name]


def fixture_batch(name):
    return ScenarioBatch.from_scenarios([load_fixture(name)])


def close(a, b, rtol=RTOL, atol=ATOL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return bool(np.all(np.abs(a - b) <= atol + rtol * np.abs(b)))


def maxdiff(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b))) if a.size else 0.0


SEG_FIELDS = ("beg_t", "end_t", "t", "beg_l", "end_l", "upp_skew", "upp_bias", "down_skew", "down_bias",
              "l_upp_skew", "l_upp_bias", "l_down_skew", "l_down_bias", "merge", "split")


def segs_equal(a, b, K):
    """Bit-exact comparison of the first K cubes on every field the reference's Cube() initialises or the
    path writes.  (`t_dif` is never initialised by the reference -- cube_type.h:12-21 -- and `count` is
    bookkeeping of CollisionCheck's push loop; both are unused downstream.)"""
    a, b = np.asarray(a)[:K], np.asarray(b)[:K]
    for f in SEG_FIELDS:
        if a[f].tobytes() != b[f].tobytes():
            return False
    return True


def lu_to_qp_rows(lu, K):
    """[2, k_max, 21, 2] lane-major (l,u) rows -> the reference's row order (a7): per axis
    K x 18 segment rows, 3 initial-state rows, then 3 rows per joint.  Returns (l[42K], u[42K])."""
    out = []
    for axis in range(2):
        seg_rows = lu[axis, :K, :18].reshape(K * 18, 2)
        init_rows = lu[axis, 0, 18:21]
        joint_rows = lu[axis, 1:K, 18:21].reshape((K - 1) * 3, 2)
        out.append(np.concatenate([seg_rows, init_rows, joint_rows], axis=0))
    allrows = np.concatenate(out, axis=0)
    return allrows[:, 0].copy(), allrows[:, 1].copy()


_emu = None


def emu_lib():
    global _emu
    if _emu is None:
        _emu = ctypes.CDLL(os.path.join(ROOT, "tests", "warp_emu", "libwarp_emu.so"))
    return _emu


def emu_solve(variant, batch, weights, k_max=32, samples_cap=0, want_lu=False, **opts):
    """Run the kernels' device bodies on the host (32 lock-stepped threads per warp).  Slow: tiny batches only."""
    emu = emu_lib()
    B = batch.batch
    o = api.SpectralOptions()
    emu.emu_default_options(ctypes.byref(o))
    for k, v in opts.items():
        setattr(o, k, v)
    w = np.ascontiguousarray(np.asarray(weights, dtype=np.float64))
    arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in batch.arrays()]
    res = api.BatchResult(np.zeros(B, np.int32), np.zeros((B, k_max), api.CUBE_DTYPE), np.zeros((B, 12 * k_max)),
                          np.zeros(B), np.zeros(B), np.zeros(B, np.int32), np.zeros(B, np.int32),
                          np.zeros(B, np.int32), np.zeros(B, np.int32),
                          np.zeros((B, samples_cap, 6)) if samples_cap else None,
                          np.zeros((B, 2, k_max, 21, 2)) if want_lu else None)
    d, i = api._d, api._i
    emu.emu_solve_batch(api.VARIANT_ID[variant], B, batch.n_knots, batch.n_regions, ctypes.c_double(batch.delta_t),
                        *[d(a) for a in arrs], d(w), 0 if w.ndim == 1 else 1, k_max, ctypes.byref(o), i(res.K),
                        res.segs.ctypes.data_as(ctypes.c_void_p), d(res.ctrl), d(res.obj), d(res.a_cost),
                        i(res.status), i(res.iters), i(res.flags), i(res.npts), d(res.samples), samples_cap,
                        d(res.lu))
    return res


def emu_bounds(obstacles, n_obs, n_knots, r_cap, road=api.ROAD):
    """bounds.cuh's warp body on the host (tests/warp_emu): (s_bounds, l_bounds, n_lanes)."""
    emu = emu_lib()
    obstacles = np.ascontiguousarray(obstacles, dtype=np.float64)
    B, M = obstacles.shape[:2]
    n_obs = np.ascontiguousarray(n_obs, dtype=np.int32)
    sb = np.full((B, r_cap, n_knots, 2), np.nan)
    lb = np.full((B, r_cap, n_knots, 2), np.nan)
    nl = np.zeros(B, np.int32)
    emu.emu_bounds(B, n_knots, M, r_cap, api._d(obstacles), api._i(n_obs), api._d(np.array(road, dtype=np.float64)), api._d(sb), api._d(lb),
                   api._i(nl))
    return sb, lb, nl


def assert_bounds_equal_oracle(sb, lb, nl, obstacles, n_obs, n_knots, r_cap, road=api.ROAD):
    """(s_bounds, l_bounds, n_lanes) of the bounds kernel vs oracle/bounds_oracle.py (pinned to the reference's get_bounds), bit for bit;
    the padding lanes are empty lanes over the free road.  Lane-table overflows of the kernel's small fixed tables may only
    happen where the oracle's lane count exceeds r_cap."""
    import bounds_oracle as bo
    rd = dict(s_l_l=road[0], s_u_l=road[1], d_l_l=road[2], d_u_l=road[3])
    n_over = 0
    for b in range(len(nl)):
        obs = [((o[0], o[1], o[2]), o[3], o[4], o[5]) for o in obstacles[b, :n_obs[b]]]
        want = bo.get_bounds(obs, n_knots, rd)
        if len(want) > r_cap:
            assert nl[b] == -1, b
            assert np.all(lb[b, :, :, 0] == 1.0) and np.all(lb[b, :, :, 1] == -1.0), b
            n_over += 1
            continue
        assert nl[b] == len(want), (b, nl[b], len(want))
        for r, (s, (lo, hi)) in enumerate(want):
            assert np.array_equal(sb[b, r], s), (b, r)
            assert np.all(lb[b, r, :, 0] == lo) and np.all(lb[b, r, :, 1] == hi), (b, r)
        assert np.all(sb[b, len(want):, :, 0] == road[0]) and np.all(sb[b, len(want):, :, 1] == road[1]), b
        assert np.all(lb[b, len(want):, :, 0] == 1.0) and np.all(lb[b, len(want):, :, 1] == -1.0), b
    return n_over


def decided_classes(ref, ref0, max_iter=5000, early_frac=0.6):
    """Which scenarios have a solved/failed class that the reference itself pins.

    The reference's outcome on a slowly converging QP is the state of OSQP's ADMM iterate at max_iter = 5000
    (trp_wrapper.cpp:191) and OSQP 0.5.0 picks its rho-adaptation schedule from wall-clock time (SURVEY.md
    7.3-1), so on such problems the class is not reproducible by the reference itself.  A class counts as
    decided when the reference-settings oracle (ref0) and the converged oracle (ref, tight tolerances, 50 000
    iterations) agree AND, for solved ones, ref0 stopped well before max_iter:
      decided solved  = ref0 solved with iters <= early_frac * max_iter, and the converged oracle solved it too
      decided failed  = ref0 failed and the converged oracle failed too (certified infeasible / never converges)
    Corridor-stage failures (no corridor, too many segments) are always decided (integer logic, bit-exact)."""
    st0, st1 = ref0["status"], ref["status"]
    corridor_fail = np.isin(st1, (2, 5))
    solved = (st0 <= 1) & (st1 <= 1) & (ref0["iters"] <= early_frac * max_iter)
    failed = (st0 > 1) & (st1 > 1)
    return solved | failed | corridor_fail


def qp_objective_and_violation(variant, batch, b, weights, segs, x):
    """Objective 0.5 x'Px + q'x and max bound violation of x for the QP the reference assembles for scenario b."""
    import pyoracle as po
    import scipy.sparse as sp
    from spectral_b200.wire import Scenario
    w = np.asarray(weights, dtype=np.float64)
    w = w if w.ndim == 1 else w[b]
    sc = Scenario(batch.n_knots, batch.delta_t, batch.init[b, :3], batch.init[b, 3:], batch.scalars[b], batch.s_bounds[b],
                  batch.l_bounds[b], batch.ds_bounds[b], batch.dl_bounds[b], batch.s_ref[b], batch.l_ref[b])
    qp = po.formulate(variant, sc, w, segs)
    n, m = qp["n"], qp["m"]
    Pu = sp.csc_matrix((qp["P_x"], qp["P_i"], qp["P_p"]), shape=(n, n))
    P = Pu + sp.triu(Pu, 1).T
    A = sp.csc_matrix((qp["A_x"], qp["A_i"], qp["A_p"]), shape=(m, n))
    Ax = A @ x
    viol = float(np.maximum(np.maximum(qp["l"] - Ax, Ax - qp["u"]), 0.0).max())
    return float(0.5 * x @ (P @ x) + qp["q"] @ x), viol


def highs_solution(variant, batch, b, weights, segs):
    """Optimum of the QP the reference assembles for scenario b according to HiGHS (scipy's vendored build);
    None when HiGHS is unavailable or does not report optimality.  Accurate to ~1e-4 on these problems."""
    try:
        import pyoracle as po
        import scipy.sparse as sp
        from scipy.optimize._highspy import _core as hp
    except Exception:
        return None
    from spectral_b200.wire import Scenario
    w = np.asarray(weights, dtype=np.float64)
    w = w if w.ndim == 1 else w[b]
    sc = Scenario(batch.n_knots, batch.delta_t, batch.init[b, :3], batch.init[b, 3:], batch.scalars[b], batch.s_bounds[b],
                  batch.l_bounds[b], batch.ds_bounds[b], batch.dl_bounds[b], batch.s_ref[b], batch.l_ref[b])
    qp = po.formulate(variant, sc, w, segs)
    n, m = qp["n"], qp["m"]
    Pl = sp.csc_matrix(sp.csc_matrix((qp["P_x"], qp["P_i"], qp["P_p"]), shape=(n, n)).T)
    h = hp._Highs()
    h.setOptionValue("output_flag", False)
    model = hp.HighsModel()
    lp = model.lp_
    lp.num_col_, lp.num_row_ = n, m
    lp.col_cost_ = qp["q"]
    lp.col_lower_ = np.full(n, -hp.kHighsInf)
    lp.col_upper_ = np.full(n, hp.kHighsInf)
    lp.row_lower_, lp.row_upper_ = qp["l"], qp["u"]
    lp.a_matrix_.format_ = hp.MatrixFormat.kColwise
    lp.a_matrix_.start_, lp.a_matrix_.index_, lp.a_matrix_.value_ = qp["A_p"], qp["A_i"], qp["A_x"]
    model.hessian_.dim_ = n
    model.hessian_.format_ = hp.HessianFormat.kTriangular
    model.hessian_.start_, model.hessian_.index_, model.hessian_.value_ = Pl.indptr, Pl.indices, Pl.data
    h.passModel(model)
    h.run()
    if "kOptimal" not in str(h.getModelStatus()):
        return None
    return np.array(h.getSolution().col_value)


PARITY_LOG = []  # one dict per assert_batch_parity call (tests/conftest.py prints them as JSON lines at session end)


def _emit_stats(stats):
    import json
    PARITY_LOG.append(stats)
    line = json.dumps({"parity_stats": stats})
    print(line)
    try:
        out = os.path.join(ROOT, "gpurun_out")
        if os.path.isdir(out):
            with open(os.path.join(out, "parity_stats.jsonl"), "a") as f:
                f.write(line + "\n")
    except OSError:
        pass


# ADMM-iterate parity (product with polish = 0 vs the reference-settings oracle): both run the same deterministic
# OSQP iteration (fixed adaptive-rho interval) in different floating-point orders (dense inverse vs LDL'), and the
# iteration contracts slowly on these QPs, so the two iterates at the SAME iteration count agree to the termination
# tolerance of the iteration (eps 1e-5, scaled), not to round-off: the bound is on what eps leaves open.
ITER_ATOL, ITER_RTOL = 5e-4, 5e-4


def assert_batch_parity(got, ref, label="", need_verified_frac=0.0, ref0=None, max_status_mismatch=0,
                        max_undecided_mismatch_frac=0.01, batch=None, variant=None, weights=None, got0=None,
                        min_iters_equal_frac=0.97, max_exception_frac=0.005):
    """got: api.BatchResult (GPU or emulator); ref: pyoracle.solve_batch(mode=1) dict (converged oracle);
    ref0: pyoracle.solve_batch(mode=0) dict (the reference's own OSQP settings); got0: the product run with
    polish = 0 (the reference's setting, solve_3d.cc:1243), i.e. its raw ADMM iterate.
    * integer / struct outputs bit-exact;
    * solved / failed class identical wherever the reference pins it (decided_classes); the undecided mismatches are
      counted and bounded (1 % of the batch);
    * iteration count equal to the reference-settings oracle's on the decided-solved set (the kernel runs OSQP's
      iteration: same check / adaptive-rho schedule), for at least min_iters_equal_frac of them, the rest within one
      check interval or one rho-adaptation cascade;
    * every scenario BOTH sides solve gets a numerical comparison: control points within RTOL / ATOL of the converged
      oracle where both hold a KKT-verified optimum, else (got0 given) within ITER_ATOL / ITER_RTOL of the
      reference-settings oracle's iterate; a batch with solved scenarios and nothing compared fails."""
    B = len(got.K)
    stats = {"label": label, "B": int(B)}
    assert np.array_equal(got.K, ref["K"]), "%s: K differs at %s" % (label, np.nonzero(got.K != ref["K"])[0][:8])
    for b in range(B):
        K = int(got.K[b])
        if ref["status"][b] in (2, 5):
            continue
        assert segs_equal(got.segs[b], ref["segs"][b], K), "%s: segs differ at scenario %d" % (label, b)
    corridor_fail = np.isin(ref["status"], (2, 5))
    assert np.array_equal(got.status[corridor_fail], ref["status"][corridor_fail]), label
    have_ref0 = ref0 is not None
    ref0 = ref0 if have_ref0 else ref
    st0 = ref0["status"]
    ok_ref = st0 <= 1
    decided = decided_classes(ref, ref0)
    mism = got.ok() != ok_ref
    # "solved inaccurate" AT the iteration cap is a threshold test (10 x eps) on a non-converged iterate: whether the last
    # iterate of an infeasible or very slowly converging problem squeezes under it depends on rounding-level details of
    # the iterate path -- the reference-settings oracle itself accepts 160 provably infeasible config-2 scenarios this way
    # (DESIGN.md 6.1).  Such outcomes are borderline on either side and count as undecided (about 1 in 1000 scenarios).
    cap = 5000
    borderline = ((got.status == 1) & (got.iters >= cap)) | ((st0 == 1) & (ref0["iters"] >= cap))
    decided = decided & ~borderline
    hard = mism & decided
    soft = mism & ~decided
    stats.update(decided=int(decided.sum()), class_mismatch_decided=int(hard.sum()), class_mismatch_undecided=int(soft.sum()),
                 solved_got=int(got.ok().sum()), solved_ref0=int(ok_ref.sum()))
    assert hard.sum() <= max_status_mismatch, "%s: solved/failed class differs at %d decided scenarios %s (got %s, ref %s)" % (
        label, hard.sum(), np.nonzero(hard)[0][:8], got.status[hard][:8], st0[hard][:8])
    assert soft.sum() <= max(1, int(np.ceil(max_undecided_mismatch_frac * B))), "%s: %d of %d undecided classes differ" % (
        label, soft.sum(), (~decided).sum())

    # ---- iteration-count parity with the reference-settings oracle (decided-solved scenarios)
    if have_ref0:
        ds = decided & ok_ref & got.ok() & ~corridor_fail
        if ds.any():
            di = np.abs(got.iters[ds].astype(np.int64) - ref0["iters"][ds].astype(np.int64))
            eq = float((di == 0).mean())
            stats.update(iters_compared=int(ds.sum()), iters_equal_frac=eq, iters_maxdiff=int(di.max()))
            # (count-based so that a tiny batch may hold one borderline scenario: a residual within round-off of eps at a check)
            assert (di != 0).sum() <= max(1, int(np.floor((1.0 - min_iters_equal_frac) * ds.sum()))), \
                "%s: iteration count equals the reference-settings oracle's on only %.3f of %d scenarios" % (label, eq, ds.sum())

    # ---- numerical comparison of every scenario both sides solve
    both = got.verified() & (ref["status"] <= 1) & (ref["polish"] == 2)
    solved0 = (got.status == 0) & (ref["status"] <= 1)
    if solved0.any():
        frac = (solved0 & got.verified()).sum() / solved0.sum()
        stats["verified_frac_of_solved"] = float(frac)
        assert frac >= need_verified_frac, "%s: only %.3f of the SOLVED scenarios carry a KKT-verified optimum" % (label, frac)
    exceptions, oracle_side = [], []
    max_rel = 0.0
    for b in np.nonzero(both)[0]:
        K = int(got.K[b])
        assert got.npts[b] == ref["npts"][b]
        d = np.abs(got.ctrl[b, :12 * K] - ref["ctrl"][b, :12 * K]) / (ATOL + RTOL * np.abs(ref["ctrl"][b, :12 * K]))
        if close(got.ctrl[b, :12 * K], ref["ctrl"][b, :12 * K]):
            max_rel = max(max_rel, float(d.max()))
            # (north-star tolerance 1e-5 relative on the cost; on the fixture weights the agreement is ~1e-6, with
            # near-zero random weights up to 3e-6)
            # ... or lower than the oracle's (the product's point is then the better one of two points that agree to
            # tolerance; seen with near-zero weights, where P is almost singular along some directions)
            assert close(got.obj[b], ref["obj"][b], rtol=1e-5, atol=1e-6) or \
                (got.obj[b] <= ref["obj"][b] and close(got.obj[b], ref["obj"][b], rtol=2e-5)), (label, b, got.obj[b], ref["obj"][b])
            # (the cost is quadratic in the control points: 1e-5 on them moves it by up to 2e-5 relative)
            assert close(got.a_cost[b], ref["a_cost"][b], rtol=2e-5), (label, b, got.a_cost[b], ref["a_cost"][b])
            continue
        # The control points differ beyond tolerance.  On these QPs (cond(P) up to 1e13, near-degenerate active
        # sets) two points can both satisfy a solver's KKT tolerances, agree in objective to 1e-7 relative and
        # still sit 1e-3 .. 1e-2 apart along the flat directions of P -- the converged oracle and HiGHS disagree
        # with each other at that level too (DESIGN.md, "parity").  Such a scenario counts as an exception; it
        # is accepted only if the product's point is feasible to 1e-9 for the reference-assembled QP and as
        # optimal as the oracle's to 1e-6 relative in the objective, and exceptions must stay rare.
        assert batch is not None and variant is not None and weights is not None, \
            "%s: ctrl of scenario %d off by %.3e" % (label, b, maxdiff(got.ctrl[b, :12 * K], ref["ctrl"][b, :12 * K]))
        obj_g, viol_g = qp_objective_and_violation(variant, batch, b, weights, ref["segs"][b, :K], got.ctrl[b, :12 * K])
        obj_r, _ = qp_objective_and_violation(variant, batch, b, weights, ref["segs"][b, :K], ref["ctrl"][b, :12 * K])
        assert viol_g <= 1e-9 and obj_g <= obj_r + 1e-6 * abs(obj_r), \
            "%s: ctrl of scenario %d off by %.3e and worse than the oracle (obj %.9f vs %.9f, violation %.2e)" % (
                label, b, maxdiff(got.ctrl[b, :12 * K], ref["ctrl"][b, :12 * K]), obj_g, obj_r, viol_g)
        # third opinion: HiGHS on the same reference-assembled QP.  When the product's point is at least as close
        # to the independent solver as the oracle's, the disagreement is charged to the oracle, not the product.
        xh = highs_solution(variant, batch, b, weights, ref["segs"][b, :K])
        if xh is not None and maxdiff(got.ctrl[b, :12 * K], xh) <= maxdiff(ref["ctrl"][b, :12 * K], xh):
            oracle_side.append(int(b))
            continue
        exceptions.append(int(b))
    stats.update(compared_verified=int(both.sum()), verified_max_err_in_tol_units=max_rel, exceptions=len(exceptions),
                 charged_to_oracle=len(oracle_side))
    assert len(exceptions) <= max(1, int(np.ceil(max_exception_frac * both.sum()))), "%s: %d of %d verified scenarios differ in the control points: %s" % (
        label, len(exceptions), both.sum(), exceptions[:8])

    # ---- scenarios both sides solve but without a KKT proof on one side: the raw ADMM iterates must agree
    compared_iter = 0
    compared_any = both.copy()
    if got0 is not None and have_ref0:
        assert np.array_equal(got0.K, got.K) and np.array_equal(got0.iters, got.iters), "%s: polish changed the iteration" % label
        same = got0.ok() & ok_ref & ~corridor_fail & (got0.iters == ref0["iters"]) & (ref0["iters"] < cap)
        worst = 0.0
        bad = []
        for b in np.nonzero(same)[0]:
            K = int(got.K[b])
            x0, x1 = got0.ctrl[b, :12 * K], ref0["ctrl"][b, :12 * K]
            e = float(np.max(np.abs(x0 - x1) / (ITER_ATOL + ITER_RTOL * np.abs(x1))))
            worst = max(worst, e)
            if e > 1.0:
                bad.append(int(b))
        compared_iter = int(same.sum())
        compared_any |= same
        stats.update(compared_iterate=compared_iter, iterate_max_err_in_tol_units=worst, iterate_outliers=len(bad))
        assert len(bad) <= max(1, int(0.01 * compared_iter)), "%s: ADMM iterate differs from the reference-settings oracle's at %s" % (label, bad[:8])
    both_solved = got.ok() & (ref["status"] <= 1) & ok_ref
    stats["both_solved"] = int(both_solved.sum())
    stats["compared_any"] = int(compared_any.sum())  # distinct scenarios compared numerically, by optimum, by iterate or both
    if both_solved.any():
        assert both.sum() + compared_iter > 0, "%s: %d scenarios solved on both sides and none compared numerically" % (label, both_solved.sum())
    fail = ~got.ok()
    assert np.all(got.a_cost[fail] == api.FAIL_COST), label
    _emit_stats(stats)
    return both


def oracle_pair(variant, batch, weights, nthreads=0):
    """(converged oracle, reference-settings oracle) for one batch."""
    import pyoracle as po
    return (po.solve_batch(variant, batch, weights, mode=1, nthreads=nthreads),
            po.solve_batch(variant, batch, weights, mode=0, nthreads=nthreads))
