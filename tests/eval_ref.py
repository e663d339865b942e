"""NumPy reference of spectral_eval_device (include/spectral.h) and the synthetic trajectories its tests use.

The reference converts each Bezier segment to monomial form in u with numpy.polynomial and differentiates that, an
independent formula from the Bernstein-difference sums of eval.cuh."""
from math import comb

import numpy as np
from numpy.polynomial import Polynomial

from spectral_b200 import api

MIN_T = 1e-9      # segments this short are never evaluated
TIME_TOL = 1e-9   # times in [-TIME_TOL, H + TIME_TOL] are valid
SLIVER = 8.9e-16  # CorridorSplit's 7.000000000000001 - 7 sliver
DURATIONS = tuple(round(0.1 * i, 1) for i in range(1, 11)) + (0.45, 0.7 / 3)


def bezier_poly(c, t):
    """s(u) = t sum_i c_i C(5, i) u^i (1 - u)^(5 - i) as a Polynomial in u."""
    u, v = Polynomial([0.0, 1.0]), Polynomial([1.0, -1.0])
    p = Polynomial([0.0])
    for i in range(6):
        p = p + float(c[i]) * comb(5, i) * u ** i * v ** (5 - i)
    return t * p


def horizon(segs_t, K):
    H = 0.0
    for k in range(K):
        H += float(segs_t[k])
    return H


def ref_eval_one(K, status, segs_t, ctrl, k_max, times):
    """(states [T, 6], jerk [T, 2], H) of one scenario at `times`, per the contract of spectral_eval_device."""
    T = len(times)
    st, jk = np.full((T, 6), np.nan), np.full((T, 2), np.nan)
    if status not in (api.SOLVED, api.SOLVED_INACCURATE) or not 1 <= K <= k_max:
        return st, jk, np.nan
    H = horizon(segs_t, K)
    starts, acc = [], 0.0
    for k in range(K):
        starts.append(acc)
        acc += float(segs_t[k])
    usable = [k for k in range(K) if segs_t[k] > MIN_T]
    if not usable:
        return st, jk, H
    polys = {}
    for j, tau in enumerate(times):
        if not (-TIME_TOL <= tau <= H + TIME_TOL):
            continue
        tc = min(max(tau, 0.0), H)
        k = next((k for k in usable if tc <= starts[k] + float(segs_t[k])), usable[-1])
        t = float(segs_t[k])
        u = min(max((tc - starts[k]) / t, 0.0), 1.0)
        if k not in polys:
            polys[k] = [bezier_poly(ctrl[6 * k:6 * k + 6], t), bezier_poly(ctrl[6 * K + 6 * k:6 * K + 6 * k + 6], t)]
        for ax, p in enumerate(polys[k]):
            # d/dtau = (1/t) d/du on the monomial form: s = p, ds = p'/t, dds = p''/t^2, ddds = p'''/t^3
            st[j, 3 * ax:3 * ax + 3] = [p(u), p.deriv(1)(u) / t, p.deriv(2)(u) / t ** 2]
            jk[j, ax] = p.deriv(3)(u) / t ** 3
    return st, jk, H


def ref_eval(K, status, segs, ctrl, k_max, times):
    """All scenarios; times [T] (shared) or [B, T]."""
    B = len(K)
    times = np.asarray(times, dtype=np.float64)
    out = [ref_eval_one(int(K[b]), int(status[b]), segs[b]["t"], ctrl[b], k_max, times if times.ndim == 1 else times[b])
           for b in range(B)]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out]), np.array([o[2] for o in out])


def synthetic(B, k_max=32, seed=0):
    """Random trajectories: K in [1, k_max], durations from DURATIONS (non-multiples of 0.1 included), slivers of 8.9e-16
    at the start, middle and end of some scenarios, random control points; a few failed / K = 0 / K > k_max scenarios."""
    rng = np.random.default_rng(seed)
    K = rng.integers(1, k_max + 1, B).astype(np.int32)
    segs = np.zeros((B, k_max), api.CUBE_DTYPE)
    ctrl = np.zeros((B, 12 * k_max))
    status = np.where(rng.random(B) < 0.3, api.SOLVED_INACCURATE, api.SOLVED).astype(np.int32)
    for b in range(B):
        t = rng.choice(DURATIONS, K[b])
        if K[b] >= 3 and b % 4 == 1:
            t[[0, K[b] // 2, K[b] - 1]] = SLIVER
        segs[b, :K[b]]["t"] = t
        segs[b, K[b]:]["t"] = np.nan  # never read: a read would show up as a NaN horizon
        ctrl[b, :12 * K[b]] = rng.uniform(-5.0, 5.0, 12 * K[b])
        ctrl[b, 12 * K[b]:] = np.nan
    if B >= 8:
        status[2] = api.FAIL_SOLVER
        status[5] = api.FAIL_NO_CORRIDOR
        K[6] = 0
        K[7] = k_max + 1
    return K, status, segs, ctrl


def probe_times(segs_t, K, n_random=16, seed=0):
    """0, every joint, H, H +- 5e-10, -5e-10, out of range by 1e-6, NaN and random times in [0, H]."""
    H = horizon(segs_t, K) if K > 0 else 1.0
    joints, acc = [], 0.0
    for k in range(max(K, 0)):
        acc += float(segs_t[k])
        joints.append(acc)
    if not np.isfinite(H):  # K beyond the scenario's segments (an invalid-K probe): any times do
        H, joints = 1.0, [0.5] * len(joints)
    rng = np.random.default_rng(seed)
    return np.array([0.0] + joints + [H, H + 5e-10, H - 5e-10, -5e-10, -1e-6, H + 1e-6, np.nan] +
                    list(rng.uniform(0.0, H, n_random)))


def ruiz_row_scaling(P, A, q, iters=4, lo=1e-4, hi=1e4):
    """Row factors E of OSQP's Ruiz equilibration (scaling.c: `iters` rounds on the KKT matrix [P A'; A 0] with the
    cost normalisation c between rounds), the scaling the solver's termination and polish tests are expressed in."""
    P, A, q = P.toarray(), A.toarray(), q.copy()
    E = np.ones(A.shape[0])

    def limit(v):
        v = np.where(v < lo, 1.0, v)
        return np.minimum(v, hi)

    for _ in range(iters):
        d = 1.0 / np.sqrt(limit(np.maximum(np.abs(P).max(0), np.abs(A).max(0))))
        e = 1.0 / np.sqrt(limit(np.abs(A).max(1)))
        P, A, q = d[:, None] * P * d[None, :], e[:, None] * A * d[None, :], d * q
        E *= e
        c = max(float(np.abs(P).max(0).mean()), float(limit(np.array([np.abs(q).max()]))[0]))
        c = 1.0 / float(limit(np.array([c]))[0])
        P, q = P * c, q * c
    return E


def verified_row_bounds(variant, batch, b, weights, segs, x):
    """Bound on |A x - clip(A x)| per constraint row, in the row's own units, that a KKT-verified polish guarantees:
    qp.cuh accepts the polished point only with prip <= 10 tol_p, i.e. E_r viol_r <= 1e-8 (1 + max_r E_r |A x|_r) in the
    Ruiz-scaled rows, so viol_r <= 1e-8 (1 + max_r E_r |A x|_r) / E_r.  The E_r are recomputed here from the QP the
    reference assembles (not read from the solver), hence the factor 2.  Row order: per axis (s, then l) K x 18 segment
    rows, the 3 initial-state rows, then 3 rows per joint."""
    import scipy.sparse as sp
    import pyoracle as po
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
    E = ruiz_row_scaling(P, A, qp["q"])
    nax = float(np.max(E * np.abs(A @ x)))
    return 2.0 * 1e-8 * (1.0 + nax) / E


def state_tolerances(row_bound, segs_t, K):
    """Row bounds -> allowed |init - state(0)| [6] and |left - right limit| [K-1, 6] in state units.  The rows (qp.cuh
    apply_A, the reference's FormulateProblem):
      initial state  row 18 = t_0 c_0 = s(0);  row 19 = 5 (c_1 - c_0) = ds(0);  row 20 = 20 D2c_0 = t_0 dds(0)
      joint k|k+1    row 18 = t_{k+1} c_{k+1,0} - t_k c_{k,5}                   = the s jump
                     row 19 = (c_{k,5} - c_{k,4}) - (c_{k+1,1} - c_{k+1,0})     = the ds jump / 5
                     row 20 = t_{k+1} D2c_{k,3} - t_k D2c_{k+1,0}              = t_k t_{k+1} (the dds jump) / 20
    so a row bound (e18, e19, e20) allows (e18, e19, e20 / t_0) at tau = 0 and (e18, 5 e19, 20 e20 / (t_k t_{k+1})) at a
    joint, per axis."""
    t = np.asarray(segs_t[:K], dtype=np.float64)
    init, joints = np.zeros(6), np.zeros((max(K - 1, 0), 6))
    for ax in range(2):
        base = 21 * K * ax + 18 * K
        e = row_bound[base:base + 3]
        init[3 * ax:3 * ax + 3] = [e[0], e[1], e[2] / t[0]]
        for k in range(K - 1):
            e = row_bound[base + 3 + 3 * k:base + 6 + 3 * k]
            joints[k, 3 * ax:3 * ax + 3] = [e[0], 5.0 * e[1], 20.0 * e[2] / (t[k] * t[k + 1])]
    return init, joints


def assert_close(got, want, label=""):
    """got == want to 1e-10 (1 + |want|), NaN exactly where want is NaN."""
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (label, np.argwhere(np.isnan(got) != np.isnan(want))[:5])
    m = ~np.isnan(want)
    err = np.abs(got[m] - want[m]) / (1.0 + np.abs(want[m]))
    assert err.size == 0 or err.max() <= 1e-10, (label, float(err.max()))
