"""CPU tests of the trajectory evaluator (eval.cuh, spectral_eval_device): the point body, compiled for the host from
tests/warp_emu/eval_emu.cpp, against the NumPy reference of tests/eval_ref.py, and against the reference's own sampler
(the `samples` of an emulated solve)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import eval_ref as R
import helpers as H
from spectral_b200 import api
from spectral_b200.scenarios import WEIGHTS_FILE


_lib = {}


@pytest.fixture(scope="module", autouse=True)
def eval_emu_lib(tmp_path_factory):
    """libeval_emu.so built from the current sources into a temporary directory (the same g++ flags as libwarp_emu.so:
    no FMA contraction), so that an edit of eval.cuh is always what runs and the source tree is never written."""
    out = str(tmp_path_factory.mktemp("eval_emu") / "libeval_emu.so")
    src = os.path.join(H.ROOT, "tests", "warp_emu", "eval_emu.cpp")
    r = subprocess.run(["/usr/bin/g++", "-O1", "-g", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-x", "c++",
                        "-I", os.path.join(H.ROOT, "tests", "warp_emu"), "-o", out, src], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    _lib["eval"] = ctypes.CDLL(out)
    yield
    _lib.clear()


def emu_eval(K, status, segs, ctrl, k_max, times):
    """eval.cuh's point body on the host for every (scenario, time): (states [B, T, 6], jerk [B, T, 2], horizon [B])."""
    B = len(K)
    times = np.ascontiguousarray(times, dtype=np.float64)
    T = times.shape[-1]
    st, jk, hz = np.zeros((B, T, 6)), np.zeros((B, T, 2)), np.zeros(B)
    _lib["eval"].emu_eval(B, k_max, api._i(np.ascontiguousarray(K, dtype=np.int32)), api._i(np.ascontiguousarray(status, dtype=np.int32)),
                         np.ascontiguousarray(segs).ctypes.data_as(ctypes.c_void_p), api._d(np.ascontiguousarray(ctrl)), T,
                         api._d(times), 0 if times.ndim == 1 else 1, api._d(st), api._d(jk), api._d(hz))
    return st, jk, hz


def per_scenario_times(K, segs, k_max, n_random=16):
    rows = [R.probe_times(segs[b]["t"], min(int(K[b]), k_max), n_random, seed=b) for b in range(len(K))]
    T = max(len(r) for r in rows)
    return np.stack([np.pad(r, (0, T - len(r)), constant_values=0.5) for r in rows])


def test_emu_eval_matches_numpy_reference():
    k_max = 32
    K, status, segs, ctrl = R.synthetic(64, k_max, seed=1)
    times = per_scenario_times(K, segs, k_max)
    st, jk, hz = emu_eval(K, status, segs, ctrl, k_max, times)
    rst, rjk, rhz = R.ref_eval(K, status, segs, ctrl, k_max, times)
    R.assert_close(st, rst, "states")
    R.assert_close(jk, rjk, "jerk")
    assert np.array_equal(hz, rhz, equal_nan=True)
    # the failure rows are all NaN, the out-of-range and NaN times too, and the in-range probes are not
    assert np.isnan(st[[2, 5, 6, 7]]).all() and np.isnan(hz[[2, 5, 6, 7]]).all()
    ok = np.setdiff1d(np.arange(64), [2, 5, 6, 7])
    for b in ok:
        nj = min(int(K[b]), k_max)
        bad = np.isnan(times[b]) | (times[b] < -R.TIME_TOL) | (times[b] > hz[b] + R.TIME_TOL)
        assert bad.sum() == 3                          # -1e-6, H + 1e-6, NaN
        assert np.isnan(st[b][bad]).all() and not np.isnan(st[b][~bad]).any(), b
        assert st[b, 0, 0] == st[b, 0, 0] and np.array_equal(st[b, nj + 1], st[b, nj + 2])   # H + 5e-10 clamps to H
    # shared times: one row for every scenario, identical to per-scenario times with identical rows
    shared = times[0]
    a = emu_eval(K, status, segs, ctrl, k_max, shared)
    b = emu_eval(K, status, segs, ctrl, k_max, np.tile(shared, (len(K), 1)))
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def test_emu_eval_sliver_segments_are_skipped():
    """A joint next to a sliver belongs to the evaluable segment that ends there, never to the 8.9e-16 s piece."""
    k_max = 4
    K = np.array([4], np.int32)
    status = np.array([api.SOLVED], np.int32)
    segs = np.zeros((1, k_max), api.CUBE_DTYPE)
    segs[0]["t"] = [R.SLIVER, 0.45, R.SLIVER, 0.7]
    ctrl = np.random.default_rng(3).uniform(-5, 5, (1, 12 * k_max))
    times = np.array([0.0, R.SLIVER, 0.45, 0.45 + R.SLIVER, 1.15, 2.0])
    st, jk, hz = emu_eval(K, status, segs, ctrl, k_max, times)
    assert np.isfinite(st[0, :5]).all() and np.isnan(st[0, 5]).all()
    rst, rjk, _ = R.ref_eval(K, status, segs, ctrl, k_max, times)
    R.assert_close(st, rst)
    R.assert_close(jk, rjk)
    # tau = 0 is the start of segment 1 (u = 0), the joint 0.45 its end (u = 1)
    c = ctrl[0]
    assert abs(st[0, 0, 0] - 0.45 * c[6]) < 1e-12 and abs(st[0, 2, 0] - 0.45 * c[11]) < 1e-12


def reference_grid(K, segs_t, delta):
    """The times of the reference's sampler (finalize.cuh, solve_3d.cc:1351): T_k + (l / linter) t_k, l = 1..linter."""
    out, T0 = [0.0], 0.0
    for k in range(K):
        t = float(segs_t[k])
        linter = int(t / delta)
        out += [T0 + (l / linter) * t for l in range(1, linter + 1)]
        T0 += t
    return np.array(out)


@pytest.mark.parametrize("variant", H.VARIANTS)
def test_emu_eval_on_reference_grid_equals_samples(variant):
    """Evaluated at the reference sampler's times, the trajectory equals `samples` row for row (rows >= 1 are the same
    Bezier arithmetic at nearly the same u); row 0 is the initial state, met to the feasibility of the solve."""
    from spectral_b200.scenarios import GOLDEN_W_TRP
    fixtures = ("c1", "c2", "c4_2")
    cap = 200
    n_checked = n_verified = 0
    for name in fixtures:
        batch = H.fixture_batch(name)
        w = GOLDEN_W_TRP if variant == "trp" else WEIGHTS_FILE
        got = H.emu_solve(variant, batch, w, samples_cap=cap)
        if not got.ok()[0]:
            continue
        K, n = int(got.K[0]), int(got.npts[0])
        grid = reference_grid(K, got.segs[0]["t"], batch.delta_t)
        assert len(grid) == n, (name, len(grid), n)
        st, _, _ = emu_eval(got.K, got.status, got.segs, got.ctrl, 32, grid)
        assert H.maxdiff(st[0, 1:], got.samples[0, 1:n]) <= 1e-9, name
        if got.verified()[0]:
            rows = R.verified_row_bounds(variant, batch, 0, w, got.segs[0, :K], got.ctrl[0, :12 * K])
            init_tol, _ = R.state_tolerances(rows, got.segs[0]["t"], K)
            assert (np.abs(st[0, 0] - batch.init[0]) <= init_tol).all(), (name, st[0, 0] - batch.init[0], init_tol)
            n_verified += 1
        n_checked += 1
    assert n_checked >= 2 and n_verified >= 1
