"""CPU tests of the feasibility certificate (certify.cuh, spectral_certify_device): its warp body, compiled for the host from
tests/warp_emu/certify_emu.cpp, against the rows of the QP the CPU oracle assembles (tests/certify_ref.py), on emulated
solves of every fixture, and on the scenarios it must refuse to certify."""
import ctypes
import mmap
import os
import subprocess

import numpy as np
import pytest

import certify_ref as C
import helpers as H
from spectral_b200 import api
from spectral_b200.scenarios import GOLDEN_W_CUB, GOLDEN_W_TRP

_lib = {}
K_MAX = 32


@pytest.fixture(scope="module", autouse=True)
def certify_emu_lib(tmp_path_factory):
    """libcertify_emu.so built from the current sources into a temporary directory (the g++ flags of libwarp_emu.so: no
    FMA contraction), so that an edit of certify.cuh or qp.cuh is always what runs and the source tree is never written."""
    out = str(tmp_path_factory.mktemp("certify_emu") / "libcertify_emu.so")
    src = os.path.join(H.ROOT, "tests", "warp_emu", "certify_emu.cpp")
    r = subprocess.run(["/usr/bin/g++", "-O1", "-g", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-x", "c++",
                        "-I", os.path.join(H.ROOT, "tests", "warp_emu"), "-o", out, src, "-lpthread"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    _lib["certify"] = ctypes.CDLL(out)
    yield
    _lib.clear()


def emu_certify(variant, batch, res, tol, inputs_stride=1, ds_bounds=None):
    """certify.cuh's warp body on the host for every scenario of `res`: (viol [B, 2, 4], cost [B])."""
    B = len(res.K)
    d = lambda a: np.ascontiguousarray(a, dtype=np.float64)  # noqa: E731
    keep = [d(batch.ds_bounds) if ds_bounds is None else ds_bounds, d(batch.dl_bounds), d(batch.init), d(batch.scalars)]
    tol = np.broadcast_to(np.asarray(tol, dtype=np.float64), (C.NF,)).copy()
    viol, cost = np.zeros((B, 2, C.NF)), np.zeros(B)
    K, status = np.ascontiguousarray(res.K, dtype=np.int32), np.ascontiguousarray(res.status, dtype=np.int32)
    segs, ctrl, a_cost = np.ascontiguousarray(res.segs), d(res.ctrl), d(res.a_cost)
    _lib["certify"].emu_certify(api.VARIANT_ID[variant], B, batch.n_knots, K_MAX, *[api._d(a) for a in keep], inputs_stride,
                                api._i(K), api._i(status), segs.ctypes.data_as(ctypes.c_void_p), api._d(ctrl), api._d(a_cost),
                                api._d(tol), api._d(viol), api._d(cost))
    return viol, cost


def weights(variant):
    return GOLDEN_W_TRP if variant == "trp" else GOLDEN_W_CUB


def copy_res(res, **changes):
    out = api.BatchResult(*[None if a is None else a.copy() for a in
                            (res.K, res.segs, res.ctrl, res.obj, res.a_cost, res.status, res.iters, res.flags, res.npts)])
    for k, v in changes.items():
        getattr(out, k)[...] = v
    return out


def accepted(res):
    """`res` with every solver failure relabelled SOLVED_INACCURATE (a_cost 1.0), as if its last iterate had been
    accepted: the certificate then measures the control points the solver stopped at."""
    out = copy_res(res)
    fail = out.status == api.FAIL_SOLVER
    out.status[fail] = api.SOLVED_INACCURATE
    out.a_cost[fail] = 1.0
    return out


@pytest.mark.parametrize("variant", H.VARIANTS)
def test_emu_certify_matches_oracle_on_every_fixture(variant):
    """Every fixture, solved in the emulator at the default settings and stopped early (max_iter = 25, no polish): the
    certificate equals the oracle's max(l - Ax, Ax - u, 0) per (axis, family) within the bar, its maximum is
    helpers.qp_objective_and_violation's, and the cost is a_cost exactly where the oracle certifies.  The early-stopped
    runs end as solver failures (NaN, FAIL_COST); their iterates are then certified as accepted ones."""
    tol = 1e-6
    n_checked = 0
    unconverged_families = np.zeros((2, C.NF), bool)
    for name in H.ALL_FIXTURES:
        batch = H.fixture_batch(name)
        for opts in (dict(), dict(max_iter=25, polish=0)):
            raw = H.emu_solve(variant, batch, weights(variant), **opts)
            viol, cost = emu_certify(variant, batch, raw, tol)
            if not raw.ok()[0]:
                assert np.isnan(viol[0]).all() and cost[0] == api.FAIL_COST, (name, opts)
            res = accepted(raw)
            K = int(res.K[0])
            if not res.ok()[0] or K > K_MAX:
                continue
            viol, cost = emu_certify(variant, batch, res, tol)
            got = C.check_scenario(variant, batch, 0, K, res.segs[0], res.ctrl[0], viol[0], (name, opts))
            _, v = H.qp_objective_and_violation(variant, batch, 0, weights(variant), res.segs[0, :K], res.ctrl[0, :12 * K])
            assert got.max() == v, (name, got, v)
            assert cost[0] == (res.a_cost[0] if (got <= tol).all() else api.FAIL_COST), (name, opts, viol[0])
            if opts:
                unconverged_families |= viol[0] > 0
            n_checked += 1
    assert n_checked >= 20
    # the early-stopped iterates are not feasible: the comparison is not one of zeros
    assert unconverged_families.any(axis=0).sum() >= 2, unconverged_families


def solved(variant="cub", name="c1", **opts):
    batch = H.fixture_batch(name)
    res = accepted(H.emu_solve(variant, batch, weights(variant), **opts))
    assert res.ok()[0]
    return batch, res


def test_emu_certify_refuses_what_it_cannot_certify():
    batch, res = solved()
    base, _ = emu_certify("cub", batch, res, 1.0)
    assert np.isfinite(base).all()
    for st in (api.FAIL_NO_CORRIDOR, api.FAIL_SOLVER, api.FAIL_POINTS_CHECK, api.FAIL_TOO_MANY):
        viol, cost = emu_certify("cub", batch, copy_res(res, status=st), 1.0)
        assert np.isnan(viol).all() and cost[0] == api.FAIL_COST, st
    for K in (0, -1, K_MAX + 1):
        viol, cost = emu_certify("cub", batch, copy_res(res, K=K), 1.0)
        assert np.isnan(viol).all() and cost[0] == api.FAIL_COST, K
    # a NaN or infinite control point: that axis' entries are NaN, the other axis is unchanged
    K = int(res.K[0])
    for ax, val in ((0, np.nan), (1, np.nan), (0, np.inf), (1, -np.inf)):
        bad = copy_res(res)
        bad.ctrl[0, 6 * K * ax + 6 * (K - 1) + 2] = val
        viol, cost = emu_certify("cub", batch, bad, 1.0)
        assert np.isnan(viol[0, ax]).all() and np.array_equal(viol[0, 1 - ax], base[0, 1 - ax]), (ax, val)
        assert cost[0] == api.FAIL_COST


def guarded(values, at_end):
    """A copy of `values` (float64) placed against an inaccessible page, after it (at_end) or before it: a read one element
    past that side of the array faults instead of returning a number."""
    libc = ctypes.CDLL(None, use_errno=True)
    page = mmap.PAGESIZE
    nbytes = values.nbytes
    assert nbytes <= page
    buf = mmap.mmap(-1, 3 * page)
    base = ctypes.addressof(ctypes.c_char.from_buffer(buf))
    libc.mprotect.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    assert libc.mprotect(base, page, 0) == 0 and libc.mprotect(base + 2 * page, page, 0) == 0
    off = 2 * page - nbytes if at_end else page
    arr = np.frombuffer(buf, dtype=np.float64, count=values.size, offset=off).reshape(values.shape)
    arr[...] = values
    return arr, buf


def test_emu_certify_checks_segment_ranges_before_reading():
    """Segments whose knot range leaves [0, N - 1] are refused (NaN, FAIL_COST) and ds_bounds is not read outside the
    scenario: the bounds sit against an inaccessible page on the side the bad range points to."""
    batch, res = solved()
    N, K = batch.n_knots, int(res.K[0])
    ds = np.ascontiguousarray(batch.ds_bounds, dtype=np.float64)
    cases = [("end_t", N, True), ("end_t", N + 1000, True), ("beg_t", -1, False), ("beg_t", -1000, False)]
    for field, val, at_end in cases:
        for k in (0, K - 1):
            bad = copy_res(res)
            bad.segs[field][0, k] = val
            arr, buf = guarded(ds, at_end)
            viol, cost = emu_certify("cub", batch, bad, 1.0, ds_bounds=arr)
            assert np.isnan(viol).all() and cost[0] == api.FAIL_COST, (field, val, k)
            del arr
            buf.close()
    bad = copy_res(res)   # beg_t > end_t
    bad.segs["beg_t"][0, K - 1] = bad.segs["end_t"][0, K - 1] + 1
    viol, cost = emu_certify("cub", batch, bad, 1.0)
    assert np.isnan(viol).all() and cost[0] == api.FAIL_COST
    # the in-range extremes are certifiable and read the bounds to the last knot of the guarded copy
    good = copy_res(res)
    good.segs["end_t"][0, K - 1] = N - 1
    arr, buf = guarded(ds, True)
    viol, _ = emu_certify("cub", batch, good, 1.0, ds_bounds=arr)
    assert np.isfinite(viol).all()
    C.check_scenario("cub", batch, 0, K, good.segs[0], good.ctrl[0], viol[0])
    del arr
    buf.close()


def test_emu_certify_tolerance_is_inclusive():
    batch, res = solved("trp", "c2", max_iter=25, polish=0)
    viol, _ = emu_certify("trp", batch, res, 0.0)
    tol = viol[0].max(axis=0)           # per family, over both axes
    assert (tol > 0).sum() >= 2
    _, cost = emu_certify("trp", batch, res, tol)
    assert cost[0] == res.a_cost[0]                          # viol == tol certifies
    for f in np.nonzero(tol > 0)[0]:
        t2 = tol.copy()
        t2[f] = np.nextafter(t2[f], 0.0)
        _, cost = emu_certify("trp", batch, res, t2)
        assert cost[0] == api.FAIL_COST, f


def test_emu_certify_shared_inputs_equal_tiled_inputs():
    """inputs_stride 0 (one scenario for every lane, the weight-sweep layout) gives the bytes of the same scenario tiled."""
    variant = "cub"
    batch = H.fixture_batch("c1")
    w = np.array([weights(variant), np.array(weights(variant)) * 0.5, np.array(weights(variant)) * 2.0])
    runs = [accepted(H.emu_solve(variant, batch, wi, max_iter=25, polish=0)) for wi in w]
    tiled = api.BatchResult(*[np.concatenate([getattr(r, n) for r in runs]) for n in
                              ("K", "segs", "ctrl", "obj", "a_cost", "status", "iters", "flags", "npts")])
    rep = lambda a: np.ascontiguousarray(np.repeat(a, 3, axis=0))  # noqa: E731
    from spectral_b200.wire import ScenarioBatch
    big = ScenarioBatch(batch.n_knots, batch.n_regions, batch.delta_t, *[rep(a) for a in batch.arrays()])
    a = emu_certify(variant, batch, tiled, 1e-6, inputs_stride=0)
    b = emu_certify(variant, big, tiled, 1e-6, inputs_stride=1)
    assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()
    assert np.isfinite(a[0]).all()
    for i in range(3):
        C.check_scenario(variant, batch, 0, int(tiled.K[i]), tiled.segs[i], tiled.ctrl[i], a[0][i])
