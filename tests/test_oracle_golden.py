"""CPU tests (`-m "not gpu"`): the oracle is pinned before it is trusted.

The CPU restatement (oracle/liboracle.so) is checked against
  * tests/golden/ref_segments.npz  new_corridor produced by the reference's OWN sources recompiled (a2-a4),
  * tests/golden/shipped_qp.npz    (P, q, A, l, u) captured from the reference's SHIPPED libtrp.so/libcub.so (a5-a8),
  * tests/golden/converged.npz     the converged optimum (HiGHS cross-checked when it was generated),
  * tests/golden/shipped_sampling.npz  trajectory file + return value the SHIPPED binary writes for given
                                   control points (a9 sampling, a10 cost, %.3f writer),
  * tests/golden/s1_{slt,cub}_3d_31.txt  the reference's shipped known-answer outputs (SURVEY.md D.2),
  * tests/golden/std_sort.npz      the order libstdc++'s std::sort gives equal keys (CollisionCheck's sort),
and, where oracle/_ref was built (container with /root/reference), against the recompiled reference itself.
Nothing here reads /root/reference at run time.
"""
import os

import numpy as np
import pytest

import helpers as H
import pyoracle as po
from spectral_b200.scenarios import (FEASIBLE, GOLDEN_W_CUB, GOLDEN_W_TRP, WEIGHTS_FILE, config2, load_fixture,
                                     mixed_batches, perturbed_obstacles)
from spectral_b200.wire import read_trajectory_text


def _oracle_one(variant, name, weights, mode):
    return po.solve_batch(variant, H.fixture_batch(name), weights, mode=mode, nthreads=1)


@pytest.mark.parametrize("variant", H.VARIANTS)
@pytest.mark.parametrize("name", H.ALL_FIXTURES)
def test_oracle_segments_match_reference_sources(name, variant):
    """a2-a4 bit-exact: every Cube field of new_corridor vs the recompiled reference's output."""
    r = _oracle_one(variant, name, WEIGHTS_FILE, 0)
    gs = H.golden("ref_segments")["%s/%s/segs" % (name, variant)].view(po.CUBE_DTYPE)
    assert r["K"][0] == len(gs)
    assert H.segs_equal(r["segs"][0], gs, len(gs))
    # success / failure class of the reference run (its own OSQP settings)
    ref_status = int(H.golden("ref_segments")["%s/%s/status" % (name, variant)])
    assert (r["status"][0] <= 1) == (ref_status <= 1)


@pytest.mark.parametrize("variant", H.VARIANTS)
@pytest.mark.parametrize("name", H.ALL_FIXTURES)
def test_oracle_qp_matches_shipped_binary(name, variant):
    """a5-a8: l, u, A bit-exact vs the QP the SHIPPED binaries hand to OSQP; P, q within the Eigen/libm
    evaluation-order noise documented in SURVEY.md D.6."""
    qp = H.golden("shipped_qp")
    key = "%s/%s/" % (name, variant)
    gs = H.golden("ref_segments")[key + "segs"].view(po.CUBE_DTYPE)
    got = po.formulate(variant, load_fixture(name), WEIGHTS_FILE, gs)
    assert got["n"] == 12 * len(gs) and got["m"] == 42 * len(gs)
    assert np.array_equal(got["l"], qp[key + "l"])
    assert np.array_equal(got["u"], qp[key + "u"])
    assert np.array_equal(got["A_p"], qp[key + "A_p"]) and np.array_equal(got["A_i"], qp[key + "A_i"])
    assert np.array_equal(got["A_x"], qp[key + "A_x"])
    assert np.array_equal(got["P_p"], qp[key + "P_p"]) and np.array_equal(got["P_i"], qp[key + "P_i"])
    assert np.allclose(got["P_x"], qp[key + "P_x"], rtol=1e-9, atol=0.0)
    if not name.startswith("c7"):  # c7*: the reference reads heap garbage past ref[N] (SURVEY.md E-10)
        assert np.allclose(got["q"], qp[key + "q"], rtol=0.0, atol=1e-10)


@pytest.mark.parametrize("variant", H.VARIANTS)
@pytest.mark.parametrize("name", ("c1", "c2", "c4_2", "bounds"))
def test_oracle_converged_optimum(name, variant):
    """mode 1 (tight ADMM + polish with KKT verification) reproduces the committed converged optimum,
    which was cross-checked against HiGHS when generated (oracle/gen_golden.py)."""
    conv = H.golden("converged")
    key = "%s/%s/" % (name, variant)
    r = _oracle_one(variant, name, WEIGHTS_FILE, 1)
    K = int(r["K"][0])
    assert r["status"][0] <= 1 and r["polish"][0] == 2
    assert H.close(r["ctrl"][0, :12 * K], conv[key + "ctrl"], rtol=1e-7, atol=1e-8)
    assert H.close(r["obj"][0], conv[key + "obj"], rtol=1e-9, atol=1e-7)
    assert float(conv[key + "highs_maxdiff"]) < 5e-5


@pytest.mark.parametrize("variant,weights,golden_file,tol", [
    ("trp", GOLDEN_W_TRP, "s1_slt_3d_31.txt", (0.0011, 0.0006, 0.0011, 0.0006, 0.0011, 0.0011)),
    ("cub", GOLDEN_W_CUB, "s1_cub_3d_31.txt", (0.024, 0.0006, 0.012, 0.0006, 0.015, 0.0006)),
])
def test_oracle_reproduces_shipped_known_answer(variant, weights, golden_file, tol):
    """The reference's only reproducible known-answer vectors (SURVEY.md 8c): c1.txt -> s1_*_3d_31.txt.
    The shipped files are OSQP's eps=1e-5 output printed with 3 decimals; the converged optimum sits within
    1e-3 (trp) / 2.3e-2 (cub s-axis, OSQP under-convergence) of them."""
    r = _oracle_one(variant, "c1", weights, 1)
    gold = read_trajectory_text(os.path.join(H.GOLDEN, golden_file))
    n = int(r["npts"][0])
    assert n == gold.shape[0]
    smp = r["samples"][0, :n]  # s ds dds l dl ddl ; file columns: t s l ds dl dds ddl
    cols = (smp[:, 0], smp[:, 3], smp[:, 1], smp[:, 4], smp[:, 2], smp[:, 5])
    for c in range(6):
        assert np.abs(cols[c] - gold[:, 1 + c]).max() <= tol[c], (c, np.abs(cols[c] - gold[:, 1 + c]).max())
    assert np.allclose(gold[:, 0], 0.1 * np.arange(n), atol=1e-9)


@pytest.mark.parametrize("name", ("c1", "c2", "c4_2"))
@pytest.mark.parametrize("variant", H.VARIANTS)
def test_oracle_sampling_and_cost_match_shipped_binary(name, variant):
    """a9 + a10: handed the same control points, the oracle writes the same 3-decimal trajectory and returns
    the same cost as the shipped binary did (the trp end term only when it is in bounds: weight_end_l = 0)."""
    g = H.golden("shipped_sampling")
    key = "%s/%s/" % (name, variant)
    if key + "ctrl" not in g.files:
        pytest.skip("no shipped sampling record")
    w = g[key + "weights"]
    r = _oracle_one(variant, name, w, 1)
    K = int(r["K"][0])
    assert H.close(r["ctrl"][0, :12 * K], g[key + "ctrl"], rtol=1e-6, atol=1e-7)
    traj = g[key + "traj"]
    n = int(r["npts"][0])
    assert n == traj.shape[0]
    smp = r["samples"][0, :n]
    ours = np.stack([smp[:, 0], smp[:, 3], smp[:, 1], smp[:, 4], smp[:, 2], smp[:, 5]], axis=1)
    assert np.abs(np.round(ours, 3) - traj[:, 1:7]).max() <= 1.01e-3
    if variant == "trp" and w[9] == 0.0:
        assert H.close(r["a_cost"][0], float(g[key + "retval"]), rtol=1e-5, atol=1e-6)


@pytest.mark.skipif(not po.have_reference(), reason="oracle/_ref not built (needs /root/reference at build time)")
@pytest.mark.parametrize("variant", H.VARIANTS)
def test_port_equals_recompiled_reference_on_perturbed_batch(variant):
    """The plain-C port vs the reference's own sources compiled where they lie: same corridors, statuses,
    iteration counts and control points on obstacle-perturbed scenarios (both run the same OSQP restatement)."""
    batch = perturbed_obstacles(load_fixture("c1"), 48, seed=99)
    a = po.solve_batch(variant, batch, WEIGHTS_FILE, mode=0, nthreads=0)
    b = po.solve_batch(variant, batch, WEIGHTS_FILE, mode=0, nthreads=0, kind="reference")
    assert np.array_equal(a["K"], b["K"]) and np.array_equal(a["status"], b["status"])
    for i in range(batch.batch):
        if a["status"][i] in (2, 5):
            continue
        assert H.segs_equal(a["segs"][i], b["segs"][i], int(a["K"][i]))
    ok = a["status"] <= 1
    assert ok.any()
    assert np.allclose(a["ctrl"][ok], b["ctrl"][ok], rtol=1e-9, atol=1e-9)
    assert np.allclose(a["a_cost"][ok], b["a_cost"][ok], rtol=1e-9)


def test_std_sort_restatement_equals_libstdcxx():
    """CollisionCheck's std::sort by beg_t (solve_3d.cc:630) is unstable past 16 elements; the restated
    introsort must order equal keys exactly like libstdc++ (tests/golden/std_sort.npz: the permutations the real
    std::sort with the reference's comparator produced, oracle/gen_std_sort_golden.py)."""
    z = H.golden("std_sort")
    assert int(z["n_cases"]) == 48
    for c in range(int(z["n_cases"])):
        keys = z["case%02d/keys" % c]
        assert np.array_equal(po.std_sort_check(keys, "port"), z["case%02d/perm" % c]), (c, len(keys))


def test_oracle_mixed_structure_runs_and_is_deterministic():
    for variant, batch in mixed_batches(40, seed=20230602)[:4]:
        a = po.solve_batch(variant, batch, WEIGHTS_FILE, mode=0, nthreads=0)
        b = po.solve_batch(variant, batch, WEIGHTS_FILE, mode=0, nthreads=1)
        assert np.array_equal(a["status"], b["status"]) and np.array_equal(a["ctrl"], b["ctrl"])
        assert a["K"].min() >= 0 and a["K"].max() <= 32
        assert np.all(a["a_cost"][a["status"] > 1] == 100000000000.0)


def test_config2_generator_contract():
    """SURVEY.md 8d config 2: scenario 0 is the unperturbed base, scenario b does not depend on the batch size,
    values rounded to 0.01, lo <= hi, s clamped to [0, 50]."""
    base = load_fixture("c1")
    a, b = config2(64), config2(16, first=8)
    assert np.array_equal(a.s_bounds[0], base.s_bounds) and np.array_equal(a.l_bounds[0], base.l_bounds)
    assert np.array_equal(a.s_bounds[8:24], b.s_bounds) and np.array_equal(a.l_bounds[8:24], b.l_bounds)
    assert np.all(a.s_bounds[..., 0] <= a.s_bounds[..., 1]) and np.all(a.l_bounds[..., 0] <= a.l_bounds[..., 1])
    assert a.s_bounds.min() >= 0.0 and a.s_bounds.max() <= 50.0
    assert np.allclose(a.s_bounds, np.round(a.s_bounds, 2)) and np.allclose(a.l_bounds, np.round(a.l_bounds, 2))
    assert set(FEASIBLE) <= set(H.ALL_FIXTURES)


# ---------------------------------------------------------------- downstream of the path (SURVEY.md 8f row 3)
def _rows_to_samples(rows):
    """trajectory file rows `t s l ds dl dds ddl` -> the C-ABI sample layout (s, ds, dds, l, dl, ddl)."""
    return np.stack([rows[:, 1], rows[:, 3], rows[:, 5], rows[:, 2], rows[:, 4], rows[:, 6]], axis=1)


def test_downstream_oracle_equals_reference_functions():
    """oracle/downstream_oracle.py vs tests/golden/downstream.npz, which the reference's OWN run_ego() and
    frenet_to_cartesian3D() produced (oracle/gen_downstream_golden.py executes them from /root/reference): exact."""
    import downstream_oracle as dso
    z = H.golden("downstream")
    keys = [k for k in z.files if k.endswith("/states")]
    assert len(keys) == 4
    for k in keys:
        rows = z[k.replace("/states", "/rows")]
        off = float(k.split("/off")[1].split("/")[0])
        got = dso.ego_states(_rows_to_samples(rows), off)
        assert np.array_equal(got, z[k]), k
    out = np.array([dso.frenet_to_cartesian3d(z["f2c/ref"][i], z["f2c/s_cond"][i], z["f2c/d_cond"][i]) for i in range(len(z["f2c/ref"]))])
    assert np.array_equal(out, z["f2c/out"])


# ---------------------------------------------------------------- upstream of the path (SURVEY.md 8f row 1)
def bounds_cases():
    """(obstacles [(centre, vel_s, vel_l, horizon)], s_bounds [R][N][2], l_bounds [R][N][2]) of tests/golden/bounds.npz."""
    z = H.golden("bounds")
    for c in range(int(z["n_cases"])):
        obs = [((r[0], r[1], r[2]), r[3], r[4], r[5]) for r in z["case%02d/obstacles" % c]]
        yield c, obs, z["case%02d/s_bounds" % c], z["case%02d/l_bounds" % c]


def test_bounds_oracle_equals_reference_get_bounds():
    """oracle/bounds_oracle.py vs tests/golden/bounds.npz, which the reference's OWN Car / get_bounds / lineFromPoints
    produced (oracle/gen_bounds_golden.py executes them from /root/reference/src/cart_frenet.py:644-1026): bit-exact
    on all cases (1-3 obstacles, lateral overlaps, cars entering at t0 > 0)."""
    import bounds_oracle as bo
    n = 0
    for c, obs, s_ref, l_ref in bounds_cases():
        got = bo.get_bounds(obs)
        s = np.array([g[0] for g in got])
        l = np.array([g[1] for g in got])
        assert s.shape == s_ref.shape, c
        assert np.array_equal(s, s_ref), c
        assert np.array_equal(np.broadcast_to(l[:, None, :], l_ref.shape), l_ref), c
        n += 1
    assert n >= 50
