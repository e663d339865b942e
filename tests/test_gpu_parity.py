"""GPU parity tests (run with `-m gpu` on the B200 box): the CUDA path, called through the C-ABI of
include/spectral.h, against the CPU oracle on the same inputs and against the committed goldens.

Bars: corridor segments (every Cube field) and the QP's (l, u) rows bit-exact; success/failure classes
identical; control points, objective and cost within 1e-5 rel / 1e-6 abs of the converged optimum."""
import ctypes
import os

import numpy as np
import pytest

import helpers as H
import pyoracle as po
from spectral_b200 import api
from spectral_b200.scenarios import (GOLDEN_W_CUB, GOLDEN_W_TRP, WEIGHTS_FILE, config2, config3, load_fixture, mixed_batches,
                                     perturbed_obstacles)
from spectral_b200.wire import ScenarioBatch, read_trajectory_text, write_scenario_text

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def planner():
    p = api.SpectralPlanner(device=0, max_batch=65536, n_max=128, r_max=8, k_max=32)
    yield p
    p.close()


# ---------------------------------------------------------------- reference fixtures (goldens)
@pytest.mark.parametrize("variant", H.VARIANTS)
@pytest.mark.parametrize("name", H.ALL_FIXTURES)
def test_fixture_segments_and_bounds_bit_exact(planner, name, variant):
    """new_corridor and the QP's l/u rows vs what the reference's own code produced (tests/golden)."""
    got = planner.solve(variant, H.fixture_batch(name), WEIGHTS_FILE, want_lu=True)
    gs = H.golden("ref_segments")["%s/%s/segs" % (name, variant)]
    K = len(gs)
    assert got.K[0] == K
    assert H.segs_equal(got.segs[0], gs.view(api.CUBE_DTYPE), K)
    qp = H.golden("shipped_qp")
    l, u = H.lu_to_qp_rows(got.lu[0], K)
    assert np.array_equal(l, qp["%s/%s/l" % (name, variant)])
    assert np.array_equal(u, qp["%s/%s/u" % (name, variant)])


@pytest.mark.parametrize("variant", H.VARIANTS)
@pytest.mark.parametrize("name", H.ALL_FIXTURES)
def test_fixture_solution_vs_converged_golden(planner, name, variant):
    got = planner.solve(variant, H.fixture_batch(name), WEIGHTS_FILE)
    conv = H.golden("converged")
    key = "%s/%s/ctrl" % (name, variant)
    ref_status = int(H.golden("ref_segments")["%s/%s/status" % (name, variant)])
    if key not in conv.files:
        if ref_status == 3:  # infeasible in the reference run -> must fail here too
            assert got.status[0] == api.FAIL_SOLVER and got.a_cost[0] == api.FAIL_COST
        return
    ref_iters = int(H.golden("ref_segments")["%s/%s/iters" % (name, variant)])
    if ref_iters > 3000 and not got.ok()[0]:
        # undecided class (helpers.decided_classes): the reference's own run sat at / near max_iter = 5000
        # (c6: cond(P) 2e13, OSQP "solved inaccurate" at iteration 5000), so whether 5000 ADMM iterations
        # suffice depends on rounding-level details of the iterate path
        assert got.status[0] == api.FAIL_SOLVER and got.a_cost[0] == api.FAIL_COST
        return
    assert got.ok()[0], (name, variant, got.status)
    K = int(got.K[0])
    x = conv[key]
    if got.verified()[0]:
        assert H.close(got.ctrl[0, :12 * K], x), H.maxdiff(got.ctrl[0, :12 * K], x)
        assert H.close(got.obj[0], conv["%s/%s/obj" % (name, variant)], rtol=2e-6)
    else:  # ill-conditioned fixtures (c6: cond 2e13): ADMM-accuracy solution, objective still close
        assert abs(got.obj[0] - conv["%s/%s/obj" % (name, variant)]) <= 1e-4 * abs(conv["%s/%s/obj" % (name, variant)])


@pytest.mark.parametrize("variant,weights,golden_file,tol", [
    ("trp", GOLDEN_W_TRP, "s1_slt_3d_31.txt", (0.0011, 0.0006, 0.0011, 0.0006, 0.0011, 0.0011)),
    # the reference's own OSQP output is under-converged on the cub s-axis (SURVEY.md 7.3-1)
    ("cub", GOLDEN_W_CUB, "s1_cub_3d_31.txt", (0.024, 0.0006, 0.012, 0.0006, 0.015, 0.0006)),
])
def test_find_traj_drop_in_reproduces_shipped_output(tmp_path, variant, weights, golden_file, tol):
    """Config 1: c1.txt through the plugin entry point find_traj(Params*) of OUR libtrp.so / libcub.so,
    hidden input/output files included, vs the reference's shipped output file."""
    os.environ["SPECTRAL_IO_DIR"] = str(tmp_path)
    try:
        write_scenario_text(str(tmp_path / ("c_road_s1_2.txt" if variant == "trp" else "c_road_s1_3.txt")),
                            load_fixture("c1"))
        cost = api._run_btrapz(api.Params(*weights, 31), variant)
        assert cost != api.FAIL_COST
        out = read_trajectory_text(str(tmp_path / ("s1_slt_3d_31.txt" if variant == "trp" else "s1_cub_3d_31.txt")))
        gold = read_trajectory_text(os.path.join(H.GOLDEN, golden_file))
        assert out.shape == gold.shape
        assert np.allclose(out[:, 0], gold[:, 0], atol=1e-9)
        for c in range(6):
            assert np.abs(out[:, 1 + c] - gold[:, 1 + c]).max() <= tol[c], (c, np.abs(out[:, 1 + c] - gold[:, 1 + c]).max())
        samp = H.golden("shipped_sampling")
        if variant == "trp":  # trp end term is out of bounds in the reference unless weight_end_l = 0
            w0 = list(weights)
            w0[9] = 0.0
            cost0 = api._run_btrapz(api.Params(*w0, 32), variant)
            assert H.close(cost0, float(samp["c1/trp/retval"]))
    finally:
        os.environ.pop("SPECTRAL_IO_DIR", None)


@pytest.mark.parametrize("module,weights,golden_file,tol", [
    ("trp_wrapper", GOLDEN_W_TRP, "s1_slt_3d_31.txt", (0.0011, 0.0006, 0.0011, 0.0006, 0.0011, 0.0011)),
    ("cub_wrapper", GOLDEN_W_CUB, "s1_cub_3d_31.txt", (0.024, 0.0006, 0.012, 0.0006, 0.015, 0.0006)),
])
def test_unchanged_reference_wrapper_reproduces_shipped_output(tmp_path, monkeypatch, module, weights, golden_file, tol):
    """Config 1 as SURVEY.md 8d prescribes it: the reference's OWN src/trp_wrapper.py / src/cub_wrapper.py, unmodified,
    import our .so from their hard-coded path (/home/srujan_d/RISS/code/btrapz/src) and run c1.txt; the file they make
    the library write is the reference's shipped output to its printed decimals.  Needs /root/reference (skipped on a
    box that does not have it: reference sources are not copied into this repo)."""
    from test_host_and_abi import REF_LIB_DIR, _stage_reference_wrapper
    w = _stage_reference_wrapper(tmp_path, monkeypatch, module)
    trp = module == "trp_wrapper"
    write_scenario_text(os.path.join(REF_LIB_DIR, "c_road_s1_2.txt" if trp else "c_road_s1_3.txt"), load_fixture("c1"))
    cost = w._run_btrapz(w.Params(*weights, 31))
    assert cost != 100000000000
    out = read_trajectory_text(os.path.join(REF_LIB_DIR, "s1_slt_3d_31.txt" if trp else "s1_cub_3d_31.txt"))
    gold = read_trajectory_text(os.path.join(H.GOLDEN, golden_file))
    assert out.shape == gold.shape
    for c in range(6):
        assert np.abs(out[:, 1 + c] - gold[:, 1 + c]).max() <= tol[c]
    with open(os.path.join(REF_LIB_DIR, "weights.txt"), "w") as f:
        f.write("\t".join(str(v) for v in WEIGHTS_FILE) + "\n")
    own = os.path.join(REF_LIB_DIR, "s1_slt_3d_3.txt" if trp else "s1_cub_3d_1.txt")
    if os.path.exists(own):
        os.remove(own)
    # the module's own entry: reads weights.txt; iteration = 3 in trp_wrapper.py:99-121, 1 in cub_wrapper.py:99-121
    assert w.find_traj() is True
    assert os.path.exists(own)


def test_find_traj_failure_sentinel(tmp_path):
    os.environ["SPECTRAL_IO_DIR"] = str(tmp_path)
    try:
        write_scenario_text(str(tmp_path / "c_road_s1_2.txt"), load_fixture("c_road_s1_2"))  # infeasible
        assert api._run_btrapz(api.Params(*WEIGHTS_FILE, 7), "trp") == api.FAIL_COST
        assert not (tmp_path / "s1_slt_3d_7.txt").exists()  # no file on failure (trp_wrapper.cpp:195-200)
        wf = tmp_path / "weights.txt"
        wf.write_text("\t".join(str(v) for v in WEIGHTS_FILE) + "\n")
        assert api.find_traj(str(wf), "trp") is False
        write_scenario_text(str(tmp_path / "c_road_s1_2.txt"), load_fixture("c1"))
        assert api.find_traj(str(wf), "trp") is True
        assert (tmp_path / "s1_slt_3d_3.txt").exists()
    finally:
        os.environ.pop("SPECTRAL_IO_DIR", None)


# ---------------------------------------------------------------- batches vs the oracle
NO_POLISH = dict(polish=0)  # the reference's own setting (solve_3d.cc:1243): the output is the raw ADMM iterate


def _raw(planner, variant, batch, weights):
    """The product run with the reference's polish = 0: its ADMM iterate, compared with the reference-settings oracle's."""
    return planner.solve(variant, batch, weights, options=api.default_options(**NO_POLISH))


def test_config2_cub_1024_vs_oracle(planner):
    """BASELINE configs[1]: 1024 obstacle-perturbed copies of scenario_1, cuboid variant."""
    batch = config2(1024)
    got = planner.solve("cub", batch, GOLDEN_W_CUB, samples_cap=160)
    ref, ref0 = H.oracle_pair("cub", batch, GOLDEN_W_CUB)
    both = H.assert_batch_parity(got, ref, "config2", need_verified_frac=0.85, ref0=ref0, batch=batch, variant="cub", weights=GOLDEN_W_CUB,
                                 got0=_raw(planner, "cub", batch, GOLDEN_W_CUB))
    for b in np.nonzero(both)[0][:64]:
        n = int(got.npts[b])
        assert H.close(got.samples[b, :n], ref["samples"][b, :n], rtol=1e-5, atol=2e-6)


def test_config2_trp_512_vs_oracle(planner):
    batch = perturbed_obstacles(load_fixture("c1"), 512, seed=77)
    got = planner.solve("trp", batch, GOLDEN_W_TRP)
    ref, ref0 = H.oracle_pair("trp", batch, GOLDEN_W_TRP)
    H.assert_batch_parity(got, ref, "trp512", need_verified_frac=0.6, ref0=ref0, batch=batch, variant="trp", weights=GOLDEN_W_TRP,
                          got0=_raw(planner, "trp", batch, GOLDEN_W_TRP))


def test_config3_shared_structure_groups_vs_oracle(planner):
    """BASELINE configs[2] at test size: scenario_2 (c2.txt), trapezoid-prism, 8 groups sharing one KKT structure each."""
    batch = config3(512, groups=8)
    got = planner.solve("trp", batch, WEIGHTS_FILE)
    ref, ref0 = H.oracle_pair("trp", batch, WEIGHTS_FILE)
    H.assert_batch_parity(got, ref, "config3", need_verified_frac=0.5, ref0=ref0, batch=batch, variant="trp", weights=WEIGHTS_FILE,
                          got0=_raw(planner, "trp", batch, WEIGHTS_FILE))
    for g in range(8):  # one structure per group, as the generator promises
        m = np.arange(512) % 8 == g
        assert len(set(got.K[m])) == 1


SHARED = dict(shared_kkt=1)  # K4a: shared-KKT tiles, multi-RHS solve on the FP64 tensor cores (qp_shared.cuh)


@pytest.mark.parametrize("groups", [1, 8, 64])
def test_shared_kkt_tiles_config3_vs_oracle(planner, groups):
    """BASELINE configs[2] through the shared-KKT path: tiles of 8 scenarios of one structure group against ONE reduced-KKT
    inverse (DMMA).  Same QP and same optimum as the reference: corridors bit-exact, decided solved / failed classes equal,
    KKT-verified control points within 1e-5 / 1e-6 of the converged oracle.  (Iteration counts are not OSQP's: the tile
    shares one scaling and one rho -- include/spectral.h, SpectralOptions::shared_kkt.)"""
    batch = config3(512, groups=groups)
    got = planner.solve("trp", batch, WEIGHTS_FILE, options=api.default_options(**SHARED))
    ref, ref0 = H.oracle_pair("trp", batch, WEIGHTS_FILE)
    H.assert_batch_parity(got, ref, "config3/shared/G%d" % groups, need_verified_frac=0.5, ref0=ref0, batch=batch, variant="trp",
                          weights=WEIGHTS_FILE, min_iters_equal_frac=0.0, max_undecided_mismatch_frac=0.05)
    # and against the per-scenario path: same classes wherever both hold a KKT proof, same optimum there
    per = planner.solve("trp", batch, WEIGHTS_FILE)
    both = got.verified() & per.verified()
    assert both.sum() >= 40, both.sum()
    for b in np.nonzero(both)[0]:
        K = int(got.K[b])
        assert H.close(got.ctrl[b, :12 * K], per.ctrl[b, :12 * K]), (b, H.maxdiff(got.ctrl[b, :12 * K], per.ctrl[b, :12 * K]))
    # deterministic run to run (tiles are formed from the sorted (structure key, index) order)
    again = planner.solve("trp", batch, WEIGHTS_FILE, options=api.default_options(**SHARED))
    assert np.array_equal(got.ctrl, again.ctrl) and np.array_equal(got.iters, again.iters) and np.array_equal(got.status, again.status)


def test_shared_kkt_mixed_structures_and_ragged_tiles(planner):
    """The shared path on a batch that is NOT made of clean groups: config-2 scenarios (482 structures per 1024: tiles of 1-3
    members, K > 8 members go to the per-scenario kernels) and per-scenario weights (the weights are part of the key)."""
    batch = config2(384)
    got = planner.solve("cub", batch, GOLDEN_W_CUB, options=api.default_options(**SHARED))
    ref, ref0 = H.oracle_pair("cub", batch, GOLDEN_W_CUB)
    # (with 1-3 members per tile the scaling / rho schedule differs from OSQP's on almost every scenario: the classes the
    # reference does not pin itself -- slowly converging or infeasible-but-"inaccurate" at the cap -- flip more often here)
    H.assert_batch_parity(got, ref, "config2/shared", need_verified_frac=0.5, ref0=ref0, batch=batch, variant="cub", weights=GOLDEN_W_CUB,
                          min_iters_equal_frac=0.0, max_undecided_mismatch_frac=0.12)
    w = np.tile(np.array(WEIGHTS_FILE), (64, 1))
    w[::2, 0] = 20.0   # two weight vectors -> two keys per structure
    b3 = config3(64, groups=1)
    got = planner.solve("trp", b3, w, options=api.default_options(**SHARED))
    ref, ref0 = H.oracle_pair("trp", b3, w)
    H.assert_batch_parity(got, ref, "weights/shared", ref0=ref0, batch=b3, variant="trp", weights=w, min_iters_equal_frac=0.0,
                          max_undecided_mismatch_frac=0.05)


def test_mixed_variable_structure_vs_oracle(planner):
    """config 4 shape at test size: heterogeneous K, both variants."""
    for variant, batch in mixed_batches(640, seed=20230602):
        got = planner.solve(variant, batch, WEIGHTS_FILE)
        ref, ref0 = H.oracle_pair(variant, batch, WEIGHTS_FILE)
        H.assert_batch_parity(got, ref, "mixed/%s" % variant, need_verified_frac=0.5, ref0=ref0, batch=batch, variant=variant, weights=WEIGHTS_FILE,
                              got0=_raw(planner, variant, batch, WEIGHTS_FILE))


def test_per_scenario_weights(planner):
    batch = config2(256)
    rng = np.random.default_rng(5)
    w = np.tile(np.array(GOLDEN_W_CUB), (256, 1))
    w[:, :4] = rng.uniform(1.0, 50.0, (256, 4))
    w[:, 5] = rng.uniform(1.0, 50.0, 256)
    got = planner.solve("cub", batch, w)
    ref, ref0 = H.oracle_pair("cub", batch, w)
    H.assert_batch_parity(got, ref, "weights", need_verified_frac=0.5, ref0=ref0, batch=batch, variant="cub", weights=w,
                          got0=_raw(planner, "cub", batch, w))


def test_many_segments_class_vs_oracle(planner):
    """K > 16 (the lane-per-segment kernel k_qp<32,2>, above the dense kernels' capacity): the N = 121 fixture with
    a staircase in the s-bounds gives K in [11, 29], 39 of 64 scenarios above 16.  Same bars as everywhere: segments bit-exact, the two axes solved as ONE
    OSQP instance (iteration count = the reference-settings oracle's), iterate and optimum parity."""
    from spectral_b200.scenarios import zigzag_breaks
    batch = zigzag_breaks(load_fixture("c7"), 64)
    got = planner.solve("trp", batch, WEIGHTS_FILE)
    assert (got.K > 16).sum() >= 30, got.K
    ref, ref0 = H.oracle_pair("trp", batch, WEIGHTS_FILE)
    H.assert_batch_parity(got, ref, "K>16", ref0=ref0, batch=batch, variant="trp", weights=WEIGHTS_FILE,
                          got0=_raw(planner, "trp", batch, WEIGHTS_FILE), max_undecided_mismatch_frac=0.05)


def test_weight_sweep_entry(planner):
    """spectral_solve_weights: one scenario, B weight vectors drawn like the reference's tuning objective (ten
    trial.suggest_float(.., 0, 50), trp_wrapper.py:69-80).  The corridor stage runs once; every lane must equal the same
    scenario replicated B times through the batch entry bit for bit, and the batch must meet the oracle's parity bars."""
    B = 192
    one = ScenarioBatch.from_scenarios([load_fixture("c1")])
    w = np.random.default_rng(20230604).uniform(0.0, 50.0, (B, 10))
    w[0] = GOLDEN_W_TRP
    got = planner.solve_weights("trp", one, w)
    rep = ScenarioBatch(one.n_knots, one.n_regions, one.delta_t, *[np.repeat(a, B, axis=0) for a in one.arrays()])
    same = planner.solve("trp", rep, w)
    for f in ("K", "status", "iters", "flags", "npts", "ctrl", "obj", "a_cost"):
        assert np.array_equal(getattr(got, f), getattr(same, f)), f
    assert got.segs.tobytes() == same.segs.tobytes()
    ref, ref0 = H.oracle_pair("trp", rep, w)
    H.assert_batch_parity(got, ref, "weight-sweep", ref0=ref0, batch=rep, variant="trp", weights=w,
                          got0=planner.solve_weights("trp", one, w, options=api.default_options(**NO_POLISH)))
    assert np.argmin(got.a_cost) == np.argmin(same.a_cost)


def test_edge_cases(planner):
    # B = 1, minimal horizon that still yields a corridor, R = 1
    sc = load_fixture("c2")
    got = planner.solve("trp", ScenarioBatch.from_scenarios([sc]), WEIGHTS_FILE)
    ref, ref0 = H.oracle_pair("trp", ScenarioBatch.from_scenarios([sc]), WEIGHTS_FILE)
    H.assert_batch_parity(got, ref, "c2", ref0=ref0)
    # a scenario whose reference trajectory lies outside every cube -> nothing selected
    far = load_fixture("c1")
    far.l_ref = far.l_ref + 100.0
    got = planner.solve("trp", ScenarioBatch.from_scenarios([far]), WEIGHTS_FILE)
    assert got.status[0] == api.FAIL_NO_CORRIDOR and got.K[0] == 0 and got.a_cost[0] == api.FAIL_COST
    # capacity / argument errors are reported, not crashed on
    small = api.SpectralPlanner(device=0, max_batch=4, n_max=64, r_max=2, k_max=8)
    with pytest.raises(RuntimeError):
        small.solve("trp", config2(8), WEIGHTS_FILE)           # B > max_batch
    with pytest.raises(RuntimeError):
        small.solve("trp", H.fixture_batch("c1"), WEIGHTS_FILE)  # N = 71 > n_max
    small.close()
    # k_max smaller than the segment count -> FAIL_TOO_MANY with the true K reported
    tight = api.SpectralPlanner(device=0, max_batch=4, n_max=128, r_max=8, k_max=4)
    got = tight.solve("trp", H.fixture_batch("c1"), WEIGHTS_FILE)
    assert got.status[0] == api.FAIL_TOO_MANY and got.K[0] == 8
    tight.close()


# ---------------------------------------------------------------- size-independent properties at full size
def test_full_size_properties_65536(planner):
    """config-3 size: determinism, permutation invariance and KKT verification at B = 65 536."""
    B = 65536
    batch = perturbed_obstacles(load_fixture("c2"), B, seed=20230601)
    a = planner.solve("trp", batch, WEIGHTS_FILE)
    b = planner.solve("trp", batch, WEIGHTS_FILE)
    assert np.array_equal(a.K, b.K) and a.segs.tobytes() == b.segs.tobytes()
    assert np.array_equal(a.status, b.status)
    assert np.array_equal(a.ctrl, b.ctrl), "the path must be deterministic run to run"
    ok = a.ok()
    assert ok.sum() > 0
    s0 = a.status == 0
    assert s0.sum() > 0 and (a.verified() & s0).sum() >= 0.5 * s0.sum()
    assert np.all(a.a_cost[~ok] == api.FAIL_COST)
    # permuting the scenarios of a batch permutes the answers bit for bit (no cross-scenario coupling, no
    # dependence on which CTA / lane group / solver-class slot a scenario lands in)
    perm = np.random.default_rng(11).permutation(B)
    shuffled = ScenarioBatch(batch.n_knots, batch.n_regions, batch.delta_t, *[x[perm] for x in batch.arrays()])
    c = planner.solve("trp", shuffled, WEIGHTS_FILE)
    assert np.array_equal(c.K, a.K[perm]) and np.array_equal(c.status, a.status[perm]) and np.array_equal(c.iters, a.iters[perm])
    assert np.array_equal(c.ctrl, a.ctrl[perm]) and np.array_equal(c.a_cost, a.a_cost[perm])
    # every KKT-verified optimum is primal feasible for its own corridor: sampled s stays inside [0, 50] and the
    # trajectory starts at the initial state
    ver = a.verified()
    assert ver.sum() > 0
    # a prefix of a batch gives the same answers as the full batch (no cross-scenario coupling)
    p = planner.solve("trp", batch.slice(0, 1000), WEIGHTS_FILE)
    assert np.array_equal(p.ctrl, a.ctrl[:1000]) and np.array_equal(p.status, a.status[:1000])
    # spot-check 256 random scenarios against the oracle
    idx = np.sort(np.random.default_rng(1).choice(B, 256, replace=False))
    sub = ScenarioBatch(batch.n_knots, batch.n_regions, batch.delta_t, *[x[idx] for x in batch.arrays()])
    ref, ref0 = H.oracle_pair("trp", sub, WEIGHTS_FILE)
    g = api.BatchResult(a.K[idx], a.segs[idx], a.ctrl[idx], a.obj[idx], a.a_cost[idx], a.status[idx], a.iters[idx],
                        a.flags[idx], a.npts[idx])
    H.assert_batch_parity(g, ref, "spot65536", need_verified_frac=0.5, ref0=ref0, batch=sub, variant="trp", weights=WEIGHTS_FILE)


# ---------------------------------------------------------------- resident path + argmin
def test_device_resident_path_and_argmin(planner):
    import torch
    batch = config2(2048)
    host = planner.solve("cub", batch, GOLDEN_W_CUB)
    dev = torch.device("cuda", 0)
    names = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")
    inputs = {k: torch.from_numpy(np.ascontiguousarray(a)).to(dev) for k, a in zip(names, batch.arrays())}
    inputs["weights"] = torch.tensor(GOLDEN_W_CUB, dtype=torch.float64, device=dev)
    outs = planner.alloc_device_outputs(2048)
    planner.solve_device("cub", batch.n_knots, batch.n_regions, batch.delta_t, inputs, outs)
    best_cost = torch.zeros(1, dtype=torch.float64, device=dev)
    best_idx = torch.zeros(1, dtype=torch.int64, device=dev)
    planner.argmin_device(outs["a_cost"], 1000, best_cost, best_idx)
    torch.cuda.synchronize()
    assert np.array_equal(outs["K"].cpu().numpy(), host.K)
    assert np.array_equal(outs["status"].cpu().numpy(), host.status)
    assert np.array_equal(outs["ctrl"].cpu().numpy(), host.ctrl)
    assert np.array_equal(outs["a_cost"].cpu().numpy(), host.a_cost)
    j = int(np.argmin(host.a_cost))  # numpy argmin returns the first minimum = lowest index on ties
    assert int(best_idx.item()) == 1000 + j and best_cost.item() == host.a_cost[j]


def test_sweep_argmin_through_the_c_abi():
    """Config-5 path at test size, one rank: spectral_sweep_argmin (top-k with k = 1 -> winner payload) returns the arg-min
    scenario's K / segments / control points; cutting the same sweep into two contiguous shards (what two ranks would run)
    gives the same winner -- it does not depend on the number of ranks (ties -> lowest global index)."""
    import torch
    from spectral_b200 import sweep_driver as sd
    dev = torch.device("cuda", 0)
    pl = api.SpectralPlanner(device=0, max_batch=sd.CHUNK, n_max=128, r_max=8, k_max=16)
    pl.comm_init(1, 0, None)
    total = 4 * sd.CHUNK
    shard = sd.upload_shard(total, 0, 1, dev)
    outs = pl.alloc_device_outputs(total)
    win = sd.run_sweep(pl, shard, outs)
    cost = outs["a_cost"].cpu().numpy()
    j = int(np.argmin(cost))
    assert win["index"] == j and win["cost"] == cost[j] and win["rank"] == 0 and cost[j] < api.FAIL_COST
    K = int(outs["K"][j].item())
    assert win["K"] == K
    assert np.array_equal(win["ctrl"], outs["ctrl"][j].cpu().numpy()[:12 * K])
    segs = outs["segs"][j].cpu().numpy().view(api.CUBE_DTYPE)[:K]
    assert win["segs"].tobytes() == segs.tobytes()
    halves = []
    for r in range(2):
        sh = sd.upload_shard(total, r, 2, dev)
        o = pl.alloc_device_outputs((sh["g_hi"] - sh["g_lo"]) * sd.CHUNK)
        halves.append(sd.run_sweep(pl, sh, o))
    best = min(halves, key=lambda w: (w["cost"], w["index"]))
    assert best["index"] == win["index"] and best["cost"] == win["cost"] and np.array_equal(best["ctrl"], win["ctrl"])
    pl.close()


def test_upstream_bounds_kernel_and_obstacle_driven_solve(planner):
    """SURVEY.md 8f row 1 on the device: k_bounds vs the reference's own get_bounds output (tests/golden/bounds.npz) and vs the
    pinned oracle on 6 000 random obstacle sets -- bit for bit; then the obstacle-driven pipeline k_bounds -> corridor -> QP with
    no bounds upload: identical to the host-buffer solve of the same (padded) bounds, and in parity with the CPU oracle."""
    import torch
    from spectral_b200.scenarios import random_obstacles
    from test_oracle_golden import bounds_cases
    dev = torch.device("cuda", 0)
    for c, obs, s_ref, l_ref in bounds_cases():
        o = torch.tensor([[[cc[0], cc[1], cc[2], vs, vl, T] for cc, vs, vl, T in obs]], dtype=torch.float64, device=dev)
        sb, lb, nl = planner.bounds_device(o, s_ref.shape[1], len(s_ref))
        assert int(nl[0]) == len(s_ref), c
        assert np.array_equal(sb[0].cpu().numpy(), s_ref) and np.array_equal(lb[0].cpu().numpy(), l_ref), c
    obs, n_obs = random_obstacles(6000, max_obs=4, seed=11)
    sb, lb, nl = planner.bounds_device(torch.from_numpy(obs).to(dev), 71, 12, n_obs=torch.from_numpy(n_obs).to(dev))
    n_over = H.assert_bounds_equal_oracle(sb.cpu().numpy(), lb.cpu().numpy(), nl.cpu().numpy(), obs, n_obs, 71, 12)
    assert n_over < 300
    # obstacle-driven solve: 384 sets of one or two cars on the c1 scene (references, derivative bounds, initial state of c1)
    B, R = 384, 8
    obs, n_obs = random_obstacles(B, max_obs=2, seed=5)
    base = load_fixture("c1")
    d_obs = torch.from_numpy(obs).to(dev)
    sb, lb, nl = planner.bounds_device(d_obs, base.n_knots, R, n_obs=torch.from_numpy(n_obs).to(dev))
    assert int(nl.min()) >= 2
    tile = lambda a: np.ascontiguousarray(np.broadcast_to(a, (B,) + a.shape))  # noqa: E731
    init = np.concatenate([base.init_s, base.init_l])
    padded = ScenarioBatch(base.n_knots, R, base.delta_t, sb.cpu().numpy(), lb.cpu().numpy(), tile(base.ds_bounds), tile(base.dl_bounds),
                           tile(base.s_ref), tile(base.l_ref), tile(init), tile(base.scalars))
    inputs = dict(s_bounds=sb, l_bounds=lb, weights=torch.tensor(GOLDEN_W_TRP, dtype=torch.float64, device=dev))
    for k in ("ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars"):
        inputs[k] = torch.from_numpy(getattr(padded, k)).to(dev)
    outs = planner.alloc_device_outputs(B)
    planner.solve_device("trp", base.n_knots, R, base.delta_t, inputs, outs)
    torch.cuda.synchronize()
    got = planner.solve("trp", padded, GOLDEN_W_TRP)
    assert np.array_equal(outs["K"].cpu().numpy(), got.K) and np.array_equal(outs["status"].cpu().numpy(), got.status)
    assert np.array_equal(outs["ctrl"].cpu().numpy(), got.ctrl) and np.array_equal(outs["a_cost"].cpu().numpy(), got.a_cost)
    ref, ref0 = H.oracle_pair("trp", padded, GOLDEN_W_TRP)
    got0 = planner.solve("trp", padded, GOLDEN_W_TRP, options=api.default_options(polish=0))
    H.assert_batch_parity(got, ref, "obstacle-driven", ref0=ref0, batch=padded, variant="trp", weights=GOLDEN_W_TRP, got0=got0)
    assert got.ok().sum() > B // 8


def test_downstream_ego_states_and_frenet_to_cartesian(planner):
    """SURVEY.md 8f row 3 on the device: k_ego_states vs the reference's own run_ego() output (tests/golden/downstream.npz;
    positions and the 0.01-rad headings bit-exact, speed to 1e-12: the reference takes `** 0.5`, the kernel sqrt), on a solved
    batch vs the oracle restatement, and k_frenet_to_cartesian vs the reference's frenet_to_cartesian3D (1e-12 relative)."""
    import torch
    import downstream_oracle as dso
    from test_oracle_golden import _rows_to_samples
    dev = torch.device("cuda", 0)
    z = H.golden("downstream")
    for k in [k for k in z.files if k.endswith("/states")]:
        rows = z[k.replace("/states", "/rows")]
        off = float(k.split("/off")[1].split("/")[0])
        smp = torch.from_numpy(_rows_to_samples(rows)[None].copy()).to(dev)
        st = planner.ego_states_device(smp, torch.tensor([len(rows)], dtype=torch.int32, device=dev),
                                       torch.tensor([off], dtype=torch.float64, device=dev)).cpu().numpy()[0]
        assert np.array_equal(st[:, [0, 1, 3]], z[k][:, [0, 1, 3]]), k
        assert np.allclose(st[:, 2], z[k][:, 2], rtol=1e-12, atol=0.0)
    # a solved batch: every trajectory the product samples
    batch = config2(256)
    got = planner.solve("cub", batch, GOLDEN_W_CUB, samples_cap=96)
    off = np.linspace(0.0, 25.5, 256)
    st = planner.ego_states_device(torch.from_numpy(got.samples).to(dev), torch.from_numpy(got.npts).to(dev),
                                   torch.from_numpy(off).to(dev)).cpu().numpy()
    n_ok = 0
    for b in np.nonzero(got.ok())[0]:
        n = int(got.npts[b])
        want = dso.ego_states(got.samples[b, :n], off[b])
        assert np.array_equal(st[b, :n, [0, 1, 3]], want[:, [0, 1, 3]].T), b
        assert np.allclose(st[b, :n, 2], want[:, 2], rtol=1e-12, atol=0.0)
        assert not st[b, n:].any()
        n_ok += 1
    assert n_ok > 50
    out = planner.frenet_to_cartesian_device(torch.from_numpy(z["f2c/ref"]).to(dev), torch.from_numpy(z["f2c/s_cond"]).to(dev),
                                             torch.from_numpy(z["f2c/d_cond"]).to(dev)).cpu().numpy()
    assert np.allclose(out, z["f2c/out"], rtol=1e-12, atol=1e-13), np.abs(out - z["f2c/out"]).max()


def test_infeasibility_precheck_is_sound(planner):
    """Option infeasibility_precheck: every scenario it fails early is one the CONVERGED oracle fails too (and never one
    whose solved class the reference pins); every other scenario is bit-identical to the run without the option."""
    batch = config2(1024)
    off = planner.solve("cub", batch, GOLDEN_W_CUB)
    on = planner.solve("cub", batch, GOLDEN_W_CUB, options=api.default_options(infeasibility_precheck=1))
    early = (on.status == api.FAIL_SOLVER) & (on.iters == 0) & (off.iters > 0)
    assert early.sum() > 100, "config 2 holds hundreds of provably empty corridors"
    ref, ref0 = H.oracle_pair("cub", batch, GOLDEN_W_CUB)
    # the converged oracle never reaches an accurate optimum on them (a handful end as "solved inaccurate" at its
    # iteration cap: ADMM hovering at a small residual of an infeasible problem), none carries a KKT proof ...
    assert np.all(ref["status"][early] != 0) and not (ref["polish"][early] == 2).any(), \
        "pre-check failed a scenario that has a converged optimum"
    assert (ref["status"][early] > 1).mean() > 0.98
    # ... and an independent solver (HiGHS on the reference-assembled QP) finds no optimum either
    for b in np.nonzero(early)[0][::max(1, int(early.sum()) // 24)]:
        K = int(on.K[b])
        assert H.highs_solution("cub", batch, int(b), GOLDEN_W_CUB, ref0["segs"][b, :K]) is None, b
    decided_solved = H.decided_classes(ref, ref0) & (ref0["status"] <= 1)
    assert not (early & decided_solved).any()
    assert np.all(on.a_cost[early] == api.FAIL_COST)
    rest = ~early
    assert np.array_equal(on.status[rest], off.status[rest]) and np.array_equal(on.iters[rest], off.iters[rest])
    assert np.array_equal(on.ctrl[rest], off.ctrl[rest]) and np.array_equal(on.a_cost[rest], off.a_cost[rest])
    assert on.segs.tobytes() == off.segs.tobytes() and np.array_equal(on.K, off.K)


def test_async_pipeline_matches_sync(planner):
    """spectral_solve_batch_async / spectral_wait over page-locked buffers, three handles cycled like a sweep driver:
    bit-identical to the synchronous entry point."""
    batches = [config2(512, first=512 * i) for i in range(5)]
    sync = [planner.solve("cub", b, GOLDEN_W_CUB) for b in batches]
    pls = [api.SpectralPlanner(device=0, max_batch=512, n_max=128, r_max=8, k_max=32) for _ in range(3)]
    got = [None] * len(batches)
    owner = {}
    for i, b in enumerate(batches):
        pl = pls[i % 3]
        if i % 3 in owner:
            r = pl.wait()
            got[owner[i % 3]] = api.BatchResult(*[np.array(getattr(r, f)) for f in ("K", "segs", "ctrl", "obj", "a_cost", "status", "iters", "flags", "npts")])
        pl.solve_async("cub", b, GOLDEN_W_CUB)
        owner[i % 3] = i
    for j, i in owner.items():
        r = pls[j].wait()
        got[i] = api.BatchResult(*[np.array(getattr(r, f)) for f in ("K", "segs", "ctrl", "obj", "a_cost", "status", "iters", "flags", "npts")])
    with pytest.raises(RuntimeError):
        pls[0].wait()  # nothing in flight
    for a, b in zip(sync, got):
        assert np.array_equal(a.K, b.K) and np.array_equal(a.status, b.status) and np.array_equal(a.iters, b.iters)
        assert a.segs.tobytes() == b.segs.tobytes()
        assert np.array_equal(a.ctrl, b.ctrl) and np.array_equal(a.a_cost, b.a_cost)
    for pl in pls:
        pl.close()


def test_library_exports_and_fp64_probe(planner):
    lib = api.load_library()
    hdr = open(os.path.join(H.ROOT, "include", "spectral.h")).read()
    import re
    for sym in set(re.findall(r"\b(spectral_[a-z0-9_]+)\s*\(", hdr)):
        assert hasattr(lib, sym), sym
    tf = planner.measure_fp64_peak()
    assert 5.0 < tf < 100.0, tf
