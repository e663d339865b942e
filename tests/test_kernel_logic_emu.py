"""CPU tests (`-m "not gpu"`): the kernels' device bodies (spectral_b200/csrc/*.cuh), compiled for the host by
tests/warp_emu (one warp = 32 lock-stepped threads, warp votes/shuffles emulated), against the goldens and the
CPU oracle.  This checks the kernel LOGIC where no GPU exists; the GPU parity tests proper are in
test_gpu_parity.py.  The emulator is test infrastructure, never a product path."""
import numpy as np
import pytest

import helpers as H
import pyoracle as po
from spectral_b200 import api
from spectral_b200.scenarios import GOLDEN_W_TRP, WEIGHTS_FILE, config2, load_fixture, mixed_batches
from spectral_b200.wire import ScenarioBatch


@pytest.mark.parametrize("variant", H.VARIANTS)
@pytest.mark.parametrize("name", H.ALL_FIXTURES)
def test_emu_corridor_and_bounds_bit_exact(name, variant):
    """K1 + K2 (corridor.cuh) and the K3 row assembly of qp.cuh: segments and (l, u) rows bit-exact."""
    got = H.emu_solve(variant, H.fixture_batch(name), WEIGHTS_FILE, want_lu=True, max_iter=25, polish=0)
    gs = H.golden("ref_segments")["%s/%s/segs" % (name, variant)].view(api.CUBE_DTYPE)
    K = len(gs)
    assert got.K[0] == K
    assert H.segs_equal(got.segs[0], gs, K)
    qp = H.golden("shipped_qp")
    l, u = H.lu_to_qp_rows(got.lu[0], K)
    assert np.array_equal(l, qp["%s/%s/l" % (name, variant)])
    assert np.array_equal(u, qp["%s/%s/u" % (name, variant)])


def test_emu_corridors_on_perturbed_and_mixed_batches():
    cases = [("cub", config2(24))] + mixed_batches(40, seed=20230602)[:4]
    for variant, batch in cases:
        got = H.emu_solve(variant, batch, WEIGHTS_FILE, max_iter=25, polish=0)
        ref = po.solve_batch(variant, batch, WEIGHTS_FILE, mode=0, nthreads=0)
        assert np.array_equal(got.K, ref["K"])
        for b in range(batch.batch):
            if ref["status"][b] in (2, 5):
                assert got.status[b] == ref["status"][b]
                continue
            assert H.segs_equal(got.segs[b], ref["segs"][b], int(got.K[b])), (variant, b)


def test_emu_full_solve_c2_matches_converged_oracle():
    """K3 + K4b + polish + K5 on an easy fixture (a few hundred ADMM iterations): control points, objective,
    samples and cost vs the converged oracle."""
    batch = ScenarioBatch.from_scenarios([load_fixture("c2")])
    got = H.emu_solve("trp", batch, GOLDEN_W_TRP, samples_cap=160)
    ref, ref0 = H.oracle_pair("trp", batch, GOLDEN_W_TRP)
    both = H.assert_batch_parity(got, ref, "emu/c2", need_verified_frac=1.0, ref0=ref0)
    assert both.all()
    n = int(got.npts[0])
    assert H.close(got.samples[0, :n], ref["samples"][0, :n], rtol=1e-5, atol=2e-6)
    # both axes are solved as ONE OSQP instance like the reference's single osqp_solve: same iteration count
    assert int(got.iters[0]) == int(ref0["iters"][0]) < 5000


def _subset(batch, idx):
    idx = np.asarray(idx)
    return ScenarioBatch(batch.n_knots, batch.n_regions, batch.delta_t, *[x[idx] for x in batch.arrays()])


def test_emu_dense_kernel_tracks_reference_osqp():
    """The dense-operator ADMM loop (qp_anchor.cuh, k_qpa<8> and k_qpa<10>) solves both axes of a scenario as ONE
    OSQP instance like the reference: on scenarios that converge quickly the ITERATION COUNT equals that of the
    reference-settings oracle, infeasible ones are certified at the same check, and the polished control
    points match the converged oracle.  Scenarios: K = 9 (#779), K = 10 (#508: 1200 iterations), an early
    infeasible one (#914) and the K = 8 base (#0) of config 2."""
    from spectral_b200.scenarios import GOLDEN_W_CUB
    batch = _subset(config2(1024), [0, 779, 914])
    got = H.emu_solve("cub", batch, GOLDEN_W_CUB)
    ref, ref0 = H.oracle_pair("cub", batch, GOLDEN_W_CUB)
    assert list(got.K) == [8, 9, 4]
    assert np.array_equal(got.iters, ref0["iters"]), (got.iters, ref0["iters"])
    assert np.array_equal(got.ok(), ref0["status"] <= 1)
    H.assert_batch_parity(got, ref, "emu/dense", need_verified_frac=1.0, ref0=ref0)


def test_emu_anchor_layout_equals_fullrow(monkeypatch):
    """The anchor layout (qp_anchor.cuh, the K <= 10 classes) orders the arithmetic of every iterate exactly like the
    full-row loop of qp_dense.cuh it replaces: identical control points, iteration counts and flags, bit for bit
    (K = 9 -> k_qpa<10>, an early infeasible K = 4 -> k_qpa<8>, adaptive-rho updates on the way)."""
    from spectral_b200.scenarios import GOLDEN_W_CUB
    batch = _subset(config2(1024), [779, 914])
    new = H.emu_solve("cub", batch, GOLDEN_W_CUB)
    monkeypatch.setenv("SPECTRAL_EMU_FULLROW", "1")
    old = H.emu_solve("cub", batch, GOLDEN_W_CUB)
    assert list(new.K) == [9, 4]
    assert np.array_equal(new.iters, old.iters) and np.array_equal(new.status, old.status) and np.array_equal(new.flags, old.flags)
    assert np.array_equal(new.ctrl, old.ctrl) and np.array_equal(new.obj, old.obj)


def test_emu_many_segments_joint_solve():
    """K > 16 (k_qp<32,2>: one warp per axis, joint reductions across the two warps): the iteration count equals the
    reference-settings oracle's, i.e. the two axes really are ONE OSQP instance (ADVICE r1: they were two)."""
    from spectral_b200.scenarios import zigzag_breaks
    batch = _subset(zigzag_breaks(load_fixture("c7"), 64), [8, 16])   # K = 18 (certified infeasible), K = 19 (solved)
    got = H.emu_solve("trp", batch, WEIGHTS_FILE, polish=0)
    ref0 = po.solve_batch("trp", batch, WEIGHTS_FILE, mode=0)
    assert list(got.K) == [18, 19]
    assert np.array_equal(got.iters, ref0["iters"]) and np.array_equal(got.ok(), ref0["status"] <= 1)
    assert H.maxdiff(got.ctrl[1, :12 * 19], ref0["ctrl"][1, :12 * 19]) < 1e-5


def test_emu_lane_kernel_matches_dense_kernel(monkeypatch):
    """The lane-per-segment body of k_qp<32,2> (qp.cuh, the product's kernel above the dense kernels' capacity, K > 16),
    run here at K <= 16, and the dense loop are the same OSQP iteration: same iteration count, same status, same polished
    optimum."""
    batch = ScenarioBatch.from_scenarios([load_fixture("c4_2")])
    dense = H.emu_solve("trp", batch, WEIGHTS_FILE)
    monkeypatch.setenv("SPECTRAL_EMU_LANES", "1")
    lanes = H.emu_solve("trp", batch, WEIGHTS_FILE)
    assert dense.status[0] == lanes.status[0] == 0 and dense.iters[0] == lanes.iters[0]
    assert dense.verified()[0] and lanes.verified()[0]
    K = int(dense.K[0])
    assert H.close(dense.ctrl[0, :12 * K], lanes.ctrl[0, :12 * K], rtol=1e-7, atol=1e-8)


def test_emu_failure_classes():
    far = load_fixture("c1")
    far.l_ref = far.l_ref + 100.0
    got = H.emu_solve("trp", ScenarioBatch.from_scenarios([far]), WEIGHTS_FILE, max_iter=25)
    assert got.status[0] == api.FAIL_NO_CORRIDOR and got.K[0] == 0 and got.a_cost[0] == api.FAIL_COST
    got = H.emu_solve("trp", H.fixture_batch("c1"), WEIGHTS_FILE, k_max=4, max_iter=25)
    assert got.status[0] == api.FAIL_TOO_MANY and got.K[0] == 8


def test_emu_infeasibility_precheck():
    """The optional interval pre-check (SpectralOptions.infeasibility_precheck) fails provably empty corridors before
    the first ADMM iteration and leaves the others alone (scenarios 914 and 5 of config 2 have disjoint joint intervals)."""
    from spectral_b200.scenarios import GOLDEN_W_CUB
    batch = _subset(config2(1024), [0, 914, 3, 5])
    off = H.emu_solve("cub", batch, GOLDEN_W_CUB, max_iter=100)
    on = H.emu_solve("cub", batch, GOLDEN_W_CUB, max_iter=100, infeasibility_precheck=1)
    assert list(off.iters) == [100, 100, 100, 100]
    assert list(on.iters) == [100, 0, 100, 0]
    assert on.status[1] == on.status[3] == api.FAIL_SOLVER and on.a_cost[1] == api.FAIL_COST
    assert np.array_equal(on.ctrl[[0, 2]], off.ctrl[[0, 2]])


# ---------------------------------------------------------------- upstream bound generator (bounds.cuh)
def test_emu_bounds_kernel_equals_reference_goldens():
    """bounds.cuh's warp body vs tests/golden/bounds.npz (the reference's OWN Car / get_bounds, executed from its source): the
    region bounds bit for bit on all 58 obstacle sets."""
    from test_oracle_golden import bounds_cases
    n = 0
    for c, obs, s_ref, l_ref in bounds_cases():
        o = np.array([[cc[0], cc[1], cc[2], vs, vl, T] for cc, vs, vl, T in obs])[None]
        R = len(s_ref)
        sb, lb, nl = H.emu_bounds(o, [len(obs)], s_ref.shape[1], R)
        assert nl[0] == R, (c, nl[0], R)
        assert np.array_equal(sb[0], s_ref), c
        assert np.array_equal(lb[0], l_ref), c
        n += 1
    assert n >= 50


def test_emu_bounds_kernel_random_obstacles_and_padding():
    """2 000 random obstacle sets (1-4 cars) vs the pinned oracle, with the output padded to 12 lanes; and the padding lanes
    are inert: the corridor stage on the padded regions gives the corridors of the unpadded scenario."""
    from spectral_b200.scenarios import random_obstacles
    obs, n_obs = random_obstacles(2000, max_obs=4, seed=7)
    sb, lb, nl = H.emu_bounds(obs, n_obs, 71, 12)
    n_over = H.assert_bounds_equal_oracle(sb, lb, nl, obs, n_obs, 71, 12)
    assert n_over < 100 and (nl > 0).sum() > 1900
    assert len(np.unique(nl)) >= 6
    # capacity / argument edge cases: no obstacle, more obstacles than slots, more lanes than R_cap -> n_lanes = -1 and the
    # whole output written as empty lanes (a solve on it reports "no corridor" instead of reading garbage)
    sb, lb, nl = H.emu_bounds(obs[:3], [0, 5, int(n_obs[2])], 71, 12)
    assert nl[0] == -1 and nl[1] == -1 and nl[2] > 0
    assert np.all(lb[:2, :, :, 0] == 1.0) and np.all(lb[:2, :, :, 1] == -1.0) and np.all(sb[:2, :, :, 1] == 50.0)
    sb, lb, nl = H.emu_bounds(obs[:64], n_obs[:64], 71, 2)
    assert (nl == -1).sum() > 32 and np.all(lb[nl == -1][:, :, :, 0] == 1.0)
    # padding is inert for the corridor stage: fixture c1 (2 regions) padded with 3 empty lanes
    base = H.fixture_batch("c1")
    N = base.n_knots
    pad_s = np.tile(np.array([0.0, 50.0]), (1, 3, N, 1))
    pad_l = np.tile(np.array([1.0, -1.0]), (1, 3, N, 1))
    padded = ScenarioBatch(N, base.n_regions + 3, base.delta_t, np.concatenate([base.s_bounds, pad_s], 1), np.concatenate([base.l_bounds, pad_l], 1),
                           base.ds_bounds, base.dl_bounds, base.s_ref, base.l_ref, base.init, base.scalars)
    for variant in H.VARIANTS:
        a = po.solve_batch(variant, base, WEIGHTS_FILE, mode=0, nthreads=1)
        b = po.solve_batch(variant, padded, WEIGHTS_FILE, mode=0, nthreads=1)
        assert a["K"][0] == b["K"][0] and H.segs_equal(a["segs"][0], b["segs"][0], int(a["K"][0]))
        assert np.array_equal(a["ctrl"], b["ctrl"])
        g = H.emu_solve(variant, padded, WEIGHTS_FILE, max_iter=25, polish=0)
        assert g.K[0] == a["K"][0] and H.segs_equal(g.segs[0], a["segs"][0], int(a["K"][0]))
