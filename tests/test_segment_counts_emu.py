"""CPU tests (`-m "not gpu"`) of the segment-count ladder (scenarios.segment_ladder) and of the corridor stage on regions with
many slope breaks, through the kernels' device bodies compiled for the host (tests/warp_emu) and the CPU oracle.
The same cases run on the device in test_segment_counts.py."""
import numpy as np
import pytest

import helpers as H
import pyoracle as po
from spectral_b200 import api
from spectral_b200.scenarios import GOLDEN_W_CUB, WEIGHTS_FILE, ladder_shape, segment_ladder, slope_wiggle, wiggle_batch
from spectral_b200.wire import Scenario

W = {"trp": WEIGHTS_FILE, "cub": GOLDEN_W_CUB}


@pytest.mark.parametrize("variant", H.VARIANTS)
def test_ladder_has_exactly_the_segment_count_it_is_built_for(variant):
    """Every scenario of segment_ladder(K) has K segments in the oracle, K = 1 .. 34; above 32 that is "too many segments"
    with the true count reported.  All scenarios of one K share the segment durations (one KKT structure)."""
    for K in range(1, 35):
        batch = segment_ladder(K, 8)
        assert batch.n_knots == ladder_shape(K)[0]
        ref = po.solve_batch(variant, batch, W[variant], mode=0, k_max=0, nthreads=0)   # k_max = 0: the corridor stage only
        assert np.all(ref["K"] == K), (K, ref["K"])
        assert np.all(ref["status"] == api.FAIL_TOO_MANY)
        if K <= 32:
            ref = po.solve_batch(variant, batch.slice(0, 3), W[variant], mode=0, nthreads=0)
            assert np.all(ref["K"] == K)
            t = ref["segs"][:, :K]["t"]
            assert np.all(t == t[0]), K


# class edges of the QP stage's dispatch (finalize.cuh lane_class): K <= 8 | 9-10 | 11-12 | 13-16 | 17-32
EDGES = [(1, "trp"), (8, "cub"), (9, "trp"), (10, "trp"), (11, "cub"), (12, "trp"), (13, "trp"), (16, "trp"), (17, "cub")]


@pytest.mark.parametrize("K,variant", EDGES)
def test_emu_ladder_class_edges_match_oracle(K, variant):
    """One ladder scenario per class edge through the emulated kernels: the ADMM iteration count equals the reference-settings
    oracle's, and the polished optimum is KKT-verified and within the parity tolerance of the converged oracle."""
    batch = segment_ladder(K, 2).slice(1, 2)
    got = H.emu_solve(variant, batch, W[variant])
    ref, ref0 = H.oracle_pair(variant, batch, W[variant])
    assert got.K[0] == K and H.segs_equal(got.segs[0], ref["segs"][0], K)
    assert got.status[0] == 0 and ref0["status"][0] == 0
    assert got.iters[0] == ref0["iters"][0] < 3000, (got.iters[0], ref0["iters"][0])
    assert got.verified()[0]
    if ref["polish"][0] == 2:
        assert H.close(got.ctrl[0, :12 * K], ref["ctrl"][0, :12 * K]), H.maxdiff(got.ctrl[0, :12 * K], ref["ctrl"][0, :12 * K])
    else:  # no KKT proof on the oracle's side (cub above K = 9): the emulated point must be feasible and as optimal
        obj_g, viol = H.qp_objective_and_violation(variant, batch, 0, W[variant], ref["segs"][0, :K], got.ctrl[0, :12 * K])
        obj_r, _ = H.qp_objective_and_violation(variant, batch, 0, W[variant], ref["segs"][0, :K], ref["ctrl"][0, :12 * K])
        assert viol <= 1e-9 and obj_g <= obj_r + 1e-6 * abs(obj_r), (obj_g, obj_r, viol)


@pytest.mark.parametrize("K,variant", [(26, "cub"), (32, "trp")])
def test_emu_ladder_many_segments_rows_bit_exact(K, variant):
    """K = 26 and 32 (the lane kernel's widest shapes), corridor-deep: segments and every (l, u) row of the QP bit for bit
    against the oracle's own assembly."""
    batch = segment_ladder(K, 2).slice(1, 2)
    got = H.emu_solve(variant, batch, W[variant], want_lu=True, max_iter=25, polish=0)
    ref = po.solve_batch(variant, batch, W[variant], mode=0, k_max=32, nthreads=0)
    assert got.K[0] == ref["K"][0] == K and H.segs_equal(got.segs[0], ref["segs"][0], K)
    sc = Scenario(batch.n_knots, batch.delta_t, batch.init[0, :3], batch.init[0, 3:], batch.scalars[0], batch.s_bounds[0],
                  batch.l_bounds[0], batch.ds_bounds[0], batch.dl_bounds[0], batch.s_ref[0], batch.l_ref[0])
    qp = po.formulate(variant, sc, W[variant], ref["segs"][0, :K])
    l, u = H.lu_to_qp_rows(got.lu[0], K)
    assert np.array_equal(l, qp["l"]) and np.array_equal(u, qp["u"])


# ---------------------------------------------------------------- corridor stage: regions with many slope breaks
N_RB = 131


def region_break_batch(n_breaks):
    """Two scenarios (base and perturbed) whose reference runs through region 0 (the ladder at N = 131: 13 segments) and never
    enters region 1 (lateral [10, 12]); region 1's upper s-bound has `n_breaks` slope breaks two knots apart, i.e.
    n_breaks + 1 cubes before the split, 0.2 s each but the last."""
    br = [2 * (m + 1) for m in range(n_breaks)]
    return wiggle_batch(N_RB, [], 2, regions=[(slope_wiggle(N_RB, br), 10.0, 12.0)])


def reference_region_break_batch(n_breaks, first, last):
    """Two scenarios whose region 0 carries `n_breaks` slope breaks two knots apart (knots 2 .. 2 n_breaks: pre-split cube j
    spans knots [2 j, 2 j + 2], the last one [2 n_breaks, 130]) and whose reference runs through region 0 at knots
    [first, last) and through region 1 (lateral [10, 12], no break) elsewhere: the corridor holds the cubes of region 0 that
    the reference visits, split where longer than 1 s, and region 1's one-second pieces."""
    br = [2 * (m + 1) for m in range(n_breaks)]
    b = wiggle_batch(N_RB, br, 2, regions=[(slope_wiggle(N_RB, []), 10.0, 12.0)])
    b.l_ref[:, :first] = 11.0
    b.l_ref[:, last:] = 11.0
    return b


def assert_corridor_equal_oracle(got, ref):
    assert np.array_equal(got.K, ref["K"]), (got.K, ref["K"])
    for b in range(len(got.K)):
        if ref["status"][b] in (2, 5):
            assert got.status[b] == ref["status"][b], (b, got.status[b], ref["status"][b])
        else:
            assert got.status[b] not in (2, 5)
            assert H.segs_equal(got.segs[b], ref["segs"][b], int(got.K[b])), b


# (n_breaks, the oracle's K, status) of region_break_batch: 64 breaks are 65 cubes before the split, one more than a region holds
REGION_BREAKS = [(0, 13, 0), (31, 13, 0), (32, 13, 0), (33, 13, 0), (47, 13, 0), (62, 13, 0), (63, 13, 0), (64, 0, 5)]


@pytest.mark.parametrize("variant", H.VARIANTS)
def test_emu_region_with_many_slope_breaks(variant):
    """A region the reference never enters may hold up to 63 slope breaks (64 cubes before the split, the oracle's cap) without
    changing the corridor of the scenario; 64 (the most that fit in N = 131 knots) make the scenario fail with "too many
    segments" on both sides."""
    for n, K, status in REGION_BREAKS:
        batch = region_break_batch(n)
        ref = po.solve_batch(variant, batch, W[variant], mode=0, nthreads=0)
        assert np.all(ref["K"] == K) and np.all((ref["status"] == 5) == (status == 5)), (n, ref["K"], ref["status"])
        got = H.emu_solve(variant, batch, W[variant], max_iter=25, polish=0)
        assert_corridor_equal_oracle(got, ref)


# (n_breaks, first, last) of reference_region_break_batch.  The reference either leaves region 0 early (pre-split cubes 0-14
# are selected) or enters it late, so that cubes 32-63 -- the second register slot of corridor_generate_region -- are selected,
# among them a cube longer than 1 s that the split cuts into pieces (n_breaks = 33, 40, 47: the last cube is 6.4, 5.0, 3.6 s).
REF_REGION_BREAKS = [(32, 0, 30), (40, 0, 30), (33, 60, N_RB), (40, 60, N_RB), (47, 70, N_RB), (63, 100, N_RB)]


def assert_reference_region_case(got, ref, n, first):
    """assert_corridor_equal_oracle, plus: a late entry selects region-0 cubes from pre-split cube 32 on (beg_t >= 64), and
    pieces of the split of the last cube when it is longer than 1 s."""
    assert np.all(ref["status"] != 5) and np.all(ref["K"] >= 16), (n, ref["K"])
    assert_corridor_equal_oracle(got, ref)
    if first == 0:
        return
    for b in range(len(got.K)):
        s = ref["segs"][b, :int(ref["K"][b])]
        reg0 = s[s["beg_l"] < 5.0]
        assert (reg0["beg_t"] >= 64).sum() >= 2, (n, b)
        if N_RB - 1 - 2 * n > 10:
            assert (reg0["beg_t"] >= 2 * n).sum() >= 2, (n, b)


@pytest.mark.parametrize("variant", H.VARIANTS)
def test_emu_reference_region_with_many_slope_breaks(variant):
    """The region that holds the reference has 32 .. 63 slope breaks: the same corridor as the oracle, bit for bit, also where
    the selected cubes come from the second half of the region's pre-split cubes."""
    for n, first, last in REF_REGION_BREAKS:
        batch = reference_region_break_batch(n, first, last)
        ref = po.solve_batch(variant, batch, W[variant], mode=0, k_max=32, nthreads=0)
        got = H.emu_solve(variant, batch, W[variant], max_iter=25, polish=0)
        assert_reference_region_case(got, ref, n, first)
