"""GPU tests (run with `-m gpu`): every segment count K = 1 .. 34 and every solver class of the QP stage against the CPU oracle,
on batches of exactly controlled K (scenarios.segment_ladder); handle capacities k_max below and above the class edges; the
shared-KKT tiles at every K <= 8 and every tile occupancy; all five classes in one call; regions with many slope breaks.

Solver classes (finalize.cuh lane_class): K <= 8 k_qpa<8> (or the shared-KKT tiles) | 9-10 k_qpa<10> | 11-12 k_qpd<12> |
13-16 k_qpd<16> | 17-32 k_qp<32,2>."""
import numpy as np
import pytest

import helpers as H
import pyoracle as po
from spectral_b200 import api
from spectral_b200.scenarios import GOLDEN_W_CUB, WEIGHTS_FILE, segment_ladder, wiggle_batch
from spectral_b200.wire import ScenarioBatch
from test_segment_counts_emu import (REF_REGION_BREAKS, REGION_BREAKS, assert_corridor_equal_oracle, assert_reference_region_case,
                                     reference_region_break_batch, region_break_batch)

pytestmark = pytest.mark.gpu

W = {"trp": WEIGHTS_FILE, "cub": GOLDEN_W_CUB}
B_LADDER = 8
MIX_B = 8192


@pytest.fixture(scope="module")
def planner():
    p = api.SpectralPlanner(device=0, max_batch=MIX_B, n_max=256, r_max=2, k_max=32)
    yield p
    p.close()


def _subset(batch, idx):
    idx = np.asarray(idx)
    return ScenarioBatch(batch.n_knots, batch.n_regions, batch.delta_t, *[x[idx] for x in batch.arrays()])


def _assert_same(a, b, label, rows=None):
    """Every output of BatchResult a equals b's (rows `rows` of b) bit for bit, the K-dependent ones up to each scenario's K."""
    rows = np.arange(len(b.K)) if rows is None else np.asarray(rows)
    for f in ("K", "status", "iters", "flags", "npts", "obj", "a_cost"):
        assert np.array_equal(getattr(a, f), getattr(b, f)[rows]), (label, f)
    for i, r in enumerate(rows):
        K = int(a.K[i]) if a.status[i] != api.FAIL_TOO_MANY else 0
        assert a.segs[i, :K].tobytes() == b.segs[r, :K].tobytes(), (label, i)
        assert np.array_equal(a.ctrl[i, :12 * K], b.ctrl[r, :12 * K]), (label, i)
        if a.samples is not None:
            assert np.array_equal(a.samples[i], b.samples[r]), (label, i)


# ---------------------------------------------------------------- every K from 1 to 32 vs the oracle
LADDER = {}  # (variant, K) -> (batch, got, ref, ref0): reused by the capacity test


def _ladder(planner, variant, K):
    if (variant, K) not in LADDER:
        batch = segment_ladder(K, B_LADDER)
        got = planner.solve(variant, batch, W[variant], samples_cap=256)
        ref, ref0 = H.oracle_pair(variant, batch, W[variant])
        LADDER[(variant, K)] = (batch, got, ref, ref0)
    return LADDER[(variant, K)]


@pytest.mark.parametrize("variant", H.VARIANTS)
def test_every_segment_count_vs_oracle(planner, variant):
    """K = 1 .. 32, eight scenarios each: the parity bars of the suite, and at every K at least 6 of 8 distinct scenarios (2 of
    8 at K >= 29, where the reference's own run ends near max_iter) compared numerically, by KKT-verified optimum, by ADMM
    iterate or both; the samples equal the oracle's wherever both hold a verified optimum."""
    table = []
    for K in range(1, 33):
        batch, got, ref, ref0 = _ladder(planner, variant, K)
        got0 = planner.solve(variant, batch, W[variant], options=api.default_options(polish=0))
        assert np.all(got.K == K), (K, got.K)
        both = H.assert_batch_parity(got, ref, "ladder/%s/K%d" % (variant, K), ref0=ref0, batch=batch, variant=variant,
                                     weights=W[variant], got0=got0)
        st = H.PARITY_LOG[-1]
        table.append((K, st["decided"], st.get("compared_verified", 0), st.get("compared_iterate", 0), st["compared_any"]))
        assert st["compared_any"] >= (6 if K <= 28 else 2), (K, st)
        for b in np.nonzero(both)[0]:
            if not H.close(got.ctrl[b, :12 * K], ref["ctrl"][b, :12 * K]):
                continue  # two optima apart along a flat direction of P, accepted by assert_batch_parity: their samples differ too
            n = int(got.npts[b])
            assert n == batch.n_knots == ref["npts"][b]
            assert H.close(got.samples[b, :n], ref["samples"][b, :n], rtol=1e-5, atol=2e-6), (K, b)
    print("ladder %s (K, decided, compared verified, compared iterate, compared either way): %s" % (variant, table))


@pytest.mark.parametrize("variant", H.VARIANTS)
def test_too_many_segments_reports_the_true_count(planner, variant):
    for K in (33, 34):
        batch = segment_ladder(K, B_LADDER)
        got = planner.solve(variant, batch, W[variant])
        ref = po.solve_batch(variant, batch, W[variant], mode=0, nthreads=0)
        assert np.all(ref["K"] == K) and np.all(ref["status"] == api.FAIL_TOO_MANY)
        assert np.all(got.K == K) and np.all(got.status == api.FAIL_TOO_MANY)
        assert np.all(got.a_cost == api.FAIL_COST)


# ---------------------------------------------------------------- handle capacities
CAPACITIES = (1, 7, 8, 9, 10, 11, 12, 13, 16, 17, 31, 32)
CAP_K = (1, 7, 8, 9, 10, 11, 12, 13, 16, 17, 31, 32)


def test_handle_capacity_never_changes_a_result(planner):
    """Handles with k_max in CAPACITIES (below, at and above every class edge) give every scenario with K <= k_max the result
    of the k_max = 32 handle bit for bit (the k_max strides of segs / ctrl / lu in every kernel, and the classes skipped
    because k_max rules them out), and report every other scenario as too many segments with its true K."""
    for km in CAPACITIES:
        small = api.SpectralPlanner(device=0, max_batch=B_LADDER, n_max=256, r_max=2, k_max=km)
        try:
            for i, K in enumerate(CAP_K):
                variant = H.VARIANTS[i % 2]
                batch, full, _, _ = _ladder(planner, variant, K)
                got = small.solve(variant, batch, W[variant], samples_cap=256)
                label = "k_max=%d K=%d %s" % (km, K, variant)
                if K <= km:
                    _assert_same(got, full, label)
                else:
                    assert np.all(got.K == K) and np.all(got.status == api.FAIL_TOO_MANY), label
                    assert np.all(got.a_cost == api.FAIL_COST), label
        finally:
            small.close()


# ---------------------------------------------------------------- shared-KKT tiles
GROUP_SIZES = (1, 2, 3, 5, 7, 8, 9, 16, 17)


def _grouped(K, variant):
    """One ladder batch of K segments cut into groups of GROUP_SIZES members: each group has its own weight vector, i.e. its
    own tile key, so that every tile occupancy 1 .. 8 and ragged tails (9 = 8 + 1, 17 = 2 x 8 + 1) occur."""
    B = sum(GROUP_SIZES)
    batch = segment_ladder(K, B)
    w = np.tile(np.array(W[variant], dtype=np.float64), (B, 1))
    w[:, 0] += np.repeat(np.arange(len(GROUP_SIZES)), GROUP_SIZES) * 0.5
    return batch, w


@pytest.mark.parametrize("variant", H.VARIANTS)
def test_shared_kkt_tiles_every_k_and_occupancy(planner, variant):
    """The shared-KKT path at K = 1 .. 8 with tiles of every occupancy: oracle parity at the bars of the other shared-KKT tests,
    the per-scenario path's optimum wherever both hold a KKT proof, and the same results on a k_max = 4 handle (K <= 4)."""
    shared = api.default_options(shared_kkt=1)
    tight = api.SpectralPlanner(device=0, max_batch=sum(GROUP_SIZES), n_max=256, r_max=2, k_max=4)
    try:
        for K in range(1, 9):
            batch, w = _grouped(K, variant)
            got = planner.solve(variant, batch, w, options=shared)
            ref, ref0 = H.oracle_pair(variant, batch, w)
            H.assert_batch_parity(got, ref, "shared/%s/K%d" % (variant, K), need_verified_frac=0.5, ref0=ref0, batch=batch,
                                  variant=variant, weights=w, min_iters_equal_frac=0.0, max_undecided_mismatch_frac=0.05)
            per = planner.solve(variant, batch, w)
            both = got.verified() & per.verified()
            assert both.sum() >= len(both) // 2, (K, both.sum())
            for b in np.nonzero(both)[0]:
                assert H.close(got.ctrl[b, :12 * K], per.ctrl[b, :12 * K]), (K, b, H.maxdiff(got.ctrl[b, :12 * K], per.ctrl[b, :12 * K]))
            if K <= 4:
                _assert_same(tight.solve(variant, batch, w, options=shared), got, "shared k_max=4 K=%d" % K)
    finally:
        tight.close()


# ---------------------------------------------------------------- all five classes in one call
def _five_class_batch():
    """8 192 scenarios at N = 81 with 0 .. 22 slope breaks each (knots drawn from 2, 5, .., 77): K from 8 to about 24."""
    rng = np.random.Generator(np.random.Philox(key=99))
    slots = np.arange(2, 79, 3)
    nb = rng.integers(0, 23, size=MIX_B)
    breaks = [sorted(rng.choice(slots, int(n), replace=False).tolist()) for n in nb]
    return wiggle_batch(81, breaks, MIX_B)


def _class(K):
    return np.select([K <= 8, K <= 10, K <= 12, K <= 16, K <= 32], [0, 1, 2, 3, 4], 5)


def test_all_classes_in_one_call_are_independent(planner):
    """One call holding all five solver classes, each with more scenarios than two per SM (every persistent kernel wraps its
    work queue): each class solved as its own batch gives the same outputs bit for bit, and so does a random permutation of
    the whole batch (classified out of order, the class streams running concurrently)."""
    batch = _five_class_batch()
    full = planner.solve("trp", batch, WEIGHTS_FILE)
    cls = _class(full.K)
    counts = np.bincount(cls, minlength=6)
    assert np.all(counts[:5] > 2 * 148), counts
    assert np.all(full.status != api.FAIL_TOO_MANY)
    for c in range(5):
        idx = np.nonzero(cls == c)[0]
        for lo in range(0, len(idx), 4096):
            part = idx[lo:lo + 4096]
            _assert_same(planner.solve("trp", _subset(batch, part), WEIGHTS_FILE), full, "class %d" % c, rows=part)
    perm = np.random.default_rng(3).permutation(MIX_B)
    _assert_same(planner.solve("trp", _subset(batch, perm), WEIGHTS_FILE), full, "permuted", rows=perm)


# ---------------------------------------------------------------- corridor stage: regions with many slope breaks
@pytest.mark.parametrize("variant", H.VARIANTS)
def test_region_with_many_slope_breaks(planner, variant):
    """A region the reference never enters with 0 .. 64 slope breaks, and a region holding the reference with 32 .. 63, entered
    late enough that cubes 32-63 of it are selected: the oracle's corridor bit for bit and its status (too many segments at 64
    breaks)."""
    for n, K, status in REGION_BREAKS:
        batch = region_break_batch(n)
        ref = po.solve_batch(variant, batch, W[variant], mode=0, nthreads=0)
        got = planner.solve(variant, batch, W[variant])
        assert np.all(got.K == K) and np.all((got.status == api.FAIL_TOO_MANY) == (status == api.FAIL_TOO_MANY)), (n, got.K, got.status)
        assert_corridor_equal_oracle(got, ref)
    for n, first, last in REF_REGION_BREAKS:
        batch = reference_region_break_batch(n, first, last)
        ref = po.solve_batch(variant, batch, W[variant], mode=0, nthreads=0)
        assert_reference_region_case(planner.solve(variant, batch, W[variant]), ref, n, first)
