"""Synthetic scenario batches of the shapes named in BASELINE.json (SURVEY.md section 8d).

* ``load_fixture``            the reference's input fixtures (src/c*.txt, bounds.txt), shipped parsed
                              in ``spectral_b200/data/fixtures.npz`` (written by oracle/gen_golden.py).
* ``perturbed_obstacles``     config 2 / 5: B obstacle-perturbed copies of one base scenario: per region
                              the obstacle ramp of the s-bounds is shifted by dk in {-5..5} knots and
                              ds = round(U(-2,2), 2) m, the lane edges by round(U(-0.3,0.3), 2) m.
* ``mixed_batch``             config 4: base drawn from the feasible fixtures, extra breakpoints.
Random numbers come from a counter-based generator (Philox) keyed by the seed, drawn in scenario
order, so scenario b is the same whatever the batch size; scenario 0 is the unperturbed base.
"""
from __future__ import annotations

import os
from typing import Sequence

import numpy as np

from .wire import Scenario, ScenarioBatch

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "fixtures.npz")
FIXTURES = ("c1", "c2", "c3", "c4", "c4_2", "c5", "c6", "c7", "c7_7", "c7_10", "c_road_s1", "c_road_s1_2",
            "c_road_s1_3", "bounds")
FEASIBLE = ("c1", "c2", "c3", "c4", "c4_2", "c5", "bounds")

# src/weights.txt and the golden recipes (SURVEY.md Appendix D.2)
WEIGHTS_FILE = (35.73, 41.61, 25.57, 41.59, 0.12, 10.04, 0.71, 14.3, 7.27, 32.13)
GOLDEN_W_TRP = (35.73, 41.61, 25.57, 41.59, 0.12, 10.04, 0.0, 0.0, 7.27, 32.13)
GOLDEN_W_CUB = (35.73, 41.61, 25.57, 41.59, 0.12, 10.04, 0.0, 0.0, 7.27, 0.0)

_cache = None


def load_fixture(name: str) -> Scenario:
    global _cache
    if _cache is None:
        _cache = np.load(_DATA)
    z = _cache
    g = lambda k: z["%s/%s" % (name, k)]  # noqa: E731
    init = g("init")
    return Scenario(int(g("n_knots")), float(g("delta_t")), init[:3].copy(), init[3:].copy(), g("scalars").copy(),
                    g("s_bounds").copy(), g("l_bounds").copy(), g("ds_bounds").copy(), g("dl_bounds").copy(),
                    g("s_ref").copy(), g("l_ref").copy())


def _mode(col: np.ndarray) -> float:
    vals, counts = np.unique(col, return_counts=True)
    return float(vals[np.argmax(counts)])


def perturbed_obstacles(base: Scenario, B: int, seed: int = 20230531, first: int = 0, s_max: float = 50.0) -> ScenarioBatch:
    """Scenarios [first, first+B) of the config-2 family built on `base` (vectorised over scenarios)."""
    N, R = base.n_knots, base.n_regions
    rng = np.random.Generator(np.random.Philox(key=seed))
    if first:
        rng.bit_generator.advance(first * R)  # one Philox block (4 draws) per (scenario, region)
    u = rng.random((B, R, 4))
    dk = np.floor(u[..., 0] * 11).astype(np.int64) - 5
    ds = np.round(u[..., 1] * 4.0 - 2.0, 2)
    dl_lo = np.round(u[..., 2] * 0.6 - 0.3, 2)
    dl_hi = np.round(u[..., 3] * 0.6 - 0.3, 2)
    if first == 0:
        dk[0], ds[0], dl_lo[0], dl_hi[0] = 0, 0.0, 0.0, 0.0
    return _shift_obstacles(base, dk, ds, dl_lo, dl_hi, s_max)


def _shift_obstacles(base: Scenario, dk, ds, dl_lo, dl_hi, s_max: float = 50.0) -> ScenarioBatch:
    """B copies of `base` whose obstacle ramps (the s-bound entries that differ from the region's free-road value) are
    moved by dk[B, R] knots and ds[B, R] metres and whose lane edges are moved by dl_lo / dl_hi[B, R] metres."""
    N, R = base.n_knots, base.n_regions
    B = dk.shape[0]
    idx = np.arange(N)[None, None, :] - dk[..., None]          # source knot of each destination knot
    valid = (idx >= 0) & (idx < N)
    src = np.clip(idx, 0, N - 1)
    s_out = np.empty((B, R, N, 2))
    for side in (0, 1):
        col = base.s_bounds[:, :, side]                          # [R, N]
        default = np.array([_mode(col[r]) for r in range(R)])    # the region's free-road value (0 or 50)
        is_obst = col != default[:, None]
        r_idx = np.arange(R)[None, :, None]
        moved = np.clip(np.round(col[r_idx, src] + ds[..., None], 2), 0.0, s_max)
        take = valid & is_obst[r_idx, src]
        s_out[..., side] = np.where(take, moved, default[None, :, None])
    s_out[..., 1] = np.maximum(s_out[..., 1], s_out[..., 0])     # keep lo <= hi
    l_out = np.broadcast_to(base.l_bounds, (B, R, N, 2)).copy()
    l_out[..., 0] = np.round(l_out[..., 0] + dl_lo[..., None], 2)
    l_out[..., 1] = np.round(l_out[..., 1] + dl_hi[..., None], 2)
    l_out[..., 1] = np.maximum(l_out[..., 1], l_out[..., 0])
    rep = lambda a: np.ascontiguousarray(np.broadcast_to(a, (B,) + a.shape))  # noqa: E731
    return ScenarioBatch(N, R, base.delta_t, np.ascontiguousarray(s_out), np.ascontiguousarray(l_out),
                         rep(base.ds_bounds), rep(base.dl_bounds), rep(base.s_ref), rep(base.l_ref),
                         rep(np.concatenate([base.init_s, base.init_l])), rep(base.scalars))


def config3(B: int = 65536, groups: int = 8, first: int = 0, seed: int = 20230601) -> ScenarioBatch:
    """BASELINE.json configs[2] (SURVEY.md 8d "Config 3"): scenario_2 (c2.txt, trapezoid-prism, N = 71, R = 1), variants
    that leave the KKT STRUCTURE (segment count, time allocation, weights) of their group unchanged -- only bounds,
    initial state and references differ -- in `groups` groups of distinct time allocations (scenario b belongs to group
    b % groups; the group moves the obstacle ramp by a fixed number of knots, which moves the corridor breaks).
    Within a group: the obstacle's s-bias is offset by round(U(-1,1), 2) m (slopes and breaks untouched), the ds / dl
    bound columns by round(U(-0.5,0.5), 2), the initial (ds, dl) by U(-0.5,0.5) and the reference lines by a constant
    round(U(-0.5,0.5), 2) m.  Scenario 0 is the unperturbed base."""
    base = load_fixture("c2")
    N, R = base.n_knots, base.n_regions
    rng = np.random.Generator(np.random.Philox(key=seed))
    if first:
        rng.bit_generator.advance(first * 2)  # two Philox blocks (8 draws) per scenario
    u = rng.random((B, 8))
    ids = first + np.arange(B)
    shifts = np.array([0] + [d for k in range(1, 33) for d in (k, -k)])[:max(1, groups)]
    dk = np.repeat(shifts[ids % max(1, groups)][:, None], R, axis=1)
    ds = np.repeat(np.round(u[:, 0] * 2.0 - 1.0, 2)[:, None], R, axis=1)
    zero = np.zeros((B, R))
    unperturbed = ids == 0
    ds[unperturbed] = 0.0
    b = _shift_obstacles(base, dk, ds, zero, zero, 50.0)
    off = lambda c: np.where(unperturbed, 0.0, np.round(u[:, c] - 0.5, 2))  # noqa: E731
    ds_b = b.ds_bounds.copy()
    ds_b[:, :, 1] = ds_b[:, :, 1] + off(1)[:, None]
    dl_b = b.dl_bounds.copy()
    dl_b[:, :, 1] = dl_b[:, :, 1] + off(2)[:, None]
    init = b.init.copy()
    init[:, 1] = np.maximum(init[:, 1] + np.where(unperturbed, 0.0, u[:, 3] - 0.5), 0.0)
    init[:, 4] = init[:, 4] + np.where(unperturbed, 0.0, 0.2 * (u[:, 4] - 0.5))
    s_ref = b.s_ref.copy()
    s_ref[:, 1:] = s_ref[:, 1:] + off(5)[:, None]   # knot 0 stays at the initial position
    l_ref = b.l_ref + 0.2 * off(6)[:, None]
    return ScenarioBatch(N, R, base.delta_t, b.s_bounds, b.l_bounds, ds_b, dl_b, s_ref, l_ref, init, b.scalars)


def config2(B: int = 1024, first: int = 0) -> ScenarioBatch:
    """BASELINE.json configs[1]: scenario_1 (c1.txt), cuboid variant, obstacle-perturbed copies."""
    return perturbed_obstacles(load_fixture("c1"), B, seed=20230531, first=first)


def with_extra_breaks(batch: ScenarioBatch, seed: int, max_breaks: int = 4) -> ScenarioBatch:
    """config 4 ingredient: random extra slope breaks (a 0.5 m step in the upper s-bound from a random
    knot on) so that the segment count K varies between scenarios."""
    rng = np.random.Generator(np.random.Philox(key=seed))
    B, R, N = batch.batch, batch.n_regions, batch.n_knots
    s = batch.s_bounds.copy()
    nb = rng.integers(0, max_breaks + 1, size=B)
    at = rng.integers(3, N - 3, size=(B, max_breaks))
    step = np.round(rng.random((B, max_breaks)) * 1.0 + 0.5, 2)
    knots = np.arange(N)[None, :]
    for j in range(max_breaks):
        on = (nb > j)[:, None] & (knots >= at[:, j:j + 1])
        s[:, 0, :, 1] = np.where(on, np.maximum(s[:, 0, :, 1] - step[:, j:j + 1], s[:, 0, :, 0]), s[:, 0, :, 1])
    return ScenarioBatch(N, R, batch.delta_t, s, batch.l_bounds, batch.ds_bounds, batch.dl_bounds, batch.s_ref,
                         batch.l_ref, batch.init, batch.scalars)


def mixed_batches(B: int, seed: int = 20230602, bases: Sequence[str] = ("c1", "c3", "bounds", "c2", "c4_2")):
    """config 4: heterogeneous corridor sequences.  Returns a list of (variant, ScenarioBatch): the C-ABI takes
    one (N, R, variant) per call, so a mixed sweep is a handful of calls on one stream."""
    out = []
    per = max(1, B // (2 * len(bases)))
    for i, name in enumerate(bases):
        for variant in ("trp", "cub"):
            b = perturbed_obstacles(load_fixture(name), per, seed=seed + 17 * i + (variant == "cub"))
            out.append((variant, with_extra_breaks(b, seed + 1000 + i)))
    return out


def zigzag_breaks(base: Scenario, B: int, seed: int = 4242, s_max: float = 100.0) -> ScenarioBatch:
    """Scenarios with MANY segments (K up to ~30, the class above the dense kernels' capacity): the config-2 perturbation of
    `base` plus a staircase in the upper s-bound of every region (a 0.3 .. 0.6 m step every p in {5 .. 9} knots), each
    step being a slope break of CorridorGeneration (solve_3d.cc:372-374)."""
    batch = perturbed_obstacles(base, B, seed=seed, s_max=s_max)
    rng = np.random.Generator(np.random.Philox(key=seed + 1))
    N = batch.n_knots
    period = rng.integers(5, 10, size=B)
    step = np.round(0.3 + 0.3 * rng.random(B), 2)
    knots = np.arange(N)[None, :]
    stair = ((knots // period[:, None]) % 2) * step[:, None]          # [B, N]
    s = batch.s_bounds.copy()
    s[:, :, :, 1] = np.maximum(s[:, :, :, 1] - stair[:, None, :], s[:, :, :, 0])
    return ScenarioBatch(N, batch.n_regions, batch.delta_t, s, batch.l_bounds, batch.ds_bounds, batch.dl_bounds, batch.s_ref,
                         batch.l_ref, batch.init, batch.scalars)


def slope_wiggle(n_knots: int, breaks: Sequence[int], delta_t: float = 0.1) -> np.ndarray:
    """Upper s-bound over `n_knots` knots: 200 m plus a ramp whose slope toggles between 0 and 0.5 m/s at each knot of
    `breaks` (the backward slope of knot i is the new one from i in `breaks` on).  Each toggle differs from the current
    cube's slope by more than CorridorGeneration's 0.2 threshold (solve_3d.cc:372), so each one starts a new pre-split cube
    as long as consecutive breaks are at least two knots apart and lie in [2, n_knots - 2]."""
    slope = np.zeros(n_knots)
    cur = 0.0
    at = set(int(i) for i in breaks)
    for i in range(1, n_knots):
        if i in at:
            cur = 0.5 - cur
        slope[i] = cur
    return 200.0 + np.cumsum(slope * delta_t)


def ladder_shape(K: int):
    """(n_knots, break knots) of `segment_ladder` for K segments (see there)."""
    if K < 1:
        raise ValueError("K >= 1")
    if K <= 25:
        return 10 * K + 1, []
    return 256, [15 * (m + 1) for m in range(2 * (K - 26))]


def wiggle_batch(n_knots: int, breaks, B: int, seed: int = 20231021, regions=None) -> ScenarioBatch:
    """B scenarios on a free road (one region, delta_t = 0.1 s, lateral bounds [1, 4], c2's derivative bounds and scalars)
    whose upper s-bound is `slope_wiggle(n_knots, breaks)`; `breaks` is one list for all scenarios or one list per scenario.
    The reference line is s_ref = 5 m/s * t, l_ref = 2 m, from the initial state (0, 5, 0, 2, 0, 0).  Per scenario, only
    values that cannot move a slope break vary (scenario 0 is the unperturbed base): s_ref (after knot 0) by an offset in
    [0, 1) m, l_ref by [-0.5, 0.5) m, the initial ds by [-0.5, 0.5) m/s and dl by [0, 0.1) m/s (the
    dl bounds are [0, 2.5]), the lateral bounds by [-0.3, 0.3) m each.  `regions`: extra regions appended after region 0, as a list of (s_upper [N], l_lo, l_hi)."""
    c2 = load_fixture("c2")
    N, d = n_knots, 0.1
    per = [list(breaks)] * B if len(breaks) == 0 or np.ndim(breaks[0]) == 0 else [list(b) for b in breaks]
    if len(per) != B:
        raise ValueError("one break list per scenario")
    extra = list(regions or [])
    R = 1 + len(extra)
    rng = np.random.Generator(np.random.Philox(key=seed))
    u = rng.random((B, 6))
    u[0] = 0.5
    u[0, 0] = u[0, 3] = 0.0
    sb = np.zeros((B, R, N, 2))
    lb = np.zeros((B, R, N, 2))
    for b in range(B):
        sb[b, 0, :, 1] = slope_wiggle(N, per[b], d)
    lb[:, 0, :, 0] = (1.0 + np.round(0.6 * u[:, 4] - 0.3, 2))[:, None]
    lb[:, 0, :, 1] = (4.0 + np.round(0.6 * u[:, 5] - 0.3, 2))[:, None]
    for r, (s_up, l_lo, l_hi) in enumerate(extra, start=1):
        sb[:, r, :, 1] = np.asarray(s_up)[None, :]
        lb[:, r, :, 0], lb[:, r, :, 1] = l_lo, l_hi
    t = np.arange(N) * d
    s_ref = np.tile(5.0 * t, (B, 1))
    s_ref[:, 1:] += np.round(u[:, 0], 2)[:, None]
    l_ref = np.tile(2.0 + np.round(u[:, 1] - 0.5, 2)[:, None], (1, N))
    init = np.tile(np.array([0.0, 5.0, 0.0, 2.0, 0.0, 0.0]), (B, 1))
    init[:, 1] += u[:, 2] - 0.5
    init[:, 4] += 0.1 * u[:, 3]
    rep = lambda a: np.ascontiguousarray(np.broadcast_to(a, (B,) + a.shape))  # noqa: E731
    return ScenarioBatch(N, R, d, sb, lb, rep(np.tile([0.0, 10.0], (N, 1))), rep(np.tile([0.0, 2.5], (N, 1))), s_ref, l_ref,
                         init, rep(c2.scalars))


def segment_ladder(K: int, B: int, seed: int = 20231021) -> ScenarioBatch:
    """B scenarios that all have exactly K corridor segments, for every K from 1 to 34 (K <= 32 solvable with k_max = 32,
    K >= 33 reported as too many segments), in both variants; they share one KKT structure (same K, same segment
    durations) and differ in values only (see `wiggle_batch`).
      K <= 25:  N = 10 K + 1 knots and no slope break: one pre-split cube of K seconds, split into K one-second segments.
      K >= 26:  N = 256 (without breaks: 25 one-second segments and a 0.5 s one) and 2 (K - 26) slope breaks at knots 15,
                30, 45, ...: each pair of breaks cuts 3 s of road into two 1.5 s cubes, split into 1.0 + 0.5 s each, i.e.
                four segments where there were three.
    Segments are never shorter than 0.5 s: closely spaced breaks give ill-conditioned QPs whose solved / failed class the
    reference does not pin (helpers.decided_classes)."""
    N, breaks = ladder_shape(K)
    return wiggle_batch(N, breaks, B, seed=seed + K)


def random_obstacles(B: int, max_obs: int = 3, seed: int = 20230606):
    """Obstacle sets for the upstream bound generator (spectral_bounds_device): [B, max_obs, 6] = (s, l, t0, vel_s, vel_l,
    horizon) and n_obs [B], with the value ranges of the reference's two-car scene (src/cart_frenet.py:1536-1546): lateral
    positions on a 0.25 m grid so that lane edges coincide now and then, 60 % of the cars present from t = 0 (they bound s from
    above), the others entering later (they bound s from below).  Scenarios whose cars tie in their smallest lateral edge are
    re-drawn: the reference orders such cars by object hash (not specified)."""
    rng = np.random.Generator(np.random.Philox(key=seed))
    obs = np.zeros((B, max_obs, 6))
    n_obs = np.zeros(B, np.int32)
    w_safe = 2 / 3 + 2 / 3
    for b in range(B):
        while True:
            n = int(rng.integers(1, max_obs + 1))
            o = np.zeros((max_obs, 6))
            o[:n, 0] = np.round(rng.uniform(2.0, 35.0, n), 1)
            o[:n, 1] = rng.integers(-4, 25, n) * 0.25
            o[:n, 2] = np.where(rng.random(n) < 0.6, 0.0, np.round(rng.uniform(0.5, 3.0, n), 1))
            o[:n, 3] = np.round(rng.uniform(1.0, 8.0, n), 1)
            o[:n, 4] = rng.choice([0.0, 0.0, 0.25, -0.25, 0.5], n)
            o[:n, 5] = rng.choice([3.0, 4.0, 5.0], n)
            fl = o[:n, 1] + o[:n, 4] * o[:n, 5]
            lo = np.where(o[:n, 4] >= 0, o[:n, 1] - w_safe, fl - w_safe)
            if len(set(lo.tolist())) == n:
                break
        obs[b], n_obs[b] = o, n
    return obs, n_obs
