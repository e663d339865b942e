"""BASELINE.json configs[4] (SURVEY.md 8d "Config 5"): the 1 M-scenario sweep, sharded over the GPUs of one box.

Scenarios come from the config-4 generator (mixed trapezoid-prism + cuboid corridors, K in [4, 14]; seed 20230603):
five base fixtures x two variants = ten families of obstacle-perturbed scenarios with extra slope breaks, dealt
round-robin in chunks of 8192: global scenario index = chunk * 8192 + position.  Rank r takes a CONTIGUOUS range of the
global index (SURVEY.md 8e), i.e. of chunks; no data-path collective.  The sweep ends with the ONE exchange of the path: the
best trajectory (arg-min of a_cost, ties -> lowest global index) through the C-ABI's spectral_sweep_argmin (top-k with
k = 1: NCCL all-gather of the 16-byte records, then an all-reduce of the winner's payload from its owner).  The winner
does not depend on the number of ranks.
"""
from __future__ import annotations

import numpy as np

from . import api
from .scenarios import WEIGHTS_FILE, load_fixture, perturbed_obstacles, with_extra_breaks
from .sweep import shard_range

BASES = ("c1", "c3", "bounds", "c2", "c4_2")
SEED = 20230603


CHUNK = 8192   # scenarios per generated chunk and per solve call


def chunk_spec(g: int):
    """Global chunk g -> (variant, base name, base index, first scenario of the chunk within its family).  Chunks are dealt
    round-robin over the ten (base, variant) families so that any contiguous range of chunks is a fair mix of them."""
    nfam = 2 * len(BASES)
    fam, c = g % nfam, g // nfam
    i = fam // 2
    variant = "trp" if fam % 2 == 0 else "cub"
    return variant, BASES[i], i, c * CHUNK


def make_chunk(g: int):
    """The CHUNK scenarios of global chunk g: the config-4 family (scenarios.mixed_batches) of (base, variant), obstacle
    perturbation at family position c * CHUNK .., extra slope breaks drawn from a seed that includes the chunk."""
    variant, name, i, lo = chunk_spec(g)
    b = perturbed_obstacles(load_fixture(name), CHUNK, seed=SEED + 17 * i + (variant == "cub"), first=lo)
    return variant, with_extra_breaks(b, SEED + 1000 + 7919 * g)


def upload_shard(total: int, rank: int, world: int, device):
    """Generates this rank's contiguous range of global chunks and makes it resident in HBM."""
    import torch
    nchunks = total // CHUNK
    g_lo, g_hi = shard_range(nchunks, rank, world)
    names = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")
    w_dev = torch.tensor(WEIGHTS_FILE, dtype=torch.float64, device=device)
    resident = []
    for g in range(g_lo, g_hi):
        variant, b = make_chunk(g)
        inp = {k: torch.from_numpy(np.ascontiguousarray(a)).to(device) for k, a in zip(names, b.arrays())}
        inp["weights"] = w_dev
        resident.append((variant, b.n_knots, b.n_regions, b.delta_t, inp))
    return dict(g_lo=g_lo, g_hi=g_hi, chunks=resident)


def run_sweep(planner: "api.SpectralPlanner", shard: dict, outs: dict, options=None):
    """One pass over this rank's resident shard (one solve call per chunk into slices of `outs`), then the ONE exchange of
    the path: spectral_sweep_argmin over the whole shard (collective).  Returns the winner (same on every rank)."""
    n = 0
    for variant, N, R, delta, inp in shard["chunks"]:
        view = {k: t[n:n + CHUNK] for k, t in outs.items()}
        planner.solve_device(variant, N, R, delta, inp, view, options=options)
        n += CHUNK
    if n == 0:   # a rank without work still takes part in the collective
        outs["a_cost"][:1].fill_(api.FAIL_COST)
        return planner.sweep_argmin(outs, shard["g_lo"] * CHUNK, B=1)
    return planner.sweep_argmin(outs, shard["g_lo"] * CHUNK, B=n)
