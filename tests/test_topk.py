"""Top-k selection (spectral_topk_device / spectral_sweep_topk, topk.cuh) on the GPU: exact against a NumPy reference of the
contract in include/spectral.h -- ascending (cost, global index), -0.0 == +0.0, NaN last, stored cost bits returned -- on
adversarial cost arrays, on real solves and across two NCCL ranks."""
import ctypes
import multiprocessing as mp
import queue

import numpy as np
import pytest

from spectral_b200 import api

pytestmark = pytest.mark.gpu

BIG_OFFSET = (1 << 32) + 12345
KS = (1, 2, 17, 256, 1024)
NAN_NEG = np.array([0xFFF8000000000001], dtype=np.uint64).view(np.float64)[0]   # a negative NaN with a payload


@pytest.fixture(scope="module")
def planner():
    p = api.SpectralPlanner(device=0, max_batch=1024, n_max=128, r_max=8, k_max=32)
    yield p
    p.close()


def canon_key(c):
    """The order-preserving 64-bit image of include/spectral.h's order: -0.0 -> +0.0, every NaN above +inf."""
    c = np.asarray(c, dtype=np.float64)
    u = c.view(np.uint64).copy()
    u[c == 0.0] = 0
    key = np.where((u >> np.uint64(63)) == 1, ~u, u | np.uint64(1 << 63))
    key[np.isnan(c)] = np.uint64(0xFFFFFFFFFFFFFFFF)
    return key


def ref_order(c):
    """Positions of c sorted by (canonical key, position)."""
    return np.lexsort((np.arange(len(c)), canon_key(c)))


def ref_topk(c, k, offset, order=None):
    order = ref_order(c) if order is None else order
    sel = order[:k]
    cost = np.full(k, np.inf)
    idx = np.full(k, -1, dtype=np.int64)
    cost[:len(sel)] = c[sel]
    idx[:len(sel)] = offset + sel
    return cost, idx


def adversarial(B, seed):
    """Costs rounded to 0.1 (many exact ties), 30 % failure sentinels, negative costs, +-0.0, +-inf, NaNs (both signs,
    payloads), subnormals and values next to 1e300."""
    rng = np.random.default_rng(seed)
    c = np.round(rng.uniform(-3.0, 40.0, B), 1)
    u = rng.random(B)
    c[u < 0.30] = api.FAIL_COST
    specials = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, NAN_NEG, 5e-324, -5e-324, 2.2250738585072e-308, -1.0e300,
                         1.0e300, np.nextafter(1.0e300, 0.0), -0.0, 0.0])
    m = (u >= 0.30) & (u < 0.36)
    c[m] = specials[rng.integers(0, len(specials), int(m.sum()))]
    if B >= 3:
        c[rng.integers(0, B, 3)] = -0.0
    return c


def _run(planner, c, k, offset, stream=None):
    import torch
    t = torch.from_numpy(c).cuda()
    cost, idx = planner.topk_device(t, k, index_offset=offset, stream=stream)
    torch.cuda.synchronize()
    return cost.cpu().numpy(), idx.cpu().numpy()


def _assert_same(got, want, label):
    gc, gi = got
    wc, wi = want
    assert np.array_equal(gi, wi), (label, np.nonzero(gi != wi)[0][:10])
    assert np.array_equal(gc.view(np.int64), wc.view(np.int64)), (label, np.nonzero(gc.view(np.int64) != wc.view(np.int64))[0][:10])


# ---------------------------------------------------------------- 1 + 3: exact vs NumPy, k = 1 vs argmin_device
@pytest.mark.parametrize("B,offset", [(1, 0), (31, BIG_OFFSET), (1000, 7), (65536, 0), (1048583, BIG_OFFSET)])
def test_topk_exact_vs_numpy_and_k1_equals_argmin(planner, B, offset):
    import torch
    c = adversarial(B, seed=B)
    order = ref_order(c)
    for k in KS:
        _assert_same(_run(planner, c, k, offset), ref_topk(c, k, offset, order), (B, k))
    # k = 1 against k_argmin wherever some cost is below its start value 1e300
    for variant in (c, np.where(np.isnan(c), 1.0, c), -np.abs(c)):
        if not (variant < 1e300).any():
            continue
        variant = np.ascontiguousarray(variant)
        t = torch.from_numpy(variant).cuda()
        bc = torch.zeros(1, dtype=torch.float64, device="cuda")
        bi = torch.zeros(1, dtype=torch.int64, device="cuda")
        planner.argmin_device(t, offset, bc, bi)
        tc, ti = planner.topk_device(t, 1, index_offset=offset)
        torch.cuda.synchronize()
        assert int(ti.item()) == int(bi.item())
        assert tc.cpu().numpy().view(np.int64)[0] == bc.cpu().numpy().view(np.int64)[0]


def test_topk_special_values_and_short_arrays(planner):
    """Exactly the ordering rules of the contract on a hand-written array, and k > B padding."""
    c = np.array([np.nan, 1.0, -0.0, np.inf, 0.0, -np.inf, NAN_NEG, api.FAIL_COST, -0.0, 5e-324, -5e-324])
    got = _run(planner, c, 16, 100)
    want_idx = 100 + np.array([5, 10, 2, 4, 8, 9, 1, 7, 3, 0, 6] + [-101] * 5)
    assert np.array_equal(got[1], want_idx), got[1]
    assert np.array_equal(got[0][:11].view(np.int64), c[want_idx[:11] - 100].view(np.int64))
    assert np.all(got[0][11:] == np.inf)


# ---------------------------------------------------------------- 2: ties across the threshold
def test_topk_ties_across_the_threshold(planner):
    rng = np.random.default_rng(5)
    B = 1 << 20
    c = np.round(rng.uniform(1.0, 100.0, B), 1)
    pos = np.sort(rng.choice(B, 5000, replace=False))
    c[pos] = 0.5
    cost, idx = _run(planner, c, 100, 0)
    assert np.array_equal(idx, pos[:100]) and np.all(cost == 0.5)
    # threshold at the failure sentinel: only 10 solved scenarios
    c = np.full(B, api.FAIL_COST)
    solved = rng.choice(B, 10, replace=False)
    c[solved] = rng.uniform(1.0, 2.0, 10)
    got = _run(planner, c, 100, 3)
    _assert_same(got, ref_topk(c, 100, 3), "sentinel")
    assert np.array_equal(np.sort(got[1][:10] - 3), np.sort(solved))
    fails = np.setdiff1d(np.arange(B), solved)[:90]
    assert np.array_equal(got[1][10:] - 3, fails)


# ---------------------------------------------------------------- 4: determinism across calls and streams
def test_topk_deterministic_across_calls_and_streams(planner):
    import torch
    c = adversarial(3 << 20, seed=11)
    base = torch.from_numpy(c).cuda()
    outs = []
    for _ in range(2):
        oc, oi = planner.topk_device(base, 1024)
        outs.append((oc.clone(), oi.clone()))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fresh = torch.empty_like(base)
        fresh.copy_(base)   # written by a torch kernel on the side stream, no synchronisation before the call
        oc, oi = planner.topk_device(fresh, 1024, stream=side.cuda_stream)
        outs.append((oc.clone(), oi.clone()))
    torch.cuda.synchronize()
    want = ref_topk(c, 1024, 0)
    for oc, oi in outs:
        _assert_same((oc.cpu().numpy(), oi.cpu().numpy()), want, "determinism")


# ---------------------------------------------------------------- 5: on real solves, one rank
def _merge_lists(lists, k):
    allw = [w for lst in lists for w in lst]
    key = canon_key(np.array([w["cost"] for w in allw]))
    order = np.lexsort((np.array([w["index"] for w in allw]), key))[:k]
    return [allw[j] for j in order]


def _same_winners(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x["index"] == y["index"] and x["K"] == y["K"] and x["rank"] == y["rank"]
        assert np.float64(x["cost"]).view(np.int64) == np.float64(y["cost"]).view(np.int64)
        assert x["segs"].tobytes() == y["segs"].tobytes() and x["ctrl"].tobytes() == y["ctrl"].tobytes()


def test_sweep_topk_on_real_solves(planner):
    import torch
    from spectral_b200.scenarios import GOLDEN_W_CUB, config2
    B, k = 2048, 64
    batch = config2(B)
    dev = torch.device("cuda", 0)
    pl = api.SpectralPlanner(device=0, max_batch=B, n_max=128, r_max=8, k_max=32)
    names = ("s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref", "init", "scalars")
    inputs = {n: torch.from_numpy(np.ascontiguousarray(a)).to(dev) for n, a in zip(names, batch.arrays())}
    inputs["weights"] = torch.tensor(GOLDEN_W_CUB, dtype=torch.float64, device=dev)
    outs = pl.alloc_device_outputs(B)
    pl.solve_device("cub", batch.n_knots, batch.n_regions, batch.delta_t, inputs, outs)
    wins = pl.sweep_topk(outs, 0, k)
    cost = outs["a_cost"].cpu().numpy()
    Ks = outs["K"].cpu().numpy()
    ctrl = outs["ctrl"].cpu().numpy()
    segs = outs["segs"].cpu().numpy()
    wc, wi = ref_topk(cost, k, 0)
    assert len(wins) == k
    assert np.array_equal(np.array([w["index"] for w in wins]), wi)
    assert np.array_equal(np.array([w["cost"] for w in wins]).view(np.int64), wc.view(np.int64))
    assert (cost < api.FAIL_COST).sum() > 0
    for w in wins:
        j, K = w["index"], int(Ks[w["index"]])
        assert w["rank"] == 0 and w["K"] == K
        assert w["ctrl"].tobytes() == ctrl[j, :12 * K].tobytes()
        assert w["segs"].tobytes() == segs[j].view(api.CUBE_DTYPE)[:K].tobytes()
    best = pl.sweep_argmin(outs, 0)
    assert best["index"] == wins[0]["index"] and best["cost"] == wins[0]["cost"] and best["K"] == wins[0]["K"]
    assert np.array_equal(best["ctrl"], wins[0]["ctrl"])
    # two contiguous shards, each listed on its own and merged: the same list (independent of the number of ranks)
    h = 1200
    parts = [pl.sweep_topk(outs, 0, k, B=h),
             pl.sweep_topk({n: t[h:] for n, t in outs.items()}, h, k)]
    _same_winners(_merge_lists(parts, k), wins)
    # k above the batch: min(k, B) entries; a rank without scenarios: none
    few = pl.sweep_topk({n: t[:5] for n, t in outs.items()}, 0, 16)
    assert [w["index"] for w in few] == list(ref_topk(cost[:5], 5, 0)[1])
    assert pl.sweep_topk(outs, 0, 8, B=0) == []
    pl.close()


def test_sweep_argmin_without_a_cost_below_1e300(planner):
    """Every cost NaN, every cost +inf, or a mix of NaN, +inf and values above 1e300: sweep_argmin still returns a real
    scenario, the first in top-k order, with its own K, segments and control points (zero beyond K)."""
    import torch
    total, km, off = 600, planner.k_max, 7
    _, K, segs, ctrl = _synthetic(total, km)
    mixed = np.full(total, np.nan)
    mixed[[3, 100, 450]] = [np.inf, 3e300, 2e300]
    lib = planner._lib
    for costs, j in ((np.full(total, np.nan), 0), (np.full(total, np.inf), 0), (mixed, 450)):
        outs = dict(a_cost=torch.from_numpy(costs).cuda(), K=torch.from_numpy(K).cuda(), segs=torch.from_numpy(segs).cuda(),
                    ctrl=torch.from_numpy(ctrl).cuda())
        best = planner.sweep_argmin(outs, off)
        _same_winners([best], planner.sweep_topk(outs, off, 1))
        assert best["index"] == off + j and best["rank"] == 0 and best["K"] == K[j]
        assert np.float64(best["cost"]).view(np.int64) == costs[j:j + 1].view(np.int64)[0]
        assert best["segs"].tobytes() == segs[j, :112 * K[j]].tobytes() and best["ctrl"].tobytes() == ctrl[j, :12 * K[j]].tobytes()
        out = api.SpectralOutputs()
        out.a_cost = ctypes.cast(ctypes.c_void_p(outs["a_cost"].data_ptr()), ctypes.POINTER(ctypes.c_double))
        out.K = ctypes.cast(ctypes.c_void_p(outs["K"].data_ptr()), ctypes.POINTER(ctypes.c_int))
        out.segs = outs["segs"].data_ptr()
        out.ctrl = ctypes.cast(ctypes.c_void_p(outs["ctrl"].data_ptr()), ctypes.POINTER(ctypes.c_double))
        w = api.SpectralWinner()
        assert lib.spectral_sweep_argmin(planner._h, total, ctypes.byref(out), off, ctypes.byref(w), None) == 0
        assert not any(bytes(w.segs)[112 * K[j]:]) and not any(w.ctrl[12 * K[j]:])


# ---------------------------------------------------------------- 6: two real NCCL ranks
def _synthetic(total, k_max):
    rng = np.random.default_rng(2024)
    cost = np.round(rng.uniform(0.0, 20.0, total), 1)
    cost[rng.random(total) < 0.3] = api.FAIL_COST
    K = rng.integers(1, k_max + 1, total).astype(np.int32)
    segs = rng.integers(0, 256, (total, k_max * 112)).astype(np.uint8)
    ctrl = rng.standard_normal((total, 12 * k_max))
    return cost, K, segs, ctrl


def _pack(wins):
    return [(w["cost"], w["index"], w["rank"], w["K"], w["segs"].tobytes(), w["ctrl"].tobytes()) for w in wins]


def _nccl_worker(rank, world, total, k, id_q, res_q):
    try:
        import torch
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        k_max = 16
        cost, K, segs, ctrl = _synthetic(total, k_max)
        outs = dict(a_cost=torch.from_numpy(cost).to(dev), K=torch.from_numpy(K).to(dev), segs=torch.from_numpy(segs).to(dev),
                    ctrl=torch.from_numpy(ctrl).to(dev))
        uid = api.SpectralPlanner.comm_unique_id() if rank == 0 else None
        if rank == 0:
            for _ in range(world - 1):
                id_q.put(uid)
        else:
            uid = id_q.get(timeout=120)
        pl = api.SpectralPlanner(device=rank, max_batch=1024, n_max=128, r_max=8, k_max=k_max)
        pl.comm_init(world, rank, uid)
        lo, hi = rank * total // world, (rank + 1) * total // world
        shard = {n: t[lo:hi] for n, t in outs.items()}
        sharded = pl.sweep_topk(shard, lo, k)
        # second call: rank 0 holds the whole sweep, rank 1 takes part with B_local = 0
        skew = pl.sweep_topk(outs, 0, k, B=total if rank == 0 else 0)
        # sweep_argmin is sweep_topk with k = 1, on the sharded split and on a skewed one (it needs B_local >= 1: rank 1
        # holds the last scenario only)
        lo1 = 0 if rank == 0 else total - 1
        shard1 = {n: t[lo1:] for n, t in outs.items()}
        B1 = total - 1 if rank == 0 else 1
        argmins = []
        for part, off, B_part in ((shard, lo, None), (shard1, lo1, B1)):
            argmins.append((_pack([pl.sweep_argmin(part, off, B=B_part)]), _pack(pl.sweep_topk(part, off, 1, B=B_part))))
        single = api.SpectralPlanner(device=rank, max_batch=1024, n_max=128, r_max=8, k_max=k_max)
        ref = single.sweep_topk(outs, 0, k)
        torch.cuda.synchronize()
        pl.close()
        single.close()
        res_q.put((rank, "ok", _pack(sharded), _pack(skew), _pack(ref), argmins))
    except Exception as e:  # reported to the parent, which fails the test
        res_q.put((rank, "error: %r" % (e,), None, None, None, None))


def test_sweep_topk_two_nccl_ranks():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    world, total, k = 2, 50_000, 300
    ctx = mp.get_context("spawn")
    id_q, res_q = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, total, k, id_q, res_q)) for r in range(world)]
    for p in procs:
        p.start()
    results = {}
    try:
        for _ in range(world):
            r = res_q.get(timeout=600)
            results[r[0]] = r
    except queue.Empty:
        pass
    finally:
        for p in procs:
            p.join(timeout=60)
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join(timeout=10)
    assert sorted(results) == list(range(world)), results.keys()
    for r in range(world):
        assert results[r][1] == "ok", results[r][1]
    cost, K, segs, ctrl = _synthetic(total, 16)
    ref = results[0][4]
    assert [w[1] for w in ref] == list(ref_topk(cost, k, 0)[1])
    for r in range(world):
        sharded, skew, single = results[r][2], results[r][3], results[r][4]
        assert single == ref
        # the list does not depend on the sharding; only the owning rank differs
        assert [w[:2] + w[3:] for w in sharded] == [w[:2] + w[3:] for w in ref]
        assert [w[2] for w in sharded] == [int(w[1] >= total // 2) for w in ref]
        assert [w[:2] + w[3:] for w in skew] == [w[:2] + w[3:] for w in ref] and all(w[2] == 0 for w in skew)
        for argmin, top1 in results[r][5]:
            assert argmin == top1
            assert argmin[0][:2] + argmin[0][3:] == ref[0][:2] + ref[0][3:]
    j = ref[0][1]
    assert ref[0][4] == segs[j].tobytes()[:ref[0][3] * 112] and ref[0][5] == ctrl[j, :12 * ref[0][3]].tobytes()


# ---------------------------------------------------------------- 7: invalid arguments
def test_topk_invalid_arguments(planner):
    import torch
    t = torch.zeros(8, dtype=torch.float64, device="cuda")
    for k in (0, 1025):
        with pytest.raises(ValueError):
            planner.topk_device(t, k)
        with pytest.raises(ValueError):
            planner.sweep_topk(dict(a_cost=t), 0, k)
    # tensors the kernels cannot read: refused in Python before any launch
    with pytest.raises(ValueError):
        planner.topk_device(t.cpu(), 4)                      # not on the GPU
    with pytest.raises(ValueError):
        planner.topk_device(t.float(), 4)                    # float32
    with pytest.raises(ValueError):
        planner.topk_device(torch.zeros(8, 2, dtype=torch.float64, device="cuda")[:, 0], 4)   # strided
    with pytest.raises(ValueError):
        planner.topk_device(t, 4, out_cost=torch.zeros(3, dtype=torch.float64, device="cuda"))  # too short
    with pytest.raises(ValueError):
        planner.topk_device(t, 4, index_offset=-1)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            planner.topk_device(t.to("cuda:1"), 4)           # another GPU than the planner's
    outs = planner.alloc_device_outputs(8)
    with pytest.raises(ValueError):
        planner.sweep_topk(outs, 0, 4, B=9)                  # more scenarios than the tensors hold
    with pytest.raises(ValueError):
        planner.sweep_topk(outs, 0, 4, B=-1)
    with pytest.raises(ValueError):
        planner.sweep_topk(dict(outs, K=outs["K"].long()), 0, 4)
    with pytest.raises(ValueError):
        planner.sweep_topk(dict(outs, ctrl=outs["ctrl"][:, :12]), 0, 4)
    lib, h = planner._lib, planner._h
    oc = torch.zeros(2048, dtype=torch.float64, device="cuda")
    oi = torch.zeros(2048, dtype=torch.int64, device="cuda")
    P = lambda x: ctypes.c_void_p(x.data_ptr())  # noqa: E731
    INVALID = 1
    assert lib.spectral_topk_device(h, 8, P(t), 0, 0, P(oc), P(oi), None) == INVALID
    assert lib.spectral_topk_device(h, 8, P(t), 0, 1025, P(oc), P(oi), None) == INVALID
    assert b"k must be" in lib.spectral_last_error(h)
    assert lib.spectral_topk_device(h, 0, P(t), 0, 4, P(oc), P(oi), None) == INVALID
    assert lib.spectral_topk_device(h, 8, P(t), 0, 4, None, P(oi), None) == INVALID
    assert lib.spectral_topk_device(h, 8, P(t), 0, 4, P(oc), None, None) == INVALID
    assert lib.spectral_topk_device(h, 8, None, 0, 4, P(oc), P(oi), None) == INVALID
    assert lib.spectral_topk_device(None, 8, P(t), 0, 4, P(oc), P(oi), None) == INVALID
    out = api.SpectralOutputs()
    out.a_cost = ctypes.cast(P(t), ctypes.POINTER(ctypes.c_double))
    ws = (api.SpectralWinner * 4)()
    n = ctypes.c_int()
    assert lib.spectral_sweep_topk(h, 8, ctypes.byref(out), 0, 0, ws, ctypes.byref(n), None) == INVALID
    assert lib.spectral_sweep_topk(h, 8, ctypes.byref(out), 0, 1025, ws, ctypes.byref(n), None) == INVALID
    assert lib.spectral_sweep_topk(h, -1, ctypes.byref(out), 0, 4, ws, ctypes.byref(n), None) == INVALID
    assert lib.spectral_sweep_topk(h, 8, None, 0, 4, ws, ctypes.byref(n), None) == INVALID
    assert lib.spectral_sweep_topk(h, 8, ctypes.byref(out), 0, 4, None, ctypes.byref(n), None) == INVALID
    assert lib.spectral_sweep_topk(h, 8, ctypes.byref(out), 0, 4, ws, None, None) == INVALID
    assert lib.spectral_sweep_topk(h, 8, ctypes.byref(out), 0, 4, ws, ctypes.byref(n), None) == INVALID  # K/segs/ctrl missing
    full = api.SpectralOutputs()
    full.a_cost = ctypes.cast(P(outs["a_cost"]), ctypes.POINTER(ctypes.c_double))
    full.K = ctypes.cast(P(outs["K"]), ctypes.POINTER(ctypes.c_int))
    full.segs = outs["segs"].data_ptr()
    full.ctrl = ctypes.cast(P(outs["ctrl"]), ctypes.POINTER(ctypes.c_double))
    w = api.SpectralWinner()
    assert lib.spectral_sweep_argmin(h, 8, ctypes.byref(full), -1, ctypes.byref(w), None) == INVALID
    assert b"index_offset" in lib.spectral_last_error(h)
    assert lib.spectral_sweep_argmin(h, 0, ctypes.byref(full), 0, ctypes.byref(w), None) == INVALID
    assert lib.spectral_sweep_argmin(h, 8, ctypes.byref(out), 0, ctypes.byref(w), None) == INVALID   # K/segs/ctrl missing
    assert lib.spectral_sweep_argmin(h, 8, ctypes.byref(full), 0, ctypes.byref(w), None) == 0
    # the handle still works after the refused calls
    oc2, oi2 = planner.topk_device(torch.arange(8, 0, -1, dtype=torch.float64, device="cuda"), 3)
    torch.cuda.synchronize()
    assert oi2.cpu().tolist() == [7, 6, 5]
