// spectral_b200/csrc/corridor.cuh -- K1 (corridor generation + split) and K2 (selection).
//
// Reference behaviour being reproduced bit for bit (paths relative to /root/reference/src):
//   CorridorGeneration  solve_3d.cc:323-486   | cuboid_3d.cc:301-407
//   CorridorSplit       solve_3d.cc:729-772   | cuboid_3d.cc:588-625
//   CollisionCheck      solve_3d.cc:488-714   | cuboid_3d.cc:409-573
// Mapping: one CTA per scenario, one warp per lateral region ("corridor face set").  Each warp
// stages its region's s/l bound slabs (2 x 16N bytes) into shared memory with a 1-D bulk async
// copy (TMA, cp.async.bulk + mbarrier), finds the slope breaks with ballot votes, splits its
// cubes (lane j % 32 holds pre-split cube j) and counts the reference-trajectory points inside each
// cube (lanes over knots, popc of ballots).  Warp 0 then replays the selection / dedupe / sort /
// swap / de-overlap logic, whose O(K^2) sequential parts run on lane 0 exactly as written in the
// reference (including libstdc++'s std::sort algorithm, whose result on equal keys is
// implementation-defined).
// Compile this translation unit with --fmad=false: the reference is SSE2 code without FMA.
#pragma once
#include "common.cuh"

struct CorridorArgs {
  int B, N, R, variant, k_max;
  double delta;
  const double *s_bounds, *l_bounds, *s_ref, *l_ref;
  SpectralCube *segs;  // [B][k_max]
  int *K;              // [B]
  int *status;         // [B] 0 = corridor ok, otherwise SPECTRAL_FAIL_*
};

// shared-memory carve-up (bytes), all offsets multiples of 16
struct CorridorSmem {
  int slab;       // bytes of one (lo,hi) slab: 16*N
  int off_xb;     // R slabs
  int off_yb;     // R slabs
  int off_slope;  // R * 2 * N doubles: backward slopes of the lower / upper s-bound per knot (computed once per region)
  int off_cubes;  // R * SP_REGION_CAP cubes
  int off_cnt;    // R * SP_REGION_CAP ints
  int off_ncube;  // SP_MAX_REGIONS ints
  int off_ref;    // 2 * N doubles (s_ref, l_ref), padded
  int off_sel;    // SP_SELECT_CAP cubes
  int off_ord;    // SP_SELECT_CAP ints
  int off_misc;   // 4 ints
  int off_bar;    // SP_MAX_REGIONS mbarriers
  int total;
};

SP_HD CorridorSmem corridor_smem_layout(int N, int R) {
  CorridorSmem L;
  int o = 0;
  L.slab = 16 * N;
  L.off_xb = o; o += R * L.slab;
  L.off_yb = o; o += R * L.slab;
  L.off_slope = o; o += R * L.slab;
  L.off_cubes = o; o += R * SP_REGION_CAP * (int)sizeof(SpectralCube);
  L.off_cnt = o; o += R * SP_REGION_CAP * 4;
  L.off_ncube = o; o += SP_MAX_REGIONS * 4;
  L.off_ref = o; o += ((2 * N * 8 + 15) / 16) * 16;
  L.off_sel = o; o += SP_SELECT_CAP * (int)sizeof(SpectralCube);
  L.off_ord = o; o += SP_SELECT_CAP * 4;
  L.off_misc = o; o += 16;
  L.off_bar = o; o += SP_MAX_REGIONS * 8;
  L.total = o;
  return L;
}

// ---------------------------------------------------------------------------------------------
// bulk-async (TMA 1-D) staging
#ifndef SPECTRAL_CPU_EMU
SP_DEV uint32_t sp_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
SP_DEV void sp_mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sp_smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
SP_DEV void sp_bulk_load(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   sp_smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(sp_smem_u32(bar))
               : "memory");
}
SP_DEV void sp_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sp_smem_u32(bar)), "r"(bytes) : "memory");
}
SP_DEV void sp_mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(sp_smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
#endif

SP_DEV void cube_defaults(SpectralCube &c) {  // Cube::Cube(), cube_type.h:12-21
  c.beg_t = 0; c.end_t = 0; c.t = 0.0; c.t_dif = 0.0; c.beg_l = 0.0; c.end_l = 0.0;
  c.upp_skew = 0.0; c.upp_bias = 1000.0; c.down_skew = 0.0; c.down_bias = 0.0;
  c.l_upp_skew = 0.0; c.l_upp_bias = 1000.0; c.l_down_skew = 0.0; c.l_down_bias = 0.0;
  c.merge = 0; c.split = 0; c.count = 0;
}

// inside test of CollisionCheck (solve_3d.cc:534-581); tt is the knot index as a double (:497)
SP_DEV int point_inside(const SpectralCube &c, double s, double l, double tt, double delta) {
  if (!(l <= c.end_l && l >= c.beg_l)) return 0;
  int pos = 0, neg = 0;
  double d;
  // the (beg_t - beg_t) / (end_t - end_t) factors are the reference's own (:536, :559)
  d = (s - c.down_bias) * (double)(c.beg_t - c.beg_t) - (tt - c.beg_t) * (c.upp_bias - c.down_bias);
  pos += d > 0; neg += d < 0;
  if (pos > 0 && neg > 0) return 0;
  d = (s - c.upp_bias) * (double)(c.end_t - c.beg_t) - (tt - c.beg_t) * (c.upp_skew * delta + c.upp_bias - c.upp_bias);
  pos += d > 0; neg += d < 0;
  if (pos > 0 && neg > 0) return 0;
  d = (s - c.upp_bias - c.upp_skew * delta) * (double)(c.end_t - c.end_t) -
      (tt - c.end_t) * (c.down_skew * delta + c.down_bias - c.upp_skew * delta - c.upp_bias);
  pos += d > 0; neg += d < 0;
  if (pos > 0 && neg > 0) return 0;
  d = (s - c.down_bias - c.down_skew * delta) * (double)(c.beg_t - c.end_t) -
      (tt - c.end_t) * (c.down_bias - c.down_skew * delta - c.down_bias);
  pos += d > 0; neg += d < 0;
  if (pos > 0 && neg > 0) return 0;
  return 1;
}

// ---------------------------------------------------------------------------------------------
// libstdc++ std::sort (bits/stl_algo.h) restated on an index array keyed by beg_t; run by one lane.
struct SortView {
  int *ord;
  const SpectralCube *sel;
  SP_DEV int key(int pos) const { return sel[ord[pos]].beg_t; }
};
SP_DEV void ss_unguarded_linear_insert(SortView v, int last) {
  int val = v.ord[last], kv = v.sel[val].beg_t;
  int next = last - 1;
  while (kv < v.key(next)) { v.ord[last] = v.ord[next]; last = next; --next; }
  v.ord[last] = val;
}
SP_DEV void ss_insertion_sort(SortView v, int first, int last) {
  if (first == last) return;
  for (int i = first + 1; i != last; ++i) {
    if (v.key(i) < v.key(first)) {
      int val = v.ord[i];
      for (int p = i; p > first; --p) v.ord[p] = v.ord[p - 1];
      v.ord[first] = val;
    } else ss_unguarded_linear_insert(v, i);
  }
}
SP_DEV void ss_adjust_heap(SortView v, int first, int hole, int len, int value) {
  const int top = hole;
  int second = hole;
  const int kval = v.sel[value].beg_t;
  while (second < (len - 1) / 2) {
    second = 2 * (second + 1);
    if (v.key(first + second) < v.key(first + second - 1)) second--;
    v.ord[first + hole] = v.ord[first + second]; hole = second;
  }
  if ((len & 1) == 0 && second == (len - 2) / 2) {
    second = 2 * (second + 1);
    v.ord[first + hole] = v.ord[first + second - 1]; hole = second - 1;
  }
  int parent = (hole - 1) / 2;
  while (hole > top && v.key(first + parent) < kval) {
    v.ord[first + hole] = v.ord[first + parent]; hole = parent; parent = (hole - 1) / 2;
  }
  v.ord[first + hole] = value;
}
SP_DEV void ss_heap_sort(SortView v, int first, int last) {
  int len = last - first;
  if (len >= 2) {
    int parent = (len - 2) / 2;
    for (;;) {
      int val = v.ord[first + parent];
      ss_adjust_heap(v, first, parent, len, val);
      if (parent == 0) break;
      parent--;
    }
  }
  while (last - first > 1) {
    --last;
    int val = v.ord[last];
    v.ord[last] = v.ord[first];
    ss_adjust_heap(v, first, 0, last - first, val);
  }
}
SP_DEV void ss_swap(SortView v, int a, int b) { int t = v.ord[a]; v.ord[a] = v.ord[b]; v.ord[b] = t; }
SP_DEV void std_sort_by_beg_t(SortView v, int n) {
  if (n <= 0) return;
  int depth = 0;
  for (int q = n; q > 1; q >>= 1) depth++;
  depth *= 2;
  // __introsort_loop, recursion unrolled with a small stack of (first,last,depth) ranges
  int stk_first[32], stk_last[32], stk_depth[32], sp = 0;
  int first = 0, last = n;
  for (;;) {
    while (last - first > 16) {
      if (depth == 0) { ss_heap_sort(v, first, last); break; }
      --depth;
      int mid = first + (last - first) / 2;
      int a = first + 1, b = mid, c = last - 1;
      // __move_median_to_first(first, a, b, c)
      if (v.key(a) < v.key(b)) {
        if (v.key(b) < v.key(c)) ss_swap(v, first, b);
        else if (v.key(a) < v.key(c)) ss_swap(v, first, c);
        else ss_swap(v, first, a);
      } else if (v.key(a) < v.key(c)) ss_swap(v, first, a);
      else if (v.key(b) < v.key(c)) ss_swap(v, first, c);
      else ss_swap(v, first, b);
      // __unguarded_partition(first + 1, last, first)
      int lo = first + 1, hi = last;
      const int pk = v.key(first);
      for (;;) {
        while (v.key(lo) < pk) ++lo;
        --hi;
        while (pk < v.key(hi)) --hi;
        if (!(lo < hi)) break;
        ss_swap(v, lo, hi);
        ++lo;
      }
      int cut = lo;
      // recurse on [cut, last) first, then continue with [first, cut)
      stk_first[sp] = first; stk_last[sp] = cut; stk_depth[sp] = depth; sp++;
      first = cut;
    }
    if (sp == 0) break;
    sp--;
    first = stk_first[sp]; last = stk_last[sp]; depth = stk_depth[sp];
  }
  if (n > 16) {
    ss_insertion_sort(v, 0, 16);
    for (int i = 16; i != n; ++i) ss_unguarded_linear_insert(v, i);
  } else ss_insertion_sort(v, 0, n);
}

// num / delta, IEEE.  A zero numerator (flat bounds: the common case) gives a zero of the numerator's sign for any
// positive delta; answering it directly keeps the division's slow path (taken for zero operands) out of the way.
// The division itself always runs on a non-zero numerator (1.0 stands in for the zeros), so that no lane of the warp ever
// drags the others through the out-of-line special-case routine of the double-precision division.
SP_DEV double slope_div(double num, double delta) {
  const bool zero = num == 0.0 && delta > 0.0;
  const double q = (zero ? 1.0 : num) / delta;
  return zero ? num : q;
}

// ---------------------------------------------------------------------------------------------
// K1: one warp, one region.  Returns the cube count written to `out` (shared) or -1 (capacity).
// `slope`: 2 N doubles of shared memory for this region.
SP_DEV int corridor_generate_region(int variant, int N, double delta, const double *xb, const double *yb, double *slope,
                                    SpectralCube *out, int lane) {
#define XLO(i) xb[2 * (i)]
#define XHI(i) xb[2 * (i) + 1]
#define YLO(i) yb[2 * (i)]
#define YHI(i) yb[2 * (i) + 1]
  // pre-split cube j lives in the registers of lane j % 32, slot j / 32: up to SP_REGION_CAP = 64 cubes, the oracle's cap.
  // Slots are only ever indexed with constants (both branches written out), which keeps them in registers.
  SpectralCube mine[2];
  cube_defaults(mine[0]);
  cube_defaults(mine[1]);
  int j = 0;
  // backward slopes of every knot, once (:355-356; the forward slope at a break knot i, :380-384, is the backward slope
  // of knot i + 1: same operands, same operation).  The break search below then only compares.
  double *dsk = slope, *usk = slope + N;
  for (int i = 1 + lane; i < N; i += 32) {
    dsk[i] = slope_div(XLO(i) - XLO(i - 1), delta);
    usk[i] = slope_div(XHI(i) - XHI(i - 1), delta);
  }
  sp_syncwarp();
  double cur_down = dsk[1];  // :332
  double cur_up = usk[1];    // :334
  if (lane == 0) {
    SpectralCube &c = mine[0];
    c.beg_t = 0;
    c.down_skew = cur_down; c.down_bias = XLO(0);
    c.upp_skew = cur_up; c.upp_bias = XHI(0);
    if (variant == SPECTRAL_TRP) {  // :338-341
      c.l_down_skew = slope_div(YLO(1) - YLO(0), delta); c.l_down_bias = YLO(0);
      c.l_upp_skew = slope_div(YHI(1) - YHI(0), delta); c.l_upp_bias = YHI(0);
    }
    c.beg_l = YLO(0); c.end_l = YHI(0);
  }
  j = 1;
  int i0 = 2;
  int overflow = 0;
  for (;;) {
    // next knot i in [i0, N-2] whose backward slope leaves the current cube's slope by > 0.2 (:355-374)
    int found = -1;
    for (int base = i0; base <= N - 2; base += 32) {
      int i = base + lane;
      int pred = 0;
      if (i <= N - 2) pred = (fabs(dsk[i] - cur_down) > 0.2) || (fabs(usk[i] - cur_up) > 0.2);
      unsigned m = sp_ballot(pred);
      if (m) { found = base + sp_ffs(m) - 1; break; }
    }
    if (found < 0) break;
    if (j >= SP_REGION_CAP) { overflow = 1; break; }
    const int i = found;
    if (lane == ((j - 1) & 31)) {  // :376
      if (j - 1 < 32) mine[0].end_t = i;
      else mine[1].end_t = i;
    }
    cur_down = dsk[i + 1];  // :380
    cur_up = usk[i + 1];    // :384
    if (lane == (j & 31)) {
      SpectralCube c;
      cube_defaults(c);
      c.beg_t = i;
      c.down_skew = cur_down; c.down_bias = XLO(i);
      c.upp_skew = cur_up; c.upp_bias = XHI(i);
      if (variant == SPECTRAL_TRP) {  // :360-367, backward differences at the break knot
        c.l_down_bias = YLO(i); c.l_upp_bias = YHI(i);
        c.l_down_skew = slope_div(YLO(i) - YLO(i - 1), delta);
        c.l_upp_skew = slope_div(YHI(i) - YHI(i - 1), delta);
      }
      c.beg_l = YLO(i); c.end_l = YHI(i);  // :388-389
      if (j < 32) mine[0] = c;
      else mine[1] = c;
    }
    j++;
    i0 = i + 1;
  }
  if (overflow) return -1;
  if (lane == ((j - 1) & 31)) {  // :461
    if (j - 1 < 32) mine[0].end_t = N - 1;
    else mine[1].end_t = N - 1;
  }
  const int nslot = j > 32 ? 2 : 1;

  // CorridorSplit (:729-772): each pre-split cube peels 1.0 s / 10-knot pieces off its front; cube j's pieces are written
  // after those of cubes 0 .. j-1 (a prefix sum over slot 0, then over slot 1)
  int pieces[2] = {0, 0}, pos[2] = {0, 0};
  int total = 0;
#pragma unroll
  for (int s = 0; s < 2; s++) {
    if (s >= nslot) break;
    const bool have = 32 * s + lane < j;
    mine[s].t = (mine[s].end_t - mine[s].beg_t) * delta;  // :465  (int -> double, then * delta)
    if (have) {
      double t = mine[s].t;
      while (t > 1) { t = t - 1; pieces[s]++; }
    }
    const int mycount = have ? pieces[s] + 1 : 0;
    int incl = mycount;
    for (int d = 1; d < 32; d <<= 1) {
      int o = sp_shfl_up_i(incl, d, 32);
      if (lane >= d) incl += o;
    }
    pos[s] = total + incl - mycount;
    total += sp_shfl_i(incl, 31);
  }
  if (total > SP_REGION_CAP) return -1;
#pragma unroll
  for (int s = 0; s < 2; s++) {
    if (32 * s + lane >= j) continue;
    int p_out = pos[s];
    SpectralCube rest = mine[s];
    for (int p = 0; p < pieces[s]; p++) {
      rest.t = rest.t - 1;  // :737
      SpectralCube m;
      cube_defaults(m);
      m.beg_t = rest.beg_t;
      rest.beg_t = rest.beg_t + 10;
      m.end_t = m.beg_t + 10;
      m.t = 1.0;
      m.down_skew = rest.down_skew; m.down_bias = rest.down_bias;
      if (variant == SPECTRAL_TRP) { m.l_down_skew = rest.l_down_skew; m.l_down_bias = rest.l_down_bias; }
      rest.down_bias = m.down_bias + 1.0 * m.down_skew;  // :753
      m.upp_skew = rest.upp_skew; m.upp_bias = rest.upp_bias;
      if (variant == SPECTRAL_TRP) { m.l_upp_skew = rest.l_upp_skew; m.l_upp_bias = rest.l_upp_bias; }
      m.beg_l = rest.beg_l; m.end_l = rest.end_l;
      rest.upp_bias = m.upp_bias + 1.0 * m.upp_skew;  // :764
      out[p_out++] = m;
    }
    out[p_out] = rest;
  }
  return total;
#undef XLO
#undef XHI
#undef YLO
#undef YHI
}

// One CTA per scenario; warp w handles region w.  `smem` is the CTA's dynamic shared memory.
// sync_cta() is __syncthreads() on the device.
template <typename SyncFn>
SP_DEV void corridor_cta_body(const CorridorArgs &a, int b, int warp, int lane, unsigned char *smem, SyncFn sync_cta) {
  const int N = a.N, R = a.R;
  const CorridorSmem L = corridor_smem_layout(N, R);
  double *xb = (double *)(smem + L.off_xb + warp * L.slab);
  double *yb = (double *)(smem + L.off_yb + warp * L.slab);
  double *slope = (double *)(smem + L.off_slope + warp * L.slab);
  SpectralCube *cubes = (SpectralCube *)(smem + L.off_cubes) + warp * SP_REGION_CAP;
  int *cnt = (int *)(smem + L.off_cnt) + warp * SP_REGION_CAP;
  int *ncube = (int *)(smem + L.off_ncube);
  double *sref = (double *)(smem + L.off_ref);
  double *lref = sref + N;
  SpectralCube *sel = (SpectralCube *)(smem + L.off_sel);
  int *ord = (int *)(smem + L.off_ord);
  int *misc = (int *)(smem + L.off_misc);

  const double *g_xb = a.s_bounds + ((size_t)b * R + warp) * 2 * N;
  const double *g_yb = a.l_bounds + ((size_t)b * R + warp) * 2 * N;
#ifndef SPECTRAL_CPU_EMU
  // TMA 1-D bulk copies of the two 16N-byte slabs, completion on this warp's mbarrier
  uint64_t *bar = (uint64_t *)(smem + L.off_bar) + warp;
  if (lane == 0) sp_mbar_init(bar, 1);
  sp_syncwarp();
  if (lane == 0) {
    sp_mbar_expect_tx(bar, 2u * (uint32_t)L.slab);
    sp_bulk_load(xb, g_xb, (uint32_t)L.slab, bar);
    sp_bulk_load(yb, g_yb, (uint32_t)L.slab, bar);
  }
#else
  for (int i = lane; i < 2 * N; i += 32) { xb[i] = g_xb[i]; yb[i] = g_yb[i]; }
#endif
  // reference trajectory: coalesced loads by all warps of the CTA
  for (int i = warp * 32 + lane; i < N; i += 32 * R) {
    sref[i] = a.s_ref[(size_t)b * N + i];
    lref[i] = a.l_ref[(size_t)b * N + i];
  }
#ifndef SPECTRAL_CPU_EMU
  sp_mbar_wait(bar, 0);
#else
  sp_syncwarp();
#endif

  int n = corridor_generate_region(a.variant, N, a.delta, xb, yb, slope, cubes, lane);
  if (lane == 0) ncube[warp] = n;
  sync_cta();  // cubes + refs visible

  // inside counts of this region's cubes: lanes over knots, popc(ballot) (solve_3d.cc:529-584)
  if (n > 0) {
    // The first and the third edge test of point_inside are  -(t - beg_t) a1  and  -(t - end_t) a3  (their other terms are
    // multiplied by the reference's (beg_t - beg_t) / (end_t - end_t) = 0).  With a1 > 0 and a3 < 0 -- every cube whose upper
    // face lies above its lower face -- they have strictly opposite signs for every knot outside [beg_t, end_t], i.e. such
    // a knot is never inside: only the cube's own knots need the test.  After the split a cube spans at most 11 knots, so
    // TWO cubes share one ballot (lanes 0-15: cube k, lanes 16-31: cube k + 1).  Any other cube takes the full scan.
    for (int k = 0; k < n; k += 2) {
      const int half = lane >> 4, l16 = lane & 15, kk = k + half;
      const bool have = kk < n;
      const SpectralCube c = cubes[have ? kk : k];
      const double a1 = c.upp_bias - c.down_bias;
      const double a3 = c.down_skew * a.delta + c.down_bias - c.upp_skew * a.delta - c.upp_bias;
      const int len = c.end_t - c.beg_t + 1;
      const bool fast = have && a1 > 0.0 && a3 < 0.0 && c.beg_t >= 0 && len >= 1 && len <= 16 && c.end_t < N;
      int in = 0;
      if (fast && l16 < len) {
        const int i = c.beg_t + l16;
        in = point_inside(c, sref[i], lref[i], (double)i, a.delta);
      }
      const unsigned m = sp_ballot(in);
      if (fast && l16 == 0) cnt[kk] = sp_popc(half ? (m >> 16) : (m & 0xffffu));
      // the full scan for the cubes of this pair that are not "fast" (warp-uniform: the flags of lanes 0 and 16)
      const int fa = sp_shfl_i(fast ? 1 : 0, 0), fb = sp_shfl_i(fast ? 1 : 0, 16);
      for (int which = 0; which < 2; which++) {
        const int kf = k + which;
        if ((which == 0 ? fa : fb) || kf >= n) continue;
        const SpectralCube cf = cubes[kf];
        int total = 0;
        for (int base = 0; base < N; base += 32) {
          const int i = base + lane;
          int inf = 0;
          if (i < N) inf = point_inside(cf, sref[i], lref[i], (double)i, a.delta);
          total += sp_popc(sp_ballot(inf));
        }
        if (lane == 0) cnt[kf] = total;
      }
    }
  }
  sync_cta();
  if (warp != 0) return;

  // ---- K2 on warp 0
  int bad = 0;
  for (int r = 0; r < R; r++) bad |= (ncube[r] < 0);
  if (bad) {
    if (lane == 0) { a.K[b] = 0; a.status[b] = SPECTRAL_FAIL_TOO_MANY; }
    return;
  }
  // every third inside point pushes the cube it fell in; `count` is carried across cubes and
  // regions, so a cube is pushed iff floor((T+c)/3) > floor(T/3) with T the running total before it.
  // Duplicates are erased later by exact equality (:617-628) keeping first occurrences, so each
  // distinct cube is appended once, in first-push order.
  const SpectralCube *all = (const SpectralCube *)(smem + L.off_cubes);
  const int *allcnt = (const int *)(smem + L.off_cnt);
  int T = 0, nsel = 0, overflow = 0;
  for (int r = 0; r < R; r++) {
    for (int k = 0; k < ncube[r]; k++) {
      const int c = allcnt[r * SP_REGION_CAP + k];
      const int pushed = ((T + c) / 3) > (T / 3);
      T += c;
      if (!pushed) continue;
      const SpectralCube &cand = all[r * SP_REGION_CAP + k];
      int dup = 0;
      for (int base = 0; base < nsel; base += 32) {
        int i = base + lane;
        int eq = 0;
        if (i < nsel) {
          const SpectralCube &o = sel[i];
          eq = o.beg_t == cand.beg_t && o.end_t == cand.end_t && o.down_bias == cand.down_bias &&
               o.down_skew == cand.down_skew && o.upp_bias == cand.upp_bias && o.upp_skew == cand.upp_skew &&
               o.beg_l == cand.beg_l && o.end_l == cand.end_l;
        }
        dup |= sp_any(eq);
      }
      if (dup) continue;
      if (nsel >= SP_SELECT_CAP) { overflow = 1; continue; }
      if (lane == 0) { sel[nsel] = cand; sel[nsel].count = 3; ord[nsel] = nsel; }
      nsel++;
      sp_syncwarp();
    }
  }
  if (overflow || nsel == 0) {
    if (lane == 0) { a.K[b] = 0; a.status[b] = overflow ? SPECTRAL_FAIL_TOO_MANY : SPECTRAL_FAIL_NO_CORRIDOR; }
    return;
  }
  sp_syncwarp();
  if (lane == 0) {
    const double delta = a.delta;
    SortView v{ord, sel};
#define S_(p) sel[ord[p]]
    if (a.variant == SPECTRAL_TRP) {
      std_sort_by_beg_t(v, nsel);  // :630
      for (int i = 0; i < nsel - 1; i++) {  // lateral-continuity swap pass (:639-673)
        for (int j = i + 1; j < nsel; j++) {
          if (S_(i).beg_l == S_(j).beg_l && j - i == 1) break;
          for (int k = j + 1; k < nsel; k++) {
            if (S_(i).beg_l == S_(k).beg_l && S_(i).end_t == S_(k).beg_t) { ss_swap(v, j, k); break; }
          }
        }
      }
      for (int i = 0; i < nsel - 1; i++) {  // de-overlap, only j = i+1 (:678-703)
        const int j = i + 1;
        SpectralCube &ci = S_(i), &cj = S_(j);
        if (ci.beg_t == cj.beg_t && ci.end_t == cj.end_t) {
          int diff = (ci.end_t - ci.beg_t) / 2;
          ci.end_t = ci.end_t - diff;
          ci.t = (ci.end_t - ci.beg_t) * delta;
          cj.beg_t = cj.beg_t + diff;
          cj.t = (cj.end_t - cj.beg_t) * delta;
        } else if (ci.beg_t > cj.beg_t && ci.end_t <= cj.end_t) {
          int diff = (ci.end_t - ci.beg_t) / 2;
          if (diff > 1) { ci.end_t = ci.end_t - diff; ci.t = (ci.end_t - ci.beg_t) * delta; }
          cj.beg_t = ci.end_t;
          cj.t = (cj.end_t - cj.beg_t) * delta;
        }
      }
    } else {
      for (int i = 0; i < nsel - 1; i++) {  // cuboid_3d.cc:553-567: all pairs, /3, no extra branch
        for (int j = i + 1; j < nsel; j++) {
          SpectralCube &ci = S_(i), &cj = S_(j);
          if (ci.beg_t == cj.beg_t && ci.end_t == cj.end_t) {
            int diff = (ci.end_t - ci.beg_t) / 3;
            ci.end_t = ci.end_t - diff;
            ci.t = (ci.end_t - ci.beg_t) * delta;
            cj.beg_t = cj.beg_t + diff;
            cj.t = (cj.end_t - cj.beg_t) * delta;
          }
        }
      }
    }
#undef S_
    misc[0] = nsel;
  }
  sp_syncwarp();
  const int K = nsel;
  if (K > a.k_max) {
    if (lane == 0) { a.K[b] = K; a.status[b] = SPECTRAL_FAIL_TOO_MANY; }
    return;
  }
  // write new_corridor: K cubes of 14 x 8-byte words, lanes strided over words
  {
    const unsigned long long *src;
    unsigned long long *dst = (unsigned long long *)(a.segs + (size_t)b * a.k_max);
    for (int w = lane; w < K * 14; w += 32) {
      int k = w / 14, f = w - 14 * k;
      src = (const unsigned long long *)(sel + ord[k]);
      unsigned long long word = src[f];
      if (f == 13) word &= 0xffffffff0000ffffull;  // bytes 106-107 are struct padding: keep the output deterministic
      dst[(size_t)k * 14 + f] = word;
    }
  }
  if (lane == 0) { a.K[b] = K; a.status[b] = 0; }
}
