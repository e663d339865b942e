// spectral_b200/csrc/qp_dense.cuh -- K4: the batched ADMM (OSQP-equivalent) hot loop, dense-operator form.
//
// Replaces the iteration that the reference delegates to OSQP (osqp_solve, called at solve_3d.cc:1249 |
// cuboid_3d.cc:1108 with the settings of solve_3d.cc:1235-1243,1446-1462) for scenarios with at most
// KC <= 16 Bezier segments (k_qpd is instantiated for KC = 12, 16; the KC <= 10 classes run the anchor layout of qp_anchor.cuh,
// which shares this file's setup, layout and check code).  One CTA = one scenario = both axis problems (s and l), solved as ONE OSQP
// instance like the reference does: one cost scaling c, one rho, joint termination and infeasibility norms.
//
// Why this form.  The lane-per-segment loop of qp.cuh (block-tridiagonal Cholesky, one lane per segment)
// spends its time in 2K dependent neighbour-to-neighbour hops per iteration and leaves 3/4 of the SM idle
// at the batch sizes of BASELINE.json (ncu, profiles/r1_qp_lanes.md: 13 k cycles per iteration, FP64 pipe
// 5 % busy).  Here the reduced KKT matrix S = P + sigma I + A' rho A of one axis (n = 6 KC <= 60) is inverted
// ONCE per rho (setup and the rare adaptive-rho updates) and the inverse G = S^-1 is kept in REGISTERS, one
// row per thread pair (n/2 doubles each), so the per-iteration solve x~ = G g is n/2 independent FMAs per thread with the
// right-hand side broadcast from shared memory: no dependent chain, no shuffles.  A and A' are never stored:
// their rows are finite-difference stencils of the control points (solve_3d.cc:823-949), applied from
// zero-padded shared-memory arrays so that every thread runs the same instruction stream.
//
// Three thread layouts, each the measured winner of its class (profiles/r1_qpd_staging.md):
//   KC = 12       row pairs (below): 2 chunks per row of G, 160 threads per axis, 168 registers, staged loads  qpd_block
//   KC = 8, 10    full rows: one thread per variable holds its whole row of G, 64 threads per axis, 255
//                 registers, four generic row slots per thread                                              qpd_block1
//                 (replaced by the anchor layout of qp_anchor.cuh; kept as its bit-exact reference in the emulator tests)
//   KC = 16       quarter rows: 4 chunks per row, one constraint row per thread, 384 threads per axis        qpd_block4
//                 (KC = 12 ran this layout at 7.7 ms; as staged row pairs, one CTA per SM at 320 threads: 6.4 ms)
// (A v-major layout, chunk index uniform per warp and partial sums through shared memory, measured slower for K <= 8: 14.6
// against 11.6 ms, profiles/r1_qpd_staging.md.)
//
// Thread map of the row-pair layout (per axis TA = 2n threads rounded up to whole warps: 96 for KC = 8; CTA = 2 TA):
//   thread (v, h) = ta >> 1, ta & 1 : half row h of G (n/2 doubles in registers); the h = 0 thread also owns the
//                                     relaxed iterate x_v, gathers (A' v)_v and publishes x~_v
//   row slots                       : every thread owns up to two "difference" rows (containment, velocity,
//                                     acceleration, jerk: one code path, the order of the finite difference is
//                                     selected per row) or one difference row and one continuity/init row; their
//                                     w = z + y / rho, clip(w), l, u, rho live in registers
// Per iteration (3 CTA barriers):  S2 gather g = A'(rho (2 clip(w) - w)) + sigma x - q   (13 LDS + 16 FMA)
//                                  S3 x~ = G g: n/2 FMAs per thread + one shuffle, x = alpha x~ + (1 - alpha) x
//                                  S1 z~ = A x~ (stencil), w += alpha (z~ - clip(w)), next v   (per row slot)
// Every check_termination iterations the residual / infeasibility norms of OSQP are evaluated in the same
// layout (CTA-wide reductions); adaptive-rho updates re-run the factorisation of qp.cuh on warp 0 and
// rebuild G.  Setup (K3 assembly, Ruiz scaling), factorisation, polish and outputs are the lane-per-segment
// code of qp.cuh, executed by warp 0.
#pragma once
#include "common.cuh"
#include "qp.cuh"

#define QPD_VB 38         // doubles per segment block of the padded row-value array V (38 = 6 mod 16: the gather of
                          // variable v = 6k + j hits bank pair v mod 16, conflict free)
#define QPD_V0 0          // containment rows      V0[i], i = 0..5
#define QPD_V1 7          // velocity rows         V1[i] at 7 + i,  i = -1..5 (pads at 6, 12)
#define QPD_V2 15         // acceleration rows     V2[i] at 15 + i, i = -2..5 (pads at 13, 14, 19, 20)
#define QPD_V3 24         // jerk rows             V3[i] at 24 + i, i = -3..5 (pads at 21..23, 27..29)
#define QPD_VC 30         // continuity/init rows  Vc[r] at 30 + r
#define QPD_CP 3          // leading pads of the control-point arrays C / XR (window of the first continuity rows)
#define QPD_LS 24         // doubles of lane state per segment: t, tp, tn, q[6], sig[6], cD[6]
#define QPD_NRED 10

template <int KC>
struct QpdLayout {
  // Full-row layout: ONE thread per variable holds its whole row of G (n doubles) -- 64 threads per axis, 128 per CTA, up to
  // 255 registers, still two CTAs per SM.  No chunk reduction (no shuffles), the g vector is read with every lane on the same
  // address (one wavefront per LDS.128), the gather runs on all variable lanes, and every thread carries ceil(21 KC / 64)
  // constraint rows whose loads and updates interleave (ILP instead of TLP: the kernel is latency-bound and every wider layout
  // tried lost to its extra barriers and instructions, profiles/r1_qpd_staging.md).
  // Measured (profiles/r1_qpd_staging.md): K <= 10: 9.95 ms (row pairs at 128 registers) -> 7.85 ms; K <= 8: 10.0 ms against
  // 10.6 ms of the staged row-pair layout at 168 registers (same box), once g is staged in groups of 24 doubles.
  static constexpr bool ROWFULL = KC <= 10;    // thread t = variable t, whole row of G, NSLOT generic row slots
  // Chunks per row of G (= threads per variable).  Measured on B200 (profiles/r1_qpd_nch.md): 2 chunks beat 4 for the
  // common K <= 8 class -- with 4, the warps run the variable gather with a quarter of their lanes and the total
  // instruction / shared-memory wavefront count per iteration rises 59 % / 69 %.  4 chunks (a quarter row of G and at
  // most one constraint row per thread) are kept where 2 would not fit the register file (KC >= 12).
  static constexpr int NCH = ROWFULL ? 1 : (KC >= 16 ? 4 : 2);  // threads per variable (chunks per row of G)
  // Staged loads (a run of loads, a fence, then the arithmetic) need temporaries for everything in flight: they pay where
  // the register budget has room (KC <= 8: 168 registers, measured 14.9 -> 12.5 ms) and spill where it has not (KC = 10 at
  // 128 registers: 9.5 -> 12.2 ms, in groups of 10 doubles: 9.65 -> 10.2 ms; KC >= 12 at 96 / 80: 8.0 -> 8.9 ms) --
  // profiles/r1_qpd_staging.md.
  static constexpr bool STAGE = KC <= 8 || KC == 12;       // S3: the whole g chunk in flight (CH doubles of temporaries)
  static constexpr bool LU_REG = KC <= 8 || KC == 12;      // (l, u) of the row slots in registers instead of one LDS.128 per slot and iteration
  static constexpr bool STAGE_ROWS = KC <= 8 || KC == 12;  // S2 / S1: 13 - 18 doubles of temporaries (KC = 10 at 128 registers: 9.5 -> 10.6 ms)
  static_assert(KC % NCH == 0, "the chunks of a row of G split the segments evenly");
  static constexpr int N = 6 * KC;             // variables per axis
  static constexpr int CH = N / NCH;           // columns of G per thread
  static constexpr int KB = KC / NCH;          // segments per chunk
  static constexpr int ROWS = 21 * KC;         // constraint rows per axis
  static constexpr int NN = 18 * KC;           // difference rows (containment, velocity, acceleration, jerk)
  static constexpr int NJ = 3 * KC;            // continuity / initial-state rows
  static constexpr int TA = ((NCH * N + 31) / 32) * 32;  // threads per axis problem
  static constexpr int NWARPS = 2 * TA / 32;             // warps per CTA
  // row slots.  NCH = 2: threads [T0, TA) own two difference rows (slots A, B), threads [0, T0) one difference row
  // (slot A) and, below NJ, one continuity row (slot J).  NCH = 4: thread t owns difference row t (t < NN) or
  // continuity row t - NN.
  static constexpr bool TWO_SLOTS = NCH == 2;
  static constexpr int T0 = TWO_SLOTS ? ((NJ + 31) / 32) * 32 : 0;
  static constexpr int TN = TA - T0;
  // row slots per thread.  Chunked layouts (NCH = 2, 4): 3 (difference rows A, B and one continuity row J).  Full-row layout: NDS slots of
  // difference rows and NJS slots of continuity / init rows, so that every slot is one kind of row on all threads.
  static constexpr int NDS = (NN + TA - 1) / TA;   // full-row layout: slots of difference rows (slot s = row s TA + t) ...
  static constexpr int NJS = (NJ + TA - 1) / TA;   // ... followed by slots of continuity / initial-state rows
  static constexpr int NSLOT = ROWFULL ? NDS + NJS : 3;
  static_assert(ROWFULL || (TWO_SLOTS ? (2 * TN + T0 >= NN) : (TA >= ROWS)), "row slots");
  static constexpr int LPA = KC <= 8 ? 8 : 16; // lanes per axis of the lane-per-segment (control) code
  static constexpr int STR = LPA;              // its shared-memory stride
  // per-axis shared memory (doubles)
  static constexpr int O_CTRL = 0;                                   // W, L, U, RHO, P slots of qp.cuh
  static constexpr int O_FS = O_CTRL + QP_SM_DOUBLES_PER_LANE * STR; // factor store [LPA][57]
  static constexpr int O_LS = O_FS + 57 * LPA;                       // lane state [LPA][QPD_LS]
  static constexpr int O_V = O_LS + QPD_LS * LPA;                    // V[(KC+1)][QPD_VB]
  static constexpr int O_GV = O_V + QPD_VB * (KC + 1);               // g[N]  (even offset: 16-byte aligned)
  static constexpr int O_C = O_GV + N;                               // x~: QPD_CP pads + N + pads
  static constexpr int O_XR = O_C + N + 8;                           // relaxed x for the checks, same shape
  static constexpr int O_CE = O_XR + N + 8;                          // continuity row coefficients [3KC][6]
  static constexpr int O_VCF = O_CE + 18 * KC;                       // continuity gather coefficients [N][3]
  static constexpr int O_LU = ((O_VCF + 3 * N + 1) / 2) * 2;         // (l, u) of the row slots [NSLOT][TA] pairs (16-byte aligned)
  static constexpr int O_V2 = O_LU + 2 * NSLOT * TA;                 // second row-value array (checks: y next to delta y)
  static constexpr int AXIS = O_V2 + ((QPD_VB * (KC + 1) + 1) / 2) * 2;       // doubles per axis (even)
  // per-CTA tail: reduction scratch [NWARPS][QPD_NRED], eqmask ints [2][LPA]
  static constexpr int O_RED = 2 * AXIS;
  static constexpr int O_EQ = O_RED + NWARPS * QPD_NRED;
  // with LPA = 8 the upper half of warp 0 holds no problem: its lanes run the lane-per-segment code on a
  // scratch copy of the control slots so that they never touch the real ones
  static constexpr int O_DUMMY = O_EQ + LPA;  // (2 * LPA ints before it)
  // one scratch copy per idle lane group (32 / LPA - 2 of them), so that no two threads ever touch the same address
  static constexpr int DUMMY_GROUPS = 2 * LPA < 32 ? 32 / LPA - 2 : 0;
  static constexpr int TOTAL = O_DUMMY + DUMMY_GROUPS * QP_SM_DOUBLES_PER_LANE * STR;
  static constexpr int BYTES = TOTAL * 8;
};

// 16-byte shared-memory load as an ordered (volatile) statement: a run of these is issued back to back, so their
// latencies overlap instead of each load being consumed before the next one is issued
SP_DEV void qpd_lds2(const double *p, double &a, double &b) {
#ifdef SPECTRAL_CPU_EMU
  a = p[0]; b = p[1];
#else
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "r"((unsigned)__cvta_generic_to_shared(p)));
#endif
}
template <bool ON>
SP_DEV void qpd_sched_fence_if() {
#ifndef SPECTRAL_CPU_EMU
  if (ON) asm volatile("fence.acq_rel.cta;" ::: "memory");
#endif
}
SP_DEV void qpd_sched_fence() {
#ifndef SPECTRAL_CPU_EMU
  asm volatile("fence.acq_rel.cta;" ::: "memory");
#endif
}
// clip(w, [l, u]) as two compare-selects (fmin/fmax expand to NaN-propagation sequences four times as long)
SP_DEV double qpd_clip(double w, double l, double u) {
  const double a = w < l ? l : w;
  return a > u ? u : a;
}

// (A' V)_v for variable (k, j): vb = V block of segment k, vk = V block holding the continuity rows that
// touch this variable (own segment for j < 3, next segment for j >= 3), vc = their three coefficients
SP_DEV double qpd_gather(const double *vb, const double *vk, int j, double tk, double vc0, double vc1, double vc2) {
  double g = tk * vb[QPD_V0 + j];
  g += 5.0 * (vb[QPD_V1 + j - 1] - vb[QPD_V1 + j]);
  g += 20.0 * ((vb[QPD_V2 + j - 2] - vb[QPD_V2 + j - 1]) - (vb[QPD_V2 + j - 1] - vb[QPD_V2 + j]));
  const double a0 = vb[QPD_V3 + j - 3], a1 = vb[QPD_V3 + j - 2], a2 = vb[QPD_V3 + j - 1], a3 = vb[QPD_V3 + j];
  g += 60.0 * ((a0 - a3) + 3.0 * (a2 - a1));
  g += vc0 * vk[QPD_VC] + vc1 * vk[QPD_VC + 1] + vc2 * vk[QPD_VC + 2];
  return g;
}

// difference rows: order-d finite difference of the control points at cp, d = 0..3 (solve_3d.cc:823-888):
//   containment t c_i | velocity 5 (c_{i+1} - c_i) | acceleration 20 (c_i - 2 c_{i+1} + c_{i+2}) | jerk 60 (...)
// One code path for all four: the window cp[0..3] is always read (the arrays are padded), the order selects.
SP_DEV double qpd_diff_row(const double *cp, int order, double scale) {
  const double c0 = cp[0], c1 = cp[1], c2 = cp[2], c3 = cp[3];
  const double d1 = c1 - c0, e1 = c2 - c1, f1 = c3 - c2;
  const double d2 = e1 - d1, e2 = f1 - e1;
  const double d3 = e2 - d2;
  const double lo = order == 0 ? c0 : d1, hi = order == 2 ? d2 : d3;
  return scale * (order < 2 ? lo : hi);
}
// continuity / initial-state rows (solve_3d.cc:896-949): six coefficients on [c_{k-1,3..5}, c_{k,0..2}]
SP_DEV double qpd_join_row(const double *cp, const double *ce) {
  return (ce[0] * cp[0] + ce[1] * cp[1]) + (ce[2] * cp[2] + ce[3] * cp[3]) + (ce[4] * cp[4] + ce[5] * cp[5]);
}

struct QpdLU { double l, u; };
struct QpdRow {
  double w, p, rho;        // w = z + y / rho, p = clip(w, l, u); (l, u) live in shared memory (QpdLayout::O_LU)
  double scale;            // difference rows: t_k, 5, 20 or 60
  int coff;                // offset of the stencil window in C / XR
  int voff;                // offset of this row's value in V
  int meta;                // bits 0-1 difference order, bit 3 valid, bit 4 equality row, bits 8-15 segment, 16.. row in slots (r)
  double er, ier;          // Ruiz row scaling E_r = sqrt(rho_r c / (rhobar eqfac)) and 1 / E_r: invariant under adaptive rho (checks only)
};

// Chunk h of row v of G = S^-1: the NCH threads (v, 0..NCH-1), adjacent lanes, run the block forward / backward
// substitution of qp.cuh's factor (read from shared memory, broadcast) on e_v, each on its own KC/NCH segments,
// handing the 3-value carry to the neighbour lane by shuffle.
template <int KC>
SP_DEV void qpd_inverse_chunk(const double *fs, int v, int h, double *g) {
  constexpr int KB = QpdLayout<KC>::KB, NCH = QpdLayout<KC>::NCH;
  const int kv = v / 6, iv = v - 6 * kv;
  const int kbase = h * KB;
  double c3 = 0.0, c4 = 0.0, c5 = 0.0;  // y_{k-1}[3..5]
#pragma unroll
  for (int phase = 0; phase < NCH; phase++) {
    if (h == phase) {
#pragma unroll
      for (int kb = 0; kb < KB; kb++) {
        const int k = kbase + kb;
        const double *F = fs + 57 * k;
#pragma unroll
        for (int a = 0; a < 6; a++) {
          double y = 0.0;
          if (k == kv && a >= iv) y = F[LT(a, 0) + iv];
          y -= F[21 + a * 3 + 0] * c3 + F[21 + a * 3 + 1] * c4 + F[21 + a * 3 + 2] * c5;  // C_0 = 0
          g[6 * kb + a] = y;
        }
        c3 = g[6 * kb + 3]; c4 = g[6 * kb + 4]; c5 = g[6 * kb + 5];
      }
    }
    if (phase + 1 < NCH) {  // lane h + 1 takes over with lane h's carry
      const double t3 = sp_shfl_up(c3, 1, NCH), t4 = sp_shfl_up(c4, 1, NCH), t5 = sp_shfl_up(c5, 1, NCH);
      if (h == phase + 1) { c3 = t3; c4 = t4; c5 = t5; }
    }
  }
  double n0 = 0.0, n1 = 0.0, n2 = 0.0;  // x_{k+1}[0..2]
#pragma unroll
  for (int phase = NCH - 1; phase >= 0; phase--) {
    if (h == phase) {
#pragma unroll
      for (int kb = KB - 1; kb >= 0; kb--) {
        const int k = kbase + kb;
        const double *F = fs + 57 * k;
#pragma unroll
        for (int i = 0; i < 6; i++) {
          double x = 0.0;
#pragma unroll
          for (int a = i; a < 6; a++) x += F[LT(a, i)] * g[6 * kb + a];
          x -= F[39 + i * 3 + 0] * n0 + F[39 + i * 3 + 1] * n1 + F[39 + i * 3 + 2] * n2;  // E of the last segment = 0
          g[6 * kb + i] = x;
        }
        n0 = g[6 * kb + 0]; n1 = g[6 * kb + 1]; n2 = g[6 * kb + 2];
      }
    }
    if (phase > 0) {  // lane h - 1 takes over with lane h's x
      const double t0 = sp_shfl_down(n0, 1, NCH), t1 = sp_shfl_down(n1, 1, NCH), t2 = sp_shfl_down(n2, 1, NCH);
      if (h == phase - 1) { n0 = t0; n1 = t1; n2 = t2; }
    }
  }
}

// thread -> (variable v, chunk h) of the G layout; threads beyond NCH N hold nothing (v = N)
template <int KC>
SP_DEV void qpd_map(int ta, int &v, int &h) {
  v = ta / QpdLayout<KC>::NCH; h = ta % QpdLayout<KC>::NCH;
}

// CTA-wide reduction of QPD_NRED values: slots 0..8 max (of non-negative norms), slot 9 sum.  All threads return the
// result in r[].  Two levels, both inside a warp: every warp reduces its lanes, lane 0 publishes the ten values, then
// every warp reduces the per-warp values (lane w reads warp w's) -- no serial loop over the warps, no fmax sequences.
// The sum is a fixed shuffle tree on both levels, so the result does not depend on scheduling.
template <typename SyncFn>
SP_DEV void qpd_reduce(double r[QPD_NRED], double *red, int warp, int lane, int nwarps, SyncFn sync_cta) {
#pragma unroll
  for (int i = 0; i < QPD_NRED - 1; i++) r[i] = sp_warp_max_nonneg(r[i]);
  r[QPD_NRED - 1] = sp_group_sum(r[QPD_NRED - 1], 32);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < QPD_NRED; i++) red[warp * QPD_NRED + i] = r[i];
  }
  sync_cta();
  const double *mine = red + (lane < nwarps ? lane : 0) * QPD_NRED;
#pragma unroll
  for (int i = 0; i < QPD_NRED - 1; i++) r[i] = sp_warp_max_nonneg(lane < nwarps ? mine[i] : 0.0);
  r[QPD_NRED - 1] = sp_group_sum(lane < nwarps ? mine[QPD_NRED - 1] : 0.0, 32);
  sync_cta();  // red[] may be reused
}

// warp 0: (re)factorise S for the current RHO slots and publish the factor; returns bad pivot flag (joint)
template <int KC>
SP_DEV_NOINLINE int qpd_refactor(double *smc, double *fs, const QpLane &Q, bool publish) {
  constexpr int LPA = QpdLayout<KC>::LPA, STR = QpdLayout<KC>::STR;
  QpFactor F;
  int bad = qp_factorize<LPA, STR>(smc, Q.seg, QP_SM_RHO, Q.sig, Q.t, Q.tp, Q.tn, Q.first, Q.last, Q.active, Q.seg, Q.kmaxw, 0u,
                                   Q.eqmask, 0.0, F);
  bad = sp_group_or(bad, 2 * LPA);
  if (publish) {
    double *dst = fs + 57 * Q.seg;
#pragma unroll
    for (int e = 0; e < 21; e++) dst[e] = F.Linv[e];
#pragma unroll
    for (int e = 0; e < 18; e++) { dst[21 + e] = F.C[e]; dst[39 + e] = F.E[e]; }
  }
  return bad;
}

SP_DEV void qpd_store_lane(const QpLane &Q, double *ls, int *eq) {
  double *d = ls + QPD_LS * Q.seg;
  d[0] = Q.t; d[1] = Q.tp; d[2] = Q.tn;
#pragma unroll
  for (int j = 0; j < 6; j++) { d[3 + j] = Q.q[j]; d[9 + j] = Q.sig[j]; d[15 + j] = Q.cD[j]; }
  eq[Q.seg] = (int)Q.eqmask;
}

// rebuilds the lane state of a control lane from shared memory (everything but c / rhobar, passed in)
SP_DEV void qpd_load_lane(QpLane &Q, const QpArgs &a, int ap, int seg, const double *ls, const int *eq, double c, double rhobar,
                          bool real) {
  Q.b = a.list[ap >> 1]; Q.axis = ap & 1; Q.K = a.K[Q.b]; Q.seg = seg; Q.kmaxw = Q.K;
  Q.have = real; Q.active = real && seg < Q.K; Q.first = seg == 0; Q.last = seg == Q.K - 1;
  const double *d = ls + QPD_LS * seg;
  Q.t = d[0]; Q.tp = d[1]; Q.tn = d[2];
#pragma unroll
  for (int j = 0; j < 6; j++) { Q.q[j] = d[3 + j]; Q.sig[j] = d[9 + j]; Q.cD[j] = d[15 + j]; }
  Q.c = c; Q.rhobar = rhobar; Q.eqmask = (unsigned)eq[seg]; Q.pre = 0; Q.xch = nullptr;
}

// warp 0: K3 assembly, Ruiz scaling, per-row rho, stencil tables, first factorisation.
// Publishes (c, state) in red[0..1].
template <int KC>
SP_DEV_NOINLINE void qpd_control_setup(const QpArgs &a, int slot, int lane, double *smem) {
  using L = QpdLayout<KC>;
  constexpr int LPA = L::LPA, STR = L::STR, JW = 2 * L::LPA;
  double *red = smem + L::O_RED;
  int *eqm = (int *)(smem + L::O_EQ);
  const int cgrp = lane / LPA, cseg = lane % LPA, caxis = cgrp & 1;
  const bool creal = lane < JW;  // lanes beyond the two axis groups idle on scratch slots
  double *smc = creal ? smem + caxis * L::AXIS + L::O_CTRL : smem + L::O_DUMMY + (cgrp - 2) * QP_SM_DOUBLES_PER_LANE * STR;
  double *cfs = smem + caxis * L::AXIS + L::O_FS;
  double *cls = smem + caxis * L::AXIS + L::O_LS;
  int *ceq = eqm + caxis * LPA;
  const int cap = 2 * slot + caxis;
  (void)red; (void)cfs; (void)cls; (void)ceq; (void)cap; (void)smc; (void)cseg; (void)STR;
  int state = QP_RUNNING;
  {
    QpLane Q;
    qp_setup<LPA, STR, JW>(a, cap, creal, cseg, cseg, smc, Q);
    if (creal) qpd_store_lane(Q, cls, ceq);
    if (creal && cseg < KC) {
      // stencil tables of the dense loop: continuity row coefficients, continuity gather coefficients
      double *ce = smem + caxis * L::AXIS + L::O_CE + 18 * cseg;
      double *vcf = smem + caxis * L::AXIS + L::O_VCF + 18 * cseg;
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int j = 0; j < 3; j++) {
          ce[6 * r + j] = Q.active ? prev_coef(18 + r, j, Q.t, Q.tp, Q.first) : 0.0;
          ce[6 * r + 3 + j] = Q.active ? row_coef(18 + r, j, Q.t, Q.tp, Q.first) : 0.0;
          vcf[3 * j + r] = Q.active ? row_coef(18 + r, j, Q.t, Q.tp, Q.first) : 0.0;                          // own rows, j < 3
          vcf[3 * (3 + j) + r] = (Q.active && !Q.last) ? prev_coef(18 + r, j, Q.tn, Q.t, false) : 0.0;       // next segment's rows
        }
    }
    const int bad = qpd_refactor<KC>(smc, cfs, Q, creal);
    if (bad || Q.pre) state = QP_ST_INFEASIBLE;  // Q.pre of lane 0 = OR over both axes of the scenario
    if (lane == 0) { red[0] = Q.c; red[1] = (double)state; }
  }
}

// warp 0: adaptive-rho refactorisation; publishes the bad-pivot flag in red[0]
template <int KC>
SP_DEV_NOINLINE void qpd_control_refactor(const QpArgs &a, int slot, int lane, double *smem, double c_scale, double rhobar) {
  using L = QpdLayout<KC>;
  constexpr int LPA = L::LPA, STR = L::STR, JW = 2 * L::LPA;
  double *red = smem + L::O_RED;
  int *eqm = (int *)(smem + L::O_EQ);
  const int cgrp = lane / LPA, cseg = lane % LPA, caxis = cgrp & 1;
  const bool creal = lane < JW;  // lanes beyond the two axis groups idle on scratch slots
  double *smc = creal ? smem + caxis * L::AXIS + L::O_CTRL : smem + L::O_DUMMY + (cgrp - 2) * QP_SM_DOUBLES_PER_LANE * STR;
  double *cfs = smem + caxis * L::AXIS + L::O_FS;
  double *cls = smem + caxis * L::AXIS + L::O_LS;
  int *ceq = eqm + caxis * LPA;
  const int cap = 2 * slot + caxis;
  (void)red; (void)cfs; (void)cls; (void)ceq; (void)cap; (void)smc; (void)cseg; (void)STR;
  QpLane Q;
  qpd_load_lane(Q, a, cap, cseg, cls, ceq, c_scale, rhobar, creal);
  const int bad = qpd_refactor<KC>(smc, cfs, Q, creal);
  if (lane == 0) red[0] = (double)bad;
}

// warp 0: final status at max_iter, polish, outputs (qp_finish of qp.cuh)
template <int KC>
SP_DEV_NOINLINE void qpd_control_finish(const QpArgs &a, int slot, int lane, double *smem, double c_scale, double rhobar, int state,
                                        int iters) {
  using L = QpdLayout<KC>;
  constexpr int LPA = L::LPA, STR = L::STR, JW = 2 * L::LPA;
  double *red = smem + L::O_RED;
  int *eqm = (int *)(smem + L::O_EQ);
  const int cgrp = lane / LPA, cseg = lane % LPA, caxis = cgrp & 1;
  const bool creal = lane < JW;  // lanes beyond the two axis groups idle on scratch slots
  double *smc = creal ? smem + caxis * L::AXIS + L::O_CTRL : smem + L::O_DUMMY + (cgrp - 2) * QP_SM_DOUBLES_PER_LANE * STR;
  double *cfs = smem + caxis * L::AXIS + L::O_FS;
  double *cls = smem + caxis * L::AXIS + L::O_LS;
  int *ceq = eqm + caxis * LPA;
  const int cap = 2 * slot + caxis;
  (void)red; (void)cfs; (void)cls; (void)ceq; (void)cap; (void)smc; (void)cseg; (void)STR;
  QpLane Q;
  qpd_load_lane(Q, a, cap, cseg, cls, ceq, c_scale, rhobar, creal);
  double x[6];
  const double *xs = smem + caxis * L::AXIS + L::O_XR + QPD_CP + 6 * (cseg < KC ? cseg : 0);
#pragma unroll
  for (int j = 0; j < 6; j++) x[j] = (creal && cseg < KC) ? xs[j] : 0.0;
  qp_finish<LPA, STR, JW>(a, smc, cseg, Q, x, creal ? state : QP_ST_MAXITER, iters);
}

// ------------------------------------------------------------------ the CTA body
// decode a difference-row index e in [0, 18 KC): order (0 containment .. 3 jerk), segment k, index i
template <int KC>
SP_DEV void qpd_decode_diff(int e, int &order, int &k, int &i) {
  // within an order the SEGMENT index runs fastest: consecutive lanes then read stencil windows 6 doubles apart and write
  // V entries 38 doubles apart -- both = 6 mod 16, i.e. the 16 lanes of an 8-byte shared-memory wavefront hit 16 distinct
  // bank pairs (with the index i fastest the windows jump at every segment boundary and the accesses took 4 wavefronts
  // instead of 2: profiles/r1_qpd_hotloop.md)
  int ep;
  if (e < 6 * KC) { order = 0; ep = e; }
  else if (e < 11 * KC) { order = 1; ep = e - 6 * KC; }
  else if (e < 15 * KC) { order = 2; ep = e - 11 * KC; }
  else { order = 3; ep = e - 15 * KC; }
  i = ep / KC; k = ep - KC * i;
}

template <int KC>
SP_DEV_NOINLINE void qpd_build_g(const double *fs, int v, int h, bool isg, double *out) {
  double g[QpdLayout<KC>::CH];
  qpd_inverse_chunk<KC>(fs, v, h, g);
#pragma unroll
  for (int e = 0; e < QpdLayout<KC>::CH; e++) out[e] = isg ? g[e] : 0.0;
}

// initial state of a difference-row slot: e = row index in [0, 18 KC) or < 0 (no row)
template <int KC>
SP_DEV void qpd_init_diff(QpdRow &r, QpdLU &lu, int e, int K, const double *ctl, const double *lsx, const int *eqa, double c_over_rhobar) {
  using L = QpdLayout<KC>;
  constexpr int STR = L::STR;
  int order = 0, k = 0, i = 0;
  const bool valid = e >= 0 && e < L::NN;
  if (valid) qpd_decode_diff<KC>(e, order, k, i);
  const int r_old = (order == 0 ? 0 : order == 1 ? 6 : order == 2 ? 11 : 15) + i;
  const int vbase = order == 0 ? QPD_V0 : order == 1 ? QPD_V1 : order == 2 ? QPD_V2 : QPD_V3;
  const bool live = valid && k < K;  // rows of unused segments stay inert: rho = 0, v = 0
  const int ooff = r_old * STR + k;
  const int eq = live ? ((eqa[k] >> r_old) & 1) : 0;
  r.coff = QPD_CP + 6 * k + i;
  r.voff = QPD_VB * k + vbase + i;
  r.meta = order | (valid ? 8 : 0) | (eq ? 16 : 0) | (k << 8) | (r_old << 16);
  r.scale = order == 0 ? (live ? lsx[QPD_LS * k] : 0.0) : (order == 1 ? 5.0 : (order == 2 ? 20.0 : 60.0));
  r.w = 0.0; r.p = 0.0;
  lu.l = live ? ctl[QP_SM_L * STR + ooff] : -1.0;
  lu.u = live ? ctl[QP_SM_U * STR + ooff] : 1.0;
  r.rho = live ? ctl[QP_SM_RHO * STR + ooff] : 0.0;
  r.er = sqrt(r.rho * c_over_rhobar * (eq ? 1e-3 : 1.0));
  r.ier = r.er > 0.0 ? 1.0 / r.er : 0.0;
}

// initial state of a continuity / initial-state row slot: ej = row index in [0, 3 KC) or < 0 (no row)
template <int KC>
SP_DEV void qpd_init_join(QpdRow &rj, QpdLU &lu, int ej, int K, const double *ctl, const int *eqa, double c_over_rhobar) {
  using L = QpdLayout<KC>;
  constexpr int STR = L::STR;
  const bool jvalid = ej >= 0 && ej < L::NJ;
  const int k = jvalid ? ej / 3 : 0, rr = jvalid ? ej - 3 * k : 0;
  const int r_old = 18 + rr;
  const bool live = jvalid && k < K;
  const int ooff = r_old * STR + k;
  const int eq = live ? ((eqa[k] >> r_old) & 1) : 0;
  rj.coff = 6 * k;  // window [c_{k-1,3..5}, c_{k,0..2}] starts at QPD_CP + 6k - 3
  rj.voff = QPD_VB * k + QPD_VC + rr;
  rj.meta = (jvalid ? 8 : 0) | (eq ? 16 : 0) | (k << 8) | (r_old << 16);
  rj.scale = 0.0;
  rj.w = 0.0; rj.p = 0.0;
  lu.l = live ? ctl[QP_SM_L * STR + ooff] : -1.0;
  lu.u = live ? ctl[QP_SM_U * STR + ooff] : 1.0;
  rj.rho = live ? ctl[QP_SM_RHO * STR + ooff] : 0.0;
  rj.er = sqrt(rj.rho * c_over_rhobar * (eq ? 1e-3 : 1.0));
  rj.ier = rj.er > 0.0 ? 1.0 / rj.er : 0.0;
}
// a row slot of the unified numbering: [0, NN) difference rows, [NN, ROWS) continuity / initial-state rows, else none
template <int KC>
SP_DEV void qpd_init_row(QpdRow &r, QpdLU &lu, int e, int K, const double *ctl, const double *lsx, const int *eqa, double c_over_rhobar) {
  using L = QpdLayout<KC>;
  if (e >= L::NN && e < L::ROWS) qpd_init_join<KC>(r, lu, e - L::NN, K, ctl, eqa, c_over_rhobar);
  else qpd_init_diff<KC>(r, lu, e < L::NN ? e : -1, K, ctl, lsx, eqa, c_over_rhobar);
}
SP_DEV bool qpd_row_is_join(const QpdRow &r) { return (r.meta >> 16) >= 18; }
// (A x)_row for any row slot: xbase = the padded control-point array (C or XR) of the axis
template <int KC>
SP_DEV double qpd_row_eval(const QpdRow &r, const double *xbase, const double *smx) {
  using L = QpdLayout<KC>;
  if (qpd_row_is_join(r)) {
    const double *cej = smx + L::O_CE + 6 * (3 * ((r.meta >> 8) & 0xff) + ((r.meta >> 16) - 18));
    return qpd_join_row(xbase + r.coff, cej);
  }
  return qpd_diff_row(xbase + r.coff, r.meta & 3, r.scale);
}

// max as one compare-select (fmax expands to a NaN-propagation sequence four times as long); a NaN in b is dropped
SP_DEV double qpd_max(double a, double b) { return b > a ? b : a; }
// check iterations: delta y of a row -> V, its scaled norm (red_v[7]) and the support-function term (red_v[9])
SP_DEV void qpd_check_dy(const QpdRow &r, const QpdLU &b, double yo, double *vv, double c_scale, double c_over_rhobar, double *red_v) {
  if (!(r.meta & 8)) return;
  const double dy = r.rho * (r.w - r.p) - yo;
  vv[r.voff] = dy;
  if (r.rho > 0.0) {
    red_v[7] = qpd_max(red_v[7], fabs(c_scale * dy * r.ier));
    red_v[9] += c_scale * (b.u * qpd_max(dy, 0.0) + b.l * (dy < 0.0 ? dy : 0.0));
  }
}
// check iterations: primal residual terms of a row, ax = (A x)_row
SP_DEV void qpd_check_resid(const QpdRow &r, double ax, double c_over_rhobar, double *red_v) {
  if (!(r.meta & 8) || !(r.rho > 0.0)) return;
  const double Er = r.er;
  red_v[0] = qpd_max(red_v[0], Er * fabs(ax - r.p));
  red_v[2] = qpd_max(red_v[2], Er * fabs(r.p));
  red_v[3] = qpd_max(red_v[3], Er * fabs(ax));
}
// adaptive rho: keep (z, y), w' = z + y / rho'; publish the new rho in the lane-per-segment RHO slots
SP_DEV void qpd_rescale_row(QpdRow &r, double ratio, int K, double *ctl_rho, int str) {
  if (!(r.meta & 8)) return;
  r.w = r.p + (r.w - r.p) / ratio;  // (rare: only when rho is re-tuned)
  r.rho *= ratio;
  const int k = (r.meta >> 8) & 0xff;
  if (k < K) ctl_rho[(r.meta >> 16) * str + k] = r.rho;
}
SP_DEV void qpd_handback_row(const QpdRow &r, int K, double *ctl, int str) {
  const int k = (r.meta >> 8) & 0xff;
  if (!(r.meta & 8) || k >= K) return;
  const int ooff = (r.meta >> 16) * str + k;
  ctl[QP_SM_W * str + ooff] = r.w;
  ctl[QP_SM_RHO * str + ooff] = r.rho;
}

// one ADMM row update: w += alpha (z~ - clip(w)); returns v = rho (2 clip(w) - w) of the new w
SP_DEV double qpd_row_update(QpdRow &r, const QpdLU &b, double zt, double alpha) {
  const double wn = r.w + alpha * (zt - r.p);
  const double pn = qpd_clip(wn, b.l, b.u);
  r.w = wn; r.p = pn;
  return r.rho * (2.0 * pn - wn);
}

// The per-thread state of the dense loop.  It lives in local memory in the CTA body; qpd_block loads what it needs
// into registers for a block of iterations, qpd_check / qpd_build_g work on it in place.
template <int CHN, int NS = 3>
struct QpdIOT {
  double G[CHN];    // this thread's chunk of its row of G = S^-1
  QpdRow rows[NS];  // row slots (chunked layouts: difference rows A, B and continuity row J); unused ones have meta bit 3 clear
  double yo[NS];    // multipliers before the check iteration's update
  double xv, sigv, qv, tkv;  // variable thread: relaxed iterate, sigma, q, segment duration
  double c_scale, rhobar;
  int state, need_g, it;
};

// A block of `n` ADMM iterations in the fast layout (3 CTA barriers each), out of line: only the hot state is live.
//   S2  g = A' v + sigma x - q              (V holds v = rho (2 clip(w) - w); zeros on the cold start)
//   S3  x~ = G g (one chunk of the row per thread, the partner lanes hold the others), x = alpha x~ + (1 - alpha) x
//   S1  z~ = A x~ (stencils), w += alpha (z~ - clip(w)), next v -> V
template <int KC, typename SyncFn>
SP_DEV_NOINLINE void qpd_block(QpdIOT<QpdLayout<KC>::CH, QpdLayout<KC>::NSLOT> &io, double *smx, int ta, int n, double alpha, SyncFn sync_cta) {
  using L = QpdLayout<KC>;
  constexpr int N = L::N, CH = L::CH, TA = L::TA;
  const int v = ta / L::NCH, h = ta % L::NCH;
  const bool isg = v < N;
  const bool isvar = isg && h == 0;
  const int vk = isg ? v / 6 : 0, vj = isg ? v - 6 * vk : 0;
  const double *vb = smx + L::O_V + QPD_VB * vk;
  const double *vkk = smx + L::O_V + QPD_VB * (vj < 3 ? vk : vk + 1);
  const double *vcf = smx + L::O_VCF + 3 * (isg ? v : 0);  // continuity gather coefficients (zero for unused segments)
  double *gvp = smx + L::O_GV + (isg ? v : 0);
  const double *gvh = smx + L::O_GV + CH * h;
  double *cx = smx + L::O_C;
  double *cxp = cx + QPD_CP + (isg ? v : 0);
  double *vv = smx + L::O_V;
  const QpdLU *lua = (const QpdLU *)(smx + L::O_LU) + ta, *lub = lua + TA, *luj = lub + TA;
  // second slot of the thread: difference row B (threads >= T0) or continuity row J (threads < T0), never both
  const bool second_is_b = L::TWO_SLOTS && ta >= L::T0;
  const int i2 = second_is_b ? 1 : 2;
  QpdRow ra = io.rows[0], r2 = io.rows[i2];
  const double *cej = smx + L::O_CE + 6 * ((!second_is_b && (r2.meta & 8)) ? 3 * ((r2.meta >> 8) & 0xff) + ((r2.meta >> 16) - 18) : 0);
  const double *cpa = cx + ra.coff, *cp2 = cx + r2.coff;  // stencil windows of the row slots
  double *vpa = vv + ra.voff, *vp2 = vv + r2.voff;        // their V entries
  const QpdLU *lu2 = second_is_b ? lub : luj;
  const bool va = ra.meta & 8, v2 = r2.meta & 8;
  const int oa = ra.meta & 3, ob = r2.meta & 3;
  double xv = io.xv;
  const double sigv = io.sigv, qv = io.qv, tkv = io.tkv;
  double G[CH];
#pragma unroll
  for (int e = 0; e < CH; e++) G[e] = io.G[e];
  // where the register budget allows, the (l, u) pairs of both slots stay in registers for the whole block
  constexpr bool LU_REG = L::LU_REG;
  const QpdLU la_r = lua[0], l2_r = lu2[0];
  double yoa = 0.0, yo2 = 0.0;
  for (int i = 0; i < n; i++) {
    if (i == n - 1) { yoa = ra.rho * (ra.w - ra.p); yo2 = r2.rho * (r2.w - r2.p); }
    if (isvar) {  // S2: the 13 loads of the gather in one run, then the arithmetic of qpd_gather
      const double g0 = vb[QPD_V0 + vj], g1a = vb[QPD_V1 + vj - 1], g1b = vb[QPD_V1 + vj];
      const double g2a = vb[QPD_V2 + vj - 2], g2b = vb[QPD_V2 + vj - 1], g2c = vb[QPD_V2 + vj];
      const double g3a = vb[QPD_V3 + vj - 3], g3b = vb[QPD_V3 + vj - 2], g3c = vb[QPD_V3 + vj - 1], g3d = vb[QPD_V3 + vj];
      const double c0 = vkk[QPD_VC], c1 = vkk[QPD_VC + 1], c2 = vkk[QPD_VC + 2];
      const double f0 = vcf[0], f1 = vcf[1], f2 = vcf[2];  // (hoisting these into registers too costs more than it saves: 10.5 -> 11.4 ms)
      qpd_sched_fence_if<L::STAGE_ROWS>();
      double g = tkv * g0;
      g += 5.0 * (g1a - g1b);
      g += 20.0 * ((g2a - g2b) - (g2b - g2c));
      g += 60.0 * ((g3a - g3d) + 3.0 * (g3c - g3b));
      g += f0 * c0 + f1 * c1 + f2 * c2;
      *gvp = g + sigv * xv - qv;
    }
    sync_cta();
    {
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
      static_assert(CH % 4 == 0, "g chunks are loaded in 16-byte pairs and summed in four chains");
      // the g chunk: a run of loads, a scheduling fence where the register budget allows (L::STAGE), the FMAs (ptxas
      // otherwise consumes each load before issuing the next)
      double gl[CH];
#pragma unroll
      for (int e = 0; e < CH; e += 2) qpd_lds2(gvh + e, gl[e], gl[e + 1]);
      qpd_sched_fence_if<L::STAGE>();
#pragma unroll
      for (int e = 0; e < CH; e += 4) {
        a0 += G[e] * gl[e]; a1 += G[e + 1] * gl[e + 1]; a2 += G[e + 2] * gl[e + 2]; a3 += G[e + 3] * gl[e + 3];
      }
      double xt = (a0 + a1) + (a2 + a3);
      xt += sp_shfl_xor(xt, 1);
      if (L::NCH == 4) xt += sp_shfl_xor(xt, 2);
      if (isvar) {
        xv = alpha * xt + (1.0 - alpha) * xv;
        *cxp = xt;
      }
    }
    sync_cta();
    // S1: the two row slots of a thread as one straight-line stream (loads of both first, then both updates), chosen by a
    // warp-uniform branch: threads >= T0 own two difference rows, threads < T0 a difference row and a continuity row.
    // Slots without a row compute on valid dummy addresses and skip the store.
    if (second_is_b) {
      const double a0 = cpa[0], a1 = cpa[1], a2 = cpa[2], a3 = cpa[3];
      const double b0 = cp2[0], b1 = cp2[1], b2 = cp2[2], b3 = cp2[3];
      const QpdLU la = LU_REG ? la_r : lua[0], lb = LU_REG ? l2_r : lu2[0];
      qpd_sched_fence_if<L::STAGE_ROWS>();
      const double wa[4] = {a0, a1, a2, a3}, wb[4] = {b0, b1, b2, b3};
      const double za = qpd_diff_row(wa, oa, ra.scale), zb = qpd_diff_row(wb, ob, r2.scale);
      const double ua = qpd_row_update(ra, la, za, alpha), ub = qpd_row_update(r2, lb, zb, alpha);
      if (va) *vpa = ua;
      if (v2) *vp2 = ub;
    } else {
      const double a0 = cpa[0], a1 = cpa[1], a2 = cpa[2], a3 = cpa[3];
      const double j0 = cp2[0], j1 = cp2[1], j2 = cp2[2], j3 = cp2[3], j4 = cp2[4], j5 = cp2[5];
      const double e0 = cej[0], e1 = cej[1], e2 = cej[2], e3 = cej[3], e4 = cej[4], e5 = cej[5];
      const QpdLU la = LU_REG ? la_r : lua[0], lj = LU_REG ? l2_r : lu2[0];
      qpd_sched_fence_if<L::STAGE_ROWS>();
      const double wa[4] = {a0, a1, a2, a3};
      const double za = qpd_diff_row(wa, oa, ra.scale);
      const double zj = (e0 * j0 + e1 * j1) + (e2 * j2 + e3 * j3) + (e4 * j4 + e5 * j5);
      const double ua = qpd_row_update(ra, la, za, alpha), uj = qpd_row_update(r2, lj, zj, alpha);
      if (va) *vpa = ua;
      if (v2) *vp2 = uj;
    }
    sync_cta();
  }
  io.rows[0].w = ra.w; io.rows[0].p = ra.p;
  io.rows[i2].w = r2.w; io.rows[i2].p = r2.p;
  io.yo[0] = yoa; io.yo[1] = 0.0; io.yo[2] = 0.0; io.yo[i2] = yo2;
  io.xv = xv;
}

// The NCH = 4 form of qpd_block: a thread is (v, h) = quarter row h of G for variable v in S3, one term of the
// variable's gather in S2 (all lanes busy: the same four-load / four-FMA stream with per-thread coefficients, summed by
// two butterfly shuffles) and exactly ONE constraint row in S1 (difference row ta < NN, continuity row NN <= ta < ROWS).
//   h = 0: t_k V0[j] + 5 (V1[j-1] - V1[j]) + sigma x - q      h = 1: 20 (V2[j-2] - 2 V2[j-1] + V2[j])
//   h = 2: 60 (V3[j-3] - 3 V3[j-2] + 3 V3[j-1] - V3[j])        h = 3: the three continuity rows that touch the variable
template <int KC, typename SyncFn>
SP_DEV_NOINLINE void qpd_block4(QpdIOT<QpdLayout<KC>::CH, QpdLayout<KC>::NSLOT> &io, double *smx, int ta, int n, double alpha, SyncFn sync_cta) {
  using L = QpdLayout<KC>;
  constexpr int N = L::N, CH = L::CH, TA = L::TA;
  static_assert(L::NCH == 4 && !L::TWO_SLOTS, "one row per thread");
  const int v = ta >> 2, h = ta & 3;
  const bool isg = v < N;
  const bool isvar = isg && h == 0;
  const int vk = isg ? v / 6 : 0, vj = isg ? v - 6 * vk : 0;
  const double *vb = smx + L::O_V + QPD_VB * vk;
  double *gvp = smx + L::O_GV + (isg ? v : 0);
  const double *gvh = smx + L::O_GV + CH * h;
  double *cxp = smx + L::O_C + QPD_CP + (isg ? v : 0);
  const double *gp0 = vb, *gp1 = vb;
  double gc0 = 0.0, gc1 = 0.0, gc2 = 0.0, gc3 = 0.0;
  if (isg) {
    if (h == 0) { gp0 = vb + QPD_V0 + vj; gp1 = vb + QPD_V1 + vj - 1; gc0 = io.tkv; gc1 = 5.0; gc2 = -5.0; }
    else if (h == 1) { gp1 = vb + QPD_V2 + vj - 2; gc1 = 20.0; gc2 = -40.0; gc3 = 20.0; }
    else if (h == 2) { gp0 = vb + QPD_V3 + vj - 3; gp1 = gp0 + 1; gc0 = 60.0; gc1 = -180.0; gc2 = 180.0; gc3 = -60.0; }
    else {
      const double *vcf = smx + L::O_VCF + 3 * v;  // continuity gather coefficients (zero for unused segments)
      gp1 = smx + L::O_V + QPD_VB * (vj < 3 ? vk : vk + 1) + QPD_VC; gc1 = vcf[0]; gc2 = vcf[1]; gc3 = vcf[2];
    }
  }
  // the thread's row
  const bool isj = io.rows[2].meta & 8;
  const int ri = isj ? 2 : 0;
  QpdRow r = io.rows[ri];
  const bool rvalid = r.meta & 8;
  const int order = r.meta & 3;
  const double *cp = smx + L::O_C + r.coff;
  double *vp = smx + L::O_V + r.voff;
  const QpdLU *lu = (const QpdLU *)(smx + L::O_LU) + ta + (isj ? 2 * TA : 0);
  const double *cej = smx + L::O_CE + 6 * (isj ? 3 * ((r.meta >> 8) & 0xff) + ((r.meta >> 16) - 18) : 0);
  double xv = io.xv;
  const double sigv = io.sigv, qv = io.qv;
  double G[CH];
#pragma unroll
  for (int e = 0; e < CH; e++) G[e] = io.G[e];
  double yo = 0.0;
  for (int i = 0; i < n; i++) {
    if (i == n - 1) yo = r.rho * (r.w - r.p);
    {  // S2
      const double l0 = gp0[0], l1 = gp1[0], l2 = gp1[1], l3 = gp1[2];
      double p = (gc0 * l0 + gc1 * l1) + (gc2 * l2 + gc3 * l3);
      p += sigv * xv - qv;  // zero except on the variable thread
      p += sp_shfl_xor(p, 1);
      p += sp_shfl_xor(p, 2);
      if (isvar) *gvp = p;
    }
    sync_cta();
    {  // S3
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
      static_assert(CH % 2 == 0, "g chunks are loaded in 16-byte pairs");
      double gl[CH];
#pragma unroll
      for (int e = 0; e < CH; e += 2) qpd_lds2(gvh + e, gl[e], gl[e + 1]);
#pragma unroll
      for (int e = 0; e + 3 < CH; e += 4) {
        a0 += G[e] * gl[e]; a1 += G[e + 1] * gl[e + 1]; a2 += G[e + 2] * gl[e + 2]; a3 += G[e + 3] * gl[e + 3];
      }
#pragma unroll
      for (int e = CH & ~3; e < CH; e++) a0 += G[e] * gl[e];
      double xt = (a0 + a1) + (a2 + a3);
      xt += sp_shfl_xor(xt, 1);
      xt += sp_shfl_xor(xt, 2);
      if (isvar) {
        xv = alpha * xt + (1.0 - alpha) * xv;
        *cxp = xt;
      }
    }
    sync_cta();
    if (rvalid) {  // S1
      const QpdLU b = lu[0];
      const double zt = isj ? qpd_join_row(cp, cej) : qpd_diff_row(cp, order, r.scale);
      *vp = qpd_row_update(r, b, zt, alpha);
    }
    sync_cta();
  }
  io.rows[ri].w = r.w; io.rows[ri].p = r.p;
  io.yo[0] = 0.0; io.yo[1] = 0.0; io.yo[2] = 0.0; io.yo[ri] = yo;
  io.xv = xv;
}

// The full-row form of the block (QpdLayout::ROWFULL): thread t < N is variable t and holds ROW t of G entirely; every thread
// carries NSLOT constraint rows (slot s = row s TA + t of the unified numbering).  Three barriers per iteration:
//   S2  g_t = (A' V)_t + sigma x - q          13 loads in one run, then the arithmetic
//   S3  x~_t = G[t][:] . g                     g read by every lane from the same address (one wavefront per LDS.128),
//                                               in groups of GRP doubles: loads, scheduling fence, FMAs
//   S1  the thread's rows: z~ = (A x~)_row, w += alpha (z~ - clip(w)), next v -> V; all-difference slots as one
//       straight-line stream, the slot(s) that mix difference and continuity rows behind a branch
template <int KC, typename SyncFn>
SP_DEV_NOINLINE void qpd_block1(QpdIOT<QpdLayout<KC>::CH, QpdLayout<KC>::NSLOT> &io, double *smx, int ta, int n, double alpha,
                                SyncFn sync_cta) {
  using L = QpdLayout<KC>;
  constexpr int N = L::N, TA = L::TA, NS = L::NSLOT, NN = L::NN;
  static_assert(L::ROWFULL && L::NCH == 1 && N % 4 == 0, "full-row layout");
  // doubles of g in flight per group: KC = 10 measured 8.05 ms with 12, 7.85 ms with 20, 8.2 ms with 30 (spills)
  constexpr int GRP = (N % 24 == 0) ? 24 : ((N % 20 == 0) ? 20 : 12);  // (KC = 8: 10.57 ms with 12, 10.0 ms with 24)
  static_assert(N % GRP == 0, "g in whole groups");
  constexpr int ND = L::NDS;   // slots 0 .. ND-1 hold difference rows, slots ND .. NS-1 continuity / initial-state rows
  const int v = ta;
  const bool isg = v < N;
  const int vk = isg ? v / 6 : 0, vj = isg ? v - 6 * vk : 0;
  const double *vb = smx + L::O_V + QPD_VB * vk;
  const double *vkk = smx + L::O_V + QPD_VB * (vj < 3 ? vk : vk + 1);
  const double *vcf = smx + L::O_VCF + 3 * (isg ? v : 0);  // continuity gather coefficients (zero for unused segments)
  double *gvp = smx + L::O_GV + (isg ? v : 0);
  const double *gv = smx + L::O_GV;
  double *cx = smx + L::O_C;
  double *cxp = cx + QPD_CP + (isg ? v : 0);
  double *vv = smx + L::O_V;
  const QpdLU *lu0 = (const QpdLU *)(smx + L::O_LU) + ta;
  QpdRow r[NS];
#pragma unroll
  for (int sl = 0; sl < NS; sl++) r[sl] = io.rows[sl];
  double xv = io.xv;
  const double sigv = io.sigv, qv = io.qv, tkv = io.tkv;
  double G[N];
#pragma unroll
  for (int e = 0; e < N; e++) G[e] = io.G[e];
  const double f0 = vcf[0], f1 = vcf[1], f2 = vcf[2];  // continuity gather coefficients: constants of the block
  QpdLU lub[NS];                                          // and the (l, u) pairs of the row slots
#pragma unroll
  for (int sl = 0; sl < NS; sl++) lub[sl] = lu0[sl * TA];
  double yo[NS];
#pragma unroll
  for (int sl = 0; sl < NS; sl++) yo[sl] = 0.0;
  for (int i = 0; i < n; i++) {
    if (i == n - 1) {
#pragma unroll
      for (int sl = 0; sl < NS; sl++) yo[sl] = r[sl].rho * (r[sl].w - r[sl].p);
    }
    if (isg) {  // S2
      const double g0 = vb[QPD_V0 + vj], g1a = vb[QPD_V1 + vj - 1], g1b = vb[QPD_V1 + vj];
      const double g2a = vb[QPD_V2 + vj - 2], g2b = vb[QPD_V2 + vj - 1], g2c = vb[QPD_V2 + vj];
      const double g3a = vb[QPD_V3 + vj - 3], g3b = vb[QPD_V3 + vj - 2], g3c = vb[QPD_V3 + vj - 1], g3d = vb[QPD_V3 + vj];
      const double c0 = vkk[QPD_VC], c1 = vkk[QPD_VC + 1], c2 = vkk[QPD_VC + 2];
      qpd_sched_fence();
      const double t01 = tkv * g0 + 5.0 * (g1a - g1b);
      const double t2 = 20.0 * ((g2a - g2b) - (g2b - g2c));
      const double t3 = 60.0 * ((g3a - g3d) + 3.0 * (g3c - g3b));
      const double tc = (f0 * c0 + f1 * c1) + (f2 * c2 + (sigv * xv - qv));
      *gvp = (t01 + t2) + (t3 + tc);
    }
    sync_cta();
    {  // S3
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
      for (int g0 = 0; g0 < N; g0 += GRP) {
        double gl[GRP];
#pragma unroll
        for (int e = 0; e < GRP; e += 2) qpd_lds2(gv + g0 + e, gl[e], gl[e + 1]);
        qpd_sched_fence();
#pragma unroll
        for (int e = 0; e < GRP; e += 4) {
          a0 += G[g0 + e] * gl[e]; a1 += G[g0 + e + 1] * gl[e + 1]; a2 += G[g0 + e + 2] * gl[e + 2]; a3 += G[g0 + e + 3] * gl[e + 3];
        }
      }
      const double xt = (a0 + a1) + (a2 + a3);
      if (isg) {
        xv = alpha * xt + (1.0 - alpha) * xv;
        *cxp = xt;
      }
    }
    sync_cta();
    {  // S1: every slot is one kind of row on all threads -> one straight-line stream: loads, fence, updates
      double win[ND][4], jw[NS - ND][6], jc[NS - ND][6];
#pragma unroll
      for (int sl = 0; sl < ND; sl++) {
        const double *cp = cx + r[sl].coff;
        win[sl][0] = cp[0]; win[sl][1] = cp[1]; win[sl][2] = cp[2]; win[sl][3] = cp[3];
      }
#pragma unroll
      for (int sl = ND; sl < NS; sl++) {
        const double *cp = cx + r[sl].coff;
        const double *ce = smx + L::O_CE + 6 * (3 * ((r[sl].meta >> 8) & 0xff) + (((r[sl].meta >> 16) & 0xff) - 18 > 0 ? ((r[sl].meta >> 16) & 0xff) - 18 : 0));
#pragma unroll
        for (int m = 0; m < 6; m++) { jw[sl - ND][m] = cp[m]; jc[sl - ND][m] = ce[m]; }
      }
      qpd_sched_fence();
#pragma unroll
      for (int sl = 0; sl < ND; sl++) {
        const double zt = qpd_diff_row(win[sl], r[sl].meta & 3, r[sl].scale);
        const double u = qpd_row_update(r[sl], lub[sl], zt, alpha);
        if (r[sl].meta & 8) vv[r[sl].voff] = u;
      }
#pragma unroll
      for (int sl = ND; sl < NS; sl++) {
        const double *w6 = jw[sl - ND], *c6 = jc[sl - ND];
        const double zt = (c6[0] * w6[0] + c6[1] * w6[1]) + (c6[2] * w6[2] + c6[3] * w6[3]) + (c6[4] * w6[4] + c6[5] * w6[5]);
        const double u = qpd_row_update(r[sl], lub[sl], zt, alpha);
        if (r[sl].meta & 8) vv[r[sl].voff] = u;
      }
    }
    sync_cta();
  }
#pragma unroll
  for (int sl = 0; sl < NS; sl++) { io.rows[sl].w = r[sl].w; io.rows[sl].p = r[sl].p; io.yo[sl] = yo[sl]; }
  io.xv = xv;
}

// OSQP's termination test (residuals in the scaled space, scaled_termination = 1), primal-infeasibility
// certificate and adaptive-rho rule, evaluated CTA-wide = jointly over the s and l problems of the scenario.
// Called by all threads of the CTA on check iterations.
template <int KC, typename SyncFn>
SP_DEV_NOINLINE void qpd_check(const QpArgs &a, int slot, int tid, double *smem, QpdIOT<QpdLayout<KC>::CH, QpdLayout<KC>::NSLOT> &io, SyncFn sync_cta) {
  using L = QpdLayout<KC>;
  constexpr int N = L::N, LPA = L::LPA, STR = L::STR, TA = L::TA;
  (void)LPA;
  const SpOptionsDev &o = a.opt;
  const int warp = tid >> 5, lane = tid & 31;
  const int axis = tid / TA, ta = tid - axis * TA;
  double *smx = smem + axis * L::AXIS;
  double *red = smem + L::O_RED;
  const int K = a.K[a.list[slot]];
  const double *ctl = smx + L::O_CTRL;
  const double *lsx = smx + L::O_LS;
  constexpr int NS = L::NSLOT;
  const QpdLU *lu0 = (const QpdLU *)(smx + L::O_LU) + ta;  // slot s: lu0[s * TA]
  int v, h;
  qpd_map<KC>(ta, v, h);
  const bool isg = v < N;
  const bool isvar = isg && h == 0;
  const int vk = isg ? v / 6 : 0, vj = isg ? v - 6 * vk : 0;
  const double *vb = smx + L::O_V + QPD_VB * vk;
  const double *vkk = smx + L::O_V + QPD_VB * (vj < 3 ? vk : vk + 1);
  const double *vcf = smx + L::O_VCF + 3 * (isg ? v : 0);
  double *xr = smx + L::O_XR;
  double *vv = smx + L::O_V;
  const double c_scale = io.c_scale, xv = io.xv, qv = io.qv, tkv = io.tkv;
  double rhobar = io.rhobar;
  int state = io.state;
  const int it = io.it;

  // value copies of the row slots: the shared-memory stores below go through generic pointers, and with the slots read
  // through `io` (local memory) every one of them forces the fields to be re-loaded
  QpdRow rows[NS];
  double yo_[NS];
  QpdLU lus[NS];
#pragma unroll
  for (int sl = 0; sl < NS; sl++) { rows[sl] = io.rows[sl]; yo_[sl] = io.yo[sl]; lus[sl] = lu0[sl * TA]; }
  double red_v[QPD_NRED];
#pragma unroll
  for (int i = 0; i < QPD_NRED; i++) red_v[i] = 0.0;
  const double c_over_rhobar = c_scale / rhobar;
  // One pass: delta y -> V and y -> V2 (and the relaxed x -> XR), ONE barrier, then both gathers A' delta y and A' y, P x
  // and the row residuals as independent instruction streams.
  double *vv2 = smx + L::O_V2;
#pragma unroll
  for (int sl = 0; sl < NS; sl++) {
    const QpdRow &r = rows[sl];
    qpd_check_dy(r, lus[sl], yo_[sl], vv, c_scale, c_over_rhobar, red_v);
    if (r.meta & 8) vv2[r.voff] = r.rho * (r.w - r.p);  // y
  }
  if (isvar) xr[QPD_CP + v] = xv;
  sync_cta();
  if (isvar) {
    const double cDv = vk < K ? lsx[QPD_LS * vk + 15 + vj] : 0.0;
    const double atd = qpd_gather(vb, vkk, vj, tkv, vcf[0], vcf[1], vcf[2]);
    const double aty = qpd_gather(vb + (L::O_V2 - L::O_V), vkk + (L::O_V2 - L::O_V), vj, tkv, vcf[0], vcf[1], vcf[2]);
    double px = 0.0;
    const double *pk = ctl + QP_SM_P * STR + vk;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      const int e = (i >= vj) ? LT(i, vj) : LT(vj, i);
      px += pk[e * STR] * xr[QPD_CP + 6 * vk + i];
    }
    if (vk >= K) px = 0.0;
    red_v[8] = fabs(cDv * atd);
    red_v[1] = cDv * fabs(px + qv + aty);
    red_v[4] = cDv * fabs(qv);
    red_v[5] = cDv * fabs(px);
    red_v[6] = cDv * fabs(aty);
  }
#pragma unroll
  for (int sl = 0; sl < NS; sl++) qpd_check_resid(rows[sl], qpd_row_eval<KC>(rows[sl], xr, smx), c_over_rhobar, red_v);
  qpd_reduce(red_v, red, warp, lane, L::NWARPS, sync_cta);
  const double pri = red_v[0], dua = red_v[1], nz = red_v[2], nax = red_v[3], nq = red_v[4], npx = red_v[5], naty = red_v[6];
  const double nd = red_v[7], na = red_v[8], lhs = red_v[9];
  const double eps_p = o.eps_abs + o.eps_rel * fmax(nz, nax);
  const double eps_d = o.eps_abs + o.eps_rel * fmax(nq, fmax(npx, naty));
  if (pri < eps_p && dua < eps_d) state = QP_ST_SOLVED;
  else if (!(pri < eps_p) && nd > o.eps_pinf && lhs < -o.eps_pinf * nd && na < o.eps_pinf * nd) state = QP_ST_INFEASIBLE;
  // adaptive rho (OSQP's rule, every adaptive_rho_interval iterations)
  if (state == QP_RUNNING && o.adapt_every > 0 && (it % o.adapt_every == 0)) {
    const double pr = pri / (fmax(nz, nax) + 1e-10);
    const double dr = dua / (fmax(nq, fmax(npx, naty)) + 1e-10);
    double est = rhobar * sqrt(pr / (dr + 1e-10));
    est = fmin(fmax(est, 1e-6), 1e6);
    if (est > rhobar * o.adapt_tol || est < rhobar / o.adapt_tol) {
      const double ratio = est / rhobar;
      double *ctlw = smx + L::O_CTRL;
#pragma unroll
      for (int sl = 0; sl < NS; sl++) { qpd_rescale_row(rows[sl], ratio, K, ctlw + QP_SM_RHO * STR, STR); io.rows[sl].w = rows[sl].w; io.rows[sl].rho = rows[sl].rho; }
      rhobar = est;
      sync_cta();
      if (warp == 0) qpd_control_refactor<KC>(a, slot, lane, smem, c_scale, rhobar);
      sync_cta();
      if (red[0] != 0.0) state = QP_ST_INFEASIBLE;
      io.need_g = 1;
    }
  }
  io.rhobar = rhobar;
  io.state = state;
}

// slot: index of the scenario in this class' list.  tid in [0, 2 TA).  smem: QpdLayout<KC>::BYTES, 16-byte aligned.
template <int KC, typename SyncFn>
SP_DEV void qpd_cta_body(const QpArgs &a, int slot, int tid, double *smem, SyncFn sync_cta) {
  using L = QpdLayout<KC>;
  constexpr int N = L::N, CH = L::CH, LPA = L::LPA, STR = L::STR, TA = L::TA;
  if (slot >= *a.count) return;
  const SpOptionsDev &o = a.opt;
  const int warp = tid >> 5, lane = tid & 31;
  const int axis = tid / TA, ta = tid - axis * TA;
  double *smx = smem + axis * L::AXIS;  // this thread's axis region (fast layout)
  double *red = smem + L::O_RED;
  const int *eqm = (const int *)(smem + L::O_EQ);
  const int b = a.list[slot];
  const int K = a.K[b];

  // ---------------- setup on warp 0: K3 assembly, Ruiz scaling, rho, first factorisation ----------------
  // (warp 0 doubles as the control warp: adjacent lane groups hold the s-axis and the l-axis problem in the
  // lane-per-segment layout of qp.cuh, see qpd_control_*)
  double c_scale = 1.0, rhobar = o.rho0;
  int state = QP_RUNNING;
  if (warp == 0) qpd_control_setup<KC>(a, slot, lane, smem);
  // zero the padded arrays of the fast layout (V incl. pads and the extra block, C / XR incl. pads)
  for (int i = ta; i < QPD_VB * (KC + 1); i += TA) { smx[L::O_V + i] = 0.0; smx[L::O_V2 + i] = 0.0; }
  for (int i = ta; i < N + 8; i += TA) { smx[L::O_C + i] = 0.0; smx[L::O_XR + i] = 0.0; }
  sync_cta();
  c_scale = red[0];
  state = (int)red[1];
  sync_cta();

  // ---------------- fast-layout state (lives in local memory; qpd_block keeps it in registers while it iterates) ----------------
  const double *ctl = smx + L::O_CTRL;
  const double *lsx = smx + L::O_LS;
  QpdIOT<CH, L::NSLOT> io;
  QpdLU *lu0 = (QpdLU *)(smx + L::O_LU) + ta;  // bounds of this thread's row slots: lu0[s * TA]
  if constexpr (L::ROWFULL) {
#pragma unroll
    for (int sl = 0; sl < L::NSLOT; sl++) {
      if (sl < L::NDS) qpd_init_diff<KC>(io.rows[sl], lu0[sl * TA], sl * TA + ta < L::NN ? sl * TA + ta : -1, K, ctl, lsx, eqm + axis * LPA, c_scale / rhobar);
      else qpd_init_join<KC>(io.rows[sl], lu0[sl * TA], (sl - L::NDS) * TA + ta, K, ctl, eqm + axis * LPA, c_scale / rhobar);
    }
  } else {
    int ea, eb, ej;
    if (L::TWO_SLOTS) {
      if (ta >= L::T0) { ea = ta - L::T0; eb = L::TN + (ta - L::T0); }
      else { ea = 2 * L::TN + ta; eb = -1; }
      ej = ta < L::NJ ? ta : -1;
    } else {
      ea = ta < L::NN ? ta : -1; eb = -1;
      ej = (ta >= L::NN && ta < L::ROWS) ? ta - L::NN : -1;
    }
    qpd_init_diff<KC>(io.rows[0], lu0[0], ea, K, ctl, lsx, eqm + axis * LPA, c_scale / rhobar);
    qpd_init_diff<KC>(io.rows[1], lu0[TA], eb, K, ctl, lsx, eqm + axis * LPA, c_scale / rhobar);
    qpd_init_join<KC>(io.rows[2], lu0[2 * TA], ej, K, ctl, eqm + axis * LPA, c_scale / rhobar);
  }
  // G thread (v, h); the h = 0 thread is the variable thread of v
  int v, h;
  qpd_map<KC>(ta, v, h);
  const bool isg = v < N;
  const bool isvar = isg && h == 0;
  const int vk = isg ? v / 6 : 0, vj = isg ? v - 6 * vk : 0;
  io.xv = 0.0; io.sigv = 0.0; io.qv = 0.0; io.tkv = 0.0;
  if (isvar && vk < K) {
    const double *d = lsx + QPD_LS * vk;
    io.tkv = d[0]; io.qv = d[3 + vj]; io.sigv = d[9 + vj];
  }
  io.c_scale = c_scale; io.rhobar = rhobar; io.state = state; io.need_g = 1; io.it = 0;
  sync_cta();

  // ---------------- ADMM ----------------
  // Blocked by check interval: qpd_block runs the plain iterations out of line with only the hot state live (the chunk
  // of G, the row slots, the variable) -- no spills in the loop; the check iteration is one more single-iteration
  // block bracketed by the multiplier capture and qpd_check.
  int iters = 0;
  int it = 1;
  double *vv = smx + L::O_V;
  while (it <= o.max_iter && io.state == QP_RUNNING) {
    if (io.need_g) {  // after setup and after every adaptive-rho refactorisation
      qpd_build_g<KC>(smx + L::O_FS, isg ? v : 0, h, isg, io.G);
      io.need_g = 0;
    }
    int it_end = o.max_iter;  // last iteration of this block (inclusive): the next check iteration
    if (o.check_every > 0) {
      const int nxt = ((it + o.check_every - 1) / o.check_every) * o.check_every;
      it_end = nxt < it_end ? nxt : it_end;
    }
    const bool check = (o.check_every > 0) && (it_end % o.check_every == 0);
    // one out-of-line call per check interval; before its LAST iteration the block captures the multipliers
    // y = rho (w - clip(w)) of the thread's rows (io.yo) for the delta y of the check
    if constexpr (L::ROWFULL) qpd_block1<KC>(io, smx, ta, it_end - it + 1, o.alpha, sync_cta);
    else if constexpr (L::NCH == 4) qpd_block4<KC>(io, smx, ta, it_end - it + 1, o.alpha, sync_cta);
    else qpd_block<KC>(io, smx, ta, it_end - it + 1, o.alpha, sync_cta);
    iters = it_end;
    it = it_end + 1;
    if (!check) continue;
    // termination / infeasibility check + adaptive rho (out of line, see qpd_check)
    io.it = iters;
    qpd_check<KC>(a, slot, tid, smem, io, sync_cta);
    // V must hold v = rho (2 clip(w) - w) again for the next iteration
    {  // (values first, stores after: the stores go through generic pointers and would force `io` to be re-read)
      double vnew[L::NSLOT];
      int voffs[L::NSLOT];
#pragma unroll
      for (int r = 0; r < L::NSLOT; r++) {
        vnew[r] = io.rows[r].rho * (2.0 * io.rows[r].p - io.rows[r].w);
        voffs[r] = (io.rows[r].meta & 8) ? io.rows[r].voff : -1;
      }
#pragma unroll
      for (int r = 0; r < L::NSLOT; r++)
        if (voffs[r] >= 0) vv[voffs[r]] = vnew[r];
    }
    sync_cta();
  }
  state = io.state;
  rhobar = io.rhobar;
  const double xv = io.xv;
  double *xr = smx + L::O_XR;

  // ---------------- hand the iterate back to the lane-per-segment layout: W slots, rho, x ----------------
  {
    double *ctlw = smx + L::O_CTRL;
#pragma unroll
    for (int sl = 0; sl < L::NSLOT; sl++) qpd_handback_row(io.rows[sl], K, ctlw, STR);
    if (isvar) xr[QPD_CP + v] = xv;
  }
  sync_cta();
  if (warp != 0) return;
  qpd_control_finish<KC>(a, slot, lane, smem, c_scale, rhobar, state, iters);
}
