// spectral_b200/csrc/qp_shared4.cuh -- K4a: the shared-KKT tile kernel k_qps4, four warps per tile.
//
// The tile structure, the keys, and the prepare / finish kernels around this one are in qp_shared.cuh (read that header first).
// Layout.  One CTA = one tile = 4 warps = (axis, half): lane 4n + q of warp (axis, h) owns ONE segment, seg = 4h + q, of
// scenario n = 0..7: its 6 control points and its 21 constraint rows (w in registers, l, u in shared memory, lane-interleaved).
// The stencils A x and A' v of a segment are thread-local (apply_A / apply_AT of qp.cuh); only the three continuity rows at a
// segment boundary travel, by quad shuffle inside a warp.  The DMMA (mma.sync.m8n8k4.f64) computes X~' = [g]' G with the 8
// scenarios of the tile as the M dimension: the A fragments are the threads' own gather values, the B fragments G from shared
// memory, the C fragments the threads' own outputs x~ -- no data movement between the gather, the contraction and the row update.
// Why four warps: the two-warp layout measured in round 2 (one warp per axis, two segments per thread, w rows in shared memory)
// was bound by shared-memory CAPACITY, not by any pipe: 110 KB per tile -> two tiles = four warps per SM, one warp per
// scheduler, every dependent-instruction latency exposed (profiles/r2_qps_full.md: sm__warps_active 5.6 %, stall "wait" 2.2 per
// issue).  Here there are twice the warps per byte of shared memory and half the serial work per thread.
//
// DMMA split.  The k dimension of X~' = [g]' G (48 variables of an axis) is split between the two warps of the axis: warp h
// contracts its own 24 gather values (6 k-steps x 4 quad lanes) against ALL 48 columns (6 n-tiles) -- 36 DMMAs per warp,
// 72 per axis.  The column order of its B fragments puts its OWN segments' outputs in n-tiles 0..2 and the OTHER
// warp's in n-tiles 3..5, so that thread (n, q) holds the partial sums of exactly its own six outputs and of the six outputs
// of thread (n, q) of the other warp: one 6-double store, one named barrier over the 64 threads of the axis, one 6-double
// load complete x~.  The continuity rows couple segment 3 (warp 0, q = 3) with segment 4 (warp 1, q = 0): x~ of segment 3's
// last three control points travels with the first exchange, the join rows' values with a second barrier.
#pragma once
#include "qp_shared.cuh"

#define QPS4_XCH (2 * 2 * 6 * 32)   // [axis][h][j][lane]: partial sums for the other warp
#define QPS4_EXT (2 * 3 * 32)       // [axis][j][lane]: warp 0's own partial sums of control points 3..5 (for segment 4's join rows)
#define QPS4_NXT (2 * 3 * 8)        // [axis][row 18..20][scenario]: join-row values of segment 4 (for segment 3's gather)

// shared memory of one four-warp tile CTA (doubles).  The w rows live in REGISTERS (21 per thread: one segment), so the row
// arrays hold only l and u, which leaves room for the exchange buffers at two tiles per SM.
struct Qps4Smem {
  static constexpr int O_ROWS = 0;                          // [axis][slot L/U][h][21][32]
  static constexpr int ROWS_AXIS = 2 * 2 * QPS_ROWSZ;
  static constexpr int O_GF = O_ROWS + 2 * ROWS_AXIS;       // [axis][h][36][32]
  static constexpr int O_CTL = O_GF + 2 * QPS_NFRAG * 32;   // [axis][63][8]: P, RHO and E_r slots, stride 8 (see QPS_RHO / QPS_ER)
  static constexpr int CTL_AXIS = 63 * 8;
  static constexpr int O_SEG = O_CTL + 2 * CTL_AXIS;        // [axis][8][16]: t, tp, tn, pad, sig[6], cD[6]
  static constexpr int O_FLAG = O_SEG + 2 * 8 * 16;         // [2] cross-axis flags (bad pivot)
  static constexpr int O_X4 = O_FLAG + 8;                   // [axis][h][6][32] partial sums for the other warp
  static constexpr int O_EXT = O_X4 + QPS4_XCH;             // [axis][3][32]
  static constexpr int O_NXT = O_EXT + QPS4_EXT;            // [axis][parity][3][8]
  static constexpr int O_RED4 = O_NXT + 2 * QPS4_NXT;       // [warp][scenario][QPD_NRED] reduction exchange of the check
  static constexpr int TOTAL = O_RED4 + 4 * 8 * QPD_NRED;
  static constexpr int BYTES = TOTAL * 8;
};

// One ADMM row pass over the thread's segment, rows [RB, RE), with the w rows in registers: w += alpha (z~ - clip(w)),
// v = rho (2 clip(w) - w) of the new w.  Loads (l, u, rho) staged in groups of CH rows.  CHECK: also the multiplier step
// dy = y_new - y_old and its norm terms.  The update is branch-free: a finished member runs it with alpha = 0.
template <bool CHECK, int RB, int RE, int CH>
SP_DEV void qps4_row_pass(double w[QP_ROWS], const double *__restrict__ rl, const double *__restrict__ ru, const double *__restrict__ rho,
                          const double z[QP_ROWS], int lane, double alpha_eff, double v[QP_ROWS], double dy[QP_ROWS],
                          const double *__restrict__ er_c, double c_scale, double &nd, double &lhs) {
  static_assert((RE - RB) % CH == 0, "whole groups");
#pragma unroll
  for (int r0 = RB; r0 < RE; r0 += CH) {
    double l[CH], u[CH], rh[CH];
#pragma unroll
    for (int j = 0; j < CH; j++) {
      l[j] = qps_lds(rl + (r0 + j) * 32 + lane); u[j] = qps_lds(ru + (r0 + j) * 32 + lane);
      rh[j] = qps_lds(rho + (r0 + j) * 8);
    }
#pragma unroll
    for (int j = 0; j < CH; j++) {
      const int r = r0 + j;
      const double p = qpd_clip(w[r], l[j], u[j]);
      const double wn = w[r] + alpha_eff * (z[r] - p);
      const double pn = qpd_clip(wn, l[j], u[j]);
      v[r] = rh[j] * (2.0 * pn - wn);
      if (CHECK) {
        const double d = rh[j] * (wn - pn) - rh[j] * (w[r] - p);
        dy[r] = d;
        const double live = rh[j] > 0.0 ? 1.0 : 0.0;
        nd = qpd_max(nd, live * fabs(c_scale * d / er_c[r * 8]));
        lhs += live * (c_scale * (u[j] * qpd_max(d, 0.0) + l[j] * (d < 0.0 ? d : 0.0)));
      }
      w[r] = wn;
    }
  }
}

// position of element (v, c) of G in the four-warp fragment array: B fragment (warp half h, k-step s, n-tile nt) at lane
SP_DEV int qps4_frag_index(int v, int c) {
  const int h = v / 24, kk = (v % 24) / 6, s = v % 6;
  const int ch = c / 24, cq = (c % 24) / 6, j = c % 6;
  const int nt = (j >> 1) + (ch == h ? 0 : 3), r = 2 * cq + (j & 1);
  return ((h * 6 + s) * 6 + nt) * 32 + r * 4 + kk;
}

// one warp: (re)factorise S for the RHO slots in ctl and rebuild BOTH halves' B fragments of G = S^-1
SP_DEV int qps4_build_g(const double *ctl, double *fs, double *gf, const double *segc, int lane, int K) {
  const int seg = lane & 7;
  const double *sc = segc + 16 * seg;
  double sig[6];
#pragma unroll
  for (int j = 0; j < 6; j++) sig[j] = sc[4 + j];
  QpFactor F;
  int bad = qp_factorize<8, 8>(ctl, seg, QPS_RHO, sig, sc[0], sc[1], sc[2], seg == 0, seg == K - 1, seg < K, seg, K, 0u, 0u, 0.0, F);
  bad = sp_group_or(bad, 8);
  if (lane < 8) {
    double *dst = fs + 57 * seg;
#pragma unroll
    for (int e = 0; e < 21; e++) dst[e] = F.Linv[e];
#pragma unroll
    for (int e = 0; e < 18; e++) { dst[21 + e] = F.C[e]; dst[39 + e] = F.E[e]; }
  }
  sp_syncwarp();
  for (int v = lane; v < 64; v += 32) {
    double g[QPS_N];
    qpd_inverse_chunk<QPS_KC>(fs, v < QPS_N ? v : 0, 0, g);
    if (v < QPS_N) {
#pragma unroll
      for (int c = 0; c < QPS_N; c++) gf[qps4_frag_index(v, c)] = g[c];
    }
  }
  sp_syncwarp();
  return bad;
}

// The tile body: `tid` in [0, 128).  sync_axis(axis): named barrier over the 64 threads of one axis.
template <typename SyncFn, typename SyncAxisFn>
SP_DEV void qps4_tile_body(const QpsArgs &A, int tile, int cta, int tid, double *smem, SyncFn sync_cta, SyncAxisFn sync_axis) {
  using S = Qps4Smem;
  using S4 = Qps4Smem;
  const QpArgs &a = A.q;
  const SpOptionsDev &o = a.opt;
  const int warp = tid >> 5, lane = tid & 31;
  const int axis = warp >> 1, h = warp & 1;
  const int n = lane >> 2, q = lane & 3;
  const int seg = 4 * h + q;
  const int cnt = A.tile_count[tile];
  const int b = A.sorted[A.tile_start[tile] + (n < cnt ? n : 0)];
  const bool have = n < cnt;
  double *rows = smem + S::O_ROWS + axis * S::ROWS_AXIS;
  double *gf = smem + S::O_GF + axis * QPS_NFRAG * 32;
  double *ctl = smem + S::O_CTL + axis * S::CTL_AXIS - QP_SM_P * 8;  // virtual base (see QPS_RHO)
  double *fs = A.fs_scratch + ((size_t)cta * 2 + axis) * 57 * 8;
  double *segc = smem + S::O_SEG + axis * 8 * 16;
  double *x4 = smem + S4::O_X4 + axis * (2 * 6 * 32);
  double *ext = smem + S4::O_EXT + axis * (3 * 32);
  double *nxt2 = smem + S4::O_NXT + axis * (2 * 3 * 8);
  int nxp = 0;   // parity of the join-row exchange buffer (two consecutive exchanges never share a buffer)
  double *red4 = smem + S4::O_RED4;
  const QpsTileBlk &B = A.blk[2 * tile + axis];
  const int K = B.K;
  const double c_scale = B.c;
  double rhobar = B.rhobar;

  // ---------------- load the tile structure and the members' rows ----------------
  if (h == 0) {
    for (int e = lane; e < 21 * 8; e += 32) {
      ctl[QPS_RHO * 8 + e] = (&B.rho[0][0])[e];
      ctl[QP_SM_P * 8 + e] = (&B.P[0][0])[e];
    }
    if (lane < 8) {
      double *sc = segc + 16 * lane;
      sc[0] = B.t[lane]; sc[1] = B.tp[lane]; sc[2] = B.tn[lane]; sc[3] = 0.0;
#pragma unroll
      for (int j = 0; j < 6; j++) { sc[4 + j] = B.sig[lane][j]; sc[10 + j] = B.cD[lane][j]; }
    }
  }
  double *rl = rows + (0 * 2 + h) * QPS_ROWSZ, *ru = rows + (1 * 2 + h) * QPS_ROWSZ;
  double qv[6], x[6], xt[6], w[QP_ROWS];
  {
    const bool act = have && seg < K;
    const double *lu = a.lu + (((size_t)b * 2 + axis) * a.k_max + seg) * QP_ROWS * 2;
    const double *qs = A.qv + (((size_t)b * 2 + axis) * 8 + seg) * 6;
#pragma unroll
    for (int r = 0; r < QP_ROWS; r++) {
      w[r] = 0.0;
      rl[r * 32 + lane] = act ? lu[2 * r] : -1.0;
      ru[r * 32 + lane] = act ? lu[2 * r + 1] : 1.0;
    }
#pragma unroll
    for (int j = 0; j < 6; j++) { qv[j] = act ? qs[j] : 0.0; x[j] = 0.0; xt[j] = 0.0; }
  }
  sync_axis(axis);
  // E_r of the tile scaling (invariant under rho updates): [row][seg]
  if (h == 0) {
    for (int e = lane; e < 21 * 8; e += 32) {
      const int r = e >> 3, sg = e & 7;
      const int eq = (B.eqmask[sg] >> r) & 1;
      const double rh = ctl[QPS_RHO * 8 + e];
      ctl[QPS_ER * 8 + e] = (sg < K && rh > 0.0) ? sqrt(rh * (c_scale / rhobar) * (eq ? 1e-3 : 1.0)) : 1.0;
    }
    sp_syncwarp();
  }
  int bad = 0;
  if (h == 0) bad = qps4_build_g(ctl, fs, gf, segc, lane, K);
  {  // a failed factorisation on either axis fails the tile on both (all four warps must hold the same states)
    double *flag = smem + S::O_FLAG;
    if (h == 0 && lane == 0) flag[axis] = (double)bad;
    sync_cta();
    bad = (flag[0] != 0.0 || flag[1] != 0.0) ? 1 : 0;
    sync_cta();
  }

  // per-thread segment constants
  const double tS = segc[16 * seg], tpS = segc[16 * seg + 1], tnS = segc[16 * seg + 2];
  const bool firstS = seg == 0, lastS = seg == K - 1, actS = seg < K;
  const double *rho_c = ctl + QPS_RHO * 8 + seg, *er_c = ctl + QPS_ER * 8 + seg;
  const double *sg_c = segc + 16 * seg + 4, *cD_c = segc + 16 * seg + 10;
  const double *gfw = gf + (size_t)h * 36 * 32 + lane;
  int state = (have && K > 0) ? QP_RUNNING : QP_ST_MAXITER;
  if (have && (bad || A.st[4 * b + 3])) state = QP_ST_INFEASIBLE;
  int iters = 0;
  const double alpha = o.alpha;

  // join-row values of the NEXT segment (rows 18..20 of seg + 1) for this segment's gather, from v18..v20 of every thread
  auto next_join = [&](double v18, double v19, double v20, double &n18, double &n19, double &n20) {
    double *nxt = nxt2 + nxp * 24;
    nxp ^= 1;
    if (h == 1 && q == 0) { nxt[0 * 8 + n] = v18; nxt[1 * 8 + n] = v19; nxt[2 * 8 + n] = v20; }
    sync_axis(axis);
    n18 = sp_shfl_down(v18, 1, 4); n19 = sp_shfl_down(v19, 1, 4); n20 = sp_shfl_down(v20, 1, 4);
    if (q == 3) {
      if (h == 0) { n18 = nxt[0 * 8 + n]; n19 = nxt[1 * 8 + n]; n20 = nxt[2 * 8 + n]; }
      else { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
    }
    if (lastS || !actS) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
  };

  // g of the cold start: w = 0 -> v = 0 -> g = -q
  double g[6];
#pragma unroll
  for (int j = 0; j < 6; j++) g[j] = -qv[j];

  for (int it = 1; it <= o.max_iter; it++) {
    const bool run = state == QP_RUNNING;
    if (!sp_any(run)) break;   // (all four warps hold the same states: they leave together)
    const bool check = (o.check_every > 0) && (it % o.check_every == 0);
    // ---- S3: this warp's k-half of X~' = g' G on the FP64 tensor pipe (36 DMMAs), then the exchange of the partial sums
    double acc[12];
#pragma unroll
    for (int j = 0; j < 12; j++) acc[j] = 0.0;
#pragma unroll
    for (int s = 0; s < 6; s++) {
      double bf[6];
#pragma unroll
      for (int nt = 0; nt < 6; nt++) bf[nt] = qps_lds(gfw + (s * 6 + nt) * 32);
#pragma unroll
      for (int nt = 0; nt < 6; nt++) qps_dmma(g[s], bf[nt], acc[2 * nt], acc[2 * nt + 1]);
    }
    {
      double *mine = x4 + (size_t)h * 6 * 32 + lane;
#pragma unroll
      for (int j = 0; j < 6; j++) mine[j * 32] = acc[6 + j];
      if (h == 0) { ext[0 * 32 + lane] = acc[3]; ext[1 * 32 + lane] = acc[4]; ext[2 * 32 + lane] = acc[5]; }
    }
    sync_axis(axis);
    double p3, p4, p5;
    {
      const double *theirs = x4 + (size_t)(1 - h) * 6 * 32 + lane;
      // (h = 0: own + received; h = 1: received + own -- both warps add warp 0's partial sum first, so that the value of a
      //  control point is the same whoever computes it)
#pragma unroll
      for (int j = 0; j < 6; j++) xt[j] = h == 0 ? acc[j] + theirs[j * 32] : theirs[j * 32] + acc[j];
      p3 = sp_shfl_up(xt[3], 1, 4); p4 = sp_shfl_up(xt[4], 1, 4); p5 = sp_shfl_up(xt[5], 1, 4);
      if (h == 1 && q == 0) {   // segment 4: the previous segment lives in warp 0, lane + 3
        const double *w1 = x4 + (size_t)1 * 6 * 32 + lane + 3;
        p3 = ext[0 * 32 + lane + 3] + w1[3 * 32];
        p4 = ext[1 * 32 + lane + 3] + w1[4 * 32];
        p5 = ext[2 * 32 + lane + 3] + w1[5 * 32];
      }
    }
    if (run) {
#pragma unroll
      for (int j = 0; j < 6; j++) x[j] = alpha * xt[j] + (1.0 - alpha) * x[j];
      iters = it;
    }
    // ---- S1 + S2: the three join rows first (the neighbour needs their values), then the difference rows; gather
    const double alpha_eff = run ? alpha : 0.0;  // a finished member keeps its state
    double z[QP_ROWS], v[QP_ROWS], dy[QP_ROWS];
    double nd = 0.0, lhs = 0.0;
    apply_A(xt, p3, p4, p5, tS, tpS, firstS, z);
    if (check) qps4_row_pass<true, 18, 21, 3>(w, rl, ru, rho_c, z, lane, alpha_eff, v, dy, er_c, c_scale, nd, lhs);
    else qps4_row_pass<false, 18, 21, 3>(w, rl, ru, rho_c, z, lane, alpha_eff, v, dy, nullptr, c_scale, nd, lhs);
    double *nxt = nxt2 + nxp * 24;
    nxp ^= 1;
    if (h == 1 && q == 0) { nxt[0 * 8 + n] = v[18]; nxt[1 * 8 + n] = v[19]; nxt[2 * 8 + n] = v[20]; }
    if (check) qps4_row_pass<true, 0, 18, 6>(w, rl, ru, rho_c, z, lane, alpha_eff, v, dy, er_c, c_scale, nd, lhs);
    else qps4_row_pass<false, 0, 18, 6>(w, rl, ru, rho_c, z, lane, alpha_eff, v, dy, nullptr, c_scale, nd, lhs);
    sync_axis(axis);
    double n18 = sp_shfl_down(v[18], 1, 4), n19 = sp_shfl_down(v[19], 1, 4), n20 = sp_shfl_down(v[20], 1, 4);
    if (q == 3) {
      if (h == 0) { n18 = nxt[0 * 8 + n]; n19 = nxt[1 * 8 + n]; n20 = nxt[2 * 8 + n]; }
      else { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
    }
    if (lastS || !actS) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
    apply_AT(v, n18, n19, n20, tS, tpS, tnS, firstS, g);
#pragma unroll
    for (int j = 0; j < 6; j++) g[j] += sg_c[j] * x[j] - qv[j];
    if (!check) continue;

    // ---- termination check (OSQP's test in the tile scaling), joint over the two axes of each scenario
    double red_v[QPD_NRED];
#pragma unroll
    for (int i = 0; i < QPD_NRED; i++) red_v[i] = 0.0;
    red_v[7] = nd; red_v[9] = lhs;
    {
      // A x (relaxed x), A' y, A' dy, P x of the thread's segment
      double ax[QP_ROWS], y[QP_ROWS];
      {
        double r3 = sp_shfl_up(x[3], 1, 4), r4 = sp_shfl_up(x[4], 1, 4), r5 = sp_shfl_up(x[5], 1, 4);
        // segment 4 needs segment 3's relaxed control points: through the exchange buffer
        if (h == 0 && q == 3) { ext[0 * 32 + lane] = x[3]; ext[1 * 32 + lane] = x[4]; ext[2 * 32 + lane] = x[5]; }
        sync_axis(axis);
        if (h == 1 && q == 0) { r3 = ext[0 * 32 + lane + 3]; r4 = ext[1 * 32 + lane + 3]; r5 = ext[2 * 32 + lane + 3]; }
        apply_A(x, r3, r4, r5, tS, tpS, firstS, ax);
      }
#pragma unroll
      for (int r = 0; r < QP_ROWS; r++) {
        const double p = qpd_clip(w[r], rl[r * 32 + lane], ru[r * 32 + lane]);
        const double rh = rho_c[r * 8];
        y[r] = rh * (w[r] - p);
        if (rh > 0.0 && actS) {
          const double E = er_c[r * 8];
          red_v[0] = qpd_max(red_v[0], E * fabs(ax[r] - p));
          red_v[2] = qpd_max(red_v[2], E * fabs(p));
          red_v[3] = qpd_max(red_v[3], E * fabs(ax[r]));
        }
      }
      double aty[6], atd[6];
      {
        double m18, m19, m20;
        next_join(y[18], y[19], y[20], m18, m19, m20);
        apply_AT(y, m18, m19, m20, tS, tpS, tnS, firstS, aty);
        next_join(dy[18], dy[19], dy[20], m18, m19, m20);
        apply_AT(dy, m18, m19, m20, tS, tpS, tnS, firstS, atd);
      }
      if (actS) {
        double px[6];
        apply_P<8>(ctl, seg, x, px);
#pragma unroll
        for (int j = 0; j < 6; j++) {
          red_v[8] = qpd_max(red_v[8], fabs(cD_c[j] * atd[j]));
          red_v[1] = qpd_max(red_v[1], cD_c[j] * fabs(px[j] + qv[j] + aty[j]));
          red_v[4] = qpd_max(red_v[4], cD_c[j] * fabs(qv[j]));
          red_v[5] = qpd_max(red_v[5], cD_c[j] * fabs(px[j]));
          red_v[6] = qpd_max(red_v[6], cD_c[j] * fabs(aty[j]));
        }
      }
    }
    // reduce over the quad, then across the four warps of the tile
#pragma unroll
    for (int i = 0; i < QPD_NRED - 1; i++) {
      red_v[i] = qpd_max(red_v[i], sp_shfl_xor(red_v[i], 1));
      red_v[i] = qpd_max(red_v[i], sp_shfl_xor(red_v[i], 2));
    }
    red_v[9] += sp_shfl_xor(red_v[9], 1);
    red_v[9] += sp_shfl_xor(red_v[9], 2);
    if (q == 0) {
#pragma unroll
      for (int i = 0; i < QPD_NRED; i++) red4[(warp * 8 + n) * QPD_NRED + i] = red_v[i];
    }
    sync_cta();
    {
      const double *o0 = red4 + (0 * 8 + n) * QPD_NRED, *o1 = red4 + (1 * 8 + n) * QPD_NRED;
      const double *o2 = red4 + (2 * 8 + n) * QPD_NRED, *o3 = red4 + (3 * 8 + n) * QPD_NRED;
#pragma unroll
      for (int i = 0; i < QPD_NRED - 1; i++) red_v[i] = qpd_max(qpd_max(o0[i], o1[i]), qpd_max(o2[i], o3[i]));
      red_v[9] = (o0[9] + o1[9]) + (o2[9] + o3[9]);
    }
    sync_cta();
    const double pri = red_v[0], dua = red_v[1], nz = red_v[2], nax = red_v[3], nq = red_v[4], npx = red_v[5], naty = red_v[6];
    const double ndn = red_v[7], na = red_v[8], lh = red_v[9];
    const double eps_p = o.eps_abs + o.eps_rel * fmax(nz, nax);
    const double eps_d = o.eps_abs + o.eps_rel * fmax(nq, fmax(npx, naty));
    if (run) {
      if (pri < eps_p && dua < eps_d) state = QP_ST_SOLVED;
      else if (!(pri < eps_p) && ndn > o.eps_pinf && lh < -o.eps_pinf * ndn && na < o.eps_pinf * ndn) state = QP_ST_INFEASIBLE;
    }
    // ---- tile rho: OSQP's estimate per member, geometric mean over the members still running
    if (o.adapt_every > 0 && (it % o.adapt_every == 0)) {
      const bool still = state == QP_RUNNING;
      const double pr = pri / (fmax(nz, nax) + 1e-10);
      const double dr = dua / (fmax(nq, fmax(npx, naty)) + 1e-10);
      double est = rhobar * sqrt(pr / (dr + 1e-10));
      est = fmin(fmax(est, 1e-6), 1e6);
      double ls = (still && q == 0) ? log(est) : 0.0, lc = (still && q == 0) ? 1.0 : 0.0;
#pragma unroll
      for (int m = 16; m > 0; m >>= 1) { ls += sp_shfl_xor(ls, m); lc += sp_shfl_xor(lc, m); }
      if (lc > 0.0) {
        const double tile_est = exp(ls / lc);
        if (tile_est > rhobar * o.adapt_tol || tile_est < rhobar / o.adapt_tol) {
          const double ratio = tile_est / rhobar;
#pragma unroll
          for (int r = 0; r < QP_ROWS; r++) {
            const double p = qpd_clip(w[r], rl[r * 32 + lane], ru[r * 32 + lane]);
            w[r] = p + (w[r] - p) / ratio;  // keep (z, y): w' = z + y / rho'
          }
          sync_axis(axis);   // (every thread has read the old rho slots it needs: none are read between the check and here)
          if (h == 0) {
            for (int e = lane; e < 21 * 8; e += 32) ctl[QPS_RHO * 8 + e] *= ratio;
            sp_syncwarp();
          }
          rhobar = tile_est;
          int b2 = 0;
          if (h == 0) b2 = qps4_build_g(ctl, fs, gf, segc, lane, K);
          {
            double *flag = smem + S::O_FLAG;
            if (h == 0 && lane == 0) flag[axis] = (double)b2;
            sync_cta();
            b2 = (flag[0] != 0.0 || flag[1] != 0.0) ? 1 : 0;
            sync_cta();
          }
          if (b2 && state == QP_RUNNING) state = QP_ST_INFEASIBLE;
          // v and g of the rescaled rows
#pragma unroll
          for (int r = 0; r < QP_ROWS; r++) {
            const double p = qpd_clip(w[r], rl[r * 32 + lane], ru[r * 32 + lane]);
            v[r] = rho_c[r * 8] * (2.0 * p - w[r]);
          }
          double m18, m19, m20;
          next_join(v[18], v[19], v[20], m18, m19, m20);
          apply_AT(v, m18, m19, m20, tS, tpS, tnS, firstS, g);
#pragma unroll
          for (int j = 0; j < 6; j++) g[j] += sg_c[j] * x[j] - qv[j];
        }
      }
    }
  }

  // ---------------- hand off to k_qps_finish: w rows, relaxed x, state, iterations; the tile's final rho ----------------
  if (have) {
    double *dw = A.wrows + (((size_t)b * 2 + axis) * 8 + seg) * QP_ROWS;
#pragma unroll
    for (int r = 0; r < QP_ROWS; r++) dw[r] = w[r];
    double *dx = A.xout + ((size_t)b * 2 + axis) * QPS_N + 6 * seg;
#pragma unroll
    for (int j = 0; j < 6; j++) dx[j] = x[j];
    if (q == 0 && warp == 0) { A.st[4 * b + 0] = state; A.st[4 * b + 1] = iters; A.st[4 * b + 2] = tile; }
  }
  sync_cta();
  if (h == 0) {
    QpsTileBlk &Bw = A.blk[2 * tile + axis];
    for (int e = lane; e < 21 * 8; e += 32) (&Bw.rho[0][0])[e] = ctl[QPS_RHO * 8 + e];
    if (lane == 0) Bw.rhobar = rhobar;
  }
}
