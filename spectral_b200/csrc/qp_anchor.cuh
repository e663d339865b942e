// spectral_b200/csrc/qp_anchor.cuh -- K4: the dense-operator ADMM hot loop in the ANCHOR layout (KC <= 10).
//
// Same OSQP iteration as qp_dense.cuh (it replaces the loop behind osqp_solve, solve_3d.cc:1249 | cuboid_3d.cc:1108,
// settings solve_3d.cc:1235-1243,1446-1462), same setup / factorisation / polish code on warp 0, same shared-memory
// layout (QpdLayout<KC>) -- only the thread map of the iteration changes, to cut what bounded the full-row layout
// (profiles/r1_qpd_full.md: 3 CTA barriers and ~430 shared-memory wavefronts per iteration, 3/4 of them in the
// stencil stages S1 / S2 that round-trip every row value through the V array):
//
//   thread (k, i) = control point i of segment k (five segments = 30 lanes per warp, two warps per axis) holds
//     * its whole row of G = S^-1                                        (as in the full-row layout)
//     * the four difference rows ANCHORED at i: containment i, velocity i (i <= 4), acceleration i (i <= 3),
//       jerk i (i <= 2)  -- their stencil windows all start at c_i, so ONE window c_i..c_{i+3} serves all four
//     * one continuity / initial-state row: lanes i < 3 row (k, i); lanes i >= 3 a REDUNDANT copy of row (k+1, i-3), so
//       that the three join rows a variable touches always sit in its own segment's lanes (no cross-warp traffic)
//   with (w, clip(w), l, u, rho) of its five rows in registers.
//   S2  g = A' v + sigma x - q   v = rho (2 clip(w) - w) straight from registers; the adjoint stencils take their
//                                neighbours' v by warp shuffle (6 + 3 shuffles), nothing goes through shared memory
//   S3  x~ = G g                 g broadcast from shared memory (one wavefront per LDS.128), n FMAs per thread
//   S1  z~ = A x~, w += alpha (z~ - clip(w))    one 3-load window + one 6-load join window per thread
//   Two barriers per iteration, each over the 64 threads of ONE axis (named barriers): the s and l problems of a
//   scenario only meet in the termination check.
// The arithmetic of every output is ordered exactly as in qp_dense.cuh's full-row loop, so both produce the same
// iterates bit for bit (tests/test_kernel_logic_emu.py::test_emu_anchor_layout_equals_fullrow).
#pragma once
#include "qp_dense.cuh"

#define QPA_SPW 5  // segments per warp
// doubles of g in flight per group in S3
SP_HD constexpr int qpa_grp(int N) { return (N % 24 == 0) ? 24 : ((N % 20 == 0) ? 20 : 12); }

template <int N>
struct QpaIO {
  double G[N];                                       // this thread's row of G = S^-1
  double w[5], p[5], l[5], u[5], rho[5], er[5], ier[5], yo[5];  // row slots: containment, velocity, acceleration, jerk, join
  double ce[6];                                      // coefficients of the join row on [c_{kj-1,3..5}, c_{kj,0..2}]
  double f0, f1, f2;                                 // coefficients of the three join rows in this variable's gather
  double tkv, sigv, qv, xv;                          // segment duration, sigma, q, relaxed iterate of the variable
  double c_scale, rhobar;
  int live;   // bits 0..4: slot holds a live row (rho > 0 possible), bit 5: the join slot is the primary copy
  int kj;     // segment of the join row
  int state, need_g, it;
  int K;      // segment count of the scenario (the check would otherwise chase a.K[a.list[slot]] through L2 every 25 iterations)
};

// thread map: ta in [0, TA) -> (variable v or -1)
template <int KC>
SP_DEV void qpa_map(int ta, int &seg, int &i, bool &isvar) {
  const int lane = ta & 31, wa = ta >> 5;
  const int sl = lane / 6;
  i = lane - 6 * sl;
  seg = QPA_SPW * wa + sl;
  isvar = lane < 6 * QPA_SPW && seg < KC;
}

// (A' v)_j + rest for this thread's variable from the five row values of the segment's lanes (warp shuffles).
// vv[0..3]: values of the difference rows anchored at this lane, vv[4]: value of the lane's join row.
// Arithmetic ordered as qpd_block1's S2.
template <bool CHECK_ORDER>
SP_DEV double qpa_gather(const double vv[5], int lane, int jsrc, double tkv, double f0, double f1, double f2, double rest) {
  const double u11 = sp_shfl_up(vv[1], 1, 32);
  const double u21 = sp_shfl_up(vv[2], 1, 32), u22 = sp_shfl_up(vv[2], 2, 32);
  const double u31 = sp_shfl_up(vv[3], 1, 32), u32 = sp_shfl_up(vv[3], 2, 32), u33 = sp_shfl_up(vv[3], 3, 32);
  const double c0 = sp_shfl(vv[4], jsrc), c1 = sp_shfl(vv[4], jsrc + 1), c2 = sp_shfl(vv[4], jsrc + 2);
  // lanes below the shuffle distance have no lower neighbour (elsewhere the neighbour across a segment boundary holds
  // a row that does not exist: rho = 0, value 0)
  const double g1a = lane >= 1 ? u11 : 0.0;
  const double g2b = lane >= 1 ? u21 : 0.0, g2a = lane >= 2 ? u22 : 0.0;
  const double g3c = lane >= 1 ? u31 : 0.0, g3b = lane >= 2 ? u32 : 0.0, g3a = lane >= 3 ? u33 : 0.0;
  if (CHECK_ORDER) {  // summation order of qpd_gather (the termination check's A' y and A' delta y)
    double g = tkv * vv[0];
    g += 5.0 * (g1a - vv[1]);
    g += 20.0 * ((g2a - g2b) - (g2b - vv[2]));
    g += 60.0 * ((g3a - vv[3]) + 3.0 * (g3c - g3b));
    g += f0 * c0 + f1 * c1 + f2 * c2;
    return g;
  }
  const double t01 = tkv * vv[0] + 5.0 * (g1a - vv[1]);
  const double t2 = 20.0 * ((g2a - g2b) - (g2b - vv[2]));
  const double t3 = 60.0 * ((g3a - vv[3]) + 3.0 * (g3c - g3b));
  const double tc = (f0 * c0 + f1 * c1) + (f2 * c2 + rest);
  return (t01 + t2) + (t3 + tc);
}

// A block of n ADMM iterations (out of line: only the hot state is live).  The axis AX is a template parameter, so that the
// barrier ids become immediates without predication.
template <int KC, int AX, typename SyncAxisFn>
SP_DEV_NOINLINE void qpa_block(QpaIO<6 * KC> &io, double *smx, int ta, int n, double alpha, SyncAxisFn sync_axis_fn) {
  using L = QpdLayout<KC>;
  constexpr int N = L::N;
  constexpr int GRP = qpa_grp(N);
  static_assert(N % GRP == 0 && GRP % 4 == 0, "g in whole groups");
  int seg, i;
  bool isvar;
  qpa_map<KC>(ta, seg, i, isvar);
  const int lane = ta & 31;
  const int v = isvar ? 6 * seg + i : 0;
  const int jsrc = 6 * (lane / 6) + 3 * (i / 3);
  const double *gv = smx + L::O_GV;
  double *gvp = smx + L::O_GV + v;
  double *cxp = smx + L::O_C + QPD_CP + v;
  const double *cpj = smx + L::O_C + QPD_CP + 6 * io.kj - 3;
  double w[5], p[5], l[5], u[5], rho[5], yo[5];
#pragma unroll
  for (int s = 0; s < 5; s++) { w[s] = io.w[s]; p[s] = io.p[s]; l[s] = io.l[s]; u[s] = io.u[s]; rho[s] = io.rho[s]; yo[s] = 0.0; }
  double ce[6];
#pragma unroll
  for (int m = 0; m < 6; m++) ce[m] = io.ce[m];
  const double f0 = io.f0, f1 = io.f1, f2 = io.f2, tkv = io.tkv, sigv = io.sigv, qv = io.qv;
  double xv = io.xv;
  double G[N];
#pragma unroll
  for (int e = 0; e < N; e++) G[e] = io.G[e];
  for (int it = 0; it < n; it++) {
    if (it == n - 1) {
#pragma unroll
      for (int s = 0; s < 5; s++) yo[s] = rho[s] * (w[s] - p[s]);
    }
    {  // S2
      double vv[5];
#pragma unroll
      for (int s = 0; s < 5; s++) vv[s] = rho[s] * (2.0 * p[s] - w[s]);
      const double g = qpa_gather<false>(vv, lane, jsrc, tkv, f0, f1, f2, sigv * xv - qv);
      if (isvar) *gvp = g;
    }
    sync_axis_fn(AX);
    double xt;
    {  // S3
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
      for (int g0 = 0; g0 < N; g0 += GRP) {
        double gl[GRP];
#pragma unroll
        for (int e = 0; e < GRP; e += 2) qpd_lds2(gv + g0 + e, gl[e], gl[e + 1]);
#pragma unroll
        for (int e = 0; e < GRP; e += 4) {
          a0 += G[g0 + e] * gl[e]; a1 += G[g0 + e + 1] * gl[e + 1]; a2 += G[g0 + e + 2] * gl[e + 2]; a3 += G[g0 + e + 3] * gl[e + 3];
        }
      }
      xt = (a0 + a1) + (a2 + a3);
      if (isvar) {
        xv = alpha * xt + (1.0 - alpha) * xv;
        *cxp = xt;
      }
    }
    sync_axis_fn(AX);
    {  // S1
      const double c1 = cxp[1], c2 = cxp[2], c3 = cxp[3];
      const double j0 = cpj[0], j1 = cpj[1], j2 = cpj[2], j3 = cpj[3], j4 = cpj[4], j5 = cpj[5];
      const double c0 = xt;
      const double d1 = c1 - c0, e1 = c2 - c1, f1_ = c3 - c2;
      const double d2 = e1 - d1, e2 = f1_ - e1;
      const double d3 = e2 - d2;
      double z[5];
      z[0] = tkv * c0; z[1] = 5.0 * d1; z[2] = 20.0 * d2; z[3] = 60.0 * d3;
      z[4] = (ce[0] * j0 + ce[1] * j1) + (ce[2] * j2 + ce[3] * j3) + (ce[4] * j4 + ce[5] * j5);
#pragma unroll
      for (int s = 0; s < 5; s++) {
        const double wn = w[s] + alpha * (z[s] - p[s]);
        p[s] = qpd_clip(wn, l[s], u[s]);
        w[s] = wn;
      }
    }
  }
#pragma unroll
  for (int s = 0; s < 5; s++) { io.w[s] = w[s]; io.p[s] = p[s]; io.yo[s] = yo[s]; }
  io.xv = xv;
}

// OSQP's termination test / primal-infeasibility certificate / adaptive-rho rule, CTA-wide (= jointly over the s and l
// problems), in the anchor layout.  Same quantities as qpd_check.
// Returns state | need_g << 8 (the caller keeps both in registers: reading them back from the state block costs an L2 round
// trip per block of iterations).
template <int KC, typename SyncFn>
SP_DEV_NOINLINE int qpa_check(const QpArgs &a, int slot, int tid, double *smem, QpaIO<6 * KC> &io, SyncFn sync_cta) {
  using L = QpdLayout<KC>;
  constexpr int STR = L::STR, TA = L::TA;
  const SpOptionsDev &o = a.opt;
  const int warp = tid >> 5, lane = tid & 31;
  const int axis = tid / TA, ta = tid - axis * TA;
  double *smx = smem + axis * L::AXIS;
  double *red = smem + L::O_RED;
  const double *ctl = smx + L::O_CTRL;
  const double *lsx = smx + L::O_LS;
  int seg, i;
  bool isvar;
  qpa_map<KC>(ta, seg, i, isvar);
  const int v = isvar ? 6 * seg + i : 0;
  const int jsrc = 6 * (lane / 6) + 3 * (i / 3);
  double *xr = smx + L::O_XR;
  // The whole per-thread state lives in local memory across the out-of-line calls, and with two CTAs per SM the stacks do
  // not fit L1: every first touch is an L2 round trip (~230 cycles; r2 profile: 40 % of the check's samples were
  // long-scoreboard stalls at a dozen separate use sites).  Pull every field the check needs into registers in ONE run of
  // loads behind a fence, so that the round trips overlap.
  const int K = io.K;
  const double c_scale = io.c_scale, xv = io.xv, qv = io.qv, tkv = io.tkv, io_f0 = io.f0, io_f1 = io.f1, io_f2 = io.f2;
  double rhobar = io.rhobar;
  int state = io.state, need_g = 0;
  const int it = io.it;
  const int live = io.live;
  const int io_kj = io.kj;
  double w[5], p[5], l[5], u[5], rho[5], er[5], ier[5], yo[5], ce[6], y[5], dy[5];
#pragma unroll
  for (int s = 0; s < 5; s++) {
    w[s] = io.w[s]; p[s] = io.p[s]; l[s] = io.l[s]; u[s] = io.u[s]; rho[s] = io.rho[s]; er[s] = io.er[s]; ier[s] = io.ier[s];
    yo[s] = io.yo[s];
  }
#pragma unroll
  for (int m = 0; m < 6; m++) ce[m] = io.ce[m];
  qpd_sched_fence();
  double red_v[QPD_NRED];
#pragma unroll
  for (int r = 0; r < QPD_NRED; r++) red_v[r] = 0.0;
  const double c_over_rhobar = c_scale / rhobar;
  (void)c_over_rhobar;
#pragma unroll
  for (int s = 0; s < 5; s++) {
    y[s] = rho[s] * (w[s] - p[s]);
    dy[s] = y[s] - yo[s];
    const bool counted = ((live >> s) & 1) && (s < 4 || (live & 32));  // the redundant join copies count once
    if (counted && rho[s] > 0.0) {
      red_v[7] = qpd_max(red_v[7], fabs(c_scale * dy[s] * ier[s]));
      red_v[9] += c_scale * (u[s] * qpd_max(dy[s], 0.0) + l[s] * (dy[s] < 0.0 ? dy[s] : 0.0));
    }
  }
  if (isvar) xr[QPD_CP + v] = xv;
  sync_cta();
  const double atd = qpa_gather<true>(dy, lane, jsrc, tkv, io_f0, io_f1, io_f2, 0.0);
  const double aty = qpa_gather<true>(y, lane, jsrc, tkv, io_f0, io_f1, io_f2, 0.0);
  if (isvar) {
    const double cDv = seg < K ? lsx[QPD_LS * seg + 15 + i] : 0.0;
    double px = 0.0;
    const double *pk = ctl + QP_SM_P * STR + seg;
#pragma unroll
    for (int m = 0; m < 6; m++) {
      const int e = (m >= i) ? LT(m, i) : LT(i, m);
      px += pk[e * STR] * xr[QPD_CP + 6 * seg + m];
    }
    if (seg >= K) px = 0.0;
    red_v[8] = fabs(cDv * atd);
    red_v[1] = cDv * fabs(px + qv + aty);
    red_v[4] = cDv * fabs(qv);
    red_v[5] = cDv * fabs(px);
    red_v[6] = cDv * fabs(aty);
  }
  {
    const double *cp = xr + QPD_CP + v;
    const double *cpj = xr + QPD_CP + 6 * io_kj - 3;
    const double c0 = cp[0], c1 = cp[1], c2 = cp[2], c3 = cp[3];
    const double d1 = c1 - c0, e1 = c2 - c1, f1_ = c3 - c2;
    const double d2 = e1 - d1, e2 = f1_ - e1;
    const double d3 = e2 - d2;
    double ax[5];
    ax[0] = tkv * c0; ax[1] = 5.0 * d1; ax[2] = 20.0 * d2; ax[3] = 60.0 * d3;
    ax[4] = (ce[0] * cpj[0] + ce[1] * cpj[1]) + (ce[2] * cpj[2] + ce[3] * cpj[3]) + (ce[4] * cpj[4] + ce[5] * cpj[5]);
#pragma unroll
    for (int s = 0; s < 5; s++) {
      const bool counted = ((live >> s) & 1) && (s < 4 || (live & 32));
      if (counted && rho[s] > 0.0) {
        red_v[0] = qpd_max(red_v[0], er[s] * fabs(ax[s] - p[s]));
        red_v[2] = qpd_max(red_v[2], er[s] * fabs(p[s]));
        red_v[3] = qpd_max(red_v[3], er[s] * fabs(ax[s]));
      }
    }
  }
  qpd_reduce(red_v, red, warp, lane, L::NWARPS, sync_cta);
  const double pri = red_v[0], dua = red_v[1], nz = red_v[2], nax = red_v[3], nq = red_v[4], npx = red_v[5], naty = red_v[6];
  const double nd = red_v[7], na = red_v[8], lhs = red_v[9];
  const double eps_p = o.eps_abs + o.eps_rel * fmax(nz, nax);
  const double eps_d = o.eps_abs + o.eps_rel * fmax(nq, fmax(npx, naty));
  if (pri < eps_p && dua < eps_d) state = QP_ST_SOLVED;
  else if (!(pri < eps_p) && nd > o.eps_pinf && lhs < -o.eps_pinf * nd && na < o.eps_pinf * nd) state = QP_ST_INFEASIBLE;
  if (state == QP_RUNNING && o.adapt_every > 0 && (it % o.adapt_every == 0)) {
    const double pr = pri / (fmax(nz, nax) + 1e-10);
    const double dr = dua / (fmax(nq, fmax(npx, naty)) + 1e-10);
    double est = rhobar * sqrt(pr / (dr + 1e-10));
    est = fmin(fmax(est, 1e-6), 1e6);
    if (est > rhobar * o.adapt_tol || est < rhobar / o.adapt_tol) {
      const double ratio = est / rhobar;
      double *ctl_rho = smx + L::O_CTRL + QP_SM_RHO * STR;
#pragma unroll
      for (int s = 0; s < 5; s++) {
        const double wn = p[s] + (w[s] - p[s]) / ratio;  // keep (z, y): w' = z + y / rho'
        const double rn = rho[s] * ratio;
        io.w[s] = wn; io.rho[s] = rn;
        const bool counted = ((live >> s) & 1) && (s < 4 || (live & 32));
        if (counted) {
          const int r_old = s == 0 ? i : (s == 1 ? 6 + i : (s == 2 ? 11 + i : (s == 3 ? 15 + i : 18 + (i % 3))));
          ctl_rho[r_old * STR + (s < 4 ? seg : io_kj)] = rn;
        }
      }
      rhobar = est;
      sync_cta();
      if (warp == 0) qpd_control_refactor<KC>(a, slot, lane, smem, c_scale, rhobar);
      sync_cta();
      if (red[0] != 0.0) state = QP_ST_INFEASIBLE;
      need_g = 1;
    }
  }
  io.rhobar = rhobar;
  io.state = state;
  return state | (need_g << 8);
}

// slot: index of the scenario in this class' list.  tid in [0, 2 TA).  smem: QpdLayout<KC>::BYTES, 16-byte aligned.
// sync_axis(axis) synchronises the TA threads of one axis.
template <int KC, typename SyncFn, typename SyncAxisFn>
SP_DEV void qpa_cta_body(const QpArgs &a, int slot, int tid, double *smem, SyncFn sync_cta, SyncAxisFn sync_axis_fn) {
  using L = QpdLayout<KC>;
  static_assert(L::ROWFULL && L::TA == 32 * ((KC + QPA_SPW - 1) / QPA_SPW), "anchor layout: five segments per warp, whole rows of G");
  constexpr int N = L::N, LPA = L::LPA, STR = L::STR, TA = L::TA;
  const SpOptionsDev &o = a.opt;
  const int warp = tid >> 5, lane = tid & 31;
  const int axis = tid / TA, ta = tid - axis * TA;
  double *smx = smem + axis * L::AXIS;
  double *red = smem + L::O_RED;
  const int *eqm = (const int *)(smem + L::O_EQ);
  const int b = a.list[slot];
  const int K = a.K[b];

  // ---------------- setup on warp 0 (qp_dense.cuh: K3 assembly, Ruiz scaling, rho, first factorisation) ----------------
  double c_scale = 1.0, rhobar = o.rho0;
  int state = QP_RUNNING;
  if (warp == 0) qpd_control_setup<KC>(a, slot, lane, smem);
  for (int e = ta; e < N + 8; e += TA) { smx[L::O_C + e] = 0.0; smx[L::O_XR + e] = 0.0; }
  sync_cta();
  c_scale = red[0];
  state = (int)red[1];
  sync_cta();

  // ---------------- per-thread state ----------------
  const double *ctl = smx + L::O_CTRL;
  const double *lsx = smx + L::O_LS;
  const int *eqa = eqm + axis * LPA;
  QpaIO<N> io;
  int seg, i;
  bool isvar;
  qpa_map<KC>(ta, seg, i, isvar);
  const int v = isvar ? 6 * seg + i : 0;
  {
    const double c_over_rhobar = c_scale / rhobar;
    const bool segl = isvar && seg < K;
    const int kj = i < 3 ? seg : seg + 1;
    const bool joinl = isvar && kj < K && kj < KC;
    io.kj = joinl ? kj : 0;
    io.live = (segl ? 1 : 0) | ((segl && i <= 4) ? 2 : 0) | ((segl && i <= 3) ? 4 : 0) | ((segl && i <= 2) ? 8 : 0) | (joinl ? 16 : 0) |
              ((joinl && i < 3) ? 32 : 0);
#pragma unroll
    for (int s = 0; s < 5; s++) {
      const bool lv = (io.live >> s) & 1;
      const int r_old = s == 0 ? i : (s == 1 ? 6 + i : (s == 2 ? 11 + i : (s == 3 ? 15 + i : 18 + (i % 3))));
      const int k = s < 4 ? seg : io.kj;
      const int ooff = r_old * STR + (lv ? k : 0);
      const int eq = lv ? ((eqa[k] >> r_old) & 1) : 0;
      io.w[s] = 0.0; io.p[s] = 0.0; io.yo[s] = 0.0;
      io.l[s] = lv ? ctl[QP_SM_L * STR + ooff] : -1.0;
      io.u[s] = lv ? ctl[QP_SM_U * STR + ooff] : 1.0;
      io.rho[s] = lv ? ctl[QP_SM_RHO * STR + ooff] : 0.0;
      io.er[s] = sqrt(io.rho[s] * c_over_rhobar * (eq ? 1e-3 : 1.0));
      io.ier[s] = io.er[s] > 0.0 ? 1.0 / io.er[s] : 0.0;
    }
    const double *cej = smx + L::O_CE + 6 * (3 * io.kj + (i % 3));
#pragma unroll
    for (int m = 0; m < 6; m++) io.ce[m] = joinl ? cej[m] : 0.0;
    const double *vcf = smx + L::O_VCF + 3 * v;
    io.f0 = isvar ? vcf[0] : 0.0; io.f1 = isvar ? vcf[1] : 0.0; io.f2 = isvar ? vcf[2] : 0.0;
    io.xv = 0.0; io.sigv = 0.0; io.qv = 0.0; io.tkv = 0.0;
    if (segl) {
      const double *d = lsx + QPD_LS * seg;
      io.tkv = d[0]; io.qv = d[3 + i]; io.sigv = d[9 + i];
    }
  }
  io.c_scale = c_scale; io.rhobar = rhobar; io.state = state; io.need_g = 0; io.it = 0; io.K = K;
  sync_cta();

  // ---------------- ADMM, blocked by check interval ----------------
  int iters = 0;
  int it = 1;
  int need_g = 1;
  while (it <= o.max_iter && state == QP_RUNNING) {
    if (need_g) {
      qpd_build_g<KC>(smx + L::O_FS, v, 0, isvar, io.G);
      need_g = 0;
    }
    int it_end = o.max_iter;
    if (o.check_every > 0) {
      const int nxt = ((it + o.check_every - 1) / o.check_every) * o.check_every;
      it_end = nxt < it_end ? nxt : it_end;
    }
    const bool check = (o.check_every > 0) && (it_end % o.check_every == 0);
    if (axis == 0) qpa_block<KC, 0>(io, smx, ta, it_end - it + 1, o.alpha, sync_axis_fn);
    else qpa_block<KC, 1>(io, smx, ta, it_end - it + 1, o.alpha, sync_axis_fn);
    iters = it_end;
    it = it_end + 1;
    if (!check) continue;
    io.it = iters;
    const int r = qpa_check<KC>(a, slot, tid, smem, io, sync_cta);  // (the axes ran the block independently; the check's barriers are CTA-wide)
    state = r & 0xff;
    need_g = r >> 8;
  }
  rhobar = io.rhobar;

  // ---------------- hand the iterate back to the lane-per-segment layout: W slots, rho, x ----------------
  {
    double *ctlw = smx + L::O_CTRL;
#pragma unroll
    for (int s = 0; s < 5; s++) {
      const bool counted = ((io.live >> s) & 1) && (s < 4 || (io.live & 32));
      if (!counted) continue;
      const int r_old = s == 0 ? i : (s == 1 ? 6 + i : (s == 2 ? 11 + i : (s == 3 ? 15 + i : 18 + (i % 3))));
      const int ooff = r_old * STR + (s < 4 ? seg : io.kj);
      ctlw[QP_SM_W * STR + ooff] = io.w[s];
      ctlw[QP_SM_RHO * STR + ooff] = io.rho[s];
    }
    if (isvar) smx[L::O_XR + QPD_CP + v] = io.xv;
  }
  sync_cta();
  if (warp != 0) return;
  qpd_control_finish<KC>(a, slot, lane, smem, c_scale, rhobar, state, iters);
}
