// spectral_b200/csrc/qp.cuh -- K3 (QP assembly) + K4b (batched ADMM, OSQP-equivalent) + polish.
//
// Replaces, for one axis (s or l) of one scenario ("axis problem"), what the reference does in
//   FormulateProblem / CalculateKernel / CalculateAffineConstraint / CalculateOffset
//       solve_3d.cc:1143-1229, :70-224, :779-1129, :226-321   (cuboid_3d.cc: same functions)
//   Optimize -> osqp_setup / osqp_solve with the settings of solve_3d.cc:1235-1243,1446-1462.
// The reference's QP is block-diagonal in (s, l) (no row of A and no entry of P mixes the axes,
// SURVEY.md Appendix B), so the two axes are solved as independent OSQP instances; the optimum is
// the same, the iteration counts are per axis.
//
// Mapping (sm_100a): LPA lanes per axis problem (8, 16 or 32), lane k owns Bezier segment k:
// its 6 control points, its 18 containment/velocity/acceleration/jerk rows and the 3 rows that tie
// it to segment k-1 (continuity) or to the initial state (k = 0) -- 21 rows per lane, always.
// A is never materialised: its rows are difference stencils (5(c[i+1]-c[i]), 20(..), 60(..)).
// The reduced KKT matrix S = P + diag(sigma_j) + A' diag(rho_r) A is block tridiagonal with 6x6
// diagonal blocks and 3x3 couplings; its block Cholesky factor is kept in REGISTERS in the form
//   Linv_k (inverse of the diagonal factor, 21), C_k = Linv_k B_k (6x3), E_k = Linv_k' B_{k+1}' (6x3)
// so that a solve is two lane-parallel triangular mat-vecs plus two short neighbour-to-neighbour
// sweeps (3 FMAs x 3 rows on the critical path per hop).  Iteration state w (= z + y/rho, from which
// both z = clip(w) and y = rho (w - z) follow), the bounds l, u, the per-row rho and the segment's P
// block live in SHARED memory, lane-interleaved (conflict free).
// OSQP's Ruiz equilibration (D, E, c) is applied implicitly: scaled ADMM is identical to unscaled
// ADMM with rho_r = rho * E_r^2 / c and sigma_j = sigma / (c D_j^2); residual norms for termination
// (scaled_termination = 1) are evaluated with the same D, E, c.
#pragma once
#include "common.cuh"

#define QP_ROWS 21
#define QP_SM_W 0
#define QP_SM_L 21
#define QP_SM_U 42
#define QP_SM_RHO 63
#define QP_SM_P 84
#define QP_SM_DOUBLES_PER_LANE 105
#define QP_SMEM_PER_WARP (QP_SM_DOUBLES_PER_LANE * 32 * 8)

#define QP_XCH_DOUBLES 4                        // cross-warp exchange scratch of a two-warp joint instance (JW = 64)

#define LT(i, j) ((i) * ((i) + 1) / 2 + (j))  // packed lower triangle, i >= j

#define QP_RUNNING 0
#define QP_ST_SOLVED 1
#define QP_ST_INACCURATE 2
#define QP_ST_INFEASIBLE 3
#define QP_ST_MAXITER 4

struct QpArgs {
  int N, k_max, variant;
  double delta;
  const double *ds_bounds, *dl_bounds, *s_ref, *l_ref, *init, *scalars, *weights;
  int wstride;
  int in_stride;     // 1: one input scenario per lane; 0: every lane reads scenario 0 (weight sweep)
  const double *mqm;  // [W][2 axes][4][21] packed lower triangle of M' pQp_d M
  const SpectralCube *segs;
  const int *K;
  const int *list;   // scenario ids of this lane-class
  const int *count;  // number of entries in list
  int *next;         // persistent kernels: next list entry to take (device counter, zeroed with the counts)
  SpOptionsDev opt;
  double *ctrl;      // [B][12*k_max]
  int *axis_status;  // [B][2]
  int *axis_iters;   // [B][2]
  int *axis_polished;// [B][2]
  double *axis_obj;  // [B][2]
  double *lu;        // optional [B][2][k_max][21][2]
};

// ------------------------------------------------------------------ row stencils
// coefficient of own control point j in row r of this lane (solve_3d.cc:823-949)
SP_DEV double row_coef(int r, int j, double t, double tp, bool first) {
  if (r < 6) return j == r ? t : 0.0;
  if (r < 11) { int i = r - 6; return j == i ? -5.0 : (j == i + 1 ? 5.0 : 0.0); }
  if (r < 15) { int i = r - 11; return j == i ? 20.0 : (j == i + 1 ? -40.0 : (j == i + 2 ? 20.0 : 0.0)); }
  if (r < 18) { int i = r - 15; return j == i ? -60.0 : (j == i + 1 ? 180.0 : (j == i + 2 ? -180.0 : (j == i + 3 ? 60.0 : 0.0))); }
  if (r == 18) return j == 0 ? t : 0.0;
  if (r == 19) return first ? (j == 0 ? -5.0 : (j == 1 ? 5.0 : 0.0)) : (j == 0 ? 1.0 : (j == 1 ? -1.0 : 0.0));
  return first ? (j == 0 ? 20.0 : (j == 1 ? -40.0 : (j == 2 ? 20.0 : 0.0)))
               : (j == 0 ? -tp : (j == 1 ? 2.0 * tp : (j == 2 ? -tp : 0.0)));
}
// coefficient of the PREVIOUS segment's control point 3+j in continuity row r (18..20) of this lane
SP_DEV double prev_coef(int r, int j, double t, double tp, bool first) {
  if (first) return 0.0;
  if (r == 18) return j == 2 ? -tp : 0.0;
  if (r == 19) return j == 1 ? -1.0 : (j == 2 ? 1.0 : 0.0);
  return j == 1 ? -2.0 * t : t;
}

// z = A x restricted to this lane's 21 rows; p3..p5 = previous segment's control points 3..5
SP_DEV void apply_A(const double c[6], double p3, double p4, double p5, double t, double tp, bool first,
                    double z[QP_ROWS]) {
  double d1[5], d2[4];
#pragma unroll
  for (int i = 0; i < 6; i++) z[i] = t * c[i];
#pragma unroll
  for (int i = 0; i < 5; i++) { d1[i] = c[i + 1] - c[i]; z[6 + i] = 5.0 * d1[i]; }
#pragma unroll
  for (int i = 0; i < 4; i++) { d2[i] = d1[i + 1] - d1[i]; z[11 + i] = 20.0 * d2[i]; }
#pragma unroll
  for (int i = 0; i < 3; i++) z[15 + i] = 60.0 * (d2[i + 1] - d2[i]);
  if (first) {
    z[18] = t * c[0];
    z[19] = 5.0 * d1[0];
    z[20] = 20.0 * d2[0];
  } else {
    z[18] = t * c[0] - tp * p5;
    z[19] = (c[0] - c[1]) + (p5 - p4);
    z[20] = t * ((p3 - p4) - (p4 - p5)) - tp * d2[0];
  }
}

// g = A' v restricted to this lane's 6 variables; n18..n20 = NEXT lane's values on its rows 18..20
// (zero when this is the last segment), tn = next segment's duration
SP_DEV void apply_AT(const double v[QP_ROWS], double n18, double n19, double n20, double t, double tp, double tn,
                     bool first, double g[6]) {
#pragma unroll
  for (int i = 0; i < 6; i++) g[i] = t * v[i];
#pragma unroll
  for (int i = 0; i < 5; i++) { double e = 5.0 * v[6 + i]; g[i] -= e; g[i + 1] += e; }
#pragma unroll
  for (int i = 0; i < 4; i++) { double e = 20.0 * v[11 + i]; g[i] += e; g[i + 1] -= 2.0 * e; g[i + 2] += e; }
#pragma unroll
  for (int i = 0; i < 3; i++) {
    double e = 60.0 * v[15 + i];
    g[i] -= e; g[i + 1] += 3.0 * e; g[i + 2] -= 3.0 * e; g[i + 3] += e;
  }
  if (first) {
    g[0] += t * v[18] - 5.0 * v[19] + 20.0 * v[20];
    g[1] += 5.0 * v[19] - 40.0 * v[20];
    g[2] += 20.0 * v[20];
  } else {
    g[0] += t * v[18] + v[19] - tp * v[20];
    g[1] += -v[19] + 2.0 * tp * v[20];
    g[2] += -tp * v[20];
  }
  g[3] += tn * n20;
  g[4] += -n19 - 2.0 * tn * n20;
  g[5] += -t * n18 + n19 + tn * n20;
}

// y = P_k x with P_k packed lower triangle in shared memory
template <int STR>
SP_DEV void apply_P(const double *sm, int lane, const double x[6], double y[6]) {
#pragma unroll
  for (int i = 0; i < 6; i++) y[i] = 0.0;
#pragma unroll
  for (int i = 0; i < 6; i++)
#pragma unroll
    for (int j = 0; j <= i; j++) {
      double p = sm[(QP_SM_P + LT(i, j)) * STR + lane];
      y[i] += p * x[j];
      if (i != j) y[j] += p * x[i];
    }
}

// ------------------------------------------------------------------ joint reductions
// Reductions over the JW lanes that form ONE OSQP instance (the s-axis and the l-axis problem of a scenario, solved jointly
// like the reference does).  JW <= 32: adjacent lane groups of one warp.  JW = 64 (LPA = 32, K > 16): the two axis problems
// sit in the two WARPS of one CTA and meet through `xch` (QP_XCH_DOUBLES of shared memory) and the CTA barrier; both
// warps take every joint decision from the same reduced values, so they reach every barrier together.
template <int JW>
SP_DEV double qp_joint_max(double v, double *xch) {
  if (JW <= 32) return sp_group_max(v, JW);
  v = sp_group_max(v, 32);
  const int w = sp_warp_in_cta() & 1;
  xch[w] = v;  // (every lane writes the same value)
  sp_sync_cta();
  const double r = fmax(xch[0], xch[1]);
  sp_sync_cta();
  return r;
}
template <int JW>
SP_DEV double qp_joint_sum(double v, double *xch) {
  if (JW <= 32) return sp_group_sum(v, JW);
  v = sp_group_sum(v, 32);
  const int w = sp_warp_in_cta() & 1;
  xch[w] = v;
  sp_sync_cta();
  const double r = xch[0] + xch[1];
  sp_sync_cta();
  return r;
}
template <int JW>
SP_DEV int qp_joint_or(int v, double *xch) {
  if (JW <= 32) return sp_group_or(v, JW);
  return qp_joint_max<JW>(sp_group_or(v, 32) ? 1.0 : 0.0, xch) != 0.0 ? 1 : 0;
}

// ------------------------------------------------------------------ factorisation of S
struct QpFactor {
  double Linv[21];  // inverse of the diagonal Cholesky block (lower triangular)
  double C[18];     // Linv * B_k            (6x3, row major)   forward sweep
  double E[18];     // Linv' * B_{k+1}'      (6x3, row major)   backward sweep
};

// Builds S from (P block in smem, sig[6], rho[21] in smem slot `rho_slot`) and factorises it.
// Returns 0 on success, 1 if a pivot was not positive (lane-local flag; caller reduces).
template <int LPA, int STR>
// pol_scale == 0: ADMM mode, row penalty = rho slot.  pol_scale > 0: polish mode, row penalty =
// rho slot * pol_scale (/1e3 on equality rows) on the rows of `actmask`, zero elsewhere.
SP_DEV int qp_factorize(const double *sm, int lane, int rho_slot, const double sig[6], double t, double tp, double tn,
                        bool first, bool last, bool active, int seg, int kmaxw, unsigned actmask, unsigned eqmask,
                        double pol_scale, QpFactor &F) {
  double S[21], Bo[9];
  // diagonal block: P + sigma + own rows
#pragma unroll
  for (int i = 0; i < 6; i++)
#pragma unroll
    for (int j = 0; j <= i; j++) S[LT(i, j)] = sm[(QP_SM_P + LT(i, j)) * STR + lane] + (i == j ? sig[i] : 0.0);
#pragma unroll
  for (int e = 0; e < 9; e++) Bo[e] = 0.0;
  double rj[3];
#pragma unroll
  for (int r = 0; r < QP_ROWS; r++) {
    double rho = sm[(rho_slot + r) * STR + lane];
    if (pol_scale > 0.0) rho = ((actmask >> r) & 1u) ? rho * pol_scale * (((eqmask >> r) & 1u) ? 1e-3 : 1.0) : 0.0;
    if (r >= 18) rj[r - 18] = rho;
#pragma unroll
    for (int i = 0; i < 6; i++) {
      const double ai = row_coef(r, i, t, tp, first);
      if (ai == 0.0) continue;
#pragma unroll
      for (int j = 0; j <= i; j++) {
        const double aj = row_coef(r, j, t, tp, first);
        if (aj != 0.0) S[LT(i, j)] += rho * ai * aj;
      }
      if (r >= 18 && i < 3) {
#pragma unroll
        for (int j = 0; j < 3; j++) Bo[i * 3 + j] += rho * ai * prev_coef(r, j, t, tp, first);
      }
    }
  }
  // next lane's continuity rows touch my control points 3..5
  {
    double n0 = sp_shfl_down(rj[0], 1, LPA), n1 = sp_shfl_down(rj[1], 1, LPA), n2 = sp_shfl_down(rj[2], 1, LPA);
    if (last) { n0 = 0.0; n1 = 0.0; n2 = 0.0; }
    const double rn[3] = {n0, n1, n2};
#pragma unroll
    for (int r = 18; r < 21; r++)
#pragma unroll
      for (int i = 0; i < 3; i++) {
        const double bi = prev_coef(r, i, tn, t, false);
#pragma unroll
        for (int j = 0; j <= i; j++) S[LT(3 + i, 3 + j)] += rn[r - 18] * bi * prev_coef(r, j, tn, t, false);
      }
  }
  if (!active) {
#pragma unroll
    for (int i = 0; i < 6; i++)
#pragma unroll
      for (int j = 0; j <= i; j++) S[LT(i, j)] = (i == j) ? 1.0 : 0.0;
#pragma unroll
    for (int e = 0; e < 9; e++) Bo[e] = 0.0;
  }
  int bad = 0;
  double Bk[9];
#pragma unroll
  for (int e = 0; e < 9; e++) Bk[e] = 0.0;
#pragma unroll
  for (int e = 0; e < 21; e++) F.Linv[e] = 0.0;
  for (int step = 0; step < kmaxw; step++) {
    // lower-right 3x3 of the previous lane's Linv (its inverse-transpose multiplies my coupling)
    double u[6];
    u[0] = sp_shfl_up(F.Linv[LT(3, 3)], 1, LPA);
    u[1] = sp_shfl_up(F.Linv[LT(4, 3)], 1, LPA);
    u[2] = sp_shfl_up(F.Linv[LT(4, 4)], 1, LPA);
    u[3] = sp_shfl_up(F.Linv[LT(5, 3)], 1, LPA);
    u[4] = sp_shfl_up(F.Linv[LT(5, 4)], 1, LPA);
    u[5] = sp_shfl_up(F.Linv[LT(5, 5)], 1, LPA);
    if (seg == step) {
      if (step > 0 && active) {
        // B_k = Bo * Linv_prev[3..5,3..5]' ; U[a][b] = Lp(3+b,3+a), a <= b
#pragma unroll
        for (int i = 0; i < 3; i++) {
          const double b0 = Bo[i * 3 + 0], b1 = Bo[i * 3 + 1], b2 = Bo[i * 3 + 2];
          Bk[i * 3 + 0] = b0 * u[0];
          Bk[i * 3 + 1] = b0 * u[1] + b1 * u[2];
          Bk[i * 3 + 2] = b0 * u[3] + b1 * u[4] + b2 * u[5];
        }
#pragma unroll
        for (int i = 0; i < 3; i++)
#pragma unroll
          for (int j = 0; j <= i; j++)
            S[LT(i, j)] -= Bk[i * 3 + 0] * Bk[j * 3 + 0] + Bk[i * 3 + 1] * Bk[j * 3 + 1] + Bk[i * 3 + 2] * Bk[j * 3 + 2];
      }
      // Cholesky of the 6x6 block, then its inverse
      double Lc[21];
#pragma unroll
      for (int j = 0; j < 6; j++) {
        double d = S[LT(j, j)];
#pragma unroll
        for (int k = 0; k < j; k++) d -= Lc[LT(j, k)] * Lc[LT(j, k)];
        if (!(d > 0.0)) { bad = 1; d = 1.0; }
        const double ljj = sqrt(d);
        Lc[LT(j, j)] = ljj;
        const double inv = 1.0 / ljj;
#pragma unroll
        for (int i = j + 1; i < 6; i++) {
          double s = S[LT(i, j)];
#pragma unroll
          for (int k = 0; k < j; k++) s -= Lc[LT(i, k)] * Lc[LT(j, k)];
          Lc[LT(i, j)] = s * inv;
        }
      }
#pragma unroll
      for (int j = 0; j < 6; j++) {
        F.Linv[LT(j, j)] = 1.0 / Lc[LT(j, j)];
#pragma unroll
        for (int i = j + 1; i < 6; i++) {
          double s = 0.0;
#pragma unroll
          for (int k = j; k < i; k++) s -= Lc[LT(i, k)] * F.Linv[LT(k, j)];
          F.Linv[LT(i, j)] = s / Lc[LT(i, i)];
        }
      }
    }
  }
  // C = Linv[:, 0..2] * Bk
#pragma unroll
  for (int i = 0; i < 6; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) {
      double s = 0.0;
#pragma unroll
      for (int a = 0; a < 3; a++)
        if (a <= i) s += F.Linv[LT(i, a)] * Bk[a * 3 + j];
      F.C[i * 3 + j] = s;
    }
  // E = Linv'[:, 3..5] * Bnext'
  double Bn[9];
#pragma unroll
  for (int e = 0; e < 9; e++) Bn[e] = sp_shfl_down(Bk[e], 1, LPA);
  if (last || !active) {
#pragma unroll
    for (int e = 0; e < 9; e++) Bn[e] = 0.0;
  }
#pragma unroll
  for (int i = 0; i < 6; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) {
      double s = 0.0;
#pragma unroll
      for (int a = 3; a < 6; a++)
        if (a >= i) s += F.Linv[LT(a, i)] * Bn[j * 3 + (a - 3)];
      F.E[i * 3 + j] = s;
    }
  return bad;
}

// x = S^{-1} r
template <int LPA>
SP_DEV void qp_solve(const QpFactor &F, const double r[6], double x[6], int seg, bool last, int kmaxw) {
  double y[6];
#pragma unroll
  for (int i = 0; i < 6; i++) {
    double s = 0.0;
#pragma unroll
    for (int j = 0; j <= i; j++) s += F.Linv[LT(i, j)] * r[j];
    y[i] = s;
  }
  // forward sweep: y_k -= C_k * y_{k-1}[3..5]; only rows 3..5 are on the critical path
  for (int step = 1; step < kmaxw; step++) {
    const double s0 = sp_shfl_up(y[3], 1, LPA), s1 = sp_shfl_up(y[4], 1, LPA), s2 = sp_shfl_up(y[5], 1, LPA);
    if (seg == step) {
#pragma unroll
      for (int i = 3; i < 6; i++) y[i] -= F.C[i * 3 + 0] * s0 + F.C[i * 3 + 1] * s1 + F.C[i * 3 + 2] * s2;
    }
  }
  {
    const double s0 = sp_shfl_up(y[3], 1, LPA), s1 = sp_shfl_up(y[4], 1, LPA), s2 = sp_shfl_up(y[5], 1, LPA);
    if (seg > 0) {
#pragma unroll
      for (int i = 0; i < 3; i++) y[i] -= F.C[i * 3 + 0] * s0 + F.C[i * 3 + 1] * s1 + F.C[i * 3 + 2] * s2;
    }
  }
#pragma unroll
  for (int i = 0; i < 6; i++) {
    double s = 0.0;
#pragma unroll
    for (int a = i; a < 6; a++) s += F.Linv[LT(a, i)] * y[a];
    x[i] = s;
  }
  // backward sweep: x_k -= E_k * x_{k+1}[0..2]; rows 0..2 are on the critical path
  for (int step = kmaxw - 2; step >= 0; step--) {
    const double n0 = sp_shfl_down(x[0], 1, LPA), n1 = sp_shfl_down(x[1], 1, LPA), n2 = sp_shfl_down(x[2], 1, LPA);
    if (seg == step && !last) {
#pragma unroll
      for (int i = 0; i < 3; i++) x[i] -= F.E[i * 3 + 0] * n0 + F.E[i * 3 + 1] * n1 + F.E[i * 3 + 2] * n2;
    }
  }
  {
    const double n0 = sp_shfl_down(x[0], 1, LPA), n1 = sp_shfl_down(x[1], 1, LPA), n2 = sp_shfl_down(x[2], 1, LPA);
    if (!last) {
#pragma unroll
      for (int i = 3; i < 6; i++) x[i] -= F.E[i * 3 + 0] * n0 + F.E[i * 3 + 1] * n1 + F.E[i * 3 + 2] * n2;
    }
  }
}

SP_DEV double limit_scaling(double v) {
  v = v < 1e-4 ? 1.0 : v;
  return v > 1e4 ? 1e4 : v;
}

struct QpResid {
  double pri, dua, nz, nax, nq, npx, naty;
};

// residuals of (x, w) in OSQP's scaled space; z = clip(w), y = rho (w - z).  RW = reduction width:
// LPA for one axis problem, 2*LPA for the joint (s, l) problem held by two adjacent lane groups.
template <int LPA, int STR, int RW>
SP_DEV QpResid qp_residuals(const double *sm, int lane, const double x[6], const double q[6], const double cD[6],
                            double c_over_rhobar, unsigned eqmask, double t, double tp, double tn, bool first, bool last,
                            bool active, double *xch = nullptr) {
  double Ax[QP_ROWS], y[QP_ROWS];
  {
    double p3 = sp_shfl_up(x[3], 1, LPA), p4 = sp_shfl_up(x[4], 1, LPA), p5 = sp_shfl_up(x[5], 1, LPA);
    apply_A(x, p3, p4, p5, t, tp, first, Ax);
  }
  double pri = 0.0, nz = 0.0, nax = 0.0;
#pragma unroll
  for (int r = 0; r < QP_ROWS; r++) {
    const double w = sm[(QP_SM_W + r) * STR + lane], l = sm[(QP_SM_L + r) * STR + lane], u = sm[(QP_SM_U + r) * STR + lane];
    const double rho = sm[(QP_SM_RHO + r) * STR + lane];
    const double z = fmin(fmax(w, l), u);
    y[r] = rho * (w - z);
    const double eqf = ((eqmask >> r) & 1u) ? 1e-3 : 1.0;
    const double E = sqrt(rho * c_over_rhobar * eqf);
    pri = fmax(pri, E * fabs(Ax[r] - z));
    nz = fmax(nz, E * fabs(z));
    nax = fmax(nax, E * fabs(Ax[r]));
  }
  double aty[6], px[6];
  {
    double n18 = sp_shfl_down(y[18], 1, LPA), n19 = sp_shfl_down(y[19], 1, LPA), n20 = sp_shfl_down(y[20], 1, LPA);
    if (last) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
    apply_AT(y, n18, n19, n20, t, tp, tn, first, aty);
  }
  apply_P<STR>(sm, lane, x, px);
  double dua = 0.0, nq = 0.0, npx = 0.0, naty = 0.0;
#pragma unroll
  for (int j = 0; j < 6; j++) {
    dua = fmax(dua, cD[j] * fabs(px[j] + q[j] + aty[j]));
    nq = fmax(nq, cD[j] * fabs(q[j]));
    npx = fmax(npx, cD[j] * fabs(px[j]));
    naty = fmax(naty, cD[j] * fabs(aty[j]));
  }
  QpResid R;
  if (!active) { pri = 0; dua = 0; nz = 0; nax = 0; nq = 0; npx = 0; naty = 0; }
  R.pri = qp_joint_max<RW>(pri, xch); R.dua = qp_joint_max<RW>(dua, xch); R.nz = qp_joint_max<RW>(nz, xch);
  R.nax = qp_joint_max<RW>(nax, xch); R.nq = qp_joint_max<RW>(nq, xch); R.npx = qp_joint_max<RW>(npx, xch);
  R.naty = qp_joint_max<RW>(naty, xch);
  return R;
}

// ------------------------------------------------------------------ per-lane problem state
// Lane-per-segment layout: LPA lanes hold one axis problem, lane `seg` owns segment `seg`.  JW is the
// joint width: with JW = 2*LPA the s-axis and l-axis problems of one scenario sit in adjacent lane groups
// and are solved as ONE OSQP instance like the reference does (one cost scaling c, one rho, joint
// termination / infeasibility norms, solve_3d.cc:1211-1249); with JW = LPA each axis is its own instance.
struct QpLane {
  int b, axis, K, seg, kmaxw;
  bool have, active, first, last;
  double t, tp, tn;
  double q[6], sig[6], cD[6];
  double c, rhobar;
  unsigned eqmask;
  double *xch;  // cross-warp exchange scratch (JW = 64 only)
  int pre;  // interval pre-check: the scenario's corridor is provably empty (SpectralOptions::infeasibility_precheck)
};

// K3 + Ruiz equilibration + per-row rho: fills the shared-memory slots L, U, W (= 0), P, RHO of this
// lane and the lane state.  `lane` is the shared-memory column of this lane (slot * STR + lane).
template <int LPA, int STR, int JW>
SP_DEV void qp_setup(const QpArgs &a, int ap, bool have, int seg, int lane, double *sm, QpLane &Q, double *xch = nullptr) {
  const int b = have ? a.list[ap >> 1] : 0;
  const int axis = ap & 1;
  const int K = have ? a.K[b] : 0;
  const bool active = have && seg < K;
  const bool first = seg == 0, last = seg == K - 1;
  const int kmaxw = sp_group_max_i(K, 32);
  const SpOptionsDev &o = a.opt;
  const int N = a.N;
  const double delta = a.delta;

  // ---------------- K3: assemble this lane's rows ----------------
  SpectralCube cube;
  if (active) cube = a.segs[(size_t)b * a.k_max + seg];
  else { cube.beg_t = 0; cube.end_t = 0; cube.t = 1.0; cube.beg_l = 0; cube.end_l = 0; cube.upp_skew = 0; cube.upp_bias = 0;
         cube.down_skew = 0; cube.down_bias = 0; cube.l_upp_skew = 0; cube.l_upp_bias = 0; cube.l_down_skew = 0; cube.l_down_bias = 0; }
  const double t = cube.t;
  double tp = sp_shfl_up(t, 1, LPA), tn = sp_shfl_down(t, 1, LPA);
  if (first) tp = 1.0;
  if (last || !active) tn = 1.0;
  const size_t bi = (size_t)b * a.in_stride;  // input scenario of this lane
  const double *sc = a.scalars + 10 * bi;
  const double *wv = a.weights + (size_t)(a.wstride ? b : 0) * 10;
  const double *ref = (axis == 0 ? a.s_ref : a.l_ref) + bi * N;
  const double *ini = a.init + 6 * bi + 3 * axis;
  const double invm[6] = {SP_INVM1_0, SP_INVM1_1, SP_INVM1_2, SP_INVM1_3, SP_INVM1_4, SP_INVM1_5};
  double lo[QP_ROWS], hi[QP_ROWS];
  // containment rows (solve_3d.cc:823-832, :961-977; cuboid_3d.cc:677-697, :826-827)
  if (axis == 0) {
    if (a.variant == SPECTRAL_CUB) {
      double lb = 0, ub = 100;
#pragma unroll
      for (int i = 0; i < 6; i++) {
        const double e_lo = rn_add(cube.down_bias, rn_mul(rn_mul(cube.down_skew, invm[i]), t));
        const double e_hi = rn_add(cube.upp_bias, rn_mul(rn_mul(cube.upp_skew, invm[i]), t));
        lb = (lb < e_lo) ? e_lo : lb;  // std::max(l_bound, e)
        ub = (e_hi < ub) ? e_hi : ub;  // std::min(u_bound, e)
      }
#pragma unroll
      for (int i = 0; i < 6; i++) { lo[i] = lb; hi[i] = ub; }
    } else {
#pragma unroll
      for (int i = 0; i < 6; i++) {
        lo[i] = rn_add(cube.down_bias, rn_mul(rn_mul(cube.down_skew, invm[i]), t));
        hi[i] = rn_add(cube.upp_bias, rn_mul(rn_mul(cube.upp_skew, invm[i]), t));
      }
    }
  } else {
    if (a.variant == SPECTRAL_CUB) {
#pragma unroll
      for (int i = 0; i < 6; i++) { lo[i] = cube.beg_l; hi[i] = cube.end_l; }
    } else {
#pragma unroll
      for (int i = 0; i < 6; i++) {
        lo[i] = rn_add(cube.l_down_bias, rn_mul(rn_mul(cube.l_down_skew, invm[i]), t));
        hi[i] = rn_add(cube.l_upp_bias, rn_mul(rn_mul(cube.l_upp_skew, invm[i]), t));
      }
    }
  }
  // velocity / acceleration / jerk rows (:835-888, :994-1037)
  if (axis == 0) {
    double d_lo = 0.0, d_hi = 1000.0, dd_lo = -1000.0, dd_hi = 1000.0;
    if (active) {
      const double *dsb = a.ds_bounds + bi * N * 2;
      for (int i = cube.beg_t; i <= cube.end_t; i++) {
        const double blo = dsb[2 * i], bhi = dsb[2 * i + 1];
        d_lo = (blo < d_lo) ? d_lo : blo;  // std::max(bound, cur)
        d_hi = (d_hi < bhi) ? d_hi : bhi;  // std::min(bound, cur)
        dd_lo = (sc[2] < dd_lo) ? dd_lo : sc[2];
        dd_hi = (dd_hi < sc[3]) ? dd_hi : sc[3];
      }
    }
#pragma unroll
    for (int i = 0; i < 5; i++) { lo[6 + i] = d_lo; hi[6 + i] = d_hi; }
#pragma unroll
    for (int i = 0; i < 4; i++) { lo[11 + i] = rn_mul(dd_lo, t); hi[11 + i] = rn_mul(dd_hi, t); }
#pragma unroll
    for (int i = 0; i < 3; i++) { lo[15 + i] = rn_mul(rn_mul(sc[4], t), t); hi[15 + i] = rn_mul(rn_mul(sc[5], t), t); }
  } else {
    const double *dlb = a.dl_bounds + bi * N * 2;
#pragma unroll
    for (int i = 0; i < 5; i++) { lo[6 + i] = dlb[2 * i]; hi[6 + i] = dlb[2 * i + 1]; }  // dy_bounds_[i]: control index (:1003)
#pragma unroll
    for (int i = 0; i < 4; i++) { lo[11 + i] = rn_mul(sc[6], t); hi[11 + i] = rn_mul(sc[7], t); }
#pragma unroll
    for (int i = 0; i < 3; i++) { lo[15 + i] = rn_mul(rn_mul(sc[8], t), t); hi[15 + i] = rn_mul(rn_mul(sc[9], t), t); }
  }
  if (first) {  // :896-912
    lo[18] = hi[18] = ini[0];
    lo[19] = hi[19] = ini[1];
    lo[20] = hi[20] = rn_mul(ini[2], t);
  } else {
    lo[18] = hi[18] = 0.0; lo[19] = hi[19] = 0.0; lo[20] = hi[20] = 0.0;
  }
  // optional interval pre-check (include/spectral.h: infeasibility_precheck): necessary conditions of feasibility on the
  // raw rows -- no row with l > u; the position intervals of consecutive segments meet at their joint (row 5 of segment
  // k - 1 and row 0 of segment k bound the same quantity, t_{k-1} c_{k-1,5} = t_k c_{k,0}); the initial state lies inside
  // the first segment's position / velocity / acceleration rows (rows 18..20 are equalities on the expressions of rows
  // 0, 6, 11).  OR-ed over the JW lanes that form one OSQP instance.
  // Always: OSQP's validate_data (run by osqp_setup) refuses a problem with a row l > u before the first iteration (the
  // reference then dereferences the NULL workspace, solve_3d.cc:1251); such a scenario fails with 0 iterations here.
  int pre = 0;
  bool bad = false;
  if (active) {
#pragma unroll
    for (int r = 0; r < 18; r++) bad = bad || (lo[r] > hi[r]);
  }
  if (o.precheck) {
    const double mg = o.precheck_margin;
    const double plo = sp_shfl_up(lo[5], 1, LPA), phi = sp_shfl_up(hi[5], 1, LPA);
    if (active && !first) {
      const double jl = lo[0] > plo ? lo[0] : plo, jh = hi[0] < phi ? hi[0] : phi;
      bad = bad || (jl > jh + mg);
    }
    if (active && first) {
      bad = bad || (lo[18] > hi[0] + mg) || (lo[18] < lo[0] - mg);
      bad = bad || (lo[19] > hi[6] + mg) || (lo[19] < lo[6] - mg);
      bad = bad || (lo[20] > hi[11] + mg) || (lo[20] < lo[11] - mg);
    }
  }
  pre = qp_joint_or<JW>(bad ? 1 : 0, xch);
  if (a.lu != nullptr && active) {
    double *dst = a.lu + (((size_t)b * 2 + axis) * a.k_max + seg) * QP_ROWS * 2;
#pragma unroll
    for (int r = 0; r < QP_ROWS; r++) { dst[2 * r] = lo[r]; dst[2 * r + 1] = hi[r]; }
  }
  // q (:226-321): x/y skew & bias from ref[10k], ref[10k+1] regardless of beg_t (:1159-1166);
  // ref[j >= N] reads as 0.0 like the shipped binary (SURVEY.md Appendix E-10)
  double q[6];
  {
    const double w_ref = wv[axis == 0 ? 4 : 6], w_dref = wv[axis == 0 ? 5 : 7], dref = sc[axis];
    const int j0 = 10 * seg, j1 = 10 * seg + 1;
    const double r0 = (active && j0 < N) ? ref[j0] : 0.0, r1 = (active && j1 < N) ? ref[j1] : 0.0;
    const double skew = (r1 - r0) / delta, bias = r0;
    const double t2 = t * t, t3 = t2 * t;
    double qp_[6];
#pragma unroll
    for (int i = 0; i < 6; i++) {
      double v = -2.0 * t3 * w_ref * skew / (double)(i + 2);
      v += -2.0 * t2 * w_ref * bias / (double)(i + 1);
      if (i > 0) v += -2.0 * w_dref * dref * t;
      qp_[i] = v;
    }
    const double M[6][6] = {{1, 0, 0, 0, 0, 0}, {-5, 5, 0, 0, 0, 0}, {10, -20, 10, 0, 0, 0},
                            {-10, 30, -30, 10, 0, 0}, {5, -20, 30, -20, 5, 0}, {-1, 5, -10, 10, -5, 1}};
#pragma unroll
    for (int j = 0; j < 6; j++) {
      double s = 0.0;
#pragma unroll
      for (int i = 0; i < 6; i++) s += qp_[i] * M[i][j];
      q[j] = s;
    }
    if (last && active) q[5] -= dref * 2.0 * ref[N - 1] * t;  // :268 / :315
    if (!active) {
#pragma unroll
      for (int j = 0; j < 6; j++) q[j] = 0.0;
    }
  }
  // P block (:145-222)
  {
    const double *mq = a.mqm + ((size_t)(a.wstride ? b : 0) * 2 + axis) * 84;
    const double t3 = t * t * t, it = 1.0 / t, it3 = 1.0 / t3;
#pragma unroll
    for (int e = 0; e < 21; e++) {
      double v = t3 * mq[e] + t * mq[21 + e] + mq[42 + e] * it + mq[63 + e] * it3;
      if (e == 20 && last) v += wv[8 + axis] * t * t;
      sm[(QP_SM_P + e) * STR + lane] = active ? 2.0 * v : (e == LT(0, 0) || e == LT(1, 1) || e == LT(2, 2) || e == LT(3, 3) || e == LT(4, 4) || e == LT(5, 5) ? 1.0 : 0.0);
    }
  }
#pragma unroll
  for (int r = 0; r < QP_ROWS; r++) {
    sm[(QP_SM_L + r) * STR + lane] = active ? lo[r] : -1.0;
    sm[(QP_SM_U + r) * STR + lane] = active ? hi[r] : 1.0;
    sm[(QP_SM_W + r) * STR + lane] = 0.0;
  }
  sp_syncwarp();

  // ---------------- Ruiz equilibration (OSQP scaling.c, `scaling` passes) ----------------
  double D[6], E[QP_ROWS], c = 1.0;
#pragma unroll
  for (int j = 0; j < 6; j++) D[j] = 1.0;
#pragma unroll
  for (int r = 0; r < QP_ROWS; r++) E[r] = 1.0;
  const double nvars = (double)(6 * K) * (JW / LPA);
  for (int pass = 0; pass < o.scaling; pass++) {
    double cn[6], rn_[QP_ROWS];
    // column norms of [P; A] and row norms of A in the current scaling
    double Dp3 = sp_shfl_up(D[3], 1, LPA), Dp4 = sp_shfl_up(D[4], 1, LPA), Dp5 = sp_shfl_up(D[5], 1, LPA);
    double En18 = sp_shfl_down(E[18], 1, LPA), En19 = sp_shfl_down(E[19], 1, LPA), En20 = sp_shfl_down(E[20], 1, LPA);
    if (last) { En18 = 0; En19 = 0; En20 = 0; }
    const double Dp[3] = {Dp3, Dp4, Dp5};
    const double En[3] = {En18, En19, En20};
#pragma unroll
    for (int j = 0; j < 6; j++) {
      double m = 0.0;
#pragma unroll
      for (int i = 0; i < 6; i++) {
        const double p = sm[(QP_SM_P + (i >= j ? LT(i, j) : LT(j, i))) * STR + lane];
        m = fmax(m, c * D[i] * fabs(p) * D[j]);
      }
      cn[j] = m;
    }
#pragma unroll
    for (int r = 0; r < QP_ROWS; r++) {
      double m = 0.0;
#pragma unroll
      for (int j = 0; j < 6; j++) {
        const double av = fabs(row_coef(r, j, t, tp, first));
        if (av != 0.0) {
          const double e = E[r] * av * D[j];
          m = fmax(m, e);
          cn[j] = fmax(cn[j], e);
        }
      }
      if (r >= 18) {
#pragma unroll
        for (int j = 0; j < 3; j++) m = fmax(m, E[r] * fabs(prev_coef(r, j, t, tp, first)) * Dp[j]);
      }
      rn_[r] = m;
    }
#pragma unroll
    for (int r = 18; r < 21; r++)
#pragma unroll
      for (int j = 0; j < 3; j++) cn[3 + j] = fmax(cn[3 + j], En[r - 18] * fabs(prev_coef(r, j, tn, t, false)) * D[3 + j]);
#pragma unroll
    for (int j = 0; j < 6; j++) D[j] *= 1.0 / sqrt(limit_scaling(cn[j]));
#pragma unroll
    for (int r = 0; r < QP_ROWS; r++) E[r] *= 1.0 / sqrt(limit_scaling(rn_[r]));
    // cost normalisation: mean column norm of the scaled P vs ||q||inf
    double colsum = 0.0, qn = 0.0;
#pragma unroll
    for (int j = 0; j < 6; j++) {
      double m = 0.0;
#pragma unroll
      for (int i = 0; i < 6; i++) {
        const double p = sm[(QP_SM_P + (i >= j ? LT(i, j) : LT(j, i))) * STR + lane];
        m = fmax(m, c * D[i] * fabs(p) * D[j]);
      }
      colsum += m;
      qn = fmax(qn, c * D[j] * fabs(q[j]));
    }
    if (!active) { colsum = 0.0; qn = 0.0; }
    colsum = qp_joint_sum<JW>(colsum, xch);
    qn = qp_joint_max<JW>(qn, xch);
    double ct = colsum / (nvars > 0 ? nvars : 1.0);
    qn = limit_scaling(qn);
    ct = ct > qn ? ct : qn;
    ct = 1.0 / limit_scaling(ct);
    c *= ct;
  }
  // per-row rho base, equality mask, per-variable sigma
  unsigned eqmask = 0;
  double rhobar = o.rho0;
  double sig[6], cD[6];
#pragma unroll
  for (int j = 0; j < 6; j++) { sig[j] = o.sigma / (c * D[j] * D[j]); cD[j] = c * D[j]; }
#pragma unroll
  for (int r = 0; r < QP_ROWS; r++) {
    const bool eq = (E[r] * sm[(QP_SM_U + r) * STR + lane] - E[r] * sm[(QP_SM_L + r) * STR + lane]) < 1e-4;  // RHO_TOL, scaled bounds
    if (eq) eqmask |= 1u << r;
    sm[(QP_SM_RHO + r) * STR + lane] = rhobar * (eq ? 1e3 : 1.0) * E[r] * E[r] / c;
  }
  sp_syncwarp();

  Q.b = b; Q.axis = axis; Q.K = K; Q.seg = seg; Q.kmaxw = kmaxw;
  Q.have = have; Q.active = active; Q.first = first; Q.last = last;
  Q.t = t; Q.tp = tp; Q.tn = tn; Q.c = c; Q.rhobar = rhobar; Q.eqmask = eqmask; Q.pre = pre; Q.xch = xch;
#pragma unroll
  for (int j = 0; j < 6; j++) { Q.q[j] = q[j]; Q.sig[j] = sig[j]; Q.cD[j] = cD[j]; }
}

#define QP_UNPACK_LANE(Q)                                                                              \
  const int b = Q.b, axis = Q.axis, K = Q.K, seg = Q.seg, kmaxw = Q.kmaxw;                             \
  const bool have = Q.have, active = Q.active, first = Q.first, last = Q.last;                         \
  const double t = Q.t, tp = Q.tp, tn = Q.tn, c = Q.c;                                                 \
  const unsigned eqmask = Q.eqmask;                                                                    \
  const double *q = Q.q, *sig = Q.sig, *cD = Q.cD;                                                     \
  (void)b; (void)axis; (void)K; (void)seg; (void)kmaxw; (void)have; (void)active; (void)first; (void)last; \
  (void)t; (void)tp; (void)tn; (void)c; (void)eqmask; (void)q; (void)sig; (void)cD

// A block of `n` ADMM iterations WITHOUT a termination check, fused so that every iteration makes ONE pass over the lane's
// 21 rows: the row update of iteration i (w += alpha (z~ - clip(w))) and the gather input of iteration i + 1
// (v = rho (2 clip(w') - w')) come from the same loads.  Same arithmetic per quantity as the general iteration of
// qp_admm_lanes below (which handles iteration 1, the check iterations and the rho updates), so the two can be interleaved.
// Rows are staged in groups of CH (loads, arithmetic, stores) to bound the live registers next to the factor.
SP_DEV double qp_ld(const double *p) {
#ifdef SPECTRAL_CPU_EMU
  return *p;
#else
  double a;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(a) : "r"((unsigned)__cvta_generic_to_shared(p)));
  return a;
#endif
}
template <int LPA, int STR, int RB, int RE, int CH, bool FIRST>
SP_DEV void qp_fast_rows(double *sm, int lane, const double z[QP_ROWS], double alpha_eff, double v[QP_ROWS]) {
  static_assert((RE - RB) % CH == 0, "whole groups");
#pragma unroll
  for (int r0 = RB; r0 < RE; r0 += CH) {
    double w[CH], l[CH], u[CH], rh[CH];
#pragma unroll
    for (int j = 0; j < CH; j++) {
      w[j] = qp_ld(sm + (QP_SM_W + r0 + j) * STR + lane); l[j] = qp_ld(sm + (QP_SM_L + r0 + j) * STR + lane);
      u[j] = qp_ld(sm + (QP_SM_U + r0 + j) * STR + lane); rh[j] = qp_ld(sm + (QP_SM_RHO + r0 + j) * STR + lane);
    }
#pragma unroll
    for (int j = 0; j < CH; j++) {
      const int r = r0 + j;
      if (FIRST) {   // block entry: only the gather input of the first iteration
        const double p = fmin(fmax(w[j], l[j]), u[j]);
        v[r] = rh[j] * (2.0 * p - w[j]);
      } else {
        const double p = fmin(fmax(w[j], l[j]), u[j]);
        const double wn = w[j] + alpha_eff * (z[r] - p);
        const double pn = fmin(fmax(wn, l[j]), u[j]);
        v[r] = rh[j] * (2.0 * pn - wn);
        w[j] = wn;
      }
    }
    if (!FIRST) {
#pragma unroll
      for (int j = 0; j < CH; j++) sm[(QP_SM_W + r0 + j) * STR + lane] = w[j];
    }
  }
}
template <int LPA, int STR>
SP_DEV void qp_fast_block(double *sm, int lane, const QpFactor &F, double x[6], const double q[6], const double sig[6], double t, double tp,
                          double tn, bool first, bool last, int seg, int kmaxw, double alpha, bool run, int n) {
  const double alpha_eff = run ? alpha : 0.0;   // a finished lane keeps its state
  double g[6];
  {
    double v[QP_ROWS];
    qp_fast_rows<LPA, STR, 0, 21, 7, true>(sm, lane, v, 0.0, v);
    double n18 = sp_shfl_down(v[18], 1, LPA), n19 = sp_shfl_down(v[19], 1, LPA), n20 = sp_shfl_down(v[20], 1, LPA);
    if (last) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
    apply_AT(v, n18, n19, n20, t, tp, tn, first, g);
#pragma unroll
    for (int j = 0; j < 6; j++) g[j] += sig[j] * x[j] - q[j];
  }
  for (int i = 0; i < n; i++) {
    double xt[6];
    qp_solve<LPA>(F, g, xt, seg, last, kmaxw);
    if (run) {
#pragma unroll
      for (int j = 0; j < 6; j++) x[j] = alpha * xt[j] + (1.0 - alpha) * x[j];
    }
    double v[QP_ROWS];
    {
      double p3 = sp_shfl_up(xt[3], 1, LPA), p4 = sp_shfl_up(xt[4], 1, LPA), p5 = sp_shfl_up(xt[5], 1, LPA);
      apply_A(xt, p3, p4, p5, t, tp, first, v);  // v holds z_tilde ...
    }
    qp_fast_rows<LPA, STR, 0, 21, 7, false>(sm, lane, v, alpha_eff, v);   // ... and then rho (2 clip(w') - w') row by row
    double n18 = sp_shfl_down(v[18], 1, LPA), n19 = sp_shfl_down(v[19], 1, LPA), n20 = sp_shfl_down(v[20], 1, LPA);
    if (last) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
    apply_AT(v, n18, n19, n20, t, tp, tn, first, g);
#pragma unroll
    for (int j = 0; j < 6; j++) g[j] += sig[j] * x[j] - q[j];
  }
}

// The lane-per-segment ADMM loop (OSQP iteration in w form) with the factor F in registers.
// Used by k_qp (segment counts above the dense kernel's capacity) and as the kernel-logic reference of
// the dense loop in qp_dense.cuh.
template <int LPA, int STR, int JW>
SP_DEV void qp_admm_lanes(const SpOptionsDev &o, double *sm, int lane, QpLane &Q, QpFactor &F, double x[6], int &state,
                          int &iters) {
  QP_UNPACK_LANE(Q);
  double rhobar = Q.rhobar;
  int bad = qp_factorize<LPA, STR>(sm, lane, QP_SM_RHO, sig, t, tp, tn, first, last, active, seg, kmaxw, 0u, eqmask, 0.0, F);
  bad = qp_joint_or<JW>(bad, Q.xch);

  // ---------------- ADMM (OSQP iteration in w form) ----------------
#pragma unroll
  for (int j = 0; j < 6; j++) x[j] = 0.0;
  state = (have && K > 0) ? QP_RUNNING : QP_ST_MAXITER;
  if (bad || Q.pre) state = QP_ST_INFEASIBLE;
  iters = 0;
  const double alpha = o.alpha;

  for (int it = 1; it <= o.max_iter; it++) {
    if (sp_all(state != QP_RUNNING)) break;
    const bool run = state == QP_RUNNING;
    const bool check = (o.check_every > 0) && (it % o.check_every == 0);
    if (it > 1 && !check) {
      // the iterations up to (not including) the next check, or to max_iter: the state cannot change inside the block
      int it_end = o.max_iter + 1;
      if (o.check_every > 0) {
        const int nxt = (it / o.check_every + 1) * o.check_every;
        it_end = nxt < it_end ? nxt : it_end;
      }
      qp_fast_block<LPA, STR>(sm, lane, F, x, q, sig, t, tp, tn, first, last, seg, kmaxw, alpha, run, it_end - it);
      if (run) iters = it_end - 1;
      it = it_end - 1;
      continue;
    }
    double v[QP_ROWS];
    // v = rho (2 clip(w) - w)  (= rho z - y); first iteration: z = y = 0 exactly as OSQP's cold start
#pragma unroll
    for (int r = 0; r < QP_ROWS; r++) {
      const double w = sm[(QP_SM_W + r) * STR + lane], l = sm[(QP_SM_L + r) * STR + lane], u = sm[(QP_SM_U + r) * STR + lane];
      const double rho = sm[(QP_SM_RHO + r) * STR + lane];
      const double p = fmin(fmax(w, l), u);
      v[r] = (it == 1) ? 0.0 : rho * (2.0 * p - w);
    }
    double g[6], xt[6];
    {
      double n18 = sp_shfl_down(v[18], 1, LPA), n19 = sp_shfl_down(v[19], 1, LPA), n20 = sp_shfl_down(v[20], 1, LPA);
      if (last) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
      apply_AT(v, n18, n19, n20, t, tp, tn, first, g);
    }
#pragma unroll
    for (int j = 0; j < 6; j++) g[j] += sig[j] * x[j] - q[j];
    qp_solve<LPA>(F, g, xt, seg, last, kmaxw);
    {
      double p3 = sp_shfl_up(xt[3], 1, LPA), p4 = sp_shfl_up(xt[4], 1, LPA), p5 = sp_shfl_up(xt[5], 1, LPA);
      apply_A(xt, p3, p4, p5, t, tp, first, v);  // v now holds z_tilde
    }
    // primal-infeasibility certificate needs delta_y of this iteration (only on check iterations)
    double dy_norm = 0.0, dy_lhs = 0.0;
    if (run) {
#pragma unroll
      for (int j = 0; j < 6; j++) x[j] = alpha * xt[j] + (1.0 - alpha) * x[j];
#pragma unroll
      for (int r = 0; r < QP_ROWS; r++) {
        const double w = sm[(QP_SM_W + r) * STR + lane], l = sm[(QP_SM_L + r) * STR + lane], u = sm[(QP_SM_U + r) * STR + lane];
        const double p = (it == 1) ? 0.0 : fmin(fmax(w, l), u);  // z_prev
        const double wn = (it == 1) ? alpha * v[r] : w + alpha * (v[r] - p);
        sm[(QP_SM_W + r) * STR + lane] = wn;
        if (check) {
          const double rho = sm[(QP_SM_RHO + r) * STR + lane];
          const double yo = (it == 1) ? 0.0 : rho * (w - p);
          const double yn = rho * (wn - fmin(fmax(wn, l), u));
          const double dy = yn - yo;
          v[r] = dy;
          const double eqf = ((eqmask >> r) & 1u) ? 1e-3 : 1.0;
          const double Er = sqrt(rho * (c / rhobar) * eqf);
          dy_norm = fmax(dy_norm, fabs(c * dy / Er));
          dy_lhs += c * (u * fmax(dy, 0.0) + l * fmin(dy, 0.0));
        }
      }
    }
    if (run) iters = it;
    if (check) {
      QpResid R = qp_residuals<LPA, STR, JW>(sm, lane, x, q, cD, c / rhobar, eqmask, t, tp, tn, first, last, active, Q.xch);
      const double eps_p = o.eps_abs + o.eps_rel * fmax(R.nz, R.nax);
      const double eps_d = o.eps_abs + o.eps_rel * fmax(R.nq, fmax(R.npx, R.naty));
      int newstate = QP_RUNNING;
      {
        // OSQP is_primal_infeasible: ||dy|| > eps, u'dy+ + l'dy- < -eps ||dy||, ||A'dy|| < eps ||dy||.
        // All warp collectives are executed unconditionally (groups of one warp diverge here).
        if (!active || !run) {
          dy_norm = 0.0; dy_lhs = 0.0;
#pragma unroll
          for (int r = 0; r < QP_ROWS; r++) v[r] = 0.0;
        }
        const double nd = qp_joint_max<JW>(dy_norm, Q.xch);
        const double lhs = qp_joint_sum<JW>(dy_lhs, Q.xch);
        double atd[6];
        double n18 = sp_shfl_down(v[18], 1, LPA), n19 = sp_shfl_down(v[19], 1, LPA), n20 = sp_shfl_down(v[20], 1, LPA);
        if (last) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
        apply_AT(v, n18, n19, n20, t, tp, tn, first, atd);
        double na = 0.0;
#pragma unroll
        for (int j = 0; j < 6; j++) na = fmax(na, fabs(cD[j] * atd[j]));
        if (!active || !run) na = 0.0;
        na = qp_joint_max<JW>(na, Q.xch);
        if (R.pri < eps_p && R.dua < eps_d) newstate = QP_ST_SOLVED;
        else if (!(R.pri < eps_p) && nd > o.eps_pinf && lhs < -o.eps_pinf * nd && na < o.eps_pinf * nd)
          newstate = QP_ST_INFEASIBLE;
      }
      if (run) state = newstate;
      // adaptive rho (OSQP: every adaptive_rho_interval iterations, same residuals)
      if (o.adapt_every > 0 && (it % o.adapt_every == 0)) {
        const bool still = state == QP_RUNNING;
        double pr = R.pri / (fmax(R.nz, R.nax) + 1e-10);
        double dr = R.dua / (fmax(R.nq, fmax(R.npx, R.naty)) + 1e-10);
        double est = rhobar * sqrt(pr / (dr + 1e-10));
        est = fmin(fmax(est, 1e-6), 1e6);
        const bool upd = still && (est > rhobar * o.adapt_tol || est < rhobar / o.adapt_tol);
        if (sp_any(upd)) {
          if (upd) {
            const double ratio = est / rhobar;
#pragma unroll
            for (int r = 0; r < QP_ROWS; r++) {
              const double w = sm[(QP_SM_W + r) * STR + lane], l = sm[(QP_SM_L + r) * STR + lane], u = sm[(QP_SM_U + r) * STR + lane];
              const double z = fmin(fmax(w, l), u);
              sm[(QP_SM_W + r) * STR + lane] = z + (w - z) / ratio;  // keep (z, y): w' = z + y / rho'
              sm[(QP_SM_RHO + r) * STR + lane] *= ratio;
            }
            rhobar = est;
          }
          sp_syncwarp();
          int b2 = qp_factorize<LPA, STR>(sm, lane, QP_SM_RHO, sig, t, tp, tn, first, last, active, seg, kmaxw, 0u, eqmask, 0.0, F);
          b2 = qp_joint_or<JW>(b2, Q.xch);
          if (b2 && state == QP_RUNNING) state = QP_ST_INFEASIBLE;
        }
      }
    }
  }
  Q.rhobar = rhobar;
}

// OSQP at max_iter: "solved inaccurate" if the 10x looser tolerances hold (joint norms when JW = 2*LPA)
SP_DEV int qp_maxiter_state(const SpOptionsDev &o, const QpResid &R) {
  const double ea = 10.0 * o.eps_abs, er = 10.0 * o.eps_rel;
  const bool okp = R.pri < ea + er * fmax(R.nz, R.nax);
  const bool okd = R.dua < ea + er * fmax(R.nq, fmax(R.npx, R.naty));
  const bool ok0 = R.pri < o.eps_abs + o.eps_rel * fmax(R.nz, R.nax) && R.dua < o.eps_abs + o.eps_rel * fmax(R.nq, fmax(R.npx, R.naty));
  return ok0 ? QP_ST_SOLVED : ((okp && okd) ? QP_ST_INACCURATE : QP_ST_MAXITER);
}

// Final status at max_iter, polish and outputs.  Expects the iterate in (x, W slots), the current per-row
// rho in the RHO slots and Q.rhobar.
template <int LPA, int STR, int JW>
SP_DEV void qp_finish(const QpArgs &a, double *sm, int lane, QpLane &Q, double x[6], int state, int iters) {
  QP_UNPACK_LANE(Q);
  const SpOptionsDev &o = a.opt;
  const double rhobar = Q.rhobar;
  if (JW != LPA) {
    QpResid R = qp_residuals<LPA, STR, JW>(sm, lane, x, q, cD, c / rhobar, eqmask, t, tp, tn, first, last, active, Q.xch);
    if (state == QP_RUNNING) state = qp_maxiter_state(o, R);
  }
  // per-axis residuals of the ADMM iterate: the yardstick of the polish acceptance below
  QpResid last_res = qp_residuals<LPA, STR, LPA>(sm, lane, x, q, cD, c / rhobar, eqmask, t, tp, tn, first, last, active);
  if (JW == LPA && state == QP_RUNNING) state = qp_maxiter_state(o, last_res);

  // ---------------- polish: exact optimum of the identified active set ----------------
  // Round 0 is OSQP's polish (polish.c): active set guessed from (z, y), equality-constrained KKT
  // solve regularised by delta, iterative refinement -- here in reduced form, S' = P + sigma' +
  // A' rho' A restricted to the active rows, with the same block-tridiagonal factorisation.  Further
  // rounds correct the active set (violated rows are added, rows with a wrong-signed multiplier are
  // dropped); a round that changes nothing proves the KKT conditions, i.e. optimality ("verified").
  int polished = 0;
  const bool solved = (state == QP_ST_SOLVED || state == QP_ST_INACCURATE);
  if (o.polish && sp_any(solved)) {
    unsigned lowm = 0, uppm = 0;
#pragma unroll
    for (int r = 0; r < QP_ROWS; r++) {
      const double w = sm[(QP_SM_W + r) * STR + lane], l = sm[(QP_SM_L + r) * STR + lane], u = sm[(QP_SM_U + r) * STR + lane];
      const double rho = sm[(QP_SM_RHO + r) * STR + lane];
      const double z = fmin(fmax(w, l), u), y = rho * (w - z);
      const double eqf = ((eqmask >> r) & 1u) ? 1e3 : 1.0;  // rho_r = rhobar eqfac E_r^2 / c
      const double kap = eqf * rhobar / rho;                // c / E_r^2
      bool lowa = (z - l) < -y * kap, uppa = !lowa && ((u - z) < y * kap);
      if ((eqmask >> r) & 1u) { if (!lowa && !uppa) lowa = true; }
      if (lowa) lowm |= 1u << r;
      if (uppa) uppm |= 1u << r;
    }
    // polish penalty rho'_r = E_r^2 / (c delta) = rho_r / (rhobar eqfac delta) on active rows, 0 elsewhere
    const double pol_scale = 1.0 / (rhobar * o.polish_delta);
    // The primal regularisation is decoupled from delta and kept tiny (1e-12 in the scaled space):
    // with OSQP's delta on both blocks the refinement is a proximal iteration that stalls along the
    // weakly curved directions of P (eigenvalues ~1e-9 after scaling on these problems).
    double sigp[6];
#pragma unroll
    for (int j = 0; j < 6; j++) sigp[j] = sig[j] * (1e-12 / o.sigma);
    double xp[6];
    int verified = 0, badp = 0, last_changed = 0;
    double prip = 0.0, duap = 0.0;
    const int rounds = o.polish_rounds > 0 ? o.polish_rounds : 1;
    for (int round = 0; round < rounds; round++) {
      const unsigned actm = lowm | uppm;
      sp_syncwarp();
      QpFactor Fp;
      badp = qp_factorize<LPA, STR>(sm, lane, QP_SM_RHO, sigp, t, tp, tn, first, last, active, seg, kmaxw, actm, eqmask, pol_scale, Fp);
      badp = sp_group_or(badp, LPA);
#pragma unroll
      for (int j = 0; j < 6; j++) xp[j] = 0.0;
      // y_p lives in the W slots from here on (w itself is no longer needed)
#pragma unroll
      for (int r = 0; r < QP_ROWS; r++) sm[(QP_SM_W + r) * STR + lane] = 0.0;
      for (int itp = 0; itp <= o.polish_refine; itp++) {
        double Axp[QP_ROWS], rr[QP_ROWS];
        {
          double p3 = sp_shfl_up(xp[3], 1, LPA), p4 = sp_shfl_up(xp[4], 1, LPA), p5 = sp_shfl_up(xp[5], 1, LPA);
          apply_A(xp, p3, p4, p5, t, tp, first, Axp);
        }
#pragma unroll
        for (int r = 0; r < QP_ROWS; r++) {
          const bool act = (actm >> r) & 1u;
          const double yp = sm[(QP_SM_W + r) * STR + lane];
          const double rp = act ? sm[(QP_SM_RHO + r) * STR + lane] * pol_scale * (((eqmask >> r) & 1u) ? 1e-3 : 1.0) : 0.0;
          const double bnd = ((lowm >> r) & 1u) ? sm[(QP_SM_L + r) * STR + lane] : sm[(QP_SM_U + r) * STR + lane];
          const double r2 = act ? bnd - Axp[r] : 0.0;
          Axp[r] = r2;             // keep r2
          rr[r] = rp * r2 - yp;    // rho' r2 - y_p
        }
        double g[6], px[6], dx[6];
        {
          double n18 = sp_shfl_down(rr[18], 1, LPA), n19 = sp_shfl_down(rr[19], 1, LPA), n20 = sp_shfl_down(rr[20], 1, LPA);
          if (last) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
          apply_AT(rr, n18, n19, n20, t, tp, tn, first, g);  // A'(rho' r2) - A' y_p
        }
        apply_P<STR>(sm, lane, xp, px);
#pragma unroll
        for (int j = 0; j < 6; j++) g[j] += -q[j] - px[j];
        qp_solve<LPA>(Fp, g, dx, seg, last, kmaxw);
        {
          double p3 = sp_shfl_up(dx[3], 1, LPA), p4 = sp_shfl_up(dx[4], 1, LPA), p5 = sp_shfl_up(dx[5], 1, LPA);
          apply_A(dx, p3, p4, p5, t, tp, first, rr);  // rr now holds A dx
        }
#pragma unroll
        for (int j = 0; j < 6; j++) xp[j] += dx[j];
#pragma unroll
        for (int r = 0; r < QP_ROWS; r++) {
          const bool act = (actm >> r) & 1u;
          const double rp = sm[(QP_SM_RHO + r) * STR + lane] * pol_scale * (((eqmask >> r) & 1u) ? 1e-3 : 1.0);
          if (act) sm[(QP_SM_W + r) * STR + lane] += rp * (rr[r] - Axp[r]);
        }
      }
      // KKT check of the polished point in the scaled space + active-set correction
      double Axp[QP_ROWS], yp[QP_ROWS];
      {
        double p3 = sp_shfl_up(xp[3], 1, LPA), p4 = sp_shfl_up(xp[4], 1, LPA), p5 = sp_shfl_up(xp[5], 1, LPA);
        apply_A(xp, p3, p4, p5, t, tp, first, Axp);
      }
      double nax = 0.0, ny = 0.0;
      prip = 0.0;
#pragma unroll
      for (int r = 0; r < QP_ROWS; r++) {
        yp[r] = sm[(QP_SM_W + r) * STR + lane];
        const double l = sm[(QP_SM_L + r) * STR + lane], u = sm[(QP_SM_U + r) * STR + lane];
        const double Er = sqrt(sm[(QP_SM_RHO + r) * STR + lane] * (c / rhobar) * (((eqmask >> r) & 1u) ? 1e-3 : 1.0));
        prip = fmax(prip, Er * fmax(fmax(l - Axp[r], Axp[r] - u), 0.0));
        nax = fmax(nax, Er * fabs(Axp[r]));
        ny = fmax(ny, fabs(c * yp[r] / Er));
      }
      if (!active) { prip = 0.0; nax = 0.0; ny = 0.0; }
      prip = sp_group_max(prip, LPA);
      nax = sp_group_max(nax, LPA);
      ny = sp_group_max(ny, LPA);
      const double tol_p = 1e-9 * (1.0 + nax), tol_d = 1e-9 * (1.0 + ny);
      int changed = 0;
      if (active && !verified) {
#pragma unroll
        for (int r = 0; r < QP_ROWS; r++) {
          const double l = sm[(QP_SM_L + r) * STR + lane], u = sm[(QP_SM_U + r) * STR + lane];
          const double Er = sqrt(sm[(QP_SM_RHO + r) * STR + lane] * (c / rhobar) * (((eqmask >> r) & 1u) ? 1e-3 : 1.0));
          const unsigned bit = 1u << r;
          if (!(actm & bit)) {
            if (Er * (l - Axp[r]) > tol_p) { lowm |= bit; changed = 1; }
            else if (Er * (Axp[r] - u) > tol_p) { uppm |= bit; changed = 1; }
          } else if (!(eqmask & bit)) {
            const double ys = c * yp[r] / Er;
            if ((lowm & bit) && ys > tol_d) { lowm &= ~bit; changed = 1; }
            else if ((uppm & bit) && ys < -tol_d) { uppm &= ~bit; changed = 1; }
          }
        }
      }
      changed = sp_group_or(changed, LPA);
      double aty[6], px[6];
      {
        double n18 = sp_shfl_down(yp[18], 1, LPA), n19 = sp_shfl_down(yp[19], 1, LPA), n20 = sp_shfl_down(yp[20], 1, LPA);
        if (last) { n18 = 0.0; n19 = 0.0; n20 = 0.0; }
        apply_AT(yp, n18, n19, n20, t, tp, tn, first, aty);
      }
      apply_P<STR>(sm, lane, xp, px);
      duap = 0.0;
      double dscale = 0.0;
#pragma unroll
      for (int j = 0; j < 6; j++) {
        duap = fmax(duap, cD[j] * fabs(px[j] + q[j] + aty[j]));
        dscale = fmax(dscale, cD[j] * fmax(fabs(px[j]), fmax(fabs(q[j]), fabs(aty[j]))));
      }
      if (!active) { duap = 0.0; dscale = 0.0; }
      duap = sp_group_max(duap, LPA);
      dscale = sp_group_max(dscale, LPA);
      // stationarity and feasibility must hold too before the KKT conditions count as verified
      if (!(duap <= 1e-8 * (1.0 + dscale)) || !(prip <= 10.0 * tol_p)) changed |= 2;
#if defined(SPECTRAL_CPU_EMU) && defined(SPECTRAL_EMU_DEBUG)
      if (seg == 0 && have) printf("[emu] b=%d axis=%d round=%d nact=%d prip=%.3e duap=%.3e tol_p=%.3e tol_d=%.3e changed=%d verified=%d (admm pri %.3e dua %.3e)\n",
                                   b, axis, round, sp_popc(actm), prip, duap, tol_p, tol_d, changed, verified, last_res.pri, last_res.dua);
#endif
      if (!changed && !badp && !verified) verified = 1;
      last_changed = changed;
      if (sp_all(verified || !solved || badp || changed == 2)) break;
    }
    // acceptance (OSQP polish.c): polished residuals must beat the ADMM ones, in the scaled space
    const bool finite = (prip == prip) && (duap == duap);
    const bool better = (prip < last_res.pri && duap < last_res.dua) || (prip < last_res.pri && last_res.dua < 1e-10) ||
                        (duap < last_res.dua && last_res.pri < 1e-10);
    if (solved && !badp && finite && better) {
      polished = verified ? 3 : 1;
#pragma unroll
      for (int j = 0; j < 6; j++) x[j] = xp[j];
    }
    // diagnostics of a polish that proved nothing (flags bits 4.., include/spectral.h): why
    if (solved && !verified)
      polished |= badp ? 16 : ((last_changed & 2) ? 4 : 8);   // bad pivot | stationarity / feasibility not reached | active set still changing
    if (solved && !(polished & 1)) polished |= 32;            // polished point rejected (not better than the ADMM iterate)
  }

  // ---------------- outputs ----------------
  {
    double px[6];
    apply_P<STR>(sm, lane, x, px);
    double ob = 0.0;
#pragma unroll
    for (int j = 0; j < 6; j++) ob += x[j] * (0.5 * px[j] + q[j]);
    if (!active) ob = 0.0;
    ob = sp_group_sum(ob, LPA);
    if (active) {
      double *dst = a.ctrl + (size_t)b * 12 * a.k_max + (size_t)axis * 6 * K + 6 * seg;
#pragma unroll
      for (int j = 0; j < 6; j++) dst[j] = x[j];
    }
    if (have && seg == 0) {
      a.axis_status[2 * b + axis] = state;
      a.axis_iters[2 * b + axis] = iters;
      a.axis_polished[2 * b + axis] = polished;
      a.axis_obj[2 * b + axis] = ob;
    }
  }
}

// One warp = 32/LPA axis problems (k_qp): setup, lane-per-segment ADMM, finish.
template <int LPA, int JW>
SP_DEV void qp_warp_body(const QpArgs &a, int warp_global, int lane, double *sm, double *xch) {
  constexpr int G = 32 / LPA;
  const int cnt = *a.count;
  const int grp = lane / LPA, seg = lane % LPA;
  const int ap = warp_global * G + grp;  // axis-problem slot in this class
  if (warp_global * G >= 2 * cnt) return;
  const bool have = ap < 2 * cnt;
  QpLane Q;
  qp_setup<LPA, 32, JW>(a, ap, have, seg, lane, sm, Q, xch);
  QpFactor F;
  double x[6];
  int state, iters;
  qp_admm_lanes<LPA, 32, JW>(a.opt, sm, lane, Q, F, x, state, iters);
  qp_finish<LPA, 32, JW>(a, sm, lane, Q, x, state, iters);
}
