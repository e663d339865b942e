// spectral_b200/csrc/certify.cuh -- the primal feasibility certificate of solved trajectories (spectral_certify_device): how
// far the returned control points x are from l <= A x <= u of the QP they were solved for, per axis and row family, in the
// QP's own row units.  A and (l, u) come from apply_A and qp_rows (qp.cuh), the solver's own assembly.
// One warp per scenario, lane k = segment k (k_max <= 32), as in the solver's lane-per-segment layout.
#pragma once
#include "common.cuh"
#include "qp.cuh"

#define SP_CERT_FAMILIES 4  // position, velocity, acceleration, jerk

struct CertArgs {
  int B, N, k_max, variant;
  int in_stride;  // 1: one input scenario per output scenario; 0: every scenario reads input scenario 0 (weight sweep)
  const double *ds_bounds, *dl_bounds, *init, *scalars;
  const int *K, *status;
  const SpectralCube *segs;
  const double *ctrl, *a_cost;
  double tol[SP_CERT_FAMILIES];
  double *viol;  // [B][2][SP_CERT_FAMILIES] or NULL
  double *cost;  // [B] or NULL
};

// family of lane row r (qp_rows): rows 0..5 and 18 position, 6..10 and 19 velocity, 11..14 and 20 acceleration, 15..17 jerk
SP_DEV int cert_family(int r) { return r < 6 ? 0 : (r < 11 ? 1 : (r < 15 ? 2 : (r < 18 ? 3 : r - 18))); }

// max that keeps a NaN of either argument (fmax drops it, and a NaN row would then certify)
SP_DEV double cert_max(double a, double b) { return (a > b || a != a) ? a : b; }

// scenario b on the calling warp; every lane must call it with the same b
SP_DEV void certify_warp(const CertArgs &a, int b, int lane) {
  const double qnan = NAN;
  const int st = a.status[b], K = a.K[b];
  const bool solved = (st == SPECTRAL_SOLVED || st == SPECTRAL_SOLVED_INACCURATE) && K >= 1 && K <= a.k_max;
  const bool active = solved && lane < K;
  SpectralCube cube{};
  bool bad = false;
  if (active) {
    cube = a.segs[(size_t)b * a.k_max + lane];
    bad = !(cube.beg_t >= 0 && cube.beg_t <= cube.end_t && cube.end_t <= a.N - 1);  // the s rows read ds_bounds over it
  }
  const bool ok = solved && !sp_any(bad);  // uniform over the warp
  double v[2][SP_CERT_FAMILIES];
#pragma unroll
  for (int ax = 0; ax < 2; ax++)
#pragma unroll
    for (int f = 0; f < SP_CERT_FAMILIES; f++) v[ax][f] = qnan;
  if (ok) {
    const bool first = lane == 0;
    const double t = cube.t;
    double tp = sp_shfl_up(t, 1, 32);
    if (first) tp = 1.0;
    const size_t bi = (size_t)b * a.in_stride;
    const double *ctrl = a.ctrl + (size_t)b * 12 * a.k_max;
#pragma unroll
    for (int ax = 0; ax < 2; ax++) {
      double c[6];
#pragma unroll
      for (int i = 0; i < 6; i++) {
        c[i] = active ? ctrl[6 * K * ax + 6 * lane + i] : 0.0;
        if (!isfinite(c[i])) c[i] = qnan;  // an infinite control point makes its rows NaN, not +-inf
      }
      const double p3 = sp_shfl_up(c[3], 1, 32), p4 = sp_shfl_up(c[4], 1, 32), p5 = sp_shfl_up(c[5], 1, 32);
      double f[SP_CERT_FAMILIES] = {0.0, 0.0, 0.0, 0.0};
      if (active) {
        double z[QP_ROWS], lo[QP_ROWS], hi[QP_ROWS];
        apply_A(c, p3, p4, p5, t, tp, first, z);
        qp_rows(a, ax, true, first, cube, t, bi, a.N, a.scalars + 10 * bi, a.init + 6 * bi + 3 * ax, lo, hi);
#pragma unroll
        for (int r = 0; r < QP_ROWS; r++) {
          // max(l - Ax, Ax - u, 0); the last step also turns a -0.0 into +0.0 for the bit-pattern maximum below
          const double e = cert_max(cert_max(lo[r] - z[r], z[r] - hi[r]), 0.0);
          f[cert_family(r)] = cert_max(f[cert_family(r)], e);
        }
      }
#pragma unroll
      for (int k = 0; k < SP_CERT_FAMILIES; k++) v[ax][k] = sp_warp_max_nonneg(f[k] != f[k] ? qnan : f[k]);  // +NaN wins
    }
  }
  if (lane == 0) {
    bool cert = true;
#pragma unroll
    for (int ax = 0; ax < 2; ax++)
#pragma unroll
      for (int k = 0; k < SP_CERT_FAMILIES; k++) {
        cert = cert && v[ax][k] <= a.tol[k];  // false for NaN
        if (a.viol) a.viol[(size_t)b * 2 * SP_CERT_FAMILIES + ax * SP_CERT_FAMILIES + k] = v[ax][k];
      }
    if (a.cost) a.cost[b] = cert ? a.a_cost[b] : SPECTRAL_FAIL_COST;
  }
}
