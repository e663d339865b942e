// spectral_b200/csrc/eval.cuh -- Bezier evaluation of solved trajectories: the reference's sampler arithmetic
// (solve_3d.cc:1351-1390, shared with finalize_body) and the body of spectral_eval_device (caller-chosen times).
#pragma once
#include "common.cuh"

#define SP_EVAL_MIN_T 1e-9   // segments this short (CorridorSplit slivers) are never evaluated
#define SP_EVAL_TIME_TOL 1e-9  // times in [-tol, H + tol] are valid and clamped to [0, H]

SP_DEV void bernstein_powers(double u, double up[6], double vp[6]) {
  up[0] = 1.0; vp[0] = 1.0;
  const double v = 1 - u;
#pragma unroll
  for (int i = 1; i < 6; i++) { up[i] = up[i - 1] * u; vp[i] = vp[i - 1] * v; }
}

// (s, ds, dds, l, dl, ddl) of a segment of duration t with control points cs (s axis) and cl (l axis) at the
// Bernstein powers up[i] = u^i, vp[i] = (1 - u)^i.  k_finalize's samples come from here: any change of the
// operation order changes its samples and costs.
SP_DEV void bezier_state(const double cs[6], const double cl[6], double t, const double up[6], const double vp[6],
                         double o[6]) {
  const double bc0[6] = {1, 5, 10, 10, 5, 1}, bc1[5] = {1, 4, 6, 4, 1}, bc2[4] = {1, 3, 3, 1};
  double x = 0, y = 0, dx = 0, dy = 0, ddx = 0, ddy = 0;
#pragma unroll
  for (int i = 0; i < 6; i++) { const double bb = bc0[i] * up[i] * vp[5 - i]; x += cs[i] * bb; y += cl[i] * bb; }
#pragma unroll
  for (int i = 0; i < 5; i++) {
    const double bb = bc1[i] * up[i] * vp[4 - i];
    dx += 5.0 * (cs[i + 1] - cs[i]) * bb; dy += 5.0 * (cl[i + 1] - cl[i]) * bb;
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const double bb = bc2[i] * up[i] * vp[3 - i];
    ddx += 20.0 * (cs[i + 2] - 2.0 * cs[i + 1] + cs[i]) * bb; ddy += 20.0 * (cl[i + 2] - 2.0 * cl[i + 1] + cl[i]) * bb;
  }
  o[0] = x * t; o[1] = dx; o[2] = ddx / t; o[3] = y * t; o[4] = dy; o[5] = ddy / t;
}

// (ddds, dddl): 60 sum_i Delta^3 c_i B^2_i(u) / t^2 per axis
SP_DEV void bezier_jerk(const double cs[6], const double cl[6], double t, const double up[6], const double vp[6], double o[2]) {
  const double bc3[3] = {1, 2, 1};
  double jx = 0, jy = 0;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const double bb = bc3[i] * up[i] * vp[2 - i];
    jx += 60.0 * ((cs[i + 3] - cs[i]) - 3.0 * (cs[i + 2] - cs[i + 1])) * bb;
    jy += 60.0 * ((cl[i + 3] - cl[i]) - 3.0 * (cl[i + 2] - cl[i + 1])) * bb;
  }
  o[0] = jx / (t * t); o[1] = jy / (t * t);
}

struct EvalArgs {
  int B, T, k_max;
  int times_stride;  // 0: times[T] for every scenario; 1: times[B][T]
  const int *K, *status;
  const SpectralCube *segs;
  const double *ctrl, *times;
};

// Point j of scenario b: state[6] and jerk[2] (NaN rows for an invalid scenario or time); returns the horizon H
// (NaN for an invalid scenario).  Time model (include/spectral.h, spectral_eval_device): segment k spans
// [T_k, T_k + t_k], T_0 = 0, the durations summed in array order; a time at a joint belongs to the segment that
// ends there; segments with t_k <= SP_EVAL_MIN_T are skipped.
SP_DEV double eval_point(const EvalArgs &a, int b, int j, double state[6], double jerk[2]) {
  const double qnan = NAN;
#pragma unroll
  for (int i = 0; i < 6; i++) state[i] = qnan;
  jerk[0] = qnan; jerk[1] = qnan;
  const int st = a.status[b], K = a.K[b];
  if (!(st == SPECTRAL_SOLVED || st == SPECTRAL_SOLVED_INACCURATE) || K < 1 || K > a.k_max) return qnan;
  const SpectralCube *segs = a.segs + (size_t)b * a.k_max;
  const double *ctrl = a.ctrl + (size_t)b * 12 * a.k_max;
  const double tau = a.times[a.times_stride ? (size_t)b * a.T + j : (size_t)j];
  // one pass over the durations: H, the last evaluable segment, and the first evaluable one whose end is >= tau
  const double tq = tau < 0.0 ? 0.0 : tau;
  int sel = -1, last = -1;
  double T0 = 0.0, Tsel = 0.0, Tlast = 0.0;
  for (int k = 0; k < K; k++) {
    const double t = segs[k].t, T1 = T0 + t;
    if (t > SP_EVAL_MIN_T) {
      last = k; Tlast = T0;
      if (sel < 0 && tq <= T1) { sel = k; Tsel = T0; }
    }
    T0 = T1;
  }
  const double H = T0;
  if (!(tau >= -SP_EVAL_TIME_TOL && tau <= H + SP_EVAL_TIME_TOL)) return H;  // NaN times fail this test too
  if (last < 0) return H;  // every segment is a sliver: nothing to evaluate
  // tau in (H, H + tol] is evaluated at H, on the last evaluable segment (every later duration is a sliver); so is a tau
  // past the last evaluable segment's end (slivers at the end), where u clamps to 1
  double tc = tq;
  if (sel < 0 || tau > H) { sel = last; Tsel = Tlast; tc = tq > H ? H : tq; }
  const double t = segs[sel].t;
  double u = (tc - Tsel) / t;
  u = u < 0.0 ? 0.0 : (u > 1.0 ? 1.0 : u);
  double cs[6], cl[6];
#pragma unroll
  for (int i = 0; i < 6; i++) { cs[i] = ctrl[6 * sel + i]; cl[i] = ctrl[6 * K + 6 * sel + i]; }
  double up[6], vp[6];
  bernstein_powers(u, up, vp);
  bezier_state(cs, cl, t, up, vp, state);
  bezier_jerk(cs, cl, t, up, vp, jerk);
  return H;
}
