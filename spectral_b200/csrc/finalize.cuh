// spectral_b200/csrc/finalize.cuh -- classification by segment count, K5 (Bezier sampling + wrapper
// cost) and K6 (argmin) bodies.
//   sampling: Optimize, solve_3d.cc:1279-1392 and the CHECK at :1407
//   cost:     find_traj, trp_wrapper.cpp:217-286 | cub_wrapper.cpp:210-258
#pragma once
#include "common.cuh"
#include "eval.cuh"
#include "qp.cuh"

struct FinalArgs {
  int B, N, k_max, variant;
  double delta;
  const double *s_ref, *l_ref, *init, *weights;
  int wstride;
  int in_stride;  // 1: one input scenario per lane; 0: every lane reads scenario 0 (weight sweep, spectral_solve_weights)
  const SpectralCube *segs;
  const int *K, *cstatus, *axis_status, *axis_iters, *axis_polished;
  const double *axis_obj, *ctrl;
  // outputs (device)
  double *obj, *a_cost, *samples;
  int *status, *iters, *flags, *npts;
  int samples_cap;
};

// solver class of a scenario by segment count:
//   0: K <= 8  k_qpd<8>   1: K <= 10  k_qpd<10>   2: K <= 12  k_qpd<12>   3: K <= 16  k_qpd<16>   (dense kernels)
//   4: K <= 32  lane-per-segment k_qp<32>
#define SP_NUM_CLASSES 5
SP_DEV int lane_class(int K) { return K <= 8 ? 0 : (K <= 10 ? 1 : (K <= 12 ? 2 : (K <= 16 ? 3 : 4))); }
SP_HD int class_kcap(int cls) { return cls == 0 ? 8 : (cls == 1 ? 10 : (cls == 2 ? 12 : (cls == 3 ? 16 : 32))); }

// one thread per scenario
SP_DEV void finalize_body(const FinalArgs &a, int b) {
  const int cst = a.cstatus[b];
  const int K = a.K[b];
  int status, iters = 0, flags = 0;
  double obj = 0.0;
  if (cst != 0) {
    status = cst;
  } else {
    const int s0 = a.axis_status[2 * b], s1 = a.axis_status[2 * b + 1];
    const bool ok0 = (s0 == QP_ST_SOLVED || s0 == QP_ST_INACCURATE), ok1 = (s1 == QP_ST_SOLVED || s1 == QP_ST_INACCURATE);
    if (ok0 && ok1) status = (s0 == QP_ST_SOLVED && s1 == QP_ST_SOLVED) ? SPECTRAL_SOLVED : SPECTRAL_SOLVED_INACCURATE;
    else status = SPECTRAL_FAIL_SOLVER;  // Optimize() returns false (solve_3d.cc:1253-1260)
    const int i0 = a.axis_iters[2 * b], i1 = a.axis_iters[2 * b + 1];
    iters = i0 > i1 ? i0 : i1;
    const int p0 = a.axis_polished[2 * b], p1 = a.axis_polished[2 * b + 1];
    flags = ((p0 & 1) ? SPECTRAL_FLAG_POLISHED_S : 0) | ((p1 & 1) ? SPECTRAL_FLAG_POLISHED_L : 0) |
            ((p0 & 2) ? SPECTRAL_FLAG_VERIFIED_S : 0) | ((p1 & 2) ? SPECTRAL_FLAG_VERIFIED_L : 0) |
            (((p0 >> 2) & 15) << SPECTRAL_FLAG_DIAG_SHIFT_S) | (((p1 >> 2) & 15) << SPECTRAL_FLAG_DIAG_SHIFT_L);
    obj = a.axis_obj[2 * b] + a.axis_obj[2 * b + 1];
  }
  double cost = SPECTRAL_FAIL_COST;
  int npts = 0;
  if (status == SPECTRAL_SOLVED || status == SPECTRAL_SOLVED_INACCURATE) {
    const int N = a.N;
    const double delta = a.delta;
    const SpectralCube *segs = a.segs + (size_t)b * a.k_max;
    const double *ctrl = a.ctrl + (size_t)b * 12 * a.k_max;
    const double *wv = a.weights + (size_t)(a.wstride ? b : 0) * 10;
    const size_t bi = (size_t)b * a.in_stride;
    const double *sref = a.s_ref + bi * N, *lref = a.l_ref + bi * N;
    const double *ini = a.init + 6 * bi;
    double *smp = a.samples ? a.samples + (size_t)b * a.samples_cap * 6 : nullptr;
    int num_of_points = 1;  // solve_3d.h:114
    for (int k = 0; k < K; k++) num_of_points = (int)((double)num_of_points + segs[k].t / delta);  // int += double (:1281)
    const bool trp = a.variant == SPECTRAL_TRP;
    double s_cost = 0.0, l_cost = 0.0, smax = 0.0, lmax = 0.0;
    double prev_dds = 0.0, prev_ddl = 0.0, l_end = 0.0;
    const int end_idx = (N - 1 < num_of_points) ? N - 1 : num_of_points - 1;
    int var_index = 0;
    bool overflow = false;
    // sample i of the trajectory: (s, ds, dds, l, dl, ddl); costs accumulate on the fly.
    // ddd at i = 0 is (dd[1]-dd[0])/dt (trp_wrapper.cpp:219), i.e. the same value as at i = 1.
    auto emit = [&](double s, double ds, double dds, double l, double dl, double ddl) {
      const int i = var_index;
      if (smp && i < a.samples_cap) {
        double *o = smp + 6 * i;
        o[0] = s; o[1] = ds; o[2] = dds; o[3] = l; o[4] = dl; o[5] = ddl;
      }
      const double xr = i < N ? sref[i] : 0.0, yr = i < N ? lref[i] : 0.0;
      const double ddds = i == 0 ? 0.0 : (dds - prev_dds) / delta;
      const double dddl = i == 0 ? 0.0 : (ddl - prev_ddl) / delta;
      const double jm = i == 1 ? 2.0 : 1.0;  // the i = 0 jerk term equals the i = 1 term
      if (trp) {
        s_cost += wv[4] * (s - xr) * (s - xr) * delta + wv[5] * ds * ds * delta + wv[0] * dds * dds * delta +
                  jm * wv[1] * ddds * ddds * delta;
        l_cost += wv[6] * (l - yr) * (l - yr) * delta + wv[7] * dl * dl * delta + wv[2] * ddl * ddl * delta +
                  jm * wv[3] * dddl * dddl * delta;
      } else {
        s_cost += (s - xr) * (s - xr) * delta + ds * ds * delta + dds * dds * dds * dds * delta +
                  jm * ddds * ddds * ddds * ddds * delta;
        l_cost += (l - yr) * (l - yr) * delta + dl * dl * delta + ddl * ddl * delta + jm * dddl * dddl * delta;
      }
      smax = fmax(smax, fabs(dds));
      lmax = fmax(lmax, fabs(ddl));
      if (i == end_idx) l_end = l;
      prev_dds = dds; prev_ddl = ddl;
      var_index++;
    };
    emit(ini[0], ini[1], ini[2], ini[3], ini[4], ini[5]);  // :1325-1331
    for (int k = 0; k < K && !overflow; k++) {
      double cs[6], cl[6];
#pragma unroll
      for (int i = 0; i < 6; i++) { cs[i] = ctrl[6 * k + i]; cl[i] = ctrl[6 * K + 6 * k + i]; }
      const double t = segs[k].t;
      const int linter = (int)(t / delta);  // :1351
      for (int l = 1; l <= linter; l++) {
        if (var_index >= num_of_points) { overflow = true; break; }  // x_.at() would throw
        double up[6], vp[6], o[6];
        bernstein_powers((double)l / linter, up, vp);
        bezier_state(cs, cl, t, up, vp, o);
        emit(o[0], o[1], o[2], o[3], o[4], o[5]);
      }
    }
    if (overflow || var_index != num_of_points) {  // CHECK_EQ(var_index, num_of_points_) -> abort (:1407)
      status = SPECTRAL_FAIL_POINTS_CHECK;
    } else {
      npts = num_of_points;
      if (trp) l_cost += wv[9] * (l_end - lref[N - 1]) * (l_end - lref[N - 1]) * delta;  // trp_wrapper.cpp:269
      else { s_cost += smax * smax * smax * smax; l_cost += lmax * lmax; }                 // cub_wrapper.cpp:228,257
      cost = s_cost + l_cost;
    }
  }
  if (a.status) a.status[b] = status;
  if (a.iters) a.iters[b] = iters;
  if (a.flags) a.flags[b] = flags;
  if (a.obj) a.obj[b] = obj;
  if (a.a_cost) a.a_cost[b] = cost;
  if (a.npts) a.npts[b] = npts;
}
