// tests/warp_emu/emu_main.cpp -- TEST INFRASTRUCTURE: runs the device "bodies" of
// spectral_b200/csrc/{corridor,qp,finalize,tables}.cuh on the host, one warp = 32 pthreads in
// lock step (see warp_emu.h).  Built by tests/warp_emu/Makefile into libwarp_emu.so and used by
// tests/test_kernel_logic_emu.py to compare the kernels' logic with the CPU oracle where no GPU
// exists.  Not part of the product.
#define SPECTRAL_CPU_EMU 1
#include "../../spectral_b200/csrc/common.cuh"
#include "../../spectral_b200/csrc/bounds.cuh"
#include "../../spectral_b200/csrc/corridor.cuh"
#include "../../spectral_b200/csrc/qp.cuh"
#include "../../spectral_b200/csrc/qp_dense.cuh"
#include "../../spectral_b200/csrc/qp_anchor.cuh"
#include "../../spectral_b200/csrc/tables.cuh"
#include "../../spectral_b200/csrc/finalize.cuh"

#include <cstdlib>
#include <functional>
#include <thread>
#include <vector>

thread_local EmuWarp *emu_warp = nullptr;
thread_local int emu_lane = 0;
thread_local pthread_barrier_t *emu_cta = nullptr;
thread_local int emu_warp_id = 0;

static void run_warps(int nwarps, const std::function<void(int, int, pthread_barrier_t *)> &fn) {
  std::vector<EmuWarp> warps(nwarps);
  pthread_barrier_t cta;
  pthread_barrier_init(&cta, nullptr, 32 * nwarps);
  for (auto &w : warps) pthread_barrier_init(&w.bar, nullptr, 32);
  std::vector<std::thread> th;
  for (int w = 0; w < nwarps; w++)
    for (int l = 0; l < 32; l++)
      th.emplace_back([&, w, l]() {
        emu_warp = &warps[w];
        emu_lane = l;
        emu_cta = &cta;
        emu_warp_id = w;
        fn(w, l, &cta);
      });
  for (auto &t : th) t.join();
  for (auto &w : warps) pthread_barrier_destroy(&w.bar);
  pthread_barrier_destroy(&cta);
}

extern "C" int emu_solve_batch(int variant, int B, int N, int R, double delta, const double *s_bounds,
                               const double *l_bounds, const double *ds_bounds, const double *dl_bounds,
                               const double *s_ref, const double *l_ref, const double *init,
                               const double *scalars, const double *weights, int wstride, int k_max,
                               const SpectralOptions *opt, int *K, SpectralCube *segs, double *ctrl,
                               double *obj, double *a_cost, int *status, int *iters, int *flags, int *npts,
                               double *samples, int samples_cap, double *lu) {
  const bool force_lanes = getenv("SPECTRAL_EMU_LANES") != nullptr;  // run the lane-per-segment body of k_qp<32, 2> for every class
  const bool fullrow = getenv("SPECTRAL_EMU_FULLROW") != nullptr;     // K <= 10: the full-row loop, the anchor layout's reference
  std::vector<int> cstatus(B, 0);
  // ---- corridor kernel: one CTA per scenario, R warps
  CorridorArgs ca{B, N, R, variant, k_max, delta, s_bounds, l_bounds, s_ref, l_ref, segs, K, cstatus.data()};
  CorridorSmem L = corridor_smem_layout(N, R);
  for (int b = 0; b < B; b++) {
    std::vector<unsigned char> smem(L.total + 64);
    unsigned char *base = smem.data();
    base += (16 - ((uintptr_t)base & 15)) & 15;
    run_warps(R, [&](int w, int l, pthread_barrier_t *cta) {
      // every thread must reach the CTA barrier the same number of times: the body returns early
      // only after its last sync_cta(), as on the device
      corridor_cta_body(ca, b, w, l, base, [cta]() { pthread_barrier_wait(cta); });
    });
  }
  // ---- tables
  const int W = wstride ? B : 1;
  std::vector<double> mqm((size_t)W * 2 * 84);
  for (int w = 0; w < W; w++)
    for (int ax = 0; ax < 2; ax++) mqm_body(weights, mqm.data(), w, ax);
  // ---- classification
  std::vector<int> list[SP_NUM_CLASSES];
  for (int b = 0; b < B; b++)
    if (cstatus[b] == 0) list[lane_class(K[b])].push_back(b);
  // ---- QP kernel per lane class
  std::vector<int> axis_status(2 * B, QP_ST_MAXITER), axis_iters(2 * B, 0), axis_pol(2 * B, 0);
  std::vector<double> axis_obj(2 * B, 0.0);
  SpOptionsDev od;
  od.max_iter = opt->max_iter; od.scaling = opt->scaling; od.check_every = opt->check_termination;
  od.adapt_every = opt->adaptive_rho_interval; od.polish = opt->polish; od.polish_refine = opt->polish_refine_iter;
  od.eps_abs = opt->eps_abs; od.eps_rel = opt->eps_rel; od.eps_pinf = opt->eps_prim_inf; od.rho0 = opt->rho;
  od.sigma = opt->sigma; od.alpha = opt->alpha; od.adapt_tol = opt->adaptive_rho_tolerance; od.polish_delta = opt->polish_delta; od.polish_rounds = opt->polish_rounds;
  od.precheck = opt->infeasibility_precheck; od.precheck_margin = opt->precheck_margin;
  for (int cls = 0; cls < SP_NUM_CLASSES; cls++) {
    int cnt = (int)list[cls].size();
    if (!cnt) continue;
    QpArgs qa;
    qa.N = N; qa.k_max = k_max; qa.variant = variant; qa.delta = delta;
    qa.ds_bounds = ds_bounds; qa.dl_bounds = dl_bounds; qa.s_ref = s_ref; qa.l_ref = l_ref; qa.init = init;
    qa.scalars = scalars; qa.weights = weights; qa.wstride = wstride; qa.in_stride = 1; qa.mqm = mqm.data(); qa.segs = segs; qa.K = K;
    qa.list = list[cls].data(); qa.count = &cnt; qa.next = nullptr; qa.opt = od; qa.ctrl = ctrl; qa.axis_status = axis_status.data();
    qa.axis_iters = axis_iters.data(); qa.axis_polished = axis_pol.data(); qa.axis_obj = axis_obj.data(); qa.lu = lu;
    if (cls <= 3 && !force_lanes) {
      // dense kernel: one CTA of 2 TA threads per scenario
      const int total = cls == 0 ? QpdLayout<8>::TOTAL : cls == 1 ? QpdLayout<10>::TOTAL : cls == 2 ? QpdLayout<12>::TOTAL : QpdLayout<16>::TOTAL;
      const int nwarps = cls == 0 ? QpdLayout<8>::NWARPS : cls == 1 ? QpdLayout<10>::NWARPS : cls == 2 ? QpdLayout<12>::NWARPS : QpdLayout<16>::NWARPS;
      for (int slot = 0; slot < cnt; slot++) {
        std::vector<double> sm(total + 2);
        double *base = sm.data();
        if ((uintptr_t)base & 15) base += 1;
        pthread_barrier_t axbar[2];
        for (auto &ab : axbar) pthread_barrier_init(&ab, nullptr, 32 * nwarps / 2);
        run_warps(nwarps, [&](int w, int l, pthread_barrier_t *cta) {
          auto sync = [cta]() { pthread_barrier_wait(cta); };
          auto sync_axis = [&axbar](int axis) { pthread_barrier_wait(&axbar[axis]); };
          if (cls == 0 && !fullrow) qpa_cta_body<8>(qa, slot, 32 * w + l, base, sync, sync_axis);
          else if (cls == 1 && !fullrow) qpa_cta_body<10>(qa, slot, 32 * w + l, base, sync, sync_axis);
          else if (cls == 0) qpd_cta_body<8>(qa, slot, 32 * w + l, base, sync);
          else if (cls == 1) qpd_cta_body<10>(qa, slot, 32 * w + l, base, sync);
          else if (cls == 2) qpd_cta_body<12>(qa, slot, 32 * w + l, base, sync);
          else qpd_cta_body<16>(qa, slot, 32 * w + l, base, sync);
        });
        for (auto &ab : axbar) pthread_barrier_destroy(&ab);
      }
      continue;
    }
    // k_qp<32, 2>: one CTA of two warps per scenario (s-axis warp, l-axis warp, joint reductions)
    for (int slot = 0; slot < cnt; slot++) {
      std::vector<double> sm(2 * QP_SM_DOUBLES_PER_LANE * 32 + QP_XCH_DOUBLES);
      run_warps(2, [&](int w, int l, pthread_barrier_t *) {
        qp_warp_body<32, 64>(qa, 2 * slot + w, l, sm.data() + (size_t)w * QP_SM_DOUBLES_PER_LANE * 32,
                             sm.data() + 2 * QP_SM_DOUBLES_PER_LANE * 32);
      });
    }
  }
  // ---- finalize
  FinalArgs fa;
  fa.B = B; fa.N = N; fa.k_max = k_max; fa.variant = variant; fa.delta = delta; fa.s_ref = s_ref; fa.l_ref = l_ref;
  fa.init = init; fa.weights = weights; fa.wstride = wstride; fa.in_stride = 1; fa.segs = segs; fa.K = K; fa.cstatus = cstatus.data();
  fa.axis_status = axis_status.data(); fa.axis_iters = axis_iters.data(); fa.axis_polished = axis_pol.data();
  fa.axis_obj = axis_obj.data(); fa.ctrl = ctrl; fa.obj = obj; fa.a_cost = a_cost; fa.samples = samples;
  fa.status = status; fa.iters = iters; fa.flags = flags; fa.npts = npts; fa.samples_cap = samples_cap;
  for (int b = 0; b < B; b++) finalize_body(fa, b);
  return 0;
}

extern "C" void emu_default_options(SpectralOptions *o) {
  o->max_iter = 5000; o->eps_abs = 1e-5; o->eps_rel = 1e-5; o->eps_prim_inf = 2.5e-5; o->rho = 0.1; o->sigma = 1e-6;
  o->alpha = 1.6; o->scaling = 4; o->check_termination = 25; o->adaptive_rho_interval = 100;
  o->adaptive_rho_tolerance = 5.0; o->polish = 1; o->polish_delta = 1e-6; o->polish_refine_iter = 4; o->polish_rounds = 8;
  o->infeasibility_precheck = 0; o->precheck_margin = 1e-3; o->shared_kkt = 0;
}

// upstream bound generator (bounds.cuh): one emulated warp per scenario, the table in host memory
extern "C" void emu_bounds(int B, int N, int M, int R_cap, const double *obstacles, const int *n_obs, const double *road, double *s_bounds,
                           double *l_bounds, int *n_lanes) {
  BoundsArgs a{B, N, M, R_cap, obstacles, n_obs, road[0], road[1], road[2], road[3], s_bounds, l_bounds, n_lanes};
  std::vector<SpbTable> T(1);
  std::vector<double> line((size_t)SPB_MAX_CARS * N);
  for (int b = 0; b < B; b++)
    run_warps(1, [&](int, int lane, pthread_barrier_t *) { bounds_warp_body(a, b, lane, &T[0], line.data()); });
}
