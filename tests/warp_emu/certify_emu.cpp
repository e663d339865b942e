// tests/warp_emu/certify_emu.cpp -- TEST INFRASTRUCTURE: the warp body of spectral_certify_device
// (spectral_b200/csrc/certify.cuh) compiled for the host, for tests/test_certify_emu.py, which builds it on its own
// (g++, no FMA contraction, as libwarp_emu.so).  One emulated warp (32 lock-stepped threads) takes the scenarios in turn.
// Not part of the product.
#define SPECTRAL_CPU_EMU 1
#include "../../spectral_b200/csrc/common.cuh"
#include "../../spectral_b200/csrc/certify.cuh"

#include <thread>
#include <vector>

thread_local EmuWarp *emu_warp = nullptr;
thread_local int emu_lane = 0;
thread_local pthread_barrier_t *emu_cta = nullptr;
thread_local int emu_warp_id = 0;

// every scenario through certify_warp, outputs laid out as k_certify writes them
extern "C" void emu_certify(int variant, int B, int N, int k_max, const double *ds_bounds, const double *dl_bounds,
                            const double *init, const double *scalars, int inputs_stride, const int *K, const int *status,
                            const SpectralCube *segs, const double *ctrl, const double *a_cost, const double *tol, double *viol,
                            double *cost) {
  CertArgs a{B, N, k_max, variant, inputs_stride, ds_bounds, dl_bounds, init, scalars, K, status, segs, ctrl, a_cost,
             {tol[0], tol[1], tol[2], tol[3]}, viol, cost};
  EmuWarp w;
  pthread_barrier_init(&w.bar, nullptr, 32);
  std::vector<std::thread> th;
  for (int l = 0; l < 32; l++)
    th.emplace_back([&, l]() {
      emu_warp = &w;
      emu_lane = l;
      for (int b = 0; b < B; b++) certify_warp(a, b, l);
    });
  for (auto &t : th) t.join();
  pthread_barrier_destroy(&w.bar);
}
