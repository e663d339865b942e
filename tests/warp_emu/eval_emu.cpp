// tests/warp_emu/eval_emu.cpp -- TEST INFRASTRUCTURE: the point body of spectral_eval_device
// (spectral_b200/csrc/eval.cuh) compiled for the host, for tests/test_eval_emu.py, which builds it on its own
// (g++, no FMA contraction, as libwarp_emu.so).  The body uses no warp primitives; it runs one point per call.
// Not part of the product.
#define SPECTRAL_CPU_EMU 1
#include "../../spectral_b200/csrc/common.cuh"
#include "../../spectral_b200/csrc/eval.cuh"

thread_local EmuWarp *emu_warp = nullptr;
thread_local int emu_lane = 0;
thread_local pthread_barrier_t *emu_cta = nullptr;
thread_local int emu_warp_id = 0;

// every (b, j) through eval_point, outputs laid out as k_eval writes them
extern "C" void emu_eval(int B, int k_max, const int *K, const int *status, const SpectralCube *segs, const double *ctrl, int T,
                         const double *times, int times_stride, double *states, double *jerk, double *horizon) {
  EvalArgs a{B, T, k_max, times_stride, K, status, segs, ctrl, times};
  for (int b = 0; b < B; b++)
    for (int j = 0; j < T; j++) {
      double st[6], jk[2];
      const size_t p = (size_t)b * T + j;
      const double H = eval_point(a, b, j, st, jk);
      for (int i = 0; i < 6; i++) states[6 * p + i] = st[i];
      if (jerk) { jerk[2 * p] = jk[0]; jerk[2 * p + 1] = jk[1]; }
      if (horizon && j == 0) horizon[b] = H;
    }
}
