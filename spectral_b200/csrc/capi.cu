// spectral_b200/csrc/capi.cu -- libspectral.so: the C-ABI of include/spectral.h and the __global__
// wrappers of the QP-side kernels (tables, classify, qp<LPA>, finalize, argmin, fp64 peak probe).
// The corridor kernel lives in corridor.cu (built with --fmad=false, see corridor.cuh).
// There is no CPU path in this library: every entry point needs a CUDA device and reports
// SPECTRAL_ERR_CUDA otherwise.
#include <cuda_runtime.h>
#include <cub/cub.cuh>
#include <dlfcn.h>
#include <nccl.h>  // types only: the library is dlopen()ed at run time (spectral_comm_*), libspectral.so has no link dependency on it

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "common.cuh"
#include "bounds.cuh"
#include "corridor.cuh"
#include "downstream.cuh"
#include "eval.cuh"
#include "finalize.cuh"
#include "qp.cuh"
#include "qp_dense.cuh"
#include "qp_anchor.cuh"
#include "qp_shared.cuh"
#include "qp_shared4.cuh"
#include "tables.cuh"
#include "topk.cuh"

static_assert(SPECTRAL_NUM_CLASSES == SP_NUM_CLASSES && SPECTRAL_NUM_WORK >= 6 + SP_NUM_CLASSES, "include/spectral.h");

extern "C" void spectral_launch_corridor(const CorridorArgs &a, cudaStream_t st);  // corridor.cu
extern "C" int spectral_corridor_prepare(int N, int R, int *configured);                           // corridor.cu
extern "C" int spectral_launch_bounds(const BoundsArgs &a, int sm_count, cudaStream_t st);         // corridor.cu (same --fmad=false unit)

// ------------------------------------------------------------------ kernels
__global__ void k_tables(const double *weights, double *mqm, int W) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 2 * W) mqm_body(weights, mqm, i >> 1, i & 1);
}

__global__ void k_classify(const int *cstatus, const int *K, int B, int *lists, int *counts) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B || cstatus[b] != 0) return;
  const int cls = lane_class(K[b]);
  const int slot = atomicAdd(&counts[cls], 1);
  lists[(size_t)cls * B + slot] = b;
}

// classification that keeps scenario order (one CTA, used for small batches so runs are reproducible
// lane-for-lane; the atomic version above is used for large ones)
__global__ void k_classify_ordered(const int *cstatus, const int *K, int B, int *lists, int *counts) {
  __shared__ int base[SP_NUM_CLASSES];
  __shared__ int wsum[SP_NUM_CLASSES][32];
  if (threadIdx.x < SP_NUM_CLASSES) base[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int start = 0; start < B; start += blockDim.x) {
    const int b = start + threadIdx.x;
    int cls = -1;
    if (b < B && cstatus[b] == 0) cls = lane_class(K[b]);
    int pos[SP_NUM_CLASSES];
    for (int c = 0; c < SP_NUM_CLASSES; c++) {
      const unsigned m = __ballot_sync(0xffffffffu, cls == c);
      pos[c] = __popc(m & ((1u << lane) - 1));
      if (lane == 0) wsum[c][warp] = __popc(m);
    }
    __syncthreads();
    if (cls >= 0) {
      int off = base[cls];
      for (int w = 0; w < warp; w++) off += wsum[cls][w];
      lists[(size_t)cls * B + off + pos[cls]] = b;
    }
    __syncthreads();
    if (threadIdx.x < SP_NUM_CLASSES) {
      int tot = 0;
      for (int w = 0; w < nw; w++) tot += wsum[threadIdx.x][w];
      base[threadIdx.x] += tot;
    }
    __syncthreads();
  }
  if (threadIdx.x < SP_NUM_CLASSES) counts[threadIdx.x] = base[threadIdx.x];
}

template <int LPA, int WPB>
__global__ void __launch_bounds__(32 * WPB) k_qp(const QpArgs a) {
  extern __shared__ double qp_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // LPA = 32 (K > 16): the block's two warps are the s-axis and the l-axis problem of ONE scenario, solved jointly (JW = 64)
  static_assert(LPA < 32 || WPB == 2, "a two-warp CTA per scenario");
  // grid-stride over the class' scenarios: the launch holds at most a few CTAs per SM, not one per scenario of the batch
  constexpr int G = 32 / LPA;
  const int nblk = (2 * *a.count + G * WPB - 1) / (G * WPB);
  for (int blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    qp_warp_body<LPA, 2 * LPA>(a, blk * WPB + warp, lane, qp_smem + (size_t)warp * QP_SM_DOUBLES_PER_LANE * 32,
                               qp_smem + (size_t)WPB * QP_SM_DOUBLES_PER_LANE * 32);
    __syncthreads();
  }
}

// dense-operator ADMM kernel (qp_dense.cuh): one CTA (2 TA threads) per scenario of this class
// Persistent like k_qpa: one CTA per SM takes scenarios of the class from the device-side queue (a.next) until the list is
// drained, so a launch never holds more CTAs than the class has work for (was: B CTAs, most of them empty).
template <int KC>
__global__ void __launch_bounds__(2 * QpdLayout<KC>::TA, 1) k_qpd(const QpArgs a) {
  extern __shared__ __align__(16) double qpd_smem[];
  __shared__ int s_slot;
  for (;;) {
    if (threadIdx.x == 0) s_slot = atomicAdd(a.next, 1);
    __syncthreads();
    const int slot = s_slot;
    __syncthreads();
    if (slot >= *a.count) return;
    qpd_cta_body<KC>(a, slot, threadIdx.x, qpd_smem, []() { __syncthreads(); });
  }
}

// anchor-layout dense ADMM kernel (qp_anchor.cuh), KC <= 10.  Persistent: 2 CTAs per SM take scenarios of this class from
// a device-side queue (a.next) until the list is drained -- no empty CTAs, no ragged last wave per launch.
template <int KC>
__global__ void __launch_bounds__(2 * QpdLayout<KC>::TA, 2) k_qpa(const QpArgs a) {
  extern __shared__ __align__(16) double qpd_smem[];
  __shared__ int s_slot;
  for (;;) {
    if (threadIdx.x == 0) s_slot = atomicAdd(a.next, 1);
    __syncthreads();
    const int slot = s_slot;
    __syncthreads();
    if (slot >= *a.count) return;
    qpa_cta_body<KC>(a, slot, threadIdx.x, qpd_smem, []() { __syncthreads(); },
                     [](int axis) {  // named barrier over the TA threads of one axis (ids as immediates: ptxas reserves only three)
                       if (axis == 0) asm volatile("bar.sync 1, %0;" ::"n"(QpdLayout<KC>::TA) : "memory");
                       else asm volatile("bar.sync 2, %0;" ::"n"(QpdLayout<KC>::TA) : "memory");
                     });
  }
}

// the step after the hot path (downstream.cuh)
__global__ void k_ego_states(const double *samples, const int *npts, int cap, const double *s_offset, int off_stride, double *states, int B) {
  const int i = blockIdx.y * blockDim.x + threadIdx.x;
  const int b = blockIdx.x;
  if (b < B && i < cap) ego_state_body(samples, npts, cap, s_offset, off_stride, states, b, i);
}
__global__ void k_frenet_to_cartesian(const double *ref, const double *s_cond, const double *d_cond, double *out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) frenet_to_cartesian_body(ref, s_cond, d_cond, out, (size_t)i);
}

// weight sweep: the corridor stage ran for scenario 0 only; every lane gets its (K, segments, corridor status)
__global__ void k_broadcast_corridor(int *K, SpectralCube *segs, int *cstatus, int k_max, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B || b == 0) return;
  K[b] = K[0]; cstatus[b] = cstatus[0];
  const int n = K[0] < k_max ? K[0] : k_max;
  for (int k = 0; k < n; k++) segs[(size_t)b * k_max + k] = segs[k];
}

// ------------------------------------------------------------------ shared-KKT path (qp_shared.cuh)
// structure key of a scenario of the K <= 8 class: (K, the bit patterns of t_k, the weights when they are per scenario)
// `hint`: st[4 b + 3] of a first prepare pass run with the interval pre-check forced on = "this corridor is provably
// empty".  It is mixed into the key, so that tiles are homogeneous in it: members that converge in a few hundred iterations no
// longer idle in a tile until an infeasible member has burnt its 5000 (the hint decides tile membership only, never a status).
__global__ void k_qps_keys(const int *cstatus, const int *K, const SpectralCube *segs, int k_max, const double *weights, int wstride, int B,
                           unsigned long long *keys, int *ids, int *leader_tile, const int *hint) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  unsigned long long h = ~0ull;
  if (cstatus[b] == 0 && K[b] >= 1 && K[b] <= QPS_KC) {
    h = 0x9E3779B97F4A7C15ull ^ (unsigned long long)K[b];
    auto mix = [&h](unsigned long long w) {
      h ^= w; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 29; h *= 0x94D049BB133111EBull; h ^= h >> 32;
    };
    for (int k = 0; k < K[b]; k++) mix((unsigned long long)__double_as_longlong(segs[(size_t)b * k_max + k].t));
    if (wstride)
      for (int i = 0; i < 10; i++) mix((unsigned long long)__double_as_longlong(weights[(size_t)b * 10 + i]));
    mix(hint[4 * b + 3] ? 0x5bd1e995ull : 0x1b873593ull);
    if (h == ~0ull) h = 0x1234567ull;
  }
  keys[b] = h; ids[b] = b; leader_tile[b] = -1;
}
__global__ void k_qps_heads(const unsigned long long *keys, int B, int *head) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  head[i] = (keys[i] != ~0ull && (i == 0 || keys[i] != keys[i - 1])) ? i : 0;
}
__global__ void k_qps_flags(const unsigned long long *keys, const int *gstart, int B, int *flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  flag[i] = (keys[i] != ~0ull && ((i - gstart[i]) % QPS_TILE) == 0) ? 1 : 0;
}
__global__ void k_qps_emit(const unsigned long long *keys, const int *ids, const int *flag, const int *tidx, int B, int *tile_start,
                           int *tile_count, int *n_tiles, int *leader_tile) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  if (flag[i]) {
    int c = 1;
    while (c < QPS_TILE && i + c < B && keys[i + c] == keys[i]) c++;
    tile_start[tidx[i]] = i; tile_count[tidx[i]] = c;
    leader_tile[ids[i]] = tidx[i];
  }
  if (i == B - 1) *n_tiles = tidx[i] + flag[i];
}
__global__ void __launch_bounds__(64) k_qps_prepare(const QpsArgs A, const int *leader_tile) {
  extern __shared__ double qp_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  qps_prepare_body(A, leader_tile, blockIdx.x * 2 + warp, lane, qp_smem + (size_t)warp * QP_SM_DOUBLES_PER_LANE * 32);
}
// four warps per tile (qp_shared4.cuh): warp = (axis, half), one segment per thread
__global__ void __launch_bounds__(128, 2) k_qps4(const QpsArgs A) {
  extern __shared__ __align__(16) double qps_smem[];
  __shared__ int s_tile;
  for (;;) {
    if (threadIdx.x == 0) s_tile = atomicAdd(A.tile_next, 1);
    __syncthreads();
    const int tile = s_tile;
    __syncthreads();
    if (tile >= *A.n_tiles) return;
    qps4_tile_body(A, tile, blockIdx.x, threadIdx.x, qps_smem, []() { __syncthreads(); },
                   [](int axis) {  // named barrier over the 64 threads of one axis
                     if (axis == 0) asm volatile("bar.sync 1, 64;" ::: "memory");
                     else asm volatile("bar.sync 2, 64;" ::: "memory");
                   });
    __syncthreads();
  }
}
__global__ void __launch_bounds__(64) k_qps_finish(const QpsArgs A) {
  extern __shared__ double qp_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  qps_finish_body(A, blockIdx.x * 2 + warp, lane, qp_smem + (size_t)warp * QP_SM_DOUBLES_PER_LANE * 32);
}

// `work` (SPECTRAL_NUM_WORK doubles) accumulates what the step did, for the roofline accounting of bench.py:
//   [0] ADMM iterations summed over the axis problems     [1] their flops in the DENSE-operator count, 72 K^2 + 208 K - 24 per
//   axis-iteration (dense apply of the 6K x 6K inverse + A, A' products; 424 K - 168 above the dense kernels' capacity)
//   [2] scenarios processed   [3] scenarios solved   [4] sum of K over scenarios with a corridor (corridor kernel output bytes)
//   [5] the same iterations in the VARIABLE-STRUCTURE count of SURVEY.md 8d, 424 K - 168 per axis-iteration (block-tridiagonal
//   solve: the algorithmic minimum when no two scenarios share a KKT matrix)   [6 + c] dense-count flops of solver class c
__global__ void k_finalize(const FinalArgs a, double *work) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  double v[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  double fcls = 0.0;
  int cls = 0;
  if (b < a.B) {
    finalize_body(a, b);
    v[2] = 1.0;
    if (a.cstatus[b] == 0) {
      const double it = (double)a.axis_iters[2 * b] + (double)a.axis_iters[2 * b + 1];
      const double Kd = (double)a.K[b];
      v[0] = it;
      v[1] = it * (a.K[b] <= 16 ? 72.0 * Kd * Kd + 208.0 * Kd - 24.0 : 424.0 * Kd - 168.0);
      v[4] = Kd;
      v[5] = it * (424.0 * Kd - 168.0);
      cls = lane_class(a.K[b]);
      fcls = v[1];
      const int s0 = a.axis_status[2 * b], s1 = a.axis_status[2 * b + 1];
      v[3] = ((s0 == QP_ST_SOLVED || s0 == QP_ST_INACCURATE) && (s1 == QP_ST_SOLVED || s1 == QP_ST_INACCURATE)) ? 1.0 : 0.0;
    }
  }
#pragma unroll
  for (int i = 0; i < 6; i++)
    for (int m = 16; m > 0; m >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], m);
  if ((threadIdx.x & 31) == 0 && v[2] > 0.0) {
#pragma unroll
    for (int i = 0; i < 6; i++) atomicAdd(&work[i], v[i]);
  }
  if (fcls > 0.0) atomicAdd(&work[6 + cls], fcls);
}

// K6: (min cost, lowest index) -- two-stage, last block finishes (ticket)
struct ArgminPair { double cost; long long idx; };
__device__ __forceinline__ ArgminPair argmin_better(ArgminPair a, ArgminPair b) {
  return (b.cost < a.cost || (b.cost == a.cost && b.idx < a.idx)) ? b : a;
}
__global__ void k_argmin(const double *cost, int B, long long offset, ArgminPair *partial, unsigned *ticket,
                         double *out_cost, long long *out_idx) {
  __shared__ ArgminPair sh[32];
  __shared__ bool is_last;
  ArgminPair best{1.0e300, 0x7fffffffffffffffLL};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x)
    best = argmin_better(best, ArgminPair{cost[i], offset + i});
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int m = 16; m > 0; m >>= 1) {
    ArgminPair o{__shfl_xor_sync(0xffffffffu, best.cost, m), __shfl_xor_sync(0xffffffffu, best.idx, m)};
    best = argmin_better(best, o);
  }
  if (lane == 0) sh[warp] = best;
  __syncthreads();
  if (warp == 0) {
    best = lane < nw ? sh[lane] : ArgminPair{1.0e300, 0x7fffffffffffffffLL};
    for (int m = 16; m > 0; m >>= 1) {
      ArgminPair o{__shfl_xor_sync(0xffffffffu, best.cost, m), __shfl_xor_sync(0xffffffffu, best.idx, m)};
      best = argmin_better(best, o);
    }
    if (lane == 0) {
      partial[blockIdx.x] = best;
      __threadfence();
      is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    }
  }
  __syncthreads();
  if (is_last && warp == 0) {
    __threadfence();
    best = ArgminPair{1.0e300, 0x7fffffffffffffffLL};
    for (int i = lane; i < (int)gridDim.x; i += 32) best = argmin_better(best, partial[i]);
    for (int m = 16; m > 0; m >>= 1) {
      ArgminPair o{__shfl_xor_sync(0xffffffffu, best.cost, m), __shfl_xor_sync(0xffffffffu, best.idx, m)};
      best = argmin_better(best, o);
    }
    if (lane == 0) { *out_cost = best.cost; *out_idx = best.idx; *ticket = 0; }
  }
}

// FP64 FMA throughput probe: 8 independent chains per thread
__global__ void k_fp64_peak(double *out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-7;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------ handle
struct DevBuf {
  void *p = nullptr;
  size_t bytes = 0;
};

struct spectral_handle {
  int device = 0, max_batch = 0, n_max = 0, r_max = 0, k_max = 0, sm_count = 148;
  cudaStream_t stream = nullptr;  // used by the host-buffer entry point
  cudaStream_t side[SP_NUM_CLASSES - 1] = {};  // the solver classes run concurrently (fork / join around the QP stage)
  cudaEvent_t ev_fork = nullptr, ev_join[SP_NUM_CLASSES - 1] = {};
  std::string err;
  long long launches = 0;
  bool timing = false;
  static const int kTimingSlots = 64;  // ring of per-call event sets; nothing synchronises until get_timing
  cudaEvent_t ev[kTimingSlots][SPECTRAL_NUM_KERNELS + 1] = {};
  cudaEvent_t ev_cls[kTimingSlots][SP_NUM_CLASSES][2] = {};  // around each solver class' kernel, on that class' stream
  long long timed_calls = 0;
  double *work = nullptr;  // device counters, see k_finalize
  // intermediates
  int *cstatus = nullptr, *lists = nullptr, *counts = nullptr, *axis_status = nullptr, *axis_iters = nullptr,
      *axis_polished = nullptr;
  double *axis_obj = nullptr, *mqm = nullptr;
  ArgminPair *partial = nullptr;
  unsigned *ticket = nullptr;
  // device mirrors for the host-buffer entry point
  double *d_in[9] = {};
  size_t d_in_bytes[9] = {};
  int *d_K = nullptr, *d_status = nullptr, *d_iters = nullptr, *d_flags = nullptr, *d_npts = nullptr;
  SpectralCube *d_segs = nullptr;
  double *d_ctrl = nullptr, *d_obj = nullptr, *d_cost = nullptr, *d_samples = nullptr, *d_lu = nullptr;
  size_t d_samples_bytes = 0, d_lu_bytes = 0;
  bool qp_attr_set = false;
  // shared-KKT path (allocated on first use)
  unsigned long long *qs_keys = nullptr, *qs_keys2 = nullptr;
  int *qs_ids = nullptr, *qs_ids2 = nullptr, *qs_tmp = nullptr /* head, gstart, flag, tidx: 4 x B */, *qs_tile = nullptr /* start, count: 2 x B */,
      *qs_leader = nullptr, *qs_misc = nullptr /* n_tiles, tile_next */, *qs_st = nullptr;
  QpsTileBlk *qs_blk = nullptr;
  double *qs_lu = nullptr, *qs_qv = nullptr, *qs_w = nullptr, *qs_x = nullptr, *qs_fs = nullptr;
  void *qs_cub = nullptr;
  size_t qs_cub_bytes = 0;
  // multi-GPU exchange (spectral_comm_* / spectral_sweep_argmin)
  ncclComm_t comm = nullptr;
  int nranks = 1, rank = 0;
  double *xg_rec = nullptr;        // [1 + nranks] (cost, index) records, 16 bytes each
  unsigned char *xg_pay = nullptr; // winner payload
  // top-k selection (topk.cuh), allocated on first use: select scratch (independent of B), then the sweep_topk exchange
  TopkScratch tk{};
  double *tk_rec = nullptr;             // (2 + nranks) x k_cap 16-byte records: local, merged, gathered
  unsigned char *tk_pay = nullptr;      // [k_cap][kPayBytes] winner payloads (device)
  unsigned char *tk_hostpay = nullptr;  // the same, page-locked host copy
  double *tk_hostrec = nullptr;         // [k_cap] merged records, page-locked host copy
  int tk_cap = 0, tk_cap_ranks = 0;
  int classes_timed = 0;    // solver classes launched per call (k_max dependent)
  int corridor_smem = 0;    // dynamic shared memory the corridor kernel is opted in for on this handle's device
};

static int fail(spectral_handle *h, int code, const std::string &msg) {
  if (h) h->err = msg;
  return code;
}
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(h, SPECTRAL_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));       \
  } while (0)

extern "C" void spectral_default_options(SpectralOptions *o) {
  o->max_iter = 5000; o->eps_abs = 1e-5; o->eps_rel = 1e-5; o->eps_prim_inf = 2.5e-5; o->rho = 0.1; o->sigma = 1e-6;
  o->alpha = 1.6; o->scaling = 4; o->check_termination = 25; o->adaptive_rho_interval = 100;
  o->adaptive_rho_tolerance = 5.0; o->polish = 1; o->polish_delta = 1e-6; o->polish_refine_iter = 4; o->polish_rounds = 8;
  o->infeasibility_precheck = 0; o->precheck_margin = 1e-3; o->shared_kkt = 0;
}

extern "C" const char *spectral_last_error(const spectral_handle_t *h) { return h ? h->err.c_str() : "null handle"; }
extern "C" long long spectral_launch_count(const spectral_handle_t *h) { return h ? h->launches : 0; }

extern "C" int spectral_create(int device, int max_batch, int n_max, int r_max, int k_max, spectral_handle_t **out) {
  if (!out) return SPECTRAL_ERR_INVALID;
  *out = nullptr;
  if (max_batch <= 0 || n_max < 3 || n_max > SP_MAX_KNOTS || r_max < 1 || r_max > SP_MAX_REGIONS || k_max < 1 || k_max > 32)
    return SPECTRAL_ERR_INVALID;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device >= ndev) {
    fprintf(stderr, "libspectral: no CUDA device (this library has no CPU path)\n");
    return SPECTRAL_ERR_CUDA;
  }
  spectral_handle *h = new spectral_handle();
  h->device = device; h->max_batch = max_batch; h->n_max = n_max; h->r_max = r_max; h->k_max = k_max;
  *out = h;
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  h->sm_count = prop.multiProcessorCount;
  CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  for (auto &s : h->side) CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
  for (auto &e : h->ev_join) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  const size_t B = (size_t)max_batch;
  CK(cudaMalloc(&h->cstatus, B * 4));
  CK(cudaMalloc(&h->lists, SP_NUM_CLASSES * B * 4));
  CK(cudaMalloc(&h->counts, 4 * 2 * SP_NUM_CLASSES));  // [0, NC): list lengths, [NC, 2 NC): queue heads of the persistent kernels
  CK(cudaMalloc(&h->axis_status, 2 * B * 4));
  CK(cudaMalloc(&h->axis_iters, 2 * B * 4));
  CK(cudaMalloc(&h->axis_polished, 2 * B * 4));
  CK(cudaMalloc(&h->axis_obj, 2 * B * 8));
  CK(cudaMalloc(&h->mqm, B * 2 * 84 * 8));
  CK(cudaMalloc(&h->partial, 1024 * sizeof(ArgminPair)));
  CK(cudaMalloc(&h->ticket, 4));
  CK(cudaMemset(h->ticket, 0, 4));
  CK(cudaMalloc(&h->work, SPECTRAL_NUM_WORK * 8));
  CK(cudaMemset(h->work, 0, SPECTRAL_NUM_WORK * 8));
  for (auto &slot : h->ev)
    for (auto &e : slot) CK(cudaEventCreate(&e));
  for (auto &slot : h->ev_cls)
    for (auto &c : slot) { CK(cudaEventCreate(&c[0])); CK(cudaEventCreate(&c[1])); }
  return SPECTRAL_SUCCESS;
}

extern "C" int spectral_destroy(spectral_handle_t *h) {
  if (!h) return SPECTRAL_ERR_INVALID;
  cudaSetDevice(h->device);
  if (h->comm) spectral_comm_destroy(h);
  if (h->xg_rec) cudaFree(h->xg_rec);
  if (h->xg_pay) cudaFree(h->xg_pay);
  void *tkb[] = {h->tk.hist, h->tk.st, h->tk.block_ties, h->tk.ck, h->tk.ci, h->tk.cc, h->tk_rec, h->tk_pay};
  for (void *p : tkb) if (p) cudaFree(p);
  if (h->tk_hostpay) cudaFreeHost(h->tk_hostpay);
  if (h->tk_hostrec) cudaFreeHost(h->tk_hostrec);
  void *qsb[] = {h->qs_keys, h->qs_keys2, h->qs_ids, h->qs_ids2, h->qs_tmp, h->qs_tile, h->qs_leader, h->qs_misc, h->qs_st, h->qs_blk, h->qs_lu,
                 h->qs_qv, h->qs_w, h->qs_x, h->qs_cub, h->qs_fs};
  for (void *p : qsb) if (p) cudaFree(p);
  void *bufs[] = {h->cstatus, h->lists, h->counts, h->axis_status, h->axis_iters, h->axis_polished, h->axis_obj, h->mqm,
                  h->partial, h->ticket, h->work, h->d_K, h->d_status, h->d_iters, h->d_flags, h->d_npts, h->d_segs, h->d_ctrl,
                  h->d_obj, h->d_cost, h->d_samples, h->d_lu};
  for (void *p : bufs) if (p) cudaFree(p);
  for (auto p : h->d_in) if (p) cudaFree(p);
  for (auto &slot : h->ev)
    for (auto &e : slot) if (e) cudaEventDestroy(e);
  for (auto &slot : h->ev_cls)
    for (auto &c : slot) { if (c[0]) cudaEventDestroy(c[0]); if (c[1]) cudaEventDestroy(c[1]); }
  if (h->stream) cudaStreamDestroy(h->stream);
  for (auto &s : h->side) if (s) cudaStreamDestroy(s);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  for (auto &e : h->ev_join) if (e) cudaEventDestroy(e);
  delete h;
  return SPECTRAL_SUCCESS;
}

extern "C" int spectral_set_timing(spectral_handle_t *h, int enabled) {
  if (!h) return SPECTRAL_ERR_INVALID;
  h->timing = enabled != 0;
  h->timed_calls = 0;
  return SPECTRAL_SUCCESS;
}
extern "C" int spectral_get_timing(spectral_handle_t *h, float ms[SPECTRAL_NUM_KERNELS], int *calls) {
  if (!h || !ms) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  const int n = (int)(h->timed_calls < spectral_handle::kTimingSlots ? h->timed_calls : spectral_handle::kTimingSlots);
  for (int k = 0; k < SPECTRAL_NUM_KERNELS; k++) ms[k] = 0.f;
  for (int s = 0; s < n; s++) {
    CK(cudaEventSynchronize(h->ev[s][SPECTRAL_NUM_KERNELS - 1]));
    for (int k = 0; k < SPECTRAL_NUM_KERNELS - 1; k++) {
      float t = 0.f;
      CK(cudaEventElapsedTime(&t, h->ev[s][k], h->ev[s][k + 1]));
      ms[k] += t;
    }
  }
  if (calls) *calls = n;
  return SPECTRAL_SUCCESS;
}
extern "C" int spectral_get_class_timing(spectral_handle_t *h, float ms[SPECTRAL_NUM_CLASSES]) {
  if (!h || !ms) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  const int n = (int)(h->timed_calls < spectral_handle::kTimingSlots ? h->timed_calls : spectral_handle::kTimingSlots);
  for (int c = 0; c < SPECTRAL_NUM_CLASSES; c++) ms[c] = 0.f;
  for (int s = 0; s < n; s++)
    for (int c = 0; c < h->classes_timed && c < SPECTRAL_NUM_CLASSES; c++) {
      float t = 0.f;
      CK(cudaEventSynchronize(h->ev_cls[s][c][1]));
      CK(cudaEventElapsedTime(&t, h->ev_cls[s][c][0], h->ev_cls[s][c][1]));
      ms[c] += t;
    }
  return SPECTRAL_SUCCESS;
}
extern "C" int spectral_get_work(spectral_handle_t *h, double work[SPECTRAL_NUM_WORK], int reset) {
  if (!h || !work) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(work, h->work, SPECTRAL_NUM_WORK * 8, cudaMemcpyDeviceToHost));
  if (reset) CK(cudaMemset(h->work, 0, SPECTRAL_NUM_WORK * 8));
  return SPECTRAL_SUCCESS;
}

template <int KC>
static cudaError_t launch_qpd(spectral_handle *h, const QpArgs &qa, int B, cudaStream_t st) {
  const size_t smem = QpdLayout<KC>::BYTES;
  cudaError_t e = cudaFuncSetAttribute(k_qpd<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_qpd<KC><<<B < h->sm_count ? B : h->sm_count, 2 * QpdLayout<KC>::TA, smem, st>>>(qa);
  h->launches++;
  return cudaGetLastError();
}

template <int KC>
static cudaError_t launch_qpa(spectral_handle *h, const QpArgs &qa, int B, cudaStream_t st) {
  const size_t smem = QpdLayout<KC>::BYTES;
  cudaError_t e = cudaFuncSetAttribute(k_qpa<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int grid = B < 2 * h->sm_count ? B : 2 * h->sm_count;
  k_qpa<KC><<<grid, 2 * QpdLayout<KC>::TA, smem, st>>>(qa);
  h->launches++;
  return cudaGetLastError();
}

static int ensure_qps_buffers(spectral_handle *h) {
  const size_t Bm = (size_t)h->max_batch, km = (size_t)h->k_max;
  if (!h->qs_keys) {
    CK(cudaMalloc(&h->qs_keys, Bm * 8)); CK(cudaMalloc(&h->qs_keys2, Bm * 8));
    CK(cudaMalloc(&h->qs_ids, Bm * 4)); CK(cudaMalloc(&h->qs_ids2, Bm * 4));
    CK(cudaMalloc(&h->qs_tmp, 4 * Bm * 4)); CK(cudaMalloc(&h->qs_tile, 2 * Bm * 4));
    CK(cudaMalloc(&h->qs_leader, Bm * 4)); CK(cudaMalloc(&h->qs_misc, 2 * 4)); CK(cudaMalloc(&h->qs_st, 4 * Bm * 4));
    CK(cudaMalloc(&h->qs_blk, 2 * Bm * sizeof(QpsTileBlk)));
    CK(cudaMalloc(&h->qs_lu, Bm * 2 * km * QP_ROWS * 2 * 8));
    CK(cudaMalloc(&h->qs_fs, (size_t)2 * h->sm_count * QPS_FS_DOUBLES * 8));
    CK(cudaMalloc(&h->qs_qv, Bm * 2 * 8 * 6 * 8)); CK(cudaMalloc(&h->qs_w, Bm * 2 * 8 * QP_ROWS * 8)); CK(cudaMalloc(&h->qs_x, Bm * 2 * QPS_N * 8));
    size_t t1 = 0, t2 = 0, t3 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, h->qs_keys, h->qs_keys2, h->qs_ids, h->qs_ids2, h->max_batch);
    cub::DeviceScan::InclusiveScan(nullptr, t2, h->qs_tmp, h->qs_tmp, cub::Max(), h->max_batch);
    cub::DeviceScan::ExclusiveSum(nullptr, t3, h->qs_tmp, h->qs_tmp, h->max_batch);
    h->qs_cub_bytes = t1 > t2 ? (t1 > t3 ? t1 : t3) : (t2 > t3 ? t2 : t3);
    CK(cudaMalloc(&h->qs_cub, h->qs_cub_bytes));
  }
  return SPECTRAL_SUCCESS;
}
// Shared-KKT path for the K <= 8 class: structure keys -> sort -> tiles of <= 8 scenarios -> prepare -> tile ADMM (DMMA) -> finish
static int launch_qps(spectral_handle *h, const QpArgs &qa, const int *cstatus, int B, cudaStream_t st) {
  { const int rc = ensure_qps_buffers(h); if (rc) return rc; }
  const size_t Bm = (size_t)h->max_batch;
  int *head = h->qs_tmp, *gstart = h->qs_tmp + Bm, *flag = h->qs_tmp + 2 * Bm, *tidx = h->qs_tmp + 3 * Bm;
  int *tile_start = h->qs_tile, *tile_count = h->qs_tile + Bm;
  const int nb = (B + 255) / 256;
  CK(cudaMemsetAsync(h->qs_misc, 0, 8, st));
  const size_t sm_pf = 2 * (size_t)QP_SMEM_PER_WARP;
  const int pf_blocks = (B + 3) / 4;  // two scenarios per warp, two warps per block
  CK(cudaFuncSetAttribute(k_qps_prepare, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_pf));
  // hint pass: the K3 assembly of every scenario of the class with the interval pre-check forced on, no tile yet (leader = -1)
  QpsArgs Hh;
  memset(&Hh, 0, sizeof(Hh));
  Hh.q = qa; Hh.q.lu = h->qs_lu; Hh.q.opt.precheck = 1;
  if (!(Hh.q.opt.precheck_margin > 0.0)) Hh.q.opt.precheck_margin = 1e-3;
  Hh.blk = h->qs_blk; Hh.qv = h->qs_qv; Hh.wrows = h->qs_w; Hh.xout = h->qs_x; Hh.st = h->qs_st;
  CK(cudaMemsetAsync(h->qs_leader, 0xFF, (size_t)B * 4, st));
  k_qps_prepare<<<pf_blocks, 64, sm_pf, st>>>(Hh, h->qs_leader);
  h->launches++;
  k_qps_keys<<<nb, 256, 0, st>>>(cstatus, qa.K, qa.segs, h->k_max, qa.weights, qa.wstride, B, h->qs_keys, h->qs_ids, h->qs_leader,
                                h->qs_st);
  size_t tb = h->qs_cub_bytes;
  CK(cub::DeviceRadixSort::SortPairs(h->qs_cub, tb, h->qs_keys, h->qs_keys2, h->qs_ids, h->qs_ids2, B, 0, 64, st));
  k_qps_heads<<<nb, 256, 0, st>>>(h->qs_keys2, B, head);
  tb = h->qs_cub_bytes;
  CK(cub::DeviceScan::InclusiveScan(h->qs_cub, tb, head, gstart, cub::Max(), B, st));
  k_qps_flags<<<nb, 256, 0, st>>>(h->qs_keys2, gstart, B, flag);
  tb = h->qs_cub_bytes;
  CK(cub::DeviceScan::ExclusiveSum(h->qs_cub, tb, flag, tidx, B, st));
  k_qps_emit<<<nb, 256, 0, st>>>(h->qs_keys2, h->qs_ids2, flag, tidx, B, tile_start, tile_count, h->qs_misc, h->qs_leader);
  QpsArgs A;
  A.q = qa; A.q.lu = h->qs_lu;
  A.tile_start = tile_start; A.tile_count = tile_count; A.n_tiles = h->qs_misc; A.sorted = h->qs_ids2; A.tile_next = h->qs_misc + 1;
  A.fs_scratch = h->qs_fs;
  A.blk = h->qs_blk; A.qv = h->qs_qv; A.wrows = h->qs_w; A.xout = h->qs_x; A.st = h->qs_st;
  CK(cudaFuncSetAttribute(k_qps_finish, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_pf));
  CK(cudaFuncSetAttribute(k_qps4, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Qps4Smem::BYTES));
  k_qps_prepare<<<pf_blocks, 64, sm_pf, st>>>(A, h->qs_leader);
  const int per_sm = 2 * (Qps4Smem::BYTES + 1024 + 16) <= 227 * 1024 ? 2 : 1;
  const int grid = B < per_sm * h->sm_count ? B : per_sm * h->sm_count;
  k_qps4<<<grid, 128, Qps4Smem::BYTES, st>>>(A);
  k_qps_finish<<<pf_blocks, 64, sm_pf, st>>>(A);
  h->launches += 8;
  CK(cudaGetLastError());
  return SPECTRAL_SUCCESS;
}

template <int LPA, int WPB>
static cudaError_t launch_qp(spectral_handle *h, const QpArgs &qa, int B, cudaStream_t st) {
  constexpr int G = 32 / LPA;
  const size_t smem = (size_t)WPB * QP_SMEM_PER_WARP + QP_XCH_DOUBLES * 8;
  cudaError_t e = cudaFuncSetAttribute(k_qp<LPA, WPB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const int warps = (2 * B + G - 1) / G;
  const int blocks = (warps + WPB - 1) / WPB;
  const int cap = 8 * h->sm_count;
  k_qp<LPA, WPB><<<blocks < cap ? blocks : cap, 32 * WPB, smem, st>>>(qa);
  h->launches++;
  return cudaGetLastError();
}

static int solve_device_impl(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t, const SpectralInputs *in,
                             const SpectralOptions *opt_in, SpectralOutputs *out, void *cuda_stream, int sweep);

extern "C" int spectral_solve_batch_device(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                                           const SpectralInputs *in, const SpectralOptions *opt_in,
                                           SpectralOutputs *out, void *cuda_stream) {
  return solve_device_impl(h, variant, B, N, R, delta_t, in, opt_in, out, cuda_stream, 0);
}
extern "C" int spectral_solve_weights_device(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                                             const SpectralInputs *in, const SpectralOptions *opt_in,
                                             SpectralOutputs *out, void *cuda_stream) {
  return solve_device_impl(h, variant, B, N, R, delta_t, in, opt_in, out, cuda_stream, 1);
}

// sweep = 1: `in` holds ONE scenario and B weight vectors (weight sweep): corridor stage once, QP per lane
static int solve_device_impl(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t, const SpectralInputs *in,
                             const SpectralOptions *opt_in, SpectralOutputs *out, void *cuda_stream, int sweep) {
  if (!h || !in || !out) return SPECTRAL_ERR_INVALID;
  if (B <= 0 || B > h->max_batch || N < 3 || N > h->n_max || R < 1 || R > h->r_max)
    return fail(h, SPECTRAL_ERR_CAPACITY, "batch shape exceeds the handle's capacity");
  if (variant != SPECTRAL_TRP && variant != SPECTRAL_CUB) return fail(h, SPECTRAL_ERR_INVALID, "variant");
  if (!out->K || !out->status || !out->segs || !out->ctrl) return fail(h, SPECTRAL_ERR_INVALID, "K/status/segs/ctrl outputs are required");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  SpectralOptions opt;
  if (opt_in) opt = *opt_in; else spectral_default_options(&opt);
  const bool tm = h->timing;
  cudaEvent_t *ev = h->ev[h->timed_calls % spectral_handle::kTimingSlots];
  int evi = 0;
  if (tm) CK(cudaEventRecord(ev[evi++], st));

  // K3a: weight tables
  const int wstride = sweep ? 1 : in->weights_stride;
  const int W = wstride ? B : 1;
  k_tables<<<(2 * W + 127) / 128, 128, 0, st>>>(in->weights, h->mqm, W);
  h->launches++;
  if (tm) CK(cudaEventRecord(ev[evi++], st));

  // K1 + K2: corridors
  CorridorArgs ca{sweep ? 1 : B, N, R, variant, h->k_max, delta_t, in->s_bounds, in->l_bounds, in->s_ref, in->l_ref, out->segs, out->K, h->cstatus};
  if (spectral_corridor_prepare(N, R, &h->corridor_smem) != 0) return fail(h, SPECTRAL_ERR_CUDA, "corridor kernel: shared memory opt-in failed");
  spectral_launch_corridor(ca, st);
  h->launches++;
  CK(cudaGetLastError());
  if (sweep && B > 1) {
    k_broadcast_corridor<<<(B + 255) / 256, 256, 0, st>>>(out->K, out->segs, h->cstatus, h->k_max, B);
    h->launches++;
  }
  if (tm) CK(cudaEventRecord(ev[evi++], st));

  // classification by segment count -> lane class lists
  CK(cudaMemsetAsync(h->counts, 0, 4 * 2 * SP_NUM_CLASSES, st));
  if (B <= 4096) k_classify_ordered<<<1, 1024, 0, st>>>(h->cstatus, out->K, B, h->lists, h->counts);
  else k_classify<<<(B + 255) / 256, 256, 0, st>>>(h->cstatus, out->K, B, h->lists, h->counts);
  h->launches++;
  if (tm) CK(cudaEventRecord(ev[evi++], st));

  // K3 + K4b: QP per lane class
  QpArgs qa;
  qa.N = N; qa.k_max = h->k_max; qa.variant = variant; qa.delta = delta_t;
  qa.ds_bounds = in->ds_bounds; qa.dl_bounds = in->dl_bounds; qa.s_ref = in->s_ref; qa.l_ref = in->l_ref;
  qa.init = in->init; qa.scalars = in->scalars; qa.weights = in->weights; qa.wstride = wstride; qa.in_stride = sweep ? 0 : 1;
  qa.mqm = h->mqm; qa.segs = out->segs; qa.K = out->K;
  qa.opt.max_iter = opt.max_iter; qa.opt.scaling = opt.scaling; qa.opt.check_every = opt.check_termination;
  qa.opt.adapt_every = opt.adaptive_rho_interval; qa.opt.polish = opt.polish; qa.opt.polish_refine = opt.polish_refine_iter;
  qa.opt.eps_abs = opt.eps_abs; qa.opt.eps_rel = opt.eps_rel; qa.opt.eps_pinf = opt.eps_prim_inf; qa.opt.rho0 = opt.rho;
  qa.opt.sigma = opt.sigma; qa.opt.alpha = opt.alpha; qa.opt.adapt_tol = opt.adaptive_rho_tolerance;
  qa.opt.polish_delta = opt.polish_delta; qa.opt.polish_rounds = opt.polish_rounds;
  qa.opt.precheck = opt.infeasibility_precheck; qa.opt.precheck_margin = opt.precheck_margin;
  qa.ctrl = out->ctrl; qa.axis_status = h->axis_status; qa.axis_iters = h->axis_iters; qa.axis_polished = h->axis_polished;
  qa.axis_obj = h->axis_obj; qa.lu = out->lu;
  // the solver classes are independent: fork them onto side streams, join before K5
  CK(cudaEventRecord(h->ev_fork, st));
  for (int cls = 0; cls < SP_NUM_CLASSES; cls++) {
    if (cls > 0 && class_kcap(cls - 1) >= h->k_max) break;  // class cannot occur with this handle's k_max
    cudaStream_t cs = cls == 0 ? st : h->side[cls - 1];
    if (cls > 0) CK(cudaStreamWaitEvent(cs, h->ev_fork, 0));
    qa.list = h->lists + (size_t)cls * B; qa.count = h->counts + cls; qa.next = h->counts + SP_NUM_CLASSES + cls;
    cudaEvent_t *ec = h->ev_cls[h->timed_calls % spectral_handle::kTimingSlots][cls];
    if (tm) CK(cudaEventRecord(ec[0], cs));
    if (cls == 0 && opt.shared_kkt) { const int rc = launch_qps(h, qa, h->cstatus, B, cs); if (rc) return rc; }
    else if (cls == 0) CK((launch_qpa<8>(h, qa, B, cs)));
    else if (cls == 1) CK((launch_qpa<10>(h, qa, B, cs)));
    else if (cls == 2) CK((launch_qpd<12>(h, qa, B, cs)));
    else if (cls == 3) CK((launch_qpd<16>(h, qa, B, cs)));
    else CK((launch_qp<32, 2>(h, qa, B, cs)));
    if (tm) CK(cudaEventRecord(ec[1], cs));
    h->classes_timed = cls + 1;
    if (cls > 0) {
      CK(cudaEventRecord(h->ev_join[cls - 1], cs));
      CK(cudaStreamWaitEvent(st, h->ev_join[cls - 1], 0));
    }
  }
  if (tm) CK(cudaEventRecord(ev[evi++], st));

  // K5: sampling + cost + status merge
  FinalArgs fa;
  fa.B = B; fa.N = N; fa.k_max = h->k_max; fa.variant = variant; fa.delta = delta_t; fa.s_ref = in->s_ref; fa.l_ref = in->l_ref;
  fa.init = in->init; fa.weights = in->weights; fa.wstride = wstride; fa.in_stride = sweep ? 0 : 1; fa.segs = out->segs; fa.K = out->K;
  fa.cstatus = h->cstatus; fa.axis_status = h->axis_status; fa.axis_iters = h->axis_iters; fa.axis_polished = h->axis_polished;
  fa.axis_obj = h->axis_obj; fa.ctrl = out->ctrl; fa.obj = out->obj; fa.a_cost = out->a_cost; fa.samples = out->samples;
  fa.status = out->status; fa.iters = out->iters; fa.flags = out->flags; fa.npts = out->npts; fa.samples_cap = out->samples_cap;
  k_finalize<<<(B + 127) / 128, 128, 0, st>>>(fa, h->work);
  h->launches++;
  CK(cudaGetLastError());
  if (tm) {
    CK(cudaEventRecord(ev[evi++], st));
    h->timed_calls++;
  }
  return SPECTRAL_SUCCESS;
}

static int dev_alloc(spectral_handle *h, void **p, size_t bytes) {
  CK(cudaMalloc(p, bytes));
  return SPECTRAL_SUCCESS;
}

template <typename T>
static int ensure(spectral_handle *h, T **p, size_t *cur, size_t need) {
  if (*cur >= need && *p) return SPECTRAL_SUCCESS;
  if (*p) cudaFree(*p);
  *p = nullptr;
  CK(cudaMalloc((void **)p, need));
  *cur = need;
  return SPECTRAL_SUCCESS;
}

static int solve_async_impl(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t, const SpectralInputs *hin,
                            const SpectralOptions *opt, SpectralOutputs *hout, int sweep);
extern "C" int spectral_solve_batch_async(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                                          const SpectralInputs *hin, const SpectralOptions *opt, SpectralOutputs *hout) {
  return solve_async_impl(h, variant, B, N, R, delta_t, hin, opt, hout, 0);
}
extern "C" int spectral_solve_weights(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                                      const SpectralInputs *hin, const SpectralOptions *opt, SpectralOutputs *hout) {
  const int rc = solve_async_impl(h, variant, B, N, R, delta_t, hin, opt, hout, 1);
  if (rc) return rc;
  return spectral_wait(h);
}
static int solve_async_impl(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t, const SpectralInputs *hin,
                            const SpectralOptions *opt, SpectralOutputs *hout, int sweep) {
  if (!h || !hin || !hout) return SPECTRAL_ERR_INVALID;
  if (B <= 0 || B > h->max_batch || N < 3 || N > h->n_max || R < 1 || R > h->r_max)
    return fail(h, SPECTRAL_ERR_CAPACITY, "batch shape exceeds the handle's capacity");
  if (variant != SPECTRAL_TRP && variant != SPECTRAL_CUB) return fail(h, SPECTRAL_ERR_INVALID, "variant");
  if (!hout->K || !hout->status) return fail(h, SPECTRAL_ERR_INVALID, "K and status outputs are required");
  if (hout->samples && hout->samples_cap <= 0) return fail(h, SPECTRAL_ERR_INVALID, "samples_cap");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  const size_t b = (size_t)B, n = (size_t)N, r = (size_t)R, km = (size_t)h->k_max;
  const size_t bs = sweep ? 1 : b;  // scenarios uploaded
  const size_t in_bytes[9] = {bs * r * n * 16, bs * r * n * 16, bs * n * 16, bs * n * 16, bs * n * 8, bs * n * 8, bs * 48, bs * 80,
                              ((sweep || hin->weights_stride) ? b : 1) * 80};
  const double *src[9] = {hin->s_bounds, hin->l_bounds, hin->ds_bounds, hin->dl_bounds, hin->s_ref, hin->l_ref, hin->init,
                          hin->scalars, hin->weights};
  for (int i = 0; i < 9; i++) {
    if (!src[i]) return fail(h, SPECTRAL_ERR_INVALID, "null input");
    int rc = ensure(h, &h->d_in[i], &h->d_in_bytes[i], in_bytes[i]);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->d_in[i], src[i], in_bytes[i], cudaMemcpyHostToDevice, st));
  }
  {
    const size_t mb = (size_t)h->max_batch;
    int rc = SPECTRAL_SUCCESS;
#define DEV_ALLOC(ptr, bytes) do { if (!(ptr) && rc == SPECTRAL_SUCCESS) rc = dev_alloc(h, (void **)&(ptr), (bytes)); } while (0)
    DEV_ALLOC(h->d_K, mb * 4); DEV_ALLOC(h->d_status, mb * 4); DEV_ALLOC(h->d_iters, mb * 4); DEV_ALLOC(h->d_flags, mb * 4);
    DEV_ALLOC(h->d_npts, mb * 4); DEV_ALLOC(h->d_segs, mb * km * sizeof(SpectralCube)); DEV_ALLOC(h->d_ctrl, mb * 12 * km * 8);
    DEV_ALLOC(h->d_obj, mb * 8); DEV_ALLOC(h->d_cost, mb * 8);
#undef DEV_ALLOC
    if (rc) return rc;
  }
  if (hout->samples) { int rc = ensure(h, &h->d_samples, &h->d_samples_bytes, b * (size_t)hout->samples_cap * 48); if (rc) return rc; }
  if (hout->lu) { int rc = ensure(h, &h->d_lu, &h->d_lu_bytes, b * 2 * km * QP_ROWS * 16); if (rc) return rc; }
  SpectralInputs din = *hin;
  din.s_bounds = h->d_in[0]; din.l_bounds = h->d_in[1]; din.ds_bounds = h->d_in[2]; din.dl_bounds = h->d_in[3];
  din.s_ref = h->d_in[4]; din.l_ref = h->d_in[5]; din.init = h->d_in[6]; din.scalars = h->d_in[7]; din.weights = h->d_in[8];
  SpectralOutputs dout;
  memset(&dout, 0, sizeof(dout));
  dout.K = h->d_K; dout.segs = h->d_segs; dout.ctrl = h->d_ctrl; dout.obj = h->d_obj; dout.a_cost = h->d_cost;
  dout.status = h->d_status; dout.iters = h->d_iters; dout.flags = h->d_flags; dout.npts = h->d_npts;
  dout.samples = hout->samples ? h->d_samples : nullptr; dout.samples_cap = hout->samples_cap;
  dout.lu = hout->lu ? h->d_lu : nullptr;
  if (hout->lu) CK(cudaMemsetAsync(h->d_lu, 0, b * 2 * km * QP_ROWS * 16, st));
  CK(cudaMemsetAsync(h->d_ctrl, 0, b * 12 * km * 8, st));
  CK(cudaMemsetAsync(h->d_segs, 0, b * km * sizeof(SpectralCube), st));
  if (hout->samples) CK(cudaMemsetAsync(h->d_samples, 0, b * (size_t)hout->samples_cap * 48, st));
  int rc = solve_device_impl(h, variant, B, N, R, delta_t, &din, opt, &dout, st, sweep);
  if (rc) return rc;
#define D2H(dst, srcp, bytes) do { if (dst) CK(cudaMemcpyAsync((dst), (srcp), (bytes), cudaMemcpyDeviceToHost, st)); } while (0)
  D2H(hout->K, h->d_K, b * 4); D2H(hout->status, h->d_status, b * 4); D2H(hout->iters, h->d_iters, b * 4);
  D2H(hout->flags, h->d_flags, b * 4); D2H(hout->npts, h->d_npts, b * 4);
  D2H(hout->segs, h->d_segs, b * km * sizeof(SpectralCube)); D2H(hout->ctrl, h->d_ctrl, b * 12 * km * 8);
  D2H(hout->obj, h->d_obj, b * 8); D2H(hout->a_cost, h->d_cost, b * 8);
  D2H(hout->samples, h->d_samples, b * (size_t)hout->samples_cap * 48);
  D2H(hout->lu, h->d_lu, b * 2 * km * QP_ROWS * 16);
#undef D2H
  return SPECTRAL_SUCCESS;
}

extern "C" int spectral_wait(spectral_handle_t *h) {
  if (!h) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  return SPECTRAL_SUCCESS;
}

extern "C" int spectral_solve_batch(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                                    const SpectralInputs *hin, const SpectralOptions *opt, SpectralOutputs *hout) {
  const int rc = spectral_solve_batch_async(h, variant, B, N, R, delta_t, hin, opt, hout);
  if (rc) return rc;
  return spectral_wait(h);
}

extern "C" int spectral_host_alloc(void **p, size_t bytes) {
  if (!p) return SPECTRAL_ERR_INVALID;
  *p = nullptr;
  return cudaHostAlloc(p, bytes ? bytes : 1, cudaHostAllocDefault) == cudaSuccess ? SPECTRAL_SUCCESS : SPECTRAL_ERR_CUDA;
}
extern "C" int spectral_host_free(void *p) {
  if (!p) return SPECTRAL_SUCCESS;
  return cudaFreeHost(p) == cudaSuccess ? SPECTRAL_SUCCESS : SPECTRAL_ERR_CUDA;
}

extern "C" int spectral_argmin_device(spectral_handle_t *h, int B, const double *a_cost_dev, long long index_offset,
                                      double *out_cost_dev, long long *out_index_dev, void *cuda_stream) {
  if (!h || B <= 0 || !a_cost_dev || !out_cost_dev || !out_index_dev) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  int blocks = (B + 255) / 256;
  const int cap = h->sm_count * 4 < 1024 ? h->sm_count * 4 : 1024;
  if (blocks > cap) blocks = cap;
  k_argmin<<<blocks, 256, 0, st>>>(a_cost_dev, B, index_offset, h->partial, h->ticket, out_cost_dev, out_index_dev);
  h->launches++;
  CK(cudaGetLastError());
  return SPECTRAL_SUCCESS;
}

// ------------------------------------------------------------------ top-k selection (topk.cuh)
static int ensure_topk_scratch(spectral_handle *h, cudaStream_t st) {
  if (h->tk.cc) return SPECTRAL_SUCCESS;  // the last allocation: set only when all of them succeeded
  const size_t hist_bytes = (size_t)TK_PASSES_MAX * TK_BINS * 4;
  if (!h->tk.hist) CK(cudaMalloc(&h->tk.hist, hist_bytes));
  if (!h->tk.st) CK(cudaMalloc(&h->tk.st, sizeof(TopkState)));
  if (!h->tk.block_ties) CK(cudaMalloc(&h->tk.block_ties, TK_GRID_MAX * 4));
  if (!h->tk.ck) CK(cudaMalloc(&h->tk.ck, TK_MAX * 8));
  if (!h->tk.ci) CK(cudaMalloc(&h->tk.ci, TK_MAX * 8));
  CK(cudaMemsetAsync(h->tk.hist, 0, hist_bytes, st));  // the kernels restore zero histograms, ticket and counter behind them
  CK(cudaMemsetAsync(h->tk.st, 0, sizeof(TopkState), st));
  CK(cudaMalloc(&h->tk.cc, TK_MAX * 8));
  return SPECTRAL_SUCCESS;
}

// npass + 2 launches: the radix passes (6 implicit, 12 explicit), compaction, finish (ties + sort + output)
static int topk_run(spectral_handle *h, TopkArgs a, cudaStream_t st) {
  { const int rc = ensure_topk_scratch(h, st); if (rc) return rc; }
  a.s = h->tk;
  const long long per_block = (long long)TK_THREADS * TK_UNROLL;
  const int cap = 4 * h->sm_count < TK_GRID_MAX ? 4 * h->sm_count : TK_GRID_MAX;
  const long long want = ((long long)a.n + per_block - 1) / per_block;
  const int grid = want < cap ? (int)want : cap;
  const int npass = (a.total_bits + TK_BITS - 1) / TK_BITS;
  for (int p = 0; p < npass; p++) k_topk_pass<<<grid, TK_THREADS, 0, st>>>(a, p);
  k_topk_compact<<<grid, TK_THREADS, 0, st>>>(a);
  k_topk_finish<<<grid, TK_FIN_THREADS, 0, st>>>(a);
  h->launches += npass + 2;
  CK(cudaGetLastError());
  return SPECTRAL_SUCCESS;
}

static int topk_implicit(spectral_handle *h, int B, const double *cost, long long index_offset, int k, double *out_cost,
                         long long *out_index, int out_stride, cudaStream_t st) {
  TopkArgs a{};
  a.cost = cost; a.index = nullptr; a.index_offset = index_offset; a.cost_stride = 1;
  a.n = B; a.keff = k < B ? k : B; a.k = k; a.total_bits = 64;
  a.out_cost = out_cost; a.out_index = out_index; a.out_stride = out_stride;
  return topk_run(h, a, st);
}

extern "C" int spectral_topk_device(spectral_handle_t *h, int B, const double *a_cost_dev, long long index_offset, int k,
                                    double *out_cost_dev, long long *out_index_dev, void *cuda_stream) {
  if (!h) return SPECTRAL_ERR_INVALID;
  if (k < 1 || k > SPECTRAL_TOPK_MAX) return fail(h, SPECTRAL_ERR_INVALID, "topk: k must be in [1, SPECTRAL_TOPK_MAX]");
  if (B <= 0) return fail(h, SPECTRAL_ERR_INVALID, "topk: B must be positive");
  if (index_offset < 0) return fail(h, SPECTRAL_ERR_INVALID, "topk: index_offset must be non-negative");
  if (!a_cost_dev || !out_cost_dev || !out_index_dev) return fail(h, SPECTRAL_ERR_INVALID, "topk: NULL pointer");
  CK(cudaSetDevice(h->device));
  return topk_implicit(h, B, a_cost_dev, index_offset, k, out_cost_dev, out_index_dev, 1, (cudaStream_t)cuda_stream);
}

// ------------------------------------------------------------------ upstream of the path (SURVEY.md 8f row 1)
extern "C" int spectral_bounds_device(spectral_handle_t *h, int B, int N, int M, const double *obstacles_dev, const int *n_obs_dev,
                                      const double road[4], int R_cap, double *s_bounds_dev, double *l_bounds_dev, int *n_lanes_dev,
                                      void *cuda_stream) {
  if (!h || !obstacles_dev || !road || !s_bounds_dev || !l_bounds_dev || !n_lanes_dev) return SPECTRAL_ERR_INVALID;
  if (B <= 0 || N < 3 || N > h->n_max || M < 1 || M > SPB_MAX_CARS || R_cap < 1 || R_cap > SPB_MAX_LANES)
    return fail(h, SPECTRAL_ERR_CAPACITY, "bounds: shape exceeds the capacity (obstacles per scenario <= 4, lanes <= 24)");
  CK(cudaSetDevice(h->device));
  BoundsArgs a{B, N, M, R_cap, obstacles_dev, n_obs_dev, road[0], road[1], road[2], road[3], s_bounds_dev, l_bounds_dev, n_lanes_dev};
  if (spectral_launch_bounds(a, h->sm_count, (cudaStream_t)cuda_stream) != 0) return fail(h, SPECTRAL_ERR_CUDA, "bounds kernel: shared memory opt-in failed");
  h->launches++;
  CK(cudaGetLastError());
  return SPECTRAL_SUCCESS;
}

// ------------------------------------------------------------------ downstream of the path (SURVEY.md 8f row 3)
extern "C" int spectral_ego_states_device(spectral_handle_t *h, int B, const double *samples_dev, const int *npts_dev, int samples_cap,
                                          const double *s_offset_dev, int offset_stride, double *states_dev, void *cuda_stream) {
  if (!h || B <= 0 || samples_cap <= 0 || !samples_dev || !npts_dev || !s_offset_dev || !states_dev) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  dim3 grid(B, (samples_cap + 127) / 128);
  k_ego_states<<<grid, 128, 0, (cudaStream_t)cuda_stream>>>(samples_dev, npts_dev, samples_cap, s_offset_dev, offset_stride ? 1 : 0, states_dev, B);
  h->launches++;
  CK(cudaGetLastError());
  return SPECTRAL_SUCCESS;
}
extern "C" int spectral_frenet_to_cartesian_device(spectral_handle_t *h, long long n, const double *ref_dev, const double *s_cond_dev,
                                                   const double *d_cond_dev, double *out_dev, void *cuda_stream) {
  if (!h || n <= 0 || !ref_dev || !s_cond_dev || !d_cond_dev || !out_dev) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  k_frenet_to_cartesian<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)cuda_stream>>>(ref_dev, s_cond_dev, d_cond_dev, out_dev, n);
  h->launches++;
  CK(cudaGetLastError());
  return SPECTRAL_SUCCESS;
}

// ------------------------------------------------------------------ trajectories at caller-chosen times (eval.cuh)
// Flat grid-stride loop over the B*T points, one thread per point.  A block's points are consecutive in the output, so
// they are staged in shared memory and written back as one contiguous run (the 6- and 2-double rows would otherwise
// be strided stores); the scenario's durations and control points are read through L1.
#define EVAL_THREADS 256
__global__ void __launch_bounds__(EVAL_THREADS) k_eval(const EvalArgs a, double *states, double *jerk, double *horizon) {
  __shared__ double s_st[EVAL_THREADS * 6];
  __shared__ double s_jk[EVAL_THREADS * 2];
  __shared__ long long s_b0;
  __shared__ int s_j0;
  const long long n = (long long)a.B * a.T;
  for (long long base = (long long)blockIdx.x * EVAL_THREADS; base < n; base += (long long)gridDim.x * EVAL_THREADS) {
    if (threadIdx.x == 0) { s_b0 = base / a.T; s_j0 = (int)(base - s_b0 * a.T); }  // one 64-bit division per tile
    __syncthreads();
    const long long p = base + threadIdx.x;
    if (p < n) {
      const unsigned off = (unsigned)s_j0 + threadIdx.x;  // < 2^31 + EVAL_THREADS
      const int b = (int)(s_b0 + off / (unsigned)a.T), j = (int)(off % (unsigned)a.T);
      double st[6], jk[2];
      const double H = eval_point(a, b, j, st, jk);
#pragma unroll
      for (int i = 0; i < 6; i++) s_st[6 * threadIdx.x + i] = st[i];
      s_jk[2 * threadIdx.x] = jk[0];
      s_jk[2 * threadIdx.x + 1] = jk[1];
      if (horizon && j == 0) horizon[b] = H;
    }
    __syncthreads();
    const int cnt = n - base < EVAL_THREADS ? (int)(n - base) : EVAL_THREADS;
    double *so = states + 6 * base;
    for (int i = threadIdx.x; i < 6 * cnt; i += EVAL_THREADS) so[i] = s_st[i];
    if (jerk) {
      double *jo = jerk + 2 * base;
      for (int i = threadIdx.x; i < 2 * cnt; i += EVAL_THREADS) jo[i] = s_jk[i];
    }
    __syncthreads();
  }
}

extern "C" int spectral_eval_device(spectral_handle_t *h, int B, const SpectralOutputs *dev_out, int T, const double *times_dev,
                                    int times_stride, double *states_dev, double *jerk_dev, double *horizon_dev, void *cuda_stream) {
  if (!h) return SPECTRAL_ERR_INVALID;
  if (!dev_out || !dev_out->K || !dev_out->segs || !dev_out->ctrl || !dev_out->status)
    return fail(h, SPECTRAL_ERR_INVALID, "eval: K/segs/ctrl/status are required");
  if (!times_dev || !states_dev) return fail(h, SPECTRAL_ERR_INVALID, "eval: NULL times or states");
  if (B < 1 || T < 1) return fail(h, SPECTRAL_ERR_INVALID, "eval: B and T must be positive");
  if (times_stride != 0 && times_stride != 1) return fail(h, SPECTRAL_ERR_INVALID, "eval: times_stride must be 0 or 1");
  CK(cudaSetDevice(h->device));
  const EvalArgs a{B, T, h->k_max, times_stride, dev_out->K, dev_out->status, dev_out->segs, dev_out->ctrl, times_dev};
  const long long want = ((long long)B * T + EVAL_THREADS - 1) / EVAL_THREADS, cap = 8LL * h->sm_count;
  k_eval<<<(unsigned)(want < cap ? want : cap), EVAL_THREADS, 0, (cudaStream_t)cuda_stream>>>(a, states_dev, jerk_dev, horizon_dev);
  h->launches++;
  CK(cudaGetLastError());
  return SPECTRAL_SUCCESS;
}

// ------------------------------------------------------------------ multi-GPU best-trajectory exchange (NCCL)
namespace {
struct NcclApi {
  void *lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi *nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (!tried) {
    tried = true;
    // the soname first: in a process that already holds an NCCL (e.g. torch's bundled one) this resolves to THAT copy
    api.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!api.lib) api.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (api.lib) {
      api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.lib, "ncclGetUniqueId");
      api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.lib, "ncclCommInitRank");
      api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
      api.AllGather = (decltype(api.AllGather))dlsym(api.lib, "ncclAllGather");
      api.Broadcast = (decltype(api.Broadcast))dlsym(api.lib, "ncclBroadcast");
      api.AllReduce = (decltype(api.AllReduce))dlsym(api.lib, "ncclAllReduce");
      api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.lib, "ncclGetErrorString");
      if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllGather || !api.Broadcast || !api.AllReduce)
        api.lib = nullptr;
    }
  }
  return api.lib ? &api : nullptr;
}
struct WinnerRec { double cost; long long idx; };
// payload of a winner: K, then the segments, then the control points
constexpr size_t kPayBytes = 16 + 32 * sizeof(SpectralCube) + 12 * 32 * 8;
__global__ void k_pack_record(const double *cost, const long long *idx, WinnerRec *rec) { rec->cost = *cost; rec->idx = *idx; }
__global__ void k_pick_winner(const WinnerRec *all, int nranks, WinnerRec *win, int *win_rank) {
  ArgminPair best{1.0e300, 0x7fffffffffffffffLL};
  int br = 0;
  for (int r = 0; r < nranks; r++) {
    const ArgminPair o{all[r].cost, all[r].idx};
    const ArgminPair nb = argmin_better(best, o);
    if (nb.idx != best.idx || nb.cost != best.cost) br = r;
    best = nb;
  }
  win->cost = best.cost; win->idx = best.idx; *win_rank = br;
}
__global__ void k_pack_winner(const WinnerRec *win, long long offset, int B, int k_max, const int *K, const SpectralCube *segs, const double *ctrl,
                              unsigned char *pay) {
  const long long loc = win->idx - offset;
  if (loc < 0 || loc >= B) return;  // not this rank's scenario
  int *hdr = (int *)pay;
  const int Kw = K[loc];
  if (threadIdx.x == 0) { hdr[0] = Kw; hdr[1] = k_max; hdr[2] = 0; hdr[3] = 0; }
  SpectralCube *ps = (SpectralCube *)(pay + 16);
  double *pc = (double *)(pay + 16 + 32 * sizeof(SpectralCube));
  for (int k = threadIdx.x; k < 32; k += blockDim.x)
    if (k < Kw && k < k_max) ps[k] = segs[(size_t)loc * k_max + k];
  for (int j = threadIdx.x; j < 12 * 32; j += blockDim.x) pc[j] = (j < 12 * Kw && j < 12 * k_max) ? ctrl[(size_t)loc * 12 * k_max + j] : 0.0;
}
// top-k exchange: slot j of the payload buffer gets winner j's payload from the rank that owns it (header: K, rank, 1, 0);
// every other rank leaves the slot zero, so a byte-wise sum over ranks reproduces it exactly
__global__ void k_pack_topk(const WinnerRec *win, int rank, long long offset, int B, int k_max, const int *K, const SpectralCube *segs,
                            const double *ctrl, unsigned char *pay) {
  const int j = blockIdx.x;
  const long long idx = win[j].idx, loc = idx - offset;
  if (idx < 0 || loc < 0 || loc >= B) return;
  unsigned char *p = pay + (size_t)j * kPayBytes;
  int *hdr = (int *)p;
  const int Kw = K[loc];
  if (threadIdx.x == 0) { hdr[0] = Kw; hdr[1] = rank; hdr[2] = 1; hdr[3] = 0; }
  SpectralCube *ps = (SpectralCube *)(p + 16);
  double *pc = (double *)(p + 16 + 32 * sizeof(SpectralCube));
  for (int q = threadIdx.x; q < 32; q += blockDim.x)
    if (q < Kw && q < k_max) ps[q] = segs[(size_t)loc * k_max + q];
  for (int q = threadIdx.x; q < 12 * 32; q += blockDim.x) pc[q] = (q < 12 * Kw && q < 12 * k_max) ? ctrl[(size_t)loc * 12 * k_max + q] : 0.0;
}
// a rank without scenarios contributes k empty records (+inf, -1): ranked after every real entry by the merge
__global__ void k_empty_records(WinnerRec *rec, int k) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < k) { rec[j].cost = __longlong_as_double(0x7FF0000000000000LL); rec[j].idx = -1; }
}
}  // namespace

extern "C" int spectral_comm_unique_id(unsigned char id[128]) {
  if (!id) return SPECTRAL_ERR_INVALID;
  NcclApi *n = nccl_api();
  if (!n) return SPECTRAL_ERR_CUDA;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId");
  ncclUniqueId u;
  if (n->GetUniqueId(&u) != ncclSuccess) return SPECTRAL_ERR_CUDA;
  memcpy(id, &u, 128);
  return SPECTRAL_SUCCESS;
}
extern "C" int spectral_comm_init(spectral_handle_t *h, int nranks, int rank, const unsigned char id[128]) {
  if (!h || nranks < 1 || rank < 0 || rank >= nranks) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  if (h->comm) spectral_comm_destroy(h);
  h->nranks = nranks; h->rank = rank;
  if (h->xg_rec) { cudaFree(h->xg_rec); h->xg_rec = nullptr; }
  CK(cudaMalloc(&h->xg_rec, (size_t)(4 + nranks) * sizeof(WinnerRec)));
  if (!h->xg_pay) CK(cudaMalloc(&h->xg_pay, kPayBytes));
  if (nranks == 1) return SPECTRAL_SUCCESS;
  NcclApi *n = nccl_api();
  if (!n || !id) return fail(h, SPECTRAL_ERR_CUDA, "NCCL is not available (libnccl.so.2 could not be loaded)");
  ncclUniqueId u;
  memcpy(&u, id, 128);
  const ncclResult_t r = n->CommInitRank(&h->comm, nranks, u, rank);
  if (r != ncclSuccess) return fail(h, SPECTRAL_ERR_CUDA, std::string("ncclCommInitRank: ") + (n->GetErrorString ? n->GetErrorString(r) : "error"));
  return SPECTRAL_SUCCESS;
}
extern "C" int spectral_comm_destroy(spectral_handle_t *h) {
  if (!h) return SPECTRAL_ERR_INVALID;
  if (h->comm) {
    NcclApi *n = nccl_api();
    if (n) n->CommDestroy(h->comm);
    h->comm = nullptr;
  }
  h->nranks = 1; h->rank = 0;
  return SPECTRAL_SUCCESS;
}

extern "C" int spectral_sweep_argmin(spectral_handle_t *h, int B_local, const SpectralOutputs *dev_out, long long index_offset,
                                     SpectralWinner *winner, void *cuda_stream) {
  if (!h || !dev_out || !winner || B_local <= 0 || !dev_out->a_cost || !dev_out->K || !dev_out->segs || !dev_out->ctrl) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  if (!h->xg_rec) { const int rc = spectral_comm_init(h, 1, 0, nullptr); if (rc) return rc; }
  cudaStream_t st = (cudaStream_t)cuda_stream;
  WinnerRec *rec = (WinnerRec *)h->xg_rec;          // [0] local, [1] winner, [2 ..] gathered, [2 + nranks] scratch (cost, idx)
  WinnerRec *win = rec + 1, *all = rec + 2;
  double *tmp_cost = (double *)(rec + 2 + h->nranks);
  long long *tmp_idx = (long long *)(tmp_cost + 1);
  int *win_rank = (int *)(rec + 3 + h->nranks);
  int rc = spectral_argmin_device(h, B_local, dev_out->a_cost, index_offset, tmp_cost, tmp_idx, st);
  if (rc) return rc;
  k_pack_record<<<1, 1, 0, st>>>(tmp_cost, tmp_idx, rec);
  NcclApi *n = h->nranks > 1 ? nccl_api() : nullptr;
  if (h->nranks > 1) {
    if (!n || !h->comm) return fail(h, SPECTRAL_ERR_INVALID, "spectral_comm_init has not been called on this handle");
    if (n->AllGather(rec, all, sizeof(WinnerRec), ncclUint8, h->comm, st) != ncclSuccess) return fail(h, SPECTRAL_ERR_CUDA, "ncclAllGather");
  } else {
    CK(cudaMemcpyAsync(all, rec, sizeof(WinnerRec), cudaMemcpyDeviceToDevice, st));
  }
  k_pick_winner<<<1, 1, 0, st>>>(all, h->nranks, win, win_rank);
  k_pack_winner<<<1, 128, 0, st>>>(win, index_offset, B_local, h->k_max, dev_out->K, dev_out->segs, dev_out->ctrl, h->xg_pay);
  h->launches += 3;
  WinnerRec hw;
  int hr = 0;
  CK(cudaMemcpyAsync(&hw, win, sizeof(WinnerRec), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&hr, win_rank, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (h->nranks > 1 && n->Broadcast(h->xg_pay, h->xg_pay, kPayBytes, ncclUint8, hr, h->comm, st) != ncclSuccess)
    return fail(h, SPECTRAL_ERR_CUDA, "ncclBroadcast");
  static unsigned char hostpay[kPayBytes];  // (a handle is not thread-safe; one exchange at a time per process)
  CK(cudaMemcpyAsync(hostpay, h->xg_pay, kPayBytes, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  memset(winner, 0, sizeof(*winner));
  winner->cost = hw.cost; winner->index = hw.idx; winner->rank = hr;
  const int *hdr = (const int *)hostpay;
  winner->K = hdr[0];
  memcpy(winner->segs, hostpay + 16, 32 * sizeof(SpectralCube));
  memcpy(winner->ctrl, hostpay + 16 + 32 * sizeof(SpectralCube), 12 * 32 * 8);
  return SPECTRAL_SUCCESS;
}

extern "C" int spectral_sweep_topk(spectral_handle_t *h, int B_local, const SpectralOutputs *dev_out, long long index_offset, int k,
                                   SpectralWinner *winners, int *n_out, void *cuda_stream) {
  if (!h) return SPECTRAL_ERR_INVALID;
  if (k < 1 || k > SPECTRAL_TOPK_MAX) return fail(h, SPECTRAL_ERR_INVALID, "sweep_topk: k must be in [1, SPECTRAL_TOPK_MAX]");
  if (B_local < 0) return fail(h, SPECTRAL_ERR_INVALID, "sweep_topk: B_local must be non-negative");
  if (index_offset < 0) return fail(h, SPECTRAL_ERR_INVALID, "sweep_topk: index_offset must be non-negative");
  if (!dev_out || !winners || !n_out) return fail(h, SPECTRAL_ERR_INVALID, "sweep_topk: NULL pointer");
  if (B_local > 0 && (!dev_out->a_cost || !dev_out->K || !dev_out->segs || !dev_out->ctrl))
    return fail(h, SPECTRAL_ERR_INVALID, "sweep_topk: a_cost/K/segs/ctrl are required");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const bool multi = h->nranks > 1;
  NcclApi *n = multi ? nccl_api() : nullptr;
  if (multi && (!n || !h->comm)) return fail(h, SPECTRAL_ERR_INVALID, "spectral_comm_init has not been called on this handle");
  const int nr = multi ? h->nranks : 1;
  if (h->tk_cap < k || h->tk_cap_ranks < nr) {  // sized by k and the number of ranks, never by the batch
    if (h->tk_rec) cudaFree(h->tk_rec);
    if (h->tk_pay) cudaFree(h->tk_pay);
    if (h->tk_hostpay) cudaFreeHost(h->tk_hostpay);
    if (h->tk_hostrec) cudaFreeHost(h->tk_hostrec);
    h->tk_rec = nullptr; h->tk_pay = nullptr; h->tk_hostpay = nullptr; h->tk_hostrec = nullptr; h->tk_cap = 0;
    CK(cudaMalloc(&h->tk_rec, (size_t)(2 + nr) * k * sizeof(WinnerRec)));
    CK(cudaMalloc(&h->tk_pay, (size_t)k * kPayBytes));
    CK(cudaHostAlloc(&h->tk_hostpay, (size_t)k * kPayBytes, cudaHostAllocDefault));
    CK(cudaHostAlloc(&h->tk_hostrec, (size_t)k * sizeof(WinnerRec), cudaHostAllocDefault));
    h->tk_cap = k; h->tk_cap_ranks = nr;
  }
  WinnerRec *loc = (WinnerRec *)h->tk_rec, *merged = loc + k, *all = loc + 2 * k;
  if (B_local > 0) {
    const int rc = topk_implicit(h, B_local, dev_out->a_cost, index_offset, k, &loc->cost, &loc->idx, 2, st);
    if (rc) return rc;
  } else {
    k_empty_records<<<(k + 255) / 256, 256, 0, st>>>(loc, k);
    h->launches++;
  }
  const WinnerRec *win = loc;
  if (multi) {  // phase 1: every rank's k records -> the same select over nranks x k records (explicit indices)
    if (n->AllGather(loc, all, (size_t)k * sizeof(WinnerRec), ncclUint8, h->comm, st) != ncclSuccess) return fail(h, SPECTRAL_ERR_CUDA, "ncclAllGather");
    TopkArgs a{};
    a.cost = &all->cost; a.index = &all->idx; a.cost_stride = 2;
    a.n = nr * k; a.keff = k; a.k = k; a.total_bits = 128;
    a.out_cost = &merged->cost; a.out_index = &merged->idx; a.out_stride = 2;
    const int rc = topk_run(h, a, st);
    if (rc) return rc;
    win = merged;
  }
  // phase 2: payloads of the winners this rank owns, summed over ranks
  CK(cudaMemsetAsync(h->tk_pay, 0, (size_t)k * kPayBytes, st));
  k_pack_topk<<<k, 128, 0, st>>>(win, multi ? h->rank : 0, index_offset, B_local, h->k_max, dev_out->K, dev_out->segs, dev_out->ctrl, h->tk_pay);
  h->launches++;
  CK(cudaGetLastError());
  if (multi && n->AllReduce(h->tk_pay, h->tk_pay, (size_t)k * kPayBytes, ncclUint8, ncclSum, h->comm, st) != ncclSuccess)
    return fail(h, SPECTRAL_ERR_CUDA, "ncclAllReduce");
  WinnerRec *hrec = (WinnerRec *)h->tk_hostrec;
  CK(cudaMemcpyAsync(hrec, win, (size_t)k * sizeof(WinnerRec), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  int cnt = 0;
  while (cnt < k && hrec[cnt].idx >= 0) cnt++;
  if (cnt) {
    CK(cudaMemcpyAsync(h->tk_hostpay, h->tk_pay, (size_t)cnt * kPayBytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  for (int j = 0; j < k; j++) {
    SpectralWinner *w = winners + j;
    memset(w, 0, sizeof(*w));
    if (j >= cnt) { w->cost = __builtin_huge_val(); w->index = -1; w->rank = -1; continue; }
    const unsigned char *p = h->tk_hostpay + (size_t)j * kPayBytes;
    const int *hdr = (const int *)p;
    w->cost = hrec[j].cost; w->index = hrec[j].idx; w->rank = hdr[1]; w->K = hdr[0];
    memcpy(w->segs, p + 16, 32 * sizeof(SpectralCube));
    memcpy(w->ctrl, p + 16 + 32 * sizeof(SpectralCube), 12 * 32 * 8);
  }
  *n_out = cnt;
  return SPECTRAL_SUCCESS;
}

extern "C" int spectral_measure_fp64_peak(spectral_handle_t *h, double *tflops) {
  if (!h || !tflops) return SPECTRAL_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  const int blocks = h->sm_count * 8, threads = 256, iters = 1 << 15;
  double *buf = nullptr;
  CK(cudaMalloc(&buf, (size_t)blocks * threads * 8));
  cudaEvent_t e0, e1;
  CK(cudaEventCreate(&e0));
  CK(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 4; rep++) {
    CK(cudaEventRecord(e0, h->stream));
    k_fp64_peak<<<blocks, threads, 0, h->stream>>>(buf, iters);
    CK(cudaEventRecord(e1, h->stream));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    const double fl = 2.0 * 8.0 * (double)iters * blocks * threads;
    const double tf = fl / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(buf);
  *tflops = best;
  return SPECTRAL_SUCCESS;
}
