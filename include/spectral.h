/*
 * include/spectral.h -- C-ABI of the B200-native planning hot path (libspectral.so).
 *
 * Plain C, no C++ or torch types, caller-owned buffers, int status returns, no exceptions
 * across the boundary.  One handle per GPU; a handle is not thread-safe.
 *
 * What each entry point replaces in the reference (paths relative to /root/reference):
 *   find_traj()                 src/trp_wrapper.cpp:16-306 (libtrp.so), src/cub_wrapper.cpp:16-285
 *                               (libcub.so): exported by our libtrp.so / libcub.so with the same
 *                               signature, Params layout (include/btrapz/py_cpp_.h:6-21), hidden
 *                               input/output files and return values, so src/trp_wrapper.py:45-54 and
 *                               src/cub_wrapper.py load them unchanged.
 *   spectral_solve_batch*()     the body of find_traj between parsing and cost for B scenarios at once:
 *                               PiecewiseJerkSpeedProblem::CorridorGeneration (src/solve_3d.cc:323-486,
 *                               src/cuboid_3d.cc:301-407), CorridorSplit (:729-772 / :588-625),
 *                               CollisionCheck (:488-714 / :409-573), FormulateProblem (:1143-1229),
 *                               Optimize (:1231-1414) incl. the OSQP solve it delegates to
 *                               (osqp_setup/osqp_solve, :1246-1249) and the Bezier sampling (:1279-1392),
 *                               and the wrapper cost (src/trp_wrapper.cpp:217-286).
 *   spectral_argmin_device()    new (the reference has no batch): best trajectory of a sweep.
 *   spectral_topk_device()      new: the k best trajectories of a sweep (spectral_sweep_topk across GPUs).
 *   spectral_eval_device()      new: solved trajectories at caller-chosen times (the sampler of Optimize, :1351-1390, on
 *                               any time grid, with jerk).
 *   spectral_certify_device()   new: how far each returned trajectory is from satisfying the constraint rows of its QP
 *                               (the rows of CalculateAffineConstraint, :779-1129), and its cost with uncertified
 *                               scenarios set to the failure sentinel.
 *   SpectralCube                struct Cube, include/btrapz/cube_type.h:2-24 (same 112-byte layout).
 *   SpectralParams              struct Params, include/btrapz/py_cpp_.h:6-21 (same 88-byte layout).
 */
#ifndef SPECTRAL_H
#define SPECTRAL_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPECTRAL_TRP 0 /* trapezoid-prism corridors, reference libtrp.so (solve_3d.cc) */
#define SPECTRAL_CUB 1 /* cuboid corridors, reference libcub.so (cuboid_3d.cc) */

/* API return codes */
#define SPECTRAL_SUCCESS 0
#define SPECTRAL_ERR_INVALID 1
#define SPECTRAL_ERR_CUDA 2
#define SPECTRAL_ERR_CAPACITY 3

/* per-scenario status[] values */
#define SPECTRAL_SOLVED 0            /* OSQP status 1 */
#define SPECTRAL_SOLVED_INACCURATE 1 /* OSQP status 2; the reference accepts it (solve_3d.cc:1253) */
#define SPECTRAL_FAIL_NO_CORRIDOR 2  /* CollisionCheck selected nothing (reference: UB, solve_3d.cc:617) */
#define SPECTRAL_FAIL_SOLVER 3       /* Optimize() == false -> find_traj returns 1e11 (trp_wrapper.cpp:199) */
#define SPECTRAL_FAIL_POINTS_CHECK 4 /* CHECK_EQ(var_index, num_of_points_) would abort (solve_3d.cc:1407) */
/* SPECTRAL_FAIL_TOO_MANY: the corridor exceeds a capacity.  K[] is then
 *   0        when a region holds more than 64 cubes before the split (64 or more slope breaks) or after it,
 *   0        when CollisionCheck selects more than 64 distinct cubes (the CPU oracle reports their count here),
 *   the true segment count K when K > k_max. */
#define SPECTRAL_FAIL_TOO_MANY 5

/* per-scenario flags[] bits */
#define SPECTRAL_FLAG_POLISHED_S 1 /* s-axis control points come from an accepted polish step */
#define SPECTRAL_FLAG_POLISHED_L 2 /* l-axis likewise */
#define SPECTRAL_FLAG_VERIFIED_S 4 /* s-axis control points satisfy the KKT conditions of the QP (exact optimum) */
#define SPECTRAL_FLAG_VERIFIED_L 8 /* l-axis likewise */
#define SPECTRAL_FLAG_VERIFIED (SPECTRAL_FLAG_VERIFIED_S | SPECTRAL_FLAG_VERIFIED_L)
/* diagnostics of a polish that did not reach a KKT proof, four bits per axis (s: bits 4-7, l: bits 8-11):
 * 1 stationarity / feasibility of the polished point not reached, 2 active set still changing after polish_rounds,
 * 4 non-positive pivot in the polish factorisation, 8 polished point rejected (not better than the ADMM iterate) */
#define SPECTRAL_FLAG_DIAG_SHIFT_S 4
#define SPECTRAL_FLAG_DIAG_SHIFT_L 8

#define SPECTRAL_FAIL_COST 100000000000.0 /* the reference's failure sentinel */

/* struct Cube (cube_type.h:2-24), 112 bytes */
typedef struct {
  int beg_t, end_t;
  double t;
  double t_dif;
  double beg_l, end_l;
  double upp_skew, upp_bias, down_skew, down_bias;
  double l_upp_skew, l_upp_bias, l_down_skew, l_down_bias;
  unsigned char merge, split;
  int count;
} SpectralCube;

/* struct Params (py_cpp_.h:6-21), 88 bytes */
typedef struct {
  double s_acc_weight, s_jerk_weight, l_acc_weight, l_jerk_weight;
  double weight_s_ref, weight_ds_ref, weight_l_ref, weight_dl_ref;
  double weight_end_s, weight_end_l;
  int iteration;
} SpectralParams;

/* Inputs of a batch of B scenarios sharing (N knots, R regions, delta_t).  All FP64, C-contiguous. */
typedef struct {
  const double *s_bounds;  /* [B][R][N][2]  (lo, hi) of s per region and knot  (set_x_bounds) */
  const double *l_bounds;  /* [B][R][N][2]  (lo, hi) of l                      (set_y_bounds) */
  const double *ds_bounds; /* [B][N][2]                                         (set_dx_bounds) */
  const double *dl_bounds; /* [B][N][2]                                         (set_dy_bounds) */
  const double *s_ref;     /* [B][N]                                            (set_x_ref) */
  const double *l_ref;     /* [B][N]                                            (set_y_ref) */
  const double *init;      /* [B][6]  s, ds, dds, l, dl, ddl at t = 0 */
  const double *scalars;   /* [B][10] ds_ref, dl_ref, dds_lo, dds_hi, ddds_lo, ddds_hi, ddl_lo, ddl_hi, dddl_lo, dddl_hi */
  const double *weights;   /* [B][10] or [1][10] in Params order (s_acc .. weight_end_l) */
  int weights_stride;      /* 1: one weight vector per scenario; 0: one for the whole batch */
} SpectralInputs;

/* Outputs.  Host-buffer entry points: any pointer except K/status may be NULL to skip it.  Device entry point
 * (spectral_solve_batch_device): K, status, segs and ctrl are required (later stages read them), the rest optional. */
typedef struct {
  int *K;             /* [B] segment count = new_corridor.size() */
  SpectralCube *segs; /* [B][k_max] the selected corridor sequence */
  double *ctrl;       /* [B][12*k_max]: s-axis control points [0,6K), l-axis [6K,12K) (OSQP x order) */
  double *obj;        /* [B] QP objective 0.5 x'Px + q'x at ctrl */
  double *a_cost;     /* [B] the wrapper's trajectory cost; 1e11 on failure */
  int *status;        /* [B] SPECTRAL_SOLVED ... */
  int *iters;         /* [B] ADMM iterations (max over the two axis problems) */
  int *flags;         /* [B] SPECTRAL_FLAG_* */
  int *npts;          /* [B] number of trajectory samples */
  double *samples;    /* [B][samples_cap][6]: s, ds, dds, l, dl, ddl per sample */
  int samples_cap;
  double *lu;         /* debug: [B][2 axes][k_max][21][2] the QP's (l, u) rows per segment lane */
} SpectralOutputs;

typedef struct {
  int max_iter;          /* 5000  (trp_wrapper.cpp:191) */
  double eps_abs;        /* 1e-5  (solve_3d.cc:1239) */
  double eps_rel;        /* 1e-5  (solve_3d.cc:1238) */
  double eps_prim_inf;   /* 2.5e-5 (solve_3d.cc:1454) */
  double rho;            /* 0.1   OSQP default */
  double sigma;          /* 1e-6  OSQP default */
  double alpha;          /* 1.6   OSQP default */
  int scaling;           /* 4     (solve_3d.cc:1242) */
  int check_termination; /* 25    OSQP default */
  int adaptive_rho_interval; /* 100 = OSQP's fixed rule; 0 disables adaptation */
  double adaptive_rho_tolerance; /* 5 */
  int polish;            /* 1: refine the ADMM solution to the exact optimum of the identified active set */
  double polish_delta;   /* 1e-6: regularisation of the active rows (OSQP's delta) */
  int polish_refine_iter;/* 4 */
  int polish_rounds;     /* 8: active-set correction rounds; a round that changes nothing verifies the KKT conditions */
  int infeasibility_precheck; /* 0 (default: every scenario goes through the reference's OSQP iteration).  1: scenarios whose
                           corridor is PROVABLY empty -- a constraint row with l > u, consecutive segments whose position
                           intervals do not meet at the joint (rows 5 of segment k and 0 of k+1 share t_k c_k5 = t_k+1 c_k+1,0,
                           solve_3d.cc:918-925), or an initial state outside the first segment's position / velocity /
                           acceleration rows (solve_3d.cc:896-912) -- fail at once instead of after up to max_iter ADMM
                           iterations.  Sound (necessary conditions of feasibility); not what the reference does: on such
                           problems its OSQP either certifies infeasibility late or stops at max_iter, sometimes with the
                           status "solved inaccurate" and a constraint-violating trajectory. */
  double precheck_margin; /* 1e-3: an interval gap must exceed this to count */
  int shared_kkt;         /* 0 (default): every scenario runs OSQP's own iteration (per-scenario Ruiz scaling and adaptive rho).
                             1: scenarios with K <= 8 that share one KKT structure (same K, same segment durations, same weights; only
                             bounds, initial state and references differ -- BASELINE configs[2]) are solved in tiles of 8 against ONE
                             reduced-KKT inverse, the per-iteration solve being a multi-right-hand-side product on the FP64 tensor cores
                             (mma.sync m8n8k4 f64).  Same QP, same ADMM, same termination test, but the scaling is the tile's first
                             member's and rho adapts per tile: the optimum and the decided solved / failed classes are the reference's,
                             the iteration counts are not OSQP's. */
} SpectralOptions;

typedef struct spectral_handle spectral_handle_t;

void spectral_default_options(SpectralOptions *opt);

/* device: CUDA ordinal.  Capacities: scenarios per call, knots, regions, segments (k_max <= 32).
 * A failed spectral_create may leave a handle in *out, so that spectral_last_error can explain the failure; that handle
 * must then be passed to spectral_destroy. */
int spectral_create(int device, int max_batch, int n_max, int r_max, int k_max, spectral_handle_t **out);
int spectral_destroy(spectral_handle_t *h);
const char *spectral_last_error(const spectral_handle_t *h);

/* Host buffers: copies in, runs the device path, copies out, synchronises.  (The end-to-end path.) */
int spectral_solve_batch(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                         const SpectralInputs *host_in, const SpectralOptions *opt,
                         SpectralOutputs *host_out);

/* The same, split for pipelining: _async enqueues the copies and kernels on the handle's own stream and returns;
 * spectral_wait() blocks until the outputs have landed.  host_in / host_out buffers must stay valid (and host_out
 * untouched) until then; with page-locked buffers (spectral_host_alloc) the copies overlap the kernels of other
 * handles, which is how a caller keeps the GPU full at small batch sizes: a few handles, round robin.
 * At most one batch in flight per handle.  (The reference's find_traj is synchronous: trp_wrapper.cpp:16-306.) */
int spectral_solve_batch_async(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                               const SpectralInputs *host_in, const SpectralOptions *opt,
                               SpectralOutputs *host_out);
int spectral_wait(spectral_handle_t *h);
/* Page-locked host memory for the buffers above (cudaHostAlloc / cudaFreeHost). */
int spectral_host_alloc(void **ptr, size_t bytes);
int spectral_host_free(void *ptr);

/* Device buffers (already resident in HBM): enqueues on `cuda_stream` (a cudaStream_t, may be NULL)
 * and returns without synchronising. */
int spectral_solve_batch_device(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                                const SpectralInputs *dev_in, const SpectralOptions *opt,
                                SpectralOutputs *dev_out, void *cuda_stream);

/* Weight sweep: ONE scenario, B candidate weight vectors -- the batch form of the reference's tuning objective
 * (src/trp_wrapper.py:56-97 run_btrapz: ten weights suggested in [0, 50] per trial, one find_traj call each).
 * `in` holds one scenario (the [B] dimension of every array except `weights` is 1) and weights[B][10] (weights_stride is
 * ignored).  The corridor stage (CorridorGeneration / CollisionCheck) runs once and is shared by all lanes: same A, same
 * (l, u); P and q per weight vector.  Outputs are per lane, laid out as for spectral_solve_batch (segs / K repeated). */
int spectral_solve_weights(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                           const SpectralInputs *host_in, const SpectralOptions *opt, SpectralOutputs *host_out);
int spectral_solve_weights_device(spectral_handle_t *h, int variant, int B, int N, int R, double delta_t,
                                  const SpectralInputs *dev_in, const SpectralOptions *opt, SpectralOutputs *dev_out, void *cuda_stream);

/* Best trajectory of a sweep: (min a_cost, lowest index on ties) over B device-resident costs.
 * out_cost/out_index are DEVICE pointers (one double / one long long); index_offset is added to the
 * local index so shards can be compared across ranks. */
int spectral_argmin_device(spectral_handle_t *h, int B, const double *a_cost_dev, long long index_offset,
                           double *out_cost_dev, long long *out_index_dev, void *cuda_stream);

/* Upstream of the path (SURVEY.md 8f row 1), device buffers, enqueued on cuda_stream: the reference's bound generator
 * src/cart_frenet.py:644-807 (Car.getCar: obstacle -> space-time prism, lateral edges), :819-830 (lineFromPoints, 0.01 rounding),
 * :833-1026 (get_bounds, 'yield' homotopy), called as in :1539-1557.
 *   obstacles [B][M][6] = (s, l, t0, vel_s, vel_l, horizon) in creation order, M <= 4; n_obs [B] (NULL: M everywhere);
 *   road[4] = (s_l_l, s_u_l, d_l_l, d_u_l) (cart_frenet.py:54-58: 0, 50, -2, 8)
 *   -> s_bounds, l_bounds [B][R_cap][N][2] in the layout of SpectralInputs and n_lanes [B] = lanes of the road found.
 * Lanes r >= n_lanes[b] are written as EMPTY lanes (l_lo = 1 > l_hi = -1, s = the free road): CollisionCheck's lateral test
 * (solve_3d.cc:534) never selects a cube of such a region, so spectral_solve_batch_device(.., R = R_cap, ..) on these arrays
 * gives the corridors and trajectories of the unpadded scenarios.  n_lanes[b] = -1: more lanes than R_cap (or than the
 * kernel's tables hold); all R_cap lanes of that scenario are then written empty, so a solve on them reports SPECTRAL_FAIL_NO_CORRIDOR.  Bit-identical to the reference's get_bounds on its
 * specified domain (cars whose smallest lateral edges tie are ordered by object hash there: creation order here). */
int spectral_bounds_device(spectral_handle_t *h, int B, int N, int M, const double *obstacles_dev, const int *n_obs_dev,
                           const double road[4], int R_cap, double *s_bounds_dev, double *l_bounds_dev, int *n_lanes_dev,
                           void *cuda_stream);

/* Downstream of the path (SURVEY.md 8f row 3), device buffers, enqueued on cuda_stream:
 * spectral_ego_states_device         run_ego() of src/cart_frenet.py:1126-1221: samples [B][cap][6] (the `samples` output:
 *                                    s, ds, dds, l, dl, ddl) + npts [B] -> states [B][cap][4] = (position along the road,
 *                                    lateral position, speed with ds floored at 5.0, heading = round(atan2(dl, ds), 2) of the
 *                                    forward difference).  s_offset [B] or [1] (offset_stride 1 / 0) is curr_state.position[0],
 *                                    added to the states i >= 1 (:1190-1191).
 * spectral_frenet_to_cartesian_device  frenet_to_cartesian3D() of src/cart_frenet.py:347-381: ref [n][6] = (rs, rx, ry, rtheta,
 *                                    rkappa, rdkappa), s_cond [n][3], d_cond [n][3] -> out [n][6] = (x, y, v, a, theta, kappa). */
int spectral_ego_states_device(spectral_handle_t *h, int B, const double *samples_dev, const int *npts_dev, int samples_cap,
                               const double *s_offset_dev, int offset_stride, double *states_dev, void *cuda_stream);
int spectral_frenet_to_cartesian_device(spectral_handle_t *h, long long n, const double *ref_dev, const double *s_cond_dev,
                                        const double *d_cond_dev, double *out_dev, void *cuda_stream);

/* Trajectories of solved scenarios evaluated at caller-chosen times (device buffers, enqueued on cuda_stream, no
 * synchronisation).  Works on any solve output, including a top-k winner or an earlier plan uploaded into [k] arrays.
 *   dev_out    K, segs, ctrl and status of B scenarios, all required, in the handle's k_max layout (as spectral_sweep_argmin).
 *   times_dev  [T] (times_stride 0: the same times for every scenario) or [B][T] (times_stride 1), seconds.
 *   states_dev [B][T][6] = (s, ds, dds, l, dl, ddl): the layout of `samples` and of SpectralInputs.init, so with T = 1 it
 *              is the next solve's init, and it feeds spectral_ego_states_device directly (samples_cap = npts = T).
 *   jerk_dev   [B][T][2] = (ddds, dddl), or NULL.      horizon_dev [B] = H, or NULL.
 * B is limited only by int (not by the handle's max_batch); B * T may exceed 2^31.
 * Time model.  tau = 0 is the initial state.  Segment k spans [T_k, T_{k+1}], T_0 = 0, T_{k+1} = T_k + segs[k].t, summed in
 *   double in array order (the corridor order, not beg_t: the cuboid variant leaves beg_t unsorted); H = T_K.  A time at a
 *   joint belongs to the segment that ends there (the reference's sampler also ends each segment at u = 1).  Segments with
 *   t_k <= 1e-9 (CorridorSplit's slivers) are never selected; a time past the last selectable segment's end evaluates it
 *   at u = 1.  u = clamp((tau - T_k) / t_k, 0, 1), c = ctrl[6k .. 6k+6) (s axis; l axis: ctrl[6K + 6k ..]),
 *     s = t_k sum c_i B5_i(u),  ds = 5 sum (c_{i+1} - c_i) B4_i(u),  dds = 20 sum D2c_i B3_i(u) / t_k,
 *     ddds = 60 sum D3c_i B2_i(u) / t_k^2            (the arithmetic of the `samples` of spectral_solve_batch*)
 *   Times in [-1e-9, H + 1e-9] are valid and clamped to [0, H], so a horizon end computed as (N - 1) delta is not lost to
 *   the rounding of the summed durations.
 * NaN rows of states and jerk: times outside that range or NaN (the scenario's horizon is still H); every row of a
 *   scenario whose status is not SOLVED or SOLVED_INACCURATE or whose K is outside [1, k_max] (its horizon is NaN too)
 *   or whose segments are all slivers (horizon H).  segs / ctrl are never read beyond K.
 * SPECTRAL_ERR_INVALID: null handle, dev_out, K/segs/ctrl/status, times_dev or states_dev; B < 1; T < 1; times_stride
 *   other than 0 or 1. */
int spectral_eval_device(spectral_handle_t *h, int B, const SpectralOutputs *dev_out, int T, const double *times_dev,
                         int times_stride, double *states_dev, double *jerk_dev, double *horizon_dev, void *cuda_stream);

/* Feasibility certificate of solved trajectories (device buffers, enqueued on cuda_stream, no synchronisation, no handle
 * scratch, one kernel launch).  It certifies PRIMAL FEASIBILITY of the returned control points for the QP they were solved
 * for, to within tol: every row l <= A x <= u of that QP, assembled by the solver's own code.  It does not certify
 * optimality.  Why it is needed: the ranking entry points (argmin, top-k, sweep) rank on a_cost alone, and a scenario with
 * status SOLVED_INACCURATE (accepted as the reference does, solve_3d.cc:1253) may carry a trajectory that leaves its
 * corridor -- on infeasible problems OSQP can stop "solved inaccurate" at max_iter.
 *   dev_in        ds_bounds, dl_bounds, init and scalars are required; the other fields are ignored and may be NULL (no row
 *                 depends on the weights or the references).  inputs_stride 1: B scenarios in the layout of
 *                 spectral_solve_batch*; 0: one scenario for every b (the layout of spectral_solve_weights*).
 *   dev_out       K, segs, ctrl and status of B scenarios, in the handle's k_max layout; a_cost too when cost_dev is given.
 *   tol           host array, one acceptable violation per row family, each >= 0.
 *   viol_dev      [B][2][SPECTRAL_CERT_FAMILIES] (axis s = 0, l = 1; family): the largest max(l - Ax, Ax - u, 0) over the
 *                 axis' rows of that family, or NULL.
 *   cost_dev      [B]: a_cost[b] when every entry of viol is <= tol[family] (a NaN entry never is), else SPECTRAL_FAIL_COST;
 *                 or NULL (not both outputs).  Feed it to spectral_argmin_device / spectral_topk_device, or point
 *                 dev_out.a_cost at it for spectral_sweep_argmin / spectral_sweep_topk: the best FEASIBLE trajectories.
 * Row families, in the QP's own row units (these are the rows as assembled, not SI units: dividing by t_k or t_k^2 would be
 * meaningless on CorridorSplit's slivers, t_k ~ 1e-15 s).  Segment k of duration t_k, control points c_0..c_5 of one axis:
 *   position      t_k c_i in the corridor (6 rows); the initial position t_0 c_0 = s(0), and the joints
 *                 t_k c_{k,0} - t_{k-1} c_{k-1,5} = 0
 *   velocity      5 (c_{i+1} - c_i) in [ds_lo, ds_hi] over the segment's knots (s) / dl_bounds (l) (5 rows); the initial
 *                 velocity and the velocity joints
 *   acceleration  20 D2c_i = acc x t_k in [lo t_k, hi t_k] (4 rows); the initial acceleration x t_0, and the joints
 *                 t_k D2c_{k-1,3} - t_{k-1} D2c_{k,0} = 0 (acc x t_{k-1} t_k / 20)
 *   jerk          60 D3c_i = jerk x t_k^2 in [lo t_k^2, hi t_k^2] (3 rows)
 * NaN entries and SPECTRAL_FAIL_COST: a scenario that is not certifiable -- status other than SOLVED / SOLVED_INACCURATE,
 *   K outside [1, k_max], or a segment with beg_t / end_t outside [0, N - 1] or beg_t > end_t (checked before any read of
 *   ds_bounds, since segs may come from the caller).  A NaN or infinite control point makes its axis' entries NaN.
 * The l-axis velocity rows read dl_bounds at knots 0..4 (by control index, as the reference does, solve_3d.cc:1003), so for
 *   N < 5 they read past the scenario's [N][2] slab, as the solver does.
 * B is limited only by int (not by the handle's max_batch).
 * SPECTRAL_ERR_INVALID: null handle; variant; a required pointer NULL; both outputs NULL; B < 1; N outside [3, n_max];
 *   inputs_stride other than 0 or 1; tol NULL, or an entry negative or NaN. */
#define SPECTRAL_CERT_FAMILIES 4 /* position, velocity, acceleration, jerk (rows as assembled, see above) */
int spectral_certify_device(spectral_handle_t *h, int variant, int B, int N, const SpectralInputs *dev_in, int inputs_stride,
                            const SpectralOutputs *dev_out, const double tol[SPECTRAL_CERT_FAMILIES], double *viol_dev,
                            double *cost_dev, void *cuda_stream);

/* Multi-GPU sweep (SURVEY.md 8e): scenarios are sharded over ranks (one handle = one GPU = one rank); the ONLY exchange is
 * the best trajectory.  spectral_sweep_argmin is spectral_sweep_topk (below) with k = 1: local top-1 -> NCCL all-gather of one
 * 16-byte (cost, global index) record per rank -> the same select over those records -> the owning rank packs the winner's
 * (K, segments, control points) into a zeroed buffer, which one NCCL all-reduce hands to every rank.  Ties -> lowest global
 * index; failed scenarios carry 1e11 (the reference's sentinel, trp_wrapper.cpp:199).  The library loads libnccl.so.2 at run
 * time.
 *   spectral_comm_unique_id  rank 0 makes the id (ncclGetUniqueId); the caller ships it to the other ranks by any means
 *   spectral_comm_init       every rank, same id (ncclCommInitRank on the handle's device); nranks = 1 needs no NCCL
 *   spectral_sweep_argmin    collective over all ranks; enqueued on cuda_stream, synchronises it, fills *winner on EVERY rank.
 *                            B_local >= 1; a negative index_offset is rejected (SPECTRAL_ERR_INVALID).  A sweep whose every
 *                            cost is above 1e300 or NaN returns its first entry in top-k order: a real index, with its own
 *                            K, segments and control points.  segs and ctrl beyond K are zero. */
typedef struct {
  double cost;         /* a_cost of the best scenario (1e11: every scenario of the sweep failed) */
  long long index;     /* its global index = index_offset of the owning rank + local index */
  int rank;            /* the rank that owns it */
  int K;
  SpectralCube segs[32];
  double ctrl[12 * 32]; /* s-axis control points [0, 6K), l-axis [6K, 12K) */
} SpectralWinner;
int spectral_comm_unique_id(unsigned char id[128]);
int spectral_comm_init(spectral_handle_t *h, int nranks, int rank, const unsigned char id[128]);
int spectral_comm_destroy(spectral_handle_t *h);
int spectral_sweep_argmin(spectral_handle_t *h, int B_local, const SpectralOutputs *dev_out, long long index_offset,
                          SpectralWinner *winner, void *cuda_stream);

/* The k best trajectories of a batch / of a multi-GPU sweep (a ranked shortlist instead of the single winner above).
 *
 * Order: ascending lexicographic on (cost, global index), global index = index_offset + i (index_offset >= 0).
 *   -0.0 and +0.0 compare equal (as in spectral_argmin_device); NaN sorts after every other value, +inf included, and NaNs
 *   rank among themselves by index.  Failed scenarios (SPECTRAL_FAIL_COST) are ordinary entries: filter with
 *   cost < SPECTRAL_FAIL_COST.  The returned cost is the stored a_cost[i], bit for bit (a -0.0 comes back as -0.0).
 * 1 <= k <= SPECTRAL_TOPK_MAX.  With fewer than k entries, the trailing slots hold index = -1, cost = +inf.
 * When some cost is below 1e300, k = 1 returns exactly what spectral_argmin_device returns.
 * B is limited only by int (not by the handle's max_batch).  Deterministic: the same bits on every call, stream and SM count.
 *
 * spectral_topk_device  out_cost_dev[k] / out_index_dev[k] are DEVICE pointers.  Enqueued on cuda_stream with no host
 *                       synchronisation: an exact radix select over B costs (a fixed number of passes), compaction of the
 *                       <= k selected entries and one sort of those (DESIGN.md 3.4).  Scratch belongs to the handle, is
 *                       allocated on first use and does not grow with B; as for spectral_argmin_device, calls on one handle
 *                       must not overlap in time (one stream at a time, or ordered by events).
 * spectral_sweep_topk   collective over all ranks: local top-k -> NCCL all-gather of k 16-byte (cost, global index)
 *                       records per rank -> the same select over the nranks x k records -> each rank packs the payloads
 *                       (K, segments, control points) of the winners it owns into a zeroed [k] buffer, which one NCCL
 *                       all-reduce (sum over bytes: exactly one rank writes each byte) hands to every rank.  Fills
 *                       winners[0..k) on EVERY rank, sorted, and returns the number of real entries in *n_out
 *                       (min(k, total scenarios)); winners[j >= *n_out] have index -1, cost +inf, rank -1, K 0.
 *                       B_local = 0 is allowed: the rank takes part and contributes nothing (dev_out's arrays may then be
 *                       NULL).  Shards must not overlap in global index.  Synchronises cuda_stream.  Handles without a
 *                       communicator of more than one rank take the single-rank path (no NCCL). */
#define SPECTRAL_TOPK_MAX 1024
int spectral_topk_device(spectral_handle_t *h, int B, const double *a_cost_dev, long long index_offset, int k,
                         double *out_cost_dev, long long *out_index_dev, void *cuda_stream);
int spectral_sweep_topk(spectral_handle_t *h, int B_local, const SpectralOutputs *dev_out, long long index_offset, int k,
                        SpectralWinner *winners, int *n_out, void *cuda_stream);

/* Number of kernel launches enqueued by this handle so far (for bench accounting). */
long long spectral_launch_count(const spectral_handle_t *h);

/* Measured FP64 FMA throughput of the device in TFLOP/s (micro-benchmark kernel; used as the
 * roofline denominator of the ADMM kernel because MEASURED_PEAKS.json has no FP64 entry). */
int spectral_measure_fp64_peak(spectral_handle_t *h, double *tflops);

/* Per-kernel-class device time, measured with CUDA events recorded on the launching stream around every
 * kernel class of each solve_batch*_ call while timing is enabled.  Nothing synchronises inside the
 * calls; spectral_get_timing() waits for the recorded events and returns the SUM of milliseconds per
 * class over the last `*calls` (<= 64) calls since spectral_set_timing(h, 1). */
#define SPECTRAL_NUM_KERNELS 6 /* tables, corridor, classify, qp (all solver classes, forked streams), finalize, (argmin: not timed) */
int spectral_set_timing(spectral_handle_t *h, int enabled);
int spectral_get_timing(spectral_handle_t *h, float ms[SPECTRAL_NUM_KERNELS], int *calls);

/* The solver classes by segment count K (one kernel each, forked streams): K <= 8, <= 10, <= 12, <= 16, <= 32.
 * spectral_get_class_timing: summed device ms of each class' kernel (events on that class' stream) over the calls recorded
 * since spectral_set_timing(h, 1); classes overlap in time, so the entries do not add up to the "qp" stage time. */
#define SPECTRAL_NUM_CLASSES 5
int spectral_get_class_timing(spectral_handle_t *h, float ms[SPECTRAL_NUM_CLASSES]);

/* Work counters accumulated on the device by every solve_batch*_ call (synchronises the device):
 * work[0] ADMM iterations summed over axis problems; work[1] their flops in the dense-operator count the kernels execute
 * (72 K^2 + 208 K - 24 per axis-iteration: dense apply of the 6K x 6K inverse + A, A' products; DESIGN.md); work[2] scenarios
 * processed; work[3] scenarios solved; work[4] sum of K (segments written by the corridor kernel); work[5] the iterations
 * in the variable-structure count of SURVEY.md 8d (424 K - 168 per axis-iteration: block-tridiagonal solve, the algorithmic
 * minimum without a shared KKT matrix); work[6 + c] the dense-count flops of solver class c; the rest reserved. */
#define SPECTRAL_NUM_WORK 12
int spectral_get_work(spectral_handle_t *h, double work[SPECTRAL_NUM_WORK], int reset);

/* The reference's plugin entry point (exported by libtrp.so / libcub.so, not by libspectral.so):
 *   double find_traj(SpectralParams *p);                       trp_wrapper.cpp:20, cub_wrapper.cpp:19 */

#ifdef __cplusplus
}
#endif
#endif
