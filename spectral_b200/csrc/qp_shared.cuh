// spectral_b200/csrc/qp_shared.cuh -- K4a: the SHARED-KKT batched ADMM, multi-right-hand-side solve on the FP64 tensor pipe.
//
// BASELINE.json configs[2] / SURVEY.md 7.4 K4a.  Replaces, for scenarios that share one KKT structure (same segment count K,
// same segment durations t_k, same weights -- only bounds, initial state and references differ), the per-scenario loop behind
// osqp_solve (solve_3d.cc:1246-1249, settings :1235-1243,1446-1462): the reduced KKT operator G = (P + sigma I + A' rho A)^-1
// depends on the structure and rho only, so ONE copy of G serves a TILE of 8 scenarios, and the per-iteration solve
// X~ = G [g_1 .. g_8] becomes a dense multi-RHS contraction on mma.sync.m8n8k4.f64 (DMMA).
//
// This header holds the parts of the path around the tile kernel (k_qps4, qp_shared4.cuh, which describes its thread map and
// its DMMA fragments): the structure keys that group scenarios into tiles (k_qps_keys / heads / flags / emit in capi.cu sort
// the class by key and cut runs of equal keys into tiles of at most QPS_TILE), the per-tile structure block (QpsTileBlk) and
// the kernel arguments (QpsArgs), the DMMA and shared-memory load primitives, and the bodies of the two kernels that bracket
// the tile kernel:
//   k_qps_prepare  K3 assembly of every member (l, u, q), and for a tile's first scenario the tile's scaling, rho and P
//   k_qps_finish   status at max_iter, polish and outputs of every member (qp_finish of qp.cuh) in the tile scaling
//
// What differs from the per-scenario kernels (qp_anchor.cuh / qp_dense.cuh), and why it is a separate, opt-in path
// (SpectralOptions::shared_kkt): a shared G needs ONE scaling and ONE rho for the tile.  The Ruiz scaling (D, E, c) is taken
// from the tile's first scenario (OSQP's depends on q through the cost scaling, and q differs between the members), and rho
// adapts per TILE (OSQP's rule applied to the geometric mean of the members' estimates).  It is therefore the same QP, the
// same ADMM and the same termination test in a slightly different metric -- not OSQP's iterate sequence.  Parity is on what
// north_star pins: decided solved / failed classes and the optimum (polish + KKT proof, qp_finish), tests/test_gpu_parity.py.
// Tiles are formed deterministically (scenarios sorted by (structure key, index)), so runs are reproducible.
#pragma once
#include "qp_dense.cuh"

#define QPS_KC 8
#define QPS_N 48
#define QPS_TILE 8
#define QPS_ROWSZ (21 * 32)             // one (slot, half) plane of the row arrays: [row][lane]
#define QPS_NFRAG 72                    // B fragments of G per axis: [half][36]
// The tile's structure slots are addressed like qp.cuh's lane slots (slot * 8 + segment) through a base pointer shifted so
// that QP_SM_P is the first slot stored: P at QP_SM_P, rho at QPS_RHO, the row scalings E_r at QPS_ER.
#define QPS_RHO (QP_SM_P + 21)
#define QPS_ER (QP_SM_P + 42)
#define QPS_FS_DOUBLES (2 * 57 * 8)     // factor store of one tile CTA (global scratch: read only when G is rebuilt)

// per tile and axis; written by k_qps_prepare from the tile's first scenario, read by k_qps4 / k_qps_finish
struct QpsTileBlk {
  double t[8], tp[8], tn[8];
  double rho[21][8];   // [row][segment]: the RHO slots of qp.cuh with stride 8
  double P[21][8];     // [packed lower-triangle entry][segment]
  double sig[8][6], cD[8][6];
  double c, rhobar;
  int eqmask[8];
  int K, pad;
};

struct QpsArgs {
  QpArgs q;                 // list / count = the K <= 8 class; lu = the assembled (l, u) rows [B][2][k_max][21][2]
  const int *tile_start;    // [n_tiles] first position of the tile in `sorted`
  const int *tile_count;    // [n_tiles] 1..8
  const int *n_tiles;
  const int *sorted;        // scenario ids ordered by (structure key, index)
  int *tile_next;           // queue head of the persistent kernel
  QpsTileBlk *blk;          // [B/1][2]  (indexed by tile)
  double *qv;               // [B][2][8][6] linear cost per scenario
  double *wrows;            // [B][2][8][21] w = z + y / rho at exit
  double *xout;             // [B][2][48] relaxed iterate at exit
  int *st;                  // [B][4]: state, iters, tile, pre
  double *fs_scratch;       // [grid][QPS_FS_DOUBLES] block-Cholesky factor of the tile being (re)built
};

SP_DEV void qps_dmma(double a, double b, double &c0, double &c1) {
#ifndef SPECTRAL_CPU_EMU
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
#endif
}

SP_DEV double qps_lds(const double *p) {
#ifdef SPECTRAL_CPU_EMU
  return *p;
#else
  double a;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(a) : "r"((unsigned)__cvta_generic_to_shared(p)));
  return a;
#endif
}

// k_qps_prepare body: one warp = two scenarios of the K <= 8 class (16 lanes each: 8 segment lanes per axis).  K3 assembly
// (l, u -> a.lu, q -> qv), and for a tile's first scenario the Ruiz scaling / rho / P of the tile.
SP_DEV void qps_prepare_body(const QpsArgs &A, const int *leader_tile, int warp_global, int lane, double *sm) {
  const QpArgs &a = A.q;
  const int cnt = *a.count;
  if (warp_global * 2 >= cnt) return;
  const int grp = lane >> 3, seg = lane & 7;
  const int ap = warp_global * 4 + grp;
  const bool have = ap < 2 * cnt;
  QpLane Q;
  qp_setup<8, 32, 16>(a, ap, have, seg, lane, sm, Q);
  if (!have) return;
  const int b = Q.b, axis = Q.axis;
  double *qs = A.qv + (((size_t)b * 2 + axis) * 8 + seg) * 6;
#pragma unroll
  for (int j = 0; j < 6; j++) qs[j] = Q.q[j];
  if (seg == 0 && axis == 0) { A.st[4 * b + 0] = QP_ST_MAXITER; A.st[4 * b + 1] = 0; A.st[4 * b + 2] = -1; A.st[4 * b + 3] = Q.pre; }
  const int tile = leader_tile[b];
  if (tile < 0) return;
  QpsTileBlk &B = A.blk[2 * tile + axis];
  B.t[seg] = Q.t; B.tp[seg] = Q.tp; B.tn[seg] = Q.tn; B.eqmask[seg] = (int)Q.eqmask;
#pragma unroll
  for (int j = 0; j < 6; j++) { B.sig[seg][j] = Q.sig[j]; B.cD[seg][j] = Q.cD[j]; }
#pragma unroll
  for (int r = 0; r < QP_ROWS; r++) { B.rho[r][seg] = Q.active ? sm[(QP_SM_RHO + r) * 32 + lane] : 0.0; B.P[r][seg] = sm[(QP_SM_P + r) * 32 + lane]; }
  if (seg == 0) { B.c = Q.c; B.rhobar = Q.rhobar; B.K = Q.K; B.pad = 0; }
}

// k_qps_finish body: one warp = two scenarios; status at max_iter, polish, outputs (qp_finish of qp.cuh) in the tile scaling
SP_DEV void qps_finish_body(const QpsArgs &A, int warp_global, int lane, double *sm) {
  const QpArgs &a = A.q;
  const int cnt = *a.count;
  if (warp_global * 2 >= cnt) return;
  const int grp = lane >> 3, seg = lane & 7;
  const int ap = warp_global * 4 + grp;
  const bool have = ap < 2 * cnt;
  const int b = a.list[have ? (ap >> 1) : 0], axis = ap & 1;
  const int tile = A.st[4 * b + 2];
  const bool ok = have && tile >= 0;
  const QpsTileBlk &B = A.blk[2 * (ok ? tile : 0) + axis];
  QpLane Q;
  Q.b = b; Q.axis = axis; Q.K = ok ? a.K[b] : 0; Q.seg = seg; Q.kmaxw = sp_group_max_i(Q.K, 32);
  Q.have = ok; Q.active = ok && seg < Q.K; Q.first = seg == 0; Q.last = seg == Q.K - 1;
  Q.t = ok ? B.t[seg] : 1.0; Q.tp = ok ? B.tp[seg] : 1.0; Q.tn = ok ? B.tn[seg] : 1.0;
  Q.c = ok ? B.c : 1.0; Q.rhobar = ok ? B.rhobar : 0.1; Q.eqmask = ok ? (unsigned)B.eqmask[seg] : 0u; Q.pre = 0; Q.xch = nullptr;
  const double *qs = A.qv + (((size_t)b * 2 + axis) * 8 + seg) * 6;
  const double *lu = a.lu + (((size_t)b * 2 + axis) * a.k_max + seg) * QP_ROWS * 2;
  const double *wr = A.wrows + (((size_t)b * 2 + axis) * 8 + seg) * QP_ROWS;
  const double *xs = A.xout + ((size_t)b * 2 + axis) * QPS_N + 6 * seg;
  double x[6];
#pragma unroll
  for (int j = 0; j < 6; j++) {
    Q.q[j] = Q.active ? qs[j] : 0.0; Q.sig[j] = ok ? B.sig[seg][j] : 1.0; Q.cD[j] = ok ? B.cD[seg][j] : 1.0;
    x[j] = Q.active ? xs[j] : 0.0;
  }
#pragma unroll
  for (int r = 0; r < QP_ROWS; r++) {
    sm[(QP_SM_W + r) * 32 + lane] = Q.active ? wr[r] : 0.0;
    sm[(QP_SM_L + r) * 32 + lane] = Q.active ? lu[2 * r] : -1.0;
    sm[(QP_SM_U + r) * 32 + lane] = Q.active ? lu[2 * r + 1] : 1.0;
    sm[(QP_SM_RHO + r) * 32 + lane] = Q.active ? B.rho[r][seg] : 0.0;
    sm[(QP_SM_P + r) * 32 + lane] = ok ? B.P[r][seg] : ((r == LT(0, 0) || r == LT(1, 1) || r == LT(2, 2) || r == LT(3, 3) || r == LT(4, 4) || r == LT(5, 5)) ? 1.0 : 0.0);
  }
  sp_syncwarp();
  const int state = ok ? A.st[4 * b + 0] : QP_ST_MAXITER, iters = ok ? A.st[4 * b + 1] : 0;
  qp_finish<8, 32, 16>(a, sm, lane, Q, x, state, iters);
}
