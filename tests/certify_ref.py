"""NumPy reference of the feasibility certificate (spectral_certify_device, certify.cuh): the QP as the CPU oracle assembles
it (pyoracle.formulate), its rows grouped into the certificate's families, max(l - Ax, Ax - u, 0) per (axis, family)."""
import numpy as np

from spectral_b200 import api

NF = len(api.CERT_FAMILIES)
BAR = 1e-12   # |kernel - oracle| <= BAR * max(1, max over the family's rows of sum_i |A_ri x_i|): the two order their sums differently


def row_groups(K):
    """axis * NF + family of every row of the oracle's QP, in its row order (helpers.lu_to_qp_rows): per axis K x 18 segment
    rows, 3 initial-state rows, 3 rows per joint.  Lane rows 0-5 position, 6-10 velocity, 11-14 acceleration, 15-17 jerk;
    the initial-state and joint rows are (position, velocity, acceleration)."""
    seg = np.array([0] * 6 + [1] * 5 + [2] * 4 + [3] * 3)
    per_axis = np.concatenate([np.tile(seg, K), np.tile([0, 1, 2], K)])
    return np.concatenate([per_axis, per_axis + NF])


def oracle_qp(variant, batch, b, segs):
    """The oracle's (A, l, u) for scenario b of `batch` and the corridor `segs` (no row depends on the weights)."""
    import pyoracle as po
    import scipy.sparse as sp
    from spectral_b200.wire import Scenario
    sc = Scenario(batch.n_knots, batch.delta_t, batch.init[b, :3], batch.init[b, 3:], batch.scalars[b], batch.s_bounds[b],
                  batch.l_bounds[b], batch.ds_bounds[b], batch.dl_bounds[b], batch.s_ref[b], batch.l_ref[b])
    qp = po.formulate(variant, sc, np.ones(10), segs)
    A = sp.csc_matrix((qp["A_x"], qp["A_i"], qp["A_p"]), shape=(qp["m"], qp["n"]))
    assert qp["m"] == 42 * len(segs)
    return A, qp["l"], qp["u"]


def oracle_viol(variant, batch, b, segs, x):
    """(viol [2, NF], scale [2, NF]): the largest max(l - Ax, Ax - u, 0) and the largest sum_i |A_ri x_i| per (axis, family)."""
    A, l, u = oracle_qp(variant, batch, b, segs)
    Ax = A @ x
    e = np.maximum(np.maximum(l - Ax, Ax - u), 0.0)
    mag = abs(A) @ np.abs(x)
    g = row_groups(len(segs))
    viol, scale = np.zeros(2 * NF), np.zeros(2 * NF)
    for j in range(2 * NF):
        viol[j] = e[g == j].max()
        scale[j] = mag[g == j].max()
    return viol.reshape(2, NF), scale.reshape(2, NF)


def check_scenario(variant, batch, b, K, segs, ctrl, viol, label=""):
    """The kernel's viol [2, NF] of one certifiable scenario against the oracle at the bar; returns the oracle's viol."""
    x = ctrl[:12 * K]
    want, scale = oracle_viol(variant, batch, b, segs[:K], x)
    err = np.abs(viol - want)
    assert (err <= BAR * np.maximum(1.0, scale)).all(), (label, b, viol, want, err)
    return want


def certify_oracle(variant, batch, res, tol, bi=None):
    """Oracle viol [B, 2, NF] (NaN where not certifiable) and certified mask [B] of a BatchResult-like (K, status, segs, ctrl)."""
    B = len(res.K)
    tol = np.broadcast_to(np.asarray(tol, dtype=np.float64), (NF,))
    want = np.full((B, 2, NF), np.nan)
    for b in range(B):
        K = int(res.K[b])
        if res.status[b] <= api.SOLVED_INACCURATE and 1 <= K <= 32:
            want[b] = oracle_viol(variant, batch, b if bi is None else bi, res.segs[b, :K], res.ctrl[b, :12 * K])[0]
    cert = (want <= tol[None, None, :]).all(axis=(1, 2))
    return want, cert
