"""CPU oracle of viml_inertial_evaluate / viml_gn_step_vi (test infrastructure only).

IMUFactor::Evaluate (vins_estimator/src/factor/imu_factor.h:19-181) with IntegrationBase::evaluate (factor/integration_base.h),
restated statement by statement in scalar Python with Eigen's operation order (SURVEY.md Appendix A: Quaterniond(p[6], p[3], p[4],
p[5]), inverse() divides by the squared norm, _transformVector, toRotationMatrix, no normalisation).  sqrt_info is an input (the
reference recomputes it from the pre-integration's covariance in every Evaluate).

UNPINNED against reference code: the reference's imu_factor.h cannot be compiled into this repository's checks (it needs Eigen and
Ceres).  The pins are independent: a second restatement with numpy matrices and finite differences in the tangent space
(tests/test_inertial_cpu.py).  The prior is the C++ oracle's orc_marginalization_factor_evaluate, which is pinned against the
reference's compiled marginalization_factor.cpp.
"""
import math

import numpy as np

O_P, O_R, O_V, O_BA, O_BG = 0, 3, 6, 9, 12


# ---- Eigen quaternion / small matrix arithmetic (Appendix A) ----------------------------------------------------------------
def quat(p):                      # Quaterniond(p[6], p[3], p[4], p[5]) as (w, x, y, z)
    return (float(p[6]), float(p[3]), float(p[4]), float(p[5]))


def qmul(a, b):
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    return (aw * bw - ax * bx - ay * by - az * bz, aw * bx + ax * bw + ay * bz - az * by,
            aw * by + ay * bw + az * bx - ax * bz, aw * bz + az * bw + ax * by - ay * bx)


def qinv(q):
    w, x, y, z = q
    n2 = w * w + x * x + y * y + z * z
    return (w / n2, -x / n2, -y / n2, -z / n2)


def cross(a, b):
    return (a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])


def qrot(q, v):                   # _transformVector
    u = q[1:]
    uv = cross(u, v)
    uv = (uv[0] + uv[0], uv[1] + uv[1], uv[2] + uv[2])
    c = cross(u, uv)
    return tuple(v[k] + q[0] * uv[k] + c[k] for k in range(3))


def rotmat(q):                    # toRotationMatrix
    w, x, y, z = q
    tx, ty, tz = 2 * x, 2 * y, 2 * z
    twx, twy, twz = tx * w, ty * w, tz * w
    txx, txy, txz = tx * x, ty * x, tz * x
    tyy, tyz, tzz = ty * y, tz * y, tz * z
    return np.array([[1 - (tyy + tzz), txy - twz, txz + twy], [txy + twz, 1 - (txx + tzz), tyz - twx],
                     [txz - twy, tyz + twx, 1 - (txx + tyy)]])


def skew(v):                      # Utility::skewSymmetric
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def qleft(q):                     # Utility::Qleft
    w, v = q[0], np.array(q[1:])
    m = np.zeros((4, 4))
    m[0, 0], m[0, 1:], m[1:, 0] = w, -v, v
    m[1:, 1:] = w * np.eye(3) + skew(v)
    return m


def qright(q):                    # Utility::Qright
    w, v = q[0], np.array(q[1:])
    m = np.zeros((4, 4))
    m[0, 0], m[0, 1:], m[1:, 0] = w, -v, v
    m[1:, 1:] = w * np.eye(3) - skew(v)
    return m


def mv3(M, v):
    return tuple((M[r, 0] * v[0] + M[r, 1] * v[1]) + M[r, 2] * v[2] for r in range(3))


# ---- IMUFactor::Evaluate ----------------------------------------------------------------------------------------------------
def imu_factor_evaluate(xi, sbi, xj, sbj, preint, jac, sqrt_info, G, want_jac=True):
    """One IMU factor: residual [15] and the Ceres Jacobian blocks pose_i [15, 7], sb_i [15, 9], pose_j [15, 7], sb_j [15, 9]
    (row-major, column 6 of the pose blocks 0), or (residual, None) without Jacobians."""
    jac = np.asarray(jac, dtype=np.float64)
    sqrt_info = np.asarray(sqrt_info, dtype=np.float64)
    G = tuple(float(g) for g in G)
    Pi, Qi = tuple(map(float, xi[:3])), quat(xi)
    Pj, Qj = tuple(map(float, xj[:3])), quat(xj)
    Vi, Bai, Bgi = tuple(map(float, sbi[0:3])), tuple(map(float, sbi[3:6])), tuple(map(float, sbi[6:9]))
    Vj, Baj, Bgj = tuple(map(float, sbj[0:3])), tuple(map(float, sbj[3:6])), tuple(map(float, sbj[6:9]))
    dt = float(preint[0])
    delta_p = tuple(map(float, preint[1:4]))
    delta_q = (float(preint[7]), float(preint[4]), float(preint[5]), float(preint[6]))
    delta_v = tuple(map(float, preint[8:11]))
    lin_ba, lin_bg = tuple(map(float, preint[11:14])), tuple(map(float, preint[14:17]))
    dp_dba, dp_dbg = jac[O_P:O_P + 3, O_BA:O_BA + 3], jac[O_P:O_P + 3, O_BG:O_BG + 3]       # imu_factor.h Evaluate
    dq_dbg = jac[O_R:O_R + 3, O_BG:O_BG + 3]
    dv_dba, dv_dbg = jac[O_V:O_V + 3, O_BA:O_BA + 3], jac[O_V:O_V + 3, O_BG:O_BG + 3]
    # IntegrationBase::evaluate
    dba = tuple(Bai[k] - lin_ba[k] for k in range(3))
    dbg = tuple(Bgi[k] - lin_bg[k] for k in range(3))
    th = mv3(dq_dbg, dbg)
    cdq = qmul(delta_q, (1.0, th[0] / 2, th[1] / 2, th[2] / 2))                             # delta_q * Utility::deltaQ(dq_dbg * dbg)
    a1, a2 = mv3(dv_dba, dba), mv3(dv_dbg, dbg)
    cdv = tuple((delta_v[k] + a1[k]) + a2[k] for k in range(3))
    b1, b2 = mv3(dp_dba, dba), mv3(dp_dbg, dbg)
    cdp = tuple((delta_p[k] + b1[k]) + b2[k] for k in range(3))
    Qii = qinv(Qi)
    ap = tuple(0.5 * G[k] * dt * dt + Pj[k] - Pi[k] - Vi[k] * dt for k in range(3))
    av = tuple(G[k] * dt + Vj[k] - Vi[k] for k in range(3))
    rp = qrot(Qii, ap)
    rv = qrot(Qii, av)
    e = qmul(qinv(cdq), qmul(Qii, Qj))
    r = np.array([rp[0] - cdp[0], rp[1] - cdp[1], rp[2] - cdp[2], 2 * e[1], 2 * e[2], 2 * e[3],
                  rv[0] - cdv[0], rv[1] - cdv[1], rv[2] - cdv[2],
                  Baj[0] - Bai[0], Baj[1] - Bai[1], Baj[2] - Bai[2], Bgj[0] - Bgi[0], Bgj[1] - Bgi[1], Bgj[2] - Bgi[2]])
    res = sqrt_info @ r
    if not want_jac:
        return res, None
    RiT = rotmat(Qii)
    I3 = np.eye(3)
    jpi, jsi, jpj, jsj = np.zeros((15, 7)), np.zeros((15, 9)), np.zeros((15, 7)), np.zeros((15, 9))
    jpi[O_P:O_P + 3, 0:3] = -RiT
    jpi[O_P:O_P + 3, 3:6] = skew(rp)
    jpi[O_R:O_R + 3, 3:6] = -(qleft(qmul(qinv(Qj), Qi)) @ qright(cdq))[1:, 1:]
    jpi[O_V:O_V + 3, 3:6] = skew(rv)
    jsi[O_P:O_P + 3, 0:3] = -RiT * dt
    jsi[O_P:O_P + 3, 3:6] = -dp_dba
    jsi[O_P:O_P + 3, 6:9] = -dp_dbg
    jsi[O_R:O_R + 3, 6:9] = -qleft(qmul(qmul(qinv(Qj), Qi), delta_q))[1:, 1:] @ dq_dbg
    jsi[O_V:O_V + 3, 0:3] = -RiT
    jsi[O_V:O_V + 3, 3:6] = -dv_dba
    jsi[O_V:O_V + 3, 6:9] = -dv_dbg
    jsi[O_BA:O_BA + 3, 3:6] = -I3
    jsi[O_BG:O_BG + 3, 6:9] = -I3
    jpj[O_P:O_P + 3, 0:3] = RiT
    jpj[O_R:O_R + 3, 3:6] = qleft(qmul(qmul(qinv(cdq), Qii), Qj))[1:, 1:]
    jsj[O_V:O_V + 3, 0:3] = RiT
    jsj[O_BA:O_BA + 3, 3:6] = I3
    jsj[O_BG:O_BG + 3, 6:9] = I3
    return res, (sqrt_info @ jpi, sqrt_info @ jsi, sqrt_info @ jpj, sqrt_info @ jsj)


# ---- batch forms over viml_inertial_factors ---------------------------------------------------------------------------------
def inertial_evaluate(orc, poses, ex_pose, extra, vi, want_jac=True):
    """The viml_inertial_out arrays of a batch: IMU factors by imu_factor_evaluate, priors by the C++ oracle's
    MarginalizationFactor::Evaluate.  Prior rows past n_w are NaN."""
    NI, W = vi.NI, vi.W
    out = {"imu_residual": np.full((NI, 15), np.nan), "imu_jac_pose_i": np.full((NI, 15, 7), np.nan),
           "imu_jac_sb_i": np.full((NI, 15, 9), np.nan), "imu_jac_pose_j": np.full((NI, 15, 7), np.nan),
           "imu_jac_sb_j": np.full((NI, 15, 9), np.nan), "prior_residual": np.full((W, vi.n_max), np.nan)}
    win = vi.imu_window()
    for k in range(NI):
        w = win[k]
        (i, j), (si, sj) = vi.imu_pose[k], vi.imu_sb[k]
        r, J = imu_factor_evaluate(poses[w, i], extra[w, si:si + 9], poses[w, j], extra[w, sj:sj + 9], vi.imu_preint[k],
                                   vi.imu_jacobian[k], vi.imu_sqrt_info[k], vi.gravity, want_jac)
        out["imu_residual"][k] = r
        if want_jac:
            out["imu_jac_pose_i"][k], out["imu_jac_sb_i"][k], out["imu_jac_pose_j"][k], out["imu_jac_sb_j"][k] = J
    for w in range(W):
        n = int(vi.prior_n[w])
        if n == 0:
            continue
        nb = int(vi.prior_n_blocks[w])
        sizes, idxs, x0s, params = [], [], [], []
        for b in range(nb):
            kind, idx, size, first = (int(t) for t in vi.prior_block[w, b])
            x = poses[w, idx] if kind == 0 else ex_pose[w] if kind == 1 else extra[w, idx:idx + size]
            sizes.append(size)
            idxs.append(first)          # keep_block_idx - m with m = 0
            x0s.append(vi.prior_x0[w, b, :size])
            params.append(np.asarray(x, dtype=np.float64)[:size])
        r, _ = orc.marginalization_factor_evaluate(n, 0, sizes, idxs, x0s, vi.prior_jacobian[w, :n, :n], vi.prior_residual[w, :n],
                                                   params, want_jac=False)
        out["prior_residual"][w, :n] = r
    return out


def inertial_cost(orc, poses, ex_pose, extra, vi):
    """1/2 sum |r|^2 per window over the IMU and prior factors (NULL loss, estimator.cpp:1927, :1939)."""
    ev = inertial_evaluate(orc, poses, ex_pose, extra, vi, want_jac=False)
    cost = np.zeros(vi.W)
    for k, w in enumerate(vi.imu_window()):
        cost[w] += 0.5 * float(ev["imu_residual"][k] @ ev["imu_residual"][k])
    for w in range(vi.W):
        n = int(vi.prior_n[w])
        cost[w] += 0.5 * float(ev["prior_residual"][w, :n] @ ev["prior_residual"][w, :n])
    return cost


def gn_step_vi(orc, gn_oracle, cfg, batch, vi, extra, flags, lam=0.0):
    """The oracle's gn_step with the dense list built by this oracle at x, and cost[1] from this oracle at x+ (the true
    nonlinear cost of the IMU and prior factors instead of their linear model)."""
    ev = inertial_evaluate(orc, batch.poses, batch.ex_pose, extra, vi)
    dense = vi.to_dense(ev)
    out = gn_oracle.gn_step(cfg, batch, dense, extra, flags, lam=lam)
    # gn_step's cost[1] = visual f(x+) + the dense factors' linear model: swap the model for the re-evaluated factors
    model = np.zeros(vi.W)
    for (w, r, J, ci) in dense.factors:
        v = np.asarray(r) + np.asarray(J) @ out["dx"][w][np.asarray(ci)]
        model[w] += 0.5 * float(v @ v)
    out["cost"][:, 1] += inertial_cost(orc, out["poses"], out["ex_pose"], out["extra"], vi) - model
    return out
