"""The IMU factor restatement of tests/inertial_oracle.py (IMUFactor::Evaluate, imu_factor.h:19-181) checked without a GPU: against
a second restatement written with numpy matrices, against finite differences in the tangent space, and for its structure.  Plus
the ctypes mirror of viml_inertial_factors / viml_inertial_out."""
import ctypes as C

import numpy as np
import pytest

import inertial_oracle as io
from conftest import rel_err


# ---- a second restatement: quaternions as 4-vectors (w, x, y, z), products as Qleft matrices ------------------------------------
def _q(p):
    return np.array([p[6], p[3], p[4], p[5]], dtype=np.float64)


def _skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def _left(q):
    m = np.zeros((4, 4))
    m[0, 0], m[0, 1:], m[1:, 0] = q[0], -q[1:], q[1:]
    m[1:, 1:] = q[0] * np.eye(3) + _skew(q[1:])
    return m


def _right(q):
    m = np.zeros((4, 4))
    m[0, 0], m[0, 1:], m[1:, 0] = q[0], -q[1:], q[1:]
    m[1:, 1:] = q[0] * np.eye(3) - _skew(q[1:])
    return m


def _inv(q):
    return np.array([q[0], -q[1], -q[2], -q[3]]) / (q @ q)


def _R(q):
    """q v q* as a matrix, for any (also non-unit) q: (w^2 ... ) written as (1 - 2|u|^2) I + 2 u u^T + 2 w [u]x, which is what
    Eigen's _transformVector and toRotationMatrix both compute without normalising."""
    w, u = q[0], q[1:]
    return (1.0 - 2.0 * (u @ u)) * np.eye(3) + 2.0 * np.outer(u, u) + 2.0 * w * _skew(u)


def imu_numpy(xi, sbi, xj, sbj, pre, jac, info, G):
    dt, dp, dv = pre[0], pre[1:4], pre[8:11]
    dq = np.array([pre[7], pre[4], pre[5], pre[6]])
    ba0, bg0 = pre[11:14], pre[14:17]
    Qi, Qj = _q(xi), _q(xj)
    Ri_T = _R(_inv(Qi))
    dba, dbg = sbi[3:6] - ba0, sbi[6:9] - bg0
    cdq = _left(dq) @ np.concatenate([[1.0], 0.5 * jac[3:6, 12:15] @ dbg])
    cdv = dv + jac[6:9, 9:12] @ dba + jac[6:9, 12:15] @ dbg
    cdp = dp + jac[0:3, 9:12] @ dba + jac[0:3, 12:15] @ dbg
    a = Ri_T @ (0.5 * G * dt * dt + xj[:3] - xi[:3] - sbi[:3] * dt)
    b = Ri_T @ (G * dt + sbj[:3] - sbi[:3])
    e = _left(_inv(cdq)) @ (_left(_inv(Qi)) @ Qj)
    r = np.concatenate([a - cdp, 2.0 * e[1:], b - cdv, sbj[3:6] - sbi[3:6], sbj[6:9] - sbi[6:9]])
    J = np.zeros((15, 30))   # [pose_i(6) | sb_i(9) | pose_j(6) | sb_j(9)]
    J[0:3, 0:3], J[0:3, 3:6] = -Ri_T, _skew(a)
    J[3:6, 3:6] = -(_left(_left(_inv(Qj)) @ Qi) @ _right(cdq))[1:, 1:]
    J[6:9, 3:6] = _skew(b)
    J[0:3, 6:9], J[0:3, 9:12], J[0:3, 12:15] = -Ri_T * dt, -jac[0:3, 9:12], -jac[0:3, 12:15]
    J[3:6, 12:15] = -_left(_left(_left(_inv(Qj)) @ Qi) @ dq)[1:, 1:] @ jac[3:6, 12:15]
    J[6:9, 6:9], J[6:9, 9:12], J[6:9, 12:15] = -Ri_T, -jac[6:9, 9:12], -jac[6:9, 12:15]
    J[9:12, 9:12], J[12:15, 12:15] = -np.eye(3), -np.eye(3)
    J[0:3, 15:18] = Ri_T
    J[3:6, 18:21] = _left(_left(_left(_inv(cdq)) @ _inv(Qi)) @ Qj)[1:, 1:]
    J[6:9, 21:24], J[9:12, 24:27], J[12:15, 27:30] = Ri_T, np.eye(3), np.eye(3)
    return info @ r, info @ J, r


def _factors(pkg, W=3, seed=3, nonunit=0.0, realistic=False):
    batch = pkg.synth.make_windows(W, seed=seed, F=8)
    vi, extra = pkg.synth.make_inertial_factors(batch, seed=seed + 1, realistic=realistic)
    poses = batch.poses.copy()
    if nonunit:
        rng = np.random.default_rng(seed + 2)
        poses[..., 3:7] *= 1.0 + nonunit * rng.uniform(-1, 1, size=poses.shape[:-1] + (1,))
    return batch, poses, vi, extra


def _one(vi, poses, extra, k):
    w = vi.imu_window()[k]
    (i, j), (si, sj) = vi.imu_pose[k], vi.imu_sb[k]
    return (poses[w, i], extra[w, si:si + 9], poses[w, j], extra[w, sj:sj + 9], vi.imu_preint[k], vi.imu_jacobian[k],
            vi.imu_sqrt_info[k], vi.gravity)


@pytest.mark.parametrize("nonunit,realistic", [(0.0, False), (0.2, False), (0.2, True)])
def test_oracle_matches_numpy_restatement(pkg, nonunit, realistic):
    _, poses, vi, extra = _factors(pkg, nonunit=nonunit, realistic=realistic)
    for k in range(vi.NI):
        args = _one(vi, poses, extra, k)
        r, (jpi, jsi, jpj, jsj) = io.imu_factor_evaluate(*args)
        r2, J2, _ = imu_numpy(*[np.asarray(a, dtype=np.float64) for a in args])
        assert rel_err(r, r2) < 1e-12
        for got, ref in ((jpi[:, :6], J2[:, 0:6]), (jsi, J2[:, 6:15]), (jpj[:, :6], J2[:, 15:21]), (jsj, J2[:, 21:30])):
            assert rel_err(got, ref) < 1e-12


def test_structure(pkg):
    _, poses, vi, extra = _factors(pkg, nonunit=0.1)
    for k in range(vi.NI):
        args = list(_one(vi, poses, extra, k))
        args[6] = np.eye(15)   # unscaled Jacobians
        _, (jpi, jsi, jpj, jsj) = io.imu_factor_evaluate(*args)
        assert np.all(jpi[:, 6] == 0.0) and np.all(jpj[:, 6] == 0.0)
        for J, sign in ((jsi, -1.0), (jsj, 1.0)):   # bias rows: +-I on their own bias, 0 elsewhere
            assert np.array_equal(J[9:15, 3:9], sign * np.eye(6)) and np.all(J[9:15, 0:3] == 0.0)
        assert np.all(jpi[9:15] == 0.0) and np.all(jpj[9:15] == 0.0)


def _plus_pose(x, d):
    """ProjectionFactor::check convention: p + dp, (q * deltaQ(dtheta)).normalized()."""
    q = io.qmul(io.quat(x), (1.0, d[3] / 2, d[4] / 2, d[5] / 2))
    n = np.sqrt(sum(c * c for c in q))
    return np.array([x[0] + d[0], x[1] + d[1], x[2] + d[2], q[1] / n, q[2] / n, q[3] / n, q[0] / n])


def test_finite_differences(pkg):
    """Numeric Jacobians in the tangent space against the coded ones (unscaled: sqrt_info = I).  A sign or a transposition error
    is an O(1) discrepancy.  The rotation rows are first-order by design: the reference differentiates 2 vec(q) as if the
    residual rotation were the identity and takes dq/dbg with the uncorrected delta_q, so those rows carry an error of the order of
    the rotation residual plus |dq_dbg dbg| (both ~1e-3 here), and their bar is set from the state."""
    _, poses, vi, extra = _factors(pkg, W=2, seed=21)
    eps = 1e-6
    for k in range(vi.NI):
        xi, sbi, xj, sbj, pre, jac, _, G = _one(vi, poses, extra, k)
        I = np.eye(15)
        r0, (jpi, jsi, jpj, jsj) = io.imu_factor_evaluate(xi, sbi, xj, sbj, pre, jac, I, G)
        num = np.zeros((15, 30))
        for c in range(30):
            def f(s):
                d = np.zeros(9)
                if c < 6:
                    d[c] = s
                    return io.imu_factor_evaluate(_plus_pose(xi, d), sbi, xj, sbj, pre, jac, I, G, False)[0]
                if c < 15:
                    d[c - 6] = s
                    return io.imu_factor_evaluate(xi, sbi + d, xj, sbj, pre, jac, I, G, False)[0]
                if c < 21:
                    d[c - 15] = s
                    return io.imu_factor_evaluate(xi, sbi, _plus_pose(xj, d), sbj, pre, jac, I, G, False)[0]
                d[c - 21] = s
                return io.imu_factor_evaluate(xi, sbi, xj, sbj + d, pre, jac, I, G, False)[0]
            num[:, c] = (f(eps) - f(-eps)) / (2 * eps)
        ana = np.concatenate([jpi[:, :6], jsi, jpj[:, :6], jsj], axis=1)
        dbg = np.asarray(sbi[6:9]) - pre[14:17]
        rot_bar = 5.0 * (np.abs(r0[3:6]).max() + np.abs(jac[3:6, 12:15] @ dbg).max()) + 1e-6
        other = np.r_[0:3, 6:15]
        assert np.abs(num[other] - ana[other]).max() < 1e-6 * max(1.0, np.abs(ana[other]).max())
        assert np.abs(num[3:6] - ana[3:6]).max() < rot_bar
        assert rot_bar < 0.05   # the rotation rows are still checked far below the O(1) of a sign error


def test_struct_sizes_match_header(pkg):
    abi = pkg._abi
    assert C.sizeof(abi.InertialFactors) == 8 + 3 * 8 + 8 + 6 * 8 + 8 + 6 * 8
    assert C.sizeof(abi.InertialOut) == 6 * 8
    assert abi.InertialFactors.n_imu.offset == 32 and abi.InertialFactors.prior_n_max.offset == 88


def test_to_dense_order(pkg):
    """Per window the prior first, then the IMU factors in input order, with the documented column maps."""
    batch = pkg.synth.make_windows(3, seed=4, F=8)
    vi, extra = pkg.synth.make_inertial_factors(batch, seed=5, no_imu=(1,), no_prior=(2,))
    ev = io.inertial_evaluate(None, batch.poses, batch.ex_pose, extra, _no_prior(vi), want_jac=True)
    ev["prior_residual"] = np.zeros((vi.W, vi.n_max))
    d = vi.to_dense(ev)
    assert list(np.diff(d.window_offset)) == [1 + 10, 1, 10]
    D = batch.D
    assert list(d.factors[0][3][:6]) == list(range(6, 12)) and list(d.factors[0][3][-9:]) == list(range(D + 9, D + 18))
    assert sorted(d.factors[0][3]) == sorted(set(d.factors[0][3]))
    assert list(d.factors[1][3]) == list(vi.imu_columns(0))


def _no_prior(vi):
    """The same factors with every prior dropped (inertial_evaluate without the C++ oracle)."""
    import copy
    v = copy.copy(vi)
    v.prior_n = np.zeros_like(vi.prior_n)
    return v
