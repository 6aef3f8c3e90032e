"""The oracle against the REFERENCE'S OWN CODE (CPU tests).

oracle/_ref/libref.so is /root/reference/vins_estimator/src/factor/{projection_factor, line_projection_factor,
pose_local_parameterization, marginalization_factor}.cpp and feature_manager.cpp compiled unmodified where they lie (oracle/Makefile
`ref`), plus the four association functions of estimator.cpp (UpdateLinesInFoV, CalAngleDist, CalEulerDist,
LineCorrespondenceInFrame) cut out of that file at build time (oracle/ref_slice.py, oracle/ref_estimator.cpp), against the
Eigen / Ceres / ROS interface stand-ins of oracle/ref_shim/.  tests/golden/ref_factors.npz and ref_assoc.npz hold vectors that
library produced (tests/golden/make_ref_golden.py), so the pin also holds where the reference tree is absent."""
import os

import numpy as np
import pytest

from conftest import ROOT

GOLD = os.path.join(ROOT, "tests", "golden", "ref_factors.npz")


def _oracle_factors(pkg, orc, g):
    abi, synth = pkg._abi, pkg.synth
    cfg = synth.euroc_config(sqrt_info=float(g["pf_sqrt_info"]))
    W = g["pf_poses"].shape[0]
    off = np.searchsorted(g["pf_win"], np.arange(W + 1)).astype(np.int32)
    b = abi.Batch(g["pf_poses"], g["pf_ex"], g["pf_inv_depth"], off, g["pf_idx"], g["pf_obs"])
    op = orc.linearize_batch(cfg, b, abi.OUT_RESIDUAL_JACOBIAN)
    loff = np.searchsorted(g["lf_win"], np.arange(W + 1)).astype(np.int32)
    bl = abi.Batch(g["lf_poses"], g["lf_ex"], np.zeros((W, 1)), np.zeros(W + 1, dtype=np.int32), np.zeros(0, dtype=np.uint32),
                   np.zeros((0, 4)), loff, g["lf_frame"], g["lf_geom"])
    ol = orc.linearize_batch(cfg, bl, abi.OUT_RESIDUAL_JACOBIAN)
    return op, ol


def test_oracle_equals_reference_vectors_bit_for_bit(pkg, orc):
    """ProjectionFactor::Evaluate and LineProjectionFactor::Evaluate: the oracle restatement reproduces the reference's own code
    bit for bit on 1669 + 330 factors (window 1 has clearly non-unit quaternions)."""
    g = np.load(GOLD)
    op, ol = _oracle_factors(pkg, orc, g)
    N, NL = len(g["pf_idx"]), len(g["lf_frame"])
    for k, rk in (("pf_residual", "pf_r"), ("pf_jac_pose_i", "pf_Ji"), ("pf_jac_pose_j", "pf_Jj"), ("pf_jac_ex", "pf_Je"), ("pf_jac_feat", "pf_Jl")):
        assert np.array_equal(op[k].reshape(N, -1), g[rk].reshape(N, -1)), k
    for k, rk in (("lf_residual", "lf_r"), ("lf_jac_pose", "lf_J")):
        assert np.array_equal(ol[k].reshape(NL, -1), g[rk].reshape(NL, -1)), k


def test_pose_plus_equals_reference(pkg, orc):
    from oracle import gn_oracle
    g = np.load(GOLD)
    for x, d, o in zip(g["plus_x"], g["plus_d"], g["plus_out"]):
        assert np.abs(gn_oracle.pose_plus(x, d) - o).max() < 1e-15


def _oracle_marginalize(pkg, orc, poses, ex, dep, idx, obs, sq, loss):
    """The oracle's route to the same quantity: dense A, b by the ThreadsConstructA rule, [pose 0, landmarks | kept] ordering,
    marginalize_dense (eigen pseudo-inverse Schur complement)."""
    abi, synth = pkg._abi, pkg.synth
    cfg = synth.euroc_config(sqrt_info=sq, cauchy_a=(loss or 1.0))
    P, F = poses.shape[0], len(dep)
    b = abi.Batch(poses[None], ex[None], dep[None], np.array([0, len(idx)], dtype=np.int32), idx, obs)
    flags = abi.OUT_HB | (abi.LOSS_CAUCHY if loss else 0)
    A, bb = orc.window_dense(cfg, b, 0, flags)
    D = b.D
    perm = np.concatenate([np.arange(6), D + np.arange(F), np.arange(6, D)])
    A, bb = A[np.ix_(perm, perm)], bb[perm]
    As, bs, _, _ = orc.marginalize_dense(A, bb, 6 + F)
    return As, bs


def _check_marg(pkg, A, b, As, bs):
    n = A.shape[0]
    assert As.shape == (n, n)
    # per 6x6 block against the block's own scale
    assert pkg.parity.unit_err("S", As[None], A[None]) < 1e-8, pkg.parity.unit_err("S", As[None], A[None])
    assert pkg.parity.unit_err("g", bs[None], b[None]) < 1e-8


def test_marginalization_equals_reference_vectors(pkg, orc):
    """MarginalizationInfo::{addResidualBlockInfo, preMarginalize, marginalize} of the reference (pthread ThreadsConstructA, eigen
    pseudo-inverse, square-root factorisation) on the MARGIN_OLD projection set: J^T J and J^T r of its linearized_jacobians /
    linearized_residuals against the oracle's dense route.  (1e-8: two eigen-decompositions on each side.)"""
    g = np.load(GOLD)
    sq = float(g["pf_sqrt_info"])
    for w in range(2):
        k0, k1 = g["marg_off"][w], g["marg_off"][w + 1]
        for loss, tag in ((None, "noloss"), (1.0, "cauchy")):
            As, bs = _oracle_marginalize(pkg, orc, g["marg_poses"][w], g["marg_ex"][w], g["marg_inv_depth"][w], g["marg_idx"][k0:k1],
                                         g["marg_obs"][k0:k1], sq, loss)
            _check_marg(pkg, g[f"marg{w}_{tag}_A"], g[f"marg{w}_{tag}_b"], As, bs)


def test_line2d_and_point2flined_equal_reference_vectors(pkg, orc):
    """Line2D::Line2D(Vector4d) and Line2D::Point2Flined (feature_manager.cpp:4-15, :46-71), the building blocks of
    CalAngleDist / CalEulerDist: bit for bit, vertical segments included."""
    import ctypes as C
    g = np.load(GOLD)
    o = orc.lib()
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))   # noqa: E731
    for seg, p, want, foot in zip(g["l2d_seg"], g["l2d_p"], g["l2d_out"], g["l2d_foot"]):
        seg, p = np.ascontiguousarray(seg), np.ascontiguousarray(p)
        a, f = np.zeros(7), np.zeros(2)
        o.orc_line2d(dp(seg), dp(a))
        o.orc_point2flined(dp(seg), dp(p), dp(f))
        assert np.array_equal(a, want) and np.array_equal(f, foot, equal_nan=True)


def test_triangulate_reference_vectors_vs_numpy_svd(pkg):
    """FeatureManager::triangulate of the reference (its JacobiSVD is the stand-in's) against numpy's LAPACK SVD on the same DLT
    rows: the check that the -m gpu test of viml_triangulate_batch uses a sound expectation."""
    g = np.load(GOLD)
    synth = pkg.synth

    def rot(q7):
        return synth._rot_from_quat(q7[3:7] / np.linalg.norm(q7[3:7]))

    poses, ex = g["tri_poses"], g["tri_ex"]
    ric, tic = rot(ex), ex[:3]
    for l in range(len(g["tri_start"])):
        i = int(g["tri_start"][l])
        obs = g["tri_pts"][g["tri_off"][l]:g["tri_off"][l + 1]]
        R0, t0 = rot(poses[i]) @ ric, poses[i, :3] + rot(poses[i]) @ tic
        rows = []
        for k, p in enumerate(obs):
            R1, t1 = rot(poses[i + k]) @ ric, poses[i + k, :3] + rot(poses[i + k]) @ tic
            t, R = R0.T @ (t1 - t0), R0.T @ R1
            Pm = np.concatenate([R.T, (-R.T @ t)[:, None]], 1)
            f = p / np.linalg.norm(p)
            rows += [f[0] * Pm[2] - f[2] * Pm[0], f[1] * Pm[2] - f[2] * Pm[1]]
        V = np.linalg.svd(np.array(rows))[2][-1]
        d = V[2] / V[3]
        d = 5.0 if d < 0.1 else d
        assert abs(d - g["tri_depth"][l]) <= 1e-7 * abs(d), (l, d, g["tri_depth"][l])


def test_live_reference_library(pkg, orc):
    """Where oracle/_ref/libref.so exists (this container; prebuilt on the GPU box): fresh random inputs, not the committed ones."""
    from oracle import ref
    if not ref.available():
        pytest.skip("oracle/_ref/libref.so not built (reference tree absent)")
    synth = pkg.synth
    rng = np.random.default_rng(99)
    b = synth.make_windows(2, seed=777)
    sq = 123.0
    for k in rng.choice(b.NP, 200, replace=False):
        w = int(np.searchsorted(b.pf_window_offset, k, side="right") - 1)
        i, j, l = int(b.pf_idx[k] & 0xff), int((b.pf_idx[k] >> 8) & 0xff), int(b.pf_idx[k] >> 16)
        pi, pj = [b.pf_obs[k, 0], b.pf_obs[k, 1], 1.0], [b.pf_obs[k, 2], b.pf_obs[k, 3], 1.0]
        r1, J1 = ref.projection_evaluate(pi, pj, sq, b.poses[w, i], b.poses[w, j], b.ex_pose[w], b.inv_depth[w, l])
        r2, J2 = orc.projection_evaluate(pi, pj, sq, b.poses[w, i], b.poses[w, j], b.ex_pose[w], b.inv_depth[w, l])
        assert np.array_equal(r1, r2)
        for a, c in zip(J1, J2):
            assert np.array_equal(a.reshape(-1), np.asarray(c).reshape(-1))
    m = synth.make_windows(1, seed=778, P=5, F=25, all_start_zero=True, lines_per_frame=0)
    idx = m.pf_idx
    A, bb, mm = ref.marginalize_old(m.poses[0], m.ex_pose[0], m.inv_depth[0], (idx >> 8) & 0xff, idx >> 16, m.pf_obs, sq, 1.0)
    assert mm == 6 + 25
    As, bs = _oracle_marginalize(pkg, orc, m.poses[0], m.ex_pose[0], m.inv_depth[0], idx, m.pf_obs, sq, 1.0)
    _check_marg(pkg, A, bb, As, bs)


ASSOC_KEYS = ("match_index", "err", "projected", "fov_count", "fov_index")


def _same(a, b, k):
    if a.dtype.kind == "f":
        assert np.array_equal(a, b, equal_nan=True), k
    else:
        assert np.array_equal(a, b), k


def test_association_oracle_equals_reference_vectors(pkg, orc):
    """tests/golden/ref_assoc.npz: outputs of the reference's own UpdateLinesInFoV + LineCorrespondenceInFrame (+ CalAngleDist,
    CalEulerDist, Line2D, Point2Flined) on threshold-hugging queries; the oracle reproduces them bit for bit — FoV lists,
    chosen map index, errA / errD / overlap as float32, projected segment."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_assoc.npz"))
    for c in range(int(g["n_cases"])):
        cfg = pkg.synth.euroc_config(angle_th=float(g[f"c{c}_angle_th"]), overlap_th=float(g[f"c{c}_overlap_th"]))
        cex = g[f"c{c}_cull_ex"] if f"c{c}_cull_ex" in g.files else None
        nl = g[f"c{c}_n_lines2d"] if f"c{c}_n_lines2d" in g.files else None
        res = orc.line_associate(cfg, g["lines"], g[f"c{c}_cull"], g[f"c{c}_match"], g[f"c{c}_ex"], g[f"c{c}_lines2d"],
                                 n_lines2d=nl, fov_capacity=int(g[f"c{c}_fov_capacity"]), nthreads=4, cull_ex_pose=cex)
        L = g[f"c{c}_lines2d"].shape[1]
        for k in ASSOC_KEYS:
            a, b = res[k], g[f"c{c}_{k}"]
            if nl is not None and k in ("match_index", "err", "projected"):   # rows beyond a pose's own count are not outputs
                valid = np.arange(L)[None, :] < nl[:, None]
                a, b = a[valid], b[valid]
            _same(a, b, (c, k))
        assert float(g[f"c{c}_overlap_th"]) >= 1.0 or (g[f"c{c}_match_index"] >= 0).mean() > 0.2


@pytest.mark.parametrize("name", ["assoc_euroc_v1.npz", "assoc_euroc_v2.npz"])
def test_association_golden_on_reference_maps_equals_reference_functions(pkg, orc, name):
    """The committed association fixtures on the reference's real EuRoC line maps were written by the oracle; the reference's own
    functions give the same lists, indices, errors and projected segments, bit for bit.  The fixture therefore is the reference's
    output: where oracle/_ref/libref.so is not built, the oracle is held to it on every key (lists, indices, all three errors and
    every projected segment, at the fixture's list capacity)."""
    from oracle import ref
    impl = ref if ref.available() else orc
    g = np.load(os.path.join(ROOT, "tests", "golden", name))
    c = g["cfg"]
    cfg = pkg._abi.make_config(fx=c[0], fy=c[1], cx=c[2], cy=c[3], width=int(c[4]), height=int(c[5]), Rbw=g["Rbw"], Tbw=g["Tbw"],
                               overlap_th=c[6], dist_th=c[7], angle_th=c[8])
    res = impl.line_associate(cfg, g["lines"], g["cull"], g["match"], g["ex"], g["lines2d"], fov_capacity=g["fov_index"].shape[1], nthreads=8)
    for k in ASSOC_KEYS:
        _same(res[k], g[k], k)


def test_live_reference_association(pkg, orc):
    """Fresh random queries through both: drifting match poses, a frame-entry extrinsic that differs from the current one, ragged
    line counts, duplicated map lines (distance ties are decided by list order)."""
    from oracle import ref
    if not ref.available():
        pytest.skip("oracle/_ref/libref.so not built (reference tree absent)")
    synth = pkg.synth
    ext = (150.0, 150.0, 20.0)
    lines = synth.make_line_map(5000, seed=31, extent=ext)
    lines = np.concatenate([lines, lines[:300]])
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 6, L=80, n_true=40, seed=32, extent=ext, pose_drift=True)
    rng = np.random.default_rng(33)
    cex = ex.copy()
    cex[:, :3] += 0.01 * rng.standard_normal((len(ex), 3))
    nl = rng.integers(0, 81, len(ex)).astype(np.int32)
    for ang, ov in ((0.1745, 0.45), (0.3, 0.0), (3.2, 0.45)):
        cfg = synth.euroc_config(angle_th=ang, overlap_th=ov)
        a = orc.line_associate(cfg, lines, cull, match, ex, l2d, n_lines2d=nl, fov_capacity=4000, nthreads=8, cull_ex_pose=cex)
        b = ref.line_associate(cfg, lines, cull, match, ex, l2d, n_lines2d=nl, fov_capacity=4000, nthreads=8, cull_ex_pose=cex)
        valid = np.arange(80)[None, :] < nl[:, None]
        for k in ASSOC_KEYS:
            if k in ("match_index", "err", "projected"):
                _same(a[k][valid], b[k][valid], (ang, k))
            else:
                _same(a[k], b[k], (ang, k))
