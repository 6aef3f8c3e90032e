"""ctypes mirror of include/viml.h (struct layouts, flags, error codes).

Shared by the product binding (this package) and by the test-only oracle binding (oracle/oracle.py), so
that both sides of a parity test are driven with the very same structs.
"""
import ctypes as C

import numpy as np

VIML_OK = 0
VIML_ERR_INVALID = -1
VIML_ERR_CUDA = -2
VIML_ERR_NO_DEVICE = -3
VIML_ERR_NOMAP = -4
VIML_ERR_UNSUPPORTED = -5

OUT_RESIDUAL_JACOBIAN = 0x01
OUT_HB = 0x02
OUT_SCHUR = 0x04
LOSS_CAUCHY = 0x10
S_PACKED = 0x20
PTRS_DEVICE = 0x100
FOV_CACHED = 0x200
FOV_SLOTS = 11
BLOCK_POSE, BLOCK_EX, BLOCK_EXTRA = 0, 1, 2
PRIOR_X0_STRIDE = 9
SOLVE_NO_CONVERGENCE, SOLVE_FUNCTION_TOL, SOLVE_PARAMETER_TOL, SOLVE_MIN_RADIUS, SOLVE_FAILURE = 0, 1, 2, 3, 4

c_double_p = C.POINTER(C.c_double)
c_float_p = C.POINTER(C.c_float)
c_int32_p = C.POINTER(C.c_int32)
c_uint32_p = C.POINTER(C.c_uint32)


class Config(C.Structure):
    """viml_config — estimator.cpp:54-124 fields read by the hot path."""

    _fields_ = [
        ("fx", C.c_double), ("fy", C.c_double), ("cx", C.c_double), ("cy", C.c_double),
        ("width", C.c_int32), ("height", C.c_int32),
        ("Rbw", C.c_double * 9), ("Tbw", C.c_double * 3),
        ("overlap_th", C.c_double), ("dist_th", C.c_double), ("angle_th", C.c_double),
        ("sqrt_info", C.c_double), ("cauchy_a", C.c_double),
    ]


class WindowBatch(C.Structure):
    _fields_ = [
        ("n_windows", C.c_int32), ("poses_per_window", C.c_int32),
        ("feats_per_window", C.c_int32), ("reserved0", C.c_int32),
        ("poses", C.c_void_p), ("ex_pose", C.c_void_p), ("inv_depth", C.c_void_p),
        ("n_point_factors", C.c_int64),
        ("pf_window_offset", C.c_void_p), ("pf_idx", C.c_void_p), ("pf_obs", C.c_void_p),
        ("pf_pts_i_z", C.c_void_p),
        ("n_line_factors", C.c_int64),
        ("lf_window_offset", C.c_void_p), ("lf_frame", C.c_void_p), ("lf_geom", C.c_void_p),
        ("feat_obs", C.c_void_p), ("pf_obs_j", C.c_void_p),
        ("feat_obs_f32", C.c_void_p), ("pf_obs_j_f32", C.c_void_p),
        ("lf_map_index", C.c_void_p), ("lf_seg2d_f32", C.c_void_p),
    ]


LIN_OUT_FIELDS = ("pf_residual", "pf_jac_pose_i", "pf_jac_pose_j", "pf_jac_ex", "pf_jac_feat",
                  "lf_residual", "lf_jac_pose", "H_pp", "H_lp", "H_ll", "b_p", "b_l", "S", "g")


class LinearizeOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in LIN_OUT_FIELDS]


class MargBatch(C.Structure):
    _fields_ = [("n_problems", C.c_int32), ("pos", C.c_int32), ("m", C.c_int32),
                ("reserved0", C.c_int32), ("eps", C.c_double), ("A", C.c_void_p), ("b", C.c_void_p)]


class MargOut(C.Structure):
    _fields_ = [("A_schur", C.c_void_p), ("b_schur", C.c_void_p),
                ("linearized_jacobians", C.c_void_p), ("linearized_residuals", C.c_void_p)]


class AssocQuery(C.Structure):
    _fields_ = [("n_poses", C.c_int32), ("lines_per_pose", C.c_int32),
                ("cull_poses", C.c_void_p), ("match_poses", C.c_void_p), ("ex_pose", C.c_void_p),
                ("lines2d", C.c_void_p), ("n_lines2d", C.c_void_p), ("cull_ex_pose", C.c_void_p), ("fov_slot", C.c_void_p)]


class AssocOut(C.Structure):
    _fields_ = [("match_index", C.c_void_p), ("err", C.c_void_p), ("projected", C.c_void_p),
                ("fov_count", C.c_void_p), ("fov_index", C.c_void_p),
                ("fov_capacity", C.c_int32), ("reserved0", C.c_int32), ("fov_mask", C.c_void_p)]


class DenseFactors(C.Structure):
    """viml_dense_factors — evaluated residual / Jacobian blocks of the prior and IMU factors (CSR over factors)."""

    _fields_ = [("extra_dim", C.c_int32), ("reserved0", C.c_int32), ("n_factors", C.c_int64),
                ("window_offset", C.c_void_p), ("row_offset", C.c_void_p), ("col_offset", C.c_void_p), ("jac_offset", C.c_void_p),
                ("col_index", C.c_void_p), ("residual", C.c_void_p), ("jacobian", C.c_void_p)]


class TriangulateIn(C.Structure):
    _fields_ = [("n_windows", C.c_int32), ("poses_per_window", C.c_int32), ("poses", C.c_void_p), ("ex_pose", C.c_void_p),
                ("n_features", C.c_int64), ("feat_window", C.c_void_p), ("start_frame", C.c_void_p), ("obs_offset", C.c_void_p),
                ("points", C.c_void_p)]


class ReducedOut(C.Structure):
    _fields_ = [("Sx", C.c_void_p), ("gx", C.c_void_p)]


class GnOptions(C.Structure):
    _fields_ = [("lambda_", C.c_double), ("reserved0", C.c_double)]


class GnOut(C.Structure):
    _fields_ = [("poses", C.c_void_p), ("ex_pose", C.c_void_p), ("inv_depth", C.c_void_p), ("extra", C.c_void_p),
                ("dx", C.c_void_p), ("cost", C.c_void_p), ("solved", C.c_void_p)]


class SolveOptions(C.Structure):
    """viml_solve_options — the trust-region loop of viml_solve_vi (Ceres' defaults in Context.solve_vi)."""

    _fields_ = [("max_iterations", C.c_int32), ("max_consecutive_invalid", C.c_int32), ("initial_radius", C.c_double),
                ("max_radius", C.c_double), ("min_radius", C.c_double), ("min_relative_decrease", C.c_double),
                ("function_tolerance", C.c_double), ("parameter_tolerance", C.c_double)]


SOLVE_OUT_FIELDS = ("poses", "ex_pose", "inv_depth", "extra", "status", "iterations", "accepted", "cost", "radius", "trace")


class SolveOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in SOLVE_OUT_FIELDS]


class Dense:
    """Host-side container of one viml_dense_factors: a list of (window, residual [n], jacobian [n, c], col_index [c]) tuples
    sorted by window."""

    def __init__(self, W, extra_dim, factors):
        self.W, self.X = W, int(extra_dim)
        factors = sorted(factors, key=lambda f: f[0])
        self.factors = factors
        cnt = np.bincount([f[0] for f in factors], minlength=W) if factors else np.zeros(W, dtype=np.int64)
        self.window_offset = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
        rows = [len(f[1]) for f in factors]
        cols = [len(f[3]) for f in factors]
        self.row_offset = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
        self.col_offset = np.concatenate([[0], np.cumsum(cols)]).astype(np.int64)
        self.jac_offset = np.concatenate([[0], np.cumsum([r * c for r, c in zip(rows, cols)])]).astype(np.int64)
        self.col_index = np.ascontiguousarray(np.concatenate([np.asarray(f[3]) for f in factors]) if factors else np.zeros(0), dtype=np.int32)
        self.residual = np.ascontiguousarray(np.concatenate([np.asarray(f[1], dtype=np.float64) for f in factors]) if factors else np.zeros(0))
        self.jacobian = np.ascontiguousarray(np.concatenate([np.asarray(f[2], dtype=np.float64).reshape(-1) for f in factors])
                                             if factors else np.zeros(0))

    def arrays(self):
        return {k: getattr(self, k) for k in ("window_offset", "row_offset", "col_offset", "jac_offset", "col_index", "residual", "jacobian")}

    def struct(self, arrays=None):
        a = self.arrays() if arrays is None else arrays
        s = DenseFactors()
        s.extra_dim, s.n_factors = self.X, len(self.factors)
        for k in a:
            setattr(s, k, ptr(a[k]))
        return s


class InertialFactors(C.Structure):
    """viml_inertial_factors — the window's IMU factors (pre-integration outputs) and the prior of the last marginalisation."""

    _fields_ = [("extra_dim", C.c_int32), ("reserved0", C.c_int32), ("gravity", C.c_double * 3), ("n_imu", C.c_int64),
                ("imu_window_offset", C.c_void_p), ("imu_pose", C.c_void_p), ("imu_sb", C.c_void_p), ("imu_preint", C.c_void_p),
                ("imu_jacobian", C.c_void_p), ("imu_sqrt_info", C.c_void_p),
                ("prior_n_max", C.c_int32), ("prior_max_blocks", C.c_int32), ("prior_n", C.c_void_p), ("prior_jacobian", C.c_void_p),
                ("prior_residual", C.c_void_p), ("prior_n_blocks", C.c_void_p), ("prior_block", C.c_void_p), ("prior_x0", C.c_void_p)]


INERTIAL_OUT_FIELDS = ("imu_residual", "imu_jac_pose_i", "imu_jac_sb_i", "imu_jac_pose_j", "imu_jac_sb_j", "prior_residual")


class InertialOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in INERTIAL_OUT_FIELDS]


class Inertial:
    """Host-side container of one viml_inertial_factors (numpy arrays, shapes as in viml.h).

    imu_preint rows are [sum_dt, delta_p(3), delta_q(4, x y z w), delta_v(3), linearized_ba(3), linearized_bg(3)]; imu_jacobian and
    imu_sqrt_info are row-major 15 x 15.  prior_block rows are [kind, index, size, first column]."""

    INT_FIELDS = ("imu_window_offset", "imu_pose", "imu_sb", "prior_n", "prior_n_blocks", "prior_block")
    FIELDS = ("imu_window_offset", "imu_pose", "imu_sb", "imu_preint", "imu_jacobian", "imu_sqrt_info",
              "prior_n", "prior_jacobian", "prior_residual", "prior_n_blocks", "prior_block", "prior_x0")

    def __init__(self, W, P, extra_dim, gravity, imu_window_offset, imu_pose, imu_sb, imu_preint, imu_jacobian, imu_sqrt_info,
                 prior_n, prior_jacobian, prior_residual, prior_n_blocks, prior_block, prior_x0):
        self.W, self.P, self.X = int(W), int(P), int(extra_dim)
        self.gravity = np.asarray(gravity, dtype=np.float64).reshape(3)
        loc = dict(locals())
        for k in self.FIELDS:
            setattr(self, k, np.ascontiguousarray(loc[k], dtype=np.int32 if k in self.INT_FIELDS else np.float64))
        self.imu_pose = self.imu_pose.reshape(-1, 2)
        self.imu_sb = self.imu_sb.reshape(-1, 2)
        self.imu_preint = self.imu_preint.reshape(-1, 17)
        self.imu_jacobian = self.imu_jacobian.reshape(-1, 15, 15)
        self.imu_sqrt_info = self.imu_sqrt_info.reshape(-1, 15, 15)
        n_max = self.prior_jacobian.shape[1] if self.prior_jacobian.ndim == 3 else 0
        self.prior_jacobian = self.prior_jacobian.reshape(self.W, n_max, n_max)
        self.prior_residual = self.prior_residual.reshape(self.W, n_max)
        self.prior_block = self.prior_block.reshape(self.W, -1, 4)
        self.prior_x0 = self.prior_x0.reshape(self.W, -1, PRIOR_X0_STRIDE)
        assert self.imu_window_offset.shape == (self.W + 1,) and self.prior_n.shape == (self.W,)

    NI = property(lambda s: int(s.imu_pose.shape[0]))
    n_max = property(lambda s: int(s.prior_jacobian.shape[1]))
    max_blocks = property(lambda s: int(s.prior_block.shape[1]))
    D = property(lambda s: 6 * (s.P + 1))

    def arrays(self):
        return {k: getattr(self, k) for k in self.FIELDS}

    def struct(self, arrays=None):
        a = self.arrays() if arrays is None else arrays
        s = InertialFactors()
        s.extra_dim, s.n_imu = self.X, self.NI
        for k in range(3):
            s.gravity[k] = float(self.gravity[k])
        s.prior_n_max, s.prior_max_blocks = self.n_max, self.max_blocks
        for k in self.FIELDS:
            setattr(s, k, ptr(a[k]))
        return s

    def imu_window(self):
        return np.repeat(np.arange(self.W), np.diff(self.imu_window_offset))

    def imu_columns(self, k):
        """Tangent columns of IMU factor k's reduced 15 x 30 block: [pose_i(6) | sb_i(9) | pose_j(6) | sb_j(9)]."""
        (i, j), (si, sj) = self.imu_pose[k], self.imu_sb[k]
        D = self.D
        return np.concatenate([6 * i + np.arange(6), D + si + np.arange(9), 6 * j + np.arange(6), D + sj + np.arange(9)])

    def prior_columns(self, w):
        """Tangent column of each of the n_w local columns of window w's prior."""
        n = int(self.prior_n[w])
        cols = np.full(n, -1, dtype=np.int64)
        for kind, idx, size, first in self.prior_block[w, :self.prior_n_blocks[w]]:
            local = 6 if size == 7 else size
            t0 = 6 * idx if kind == BLOCK_POSE else 6 * self.P if kind == BLOCK_EX else self.D + idx
            cols[first:first + local] = t0 + np.arange(local)
        return cols

    def to_dense(self, ev):
        """The viml_dense_factors of an evaluation (dict of the viml_inertial_out arrays): per window the prior, then its IMU factors
        in input order — the order viml_gn_step_vi assembles them in."""
        fs = []
        win = self.imu_window()
        for w in range(self.W):
            n = int(self.prior_n[w])
            if n > 0:
                fs.append((w, ev["prior_residual"][w, :n], self.prior_jacobian[w, :n, :n], self.prior_columns(w)))
            for k in range(self.imu_window_offset[w], self.imu_window_offset[w + 1]):
                J = np.concatenate([ev["imu_jac_pose_i"][k][:, :6], ev["imu_jac_sb_i"][k], ev["imu_jac_pose_j"][k][:, :6],
                                    ev["imu_jac_sb_j"][k]], axis=1)
                fs.append((w, ev["imu_residual"][k], J, self.imu_columns(k)))
        assert all(f[0] == w for f, w in zip(fs, sorted(f[0] for f in fs)))
        return Dense(self.W, self.X, fs)


def ptr(a):
    """Address of a numpy array (host) or an int device pointer; None -> NULL."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return int(a)
    if hasattr(a, "data_ptr"):  # torch tensor (host pinned or device)
        return int(a.data_ptr())
    assert a.flags["C_CONTIGUOUS"], "ABI buffers must be C-contiguous"
    return a.ctypes.data


def make_config(fx=461.6, fy=460.3, cx=363.0, cy=248.1, width=752, height=480, Rbw=None, Tbw=None,
                overlap_th=0.45, dist_th=50.0, angle_th=0.1745, sqrt_info=460.0 / 1.5, cauchy_a=1.0):
    """Defaults are EuRoC cam0 and the thresholds of benchmark_publisher/config/V1_01_easy/sensor.yaml."""
    cfg = Config()
    cfg.fx, cfg.fy, cfg.cx, cfg.cy = fx, fy, cx, cy
    cfg.width, cfg.height = width, height
    R = np.eye(3) if Rbw is None else np.asarray(Rbw, dtype=np.float64).reshape(3, 3)
    T = np.zeros(3) if Tbw is None else np.asarray(Tbw, dtype=np.float64).reshape(3)
    for k in range(9):
        cfg.Rbw[k] = float(R.reshape(-1)[k])
    for k in range(3):
        cfg.Tbw[k] = float(T[k])
    cfg.overlap_th, cfg.dist_th, cfg.angle_th = overlap_th, dist_th, angle_th
    cfg.sqrt_info, cfg.cauchy_a = sqrt_info, cauchy_a
    return cfg


class Batch:
    """Host-side container of one viml_window_batch (numpy arrays, SoA as in viml.h)."""

    def __init__(self, poses, ex_pose, inv_depth, pf_window_offset, pf_idx, pf_obs,
                 lf_window_offset=None, lf_frame=None, lf_geom=None, pf_pts_i_z=None, lf_seg2d=None, lf_map_index=None):
        self.poses = np.ascontiguousarray(poses, dtype=np.float64)
        self.ex_pose = np.ascontiguousarray(ex_pose, dtype=np.float64)
        self.inv_depth = np.ascontiguousarray(inv_depth, dtype=np.float64)
        self.pf_window_offset = np.ascontiguousarray(pf_window_offset, dtype=np.int32)
        self.pf_idx = np.ascontiguousarray(pf_idx, dtype=np.uint32)
        self.pf_obs = np.ascontiguousarray(pf_obs, dtype=np.float64).reshape(-1, 4)
        self.pf_pts_i_z = None if pf_pts_i_z is None else np.ascontiguousarray(pf_pts_i_z, dtype=np.float64)
        W = self.poses.shape[0]
        if lf_window_offset is None:
            lf_window_offset = np.zeros(W + 1, dtype=np.int32)
            lf_frame = np.zeros(0, dtype=np.int32)
            lf_geom = np.zeros((9, 0), dtype=np.float64)
        self.lf_window_offset = np.ascontiguousarray(lf_window_offset, dtype=np.int32)
        self.lf_frame = np.ascontiguousarray(lf_frame, dtype=np.int32)
        self.lf_geom = np.ascontiguousarray(lf_geom, dtype=np.float64).reshape(9, -1)
        # optional line-table form of lf_geom (viml.h): the detected 2D segments as float32 and the map line of every factor
        self.lf_seg2d = None if lf_seg2d is None else np.ascontiguousarray(lf_seg2d, dtype=np.float32).reshape(-1, 4)
        self.lf_map_index = None if lf_map_index is None else np.ascontiguousarray(lf_map_index, dtype=np.int32)
        assert self.poses.ndim == 3 and self.poses.shape[2] == 7
        assert self.ex_pose.shape == (W, 7) and self.inv_depth.shape[0] == W
        assert self.pf_window_offset.shape == (W + 1,) and self.lf_window_offset.shape == (W + 1,)

    W = property(lambda s: s.poses.shape[0])
    P = property(lambda s: s.poses.shape[1])
    F = property(lambda s: s.inv_depth.shape[1])
    D = property(lambda s: 6 * (s.poses.shape[1] + 1))
    NP = property(lambda s: int(s.pf_idx.shape[0]))
    NL = property(lambda s: int(s.lf_frame.shape[0]))

    def arrays(self):
        return {k: getattr(self, k) for k in ("poses", "ex_pose", "inv_depth", "pf_window_offset", "pf_idx",
                                              "pf_obs", "pf_pts_i_z", "lf_window_offset", "lf_frame", "lf_geom")}

    def struct(self, arrays=None):
        a = self.arrays() if arrays is None else arrays
        s = WindowBatch()
        s.n_windows, s.poses_per_window, s.feats_per_window = self.W, self.P, self.F
        s.poses, s.ex_pose, s.inv_depth = ptr(a["poses"]), ptr(a["ex_pose"]), ptr(a["inv_depth"])
        s.n_point_factors = self.NP
        s.pf_window_offset, s.pf_idx, s.pf_obs = ptr(a["pf_window_offset"]), ptr(a["pf_idx"]), ptr(a.get("pf_obs"))
        if a.get("pf_obs") is None:   # observation table instead of per-factor pairs (viml.h, viml_window_batch)
            if a.get("feat_obs_f32") is not None:
                s.feat_obs_f32, s.pf_obs_j_f32 = ptr(a["feat_obs_f32"]), ptr(a["pf_obs_j_f32"])
            else:
                s.feat_obs, s.pf_obs_j = ptr(a["feat_obs"]), ptr(a["pf_obs_j"])
        s.pf_pts_i_z = ptr(a.get("pf_pts_i_z"))
        s.n_line_factors = self.NL
        s.lf_window_offset, s.lf_frame, s.lf_geom = ptr(a["lf_window_offset"]), ptr(a["lf_frame"]), ptr(a.get("lf_geom"))
        if a.get("lf_geom") is None and self.NL > 0:   # line table instead of the nine geometry planes
            s.lf_map_index, s.lf_seg2d_f32 = ptr(a["lf_map_index"]), ptr(a["lf_seg2d_f32"])
        return s

    def obs_table(self, f32=False):
        """The observation-table form of pf_obs: (feat_obs [W][F][2], pf_obs_j [NP][2]).  Raises when the factors of a feature
        do not share pts_i (then only the per-factor form describes the batch).  f32=True: as float32 arrays, for observations
        that are float32 values (raises when they are not)."""
        W, F = self.W, self.F
        win = np.repeat(np.arange(W, dtype=np.int64), np.diff(self.pf_window_offset))
        key = win * F + (self.pf_idx >> 16).astype(np.int64)
        feat_obs = np.zeros((W * F, 2))
        feat_obs[key] = self.pf_obs[:, :2]          # one of the factors' pts_i per feature ...
        if not np.array_equal(feat_obs[key], self.pf_obs[:, :2]):   # ... which every other factor must repeat
            raise ValueError("pts_i differs between the factors of a feature")
        feat_obs, obs_j = feat_obs.reshape(W, F, 2), np.ascontiguousarray(self.pf_obs[:, 2:])
        if f32:
            f32s = feat_obs.astype(np.float32), obs_j.astype(np.float32)
            if not (np.array_equal(f32s[0].astype(np.float64), feat_obs) and np.array_equal(f32s[1].astype(np.float64), obs_j)):
                raise ValueError("observations are not float32 values")
            return f32s
        return feat_obs, obs_j

    def out_shapes(self):
        W, F, D, NP, NL = self.W, self.F, self.D, self.NP, self.NL
        return {"pf_residual": (NP, 2), "pf_jac_pose_i": (NP, 14), "pf_jac_pose_j": (NP, 14),
                "pf_jac_ex": (NP, 14), "pf_jac_feat": (NP, 2), "lf_residual": (NL, 2), "lf_jac_pose": (NL, 14),
                "H_pp": (W, D, D), "H_lp": (W, F, D), "H_ll": (W, F), "b_p": (W, D), "b_l": (W, F),
                "S": (W, D, D), "g": (W, D), "S_packed": (W, D * (D + 1) // 2)}

    def alloc_out(self, flags, fill=np.nan):
        """numpy output buffers for the requested modes, NaN-filled so unwritten entries are caught."""
        sh = self.out_shapes()
        names = []
        if flags & OUT_RESIDUAL_JACOBIAN:
            names += ["pf_residual", "pf_jac_pose_i", "pf_jac_pose_j", "pf_jac_ex", "pf_jac_feat",
                      "lf_residual", "lf_jac_pose"]
        if flags & OUT_HB:
            names += ["H_pp", "H_lp", "H_ll", "b_p", "b_l"]
        if flags & OUT_SCHUR:
            names += ["S", "g"]
        return {n: np.full(sh[n], fill, dtype=np.float64) for n in names}

    def slice_windows(self, lo, hi):
        """Sub-batch of windows [lo, hi) (used to shard windows over ranks)."""
        p0, p1 = int(self.pf_window_offset[lo]), int(self.pf_window_offset[hi])
        l0, l1 = int(self.lf_window_offset[lo]), int(self.lf_window_offset[hi])
        return Batch(self.poses[lo:hi], self.ex_pose[lo:hi], self.inv_depth[lo:hi],
                     self.pf_window_offset[lo:hi + 1] - p0, self.pf_idx[p0:p1], self.pf_obs[p0:p1],
                     self.lf_window_offset[lo:hi + 1] - l0, self.lf_frame[l0:l1], self.lf_geom[:, l0:l1],
                     None if self.pf_pts_i_z is None else self.pf_pts_i_z[p0:p1],
                     None if self.lf_seg2d is None else self.lf_seg2d[l0:l1],
                     None if self.lf_map_index is None else self.lf_map_index[l0:l1])


def out_struct(bufs):
    o = LinearizeOut()
    for n in LIN_OUT_FIELDS:
        setattr(o, n, ptr(bufs.get(n)))
    if bufs.get("S") is None and bufs.get("S_packed") is not None:   # VIML_S_PACKED: the S pointer receives the upper triangle
        o.S = ptr(bufs["S_packed"])
    return o


def unpack_upper(Sp, D):
    """[W, D(D+1)/2] upper triangles (VIML_S_PACKED) -> full symmetric [W, D, D]."""
    W = Sp.shape[0]
    S = np.zeros((W, D, D))
    iu = np.triu_indices(D)
    S[:, iu[0], iu[1]] = Sp
    S[:, iu[1], iu[0]] = Sp
    return S
