"""tc-viml_b200 — B200-native linearisation hot path of TC-VIML.

The product is the C-ABI library csrc/ -> libviml_b200.so (hand-written sm_100a CUDA) plus the C++ host
shim under host/ that keeps the reference's class interfaces.  This Python module is only a thin ctypes
binding of the C-ABI for tests and bench.py.  There is no CPU fallback: if the library is missing or no
CUDA device is usable, construction fails loudly.
"""
import ctypes as C
import os

import numpy as np

from . import _abi, build, parity, shard, synth  # noqa: F401
from ._abi import (LOSS_CAUCHY, OUT_HB, OUT_RESIDUAL_JACOBIAN, OUT_SCHUR, PTRS_DEVICE, S_PACKED, Batch,  # noqa: F401
                   make_config)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VIML_LIB_PATH") or os.path.join(_HERE, "libviml_b200.so")   # override: A/B runs of kernel variants
_LIB = None

# every symbol include/viml.h declares
ABI_SYMBOLS = (
    "viml_abi_version", "viml_create", "viml_destroy", "viml_last_error", "viml_sync", "viml_stream",
    "viml_host_alloc", "viml_host_free", "viml_device_alloc", "viml_device_free", "viml_memcpy_h2d",
    "viml_memcpy_d2h", "viml_kernel_launches", "viml_profile_begin", "viml_profile_end", "viml_kernel_name",
    "viml_microbench_fp64", "viml_microbench_dmma", "viml_selftest_division", "viml_set_map", "viml_linearize_batch",
    "viml_marginalize_batch", "viml_line_associate", "viml_assoc_stats", "viml_allreduce_hb",
    "viml_load_line_map", "viml_reduced_system", "viml_reduced_from_schur", "viml_gn_step",
    "viml_fov_update", "viml_fov_slide", "viml_track_gate", "viml_triangulate_batch",
    "viml_inertial_evaluate", "viml_gn_step_vi", "viml_solve_vi",
)


class VimlError(RuntimeError):
    pass


def load_library():
    """dlopen libviml_b200.so and check every ABI symbol.  Works without a GPU (no device call)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise VimlError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (build()) first; "
                        "there is no CPU fallback for the hot path")
    lib = C.CDLL(LIB_PATH)
    for s in ABI_SYMBOLS:
        if not hasattr(lib, s):
            raise VimlError(f"libviml_b200.so does not export {s}")
    lib.viml_last_error.restype = C.c_char_p
    lib.viml_last_error.argtypes = [C.c_void_p]
    lib.viml_stream.restype = C.c_void_p
    lib.viml_stream.argtypes = [C.c_void_p]
    lib.viml_kernel_launches.restype = C.c_int64
    lib.viml_kernel_launches.argtypes = [C.c_void_p]
    lib.viml_kernel_name.restype = C.c_char_p
    lib.viml_kernel_name.argtypes = [C.c_int]
    lib.viml_profile_begin.argtypes = [C.c_void_p]
    lib.viml_profile_end.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]
    lib.viml_microbench_fp64.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.viml_microbench_dmma.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    lib.viml_selftest_division.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    lib.viml_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(_abi.Config), C.c_int]
    lib.viml_destroy.argtypes = [C.c_void_p]
    lib.viml_sync.argtypes = [C.c_void_p]
    lib.viml_set_map.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    lib.viml_linearize_batch.argtypes = [C.c_void_p, C.POINTER(_abi.WindowBatch), C.POINTER(_abi.LinearizeOut), C.c_uint32]
    lib.viml_marginalize_batch.argtypes = [C.c_void_p, C.POINTER(_abi.MargBatch), C.POINTER(_abi.MargOut), C.c_uint32]
    lib.viml_line_associate.argtypes = [C.c_void_p, C.POINTER(_abi.AssocQuery), C.POINTER(_abi.AssocOut), C.c_uint32]
    lib.viml_assoc_stats.argtypes = [C.c_void_p] + [C.POINTER(C.c_int64)] * 4
    lib.viml_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    lib.viml_host_free.argtypes = [C.c_void_p]
    lib.viml_device_alloc.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.c_size_t]
    lib.viml_device_free.argtypes = [C.c_void_p, C.c_void_p]
    lib.viml_memcpy_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.viml_memcpy_d2h.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.viml_allreduce_hb.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]
    lib.viml_fov_update.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
    lib.viml_fov_slide.argtypes = [C.c_void_p, C.c_int32]
    lib.viml_track_gate.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
    lib.viml_triangulate_batch.argtypes = [C.c_void_p, C.POINTER(_abi.TriangulateIn), C.c_double, C.c_void_p, C.c_uint32]
    lib.viml_load_line_map.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_int64)]
    lib.viml_reduced_system.argtypes = [C.c_void_p, C.POINTER(_abi.WindowBatch), C.POINTER(_abi.DenseFactors),
                                        C.POINTER(_abi.ReducedOut), C.c_uint32]
    lib.viml_reduced_from_schur.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(_abi.DenseFactors),
                                            C.POINTER(_abi.ReducedOut), C.c_uint32]
    lib.viml_gn_step.argtypes = [C.c_void_p, C.POINTER(_abi.WindowBatch), C.POINTER(_abi.DenseFactors), C.c_void_p,
                                 C.POINTER(_abi.GnOptions), C.POINTER(_abi.GnOut), C.c_uint32]
    lib.viml_inertial_evaluate.argtypes = [C.c_void_p, C.POINTER(_abi.WindowBatch), C.c_void_p, C.POINTER(_abi.InertialFactors),
                                           C.POINTER(_abi.InertialOut), C.c_uint32]
    lib.viml_gn_step_vi.argtypes = [C.c_void_p, C.POINTER(_abi.WindowBatch), C.POINTER(_abi.InertialFactors), C.c_void_p,
                                    C.POINTER(_abi.GnOptions), C.POINTER(_abi.GnOut), C.c_uint32]
    lib.viml_solve_vi.argtypes = [C.c_void_p, C.POINTER(_abi.WindowBatch), C.POINTER(_abi.InertialFactors), C.c_void_p,
                                  C.POINTER(_abi.SolveOptions), C.POINTER(_abi.SolveOut), C.c_uint32]
    _LIB = lib
    return lib


class PinnedArray:
    """numpy view over cudaHostAlloc'ed memory (viml_host_alloc)."""

    def __init__(self, shape, dtype):
        lib = load_library()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        rc = lib.viml_host_alloc(C.byref(p), max(self.nbytes, 1))
        if rc != 0:
            raise VimlError(f"viml_host_alloc failed ({rc})")
        self._p = p
        buf = (C.c_byte * max(self.nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._p is not None:
            self.array = None
            load_library().viml_host_free(self._p)
            self._p = None


def pinned_like(a):
    pa = PinnedArray(a.shape, a.dtype)
    pa.array[...] = a
    return pa


class Context:
    """One viml_ctx (one CUDA device, one stream).  Mirrors the C-ABI one to one."""

    def __init__(self, cfg, device=0):
        self.lib = load_library()
        self.cfg = cfg
        h = C.c_void_p()
        rc = self.lib.viml_create(C.byref(h), C.byref(cfg), int(device))
        if rc != 0:
            raise VimlError(f"viml_create failed with {rc}: no usable CUDA device and no CPU fallback")
        self.h = h
        self.n_map = 0

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def close(self):
        if getattr(self, "h", None):
            self.lib.viml_destroy(self.h)
            self.h = None

    def _check(self, rc):
        if rc != 0:
            raise VimlError(f"viml error {rc}: {self.lib.viml_last_error(self.h).decode()}")

    def sync(self):
        self._check(self.lib.viml_sync(self.h))

    def stream(self):
        return self.lib.viml_stream(self.h)

    def kernel_launches(self):
        return int(self.lib.viml_kernel_launches(self.h))

    def profile_begin(self):
        self._check(self.lib.viml_profile_begin(self.h))

    def profile_end(self):
        """{kernel name: (total ms, launches)} for every kernel launched since profile_begin."""
        ms = (C.c_double * 16)()
        n = (C.c_int64 * 16)()
        self._check(self.lib.viml_profile_end(self.h, ms, n))
        return {self.lib.viml_kernel_name(k).decode(): (ms[k], n[k]) for k in range(16) if n[k] > 0}

    def microbench_fp64(self):
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        self._check(self.lib.viml_microbench_fp64(self.h, C.byref(a), C.byref(b)))
        self._check(self.lib.viml_microbench_dmma(self.h, C.byref(c)))
        return a.value, b.value, c.value

    # -- device memory helpers (for the resident-input benchmark path) --
    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._check(self.lib.viml_device_alloc(self.h, C.byref(p), max(int(nbytes), 1)))
        return p.value

    def device_free(self, p):
        self._check(self.lib.viml_device_free(self.h, p))

    def h2d(self, dptr, arr):
        self._check(self.lib.viml_memcpy_h2d(self.h, dptr, _abi.ptr(arr), arr.nbytes))

    def d2h(self, arr, dptr):
        self._check(self.lib.viml_memcpy_d2h(self.h, _abi.ptr(arr), dptr, arr.nbytes))

    def to_device(self, arr):
        d = self.device_alloc(arr.nbytes)
        self.h2d(d, arr)
        return d

    # -- ABI calls --
    def set_map(self, lines_xyzxyz):
        lines = np.ascontiguousarray(lines_xyzxyz, dtype=np.float64).reshape(-1, 6)
        self._check(self.lib.viml_set_map(self.h, _abi.ptr(lines), len(lines)))
        self.n_map = len(lines)

    def load_line_map(self, path):
        """viml_load_line_map: read a line_3d.txt prior map (parameters.cpp:50-59) and install it."""
        n = C.c_int64()
        self._check(self.lib.viml_load_line_map(self.h, os.fsencode(path), C.byref(n)))
        self.n_map = int(n.value)
        return self.n_map

    @staticmethod
    def _batch_struct(batch, obs_table, line_table=False):
        """viml_window_batch of host arrays; obs_table=True / "f32": observations as feat_obs + pf_obs_j (pf_obs NULL);
        line_table=True: line factors as lf_map_index + lf_seg2d_f32 (lf_geom NULL; the map must be set)."""
        if not obs_table and not line_table:
            return batch.struct(), None
        arrs = batch.arrays()
        if obs_table:
            arrs["pf_obs"] = None
            if obs_table == "f32":
                arrs["feat_obs_f32"], arrs["pf_obs_j_f32"] = batch.obs_table(f32=True)
            else:
                arrs["feat_obs"], arrs["pf_obs_j"] = batch.obs_table()
        if line_table:
            assert batch.lf_map_index is not None and batch.lf_seg2d is not None, "batch has no line table (synth.with_line_map)"
            arrs["lf_geom"] = None
            arrs["lf_map_index"], arrs["lf_seg2d_f32"] = batch.lf_map_index, batch.lf_seg2d
        return batch.struct(arrs), arrs

    def reduced_system(self, batch, dense, flags, obs_table=False, line_table=False):
        """viml_reduced_system with host buffers: (Sx [W,Dx,Dx], gx [W,Dx])."""
        X = dense.X if dense is not None else 0
        Dx = batch.D + X
        Sx, gx = np.full((batch.W, Dx, Dx), np.nan), np.full((batch.W, Dx), np.nan)
        s, _keep = self._batch_struct(batch, obs_table, line_table)
        d = dense.struct() if dense is not None else None
        o = _abi.ReducedOut()
        o.Sx, o.gx = _abi.ptr(Sx), _abi.ptr(gx)
        self._check(self.lib.viml_reduced_system(self.h, C.byref(s), C.byref(d) if d is not None else None, C.byref(o),
                                                 flags & ~PTRS_DEVICE))
        return Sx, gx

    def gn_step(self, batch, dense, extra, flags, lam=0.0, obs_table=False, line_table=False):
        """viml_gn_step with host buffers: dict(poses, ex_pose, inv_depth, extra, dx, cost, solved)."""
        X = dense.X if dense is not None else 0
        W, Dx = batch.W, batch.D + X
        res = {"poses": np.full_like(batch.poses, np.nan), "ex_pose": np.full_like(batch.ex_pose, np.nan),
               "inv_depth": np.full_like(batch.inv_depth, np.nan), "extra": np.full((W, X), np.nan),
               "dx": np.full((W, Dx), np.nan), "cost": np.full((W, 3), np.nan), "solved": np.full(W, -1, dtype=np.int32)}
        s, _keep = self._batch_struct(batch, obs_table, line_table)
        d = dense.struct() if dense is not None else None
        ex = None if extra is None else np.ascontiguousarray(extra, dtype=np.float64)
        opt = _abi.GnOptions()
        opt.lambda_ = float(lam)
        o = _abi.GnOut()
        for k in ("poses", "ex_pose", "inv_depth", "dx", "cost", "solved"):
            setattr(o, k, _abi.ptr(res[k]))
        o.extra = _abi.ptr(res["extra"]) if X > 0 else None
        self._check(self.lib.viml_gn_step(self.h, C.byref(s), C.byref(d) if d is not None else None, _abi.ptr(ex), C.byref(opt),
                                          C.byref(o), flags & ~PTRS_DEVICE))
        return res

    def inertial_evaluate(self, batch, extra, vi):
        """viml_inertial_evaluate with host buffers at the state (batch.poses, batch.ex_pose, extra [W, X]): dict of the
        viml_inertial_out arrays (imu_residual [NI,15], imu_jac_pose_i [NI,15,7], imu_jac_sb_i [NI,15,9], imu_jac_pose_j,
        imu_jac_sb_j, prior_residual [W,n_max]; prior rows past n_w are NaN)."""
        NI, W = vi.NI, batch.W
        res = {"imu_residual": np.full((NI, 15), np.nan), "imu_jac_pose_i": np.full((NI, 15, 7), np.nan),
               "imu_jac_sb_i": np.full((NI, 15, 9), np.nan), "imu_jac_pose_j": np.full((NI, 15, 7), np.nan),
               "imu_jac_sb_j": np.full((NI, 15, 9), np.nan), "prior_residual": np.full((W, vi.n_max), np.nan)}
        s = batch.struct()
        ex = None if extra is None else np.ascontiguousarray(extra, dtype=np.float64)
        v = vi.struct()
        o = _abi.InertialOut()
        for k in _abi.INERTIAL_OUT_FIELDS:
            setattr(o, k, _abi.ptr(res[k]) if res[k].size else None)
        self._check(self.lib.viml_inertial_evaluate(self.h, C.byref(s), _abi.ptr(ex), C.byref(v), C.byref(o), 0))
        return res

    def gn_step_vi(self, batch, vi, extra, flags, lam=0.0, obs_table=False, line_table=False):
        """viml_gn_step_vi with host buffers: dict(poses, ex_pose, inv_depth, extra, dx, cost, solved)."""
        X = vi.X
        W, Dx = batch.W, batch.D + X
        res = {"poses": np.full_like(batch.poses, np.nan), "ex_pose": np.full_like(batch.ex_pose, np.nan),
               "inv_depth": np.full_like(batch.inv_depth, np.nan), "extra": np.full((W, X), np.nan),
               "dx": np.full((W, Dx), np.nan), "cost": np.full((W, 3), np.nan), "solved": np.full(W, -1, dtype=np.int32)}
        s, _keep = self._batch_struct(batch, obs_table, line_table)
        v = vi.struct()
        ex = None if extra is None else np.ascontiguousarray(extra, dtype=np.float64)
        opt = _abi.GnOptions()
        opt.lambda_ = float(lam)
        o = _abi.GnOut()
        for k in ("poses", "ex_pose", "inv_depth", "dx", "cost", "solved"):
            setattr(o, k, _abi.ptr(res[k]))
        o.extra = _abi.ptr(res["extra"]) if X > 0 else None
        self._check(self.lib.viml_gn_step_vi(self.h, C.byref(s), C.byref(v), _abi.ptr(ex), C.byref(opt), C.byref(o),
                                             flags & ~PTRS_DEVICE))
        return res

    @staticmethod
    def solve_options(max_iterations=50, max_consecutive_invalid=5, initial_radius=1e4, max_radius=1e16, min_radius=1e-32,
                      min_relative_decrease=1e-3, function_tolerance=1e-6, parameter_tolerance=1e-8):
        """viml_solve_options; the defaults are ceres::Solver::Options'."""
        o = _abi.SolveOptions()
        o.max_iterations, o.max_consecutive_invalid = int(max_iterations), int(max_consecutive_invalid)
        o.initial_radius, o.max_radius, o.min_radius = float(initial_radius), float(max_radius), float(min_radius)
        o.min_relative_decrease, o.function_tolerance = float(min_relative_decrease), float(function_tolerance)
        o.parameter_tolerance = float(parameter_tolerance)
        return o

    def solve_vi(self, batch, vi, extra, flags, max_iterations=50, max_consecutive_invalid=5, initial_radius=1e4,
                 max_radius=1e16, min_radius=1e-32, min_relative_decrease=1e-3, function_tolerance=1e-6, parameter_tolerance=1e-8,
                 obs_table=False, line_table=False):
        """viml_solve_vi with host buffers: dict(poses, ex_pose, inv_depth, extra, status, iterations, accepted, cost [W,2],
        radius [W], trace [W,max_iterations,4])."""
        X, W = vi.X, batch.W
        res = {"poses": np.full_like(batch.poses, np.nan), "ex_pose": np.full_like(batch.ex_pose, np.nan),
               "inv_depth": np.full_like(batch.inv_depth, np.nan), "extra": np.full((W, X), np.nan),
               "status": np.full(W, -1, dtype=np.int32), "iterations": np.full(W, -1, dtype=np.int32),
               "accepted": np.full(W, -1, dtype=np.int32), "cost": np.full((W, 2), np.nan), "radius": np.full(W, np.nan),
               "trace": np.full((W, max(int(max_iterations), 0), 4), -1.0)}
        s, _keep = self._batch_struct(batch, obs_table, line_table)
        v = vi.struct()
        ex = None if extra is None else np.ascontiguousarray(extra, dtype=np.float64)
        opt = self.solve_options(max_iterations, max_consecutive_invalid, initial_radius, max_radius, min_radius,
                                 min_relative_decrease, function_tolerance, parameter_tolerance)
        o = _abi.SolveOut()
        for k in _abi.SOLVE_OUT_FIELDS:
            setattr(o, k, _abi.ptr(res[k]))
        o.extra = _abi.ptr(res["extra"]) if X > 0 else None
        self._check(self.lib.viml_solve_vi(self.h, C.byref(s), C.byref(v), _abi.ptr(ex), C.byref(opt), C.byref(o),
                                           flags & ~PTRS_DEVICE))
        return res

    def linearize(self, batch, flags, out=None, obs_table=False, line_table=False):
        """viml_linearize_batch with host buffers; returns dict of numpy outputs.  obs_table=True passes the observations as
        the per-feature table (feat_obs + pf_obs_j) instead of pf_obs, obs_table="f32" as the float32 table."""
        bufs = batch.alloc_out(flags) if out is None else out
        s, _keep = self._batch_struct(batch, obs_table, line_table)
        o = _abi.out_struct(bufs)
        self._check(self.lib.viml_linearize_batch(self.h, C.byref(s), C.byref(o), flags & ~PTRS_DEVICE))
        return bufs

    def linearize_raw(self, batch_struct, out_struct, flags):
        self._check(self.lib.viml_linearize_batch(self.h, C.byref(batch_struct), C.byref(out_struct), flags))

    def marginalize(self, A, b, m, eps=1e-8, want_lin=True):
        A = np.ascontiguousarray(A, dtype=np.float64)
        b = np.ascontiguousarray(b, dtype=np.float64)
        if A.ndim == 2:
            A, b = A[None], b[None]
        K, pos = A.shape[0], A.shape[1]
        n = pos - m
        res = {"A_schur": np.full((K, n, n), np.nan), "b_schur": np.full((K, n), np.nan)}
        if want_lin:
            res["linearized_jacobians"] = np.full((K, n, n), np.nan)
            res["linearized_residuals"] = np.full((K, n), np.nan)
        i = _abi.MargBatch()
        i.n_problems, i.pos, i.m, i.eps, i.A, i.b = K, pos, m, eps, _abi.ptr(A), _abi.ptr(b)
        o = _abi.MargOut()
        o.A_schur, o.b_schur = _abi.ptr(res["A_schur"]), _abi.ptr(res["b_schur"])
        o.linearized_jacobians = _abi.ptr(res.get("linearized_jacobians"))
        o.linearized_residuals = _abi.ptr(res.get("linearized_residuals"))
        self._check(self.lib.viml_marginalize_batch(self.h, C.byref(i), C.byref(o), 0))
        return res

    def fov_update(self, slot, pose, ex_pose):
        """viml_fov_update: UpdateLinesInFoV(slot) with the list kept on the device; returns its length."""
        p = np.ascontiguousarray(pose, dtype=np.float64)
        e = np.ascontiguousarray(ex_pose, dtype=np.float64)
        n = C.c_int32()
        self._check(self.lib.viml_fov_update(self.h, int(slot), _abi.ptr(p), _abi.ptr(e), C.byref(n)))
        return int(n.value)

    def fov_slide(self, marginalize_old):
        self._check(self.lib.viml_fov_slide(self.h, 1 if marginalize_old else 0))

    def triangulate(self, poses, ex_pose, feat_window, start_frame, obs_offset, points, init_depth=5.0):
        """viml_triangulate_batch with host buffers: estimated depth per feature."""
        arrs = [np.ascontiguousarray(poses, dtype=np.float64), np.ascontiguousarray(ex_pose, dtype=np.float64),
                np.ascontiguousarray(feat_window, dtype=np.int32), np.ascontiguousarray(start_frame, dtype=np.int32),
                np.ascontiguousarray(obs_offset, dtype=np.int64), np.ascontiguousarray(points, dtype=np.float64)]
        t = _abi.TriangulateIn()
        t.n_windows, t.poses_per_window = arrs[0].shape[0], arrs[0].shape[1]
        t.poses, t.ex_pose, t.feat_window, t.start_frame, t.obs_offset, t.points = [_abi.ptr(a) for a in arrs]
        t.n_features = len(arrs[2])
        depth = np.full(len(arrs[2]), np.nan)
        self._check(self.lib.viml_triangulate_batch(self.h, C.byref(t), float(init_depth), _abi.ptr(depth), 0))
        return depth

    def track_gate(self, track_offset, line_index):
        """viml_track_gate with host buffers: (credible_line [Nobs] bool, credible_matching [T] bool)."""
        off = np.ascontiguousarray(track_offset, dtype=np.int32)
        idx = np.ascontiguousarray(line_index, dtype=np.int32)
        T = len(off) - 1
        cl, cm = np.full(max(len(idx), 1), 255, dtype=np.uint8), np.full(max(T, 1), 255, dtype=np.uint8)
        self._check(self.lib.viml_track_gate(self.h, T, _abi.ptr(off), _abi.ptr(idx), _abi.ptr(cl), _abi.ptr(cm), 0))
        return cl[:len(idx)].astype(bool), cm[:T].astype(bool)

    def associate(self, cull_poses, match_poses, ex_pose, lines2d, n_lines2d=None, fov_capacity=0,
                  want_mask=False, cull_ex_pose=None, cached=False, fov_slot=None):
        """viml_line_associate with host buffers; returns dict of numpy outputs.  cached=True matches against the FoV lists
        kept on the device by fov_update / fov_slide (VIML_FOV_CACHED)."""
        keep = [None if x is None else np.ascontiguousarray(x, dtype=np.float64)
                for x in (cull_poses, match_poses, ex_pose, lines2d)]
        Pq, L = keep[3].shape[0], keep[3].shape[1]
        q = _abi.AssocQuery()
        q.n_poses, q.lines_per_pose = Pq, L
        q.cull_poses, q.match_poses, q.ex_pose, q.lines2d = [_abi.ptr(k) for k in keep]
        nl = None if n_lines2d is None else np.ascontiguousarray(n_lines2d, dtype=np.int32)
        q.n_lines2d = _abi.ptr(nl)
        cex = None if cull_ex_pose is None else np.ascontiguousarray(cull_ex_pose, dtype=np.float64)
        q.cull_ex_pose = _abi.ptr(cex)
        fs = None if fov_slot is None else np.ascontiguousarray(fov_slot, dtype=np.int32)
        q.fov_slot = _abi.ptr(fs)
        res = {"match_index": np.full((Pq, L), -2, dtype=np.int32),
               "err": np.full((Pq, L, 3), np.nan, dtype=np.float32),
               "projected": np.full((Pq, L, 4), np.nan), "fov_count": np.zeros(Pq, dtype=np.int32)}
        if fov_capacity:
            res["fov_index"] = np.full((Pq, fov_capacity), -1, dtype=np.int32)
        if want_mask:
            res["fov_mask"] = np.zeros((Pq, (self.n_map + 31) // 32), dtype=np.uint32)
        o = _abi.AssocOut()
        o.match_index, o.err, o.projected, o.fov_count = [_abi.ptr(res[k]) for k in ("match_index", "err", "projected", "fov_count")]
        o.fov_index, o.fov_capacity, o.fov_mask = _abi.ptr(res.get("fov_index")), fov_capacity, _abi.ptr(res.get("fov_mask"))
        self._check(self.lib.viml_line_associate(self.h, C.byref(q), C.byref(o), _abi.FOV_CACHED if cached else 0))
        return res

    def selftest_division(self, a, b):
        a = np.ascontiguousarray(a, dtype=np.float64)
        b = np.ascontiguousarray(b, dtype=np.float64)
        m = C.c_int64()
        self._check(self.lib.viml_selftest_division(self.h, _abi.ptr(a), _abi.ptr(b), a.size, C.byref(m)))
        return m.value

    def assoc_stats(self):
        v = [C.c_int64() for _ in range(4)]
        self._check(self.lib.viml_assoc_stats(self.h, *[C.byref(x) for x in v]))
        return tuple(x.value for x in v)   # gate tests, gated pairs, overlap-scored, distance-scored

    def associate_raw(self, q, o, flags):
        self._check(self.lib.viml_line_associate(self.h, C.byref(q), C.byref(o), flags))
