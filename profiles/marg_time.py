"""Times viml_marginalize_vi (MARGIN_OLD, device pointers) against the route a caller had before it, driven batch-wide from Python
with host buffers: select the point factors with i == 0, viml_linearize_batch(VIML_OUT_SCHUR), viml_inertial_evaluate, the prior and
the IMU factors with pose i = 0 as viml_dense_factors, viml_reduced_from_schur, a numpy gather of [pose 0, speed-bias 0 | kept] and
viml_marginalize_batch.  1024 EuRoC-shaped windows (synth.make_windows(1024, seed=9) + make_inertial_factors), the two alternated in
one run: wall time per call around a synchronise after a warm-up, median of five alternations of five calls each; the per-kernel
device times of one viml_marginalize_vi call (the library's event pairs) in a separate pass; and the agreement of the two routes
(J^T J and J^T r of the returned priors).  The card's name and power limit are read in the same run.
usage (on a GPU box, from the repo root): python profiles/marg_time.py"""
import ctypes as C
import importlib
import json
import subprocess
import sys
import time

sys.path.insert(0, ".")
import numpy as np  # noqa: E402

pkg = importlib.import_module("tc-viml_b200")
abi, synth = pkg._abi, pkg.synth
REPS, N = 5, 5


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


res = {"card (name, power limit, max SM clock)": card(), "windows": 1024}
with pkg.Context(synth.euroc_config()) as c:
    b = synth.make_windows(1024, seed=9)
    vi, extra = synth.make_inertial_factors(b, seed=5)
    W, P, D, X, n_max = b.W, b.P, b.D, vi.X, vi.n_max
    mb = 2 * P + 1
    margin = np.zeros(W, np.int32)
    bd = b.struct({k: (None if a is None else c.to_device(np.ascontiguousarray(a))) for k, a in b.arrays().items()})
    vd = vi.struct({k: c.to_device(np.ascontiguousarray(a)) for k, a in vi.arrays().items()})
    exd, mgd = c.to_device(extra), c.to_device(margin)
    po = abi.PriorOut()
    po.prior_n_max, po.prior_max_blocks = n_max, mb
    sizes = {"prior_n": W * 4, "prior_jacobian": W * n_max * n_max * 8, "prior_residual": W * n_max * 8, "prior_n_blocks": W * 4,
             "prior_block": W * mb * 16, "prior_x0": W * mb * 72}
    for k, nb in sizes.items():
        setattr(po, k, c.device_alloc(nb))

    def new():
        c._check(c.lib.viml_marginalize_vi(c.h, C.byref(bd), C.byref(vd), exd, mgd, C.byref(po), abi.LOSS_CAUCHY | abi.PTRS_DEVICE))
        c.sync()

    # the route before: every window's selection and gather from Python (MARGIN_OLD of synth's windows: pose 0 and speed-bias 0
    # marginalised, poses 1..P-1, the extrinsic and speed-bias 1 kept, the same for every window)
    drop = list(range(6)) + list(range(D, D + 9))
    keep = list(range(6, 6 * P + 6)) + list(range(D + 9, D + 18))
    order = np.array(drop + keep)

    def old():
        win = np.repeat(np.arange(W), np.diff(b.pf_window_offset))
        sel = (b.pf_idx & 0xff) == 0
        off = np.concatenate([[0], np.cumsum(np.bincount(win[sel], minlength=W))]).astype(np.int32)
        sb = abi.Batch(b.poses, b.ex_pose, b.inv_depth, off, b.pf_idx[sel], b.pf_obs[sel])
        lin = c.linearize(sb, abi.OUT_SCHUR | abi.LOSS_CAUCHY)
        ev = c.inertial_evaluate(b, extra, vi)
        dense = vi.to_dense(ev)
        imu_w, imu_i = vi.imu_window(), vi.imu_pose[:, 0]
        keepf, k = [], 0
        for w in range(W):   # per window: the prior, then its IMU factors (to_dense's order)
            if vi.prior_n[w] > 0:
                keepf.append(dense.factors[k])
                k += 1
            for f in range(vi.imu_window_offset[w], vi.imu_window_offset[w + 1]):
                if imu_i[f] == 0 and vi.imu_preint[f, 0] < 10.0:
                    keepf.append(dense.factors[k])
                k += 1
        d = abi.Dense(W, X, keepf)
        Sx, gx = np.full((W, D + X, D + X), np.nan), np.full((W, D + X), np.nan)
        ro = abi.ReducedOut()
        ro.Sx, ro.gx = abi.ptr(Sx), abi.ptr(gx)
        c._check(c.lib.viml_reduced_from_schur(c.h, W, D, abi.ptr(lin["S"]), abi.ptr(lin["g"]), C.byref(d.struct()), C.byref(ro), 0))
        A = np.ascontiguousarray(Sx[:, order][:, :, order])
        bb = np.ascontiguousarray(gx[:, order])
        return c.marginalize(A, bb, len(drop))

    arms = {"viml_marginalize_vi (device pointers)": new, "route before (host buffers, Python glue)": old}
    for f in arms.values():
        f()
    walls = {k: [] for k in arms}
    for _ in range(REPS):
        for name, f in arms.items():
            t = time.perf_counter()
            for _ in range(N):
                f()
            walls[name].append((time.perf_counter() - t) / N * 1e3)
    for name in arms:
        res[name] = {"wall_ms_median": float(np.median(walls[name])), "wall_ms_min_max": [min(walls[name]), max(walls[name])]}
    c.profile_begin()
    new()
    res["kernels of one viml_marginalize_vi call (ms, launches)"] = c.profile_end()
    # agreement: J^T J and J^T r of both routes
    got = {}
    for k, nb in sizes.items():
        a = np.empty(nb // (4 if k in ("prior_n", "prior_n_blocks", "prior_block") else 8),
                     np.int32 if k in ("prior_n", "prior_n_blocks", "prior_block") else np.float64)
        c.d2h(a, getattr(po, k))
        got[k] = a
    c.sync()
    ref = old()
    n = len(keep)
    J = got["prior_jacobian"].reshape(W, n_max, n_max)[:, :n, :n]
    r = got["prior_residual"].reshape(W, n_max)[:, :n]
    J1, r1 = ref["linearized_jacobians"], ref["linearized_residuals"]
    JtJ, J1tJ1 = np.einsum("wki,wkj->wij", J, J), np.einsum("wki,wkj->wij", J1, J1)
    res["prior_n"] = sorted(set(int(x) for x in got["prior_n"]))
    res["max rel diff J^T J (per window)"] = float(max(np.abs(JtJ[w] - J1tJ1[w]).max() / np.abs(J1tJ1[w]).max() for w in range(W)))
    Jr, J1r1 = np.einsum("wki,wk->wi", J, r), np.einsum("wki,wk->wi", J1, r1)
    res["max rel diff J^T r (per window)"] = float(max(np.abs(Jr[w] - J1r1[w]).max() / np.abs(J1r1[w]).max() for w in range(W)))
print(json.dumps(res, indent=1))
