"""Times viml_solve_vi with the Levenberg-Marquardt strategy against VIML_SOLVE_DOGLEG (max_iterations = 10, default options otherwise)
on 1024 EuRoC-shaped windows (synth.make_windows(1024, seed=9) + make_inertial_factors) with device pointers, the two alternated in
one run: wall time around a synchronise and K_GN device time (the library's per-kernel event pairs) per call, five alternations of
ten calls each; also the iteration / acceptance / status distribution and the cost reached.  The card's name and power limit are
read in the same run.
usage (on a GPU box, from the repo root): python profiles/dogleg_time.py"""
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
M, REPS, N = 10, 5, 10
STATUS = ["no_convergence", "function_tol", "parameter_tol", "min_radius", "failure"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


res = {"card (name, power limit, max SM clock)": card(), "windows": 1024, "max_iterations": M}
with pkg.Context(synth.euroc_config()) as c:
    b = synth.make_windows(1024, seed=9)
    vi, extra = synth.make_inertial_factors(b, seed=5)
    W, X = b.W, vi.X
    bd = b.struct({k: (None if a is None else c.to_device(np.ascontiguousarray(a))) for k, a in b.arrays().items()})
    vd = vi.struct({k: c.to_device(np.ascontiguousarray(a)) for k, a in vi.arrays().items()})
    exd = c.to_device(extra)
    so = abi.SolveOut()
    for k, cnt, size in (("poses", b.poses.size, 8), ("ex_pose", b.ex_pose.size, 8), ("inv_depth", b.inv_depth.size, 8),
                         ("extra", W * X, 8), ("status", W, 4), ("iterations", W, 4), ("accepted", W, 4), ("cost", 2 * W, 8),
                         ("radius", W, 8), ("trace", W * M * 4, 8)):
        setattr(so, k, c.device_alloc(cnt * size))
    opt = c.solve_options(max_iterations=M)
    arms = {"levenberg_marquardt": abi.LOSS_CAUCHY | abi.PTRS_DEVICE,
            "dogleg": abi.LOSS_CAUCHY | abi.PTRS_DEVICE | abi.SOLVE_DOGLEG}

    def run(flags):
        c._check(c.lib.viml_solve_vi(c.h, C.byref(bd), C.byref(vd), exd, C.byref(opt), C.byref(so), flags))
        c.sync()

    walls = {k: [] for k in arms}
    kgn = {k: [] for k in arms}
    for f in arms.values():   # warm-up of both
        run(f)
    for _ in range(REPS):
        for name, f in arms.items():
            t = time.perf_counter()
            for _ in range(N):
                run(f)
            walls[name].append((time.perf_counter() - t) / N * 1e3)
            c.profile_begin()
            for _ in range(N):
                run(f)
            pr = c.profile_end()
            kgn[name].append(pr.get("gn_step", (float("nan"), 0))[0] / N)
    for name, f in arms.items():
        run(f)
        it, st, acc, cost = np.zeros(W, np.int32), np.zeros(W, np.int32), np.zeros(W, np.int32), np.zeros((W, 2))
        for a, p in ((it, so.iterations), (st, so.status), (acc, so.accepted), (cost, so.cost)):
            c.d2h(a, p)
        c.sync()
        res[name] = {"wall_ms_median": float(np.median(walls[name])), "wall_ms_min_max": [min(walls[name]), max(walls[name])],
                     "kgn_ms_median": float(np.median(kgn[name])), "kgn_ms_min_max": [min(kgn[name]), max(kgn[name])],
                     "iterations": {int(k): int(v) for k, v in zip(*np.unique(it, return_counts=True))},
                     "accepted": {int(k): int(v) for k, v in zip(*np.unique(acc, return_counts=True))},
                     "status": {STATUS[int(k)]: int(v) for k, v in zip(*np.unique(st, return_counts=True))},
                     "cost_sum_x0_final": [float(cost[:, 0].sum()), float(cost[:, 1].sum())]}
print(json.dumps(res, indent=1))
