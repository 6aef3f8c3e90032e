"""Times one viml_solve_vi call (max_iterations = 10) against the same ten steps driven from the host, on 1024 EuRoC-shaped windows
(synth.make_windows(1024, seed=9) + make_inertial_factors) with device pointers (VIML_PTRS_DEVICE).

  solve    one viml_solve_vi call: wall time around a synchronise, K_GN device time and the device time of every kernel;
  host     what a caller of viml_gn_step_vi can do: ten times (step, read back cost and solved, decide on the host with one lambda for
           the batch: keep x+ when the batch cost fell and halve lambda, else keep x and multiply it by 10);
  waste    the rounds enqueued after every window had stopped: the same solve with max_iterations = the largest iteration count
           (which gives the same result), timed the same way, subtracted from the 10-round call; and, since on this batch few
           windows stop early, the cost of such a round on its own: a solve whose function_tolerance stops every window after its
           first step, with 10 rounds against 1.
Also the distribution of iterations and status, and the card's name and power limit, read in the same run.
usage (on a GPU box, from the repo root): python profiles/solve_time.py"""
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
cfg = synth.euroc_config()
M = 10
STATUS = ["no_convergence", "function_tol", "parameter_tol", "min_radius", "failure"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def wall(fn, n=10):
    fn()
    t = time.perf_counter()
    for _ in range(n):
        fn()
    return (time.perf_counter() - t) / n * 1e3


def device(c, fn, n=10):
    """(K_GN ms, all kernels ms) per call."""
    fn()
    c.profile_begin()
    for _ in range(n):
        fn()
    pr = c.profile_end()
    return pr.get("gn_step", (float("nan"), 0))[0] / n, sum(v[0] for v in pr.values()) / n


res = {"card (name, power limit, max SM clock)": card(), "windows": 1024, "max_iterations": M}
with pkg.Context(cfg) as c:
    b = synth.make_windows(1024, seed=9)
    vi, extra = synth.make_inertial_factors(b, seed=5)
    W, X, Dx = b.W, vi.X, b.D + vi.X
    flags = abi.LOSS_CAUCHY | abi.PTRS_DEVICE
    bd_arrays = {k: (None if a is None else c.to_device(np.ascontiguousarray(a))) for k, a in b.arrays().items()}
    bd = b.struct(bd_arrays)
    vd = vi.struct({k: c.to_device(np.ascontiguousarray(a)) for k, a in vi.arrays().items()})
    exd = c.to_device(extra)

    # -- one solve
    so = abi.SolveOut()
    for k, cnt, size in (("poses", b.poses.size, 8), ("ex_pose", b.ex_pose.size, 8), ("inv_depth", b.inv_depth.size, 8),
                         ("extra", W * X, 8), ("status", W, 4), ("iterations", W, 4), ("accepted", W, 4), ("cost", 2 * W, 8),
                         ("radius", W, 8), ("trace", W * M * 4, 8)):
        setattr(so, k, c.device_alloc(cnt * size))

    def solve(m, **kw):
        opt = c.solve_options(max_iterations=m, **kw)

        def run():
            c._check(c.lib.viml_solve_vi(c.h, C.byref(bd), C.byref(vd), exd, C.byref(opt), C.byref(so), flags))
            c.sync()
        return run
    solve_wall = wall(solve(M))
    solve_kgn, solve_all = device(c, solve(M))
    it, st, acc = np.zeros(W, np.int32), np.zeros(W, np.int32), np.zeros(W, np.int32)
    c.d2h(it, so.iterations)
    c.d2h(st, so.status)
    c.d2h(acc, so.accepted)
    cost = np.zeros((W, 2))
    c.d2h(cost, so.cost)
    c.sync()
    last = int(it.max())
    res["solve"] = {"wall_ms": solve_wall, "kgn_ms": solve_kgn, "all_kernels_ms": solve_all,
                    "iterations": {int(k): int(v) for k, v in zip(*np.unique(it, return_counts=True))},
                    "accepted": {int(k): int(v) for k, v in zip(*np.unique(acc, return_counts=True))},
                    "status": {STATUS[int(k)]: int(v) for k, v in zip(*np.unique(st, return_counts=True))},
                    "cost_sum_x0_final": [float(cost[:, 0].sum()), float(cost[:, 1].sum())]}
    if last < M:
        w_wall = wall(solve(last))
        w_kgn, w_all = device(c, solve(last))
        res["waste"] = {"rounds_after_all_stopped": M - last, "wall_ms": solve_wall - w_wall, "kgn_ms": solve_kgn - w_kgn,
                        "all_kernels_ms": solve_all - w_all, "solve_with_max_iterations_%d_wall_ms" % last: w_wall}

    one_wall, (one_kgn, one_all) = wall(solve(1, function_tolerance=1e300)), device(c, solve(1, function_tolerance=1e300))
    all_wall, (all_kgn, all_all) = wall(solve(M, function_tolerance=1e300)), device(c, solve(M, function_tolerance=1e300))
    c.d2h(st, so.status)
    c.sync()
    res["stopped_round"] = {"status_after_round_0": {STATUS[int(k)]: int(v) for k, v in zip(*np.unique(st, return_counts=True))},
                            "per_round_wall_ms": (all_wall - one_wall) / (M - 1), "per_round_kgn_ms": (all_kgn - one_kgn) / (M - 1),
                            "per_round_all_kernels_ms": (all_all - one_all) / (M - 1)}

    # -- the same ten steps driven from the host
    # two state buffers: x and x+ swap on acceptance (every timed loop starts from whatever state the previous one left: the
    # kernels' time does not depend on it)
    state = [{k: c.to_device(np.ascontiguousarray(a)) for k, a in (("poses", b.poses), ("ex_pose", b.ex_pose),
                                                                   ("inv_depth", b.inv_depth), ("extra", extra))} for _ in range(2)]
    dx, dcost, dsolved = c.device_alloc(W * Dx * 8), c.device_alloc(W * 3 * 8), c.device_alloc(W * 4)
    h_cost, h_solved = pkg.PinnedArray((W, 3), np.float64), pkg.PinnedArray((W,), np.int32)

    def host_loop():
        cur = 0
        lam = 1e-4
        for _ in range(M):
            nxt = 1 - cur
            s = b.struct({**bd_arrays, **{k: state[cur][k] for k in ("poses", "ex_pose", "inv_depth")}})
            o = abi.GnOut()
            o.poses, o.ex_pose, o.inv_depth, o.extra = (state[nxt][k] for k in ("poses", "ex_pose", "inv_depth", "extra"))
            o.dx, o.cost, o.solved = dx, dcost, dsolved
            opt = abi.GnOptions()
            opt.lambda_ = lam
            c._check(c.lib.viml_gn_step_vi(c.h, C.byref(s), C.byref(vd), state[cur]["extra"], C.byref(opt), C.byref(o), flags))
            c._check(c.lib.viml_memcpy_d2h(c.h, h_cost.array.ctypes.data, dcost, W * 3 * 8))
            c._check(c.lib.viml_memcpy_d2h(c.h, h_solved.array.ctypes.data, dsolved, W * 4))
            c.sync()
            ok = h_solved.array != 0
            if ok.any() and h_cost.array[ok, 1].sum() < h_cost.array[ok, 0].sum():
                cur, lam = nxt, lam * 0.5
            else:
                lam *= 10.0
        c.sync()
    res["host_loop"] = {"wall_ms": wall(host_loop), "steps": M}
    k, a = device(c, host_loop, 3)
    res["host_loop"].update({"kgn_ms": k, "all_kernels_ms": a})
print(json.dumps(res, indent=1))
