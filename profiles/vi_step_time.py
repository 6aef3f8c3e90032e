"""Times viml_inertial_evaluate alone (4096 EuRoC-shaped windows, realistic IMU noise: about 41 K IMU factors and 4096 priors) and
viml_gn_step_vi against viml_gn_step on the same 1024 windows, with host and with device pointers (VIML_PTRS_DEVICE).  Device time
is the K_GN event pairs (profile_begin / profile_end); wall time is per call after a warm-up.
usage (on a GPU box, from the repo root): python profiles/vi_step_time.py"""
import ctypes as C
import importlib
import json
import sys
import time

sys.path.insert(0, ".")
import numpy as np  # noqa: E402

pkg = importlib.import_module("tc-viml_b200")
abi, synth = pkg._abi, pkg.synth
cfg = synth.euroc_config()
HBM_GBS = 6553.0   # B200 HBM3e peak used for the traffic fraction


def wall(fn, n=5):
    fn()
    t = time.perf_counter()
    for _ in range(n):
        fn()
    return (time.perf_counter() - t) / n * 1e3


def kgn(c, fn, n=5):
    fn()
    c.profile_begin()
    for _ in range(n):
        fn()
    pr = c.profile_end()
    return pr["gn_step"][0] / n if "gn_step" in pr else float("nan")


res = {}
with pkg.Context(cfg) as c:
    b = synth.make_windows(4096, seed=9, F=8, lines_per_frame=1)
    vi, extra = synth.make_inertial_factors(b, seed=5, realistic=True)
    NI, W, n = vi.NI, vi.W, vi.n_max
    # bytes: IMU inputs (pose/sb indices, 17 + 2 x 225 doubles) + the state read + the Ceres outputs (15 + 2 x 105 + 2 x 135);
    # prior: J (n^2) + linearized residuals + x0 + the residual written
    imu_bytes = NI * (16 + 8 * (17 + 450) + 8 * (2 * 7 + 2 * 9) + 8 * (15 + 480))
    prior_bytes = W * 8 * (n * n + 2 * n + vi.max_blocks * (abi.PRIOR_X0_STRIDE + 7 + 4))
    dev = {k: c.to_device(np.ascontiguousarray(a)) for k, a in vi.arrays().items()}
    s = b.struct({**b.arrays(), "poses": c.to_device(b.poses), "ex_pose": c.to_device(b.ex_pose)})
    v = vi.struct(dev)
    dex = c.to_device(extra)
    outs = {"imu_residual": NI * 15, "imu_jac_pose_i": NI * 105, "imu_jac_sb_i": NI * 135, "imu_jac_pose_j": NI * 105,
            "imu_jac_sb_j": NI * 135, "prior_residual": W * n}
    o = abi.InertialOut()
    for k, cnt in outs.items():
        setattr(o, k, c.device_alloc(cnt * 8))

    def ev():
        c._check(c.lib.viml_inertial_evaluate(c.h, C.byref(s), dex, C.byref(v), C.byref(o), abi.PTRS_DEVICE))
    ms = kgn(c, ev, 20)
    res["inertial_evaluate_4096"] = {"n_imu": NI, "n_prior": W, "device_ms": ms, "MB": (imu_bytes + prior_bytes) / 1e6,
                                     "frac_hbm_peak": (imu_bytes + prior_bytes) / (ms * 1e-3) / (HBM_GBS * 1e9)}

    b = synth.make_windows(1024, seed=9)
    vi, extra = synth.make_inertial_factors(b, seed=5)
    dense = vi.to_dense(c.inertial_evaluate(b, extra, vi))
    lam = 1e-4
    r = {"gn_step_host_ms": wall(lambda: c.gn_step(b, dense, extra, abi.LOSS_CAUCHY, lam=lam)),
         "gn_step_vi_host_ms": wall(lambda: c.gn_step_vi(b, vi, extra, abi.LOSS_CAUCHY, lam=lam)),
         "gn_step_kgn_ms": kgn(c, lambda: c.gn_step(b, dense, extra, abi.LOSS_CAUCHY, lam=lam)),
         "gn_step_vi_kgn_ms": kgn(c, lambda: c.gn_step_vi(b, vi, extra, abi.LOSS_CAUCHY, lam=lam))}
    # device pointers
    X, Dx = vi.X, b.D + vi.X
    bd = b.struct({k: (None if a is None else c.to_device(np.ascontiguousarray(a))) for k, a in b.arrays().items()})
    vd = vi.struct({k: c.to_device(np.ascontiguousarray(a)) for k, a in vi.arrays().items()})
    dd = dense.struct({k: c.to_device(np.ascontiguousarray(a)) for k, a in dense.arrays().items()})
    exd = c.to_device(extra)
    go = abi.GnOut()
    for k, cnt in (("poses", b.poses.size), ("ex_pose", b.ex_pose.size), ("inv_depth", b.inv_depth.size), ("extra", b.W * X),
                   ("dx", b.W * Dx), ("cost", b.W * 3), ("solved", b.W)):
        setattr(go, k, c.device_alloc(cnt * 8))
    opt = abi.GnOptions()
    opt.lambda_ = lam
    flags = abi.LOSS_CAUCHY | abi.PTRS_DEVICE

    def step_dev():
        c._check(c.lib.viml_gn_step(c.h, C.byref(bd), C.byref(dd), exd, C.byref(opt), C.byref(go), flags))
        c.sync()

    def step_vi_dev():
        c._check(c.lib.viml_gn_step_vi(c.h, C.byref(bd), C.byref(vd), exd, C.byref(opt), C.byref(go), flags))
        c.sync()
    r["gn_step_device_ms"] = wall(step_dev)
    r["gn_step_vi_device_ms"] = wall(step_vi_dev)
    res["step_1024"] = r

    # small host-pointer calls (a live sliding window): latency-bound, one copy each way
    rng = np.random.default_rng(3)
    for w in (1, 12):
        b = synth.make_windows(w, seed=9)
        vi, extra = synth.make_inertial_factors(b, seed=5)
        M = rng.standard_normal((w, 98, 90))
        A, bm = np.einsum("kij,kil->kjl", M, M), rng.standard_normal((w, 90))
        res[f"host_{w}"] = {"gn_step_vi_ms": wall(lambda: c.gn_step_vi(b, vi, extra, abi.LOSS_CAUCHY, lam=lam), 50),
                            "solve_vi_10_rounds_ms": wall(lambda: c.solve_vi(b, vi, extra, abi.LOSS_CAUCHY, max_iterations=10), 50),
                            "marginalize_90_15_ms": wall(lambda: c.marginalize(A, bm, 15), 50)}
print(json.dumps(res, indent=1))
