"""Times viml_slide_vi (MARGIN_OLD, device pointers) against the route a caller has without it: read the poses, the extra state and
the inverse depths back, slide and re-anchor them on the host (numpy, vectorised over windows and features), upload the result.  The
host route's choice of the re-anchored features (and of each one's first factor) is made once outside the timed region, as the
caller's FeatureManager already knows it; only the copies and the arithmetic are timed, which favours that route.
1024 EuRoC-shaped windows (synth.make_windows(1024, seed=9) + make_inertial_factors), the two alternated in one run: wall time per
call around a synchronise after a warm-up, median of five alternations of twenty calls each; the device time of one call's kernel
(the library's event pairs) in a separate pass; and the agreement of the two routes.  The card's name and power limit are read in
the same run.
usage (on a GPU box, from the repo root): python profiles/slide_time.py"""
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
REPS, N = 5, 20
INIT_DEPTH = 5.0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def rot(q):
    """normalized(q).toRotationMatrix() of [..., 7] pose blocks."""
    q = q[..., 3:7] / np.linalg.norm(q[..., 3:7], axis=-1, keepdims=True)
    x, y, z, w = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    return np.stack([np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], -1),
                     np.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)], -1),
                     np.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], -1)], -2)


res = {"card (name, power limit, max SM clock)": card(), "windows": 1024}
with pkg.Context(synth.euroc_config()) as c:
    b = synth.make_windows(1024, seed=9)
    vi, extra = synth.make_inertial_factors(b, seed=5)
    W, P, F, X = b.W, b.P, b.F, vi.X
    margin = np.zeros(W, np.int32)
    bd = b.struct({k: (None if a is None else c.to_device(np.ascontiguousarray(a))) for k, a in b.arrays().items()})
    exd, mgd = c.to_device(extra), c.to_device(margin)
    so = abi.SlideOut()
    sizes = {"poses": W * P * 7, "ex_pose": W * 7, "inv_depth": W * F, "extra": W * X}
    for k, n in sizes.items():
        setattr(so, k, c.device_alloc(n * 8))

    def new():
        c._check(c.lib.viml_slide_vi(c.h, C.byref(bd), exd, X, mgd, INIT_DEPTH, C.byref(so), abi.PTRS_DEVICE))
        c.sync()

    # the re-anchored features of every window and the first of their anchor-0 factors, known to the caller's FeatureManager
    win = np.repeat(np.arange(W), np.diff(b.pf_window_offset))
    a0 = np.flatnonzero((b.pf_idx & 0xff) == 0)
    key = win[a0] * F + (b.pf_idx[a0] >> 16).astype(np.int64)
    uk, first, cnt = np.unique(key, return_index=True, return_counts=True)
    sel = cnt >= 2
    rw, rf, rk = uk[sel] // F, uk[sel] % F, a0[first[sel]]
    uv = np.column_stack([b.pf_obs[rk, 0], b.pf_obs[rk, 1], np.ones(len(rk))])
    h = {"poses": np.empty((W, P, 7)), "ex_pose": np.empty((W, 7)), "inv_depth": np.empty((W, F)), "extra": np.empty((W, X))}
    hd = {k: c.device_alloc(n * 8) for k, n in sizes.items()}

    def old():
        for k in ("poses", "ex_pose", "inv_depth", "extra"):
            c.d2h(h[k], getattr(bd, k) if k != "extra" else exd)
        c.sync()
        po, ex, dep, xo = h["poses"], h["ex_pose"], h["inv_depth"], h["extra"]
        Rb0, Rb1, Ric = rot(po[:, 0]), rot(po[:, 1]), rot(ex)
        R0, R1 = Rb0 @ Ric, Rb1 @ Ric
        P0 = po[:, 0, :3] + np.einsum("wij,wj->wi", Rb0, ex[:, :3])
        P1 = po[:, 1, :3] + np.einsum("wij,wj->wi", Rb1, ex[:, :3])
        wp = np.einsum("nij,nj->ni", R0[rw], uv / dep[rw, rf][:, None]) + P0[rw]
        zj = np.einsum("ni,ni->n", R1[rw][:, :, 2], wp - P1[rw])
        out = {"poses": np.concatenate([po[:, 1:], po[:, -1:]], axis=1), "ex_pose": ex, "inv_depth": dep.copy(), "extra": xo.copy()}
        out["extra"][:, :9 * (P - 1)] = xo[:, 9:9 * P]
        out["inv_depth"][rw, rf] = np.where(zj > 0, 1.0 / np.where(zj > 0, zj, 1.0), 1.0 / INIT_DEPTH)
        for k in out:
            c.h2d(hd[k], np.ascontiguousarray(out[k]))
        c.sync()
        return out

    arms = {"viml_slide_vi (device pointers)": new, "read back, slide on the host (numpy), upload": old}
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
    res["kernels of one viml_slide_vi call (ms, launches)"] = c.profile_end()
    res["bytes moved by the kernel per window (state in and out, point-factor indices and observations read)"] = int(
        (2 * (P * 7 + 7 + X + F)) * 8 + (b.NP / W) * (4 + 32) + 8)
    got = {k: np.empty_like(h[k]) for k in h}
    for k in got:
        c.d2h(got[k], getattr(so, k))
    c.sync()
    ref = old()
    res["re-anchored features"] = int(len(rw))
    for k in got:
        res[f"max rel diff {k} (device against the host route)"] = float(np.max(np.abs(got[k] - ref[k]) / np.maximum(np.abs(ref[k]), 1e-300)))
print(json.dumps(res, indent=1))
