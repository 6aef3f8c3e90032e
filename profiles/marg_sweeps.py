"""Times viml_marginalize_batch per size n, to see whether marg_kernel's Jacobi meets its stopping rule off(A)^2 <= 1e-30 |A|_F^2
or runs to its cap of 40 sweeps.  m = 0, so each problem is one n x n Jacobi (plus the outputs); K = 296 random SPD problems
(M^T M, M of n + 8 rows) per call = two per SM of a 148-SM B200, device pointers, inputs resident in L2 (at most 78 MB at n = 256).
Device time of marg_kernel from the library's per-kernel event pairs over REPS calls after a warm-up call; reported as ms per
call and as ns per n^3 per problem.  A sweep costs ~n^3, so a jump in ns / n^3 between neighbouring n marks more sweeps.  Alongside,
the sweeps the same algorithm needs in numpy float64 (round-robin order, the kernel's rotation formulas and stopping rule; the
device contracts to FMAs, so its count may differ by one or two) for one problem of each size.
usage (on a GPU box, from the repo root): python profiles/marg_sweeps.py > profiles/marg_sweeps.txt"""
import ctypes as C
import importlib
import json
import subprocess
import sys

sys.path.insert(0, ".")
import numpy as np  # noqa: E402

pkg = importlib.import_module("tc-viml_b200")
abi, synth = pkg._abi, pkg.synth
K, REPS = 296, 5
SIZES = [16, 32, 48, 64, 96, 128, 160, 192, 224, 240, 248, 252, 253, 254, 255, 256]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def sweeps_f64(A, cap=40):
    """block_jacobi restated in numpy float64: the sweeps run before off^2 <= 1e-30 |A|_F^2 (cap: the rule was never met)."""
    a = A.copy()
    n = a.shape[0]
    ne = n + (n & 1)
    k = np.arange(ne // 2)
    offd = ~np.eye(n, dtype=bool)
    np.seterr(over="ignore", invalid="ignore", divide="ignore")   # theta overflows for tiny a_pq, as on the device: t = 0
    for sweep in range(cap):
        off, tot = (a[offd] ** 2).sum(), (a * a).sum()
        if off <= 1e-30 * tot or off == 0:
            return sweep
        for r in range(ne - 1):
            p = np.where(k == 0, ne - 1, (r + k) % (ne - 1))
            q = (r + (ne - 1) - k) % (ne - 1)
            p, q = np.minimum(p, q), np.maximum(p, q)
            p, q = p[q < n], q[q < n]
            apq = a[p, q]
            theta = np.where(apq != 0, (a[q, q] - a[p, p]) / (2 * np.where(apq != 0, apq, 1)), 0)
            t = np.where(apq != 0, np.where(theta >= 0, 1.0, -1.0) / (np.abs(theta) + np.sqrt(theta * theta + 1)), 0)
            c = 1 / np.sqrt(t * t + 1)
            s = t * c
            ap, aq = a[:, p].copy(), a[:, q].copy()
            a[:, p], a[:, q] = c * ap - s * aq, s * ap + c * aq
            ap, aq = a[p, :].copy(), a[q, :].copy()
            a[p, :], a[q, :] = c[:, None] * ap - s[:, None] * aq, s[:, None] * ap + c[:, None] * aq
    return cap


res = {"card (name, power limit, max SM clock)": card(), "problems per call": K, "calls timed": REPS, "sizes": []}
rng = np.random.default_rng(1)
with pkg.Context(synth.euroc_config()) as c:
    for n in SIZES:
        M = rng.standard_normal((K, n + 8, n))
        A = np.ascontiguousarray(np.einsum("kri,krj->kij", M, M))
        b = rng.standard_normal((K, n))
        dA, db = c.to_device(A), c.to_device(b)
        outs = [c.device_alloc(K * n * n * 8), c.device_alloc(K * n * 8), c.device_alloc(K * n * n * 8), c.device_alloc(K * n * 8)]
        i = abi.MargBatch()
        i.n_problems, i.pos, i.m, i.eps, i.A, i.b = K, n, 0, 1e-8, dA, db
        o = abi.MargOut()
        o.A_schur, o.b_schur, o.linearized_jacobians, o.linearized_residuals = outs

        def call():
            c._check(c.lib.viml_marginalize_batch(c.h, C.byref(i), C.byref(o), abi.PTRS_DEVICE))

        call()
        c.sync()
        c.profile_begin()
        for _ in range(REPS):
            call()
        c.sync()
        ms, launches = c.profile_end()["marginalize_dense"]
        per = ms / launches
        res["sizes"].append({"n": n, "ms_per_call": per, "ns_per_n3_per_problem": per * 1e6 / K / n ** 3,
                             "sweeps_numpy_f64": sweeps_f64(A[0])})
        for p in [dA, db] + outs:
            c.device_free(p)
print(json.dumps(res, indent=1))
