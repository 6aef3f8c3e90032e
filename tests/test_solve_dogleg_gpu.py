"""viml_solve_vi with VIML_SOLVE_DOGLEG: the dogleg trust-region strategy per window on the device.

The reference is a per-window numpy dogleg over the window's whole problem, independent of the device's Schur step: H and g in the
full N x N space (poses / extrinsic, extra state, inverse depths) from the library's (or the CPU oracle's) H/b blocks plus the IMU /
prior factors' J^T J, the damped system solved densely, x+ by pose_plus, f(x+) from the library's (or the oracle's) cost at x+, and
the scalar step and policy of tests/dogleg_policy.py.  The device eliminates the landmarks and solves the reduced system with a
blocked Cholesky, so values agree to 1e-9 and the decisions exactly; bit-exact checks are only made between device runs."""
import copy
import math

import numpy as np
import pytest

import dogleg_policy as dp
import inertial_oracle as io
from conftest import rel_err
from vi_helpers import bits, inertial_only, rotate, slice_vi, solve_device

pytestmark = pytest.mark.gpu

CAUCHY, OUT_HB = 0x10, 0x02
STATE = ("poses", "ex_pose", "inv_depth", "extra")
EPS = 1e-8


def _case(pkg, W=6, seed=5, P=11, F=40, no_imu=(), perturb=(0.002, 0.01, 0.05, 0.5, 1.0)):
    """W windows whose state is moved away from the one the factors were built at; windows in no_imu carry the prior only."""
    batch = pkg.synth.make_windows(W, seed=seed, P=P, F=F)
    vi, extra = pkg.synth.make_inertial_factors(batch, seed=seed + 1, no_imu=no_imu)
    rng = np.random.default_rng(seed + 2)
    for w in range(W):
        s = perturb[w % len(perturb)]
        batch.poses[w, :, :3] += s * rng.standard_normal((P, 3))
        for p in range(P):
            batch.poses[w, p] = rotate(batch.poses[w, p], 0.5 * s * rng.standard_normal(3))
        extra[w] += s * rng.standard_normal(extra.shape[1])
    return batch, vi, extra


# ---- the numpy reference ------------------------------------------------------------------------------------------------------

def _full_system(lin, dense, D, X, F):
    """H [N, N] and g [N] of window 0 from the H/b blocks and the dense-block factors."""
    Dx = D + X
    N = Dx + F
    H, g = np.zeros((N, N)), np.zeros(N)
    H[:D, :D] = lin["H_pp"][0]
    H[Dx:, :D] = lin["H_lp"][0]
    H[:D, Dx:] = lin["H_lp"][0].T
    H[np.arange(Dx, N), np.arange(Dx, N)] = lin["H_ll"][0]
    g[:D], g[Dx:] = lin["b_p"][0], lin["b_l"][0]
    for (_, r, J, ci) in dense.factors:
        J, ci = np.asarray(J), np.asarray(ci)
        H[np.ix_(ci, ci)] += J.T @ J
        g[ci] += J.T @ np.asarray(r)
    return H, g


def _plus(b, ex, step, P, D, Dx):
    nb, nex = copy.deepcopy(b), ex.copy()
    for p in range(P):
        nb.poses[0, p] = io_pose_plus(b.poses[0, p], step[6 * p:6 * p + 6])
    nb.ex_pose[0] = io_pose_plus(b.ex_pose[0], step[6 * P:6 * P + 6])
    nex[0] = ex[0] + step[D:Dx]
    nb.inv_depth[0] = b.inv_depth[0] + step[Dx:]
    return nb, nex


def io_pose_plus(x, d):
    from oracle import gn_oracle
    return gn_oracle.pose_plus(x, d)


def _reference(system, cost, batch1, extra1, X, opt):
    """One window (batch1, extra1) solved by the numpy dogleg.  system(b, ex) -> (H, g); cost(b, ex) -> f.  Returns the solve_vi
    outputs of the window plus the dogleg case of every step and the number of steps that reused a stored one."""
    b, ex = copy.deepcopy(batch1), extra1.copy()
    P, F, D = b.P, b.F, b.D
    Dx = D + X
    st, trace, cases, reused = None, [], [], 0
    s = None
    while True:
        f = cost(b, ex)
        if st is None:
            st = dp.start(f, opt)
            if st.status is not None:
                break
        if not st.reuse:
            H, g = system(b, ex)
            keep = np.concatenate([np.ones(Dx, bool), np.diag(H)[Dx:] > EPS])
            if s is None:
                s = 1.0 / (1.0 + np.sqrt(np.diag(H)))
            d = np.sqrt(np.minimum(np.maximum(s * s * np.diag(H), 1e-6), 1e32))
            gam = np.where(keep, s * g / d, 0.0)
            w = s * gam / d
            dgn = np.zeros(Dx + F)
            valid = st.mu < dp.MAX_MU
            if valid:
                k = np.flatnonzero(keep)
                A = H[np.ix_(k, k)] + np.diag(st.mu * d[k] * d[k] / (s[k] * s[k]))
                try:
                    L = np.linalg.cholesky(A)
                    dgn[k] = -np.linalg.solve(L.T, np.linalg.solve(L, g[k]))
                except np.linalg.LinAlgError:
                    valid = False
            nv = d * dgn / s
            sc = (gam @ gam, nv @ nv, gam @ nv, w @ H @ w, w @ H @ dgn, dgn @ H @ dgn)
        else:
            reused += 1
        if valid:
            case, a, bb, norm, m = dp.step(*(float(v) for v in sc), st.radius)
            step = a * w + bb * dgn
            nb, nex = _plus(b, ex, step, P, D, Dx)
            fp = cost(nb, nex)
        else:
            case, norm, m, step, nb, nex, fp = 0, 0.0, 0.0, np.zeros(Dx + F), b, ex, f
        cases.append(case)
        step_norm = math.sqrt(float(np.sum(step[:Dx] ** 2) + np.sum((nb.inv_depth[0] - b.inv_depth[0]) ** 2)))
        x_norm = math.sqrt(float(np.sum(b.poses ** 2) + np.sum(b.ex_pose ** 2) + np.sum(b.inv_depth ** 2) + np.sum(ex ** 2)))
        acc, row = dp.advance(st, opt, f, fp, m, valid, step_norm, x_norm, norm)
        trace.append(row)
        if acc:
            b, ex = nb, nex
        if st.status is not None:
            break
    tr = np.full((opt.max_iterations, 4), np.nan)
    if trace:
        tr[:len(trace)] = trace
    return {"poses": b.poses[0], "ex_pose": b.ex_pose[0], "inv_depth": b.inv_depth[0], "extra": ex[0], "status": st.status,
            "iterations": st.iterations, "accepted": st.accepted, "cost": np.array([st.f0, st.f]), "radius": st.radius,
            "trace": tr, "cases": cases, "reused": reused}


def _library_reference(pkg, ctx, batch, vi, extra, opt):
    ref = []
    for w in range(batch.W):
        vi1 = slice_vi(pkg, vi, w)

        def system(b, ex):
            lin = ctx.linearize(b, OUT_HB | CAUCHY)
            return _full_system(lin, vi1.to_dense(ctx.inertial_evaluate(b, ex, vi1)), b.D, vi.X, b.F)

        def cost(b, ex):
            return float(ctx.gn_step_vi(b, vi1, ex, CAUCHY, lam=1.0)["cost"][0, 0])
        ref.append(_reference(system, cost, batch.slice_windows(w, w + 1), extra[w:w + 1], vi.X, opt))
    return ref


def _solve(pkg, ctx, batch, vi, extra, opt, flags=CAUCHY):
    return ctx.solve_vi(batch, vi, extra, flags | pkg.SOLVE_DOGLEG, **vars(opt))


def _decisions(trace, n, opt):
    """The accept / reject sequence of every step but the last (which may have stopped on a tolerance instead)."""
    return [bool(math.isfinite(fp) and m > 0.0 and (f - fp) / m > opt.min_relative_decrease) for f, fp, m, _ in trace[:max(n - 1, 0)]]


def _check_close(got, ref, opt, tol=1e-9):
    for w, r in enumerate(ref):
        assert (got["status"][w], got["iterations"][w], got["accepted"][w]) == (r["status"], r["iterations"], r["accepted"]), w
        n = int(r["iterations"])
        assert np.all(np.isnan(got["trace"][w, n:])), w
        assert _decisions(got["trace"][w], n, opt) == _decisions(r["trace"], n, opt), w
        assert rel_err(got["trace"][w, :n], r["trace"][:n]) < tol, w
        for k in STATE:
            assert rel_err(got[k][w], r[k]) < tol, (w, k)
        assert rel_err(got["cost"][w], r["cost"]) < tol and abs(got["radius"][w] - r["radius"]) <= tol * r["radius"], w


OPTIONS = (dp.Options(max_iterations=12, initial_radius=1e-3),
           dp.Options(max_iterations=12, initial_radius=1e-2, min_relative_decrease=0.999, max_consecutive_invalid=2),
           dp.Options(max_iterations=6)) + tuple(dp.Options(max_iterations=3, initial_radius=r) for r in (0.03, 0.1, 0.3, 1.0, 3.0))


def _run_against_reference(pkg, ctx, batch, vi, extra):
    cases, reused = set(), 0
    for opt in OPTIONS:
        got = _solve(pkg, ctx, batch, vi, extra, opt)
        ref = _library_reference(pkg, ctx, batch, vi, extra, opt)
        _check_close(got, ref, opt)
        for r in ref:
            cases |= set(r["cases"])
            reused += r["reused"]
    print("dogleg cases", sorted(cases), "reused steps", reused)
    return cases, reused


def test_against_numpy_inertial_only(pkg, ctx):
    batch, vi, extra = _case(pkg, W=5, seed=5)
    cases, reused = _run_against_reference(pkg, ctx, inertial_only(pkg, batch), vi, extra)
    assert {1, 2, 3} <= cases and reused > 0


def test_against_numpy_with_point_and_line_factors(pkg, ctx):
    batch, vi, extra = _case(pkg, W=4, seed=13, perturb=(0.002, 0.01, 0.05, 0.2))   # well-conditioned windows only
    cases, reused = _run_against_reference(pkg, ctx, batch, vi, extra)
    assert {1, 2, 3} <= cases and reused > 0


def test_against_cpu_oracle(pkg, orc, ctx, cfg):
    from oracle import gn_oracle
    batch, vi, extra = _case(pkg, W=2, seed=21, perturb=(0.01, 0.03))
    opt = dp.Options(max_iterations=5, initial_radius=1e-2)
    got = _solve(pkg, ctx, batch, vi, extra, opt)
    for w in range(2):
        vi1 = slice_vi(pkg, vi, w)

        def system(b, ex):
            lin = orc.linearize_batch(cfg, b, OUT_HB | CAUCHY)
            return _full_system(lin, vi1.to_dense(io.inertial_evaluate(orc, b.poses, b.ex_pose, ex, vi1)), b.D, vi.X, b.F)

        def cost(b, ex):
            return float(gn_oracle.window_cost(cfg, b, CAUCHY)[0] + io.inertial_cost(orc, b.poses, b.ex_pose, ex, vi1)[0])
        ref = _reference(system, cost, batch.slice_windows(w, w + 1), extra[w:w + 1], vi.X, opt)
        _check_close({k: v[w:w + 1] for k, v in got.items()}, [ref], opt)
        assert ref["accepted"] > 0


def test_unfused(pkg, ctx):
    """Dx = 201 (P = 13): the separate reduced-system and solve kernels."""
    batch, vi, extra = _case(pkg, W=3, seed=33, P=13, F=20)
    assert batch.D + vi.X == 201
    b = inertial_only(pkg, batch)
    opt = dp.Options(max_iterations=8, initial_radius=1e-2)
    got = _solve(pkg, ctx, b, vi, extra, opt)
    _check_close(got, _library_reference(pkg, ctx, b, vi, extra, opt), opt)
    assert (got["accepted"] > 0).all()


def test_window_independence(pkg, ctx):
    """Without point and line factors a window solved in a batch equals the same window solved alone, bit for bit."""
    batch, vi, extra = _case(pkg, W=5, seed=71)
    b = inertial_only(pkg, batch)
    opt = dp.Options(max_iterations=10, initial_radius=1e-2)
    got = _solve(pkg, ctx, b, vi, extra, opt)
    for w in range(b.W):
        one = _solve(pkg, ctx, b.slice_windows(w, w + 1), slice_vi(pkg, vi, w), extra[w:w + 1], opt)
        for k in one:
            assert np.array_equal(bits(got[k][w]), bits(one[k][0])), (w, k)


def test_nan_in_one_window(pkg, ctx):
    batch, vi, extra = _case(pkg, W=6, seed=51)
    b = inertial_only(pkg, batch)
    opt = dp.Options(max_iterations=6, initial_radius=1e-2)
    clean = _solve(pkg, ctx, b, vi, extra, opt)
    bad = copy.deepcopy(b)
    bad.poses[3, 4, 1] = np.nan
    got = _solve(pkg, ctx, bad, vi, extra, opt)
    assert got["status"][3] == dp.FAILURE and got["iterations"][3] == 0 and got["accepted"][3] == 0
    assert np.isnan(got["cost"][3]).all() and np.isnan(got["trace"][3]).all() and got["radius"][3] == 1e-2
    start = {"poses": bad.poses, "ex_pose": bad.ex_pose, "inv_depth": bad.inv_depth, "extra": extra}
    for k in STATE:
        assert np.array_equal(bits(got[k][3]), bits(start[k][3])), k
    others = [w for w in range(b.W) if w != 3]
    for k in clean:
        assert np.array_equal(bits(got[k][others]), bits(clean[k][others])), k


def test_prior_only_window(pkg, ctx):
    """A window with the prior alone has a singular J^T J.  The dogleg's damping mu d^2 / s^2 keeps every column's diagonal at least
    mu 1e-6 / s^2 (Ceres' clamp of the scaled diagonal), so the window still converges: its state stays finite, its cost does not
    rise, and the windows beside it are those of the batch without it."""
    batch, vi, extra = _case(pkg, W=4, seed=5, no_imu=(2,))
    b = inertial_only(pkg, batch)
    opt = dp.Options(max_iterations=12)
    got = _solve(pkg, ctx, b, vi, extra, opt)
    assert got["status"][2] != dp.FAILURE and got["accepted"][2] > 0
    for k in STATE:
        assert np.isfinite(got[k][2]).all(), k
    assert got["cost"][2, 1] <= got["cost"][2, 0]
    for w in (0, 1, 3):
        one = _solve(pkg, ctx, b.slice_windows(w, w + 1), slice_vi(pkg, vi, w), extra[w:w + 1], opt)
        for k in one:
            assert np.array_equal(bits(got[k][w]), bits(one[k][0])), (w, k)


def test_device_pointers(pkg, ctx):
    """Guarded device buffers: nothing is written outside the outputs, the inputs stay untouched, and two calls agree with each
    other and with the host flavour bit for bit (no point or line factors, whose pose blocks are summed through atomics)."""
    batch, vi, extra = _case(pkg, W=6, seed=41)
    b = inertial_only(pkg, batch)
    opt = dp.Options(max_iterations=8, initial_radius=1e-2)
    host = _solve(pkg, ctx, b, vi, extra, opt)
    for _ in range(2):
        dev = solve_device(pkg, ctx, b, vi, extra, opt, CAUCHY | pkg.SOLVE_DOGLEG)
        for k in host:
            assert np.array_equal(bits(dev[k]), bits(host[k])), k
    assert (host["accepted"] > 0).all()
