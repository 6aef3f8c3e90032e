"""viml_solve_vi: a whole Levenberg-Marquardt solve per window on the device.

The reference is a host loop per window: Context.gn_step_vi on that window sliced out alone, driven by the scalar policy of
tests/solve_policy.py.  Without point and line factors every kernel of a step is order-deterministic and a window solved in a batch
equals the same window solved alone, so the device loop must reproduce the host loop bit for bit: trace, status, counters, radius
and final state.  With point and line factors the visual pose blocks are summed through shared-memory atomics, so the decisions
must agree and the values to 1e-9."""
import copy
import ctypes as C
import math

import numpy as np
import pytest

import inertial_oracle as io
import solve_policy as sp
from conftest import rel_err
from vi_helpers import bits, device_structs, guard_all, inertial_only, rotate, slice_vi, solve_device

pytestmark = pytest.mark.gpu

FLAGS = 0x10   # VIML_LOSS_CAUCHY
STATE = ("poses", "ex_pose", "inv_depth", "extra")


def _case(pkg, W=8, seed=5, P=11, F=40, no_imu=(2,), perturb=(0.002, 0.01, 0.05, 0.5, 1.0)):
    """W windows; window w's state is moved away from the one the factors were built at by perturb[w % len(perturb)].  The
    synthetic problem is close to quadratic, so step quality stays near 1; far from the solution it drops to about 0.94, which a
    strict min_relative_decrease rejects.  Windows in no_imu carry the prior only: their system is singular."""
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


def _norms(b, ex, o):
    """|dx| (the reduced step and the landmark increments x+ - x) and |x| (every state value)."""
    step = math.sqrt(float(np.sum(o["dx"][0] ** 2) + np.sum((o["inv_depth"][0] - b.inv_depth[0]) ** 2)))
    x = math.sqrt(float(np.sum(b.poses ** 2) + np.sum(b.ex_pose ** 2) + np.sum(b.inv_depth ** 2) + np.sum(ex ** 2)))
    return step, x


def _policy_loop(step, batch1, extra1, opt):
    """One window (batch1, extra1 of one window) driven by solve_policy through step(batch, extra, lambda) -> gn_step dict."""
    b, ex = copy.deepcopy(batch1), extra1.copy()
    st, trace = None, []
    while st is None or st.status is None:
        o = step(b, ex, 1.0 / opt.initial_radius if st is None else sp.lam(st))
        if st is None:
            st = sp.start(o["cost"][0, 0], opt)
            if st.status is not None:
                break
        acc, row = sp.advance(st, opt, *o["cost"][0], int(o["solved"][0]), *_norms(b, ex, o))
        trace.append(row)
        if acc:
            b.poses[...], b.ex_pose[...], b.inv_depth[...], ex[...] = o["poses"], o["ex_pose"], o["inv_depth"], o["extra"]
    tr = np.full((opt.max_iterations, 4), np.nan)
    if trace:
        tr[:len(trace)] = trace
    return {"poses": b.poses[0], "ex_pose": b.ex_pose[0], "inv_depth": b.inv_depth[0], "extra": ex[0], "status": st.status,
            "iterations": st.iterations, "accepted": st.accepted, "cost": np.array([st.f0, st.f]), "radius": st.radius, "trace": tr}


def _host_loop(pkg, ctx, batch, vi, extra, opt, flags=FLAGS):
    """The reference: every window sliced out alone and solved by the policy loop over Context.gn_step_vi."""
    ref = []
    for w in range(batch.W):
        vi1 = slice_vi(pkg, vi, w)
        ref.append(_policy_loop(lambda b, ex, lam: ctx.gn_step_vi(b, vi1, ex, flags, lam=lam),
                                batch.slice_windows(w, w + 1), extra[w:w + 1], opt))
    return ref


def _solve(ctx, batch, vi, extra, opt, flags=FLAGS):
    return ctx.solve_vi(batch, vi, extra, flags, **vars(opt))


def _check_exact(got, ref):
    for w, r in enumerate(ref):
        for k in STATE + ("trace", "cost"):
            assert np.array_equal(bits(got[k][w]), bits(np.asarray(r[k], dtype=np.float64))), (w, k)
        assert (got["status"][w], got["iterations"][w], got["accepted"][w]) == (r["status"], r["iterations"], r["accepted"]), w
        assert got["radius"][w] == r["radius"], w


def _decisions(trace, iterations, opt):
    """The accept / reject sequence of every step but the last (which may have stopped on a tolerance instead): a valid step whose
    quality rho is above min_relative_decrease was accepted.  An unsolved step reports a model decrease of exactly 0."""
    return [bool(math.isfinite(fp) and m > 0.0 and (f - fp) / m > opt.min_relative_decrease)
            for f, fp, m, _ in trace[:max(int(iterations) - 1, 0)]]


def _check_close(got, ref, opt, tol=1e-9):
    for w, r in enumerate(ref):
        assert (got["status"][w], got["iterations"][w], got["accepted"][w]) == (r["status"], r["iterations"], r["accepted"]), w
        n = int(r["iterations"])
        assert rel_err(got["trace"][w, :n], r["trace"][:n]) < tol, w
        assert np.all(np.isnan(got["trace"][w, n:])), w
        assert _decisions(got["trace"][w], n, opt) == _decisions(r["trace"], n, opt), w
        for k in STATE:
            assert rel_err(got[k][w], r[k]) < tol, (w, k)
        assert rel_err(got["cost"][w], r["cost"]) < tol and abs(got["radius"][w] - r["radius"]) <= tol * r["radius"], w


def test_host_loop_equality_inertial_only(pkg, ctx):
    """Bit for bit against the host loop; the batch covers FAILURE (the window without IMU factors, state unchanged),
    NO_CONVERGENCE (a small cap), rejected steps and tolerance stops."""
    batch, vi, extra = _case(pkg)
    b = inertial_only(pkg, batch)
    seen, rejected = set(), 0
    for opt in (sp.Options(max_iterations=12), sp.Options(max_iterations=3),
                sp.Options(max_iterations=12, parameter_tolerance=1e-4, max_consecutive_invalid=2, min_relative_decrease=0.999)):
        got = _solve(ctx, b, vi, extra, opt)
        ref = _host_loop(pkg, ctx, b, vi, extra, opt)
        _check_exact(got, ref)
        seen |= set(int(s) for s in got["status"])
        rejected += sum(d is False for w in range(b.W) if got["status"][w] != sp.FAILURE
                        for d in _decisions(got["trace"][w], got["iterations"][w], opt))
    assert rejected > 0
    assert got["status"][2] == sp.FAILURE and got["accepted"][2] == 0
    for k in STATE:
        assert np.array_equal(bits(got[k][2]), bits({"poses": b.poses, "ex_pose": b.ex_pose, "inv_depth": b.inv_depth,
                                                        "extra": extra}[k][2])), k
    assert {sp.FAILURE, sp.NO_CONVERGENCE} <= seen and seen & {sp.FUNCTION_TOL, sp.PARAMETER_TOL}


def test_host_loop_with_point_and_line_factors(pkg, ctx):
    batch, vi, extra = _case(pkg, W=6, seed=13, no_imu=())
    opt = sp.Options(max_iterations=8)
    got = _solve(ctx, batch, vi, extra, opt)
    ref = _host_loop(pkg, ctx, batch, vi, extra, opt)
    _check_close(got, ref, opt)
    assert (got["accepted"] > 0).all()


def test_against_cpu_oracle(pkg, orc, ctx, cfg):
    from oracle import gn_oracle
    batch, vi, extra = _case(pkg, W=2, seed=21, no_imu=(), perturb=(0.01, 0.03))
    opt = sp.Options(max_iterations=4)
    got = _solve(ctx, batch, vi, extra, opt)
    for w in range(2):
        vi1 = slice_vi(pkg, vi, w)
        ref = _policy_loop(lambda b, ex, lam: io.gn_step_vi(orc, gn_oracle, cfg, b, vi1, ex, FLAGS, lam=lam),
                           batch.slice_windows(w, w + 1), extra[w:w + 1], opt)
        _check_close({k: v[w:w + 1] for k, v in got.items()}, [ref], opt)


def test_host_loop_equality_unfused(pkg, ctx):
    """Dx = 201 (P = 13): the separate reduced-system and solve kernels."""
    batch, vi, extra = _case(pkg, W=4, seed=33, P=13, F=20, no_imu=(1,))
    assert batch.D + vi.X == 201
    b = inertial_only(pkg, batch)
    opt = sp.Options(max_iterations=10)
    got = _solve(ctx, b, vi, extra, opt)
    _check_exact(got, _host_loop(pkg, ctx, b, vi, extra, opt))
    assert got["status"][1] == sp.FAILURE


def test_one_iteration_is_one_step(pkg, ctx):
    batch, vi, extra = _case(pkg)
    for b, ok in ((inertial_only(pkg, batch), True), (batch, False)):   # bit for bit without point and line factors
        got = _solve(ctx, b, vi, extra, sp.Options(max_iterations=1))
        one = ctx.gn_step_vi(b, vi, extra, FLAGS, lam=1.0 / 1e4)
        if ok:
            assert np.array_equal(got["trace"][:, 0, :3], one["cost"]) and np.all(got["trace"][:, 0, 3] == 1e-4)
        else:
            assert rel_err(got["trace"][:, 0, :3], one["cost"]) < 1e-12
        assert np.all(got["iterations"] == 1)
        for k in STATE:
            start = {"poses": b.poses, "ex_pose": b.ex_pose, "inv_depth": b.inv_depth, "extra": extra}[k]
            for w in range(b.W):
                want = one[k][w] if got["accepted"][w] else start[w]
                assert np.array_equal(got[k][w], want) if ok else rel_err(got[k][w], want) < 1e-12, (k, w)
        assert got["accepted"].sum() > 0 and (got["accepted"] == 0).any()


def test_device_pointers(pkg, ctx):
    batch, vi, extra = _case(pkg, W=6, seed=41)
    b = inertial_only(pkg, batch)
    opt = sp.Options(max_iterations=8)
    host = _solve(ctx, b, vi, extra, opt)
    for _ in range(2):   # and two calls repeat bit for bit
        dev = solve_device(pkg, ctx, b, vi, extra, opt, FLAGS)
        for k in host:
            assert np.array_equal(bits(dev[k]), bits(host[k])), k


def test_nan_in_one_window(pkg, ctx):
    batch, vi, extra = _case(pkg, W=6, seed=51, no_imu=())
    b = inertial_only(pkg, batch)
    opt = sp.Options(max_iterations=6)
    clean = _solve(ctx, b, vi, extra, opt)
    bad = copy.deepcopy(b)
    bad.poses[3, 4, 1] = np.nan
    got = _solve(ctx, bad, vi, extra, opt)
    assert got["status"][3] == sp.FAILURE and got["iterations"][3] == 0 and got["accepted"][3] == 0
    assert np.isnan(got["cost"][3]).all() and np.isnan(got["trace"][3]).all() and got["radius"][3] == 1e4
    start = {"poses": bad.poses, "ex_pose": bad.ex_pose, "inv_depth": bad.inv_depth, "extra": extra}
    for k in STATE:
        assert np.array_equal(bits(got[k][3]), bits(start[k][3])), k
    others = [w for w in range(b.W) if w != 3]
    for k in clean:
        assert np.array_equal(bits(got[k][others]), bits(clean[k][others])), k


def test_validation(pkg, ctx):
    batch, vi, extra = _case(pkg, W=2, seed=61, no_imu=())
    b = inertial_only(pkg, batch)
    bad_options = [dict(max_iterations=0), dict(max_consecutive_invalid=-1), dict(min_radius=0.0), dict(min_radius=-1.0),
                   dict(initial_radius=1e-40), dict(initial_radius=1e17), dict(max_radius=math.inf), dict(initial_radius=math.nan),
                   dict(min_relative_decrease=-1e-3), dict(function_tolerance=-1.0), dict(parameter_tolerance=-1.0),
                   dict(function_tolerance=math.nan)]
    for kw in bad_options:
        with pytest.raises(pkg.VimlError, match="error -1"):
            ctx.solve_vi(b, vi, extra, FLAGS, **{"max_iterations": 3, **kw})
    # the device flavour refuses the same from the structs alone (every pointer a real device buffer)
    ins, gi, s, v = device_structs(ctx, b, vi, extra)
    W = b.W
    outs = {"poses": np.zeros_like(b.poses), "ex_pose": np.zeros_like(b.ex_pose), "inv_depth": np.zeros_like(b.inv_depth),
            "extra": np.zeros((W, vi.X)), "status": np.zeros(W, np.int32), "iterations": np.zeros(W, np.int32),
            "accepted": np.zeros(W, np.int32), "cost": np.zeros((W, 2)), "radius": np.zeros(W), "trace": np.zeros((W, 3, 4))}
    go = guard_all(ctx, outs)

    def call(opt, drop=None, flags=FLAGS | pkg.PTRS_DEVICE, n_windows=None):
        o = pkg._abi.SolveOut()
        for k in outs:
            setattr(o, k, None if k == drop else go[k].ptr)
        s2 = pkg._abi.WindowBatch.from_buffer_copy(s)
        if n_windows is not None:
            s2.n_windows = n_windows
        return ctx.lib.viml_solve_vi(ctx.h, C.byref(s2), C.byref(v), gi["extra"].ptr, C.byref(opt), C.byref(o), flags)

    for kw in bad_options:
        assert call(ctx.solve_options(**{"max_iterations": 3, **kw})) == pkg._abi.VIML_ERR_INVALID, kw
    for k in ("poses", "ex_pose", "inv_depth", "extra", "status", "iterations", "accepted", "cost"):
        assert call(ctx.solve_options(max_iterations=3), drop=k) == pkg._abi.VIML_ERR_INVALID, k
        with pytest.raises(pkg.VimlError, match="error -1"):   # the host flavour
            o = pkg._abi.SolveOut()
            res = {kk: outs[kk].copy() for kk in outs}
            for kk in outs:
                setattr(o, kk, None if kk == k else pkg._abi.ptr(res[kk]))
            ctx._check(ctx.lib.viml_solve_vi(ctx.h, C.byref(b.struct()), C.byref(vi.struct()), pkg._abi.ptr(extra),
                                             C.byref(ctx.solve_options(max_iterations=3)), C.byref(o), FLAGS))
    assert ctx.lib.viml_solve_vi(ctx.h, C.byref(s), C.byref(v), gi["extra"].ptr, None, C.byref(pkg._abi.SolveOut()),
                                 FLAGS | pkg.PTRS_DEVICE) == pkg._abi.VIML_ERR_INVALID
    # W == 0: nothing to do, in both flavours
    assert call(ctx.solve_options(max_iterations=3), n_windows=0) == pkg._abi.VIML_OK
    assert call(ctx.solve_options(max_iterations=3), n_windows=0, drop="radius", flags=FLAGS) == pkg._abi.VIML_OK
    ctx.sync()
    for k, g in go.items():   # nothing was written by the refused calls
        assert np.array_equal(bits(g.check()), bits(outs[k])), k
    for g in list(gi.values()) + list(go.values()):
        g.free()
    # the valid options pass (radius and trace are optional)
    res = ctx.solve_vi(b, vi, extra, FLAGS, max_iterations=2, min_radius=1e4, initial_radius=1e4, max_radius=1e4)
    assert (res["iterations"] >= 1).all()
