"""viml_inertial_evaluate and viml_gn_step_vi on the device: per-factor parity with the CPU oracle (tests/inertial_oracle.py),
bit-for-bit equivalence with viml_gn_step fed the same evaluated blocks, the step against the oracle's, a short solve, and
host-path validation."""
import copy
import ctypes as C

import numpy as np
import pytest

import inertial_oracle as io
from conftest import rel_err
from vi_helpers import device_structs, guard_all, inertial_only, rotate

pytestmark = pytest.mark.gpu


def _case(pkg, W=6, seed=31, extra_pad=0, F=40, gaps=True, perturb=0.0):
    """A non-adjacent IMU factor and a prior whose q0^-1 q has w < 0; with gaps, windows without IMU factors (2) and without a prior
    (3) in the middle of the batch (their systems are then singular: evaluation only).  perturb moves the state away from the
    one the factors were built at."""
    batch = pkg.synth.make_windows(W, seed=seed, F=F)
    vi, extra = pkg.synth.make_inertial_factors(batch, seed=seed + 1, no_imu=(2,) if gaps else (), no_prior=(3,) if gaps else (),
                                                extra_pad=extra_pad)
    k = int(vi.imu_window_offset[0]) + 3
    vi.imu_pose[k] = (3, 5)          # pose 3 -> pose 5 (pose 4 keeps its factor with pose 5)
    vi.imu_sb[k] = (27, 45)
    vi.prior_x0[min(1, W - 1), 2, 3:7] *= -1.0   # same rotation, w < 0 in q0^-1 q
    if perturb:
        rng = np.random.default_rng(seed + 2)
        batch.poses[..., :3] += perturb * rng.standard_normal(batch.poses[..., :3].shape)
        for w in range(batch.W):
            for p in range(batch.P):
                batch.poses[w, p] = rotate(batch.poses[w, p], 0.5 * perturb * rng.standard_normal(3))
        extra = extra + perturb * rng.standard_normal(extra.shape)
    return batch, vi, extra


def _check_eval(got, ref, vi):
    for k in range(vi.NI):
        assert rel_err(got["imu_residual"][k], ref["imu_residual"][k]) < 1e-9
        for name in ("imu_jac_pose_i", "imu_jac_sb_i", "imu_jac_pose_j", "imu_jac_sb_j"):
            assert rel_err(got[name][k], ref[name][k]) < 1e-9, (name, k)
        assert np.all(got["imu_jac_pose_i"][k][:, 6] == 0.0) and np.all(got["imu_jac_pose_j"][k][:, 6] == 0.0)
    for w in range(vi.W):
        n = int(vi.prior_n[w])
        assert rel_err(got["prior_residual"][w, :n], ref["prior_residual"][w, :n]) < 1e-9
        assert np.all(np.isnan(got["prior_residual"][w, n:]))   # rows past n_w keep the caller's content


def test_evaluate_parity_host(pkg, orc, ctx):
    batch, vi, extra = _case(pkg, extra_pad=5)
    got = ctx.inertial_evaluate(batch, extra, vi)
    ref = io.inertial_evaluate(orc, batch.poses, batch.ex_pose, extra, vi)
    _check_eval(got, ref, vi)


def _check_inputs(g, arrays):
    """Inputs come back unchanged and nothing around them was written."""
    for k, v in g.items():
        if v is not None:
            assert np.array_equal(v.check().view(np.uint8), np.ascontiguousarray(arrays[k]).view(np.uint8)), k


def test_evaluate_parity_device(pkg, orc, ctx):
    """VIML_PTRS_DEVICE: the same results, every output written inside its buffer, every input left as it was."""
    batch, vi, extra = _case(pkg, seed=41, extra_pad=3)
    ref = io.inertial_evaluate(orc, batch.poses, batch.ex_pose, extra, vi)
    ins = {"poses": batch.poses, "ex_pose": batch.ex_pose, "extra": extra, **vi.arrays()}
    gi = guard_all(ctx, ins)
    s = batch.struct({**batch.arrays(), "poses": gi["poses"].ptr, "ex_pose": gi["ex_pose"].ptr})
    v = vi.struct({k: gi[k].ptr for k in vi.arrays()})
    got = {"imu_residual": np.full((vi.NI, 15), np.nan), "imu_jac_pose_i": np.full((vi.NI, 15, 7), np.nan),
           "imu_jac_sb_i": np.full((vi.NI, 15, 9), np.nan), "imu_jac_pose_j": np.full((vi.NI, 15, 7), np.nan),
           "imu_jac_sb_j": np.full((vi.NI, 15, 9), np.nan), "prior_residual": np.full((vi.W, vi.n_max), np.nan)}
    go = guard_all(ctx, got)
    o = pkg._abi.InertialOut()
    for k in got:
        setattr(o, k, go[k].ptr)
    ctx._check(ctx.lib.viml_inertial_evaluate(ctx.h, C.byref(s), gi["extra"].ptr, C.byref(v), C.byref(o), pkg.PTRS_DEVICE))
    ctx.sync()
    got = {k: g.check() for k, g in go.items()}
    _check_inputs(gi, ins)
    for g in list(gi.values()) + list(go.values()):
        g.free()
    _check_eval(got, ref, vi)
    # repeatable bit for bit (no order-dependent accumulation in these kernels)
    again = ctx.inertial_evaluate(batch, extra, vi)
    host = ctx.inertial_evaluate(batch, extra, vi)
    for k in got:
        assert np.array_equal(again[k], host[k], equal_nan=True) and np.array_equal(got[k], host[k], equal_nan=True), k


def _gn_step_vi_device(pkg, ctx, batch, vi, extra, flags, lam):
    """viml_gn_step_vi with VIML_PTRS_DEVICE on guarded device copies of every input and output."""
    X, W, Dx = vi.X, batch.W, batch.D + vi.X
    ins, gi, s, v = device_structs(ctx, batch, vi, extra)
    outs = {"poses": np.full_like(batch.poses, np.nan), "ex_pose": np.full_like(batch.ex_pose, np.nan),
            "inv_depth": np.full_like(batch.inv_depth, np.nan), "extra": np.full((W, X), np.nan),
            "dx": np.full((W, Dx), np.nan), "cost": np.full((W, 3), np.nan), "solved": np.full(W, -1, dtype=np.int32)}
    go = guard_all(ctx, outs)
    opt = pkg._abi.GnOptions()
    opt.lambda_ = lam
    o = pkg._abi.GnOut()
    for k in outs:
        setattr(o, k, go[k].ptr)
    ctx._check(ctx.lib.viml_gn_step_vi(ctx.h, C.byref(s), C.byref(v), gi["extra"].ptr, C.byref(opt), C.byref(o),
                                       flags | pkg.PTRS_DEVICE))
    ctx.sync()
    res = {k: g.check() for k, g in go.items()}
    _check_inputs(gi, ins)
    for g in list(gi.values()) + list(go.values()):
        g.free()
    return res


def test_gn_step_vi_device_pointers(pkg, ctx):
    """VIML_PTRS_DEVICE against the host-pointer flavour on the same inputs: bit for bit without point / line factors (every
    kernel on the path is then order-deterministic), to 1e-12 with them (the visual pose blocks are summed through shared-memory
    atomics).  Outputs are written inside their buffers only, inputs are left unchanged."""
    batch, vi, extra = _case(pkg, seed=91, gaps=False, perturb=0.01)
    flags = pkg.LOSS_CAUCHY
    for b_, exact in ((inertial_only(pkg, batch), True), (batch, False)):
        h = ctx.gn_step_vi(b_, vi, extra, flags, lam=1e-3)
        d = _gn_step_vi_device(pkg, ctx, b_, vi, extra, flags, 1e-3)
        assert h["solved"].all() and np.array_equal(h["solved"], d["solved"])
        for k in ("dx", "poses", "ex_pose", "inv_depth", "extra", "cost"):
            assert np.array_equal(h[k], d[k]) if exact else rel_err(d[k], h[k]) < 1e-12, k
        if exact:   # and repeatable
            h2 = ctx.gn_step_vi(b_, vi, extra, flags, lam=1e-3)
            assert all(np.array_equal(h[k], h2[k]) for k in h)


def test_gn_step_vi_equals_gn_step_on_evaluated_blocks(pkg, ctx):
    """viml_gn_step_vi(x) against viml_gn_step(x) fed the blocks of viml_inertial_evaluate(x) in the same order.  Without point and
    line factors identical inputs go through identical deterministic kernels: bit for bit.  With them, the visual pose blocks are
    summed through shared-memory atomics in whatever order the warps finish (two viml_gn_step calls repeat to rounding only), so
    the full batch is held to 1e-12."""
    batch, vi, extra = _case(pkg, seed=51, gaps=False, perturb=0.01)
    flags = pkg.LOSS_CAUCHY
    dense = vi.to_dense(ctx.inertial_evaluate(batch, extra, vi))
    for b_, exact in ((inertial_only(pkg, batch), True), (batch, False)):
        a = ctx.gn_step_vi(b_, vi, extra, flags, lam=1e-3)
        b = ctx.gn_step(b_, dense, extra, flags, lam=1e-3)
        assert a["solved"].all() and np.array_equal(a["solved"], b["solved"])
        for k in ("dx", "poses", "ex_pose", "inv_depth", "extra"):
            assert np.array_equal(a[k], b[k]) if exact else rel_err(a[k], b[k]) < 1e-12, k
        if exact:
            assert np.array_equal(a["cost"][:, [0, 2]], b["cost"][:, [0, 2]])
        else:
            assert rel_err(a["cost"][:, [0, 2]], b["cost"][:, [0, 2]]) < 1e-12


@pytest.mark.parametrize("lam", [0.0, 1e-2])
def test_gn_step_vi_against_oracle(pkg, orc, ctx, cfg, lam):
    from oracle import gn_oracle
    batch, vi, extra = _case(pkg, seed=61, gaps=False, perturb=0.01)
    flags = pkg.LOSS_CAUCHY
    got = ctx.gn_step_vi(batch, vi, extra, flags, lam=lam)
    ref = io.gn_step_vi(orc, gn_oracle, cfg, batch, vi, extra, flags, lam=lam)
    assert np.array_equal(got["solved"], ref["solved"]) and got["solved"].all()
    for w in range(batch.W):
        for p in range(batch.P + 1):
            assert rel_err(got["dx"][w, 6 * p:6 * p + 6], ref["dx"][w, 6 * p:6 * p + 6]) < 1e-9
        for e in range(0, vi.X, 9):
            assert rel_err(got["dx"][w, batch.D + e:batch.D + e + 9], ref["dx"][w, batch.D + e:batch.D + e + 9]) < 1e-9
    for k in ("poses", "ex_pose", "inv_depth", "extra"):
        assert rel_err(got[k], ref[k]) < 1e-9, k
    for c in range(3):
        assert np.abs(got["cost"][:, c] - ref["cost"][:, c]).max() < 1e-9 * np.abs(ref["cost"][:, c]).max(), c
    # cost[1] is the nonlinear cost at x+, which differs from viml_gn_step's linear model of the same blocks
    lin = ctx.gn_step(batch, vi.to_dense(ctx.inertial_evaluate(batch, extra, vi)), extra, flags, lam=lam)
    assert np.abs(lin["cost"][:, 1] - got["cost"][:, 1]).max() > 1e-7 * np.abs(got["cost"][:, 1]).max()


def _solve(batch, extra, step, iters=5):
    """Python-driven Levenberg-Marquardt on one window: accept cost[1] < cost[0], lambda / 2 on accept, x 10 on reject.
    Returns the accepted costs and the final state."""
    b, ex, lam = copy.deepcopy(batch), extra.copy(), 1e-3
    costs = []
    for _ in range(iters):
        o = step(b, ex, lam)
        if not costs:
            costs.append(float(o["cost"][0, 0]))
        if o["solved"][0] and o["cost"][0, 1] < o["cost"][0, 0]:
            b.poses[...], b.ex_pose[...], b.inv_depth[...], ex[...] = o["poses"], o["ex_pose"], o["inv_depth"], o["extra"]
            costs.append(float(o["cost"][0, 1]))
            lam *= 0.5
        else:
            lam *= 10.0
    return np.array(costs), b, ex


@pytest.mark.parametrize("seed", [71, 72])
def test_solve_decreases_cost(pkg, orc, ctx, cfg, seed):
    from oracle import gn_oracle
    batch, vi, extra = _case(pkg, W=1, seed=seed, gaps=False, perturb=0.02)
    flags = pkg.LOSS_CAUCHY
    costs, bf, exf = _solve(batch, extra, lambda b, ex, lam: ctx.gn_step_vi(b, vi, ex, flags, lam=lam))
    assert len(costs) >= 3 and np.all(np.diff(costs) < 0.0)
    # the same loop with the IMU and prior blocks frozen at the initial state (viml_gn_step: they enter linearised)
    frozen = vi.to_dense(ctx.inertial_evaluate(batch, extra, vi))
    _, bz, exz = _solve(batch, extra, lambda b, ex, lam: ctx.gn_step(b, frozen, ex, flags, lam=lam))

    def f(b, ex):   # the true cost: visual factors + IMU and prior factors re-evaluated
        return float(gn_oracle.window_cost(cfg, b, flags)[0] + io.inertial_cost(orc, b.poses, b.ex_pose, ex, vi)[0])
    assert abs(f(bf, exf) - costs[-1]) < 1e-9 * costs[0]
    assert f(bf, exf) < f(bz, exz)


def test_validation(pkg, ctx):
    batch, vi, extra = _case(pkg, W=3, seed=81)
    flags = pkg.LOSS_CAUCHY

    def bad(mut):
        v = copy.deepcopy(vi)
        mut(v)
        for call in (lambda: ctx.inertial_evaluate(batch, extra, v), lambda: ctx.gn_step_vi(batch, v, extra, flags)):
            with pytest.raises(pkg.VimlError, match="error -1"):
                call()
    bad(lambda v: v.imu_pose.__setitem__((0, 0), batch.P))              # pose index outside [0, P)
    bad(lambda v: v.imu_pose.__setitem__((0, 1), -1))
    bad(lambda v: v.imu_sb.__setitem__((0, 1), vi.X - 8))               # sb + 9 > X
    bad(lambda v: v.prior_n.__setitem__(0, vi.n_max + 1))               # n_w > n_max
    bad(lambda v: v.prior_block.__setitem__((0, 0, 3), vi.n_max - 3))   # block columns outside [0, n_w)
    bad(lambda v: v.prior_block.__setitem__((0, 0, 2), 6))              # a pose block of size != 7
    bad(lambda v: setattr(v, "X", 233 - batch.D))                       # D + X > 232
    # X < 9 with IMU factors is refused by the device flavour too (it needs no input read back)
    v = copy.deepcopy(vi)
    v.X = 8
    st = v.struct()
    o = pkg._abi.InertialOut()
    rc = ctx.lib.viml_inertial_evaluate(ctx.h, C.byref(batch.struct()), None, C.byref(st), C.byref(o), pkg.PTRS_DEVICE)
    assert rc == pkg._abi.VIML_ERR_INVALID
    ctx.inertial_evaluate(batch, extra, vi)                             # the unmodified input passes
