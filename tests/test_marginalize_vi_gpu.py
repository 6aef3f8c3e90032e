"""viml_marginalize_vi: the next prior of every window, marginalised on the device.

The oracle builds each window's dense problem from independent pieces: the C++ oracle's window_dense for the selected point factors,
tests/inertial_oracle.py for the IMU factors, the C++ oracle's MarginalizationFactor::Evaluate for the prior, added by the
ThreadsConstructA rule in the order [marginalised blocks, landmarks | kept blocks] of tests/marg_vi_policy.py, then the C++ oracle's
MarginalizationInfo::marginalize.  Eigenvector signs are not unique, so the returned prior is compared as J^T J and J^T r, per 6 x 6
block and 6-vector (parity.unit_err; the bar of DESIGN.md section 2 for outputs of two eigen-decompositions)."""
import ctypes as C

import numpy as np
import pytest

import inertial_oracle as io
import marg_reference as mr
import marg_vi_policy as mp
from vi_helpers import bits, guard_all, inertial_only, slice_vi

pytestmark = pytest.mark.gpu

FLAGS = 0x10   # VIML_LOSS_CAUCHY
PRIOR = ("prior_n", "prior_jacobian", "prior_residual", "prior_n_blocks", "prior_block", "prior_x0")


def _case(pkg, W=4, seed=3, F=40, realistic=False, **kw):
    batch = pkg.synth.make_windows(W, seed=seed, F=F)
    vi, extra = pkg.synth.make_inertial_factors(batch, seed=seed + 1, realistic=realistic, **kw)
    return batch, vi, extra


def _plan(batch, vi, w, margin):
    p0, p1 = batch.pf_window_offset[w], batch.pf_window_offset[w + 1]
    k0, k1 = vi.imu_window_offset[w], vi.imu_window_offset[w + 1]
    n = int(vi.prior_n[w])
    blocks = vi.prior_block[w, :vi.prior_n_blocks[w]] if n > 0 else np.zeros((0, 4))
    return mp.plan(batch.P, vi.X, margin, batch.pf_idx[p0:p1], vi.imu_pose[k0:k1], vi.imu_preint[k0:k1], blocks)


def _oracle(pkg, orc, cfg, batch, vi, extra, w, margin):
    """(plan, J^T J, J^T r) of the oracle's marginalisation of window w."""
    r, A, b, m = _dense_problem(pkg, orc, cfg, batch, vi, extra, w, margin)
    _, _, lj, lr = orc.marginalize_dense(A, b, m)
    return r, lj.T @ lj, lj.T @ lr


def _dense_problem(pkg, orc, cfg, batch, vi, extra, w, margin):
    """(plan, A, b, m): window w's dense problem in the order [marginalised blocks, landmarks | kept blocks], m its marginalised
    size."""
    P, D, X, F = batch.P, batch.D, vi.X, batch.F
    r = _plan(batch, vi, w, margin)
    N = D + X + F
    H, g = np.zeros((N, N)), np.zeros(N)
    p0, p1 = batch.pf_window_offset[w], batch.pf_window_offset[w + 1]
    sel = np.flatnonzero(r["points"]) + p0
    land = []
    if len(sel):
        b1 = pkg._abi.Batch(batch.poses[w:w + 1], batch.ex_pose[w:w + 1], batch.inv_depth[w:w + 1], [0, len(sel)], batch.pf_idx[sel],
                            batch.pf_obs[sel])
        Hv, bv = orc.window_dense(cfg, b1, 0, FLAGS)
        ix = np.concatenate([np.arange(D), D + X + np.arange(F)])
        H[np.ix_(ix, ix)] += Hv
        g[ix] += bv
        land = sorted(set(int(f) for f in batch.pf_idx[sel] >> 16))
    for k in np.flatnonzero(r["imu"]) + vi.imu_window_offset[w]:
        (i, j), (si, sj) = vi.imu_pose[k], vi.imu_sb[k]
        res, (a, b, c, d) = io.imu_factor_evaluate(batch.poses[w, i], extra[w, si:si + 9], batch.poses[w, j], extra[w, sj:sj + 9],
                                                   vi.imu_preint[k], vi.imu_jacobian[k], vi.imu_sqrt_info[k], vi.gravity)
        J = np.concatenate([a[:, :6], b, c[:, :6], d], axis=1)
        cols = vi.imu_columns(k)
        H[np.ix_(cols, cols)] += J.T @ J
        g[cols] += J.T @ res
    if r["prior"]:
        n = int(vi.prior_n[w])
        ev = io.inertial_evaluate(orc, batch.poses, batch.ex_pose, extra, _slice_all_but(pkg, vi, w), want_jac=False)
        res, J = ev["prior_residual"][w, :n], vi.prior_jacobian[w, :n, :n]
        cols = vi.prior_columns(w)
        H[np.ix_(cols, cols)] += J.T @ J
        g[cols] += J.T @ res
    order = r["drop"] + [D + X + f for f in land] + r["cols"]
    return r, H[np.ix_(order, order)], g[order], len(r["drop"]) + len(land)


def _slice_all_but(pkg, vi, w):
    """vi without IMU factors (the prior of every window is evaluated; only window w's is read)."""
    W = vi.W
    return pkg._abi.Inertial(W, vi.P, vi.X, vi.gravity, np.zeros(W + 1), np.zeros((0, 2)), np.zeros((0, 2)), np.zeros((0, 17)),
                             np.zeros((0, 15, 15)), np.zeros((0, 15, 15)), vi.prior_n, vi.prior_jacobian, vi.prior_residual,
                             vi.prior_n_blocks, vi.prior_block, vi.prior_x0)


def _pad6(a):
    """Zero-pad the trailing dimensions to a multiple of 6 (parity's 6 x 6 / 6-vector units)."""
    n = a.shape[-1]
    k = -n % 6
    return np.pad(a, [(0, 0)] * (a.ndim - 2) + [(0, k)] * min(a.ndim, 2)) if a.ndim == 2 else np.pad(a, (0, k))


def _check_window(pkg, got, w, r, JtJ, Jtr, batch, extra, tol=1e-8):
    n = sum(6 if b[2] == 7 else 9 for b in r["keep"])
    assert got["prior_n"][w] == n and got["prior_n_blocks"][w] == len(r["keep"])
    assert np.array_equal(got["prior_block"][w, :len(r["keep"])], np.array(r["keep"], dtype=np.int32).reshape(-1, 4))
    x0 = mp.x0_rows(batch.P, r["src"], batch.poses[w], batch.ex_pose[w], extra[w])
    assert np.array_equal(bits(got["prior_x0"][w, :len(r["keep"])]), bits(x0))
    J, res = got["prior_jacobian"][w, :n, :n], got["prior_residual"][w, :n]
    e1 = pkg.parity.unit_err("S", _pad6(J.T @ J)[None], _pad6(JtJ)[None])
    e2 = pkg.parity.unit_err("g", _pad6(J.T @ res)[None], _pad6(Jtr)[None])
    return e1, e2


@pytest.mark.parametrize("realistic, tol", [(False, 1e-8), (True, 5e-8)])
def test_margin_old_against_oracle(pkg, orc, ctx, cfg, realistic, tol):
    """realistic=True (EuRoC IMU noise densities: bias rows of the covariance near 1e-11, sqrt_info entries near 3e5) does not reach
    1e-8: measured 3.0e-8 on J^T J and 1.1e-8 on J^T r on one B200 (default covariance: 9e-14 and 2e-14).  Against the
    extended-precision reference of the joint problem (test_margin_old_realistic_against_reference) neither side is exact and
    neither is the outlier: measured on one B200, the device is off by up to 2.6e-8 (J^T J) and 1.2e-8 (J^T r), the oracle by up to
    1.7e-8 and 9.7e-9, so their difference can reach the sum of the two.  Both are about 1e-6 of their normwise bars: the
    marginalised block has kappa ~ 1e10 (bias rows ~1e12 against pose rows ~1e2), and any backward-stable eigen route loses
    ~kappa u there.  The landmarks-first elimination of the device is not the cause: every eigenvalue of the joint Amm is kept,
    so the sequential and the joint pseudo-inverse are the same matrix."""
    batch, vi, extra = _case(pkg, realistic=realistic)
    got = ctx.marginalize_vi(batch, vi, extra, np.zeros(batch.W, np.int32), FLAGS)
    errs = []
    for w in range(batch.W):
        r, JtJ, Jtr = _oracle(pkg, orc, cfg, batch, vi, extra, w, mp.OLD)
        assert len(r["drop"]) == 15 and r["points"].any() and r["imu"].any()
        errs.append(_check_window(pkg, got, w, r, JtJ, Jtr, batch, extra))
    print("realistic", realistic, "max unit errors J^T J, J^T r:", np.max(errs, axis=0))
    assert np.max(errs) < tol


def test_margin_second_new_against_oracle(pkg, orc, ctx, cfg):
    batch, vi, extra = _case(pkg, seed=7)
    got = ctx.marginalize_vi(batch, vi, extra, np.ones(batch.W, np.int32), FLAGS)
    for w in range(batch.W):
        r, JtJ, Jtr = _oracle(pkg, orc, cfg, batch, vi, extra, w, mp.SECOND_NEW)
        assert r["drop"] == list(range(6 * (batch.P - 2), 6 * (batch.P - 1))) and not r["points"].any()
        e1, e2 = _check_window(pkg, got, w, r, JtJ, Jtr, batch, extra)
        assert e1 < 1e-8 and e2 < 1e-8, (w, e1, e2)


def _copy_case(pkg, vi, w):
    """Window w's prior without pose P-2 (MARGIN_SECOND_NEW keeps it unchanged): its pose blocks from pose 1 to P-3 only."""
    P = vi.P
    keep = [b for b in range(vi.prior_n_blocks[w]) if not (vi.prior_block[w, b, 0] == mp.POSE and vi.prior_block[w, b, 1] >= P - 2)]
    cols = np.concatenate([np.arange(vi.prior_block[w, b, 3], vi.prior_block[w, b, 3] + (6 if vi.prior_block[w, b, 2] == 7 else 9))
                           for b in keep])
    n = len(cols)
    vi.prior_jacobian[w] = 0.0
    vi.prior_jacobian[w, :n, :n] = np.eye(n) * 300.0
    vi.prior_residual[w, :n] = vi.prior_residual[w, cols]
    first = 0
    blocks, x0 = [], []
    for b in keep:
        blk = vi.prior_block[w, b].copy()
        blk[3] = first
        first += 6 if blk[2] == 7 else 9
        blocks.append(blk), x0.append(vi.prior_x0[w, b].copy())
    vi.prior_n[w], vi.prior_n_blocks[w] = n, len(keep)
    vi.prior_block[w, :len(keep)], vi.prior_x0[w, :len(keep)] = blocks, x0


def test_mixed_batch_equals_one_window_calls(pkg, ctx):
    """Both kinds, windows without prior, without IMU and without anchor-0 features, and a MARGIN_SECOND_NEW copy.  Without point
    factors every kernel is order-deterministic and a window equals its one-window call bit for bit; the fused assembly sums the
    point factors' pose blocks through shared-memory atomics, so there J^T J and J^T r must agree to 1e-9."""
    batch, vi, extra = _case(pkg, W=8, seed=11, no_imu=(2, 5), no_prior=(3,))
    # window 6: no feature anchored at frame 0 (they start at frame 1)
    p0, p1 = batch.pf_window_offset[6], batch.pf_window_offset[7]
    idx = batch.pf_idx[p0:p1]
    batch.pf_idx[p0:p1] = np.where((idx & 0xff) == 0, idx | 1, idx).astype(np.uint32)
    batch.pf_idx[p0:p1] = np.where(((batch.pf_idx[p0:p1] >> 8) & 0xff) == 1, batch.pf_idx[p0:p1] + (1 << 8), batch.pf_idx[p0:p1])
    _copy_case(pkg, vi, 7)
    margin = np.array([0, 1, 0, 0, 1, 0, 0, 1], np.int32)
    got = ctx.marginalize_vi(batch, vi, extra, margin, FLAGS)
    assert got["prior_n"][7] == vi.prior_n[7]
    n7, nb7 = int(vi.prior_n[7]), int(vi.prior_n_blocks[7])
    assert np.array_equal(got["prior_jacobian"][7, :n7, :n7], vi.prior_jacobian[7, :n7, :n7])
    assert np.array_equal(got["prior_residual"][7, :n7], vi.prior_residual[7, :n7])
    assert np.array_equal(got["prior_block"][7, :nb7], vi.prior_block[7, :nb7]) and np.array_equal(got["prior_x0"][7, :nb7], vi.prior_x0[7, :nb7])
    exact = {1, 4, 7}   # MARGIN_SECOND_NEW: the prior alone
    for w in range(batch.W):
        one = ctx.marginalize_vi(batch.slice_windows(w, w + 1), slice_vi(pkg, vi, w), extra[w:w + 1], margin[w:w + 1], FLAGS)
        n = int(one["prior_n"][0])
        for k in ("prior_n", "prior_n_blocks", "prior_block", "prior_x0"):
            assert np.array_equal(bits(got[k][w]), bits(one[k][0])), (w, k)
        J, r, J1, r1 = got["prior_jacobian"][w, :n, :n], got["prior_residual"][w, :n], one["prior_jacobian"][0, :n, :n], one["prior_residual"][0, :n]
        if w in exact:
            assert np.array_equal(bits(J), bits(J1)) and np.array_equal(bits(r), bits(r1)), w
        else:
            assert pkg.parity.unit_err("S", _pad6(J.T @ J)[None], _pad6(J1.T @ J1)[None]) < 1e-9, w
            assert pkg.parity.unit_err("g", _pad6(J.T @ r)[None], _pad6(J1.T @ r1)[None]) < 1e-9, w
    assert got["prior_n"][6] == 6 * batch.P + 9 and got["prior_n"][3] > 0   # no anchor-0 feature / no prior: still a prior


def test_zero_step_identity(pkg, ctx):
    """The returned prior evaluated at the slid linearisation point: dx = 0 in every position and vector entry; Eigen's
    q0.inverse() * q of q0 == q is the identity up to rounding (|dtheta| ~ 1e-16), so the residual is prior_residual to 1e-12."""
    batch, vi, extra = _case(pkg, W=4, seed=17)
    margin = np.array([0, 1, 0, 1], np.int32)
    got = ctx.marginalize_vi(batch, vi, extra, margin, FLAGS)
    slid = pkg._abi.Batch(batch.poses.copy(), batch.ex_pose, batch.inv_depth, batch.pf_window_offset, batch.pf_idx, batch.pf_obs)
    ex2 = extra.copy()
    for w in range(batch.W):
        slid.poses[w], ex2[w] = mp.slide_state(batch.poses[w], extra[w], margin[w])
    vi2 = pkg._abi.Inertial(vi.W, vi.P, vi.X, vi.gravity, np.zeros(vi.W + 1), np.zeros((0, 2)), np.zeros((0, 2)), np.zeros((0, 17)),
                            np.zeros((0, 15, 15)), np.zeros((0, 15, 15)), got["prior_n"], np.nan_to_num(got["prior_jacobian"]),
                            np.nan_to_num(got["prior_residual"]), got["prior_n_blocks"], np.maximum(got["prior_block"], 0),
                            np.nan_to_num(got["prior_x0"]))
    ev = ctx.inertial_evaluate(slid, ex2, vi2)
    for w in range(batch.W):
        n = int(got["prior_n"][w])
        assert n > 0
        r0 = got["prior_residual"][w, :n]
        assert np.abs(ev["prior_residual"][w, :n] - r0).max() <= 1e-12 * np.abs(r0).max(), w


def test_two_frame_chain_device_pointers(pkg, ctx):
    """solve, marginalise with device pointers, slide (numpy), solve with the new prior: equal to the host-pointer chain bit for bit
    (no point factors: every kernel is order-deterministic), and no window fails because of the prior."""
    batch, vi, extra = _case(pkg, W=6, seed=23)
    b = inertial_only(pkg, batch)
    margin = np.array([0, 0, 1, 0, 1, 0], np.int32)

    def chain(device):
        s1 = ctx.solve_vi(b, vi, extra, FLAGS, max_iterations=6)
        assert (s1["status"] != pkg._abi.SOLVE_FAILURE).all()
        b1 = pkg._abi.Batch(s1["poses"], s1["ex_pose"], s1["inv_depth"], b.pf_window_offset, b.pf_idx, b.pf_obs)
        prior = _marg_device(pkg, ctx, b1, vi, s1["extra"], margin)[0] if device else ctx.marginalize_vi(b1, vi, s1["extra"], margin, FLAGS)
        b2 = pkg._abi.Batch(b1.poses.copy(), b1.ex_pose, b1.inv_depth, b.pf_window_offset, b.pf_idx, b.pf_obs)
        e2 = s1["extra"].copy()
        for w in range(b.W):
            b2.poses[w], e2[w] = mp.slide_state(b1.poses[w], s1["extra"][w], margin[w])
        mb = prior["prior_block"].shape[1]
        vi2 = pkg._abi.Inertial(vi.W, vi.P, vi.X, vi.gravity, vi.imu_window_offset, vi.imu_pose, vi.imu_sb, vi.imu_preint, vi.imu_jacobian,
                                vi.imu_sqrt_info, prior["prior_n"], np.nan_to_num(prior["prior_jacobian"]),
                                np.nan_to_num(prior["prior_residual"]), prior["prior_n_blocks"], np.maximum(prior["prior_block"], 0)[:, :mb],
                                np.nan_to_num(prior["prior_x0"]))
        s2 = ctx.solve_vi(b2, vi2, e2, FLAGS, max_iterations=6)
        return prior, s2

    p_host, s_host = chain(False)
    p_dev, s_dev = chain(True)
    for k in PRIOR:
        assert np.array_equal(bits(p_dev[k]), bits(p_host[k])), k
    for k in s_host:
        assert np.array_equal(bits(s_dev[k]), bits(s_host[k])), k
    assert (s_host["status"] != pkg._abi.SOLVE_FAILURE).all() and (s_host["accepted"] > 0).all()


def _marg_device(pkg, ctx, batch, vi, extra, margin, n_max=None):
    """viml_marginalize_vi with VIML_PTRS_DEVICE on guarded device copies of every input and output: (outputs, inputs unchanged)."""
    W, P = batch.W, batch.P
    n_max = vi.n_max if n_max is None else n_max
    mb = 2 * P + 1
    b_in = {k: a for k, a in batch.arrays().items() if a is not None}
    ins = {**{"b_" + k: a for k, a in b_in.items()}, **{"v_" + k: a for k, a in vi.arrays().items()}, "extra": extra,
           "margin": np.ascontiguousarray(margin, np.int32)}
    gi = guard_all(ctx, ins)
    s = batch.struct({**batch.arrays(), **{k: gi["b_" + k].ptr for k in b_in}})
    v = vi.struct({k: gi["v_" + k].ptr for k in vi.arrays()})
    outs = {"prior_n": np.full(W, -1, np.int32), "prior_jacobian": np.full((W, n_max, n_max), np.nan), "prior_residual": np.full((W, n_max), np.nan),
            "prior_n_blocks": np.full(W, -1, np.int32), "prior_block": np.full((W, mb, 4), -1, np.int32), "prior_x0": np.full((W, mb, 9), np.nan)}
    go = guard_all(ctx, outs)
    o = pkg._abi.PriorOut()
    o.prior_n_max, o.prior_max_blocks = n_max, mb
    for k in outs:
        setattr(o, k, go[k].ptr)
    ctx._check(ctx.lib.viml_marginalize_vi(ctx.h, C.byref(s), C.byref(v), gi["extra"].ptr, gi["margin"].ptr, C.byref(o),
                                           FLAGS | pkg.PTRS_DEVICE))
    ctx.sync()
    res = {k: g.check() for k, g in go.items()}
    same = all(np.array_equal(bits(g.check()), bits(ins[k])) for k, g in gi.items())
    for g in list(gi.values()) + list(go.values()):
        g.free()
    return res, same


def test_device_pointers_guard_bands(pkg, ctx):
    batch, vi, extra = _case(pkg, W=5, seed=29, no_imu=(1,), no_prior=(2,))
    margin = np.array([0, 0, 0, 1, 1], np.int32)
    b = inertial_only(pkg, batch)   # deterministic kernels: the flavours agree bit for bit
    host = ctx.marginalize_vi(b, vi, extra, margin, FLAGS)
    dev, same = _marg_device(pkg, ctx, b, vi, extra, margin)
    assert same, "an input changed"
    for k in PRIOR:
        assert np.array_equal(bits(dev[k]), bits(host[k])), k
    # with point factors (the observation table too): inputs untouched, nothing written outside the outputs
    dev, same = _marg_device(pkg, ctx, batch, vi, extra, margin)
    assert same and (dev["prior_n"] >= 0).all()


def test_observation_forms_agree(pkg, ctx):
    batch, vi, extra = _case(pkg, W=3, seed=31)
    margin = np.zeros(3, np.int32)
    ref = ctx.marginalize_vi(batch, vi, extra, margin, FLAGS)
    for form in (True,):
        got = ctx.marginalize_vi(batch, vi, extra, margin, FLAGS, obs_table=form)
        for w in range(3):
            n = int(ref["prior_n"][w])
            assert got["prior_n"][w] == n
            J, r, J1, r1 = got["prior_jacobian"][w, :n, :n], got["prior_residual"][w, :n], ref["prior_jacobian"][w, :n, :n], ref["prior_residual"][w, :n]
            assert pkg.parity.unit_err("S", _pad6(J.T @ J)[None], _pad6(J1.T @ J1)[None]) < 1e-9


def test_validation(pkg, ctx):
    batch, vi, extra = _case(pkg, W=2, seed=37)
    margin = np.zeros(2, np.int32)

    def refused(b=batch, v=vi, e=extra, mg=margin, **kw):
        with pytest.raises(pkg.VimlError, match="error -1"):
            ctx.marginalize_vi(b, v, e, mg, FLAGS, **kw)

    refused(mg=np.array([0, 2], np.int32))
    refused(n_max=60)                       # the kept dimension (75) does not fit
    refused(max_blocks=4)                   # nor the block count (12)
    v = slice_vi(pkg, vi, 0)
    v = pkg._abi.Inertial(1, v.P, v.X, v.gravity, v.imu_window_offset, v.imu_pose, v.imu_sb.copy(), v.imu_preint, v.imu_jacobian,
                          v.imu_sqrt_info, v.prior_n, v.prior_jacobian, v.prior_residual, v.prior_n_blocks, v.prior_block.copy(), v.prior_x0)
    b1, e1 = batch.slice_windows(0, 1), extra[:1]
    v.imu_sb[0, 1] = 9 * 5                  # not 9 j
    refused(b1, v, e1, margin[:1])
    v.imu_sb[0, 1] = 9
    v.prior_block[0, -1, 1] = 10            # an extra block not at 9p
    refused(b1, v, e1, margin[:1])
    v.prior_block[0, -1, 1] = 9 * (v.P - 2)   # speed-bias P-2 in a MARGIN_SECOND_NEW prior
    refused(b1, v, e1, np.ones(1, np.int32))
    v.prior_block[0, -1, 1] = 9
    ctx.marginalize_vi(b1, v, e1, margin[:1], FLAGS)   # restored: accepted
    # a feature with factors both at i == 0 and i != 0
    b2 = batch.slice_windows(0, 1)
    k = int(np.flatnonzero((b2.pf_idx & 0xff) == 0)[0])
    f = int(b2.pf_idx[k] >> 16)
    b2.pf_idx = np.concatenate([b2.pf_idx, np.array([2 | (3 << 8) | (f << 16)], np.uint32)])
    b2.pf_obs = np.concatenate([b2.pf_obs, b2.pf_obs[:1]])
    b2.pf_window_offset = np.array([0, len(b2.pf_idx)], np.int32)
    b2.lf_window_offset = np.zeros(2, np.int32)
    b2.lf_frame, b2.lf_geom = np.zeros(0, np.int32), np.zeros((9, 0))
    refused(b2, v, e1, margin[:1])
    # P < 2
    b3 = pkg._abi.Batch(batch.poses[:1, :1], batch.ex_pose[:1], batch.inv_depth[:1], [0, 0], np.zeros(0, np.uint32), np.zeros((0, 4)))
    v3 = pkg._abi.Inertial(1, 1, 9, vi.gravity, [0, 0], np.zeros((0, 2)), np.zeros((0, 2)), np.zeros((0, 17)), np.zeros((0, 15, 15)),
                           np.zeros((0, 15, 15)), [0], np.zeros((1, 1, 1)), np.zeros((1, 1)), [0], np.zeros((1, 1, 4)), np.zeros((1, 1, 9)))
    refused(b3, v3, np.zeros((1, 9)), margin[:1])
    # W == 0
    b0 = pkg._abi.Batch(np.zeros((0, 11, 7)), np.zeros((0, 7)), np.zeros((0, 4)), [0], np.zeros(0, np.uint32), np.zeros((0, 4)))
    o = pkg._abi.PriorOut()
    assert ctx.lib.viml_marginalize_vi(ctx.h, C.byref(b0.struct()), C.byref(vi.struct()), pkg._abi.ptr(extra), None, C.byref(o), 0) == 0



def test_margin_old_realistic_against_reference(pkg, orc, ctx, cfg):
    """The realistic windows' priors, the device's and the C++ oracle's, each against the extended-precision reference of the joint
    problem (tests/marg_reference.py) under the bars of tests/test_marginalize_dense_gpu.py.  The device eliminates the landmarks
    first (an exact diagonal inverse) and then pose 0 and speed-bias 0 by a 15 x 15 pseudo-inverse; that equals the joint
    pseudo-inverse because every eigenvalue of the joint Amm is kept, well above eps (checked: the smallest is ~1e2 against
    eps = 1e-8 and a perturbation band of a few units).  Its rounding is held to the joint route's bar with the device's sweep
    cap: the landmark step rounds each entry of the Schur complement as the joint route's products do, and its Jacobi is smaller."""
    batch, vi, extra = _case(pkg, realistic=True)
    got = ctx.marginalize_vi(batch, vi, extra, np.zeros(batch.W, np.int32), FLAGS)
    for w in range(batch.W):
        r, A, b, m = _dense_problem(pkg, orc, cfg, batch, vi, extra, w, mp.OLD)
        ref = mr.marginalize(A, b, m)
        im = ref["Amm_info"]
        assert im["kept"].all() and not im["undecidable"] and im["dist_eps"] > 10 * im["band"], (w, im)
        n = int(got["prior_n"][w])
        J, res = got["prior_jacobian"][w, :n, :n], got["prior_residual"][w, :n]
        As, bs, lj, lr = orc.marginalize_dense(A, b, m)
        q_dev = mr.check(ref, None, None, J, res, 40, ("device", w))
        q_orc = mr.check(ref, As, bs, lj, lr, 60, ("oracle", w))
        RJ, Rr = _pad6(ref["JtJ"].astype(np.float64))[None], _pad6(ref["Jtr"].astype(np.float64))[None]
        print("window", w, "unit errors J^T J, J^T r against the reference: device",
              pkg.parity.unit_err("S", _pad6(J.T @ J)[None], RJ), pkg.parity.unit_err("g", _pad6(J.T @ res)[None], Rr),
              "oracle", pkg.parity.unit_err("S", _pad6(lj.T @ lj)[None], RJ), pkg.parity.unit_err("g", _pad6(lj.T @ lr)[None], Rr),
              "error / bar: device", q_dev, "oracle", q_orc)
