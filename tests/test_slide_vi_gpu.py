"""viml_slide_vi: the window slide and the depth re-anchoring of every window on the device.

The reference is tests/slide_policy.py, a scalar restatement with the kernel's operation order (IEEE binary64, no fused multiply-add),
so the device must reproduce it bit for bit in every observation form.  The chain test runs solve -> marginalise -> slide -> solve with
device pointers and no host step between the calls, against the same chain with the restatement's slide on the host."""
import ctypes as C

import numpy as np
import pytest

import marg_vi_policy as mp
import slide_policy as sp
from conftest import rel_err
from vi_helpers import bits, guard_all, inertial_only

pytestmark = pytest.mark.gpu

FLAGS = 0x10   # VIML_LOSS_CAUCHY
STATE = ("poses", "ex_pose", "inv_depth", "extra")


def _case(pkg, W=4, seed=3, F=40, **kw):
    batch = pkg.synth.make_windows(W, seed=seed, F=F, f32_obs=True, lines_per_frame=0)
    vi, extra = pkg.synth.make_inertial_factors(batch, seed=seed + 1, extra_pad=3, **kw)
    return batch, vi, extra


def _check_bits(got, ref):
    for k in STATE:
        assert got[k].shape == ref[k].shape and np.array_equal(bits(got[k]), bits(ref[k])), k


def _n_moved(batch, got):
    return int(np.sum(got["inv_depth"] != batch.inv_depth))


@pytest.mark.parametrize("margin", [mp.OLD, mp.SECOND_NEW])
def test_against_restatement(pkg, ctx, margin):
    batch, vi, extra = _case(pkg)
    mg = np.full(batch.W, margin, np.int32)
    got = ctx.slide_vi(batch, extra, mg, 0, init_depth=5.0)
    _check_bits(got, sp.slide_batch(batch, extra, mg, 5.0))
    assert (_n_moved(batch, got) >= 10) if margin == mp.OLD else np.array_equal(got["inv_depth"], batch.inv_depth)


def _drop(pkg, batch, keep):
    """The batch with only the point factors where keep is set."""
    win = np.repeat(np.arange(batch.W), np.diff(batch.pf_window_offset))
    off = np.concatenate([[0], np.cumsum(np.bincount(win[keep], minlength=batch.W))])
    return pkg._abi.Batch(batch.poses, batch.ex_pose, batch.inv_depth, off, batch.pf_idx[keep], batch.pf_obs[keep],
                          pf_pts_i_z=None if batch.pf_pts_i_z is None else batch.pf_pts_i_z[keep])


def test_mixed_batch(pkg, ctx):
    """Both kinds; window 2 without a feature anchored at frame 0; in window 3 a feature with a single anchor-0 factor, whose depth
    keeps its input value."""
    batch, vi, extra = _case(pkg, W=6, seed=11)
    p0, p1 = batch.pf_window_offset[2], batch.pf_window_offset[3]
    idx = batch.pf_idx[p0:p1]
    idx = np.where((idx & 0xff) == 0, idx | 1, idx).astype(np.uint32)
    batch.pf_idx[p0:p1] = np.where(((idx >> 8) & 0xff) == 1, idx + (1 << 8), idx)
    q0, q1 = batch.pf_window_offset[3], batch.pf_window_offset[4]
    f = next(f for f, k in sp.reanchored(batch.pf_idx[q0:q1]).items())
    own = np.flatnonzero((batch.pf_idx[q0:q1] >> 16) == f) + q0
    keep = np.ones(batch.NP, bool)
    keep[own[1:]] = False
    batch = _drop(pkg, batch, keep)
    margin = np.array([0, 1, 0, 0, 1, 0], np.int32)
    got = ctx.slide_vi(batch, extra, margin, 0)
    _check_bits(got, sp.slide_batch(batch, extra, margin))
    assert np.array_equal(bits(got["inv_depth"][2]), bits(batch.inv_depth[2]))
    assert got["inv_depth"][3, f] == batch.inv_depth[3, f]
    assert not np.array_equal(got["inv_depth"][0], batch.inv_depth[0])


@pytest.mark.parametrize("form", [False, True, "f32"])
@pytest.mark.parametrize("with_z", [False, True])
def test_observation_forms(pkg, ctx, form, with_z):
    batch, vi, extra = _case(pkg, W=3, seed=31)
    if with_z:
        batch.pf_pts_i_z = 1.0 + 0.01 * np.random.default_rng(5).standard_normal(batch.NP)
    margin = np.zeros(batch.W, np.int32)
    got = ctx.slide_vi(batch, extra, margin, 0, obs_table=form)
    _check_bits(got, sp.slide_batch(batch, extra, margin))


def _slide_device(pkg, ctx, batch, extra, margin, init_depth=5.0, obs_table=False):
    """viml_slide_vi with VIML_PTRS_DEVICE on guarded device copies of every input and output: (outputs, inputs unchanged)."""
    s0, arrs = ctx._batch_struct(batch, obs_table)
    arrs = batch.arrays() if arrs is None else arrs
    b_in = {k: a for k, a in arrs.items() if a is not None}
    ins = {**{"b_" + k: a for k, a in b_in.items()}, "extra": extra, "margin": np.ascontiguousarray(margin, np.int32)}
    gi = guard_all(ctx, ins)
    s = batch.struct({**{k: None for k in arrs}, **{k: gi["b_" + k].ptr for k in b_in}})
    outs = {"poses": np.full_like(batch.poses, np.nan), "ex_pose": np.full_like(batch.ex_pose, np.nan),
            "inv_depth": np.full_like(batch.inv_depth, np.nan), "extra": np.full_like(extra, np.nan)}
    go = guard_all(ctx, outs)
    o = pkg._abi.SlideOut()
    for k in outs:
        setattr(o, k, go[k].ptr)
    ctx._check(ctx.lib.viml_slide_vi(ctx.h, C.byref(s), gi["extra"].ptr, extra.shape[1], gi["margin"].ptr, init_depth, C.byref(o),
                                     pkg.PTRS_DEVICE))
    ctx.sync()
    res = {k: g.check() for k, g in go.items()}
    same = all(np.array_equal(bits(g.check()), bits(ins[k])) for k, g in gi.items())
    for g in list(gi.values()) + list(go.values()):
        g.free()
    return res, same


@pytest.mark.parametrize("form", [False, "f32"])
def test_device_pointers_guard_bands(pkg, ctx, form):
    batch, vi, extra = _case(pkg, W=5, seed=29)
    batch.pf_pts_i_z = 1.0 + 0.01 * np.random.default_rng(6).standard_normal(batch.NP)
    margin = np.array([0, 1, 0, 1, 0], np.int32)
    host = ctx.slide_vi(batch, extra, margin, 0, obs_table=form)
    dev, same = _slide_device(pkg, ctx, batch, extra, margin, obs_table=form)
    assert same, "an input changed"
    _check_bits(dev, host)


def test_validation(pkg, ctx):
    batch, vi, extra = _case(pkg, W=2, seed=37)
    margin = np.zeros(2, np.int32)

    def refused(b=batch, e=extra, mg=margin, init_depth=5.0, flags=0):
        with pytest.raises(pkg.VimlError, match="error -1"):
            if flags:
                _slide_device(pkg, ctx, b, e, mg, init_depth)
            else:
                ctx.slide_vi(b, e, mg, 0, init_depth=init_depth)

    refused(mg=np.array([0, 2], np.int32))
    refused(e=extra[:, :9 * batch.P - 1])            # X < 9P
    for d in (0.0, -1.0, np.nan, np.inf):
        refused(init_depth=d)
        refused(init_depth=d, flags=pkg.PTRS_DEVICE)
    # a feature with factors both at i == 0 and i != 0
    b2 = batch.slice_windows(0, 1)
    k = int(np.flatnonzero((b2.pf_idx & 0xff) == 0)[0])
    f = int(b2.pf_idx[k] >> 16)
    b2 = pkg._abi.Batch(b2.poses, b2.ex_pose, b2.inv_depth, [0, b2.NP + 1],
                        np.concatenate([b2.pf_idx, np.array([2 | (3 << 8) | (f << 16)], np.uint32)]),
                        np.concatenate([b2.pf_obs, b2.pf_obs[:1]]))
    refused(b2, extra[:1], margin[:1])
    # P < 2, on both flavours
    b3 = pkg._abi.Batch(batch.poses[:1, :1], batch.ex_pose[:1], batch.inv_depth[:1], [0, 0], np.zeros(0, np.uint32), np.zeros((0, 4)))
    refused(b3, np.zeros((1, 9)), margin[:1])
    refused(b3, np.zeros((1, 9)), margin[:1], flags=pkg.PTRS_DEVICE)
    # W == 0
    b0 = pkg._abi.Batch(np.zeros((0, 11, 7)), np.zeros((0, 7)), np.zeros((0, 4)), [0], np.zeros(0, np.uint32), np.zeros((0, 4)))
    o = pkg._abi.SlideOut()
    assert ctx.lib.viml_slide_vi(ctx.h, C.byref(b0.struct()), None, 99, None, 5.0, C.byref(o), 0) == 0


SOLVE_OUT = ("poses", "ex_pose", "inv_depth", "extra", "status", "iterations", "accepted", "cost")


def _inertial_with_prior(pkg, vi, prior):
    return pkg._abi.Inertial(vi.W, vi.P, vi.X, vi.gravity, vi.imu_window_offset, vi.imu_pose, vi.imu_sb, vi.imu_preint, vi.imu_jacobian,
                             vi.imu_sqrt_info, prior["prior_n"], np.nan_to_num(prior["prior_jacobian"]),
                             np.nan_to_num(prior["prior_residual"]), prior["prior_n_blocks"], np.maximum(prior["prior_block"], 0),
                             np.nan_to_num(prior["prior_x0"]))


def _chain_host(pkg, ctx, batch, vi, extra, margin, nxt):
    s1 = ctx.solve_vi(batch, vi, extra, FLAGS, max_iterations=6)
    b1 = pkg._abi.Batch(s1["poses"], s1["ex_pose"], s1["inv_depth"], batch.pf_window_offset, batch.pf_idx, batch.pf_obs)
    prior = ctx.marginalize_vi(b1, vi, s1["extra"], margin, FLAGS)
    sl = sp.slide_batch(b1, s1["extra"], margin)
    b2 = pkg._abi.Batch(sl["poses"], sl["ex_pose"], sl["inv_depth"], *nxt)
    s2 = ctx.solve_vi(b2, _inertial_with_prior(pkg, vi, prior), sl["extra"], FLAGS, max_iterations=6)
    return s1, s2


def _chain_device(pkg, ctx, batch, vi, extra, margin, nxt):
    """The same chain, every call with VIML_PTRS_DEVICE and nothing read back before the end."""
    W, P, X = batch.W, batch.P, vi.X
    n_max, mb = vi.n_max, 2 * P + 1
    ptrs = []

    def dev(a):
        ptrs.append(ctx.to_device(np.ascontiguousarray(a)))
        return ptrs[-1]

    like = {"poses": batch.poses, "ex_pose": batch.ex_pose, "inv_depth": batch.inv_depth, "extra": extra,
            "status": np.zeros(W, np.int32), "iterations": np.zeros(W, np.int32), "accepted": np.zeros(W, np.int32),
            "cost": np.zeros((W, 2))}
    bd = {k: dev(a) for k, a in batch.arrays().items() if a is not None}
    vd = {k: dev(a) for k, a in vi.arrays().items()}
    exd, mgd = dev(extra), dev(margin)
    o1, o2 = ({k: dev(np.zeros_like(a)) for k, a in like.items()} for _ in range(2))
    pz = {"prior_n": np.zeros(W, np.int32), "prior_jacobian": np.zeros((W, n_max, n_max)), "prior_residual": np.zeros((W, n_max)),
          "prior_n_blocks": np.zeros(W, np.int32), "prior_block": np.zeros((W, mb, 4), np.int32), "prior_x0": np.zeros((W, mb, 9))}
    pd = {k: dev(a) for k, a in pz.items()}
    sd = {k: dev(np.zeros_like(like[k])) for k in STATE}
    b2h = pkg._abi.Batch(batch.poses, batch.ex_pose, batch.inv_depth, *nxt)
    b2d = {k: dev(getattr(b2h, k)) for k in ("pf_window_offset", "pf_idx", "pf_obs", "lf_window_offset", "lf_frame", "lf_geom")}
    opt = ctx.solve_options(max_iterations=6)

    def solve_out(o):
        so = pkg._abi.SolveOut()
        for k in SOLVE_OUT:
            setattr(so, k, o[k])
        return so

    s1 = batch.struct({**bd, "pf_pts_i_z": None})
    v1 = vi.struct(vd)
    ctx._check(ctx.lib.viml_solve_vi(ctx.h, C.byref(s1), C.byref(v1), exd, C.byref(opt), C.byref(solve_out(o1)), FLAGS | pkg.PTRS_DEVICE))
    b1 = batch.struct({**bd, "pf_pts_i_z": None, "poses": o1["poses"], "ex_pose": o1["ex_pose"], "inv_depth": o1["inv_depth"]})
    po = pkg._abi.PriorOut()
    po.prior_n_max, po.prior_max_blocks = n_max, mb
    for k in pz:
        setattr(po, k, pd[k])
    ctx._check(ctx.lib.viml_marginalize_vi(ctx.h, C.byref(b1), C.byref(v1), o1["extra"], mgd, C.byref(po), FLAGS | pkg.PTRS_DEVICE))
    so = pkg._abi.SlideOut()
    for k in STATE:
        setattr(so, k, sd[k])
    ctx._check(ctx.lib.viml_slide_vi(ctx.h, C.byref(b1), o1["extra"], X, mgd, 5.0, C.byref(so), pkg.PTRS_DEVICE))
    s2 = b2h.struct({**b2d, "pf_pts_i_z": None, "poses": sd["poses"], "ex_pose": sd["ex_pose"], "inv_depth": sd["inv_depth"]})
    vi2h = _inertial_with_prior(pkg, vi, pz)
    v2 = vi2h.struct({**vd, **pd})
    ctx._check(ctx.lib.viml_solve_vi(ctx.h, C.byref(s2), C.byref(v2), sd["extra"], C.byref(opt), C.byref(solve_out(o2)),
                                     FLAGS | pkg.PTRS_DEVICE))
    ctx.sync()
    res = []
    for o in (o1, o2):
        r = {k: np.empty_like(like[k]) for k in SOLVE_OUT}
        for k in SOLVE_OUT:
            ctx.d2h(r[k], o[k])
        res.append(r)
    ctx.sync()
    for p in ptrs:
        ctx.device_free(p)
    return res


@pytest.mark.parametrize("points", [False, True])
def test_two_frame_chain_device_pointers(pkg, ctx, points):
    """Inertial-only windows: every kernel is order-deterministic, so the chains agree bit for bit.  With point factors the visual
    pose blocks are summed through shared-memory atomics: the 1e-9 per-unit bar."""
    batch = pkg.synth.make_windows(6, seed=23, F=40, lines_per_frame=0)
    vi, extra = pkg.synth.make_inertial_factors(batch, seed=24)
    b = batch if points else inertial_only(pkg, batch)
    margin = np.array([0, 0, 1, 0, 1, 0], np.int32)
    nxt = sp.next_structure_batch(b, margin)
    h1, h2 = _chain_host(pkg, ctx, b, vi, extra, margin, nxt)
    d1, d2 = _chain_device(pkg, ctx, b, vi, extra, margin, nxt)
    assert (h2["status"] != pkg._abi.SOLVE_FAILURE).all() and (d2["status"] != pkg._abi.SOLVE_FAILURE).all()
    assert (h2["accepted"] > 0).all()
    for h, d in ((h1, d1), (h2, d2)):
        for k in SOLVE_OUT:
            if not points:
                assert np.array_equal(bits(d[k]), bits(h[k])), k
            elif k in STATE + ("cost",):
                for w in range(b.W):
                    assert rel_err(d[k][w], h[k][w]) < 1e-9, (k, w)
    if points:
        assert len(nxt[1]) > 0
