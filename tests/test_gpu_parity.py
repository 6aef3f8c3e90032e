"""GPU parity tests (run with -m gpu on a B200): the CUDA path, driven through the C-ABI, against the CPU
oracle on the same seeded inputs and against the committed golden fixtures.

Bars (BASELINE.json north_star): association indices / inlier masks / FoV lists bit-exact; residuals,
Jacobians, H, b and the Schur complement within 1e-9 relative PER UNIT (per factor, per 6x6 block, per landmark
row: tc-viml_b200/parity.py)."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT, rel_err

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
TOL = 1e-9


def check_linearize(pkg, orc, ctx, cfg, batch, flags, tol=TOL):
    got = ctx.linearize(batch, flags)
    ref = orc.linearize_batch(cfg, batch, flags, nthreads=8)
    assert set(got) == set(ref)
    for k, v in ref.items():
        assert not np.isnan(got[k]).any(), f"{k}: unwritten entries"
        e = pkg.parity.unit_err(k, got[k], v)
        assert e < tol, (k, e)
    return got, ref


def test_single_window_cfg1(pkg, orc, ctx, cfg):
    """BASELINE.json configs[0]: one EuRoC-shaped window (11 poses, 150 features, line factors)."""
    abi = pkg._abi
    b = pkg.synth.make_windows(1, seed=101)
    for flags in (abi.OUT_RESIDUAL_JACOBIAN, abi.OUT_RESIDUAL_JACOBIAN | abi.LOSS_CAUCHY,
                  abi.OUT_HB | abi.LOSS_CAUCHY, abi.OUT_SCHUR | abi.LOSS_CAUCHY,
                  abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY, abi.OUT_HB):
        got, _ = check_linearize(pkg, orc, ctx, cfg, b, flags)
        if flags & abi.OUT_RESIDUAL_JACOBIAN:
            for k in ("pf_jac_pose_i", "pf_jac_pose_j", "pf_jac_ex", "lf_jac_pose"):
                assert np.all(got[k].reshape(-1, 2, 7)[:, :, 6] == 0.0)   # column 6 is exactly zero
        if flags & abi.OUT_HB:
            assert np.abs(got["H_pp"] - np.swapaxes(got["H_pp"], 1, 2)).max() <= 1e-9 * np.abs(got["H_pp"]).max()


def test_packed_schur_output(pkg, orc, ctx, cfg):
    """VIML_S_PACKED: the upper triangle of S, bit for bit the entries of the full output (host and device pointers)."""
    abi = pkg._abi
    b = pkg.synth.make_windows(20, seed=151)
    full = ctx.linearize(b, abi.OUT_SCHUR | abi.LOSS_CAUCHY)
    bufs = {"S_packed": np.full(b.out_shapes()["S_packed"], np.nan), "g": np.full((b.W, b.D), np.nan)}
    ctx.linearize(b, abi.OUT_SCHUR | abi.S_PACKED | abi.LOSS_CAUCHY, out=bufs)
    iu = np.triu_indices(b.D)
    assert pkg.parity.unit_err("S", abi.unpack_upper(bufs["S_packed"], b.D), full["S"]) < 1e-12
    assert pkg.parity.unit_err("g", bufs["g"], full["g"]) < 1e-12
    assert not np.isnan(bufs["S_packed"]).any()
    ref = orc.linearize_batch(cfg, b, abi.OUT_SCHUR | abi.LOSS_CAUCHY)
    assert pkg.parity.unit_err("S", abi.unpack_upper(bufs["S_packed"], b.D), ref["S"]) < TOL
    # a long window (D = 246: the packing runs on several CTAs per window)
    h = pkg.synth.make_windows(2, seed=152, P=40, F=400, lines_per_frame=2, max_len=12)
    fullh = ctx.linearize(h, abi.OUT_SCHUR | abi.LOSS_CAUCHY)
    bh = {"S_packed": np.full(h.out_shapes()["S_packed"], np.nan), "g": np.full((h.W, h.D), np.nan)}
    ctx.linearize(h, abi.OUT_SCHUR | abi.S_PACKED | abi.LOSS_CAUCHY, out=bh)
    assert not np.isnan(bh["S_packed"]).any()
    assert pkg.parity.unit_err("S", abi.unpack_upper(bh["S_packed"], h.D), fullh["S"]) < 1e-12


def test_golden_linearize(pkg, orc, ctx, cfg):
    g = np.load(os.path.join(GOLD, "linearize_cfg1.npz"))
    abi = pkg._abi
    b = abi.Batch(g["in_poses"], g["in_ex_pose"], g["in_inv_depth"], g["in_pf_window_offset"], g["in_pf_idx"],
                  g["in_pf_obs"], g["in_lf_window_offset"], g["in_lf_frame"], g["in_lf_geom"])
    flags = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    got = ctx.linearize(b, flags)
    for k in got:
        assert pkg.parity.unit_err(k, got[k], g["out_" + k]) < TOL, k


def test_batch_shapes_and_edges(pkg, orc, ctx, cfg):
    abi, synth = pkg._abi, pkg.synth
    allf = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    check_linearize(pkg, orc, ctx, cfg, synth.make_windows(37, seed=102), allf)
    # no line factors at all
    check_linearize(pkg, orc, ctx, cfg, synth.make_windows(5, seed=103, lines_per_frame=0), allf)
    # other window geometries: short window, few features; long window
    check_linearize(pkg, orc, ctx, cfg, synth.make_windows(9, seed=104, P=5, F=17, lines_per_frame=2), allf)
    check_linearize(pkg, orc, ctx, cfg, synth.make_windows(3, seed=105, P=24, F=300, lines_per_frame=3), allf)
    # ragged: windows with zero factors in the middle of the batch
    b = synth.make_windows(6, seed=106)
    keep = np.ones(b.NP, dtype=bool)
    keep[b.pf_window_offset[2]:b.pf_window_offset[3]] = False
    keep[b.pf_window_offset[5]:b.pf_window_offset[6]] = False
    off = np.concatenate([[0], np.cumsum([keep[b.pf_window_offset[w]:b.pf_window_offset[w + 1]].sum() for w in range(6)])])
    b2 = abi.Batch(b.poses, b.ex_pose, b.inv_depth, off, b.pf_idx[keep], b.pf_obs[keep], b.lf_window_offset, b.lf_frame,
                   b.lf_geom)
    check_linearize(pkg, orc, ctx, cfg, b2, allf)
    # explicit pts_i.z != 1 (ProjectionFactor divides all three components by inv_dep, projection_factor.cpp:35)
    b3 = synth.make_windows(4, seed=107)
    b3.pf_pts_i_z = 1.0 + 0.01 * np.random.default_rng(1).standard_normal(b3.NP)
    check_linearize(pkg, orc, ctx, cfg, b3, allf)
    # windows too large for the fused kernel's shared memory (> 704 factors) inside a batch that is otherwise
    # on the fast path: flagged and finished by the generic atomic kernel
    big = synth.make_windows(5, seed=112, F=160, all_start_zero=True)
    assert np.diff(big.pf_window_offset).max() > 704
    check_linearize(pkg, orc, ctx, cfg, big, allf)
    mixed = synth.make_windows(6, seed=113, F=160)
    keep = np.ones(mixed.NP, dtype=bool)          # thin out all but window 1 -> only one window is flagged
    check_linearize(pkg, orc, ctx, cfg, mixed, allf)
    # the generic path alone (test hook), same results
    os.environ["VIML_FORCE_GENERIC"] = "1"
    try:
        with pkg.Context(cfg) as cg:
            check_linearize(pkg, orc, cg, cfg, synth.make_windows(7, seed=114), allf)
    finally:
        del os.environ["VIML_FORCE_GENERIC"]
    # non-default sqrt_info / Cauchy scale
    cfg2 = synth.euroc_config(sqrt_info=120.0, cauchy_a=2.5)
    with pkg.Context(cfg2) as c2:
        check_linearize(pkg, orc, c2, cfg2, synth.make_windows(4, seed=108), allf)


def test_fused_path_extremes(pkg, orc, ctx, cfg):
    """Limits of the fused kernel's static layout (12 poses, 4-bit pose indices in the plan), degenerate pair structures
    and empty factor classes, with and without the per-factor outputs (both template instantiations)."""
    abi, synth = pkg._abi, pkg.synth
    hb = abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    allf = hb | abi.OUT_RESIDUAL_JACOBIAN
    for flags in (hb, allf):
        check_linearize(pkg, orc, ctx, cfg, synth.make_windows(6, seed=121, P=12, F=160, lines_per_frame=12), flags)
        check_linearize(pkg, orc, ctx, cfg, synth.make_windows(5, seed=122, P=2, F=9, lines_per_frame=1, start_max=0), flags)
        check_linearize(pkg, orc, ctx, cfg, synth.make_windows(4, seed=123, P=3, F=150, lines_per_frame=0, start_max=0), flags)
    # only line factors: every pose-pair block, every landmark row is a structural zero
    b = synth.make_windows(4, seed=124)
    only_lines = abi.Batch(b.poses, b.ex_pose, b.inv_depth, np.zeros(5, dtype=np.int32), b.pf_idx[:0], b.pf_obs[:0],
                           b.lf_window_offset, b.lf_frame, b.lf_geom)
    got, _ = check_linearize(pkg, orc, ctx, cfg, only_lines, abi.OUT_HB | abi.LOSS_CAUCHY)
    assert np.all(got["H_lp"] == 0.0) and np.all(got["H_ll"] == 0.0)
    # no landmarks at all (F = 0): nothing to eliminate, S and g are H_pp and b_p bit for bit (full and packed S)
    no_feats = abi.Batch(b.poses, b.ex_pose, np.zeros((b.W, 0)), np.zeros(5, dtype=np.int32), b.pf_idx[:0], b.pf_obs[:0],
                         b.lf_window_offset, b.lf_frame, b.lf_geom)
    got, _ = check_linearize(pkg, orc, ctx, cfg, no_feats, abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY)
    assert np.array_equal(got["S"], got["H_pp"]) and np.array_equal(got["g"], got["b_p"])
    bufs = no_feats.alloc_out(abi.OUT_HB | abi.OUT_SCHUR)
    del bufs["S"]
    bufs["S_packed"] = np.full(no_feats.out_shapes()["S_packed"], np.nan)
    ctx.linearize(no_feats, abi.OUT_HB | abi.OUT_SCHUR | abi.S_PACKED | abi.LOSS_CAUCHY, out=bufs)
    iu = np.triu_indices(no_feats.D)
    assert np.array_equal(bufs["S_packed"], bufs["H_pp"][:, iu[0], iu[1]]) and np.array_equal(bufs["g"], bufs["b_p"])
    # one pose pair carries every factor (all features start in frame 0 and are seen once more, in frame 1)
    b = synth.make_windows(3, seed=125, P=11, F=150, all_start_zero=True, max_len=2)
    check_linearize(pkg, orc, ctx, cfg, b, hb)
    # reproducible: per-factor outputs and the landmark part bit for bit; the pose blocks are summed through shared-memory
    # atomics in whatever order the warps finish their segments, so H_pp / b_p (and S, g) repeat to rounding only
    b = synth.make_windows(16, seed=126)
    a1 = ctx.linearize(b, allf)
    a2 = ctx.linearize(b, allf)
    for k in a1:
        if k in ("H_pp", "b_p", "S", "g"):
            assert pkg.parity.unit_err(k, a1[k], a2[k]) < 1e-12, k
        else:
            assert np.array_equal(a1[k], a2[k]), k


def test_irregular_windows(pkg, orc, ctx, cfg):
    """Factor lists outside the reference's structure (estimator.cpp:1735-1770: one anchor per feature, one factor per
    (feature, frame), i != j) are legal for the C-ABI: the plan flags such windows and they are assembled by the generic
    atomic kernel, inside a batch whose other windows stay on the fused path."""
    abi, synth = pkg._abi, pkg.synth
    allf = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    b = synth.make_windows(6, seed=131)
    idx = b.pf_idx.copy()
    o = b.pf_window_offset
    # window 1: a feature gets a second anchor;  window 3: a repeated (feature, j)
    k = o[1] + 5
    i, j, l = int(idx[k] & 0xff), int((idx[k] >> 8) & 0xff), int(idx[k] >> 16)
    i2 = (i + 1) % 11 if (i + 1) % 11 != j else (i + 2) % 11
    idx[k] = i2 | (j << 8) | (l << 16)
    idx[o[3] + 7] = idx[o[3] + 8]
    b2 = abi.Batch(b.poses, b.ex_pose, b.inv_depth, o, idx, b.pf_obs, b.lf_window_offset, b.lf_frame, b.lf_geom)
    check_linearize(pkg, orc, ctx, cfg, b2, allf)
    check_linearize(pkg, orc, ctx, cfg, b2, abi.OUT_HB | abi.LOSS_CAUCHY)
    # window 2 with the roles of i and j swapped in every factor: features now have several anchors -> generic kernel
    idx3 = b.pf_idx.copy()
    i3, j3, l3 = idx3 & 0xff, (idx3 >> 8) & 0xff, idx3 >> 16
    pos = np.arange(len(idx3))
    flip = (pos >= o[2]) & (pos < o[3])
    b3 = abi.Batch(b.poses, b.ex_pose, b.inv_depth, o, np.where(flip, j3 | (i3 << 8) | (l3 << 16), idx3).astype(np.uint32),
                   b.pf_obs, b.lf_window_offset, b.lf_frame, b.lf_geom)
    check_linearize(pkg, orc, ctx, cfg, b3, allf)
    # regular windows whose anchor is the LAST frame of every track (i > j everywhere): fused path, lo/hi roles flip
    b4 = synth.make_windows(5, seed=132, all_start_zero=True, max_len=6)
    i4, j4, l4 = b4.pf_idx & 0xff, (b4.pf_idx >> 8) & 0xff, b4.pf_idx >> 16
    b5 = abi.Batch(b4.poses, b4.ex_pose, b4.inv_depth, b4.pf_window_offset, ((10 - i4) | ((10 - j4) << 8) | (l4 << 16)).astype(np.uint32),
                   b4.pf_obs, b4.lf_window_offset, b4.lf_frame, b4.lf_geom)
    check_linearize(pkg, orc, ctx, cfg, b5, allf)
    # out-of-range indices through host pointers are rejected before anything is launched
    bad = b.pf_idx.copy()
    bad[3] = 200 | (1 << 8) | (0 << 16)
    bb = abi.Batch(b.poses, b.ex_pose, b.inv_depth, o, bad, b.pf_obs, b.lf_window_offset, b.lf_frame, b.lf_geom)
    s, oo = bb.struct(), abi.out_struct(bb.alloc_out(abi.OUT_HB))
    assert ctx.lib.viml_linearize_batch(ctx.h, C.byref(s), C.byref(oo), abi.OUT_HB) == abi.VIML_ERR_INVALID
    assert b"index" in ctx.lib.viml_last_error(ctx.h)


def test_marginalisation_stress_shape(pkg, orc, ctx, cfg):
    """cfg-4 shape at a size the dense oracle finishes in seconds: all landmarks start in frame 0."""
    abi = pkg._abi
    b = pkg.synth.make_windows(3, seed=109, P=11, F=400, all_start_zero=True, lines_per_frame=0)
    check_linearize(pkg, orc, ctx, cfg, b, abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY)
    # the full cfg-4 window shape: 2000 landmarks, ~11000 factors per window (fused kernel in its many-feature mode:
    # 16 accumulating parts per window, landmark rows by RED), DMMA Schur with K = 2000
    b = pkg.synth.make_windows(2, seed=115, P=11, F=2000, all_start_zero=True, lines_per_frame=3)
    assert np.diff(b.pf_window_offset).min() > 9000
    check_linearize(pkg, orc, ctx, cfg, b, abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY)


def test_associate_before_set_map(pkg, cfg):
    abi = pkg._abi
    with pkg.Context(cfg) as c0:
        q, o = abi.AssocQuery(), abi.AssocOut()
        pose = np.zeros((1, 7)); pose[0, 6] = 1.0
        l2d = np.zeros((1, 1, 4))
        q.n_poses, q.lines_per_pose = 1, 1
        q.cull_poses, q.ex_pose, q.lines2d = abi.ptr(pose), abi.ptr(pose), abi.ptr(l2d)
        assert c0.lib.viml_line_associate(c0.h, C.byref(q), C.byref(o), 0) == abi.VIML_ERR_NOMAP


def test_bad_arguments(pkg, ctx, cfg):
    abi = pkg._abi
    b = pkg.synth.make_windows(1, seed=110)
    s, o = b.struct(), abi.LinearizeOut()
    lib = ctx.lib
    assert lib.viml_linearize_batch(ctx.h, C.byref(s), C.byref(o), 0) == abi.VIML_ERR_INVALID
    assert lib.viml_linearize_batch(ctx.h, C.byref(s), C.byref(o), abi.OUT_HB) == abi.VIML_ERR_INVALID
    assert b"H_pp" in lib.viml_last_error(ctx.h)
    assert lib.viml_linearize_batch(ctx.h, None, C.byref(o), abi.OUT_HB) == abi.VIML_ERR_INVALID
    s.poses_per_window = 0
    assert lib.viml_linearize_batch(ctx.h, C.byref(s), C.byref(o), abi.OUT_RESIDUAL_JACOBIAN) == abi.VIML_ERR_INVALID
    # dense factors through host pointers: the CSR the kernels index through is checked before anything is launched
    b3 = pkg.synth.make_windows(3, seed=110)
    dense = pkg.synth.make_dense_factors(b3)
    Dx = b3.D + dense.X
    bs = b3.struct()
    S, g = np.zeros((b3.W, b3.D, b3.D)), np.zeros((b3.W, b3.D))
    Sx, gx = np.zeros((b3.W, Dx, Dx)), np.zeros((b3.W, Dx))
    ro = abi.ReducedOut()
    ro.Sx, ro.gx = abi.ptr(Sx), abi.ptr(gx)
    wo = dense.window_offset
    for field, i, val in (("jac_offset", 1, dense.jac_offset[1] + 1),   # a step != rows x columns
                          ("window_offset", -1, wo[-1] - 1),            # last entry != n_factors
                          ("window_offset", 1, wo[2] + 1),              # decreases in the middle
                          ("col_index", 0, Dx),                         # column outside [0, Dx)
                          ("col_index", 1, dense.col_index[0]),         # a column repeated inside factor 0
                          ("col_offset", 0, 1),                         # offsets that do not start at 0
                          ("col_offset", 1, dense.col_offset[-1] + 7)):  # past the total, then back down
        arrs = {k: v.copy() for k, v in dense.arrays().items()}
        arrs[field][i] = val
        d = dense.struct(arrs)
        assert lib.viml_reduced_system(ctx.h, C.byref(bs), C.byref(d), C.byref(ro), 0) == abi.VIML_ERR_INVALID
        assert field.encode() in lib.viml_last_error(ctx.h)
        assert lib.viml_reduced_from_schur(ctx.h, b3.W, b3.D, abi.ptr(S), abi.ptr(g), C.byref(d), C.byref(ro), 0) == abi.VIML_ERR_INVALID
        assert field.encode() in lib.viml_last_error(ctx.h)
    # a malformed window batch through host pointers: every entry point that takes one refuses it before anything is launched, with
    # viml_linearize_batch's code and message (P = 13: the steps would run the generic H/b kernels, which index without checks)
    def calls(c, bad, vi, extra, **form):
        return (lambda: c.linearize(bad, abi.OUT_HB | abi.LOSS_CAUCHY, **form),
                lambda: c.reduced_system(bad, None, abi.LOSS_CAUCHY, **form),
                lambda: c.gn_step(bad, None, None, abi.LOSS_CAUCHY, **form),
                lambda: c.gn_step_vi(bad, vi, extra, abi.LOSS_CAUCHY, **form),
                lambda: c.solve_vi(bad, vi, extra, abi.LOSS_CAUCHY, max_iterations=2, **form))

    def refusals(fns):
        msgs = []
        for fn in fns:
            with pytest.raises(pkg.VimlError) as e:
                fn()
            msgs.append(str(e.value))
        return msgs

    for P in (11, 13):
        good = pkg.synth.make_windows(3, seed=110, P=P)
        vi, extra = pkg.synth.make_inertial_factors(good, seed=111)
        for field, i, val, what in (("pf_window_offset", -1, good.NP - 1, "window offsets"),      # last entry != n_factors
                                    ("lf_window_offset", 1, good.lf_window_offset[2] + 1, "window offsets"),   # decreases
                                    ("pf_idx", 3, P | (1 << 8), "index out of range"),          # pose i == P
                                    ("lf_frame", 2, P, "index out of range")):
            arrs = {k: (None if v is None else v.copy()) for k, v in good.arrays().items()}
            arrs[field][i] = val
            msgs = refusals(calls(ctx, abi.Batch(**arrs), vi, extra))
            assert msgs[0].startswith(f"viml error {abi.VIML_ERR_INVALID}: ") and what in msgs[0], (P, field, msgs[0])
            assert msgs[1:] == msgs[:1] * 4, (P, field, msgs)
    # a line table on a context without a map
    good, _ = pkg.synth.with_line_map(pkg.synth.make_windows(3, seed=110), cfg)
    vi, extra = pkg.synth.make_inertial_factors(good, seed=111)
    with pkg.Context(cfg) as c0:
        msgs = refusals(calls(c0, good, vi, extra, line_table=True))
    assert msgs[0].startswith(f"viml error {abi.VIML_ERR_NOMAP}: ") and msgs[1:] == msgs[:1] * 4, msgs


def test_observation_table_input(pkg, orc, ctx, cfg):
    """viml_window_batch.feat_obs / pf_obs_j (pf_obs == NULL): pts_i once per feature, as FeaturePerId stores it
    (feature_manager.h:65-96; estimator.cpp:1747-1766 builds every factor of a feature from feature_per_frame[0].point).  Same
    results, bit for bit where the per-factor form is deterministic, through every entry point that takes a window batch."""
    abi, synth = pkg._abi, pkg.synth
    b = synth.make_windows(600, seed=171)       # 600 windows: the host pipeline runs in chunks
    feat_obs, obs_j = b.obs_table()
    assert feat_obs.shape == (b.W, b.F, 2) and obs_j.shape == (b.NP, 2)
    flags = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    pairs = ctx.linearize(b, flags)
    table = ctx.linearize(b, flags, obs_table=True)
    for k, v in pairs.items():
        assert not np.isnan(table[k]).any(), k
        if k.startswith(("pf_", "lf_")) or k in ("H_lp", "H_ll", "b_l"):
            assert np.array_equal(table[k], v), k
        else:
            assert pkg.parity.unit_err(k, table[k], v) < 1e-12, k
    ref = orc.linearize_batch(cfg, b.slice_windows(0, 32), flags, nthreads=8)
    for k, v in ref.items():
        n = v.shape[0]
        assert pkg.parity.unit_err(k, table[k][:n], v) < TOL, k
    # device pointers
    small = b.slice_windows(0, 16)
    fo, oj = small.obs_table()
    arrs = {k: v for k, v in small.arrays().items() if v is not None and k != "pf_obs"}
    arrs.update(feat_obs=fo, pf_obs_j=oj)
    d_in = {k: ctx.to_device(v) for k, v in arrs.items()}
    want = ctx.linearize(small, abi.OUT_HB | abi.LOSS_CAUCHY)
    d_out = {k: ctx.device_alloc(v.nbytes) for k, v in want.items()}
    ctx.linearize_raw(small.struct(d_in), abi.out_struct(d_out), abi.OUT_HB | abi.LOSS_CAUCHY | abi.PTRS_DEVICE)
    for k, v in want.items():
        back = np.empty_like(v)
        ctx.d2h(back, d_out[k])
        ctx.sync()
        assert pkg.parity.unit_err(k, back, v) < 1e-12, k
    for p in list(d_in.values()) + list(d_out.values()):
        ctx.device_free(p)
    # the solver entry points take the same batch struct
    dense = synth.make_dense_factors(small, seed=5)
    Sx0, gx0 = ctx.reduced_system(small, dense, abi.LOSS_CAUCHY)
    Sx1, gx1 = ctx.reduced_system(small, dense, abi.LOSS_CAUCHY, obs_table=True)
    assert np.abs(Sx1 - Sx0).max() <= 1e-12 * np.abs(Sx0).max() and np.abs(gx1 - gx0).max() <= 1e-12 * np.abs(gx0).max()
    extra = np.zeros((small.W, dense.X))
    g0 = ctx.gn_step(small, dense, extra, abi.LOSS_CAUCHY, lam=1e-4)
    g1 = ctx.gn_step(small, dense, extra, abi.LOSS_CAUCHY, lam=1e-4, obs_table=True)
    assert np.abs(g1["dx"] - g0["dx"]).max() <= 1e-9 * np.abs(g0["dx"]).max()
    # float32 table: observations that are float32 values (what the tracker publishes) travel as floats, same results bit for bit
    bf = synth.make_windows(600, seed=171, f32_obs=True)
    pairs32 = ctx.linearize(bf, flags)
    table32 = ctx.linearize(bf, flags, obs_table="f32")
    for k, v in pairs32.items():
        if k.startswith(("pf_", "lf_")) or k in ("H_lp", "H_ll", "b_l"):
            assert np.array_equal(table32[k], v), k
        else:
            assert pkg.parity.unit_err(k, table32[k], v) < 1e-12, k
    s32 = bf.slice_windows(0, 8)           # the small-batch staging path and the solver entry point
    a32, b32 = ctx.linearize(s32, flags), ctx.linearize(s32, flags, obs_table="f32")
    assert np.array_equal(a32["pf_jac_pose_i"], b32["pf_jac_pose_i"]) and pkg.parity.unit_err("S", b32["S"], a32["S"]) < 1e-12
    d32 = synth.make_dense_factors(s32, seed=5)
    Sa, ga = ctx.reduced_system(s32, d32, abi.LOSS_CAUCHY)
    Sb, gb = ctx.reduced_system(s32, d32, abi.LOSS_CAUCHY, obs_table="f32")
    assert np.abs(Sb - Sa).max() <= 1e-12 * np.abs(Sa).max() and np.abs(gb - ga).max() <= 1e-12 * np.abs(ga).max()
    with pytest.raises(ValueError):
        b.obs_table(f32=True)              # b's observations are full doubles
    # a batch whose factors do not share pts_i per feature has no table form
    bad = abi.Batch(b.poses, b.ex_pose, b.inv_depth, b.pf_window_offset, b.pf_idx, b.pf_obs + np.arange(b.NP)[:, None] * 1e-6,
                    b.lf_window_offset, b.lf_frame, b.lf_geom)
    with pytest.raises(ValueError):
        bad.obs_table()


def test_line_table_input(pkg, orc, cfg):
    """viml_window_batch.lf_map_index / lf_seg2d_f32 (lf_geom == NULL): a line factor given by its map line and the detected 2D segment,
    as the estimator builds it (estimator.cpp:1831-1835, feature_manager.cpp:11-13).  The device expands them with the reference's
    operation order: same outputs as the nine-plane form, bit for bit on the per-factor line outputs, through the chunked pipeline,
    the small-batch staging, device pointers and the solver entry point; errors without a map or with an index outside it."""
    abi, synth = pkg._abi, pkg.synth
    b0 = synth.make_windows(600, seed=201, f32_obs=True)
    b, lmap = synth.with_line_map(b0, cfg)
    flags = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    with pkg.Context(cfg) as c:
        with pytest.raises(pkg.VimlError):
            c.linearize(b.slice_windows(0, 4), flags, line_table=True)          # no map yet
        c.set_map(lmap)
        planes = c.linearize(b, flags)
        table = c.linearize(b, flags, obs_table="f32", line_table=True)
        for k, v in planes.items():
            assert not np.isnan(table[k]).any(), k
            if k.startswith(("pf_", "lf_")) or k in ("H_lp", "H_ll", "b_l"):
                assert np.array_equal(table[k], v), k
            else:
                assert pkg.parity.unit_err(k, table[k], v) < 1e-12, k
        ref = orc.linearize_batch(cfg, b.slice_windows(0, 16), flags, nthreads=8)
        for k, v in ref.items():
            assert pkg.parity.unit_err(k, table[k][:v.shape[0]], v) < TOL, k
        small = b.slice_windows(590, 600)                                       # staging path; map indices are absolute
        s_pl, s_tb = c.linearize(small, flags), c.linearize(small, flags, line_table=True)
        assert np.array_equal(s_tb["lf_jac_pose"], s_pl["lf_jac_pose"]) and np.array_equal(s_tb["lf_residual"], s_pl["lf_residual"])
        assert pkg.parity.unit_err("S", s_tb["S"], s_pl["S"]) < 1e-12
        # device pointers
        arrs = {k: v for k, v in small.arrays().items() if v is not None and k != "lf_geom"}
        arrs.update(lf_map_index=small.lf_map_index, lf_seg2d_f32=small.lf_seg2d)
        d_in = {k: c.to_device(v) for k, v in arrs.items()}
        want = {k: s_pl[k] for k in ("H_pp", "H_lp", "H_ll", "b_p", "b_l")}
        d_out = {k: c.device_alloc(v.nbytes) for k, v in want.items()}
        c.linearize_raw(small.struct(d_in), abi.out_struct(d_out), abi.OUT_HB | abi.LOSS_CAUCHY | abi.PTRS_DEVICE)
        for k, v in want.items():
            back = np.empty_like(v)
            c.d2h(back, d_out[k])
            c.sync()
            assert pkg.parity.unit_err(k, back, v) < 1e-12, k
        for p in list(d_in.values()) + list(d_out.values()):
            c.device_free(p)
        # solver entry point
        dense = synth.make_dense_factors(small, seed=5)
        Sa, ga = c.reduced_system(small, dense, abi.LOSS_CAUCHY)
        Sb, gb = c.reduced_system(small, dense, abi.LOSS_CAUCHY, line_table=True)
        assert np.abs(Sb - Sa).max() <= 1e-12 * np.abs(Sa).max() and np.abs(gb - ga).max() <= 1e-12 * np.abs(ga).max()
        # an index outside the map
        bad = small.slice_windows(0, 10)
        bad.lf_map_index = bad.lf_map_index.copy()
        bad.lf_map_index[3] = len(lmap)
        with pytest.raises(pkg.VimlError):
            c.linearize(bad, flags, line_table=True)


def test_small_batch_staging_matches_pipeline(pkg, ctx, cfg):
    """Host-pointer calls on small batches go through one pinned staging block each way (one H2D, one D2H); batches of 512
    windows and more go through the chunked copy pipeline.  The first 12 windows of a 600-window batch equal the same windows
    sliced out and sent alone: every mode, both observation forms."""
    abi = pkg._abi
    b = pkg.synth.make_windows(600, seed=181)
    small = b.slice_windows(0, 12)
    n = {"pf_": int(b.pf_window_offset[12]), "lf_": int(b.lf_window_offset[12])}
    for flags in (abi.OUT_RESIDUAL_JACOBIAN, abi.OUT_SCHUR | abi.LOSS_CAUCHY, abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_SCHUR,
                  abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY):
        for table in (False, True):
            staged = ctx.linearize(small, flags, obs_table=table)
            piped = ctx.linearize(b, flags, obs_table=table)
            assert set(staged) == set(piped)
            for k, v in piped.items():
                assert not np.isnan(staged[k]).any(), k
                if k.startswith(("pf_", "lf_")):
                    assert np.array_equal(staged[k], v[:n[k[:3]]]), k
                else:
                    assert pkg.parity.unit_err(k, staged[k], v[:12]) < 1e-12, k


def test_device_pointer_mode_matches_host_mode(pkg, ctx, cfg):
    """VIML_PTRS_DEVICE: inputs resident in HBM, asynchronous on the context stream."""
    abi = pkg._abi
    b = pkg.synth.make_windows(16, seed=111)
    flags = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    host = ctx.linearize(b, flags)
    d_in = {k: ctx.to_device(v) for k, v in b.arrays().items() if v is not None}
    d_out = {k: ctx.device_alloc(v.nbytes) for k, v in host.items()}
    ctx.linearize_raw(b.struct(d_in), abi.out_struct(d_out), flags | abi.PTRS_DEVICE)
    for k, v in host.items():
        back = np.empty_like(v)
        ctx.d2h(back, d_out[k])
        ctx.sync()
        if k in ("pf_residual", "pf_jac_pose_i", "pf_jac_pose_j", "pf_jac_ex", "pf_jac_feat", "lf_residual", "lf_jac_pose"):
            assert np.array_equal(back, v), k        # per-factor outputs are deterministic
        else:
            assert rel_err(back, v) < 1e-12, k       # assembled sums may differ in summation order only
    for p in list(d_in.values()) + list(d_out.values()):
        ctx.device_free(p)


def test_full_size_batch_properties(pkg, orc, ctx, cfg):
    """BASELINE.json configs[1] at full size (4096 windows): oracle on a sample of windows + properties."""
    abi = pkg._abi
    b = pkg.synth.make_windows(4096, seed=0x5EED + 2)
    flags = abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    got = ctx.linearize(b, flags)
    for k, v in got.items():
        assert np.isfinite(v).all(), k
    H = got["H_pp"]
    assert np.abs(H - np.swapaxes(H, 1, 2)).max() <= 1e-9 * np.abs(H).max()
    S = got["S"]
    assert np.abs(S - np.swapaxes(S, 1, 2)).max() <= 1e-9 * np.abs(S).max()
    # S is H_pp minus a PSD term: diagonal can only shrink
    assert np.all(np.einsum("wii->wi", S) <= np.einsum("wii->wi", H) * (1 + 1e-12) + 1e-9)
    # 256 of the 4096 windows against the oracle, per unit (per 6x6 block / landmark row)
    for w0 in (0, 777, 2048, 4032):
        sb = b.slice_windows(w0, w0 + 64)
        ref = orc.linearize_batch(cfg, sb, flags, nthreads=8)
        for k, v in ref.items():
            e = pkg.parity.unit_err(k, got[k][w0:w0 + 64], v)
            assert e < TOL, (k, w0, e)
    # linearity in the factor set: H(all) == H(first half of windows) ++ H(second half)
    half = ctx.linearize(b.slice_windows(0, 2048), abi.OUT_HB | abi.LOSS_CAUCHY)
    assert rel_err(half["H_pp"], got["H_pp"][:2048]) < 1e-12


def test_huge_window_partition_sums_to_full(pkg, orc, ctx, cfg):
    """cfg-5b shape (one long window) at a size the dense oracle handles: the per-rank partial [S | g] of the
    landmark partition (shard.split_huge_window) sum to the single-GPU result (what the NCCL all-reduce does)."""
    abi, synth, shard = pkg._abi, pkg.synth, pkg.shard
    huge = synth.make_windows(1, seed=121, P=40, F=300, lines_per_frame=2, max_len=12)
    flags = abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    got, ref = check_linearize(pkg, orc, ctx, cfg, huge, flags)
    acc = np.zeros(huge.D * huge.D + huge.D)
    owned = 0
    for r in range(4):
        part = shard.split_huge_window(huge, r, 4)
        owned += part.NP + part.NL
        o = ctx.linearize(part, abi.OUT_SCHUR | abi.LOSS_CAUCHY)
        acc += shard.pack_sg(o["S"][0], o["g"][0])
    assert owned == huge.NP + huge.NL
    accS, accg = shard.unpack_sg(acc, huge.D)
    assert pkg.parity.unit_err("S", accS[None], ref["S"]) < TOL and pkg.parity.unit_err("g", accg[None], ref["g"]) < TOL


# ---- whole-window reduced system and the Gauss-Newton step (SURVEY 8f ranks 1, 2) -----------------------------------
def make_dense(pkg, batch, seed=5):
    return pkg.synth.make_dense_factors(batch, seed)


def block_err(got, ref, bounds):
    """max over windows and (block row, block col) of max|d| / max|ref| with the given block boundaries."""
    worst = 0.0
    nb = len(bounds) - 1
    for i in range(nb):
        for j in range(nb if got.ndim == 3 else 1):
            if got.ndim == 3:
                g, r = got[:, bounds[i]:bounds[i + 1], bounds[j]:bounds[j + 1]], ref[:, bounds[i]:bounds[i + 1], bounds[j]:bounds[j + 1]]
            else:
                g, r = got[:, bounds[i]:bounds[i + 1]], ref[:, bounds[i]:bounds[i + 1]]
            sc = np.abs(r).reshape(len(r), -1).max(axis=1)
            df = np.abs(g - r).reshape(len(r), -1).max(axis=1)
            e = np.where(sc > 0, df / np.where(sc > 0, sc, 1.0), np.where(df == 0, 0.0, np.inf))
            worst = max(worst, float(e.max()))
    return worst


def check_reduced_system_and_gn_step(pkg, orc, ctx, cfg, b, flags):
    """viml_reduced_system and viml_gn_step (lambda = 0 and 1e-3) on batch b with make_dense's factors against the oracle;
    returns (dense, extra)."""
    from oracle import gn_oracle
    abi = pkg._abi
    dense = make_dense(pkg, b)
    P, D, X = b.P, b.D, dense.X
    bounds = [6 * k for k in range(P + 2)] + [D + 9 * k for k in range(1, P + 1)]
    Sx, gx = ctx.reduced_system(b, dense, flags)
    rSx, rgx, _ = gn_oracle.reduced_system(cfg, b, dense, flags)
    assert block_err(Sx, rSx, bounds) < TOL and block_err(gx, rgx, bounds) < TOL
    # without dense factors: the embedding of S, g
    S0, g0 = ctx.reduced_system(b, None, flags)
    r0 = orc.linearize_batch(cfg, b, abi.OUT_SCHUR | abi.LOSS_CAUCHY)
    assert pkg.parity.unit_err("S", S0, r0["S"]) < TOL and pkg.parity.unit_err("g", g0, r0["g"]) < TOL
    extra = 0.1 * np.random.default_rng(3).standard_normal((b.W, X))
    for lam in (0.0, 1e-3):
        got = ctx.gn_step(b, dense, extra, flags, lam=lam)
        ref = gn_oracle.gn_step(cfg, b, dense, extra, flags, lam=lam)
        assert np.array_equal(got["solved"], ref["solved"]) and got["solved"].all()
        assert block_err(got["dx"], ref["dx"], bounds) < TOL
        for k in ("poses", "ex_pose"):
            assert np.abs(got[k] - ref[k]).max() < 1e-9 * max(1.0, np.abs(ref[k]).max()), k
        # inverse depths / extra state: the increments are what is computed
        dl_g, dl_r = got["inv_depth"] - b.inv_depth, ref["inv_depth"] - b.inv_depth
        assert np.abs(dl_g - dl_r).max() < 1e-9 * np.abs(dl_r).max()
        assert np.abs(got["extra"] - ref["extra"]).max() < 1e-9 * np.abs(ref["extra"]).max()
        assert np.abs(got["cost"] - ref["cost"]).max(axis=0).max() < 1e-9 * np.abs(ref["cost"]).max()
        rel = np.abs(got["cost"] - ref["cost"]) / np.maximum(np.abs(ref["cost"]), 1e-300)
        assert rel.max() < 1e-9, rel.max()
        # identical accept / reject decisions, and the step does decrease the cost on these windows
        assert np.array_equal(got["cost"][:, 1] < got["cost"][:, 0], ref["cost"][:, 1] < ref["cost"][:, 0])
        assert (got["cost"][:, 2] > 0).all()
    return dense, extra


def test_reduced_system_and_gn_step(pkg, orc, ctx, cfg):
    from oracle import gn_oracle
    abi, synth = pkg._abi, pkg.synth
    flags = abi.LOSS_CAUCHY
    b = synth.make_windows(12, seed=141)
    dense, extra = check_reduced_system_and_gn_step(pkg, orc, ctx, cfg, b, flags)
    # P = 13: Dx = 201 is too large for the step's single kernel (reduced_kernel, then the tiled solve), and H / b come from the
    # generic atomic kernels (P > 12)
    check_reduced_system_and_gn_step(pkg, orc, ctx, cfg, synth.make_windows(12, seed=141, P=13), flags)
    # a few iterations from a perturbed state converge (cost decreases monotonically when every step is accepted)
    cur = b
    costs = []
    ex_state = extra
    for it in range(3):
        o = ctx.gn_step(cur, dense, ex_state, flags, lam=1e-4)
        costs.append(o["cost"][:, 0].sum())
        cur = abi.Batch(o["poses"], o["ex_pose"], o["inv_depth"], b.pf_window_offset, b.pf_idx, b.pf_obs, b.lf_window_offset, b.lf_frame, b.lf_geom)
        ex_state = o["extra"]
    assert costs[1] < costs[0]
    # a singular system (no dense factors, lambda = 0: gauge freedom) is reported, not solved, and the state comes back unchanged
    o = ctx.gn_step(b.slice_windows(0, 2), None, None, flags, lam=0.0)
    r = gn_oracle.gn_step(cfg, b.slice_windows(0, 2), None, None, flags, lam=0.0)
    assert np.array_equal(o["solved"], r["solved"])
    for w in range(2):
        if not o["solved"][w]:
            assert np.array_equal(o["poses"][w], b.poses[w]) and np.array_equal(o["inv_depth"][w], b.inv_depth[w])


def test_fov_cache_and_window_bookkeeping(pkg, orc, cfg):
    """SURVEY 8f rank 3: the per-slot FoV lists live on the device (viml_fov_update), move with the window (viml_fov_slide, both
    marginalisation flags, estimator.cpp:2148, :2160, :2218) and are matched against under the CURRENT poses (VIML_FOV_CACHED):
    bit for bit what the oracle gives for the frame-entry cull pose of whatever frame sits in each slot."""
    abi, synth = pkg._abi, pkg.synth
    ext = (150.0, 150.0, 20.0)
    lines = synth.make_line_map(6000, extent=ext)
    n = 16   # frames of a little sequence; the window holds 11 of them
    cull, match, ex, l2d = synth.make_assoc_queries(lines, n, L=40, n_true=14, extent=ext, pose_drift=True)
    with pkg.Context(cfg) as c:
        c.set_map(lines)
        frames = list(range(11))            # frame index sitting in each slot
        for s in range(11):
            c.fov_update(s, cull[s], ex[s])

        def check(frames):
            idx = np.array(frames)
            got = c.associate(None, match[idx], ex[idx], l2d[idx], cached=True, fov_capacity=600, want_mask=True)
            ref = orc.line_associate(cfg, lines, cull[idx], match[idx], ex[idx], l2d[idx], fov_capacity=600, want_mask=True)
            check_assoc(got, ref)

        check(frames)
        nxt = 11
        for flag_old in (True, False, True, True, False):
            c.fov_slide(flag_old)
            if flag_old:
                frames = frames[1:] + [frames[-1]]
            else:
                frames[9] = frames[10]
            check(frames)
            cnt = c.fov_update(10, cull[nxt], ex[nxt])    # the next frame enters the newest slot
            frames[10] = nxt
            assert cnt == orc.line_associate(cfg, lines, cull[nxt:nxt + 1], None, ex[nxt:nxt + 1], l2d[nxt:nxt + 1])["fov_count"][0]
            nxt += 1
            check(frames)
        # explicit slot map: poses in arbitrary slot order
        order = [7, 2, 10, 0]
        idx = np.array([frames[s] for s in order])
        got = c.associate(None, match[idx], ex[idx], l2d[idx], cached=True, fov_slot=order, want_mask=True)
        ref = orc.line_associate(cfg, lines, cull[idx], match[idx], ex[idx], l2d[idx], want_mask=True)
        check_assoc(got, ref)
        # a new map drops the cache: every slot is empty until updated again
        c.set_map(lines[:3000])
        got = c.associate(None, match[:3], ex[:3], l2d[:3], cached=True)
        assert np.all(got["match_index"] == -1) and np.all(got["fov_count"] == 0)


def test_track_gate(pkg, orc, cfg):
    """FeatureManager::removeLineOutlier on the device against the oracle's restatement (feature_manager.cpp:494-541)."""
    rng = np.random.default_rng(11)
    lines = pkg.synth.make_line_map(500, extent=(40.0, 40.0, 10.0))
    # make near-duplicates so that some LineVec differences fall on both sides of 0.1 m
    lines[250:] = lines[:250] + rng.normal(0, 0.03, (250, 6))
    T = 300
    nobs = rng.integers(0, 12, T)
    off = np.concatenate([[0], np.cumsum(nobs)]).astype(np.int32)
    idx = np.empty(off[-1], dtype=np.int32)
    for t in range(T):
        base = rng.integers(0, 250)
        pick = rng.choice([base, base + 250, rng.integers(0, 500), -1], size=nobs[t], p=[0.5, 0.3, 0.15, 0.05])
        idx[off[t]:off[t + 1]] = pick
    with pkg.Context(cfg) as c:
        c.set_map(lines)
        cl, cm = c.track_gate(off, idx)
    vec = np.where((idx >= 0)[:, None], lines[np.maximum(idx, 0), 3:] - lines[np.maximum(idx, 0), :3], 0.0)
    for t in range(T):
        if nobs[t] == 0:
            assert cm[t]
            continue
        ref_cm, ref_cl = orc.track_gate(vec[off[t]:off[t + 1]])
        assert bool(cm[t]) == bool(ref_cm), t
        assert np.array_equal(cl[off[t]:off[t + 1]], np.asarray(ref_cl, dtype=bool)), t


def test_triangulate_batch(pkg, ctx, cfg):
    """FeatureManager::triangulate (feature_manager.cpp:440-492) for a batch: the DLT rows restated with numpy and
    numpy.linalg.svd standing in for Eigen::JacobiSVD; depth = V[2] / V[3], INIT_DEPTH below 0.1."""
    synth = pkg.synth
    b = synth.make_windows(6, seed=161)
    P = b.P

    def rot(q7):
        q = q7[3:7] / np.linalg.norm(q7[3:7])
        return synth._rot_from_quat(q)

    fw, sf, off, pts, ref = [], [], [0], [], []
    rng = np.random.default_rng(2)
    for w in range(b.W):
        k0, k1 = b.pf_window_offset[w], b.pf_window_offset[w + 1]
        idx = b.pf_idx[k0:k1]
        feat = idx >> 16
        for l in np.unique(feat)[:60]:
            sel = np.nonzero(feat == l)[0]
            i = int(idx[sel[0]] & 0xff)
            js = sorted(int((idx[s] >> 8) & 0xff) for s in sel)
            if js != list(range(i + 1, i + 1 + len(js))):
                continue
            obs = [np.array([b.pf_obs[k0 + sel[0], 0], b.pf_obs[k0 + sel[0], 1], 1.0])]
            for j in js:
                s = sel[[int((idx[t] >> 8) & 0xff) for t in sel].index(j)]
                obs.append(np.array([b.pf_obs[k0 + s, 2], b.pf_obs[k0 + s, 3], 1.0]))
            if rng.uniform() < 0.1:
                obs = obs[:1]          # a single observation: rank-deficient system, still defined
            ric, tic = rot(b.ex_pose[w]), b.ex_pose[w, :3]
            R0 = rot(b.poses[w, i]) @ ric
            t0 = b.poses[w, i, :3] + rot(b.poses[w, i]) @ tic
            rows = []
            for k, p in enumerate(obs):
                R1 = rot(b.poses[w, i + k]) @ ric
                t1 = b.poses[w, i + k, :3] + rot(b.poses[w, i + k]) @ tic
                t, R = R0.T @ (t1 - t0), R0.T @ R1
                Pm = np.concatenate([R.T, (-R.T @ t)[:, None]], 1)
                f = p / np.linalg.norm(p)
                rows += [f[0] * Pm[2] - f[2] * Pm[0], f[1] * Pm[2] - f[2] * Pm[1]]
            A = np.array(rows)
            if len(obs) < 2:
                continue
            V = np.linalg.svd(A)[2][-1]
            d = V[2] / V[3]
            ref.append(5.0 if d < 0.1 else d)
            fw.append(w), sf.append(i), pts.extend(obs), off.append(off[-1] + len(obs))
    got = ctx.triangulate(b.poses, b.ex_pose, fw, sf, off, np.array(pts), init_depth=5.0)
    ref = np.array(ref)
    assert len(ref) > 200
    assert np.abs(got - ref).max() < 1e-9 * np.abs(ref).max(), np.abs(got - ref).max()
    assert np.all(np.abs(got - ref) <= 1e-7 * np.abs(ref))     # per feature (the DLT null vector amplifies rounding by the system's conditioning)


def test_triangulate_against_reference_vectors(pkg, ctx):
    """viml_triangulate_batch against depths the reference's own FeatureManager::triangulate produced (tests/golden/ref_factors.npz)."""
    g = np.load(os.path.join(GOLD, "ref_factors.npz"))
    got = ctx.triangulate(g["tri_poses"][None], g["tri_ex"][None], np.zeros(len(g["tri_start"]), dtype=np.int32), g["tri_start"], g["tri_off"],
                          g["tri_pts"], init_depth=5.0)
    assert np.all(np.abs(got - g["tri_depth"]) <= 1e-7 * np.abs(g["tri_depth"]))
    assert np.abs(got - g["tri_depth"]).max() < 1e-9 * np.abs(g["tri_depth"]).max()


def test_load_line_map(pkg, cfg, tmp_path):
    """viml_load_line_map reads line_3d.txt the way parameters.cpp:50-59 does and gives the same association as viml_set_map."""
    synth = pkg.synth
    lines = synth.make_line_map(3000, extent=(120.0, 120.0, 20.0))
    path = tmp_path / "line_3d.txt"
    with open(path, "w") as f:
        for r in lines:
            f.write(" ".join(repr(float(v)) for v in r) + "\n")
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 6, L=40, n_true=16, extent=(120.0, 120.0, 20.0))
    with pkg.Context(cfg) as c1, pkg.Context(cfg) as c2:
        assert c1.load_line_map(str(path)) == len(lines)
        c2.set_map(lines)
        a1, a2 = c1.associate(cull, match, ex, l2d, want_mask=True), c2.associate(cull, match, ex, l2d, want_mask=True)
        for k in a1:
            assert np.array_equal(a1[k], a2[k], equal_nan=True), k
        assert c1.lib.viml_load_line_map(c1.h, b"/nonexistent/line_3d.txt", None) == pkg._abi.VIML_ERR_INVALID


# ---- marginalisation ----------------------------------------------------------------------------------
def test_marginalize_dense(pkg, orc, ctx):
    rng = np.random.default_rng(7)
    for pos, m, K in ((90, 15, 5), (37, 0, 2), (120, 45, 3), (16, 15, 4)):
        A = np.empty((K, pos, pos))
        b = rng.standard_normal((K, pos))
        for k in range(K):
            M = rng.standard_normal((pos + 8, pos))
            A[k] = M.T @ M
        got = ctx.marginalize(A, b, m)
        for k in range(K):
            As, bs, lj, lr = orc.marginalize_dense(A[k], b[k], m)
            assert rel_err(got["A_schur"][k], As) < TOL and rel_err(got["b_schur"][k], bs) < TOL
            J, r = got["linearized_jacobians"][k], got["linearized_residuals"][k]
            # eigenvector signs are not unique: compare J^T J and J^T r (SURVEY.md A.3)
            assert rel_err(J.T @ J, lj.T @ lj) < TOL and rel_err(J.T @ r, lj.T @ lr) < 1e-8
    # rank-deficient marginalised block -> pseudo-inverse semantics
    pos, m = 40, 12
    M = rng.standard_normal((pos + 3, pos))
    A = M.T @ M
    A[2, :] = 0
    A[:, 2] = 0
    b = rng.standard_normal(pos)
    got = ctx.marginalize(A, b, m)
    As, bs, _, _ = orc.marginalize_dense(A, b, m)
    assert rel_err(got["A_schur"][0], As) < 1e-8 and rel_err(got["b_schur"][0], bs) < 1e-8


# ---- association -----------------------------------------------------------------------------------------
def check_assoc(got, ref, check_lists=True):
    assert np.array_equal(got["match_index"], ref["match_index"])
    assert np.array_equal(got["fov_count"], ref["fov_count"])
    if "fov_mask" in ref:
        assert np.array_equal(got["fov_mask"], ref["fov_mask"])
    if "fov_index" in ref and check_lists:
        assert np.array_equal(got["fov_index"], ref["fov_index"])
    m = ref["match_index"] >= 0
    # errD and overlap (float32) and the projected segment are bit-exact
    assert np.array_equal(got["err"][..., 1:], ref["err"][..., 1:], equal_nan=True)   # NaN = untouched ragged entries
    # every processed query, matched or not (an unmatched query returns the detected line itself, est.cpp:709, :874);
    # NaN = untouched ragged entries
    assert np.array_equal(got["projected"], ref["projected"], equal_nan=True)
    # errA goes through acos: device acos is <= 2 ulp in double, i.e. <= 1 ulp after narrowing to float
    a, b = got["err"][..., 0], ref["err"][..., 0]
    assert np.array_equal(np.isnan(a), np.isnan(b))
    a, b = np.nan_to_num(a), np.nan_to_num(b)
    assert np.all(np.abs(a - b) <= np.spacing(np.abs(b)).astype(np.float32))
    return float((a == b).mean())


@pytest.mark.parametrize("name", ["assoc_euroc_v1.npz", "assoc_euroc_v2.npz"])
def test_golden_association_on_reference_maps(pkg, name):
    g = np.load(os.path.join(GOLD, name))
    c = g["cfg"]
    cfg = pkg._abi.make_config(fx=c[0], fy=c[1], cx=c[2], cy=c[3], width=int(c[4]), height=int(c[5]), Rbw=g["Rbw"],
                               Tbw=g["Tbw"], overlap_th=c[6], dist_th=c[7], angle_th=c[8])
    with pkg.Context(cfg) as cx:
        cx.set_map(g["lines"])
        got = cx.associate(g["cull"], g["match"], g["ex"], g["lines2d"], fov_capacity=512)
    ref = {k: g[k] for k in ("match_index", "err", "projected", "fov_count", "fov_index")}
    check_assoc(got, ref)


def test_association_against_reference_vectors(pkg):
    """tests/golden/ref_assoc.npz was written by the REFERENCE's own UpdateLinesInFoV / LineCorrespondenceInFrame / CalAngleDist /
    CalEulerDist (oracle/ref_estimator.cpp; tests/golden/make_ref_golden.py) on threshold-hugging queries: the CUDA path gives the
    same FoV lists, map indices, errD, overlap and projected segments bit for bit (errA within 1 float ulp: device acos)."""
    g = np.load(os.path.join(GOLD, "ref_assoc.npz"))
    for c in range(int(g["n_cases"])):
        cfg = pkg.synth.euroc_config(angle_th=float(g[f"c{c}_angle_th"]), overlap_th=float(g[f"c{c}_overlap_th"]))
        cex = g[f"c{c}_cull_ex"] if f"c{c}_cull_ex" in g.files else None
        nl = g[f"c{c}_n_lines2d"] if f"c{c}_n_lines2d" in g.files else None
        L = g[f"c{c}_lines2d"].shape[1]
        with pkg.Context(cfg) as cx:
            cx.set_map(g["lines"])
            got = cx.associate(g[f"c{c}_cull"], g[f"c{c}_match"], g[f"c{c}_ex"], g[f"c{c}_lines2d"], n_lines2d=nl,
                               fov_capacity=int(g[f"c{c}_fov_capacity"]), cull_ex_pose=cex)
        ref = {k: g[f"c{c}_{k}"].copy() for k in ("match_index", "err", "projected", "fov_count", "fov_index")}
        if nl is not None:   # rows beyond a pose's own count are not outputs: compare the filler of the wrapper to itself
            inval = np.arange(L)[None, :] >= nl[:, None]
            for k in ("match_index", "err", "projected"):
                ref[k][inval] = got[k][inval]
        check_assoc(got, ref)


def test_association_synthetic(pkg, orc, ctx, cfg):
    synth = pkg.synth
    lines = synth.make_line_map(60000, seed=41, extent=(500.0, 500.0, 30.0))
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 97, L=300, n_true=100, seed=42, extent=(500.0, 500.0, 30.0))
    ctx.set_map(lines)
    got = ctx.associate(cull, match, ex, l2d, fov_capacity=2048, want_mask=True)
    ref = orc.line_associate(cfg, lines, cull, match, ex, l2d, fov_capacity=2048, want_mask=True, nthreads=8)
    exact = check_assoc(got, ref)
    assert (ref["match_index"] >= 0).mean() > 0.2 and exact > 0.99
    um = ref["match_index"] == -1   # an unmatched query returns the detected line itself (est.cpp:874)
    assert um.any() and np.array_equal(got["projected"][um], l2d[um]) and np.array_equal(ref["projected"][um], l2d[um])
    # same pose for cull and match (match_poses = NULL), as the cfg-3 sweep does
    got = ctx.associate(cull, None, ex, l2d)
    ref = orc.line_associate(cfg, lines, cull, None, ex, l2d, nthreads=8)
    check_assoc(got, ref)


def test_hierarchical_cull_equals_brute_force_sweep(pkg, orc, cfg):
    """The tile-rejection cull (default) and the literal all-pairs sweep (VIML_BRUTE_CULL=1) give identical masks,
    counts, lists and matches; both equal the oracle on a sample of poses."""
    synth = pkg.synth
    ext = (600.0, 600.0, 30.0)
    lines = synth.make_line_map(100001, seed=51, extent=ext)            # not a multiple of the 256-line tile
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 70, L=48, n_true=20, seed=52, extent=ext)
    # a few poses that look at the horizon: huge FoV lists, tiles straddling every frustum plane
    h = np.sqrt(0.5)
    cull[3, 3:7] = [h, 0.0, 0.0, h]      # body z (the camera axis, up to the extrinsic) turned horizontal
    cull[4, 3:7] = [0.0, h, 0.0, h]
    match[3], match[4] = cull[3], cull[4]
    res = {}
    for mode in ("0", "1"):
        os.environ["VIML_BRUTE_CULL"] = mode
        try:
            with pkg.Context(cfg) as cx:
                cx.set_map(lines)
                res[mode] = cx.associate(cull, match, ex, l2d, fov_capacity=8192, want_mask=True)
        finally:
            del os.environ["VIML_BRUTE_CULL"]
    for k in res["0"]:
        assert np.array_equal(res["0"][k], res["1"][k], equal_nan=True), k
    sel = np.array([0, 3, 4, 69])
    ref = orc.line_associate(cfg, lines, cull[sel], match[sel], ex[sel], l2d[sel], fov_capacity=8192, want_mask=True, nthreads=8)
    check_assoc({k: v[sel] for k, v in res["0"].items()}, ref)
    assert max(res["0"]["fov_count"][3], res["0"]["fov_count"][4]) > 2 * np.median(res["0"]["fov_count"])


def test_association_edges(pkg, orc, ctx, cfg):
    synth = pkg.synth
    lines = synth.make_line_map(777, seed=43, extent=(60.0, 60.0, 30.0))   # N not a multiple of 32
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 5, L=16, n_true=8, seed=44, extent=(60.0, 60.0, 30.0))
    l2d[0, 0] = [100, 100, 100, 100]      # zero-length detected line
    l2d[0, 1] = [200, 50, 200, 300]       # vertical: Point2Flined always clamps to an endpoint
    ctx.set_map(lines)
    nl = np.array([16, 0, 3, 16, 1], dtype=np.int32)
    got = ctx.associate(cull, match, ex, l2d, n_lines2d=nl, fov_capacity=64, want_mask=True)
    ref = orc.line_associate(cfg, lines, cull, match, ex, l2d, n_lines2d=nl, fov_capacity=64, want_mask=True)
    check_assoc(got, ref)                 # includes truncated fov_index (capacity 64) and untouched -2 entries
    # empty map
    ctx.set_map(np.zeros((0, 6)))
    got = ctx.associate(cull, match, ex, l2d)
    assert np.all(got["match_index"] == -1) and np.all(got["err"] == -1) and np.all(got["fov_count"] == 0)
    # poses looking away from everything: empty FoV lists
    ctx.set_map(lines + 1e5)
    got = ctx.associate(cull, match, ex, l2d)
    assert np.all(got["match_index"] == -1) and np.all(got["fov_count"] == 0)


def test_association_frame_entry_extrinsic(pkg, orc, ctx, cfg):
    """UpdateLinesInFoV runs at frame entry with the extrinsic of that moment (est.cpp:385), the match with the
    re-optimised one: cull_ex_pose != ex_pose, with and without a separate match pose, host chunks included (640 poses)."""
    synth = pkg.synth
    ext = (400.0, 400.0, 30.0)
    lines = synth.make_line_map(40000, seed=81, extent=ext)
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 640, L=24, n_true=12, seed=82, extent=ext)
    rng = np.random.Generator(np.random.PCG64(83))
    cex = ex.copy()
    cex[:, :3] += 0.01 * rng.standard_normal((len(ex), 3))
    cex[:, 3:] += 0.002 * rng.standard_normal((len(ex), 4))        # un-normalised on purpose: the path normalises
    ctx.set_map(lines)
    sel = np.array([0, 1, 159, 160, 319, 320, 479, 480, 639])       # both sides of every host-pipeline chunk boundary
    for m in (match, None):
        got = ctx.associate(cull, m, ex, l2d, fov_capacity=1024, want_mask=True, cull_ex_pose=cex)
        ref = orc.line_associate(cfg, lines, cull[sel], None if m is None else m[sel], ex[sel], l2d[sel], fov_capacity=1024,
                                 want_mask=True, nthreads=8, cull_ex_pose=cex[sel])
        check_assoc({k: v[sel] for k, v in got.items()}, ref)
    plain = ctx.associate(cull, match, ex, l2d, fov_capacity=1024)
    assert not np.array_equal(plain["fov_count"], got["fov_count"]) or not np.array_equal(plain["fov_index"], got["fov_index"])


def test_association_long_fov_lists(pkg, orc, ctx, cfg):
    """FoV lists longer than the match kernel's shared-memory stage (2048 candidate directions): the tail of the list
    is gated straight from the candidate arrays; same bits as the oracle, and the winners do come from the tail."""
    synth = pkg.synth
    ext = (70.0, 70.0, 30.0)
    lines = synth.make_line_map(9000, seed=71, extent=ext)
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 130, L=48, n_true=24, seed=72, extent=ext)
    ctx.set_map(lines)
    got = ctx.associate(cull, match, ex, l2d, fov_capacity=8192, want_mask=True)
    assert got["fov_count"].max() > 2600
    sel = np.argsort(-got["fov_count"])[:6]                       # the longest lists
    ref = orc.line_associate(cfg, lines, cull[sel], match[sel], ex[sel], l2d[sel], fov_capacity=8192, want_mask=True, nthreads=8)
    sub = {k: v[sel] for k, v in got.items()}
    check_assoc(sub, ref)
    pos = [np.searchsorted(sub["fov_index"][i, :sub["fov_count"][i]], sub["match_index"][i][sub["match_index"][i] >= 0]) for i in range(len(sel))]
    assert max(p.max() for p in pos if len(p)) >= 2048           # some matches sit beyond the staged part of the list


def test_association_angle_threshold_variants(pkg, orc):
    synth = pkg.synth
    lines = synth.make_line_map(20000, seed=45, extent=(300.0, 300.0, 30.0))
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 12, L=64, n_true=30, seed=46, extent=(300.0, 300.0, 30.0))
    for th, ov in ((0.1, 0.5), (0.18, 0.5), (0.3491, 0.3), (3.2, 0.0)):   # last: angle_th > PI lets NaN angles pass
        cfg = synth.euroc_config(angle_th=th, overlap_th=ov)
        with pkg.Context(cfg) as cx:
            cx.set_map(lines)
            got = cx.associate(cull, match, ex, l2d, want_mask=True)
        ref = orc.line_associate(cfg, lines, cull, match, ex, l2d, want_mask=True, nthreads=8)
        check_assoc(got, ref)


def test_division_with_hoisted_reciprocal_is_exact(ctx):
    """div_by (associate_kernels.cu) replays the compiler's division fast path with the reciprocal part computed once
    per divisor and falls back to `/` outside a narrower exponent range: every quotient must equal a / b bit for bit,
    over pixel-scale values, random bit patterns, subnormals, huge values, zeros, infinities and NaNs."""
    rng = np.random.Generator(np.random.PCG64(61))
    n = 1 << 21
    a = [rng.uniform(-2000, 2000, n), rng.uniform(0, 1e6, n) * rng.uniform(0, 1, n) ** 8]
    b = [rng.uniform(1e-3, 2000, n), rng.uniform(0, 800, n)]
    bits = rng.integers(0, 1 << 63, n, dtype=np.int64) * rng.choice([-1, 1], n)      # any finite / inf / NaN pattern
    a.append(bits.view(np.float64))
    b.append((rng.integers(0, 1 << 63, n, dtype=np.int64)).view(np.float64))
    mant = 1.0 + rng.integers(0, 16, n) * 2.0 ** -52                                  # mantissas next to 1 and 2
    mant2 = 2.0 - rng.integers(1, 16, n) * 2.0 ** -52
    a.append(np.concatenate([mant[: n // 2], mant2[n // 2:]]) * 2.0 ** rng.integers(-1030, 1020, n).astype(np.float64))
    b.append(np.concatenate([mant2[: n // 2], mant[n // 2:]]) * 2.0 ** rng.integers(-1030, 1020, n).astype(np.float64))
    special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, 2.2250738585072014e-308, 1.7976931348623157e308,
                        1.0, 10.0, 12.0, 3.0, 1e-200, 1e200])
    a.append(np.repeat(special, special.size))
    b.append(np.tile(special, special.size))
    with np.errstate(all="ignore"):
        for x, y in zip(a, b):
            assert ctx.selftest_division(x, y) == 0


def test_association_pruning_adversarial(pkg, orc):
    """The match kernel drops pairs through conservative overlap / distance bounds before the exact arithmetic.
    Queries built ON the thresholds: sub-segments of the projected map lines whose overlap sits within 1e-9 ... 1e-3
    of overlap_th on either side, over-long queries (the detected line becomes line2), exactly / nearly vertical and
    (near) zero-length segments, 3 px parallel offsets, duplicated map lines (distance ties -> list order)."""
    synth = pkg.synth
    ext = (300.0, 300.0, 30.0)
    lines = synth.make_line_map(20000, seed=51, extent=ext)
    lines = np.concatenate([lines, lines[:800]])                      # exact duplicates: equal distances
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 16, L=300, n_true=150, seed=52, extent=ext)
    rng = np.random.Generator(np.random.PCG64(53))
    for ang, ov in ((0.18, 0.8), (0.1, 0.5), (0.3, 0.0), (0.18, 1.0)):
        cfg = synth.euroc_config(angle_th=ang, overlap_th=ov)
        with pkg.Context(cfg) as cx:
            cx.set_map(lines)
            base = cx.associate(cull, None, ex, l2d)
            q = l2d.copy()
            for p in range(q.shape[0]):
                segs = base["projected"][p][base["match_index"][p] >= 0]
                if len(segs) == 0:
                    continue
                for i in range(q.shape[1]):
                    s = segs[i % len(segs)]
                    S, E = s[:2], s[2:]
                    d = E - S
                    Ls = np.hypot(*d)
                    if not np.isfinite(Ls) or Ls < 1e-6:
                        continue
                    u, n = d / Ls, np.array([-d[1], d[0]]) / Ls
                    eps = (0.0, 1e-9, -1e-9, 1e-6, -1e-6, 1e-4, -1e-4, 1e-3, -1e-3)[rng.integers(9)]
                    f = min(max(ov + eps, 1e-3), 1.0)
                    mode = i % 10
                    if mode == 0:
                        a, b = S, E
                    elif mode == 1:                                   # shorter query inside the candidate
                        a, b = S, S + f * Ls * u
                    elif mode == 2:                                   # hangs over the end, overlap part = f * L
                        a = S + (1 - f) * Ls * u
                        b = a + (f * Ls + 40.0) * u * (0.5 if f * Ls + 40.0 > Ls else 1.0)
                    elif mode == 3:                                   # longer query: candidate / query = f
                        ext_ = Ls / f - Ls
                        a, b = S - 0.3 * ext_ * u, E + 0.7 * ext_ * u
                    elif mode == 4:                                   # exactly vertical through the midpoint
                        mid = 0.5 * (S + E)
                        a, b = mid - [0, 0.4 * Ls], mid + [0, 0.4 * Ls]
                    elif mode == 5:                                   # nearly vertical
                        mid = 0.5 * (S + E)
                        a, b = mid - [5e-5, 0.4 * Ls], mid + [5e-5, 0.4 * Ls]
                    elif mode == 6:                                   # (near) zero length
                        mid = 0.5 * (S + E)
                        a, b = mid, mid + (1e-5 * u if i % 20 == 6 else 0.0)
                    elif mode == 7:                                   # parallel, 3 px off, same extent
                        a, b = S + 3 * n, E + 3 * n
                    elif mode == 8:                                   # reversed direction, float32-rounded
                        a, b = E.astype(np.float32), S.astype(np.float32)
                    else:                                             # rotated by about angle_th
                        c, si = np.cos(ang * (1 + eps)), np.sin(ang * (1 + eps))
                        r = np.array([c * d[0] - si * d[1], si * d[0] + c * d[1]])
                        a, b = S, S + r
                    q[p, i] = [a[0], a[1], b[0], b[1]]
            got = cx.associate(cull, None, ex, q, want_mask=True)
        ref = orc.line_associate(cfg, lines, cull, None, ex, q, want_mask=True, nthreads=8)
        check_assoc(got, ref)
        assert ov >= 1.0 or (ref["match_index"] >= 0).mean() > 0.3


def test_association_sweep_properties_large(pkg, orc, ctx, cfg):
    """cfg-3 geometry at 1/4 of the map and 1/16 of the poses: oracle on a sample of poses + invariants."""
    synth = pkg.synth
    ext = (1000.0, 1000.0, 30.0)
    lines = synth.make_line_map(250000, seed=47, extent=ext)
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 256, L=300, n_true=100, seed=48, extent=ext)
    ctx.set_map(lines)
    got = ctx.associate(cull, None, ex, l2d, fov_capacity=4096, want_mask=True)
    pop = np.array([sum(bin(int(x)).count("1") for x in row) for row in got["fov_mask"][:8]])
    assert np.array_equal(pop, got["fov_count"][:8])
    for p in range(8):   # every matched index is a member of that pose's FoV list; lists are sorted (map order)
        fl = got["fov_index"][p, :got["fov_count"][p]]
        assert np.all(np.diff(fl) > 0)
        mi = got["match_index"][p]
        assert np.all(np.isin(mi[mi >= 0], fl))
    sel = np.array([0, 1, 100, 255])
    ref = orc.line_associate(cfg, lines, cull[sel], None, ex[sel], l2d[sel], fov_capacity=4096, want_mask=True, nthreads=8)
    sub = {k: v[sel] for k, v in got.items()}
    check_assoc(sub, ref)


def test_two_devices_in_one_process(pkg, orc, cfg):
    """One process, a context on device 0 and one on device 1 (the model viml_create(device) offers): every kernel that needs a
    per-device attribute (dynamic shared memory of the fused assembly, the Schur and match kernels) must work on the second device
    too.  Skipped on a single-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    abi, synth = pkg._abi, pkg.synth
    b = synth.make_windows(24, seed=191)
    flags = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    ref = orc.linearize_batch(cfg, b, flags, nthreads=8)
    lines = synth.make_line_map(20000, seed=192, extent=(300.0, 300.0, 30.0))
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 4, L=100, n_true=50, seed=193, extent=(300.0, 300.0, 30.0))
    aref = orc.line_associate(cfg, lines, cull, match, ex, l2d, nthreads=4)
    for dev in (0, 1, 0):
        with pkg.Context(cfg, device=dev) as c:
            got = c.linearize(b, flags)
            for k, v in ref.items():
                assert pkg.parity.unit_err(k, got[k], v) < TOL, (dev, k)
            c.set_map(lines)
            a = c.associate(cull, match, ex, l2d)
            assert np.array_equal(a["match_index"], aref["match_index"]), dev


def test_allreduce_hb_two_gpus(pkg, cfg):
    """viml_allreduce_hb (the C++ hosts' all-reduce of partial [S | g], SURVEY 8e) with raw ncclComm_t handles: one
    process, two contexts on two devices, one thread per device.  Skipped on a single-GPU box."""
    import ctypes
    import threading
    import torch   # loads the bundled libnccl into the process, which is what the library dlopens
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    nccl = ctypes.CDLL("libnccl.so.2")
    comms = (ctypes.c_void_p * 2)()
    devs = (ctypes.c_int * 2)(0, 1)
    assert nccl.ncclCommInitAll(comms, 2, devs) == 0
    n = 72 * 72 + 72
    parts = [np.arange(n, dtype=np.float64) * (k + 1) + 0.25 * k for k in range(2)]
    ctxs = [pkg.Context(cfg, device=k) for k in range(2)]
    bufs = [c.to_device(p) for c, p in zip(ctxs, parts)]
    for c in ctxs:
        c.sync()
    rcs = [None, None]

    def run(k):
        rcs[k] = ctxs[k].lib.viml_allreduce_hb(ctxs[k].h, comms[k], bufs[k], n)
        ctxs[k].sync()

    th = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    [t.start() for t in th]
    [t.join(timeout=60) for t in th]
    assert rcs == [0, 0]
    for k in range(2):
        got = np.empty(n)
        ctxs[k].d2h(got, bufs[k])
        ctxs[k].sync()
        assert np.array_equal(got, parts[0] + parts[1])
        ctxs[k].device_free(bufs[k])
    for k in range(2):
        nccl.ncclCommDestroy(ctypes.c_void_p(comms[k]))
    for c in ctxs:
        c.close() if hasattr(c, "close") else None
