"""Host <-> device staging of the synchronous host-pointer calls.

A call whose staged arrays total at most 4 MB goes up in one copy and comes back in one; a larger one copies array by array.  The
first windows (problems) of a large call must equal the same windows sent alone: bit for bit where every kernel is
order-deterministic (no visual factors; the marginalisation), to 1e-12 per window where the visual pose blocks are summed through
atomics.  The linearisation pipeline (host pointers, W >= 512) must not overwrite what work still queued on the context stream reads."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FLAGS = 0x10   # VIML_LOSS_CAUCHY
ONE_COPY = 4 << 20
W_BIG, N = 32, 3


def _blind(pkg, b):
    """b without its point and line factors."""
    return pkg._abi.Batch(b.poses, b.ex_pose, b.inv_depth, np.zeros(b.W + 1, dtype=np.int32), np.zeros(0, dtype=np.uint32),
                          np.zeros((0, 4)))


def _first_vi(pkg, vi, n):
    """The inertial factors of windows [0, n)."""
    k = int(vi.imu_window_offset[n])
    return pkg._abi.Inertial(n, vi.P, vi.X, vi.gravity, vi.imu_window_offset[:n + 1], vi.imu_pose[:k], vi.imu_sb[:k],
                             vi.imu_preint[:k], vi.imu_jacobian[:k], vi.imu_sqrt_info[:k], vi.prior_n[:n], vi.prior_jacobian[:n],
                             vi.prior_residual[:n], vi.prior_n_blocks[:n], vi.prior_block[:n], vi.prior_x0[:n])


def _window_err(got, ref):
    """max over windows of max|got - ref| / max|ref| inside the window (a window whose reference is all zeros must match exactly)."""
    g, r = got.reshape(len(got), -1), ref.reshape(len(ref), -1)
    assert np.array_equal(np.isnan(g), np.isnan(r))
    g, r = np.nan_to_num(g), np.nan_to_num(r)
    scale, diff = np.abs(r).max(axis=1), np.abs(g - r).max(axis=1)
    return float(np.where(scale > 0, diff / np.where(scale > 0, scale, 1.0), np.where(diff == 0, 0.0, np.inf)).max())


def _same_windows(big, small, exact):
    for k, v in small.items():
        head = big[k][:len(v)]
        if exact or v.dtype.kind == "i":
            assert np.array_equal(head, v, equal_nan=True), k
        else:
            assert _window_err(head, v) < 1e-12, k


@pytest.mark.parametrize("visual", [False, True], ids=["no_visual", "visual"])
def test_small_calls_match_large_calls(pkg, ctx, visual):
    synth = pkg.synth
    b = synth.make_windows(W_BIG, seed=311)
    assert W_BIG * 8 * b.D * (2 * b.D + b.F) > ONE_COPY   # H_pp, S and H_lp alone: the large call copies array by array
    vi, extra = synth.make_inertial_factors(b, seed=313)
    dense = synth.make_dense_factors(b, seed=317)
    if not visual:
        b = _blind(pkg, b)
    s, vs, es = b.slice_windows(0, N), _first_vi(pkg, vi, N), extra[:N]
    ds = pkg._abi.Dense(N, dense.X, [f for f in dense.factors if f[0] < N])
    Sx, gx = ctx.reduced_system(b, dense, FLAGS)
    Sx1, gx1 = ctx.reduced_system(s, ds, FLAGS)
    _same_windows({"Sx": Sx, "gx": gx}, {"Sx": Sx1, "gx": gx1}, not visual)
    _same_windows(ctx.gn_step_vi(b, vi, extra, FLAGS, lam=1e-4), ctx.gn_step_vi(s, vs, es, FLAGS, lam=1e-4), not visual)
    _same_windows(ctx.solve_vi(b, vi, extra, FLAGS, max_iterations=3), ctx.solve_vi(s, vs, es, FLAGS, max_iterations=3), not visual)


MARG_OUT = ("A_schur", "b_schur", "linearized_jacobians", "linearized_residuals")


def _marginalize(pkg, c, A, b, m, skip):
    """viml_marginalize_batch with host buffers; the output named `skip` is passed as null."""
    abi = pkg._abi
    K, pos = A.shape[0], A.shape[1]
    n = pos - m
    res = {k: np.full((K, n, n) if k in ("A_schur", "linearized_jacobians") else (K, n), np.nan) for k in MARG_OUT if k != skip}
    i = abi.MargBatch()
    i.n_problems, i.pos, i.m, i.eps, i.A, i.b = K, pos, m, 1e-8, abi.ptr(A), abi.ptr(b)
    o = abi.MargOut()
    for k in MARG_OUT:
        setattr(o, k, abi.ptr(res.get(k)))
    c._check(c.lib.viml_marginalize_batch(c.h, C.byref(i), C.byref(o), 0))
    return res


def test_marginalize_small_calls_match_large_call(pkg, ctx):
    rng = np.random.default_rng(331)
    K, pos, m = 24, 160, 40
    assert K * pos * pos * 8 > ONE_COPY
    M = rng.standard_normal((K, pos + 8, pos))
    A = np.ascontiguousarray(np.einsum("kij,kil->kjl", M, M))
    b = rng.standard_normal((K, pos))
    for skip in (None,) + MARG_OUT:
        big = _marginalize(pkg, ctx, A, b, m, skip)
        for k in (1, 4):
            _same_windows(big, _marginalize(pkg, ctx, A[:k], b[:k], m, skip), True)


def test_pipeline_waits_for_the_context_stream(pkg, cfg):
    """Work left queued on the context stream still reads what it staged: the pose of viml_fov_update without the count, the
    expanded tables of a device-pointer viml_linearize_batch.  A host-pointer viml_linearize_batch of 600 windows issued at once
    must not overwrite them before they are read."""
    abi, synth = pkg._abi, pkg.synth
    flags = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    other = synth.make_windows(600, seed=341)
    ext = (300.0, 300.0, 30.0)
    lines = synth.make_line_map(100_000, extent=ext)
    cull, match, ex, l2d = synth.make_assoc_queries(lines, 1, L=64, n_true=24, extent=ext)
    with pkg.Context(cfg) as c:
        c.set_map(lines)
        c.linearize(other, flags)   # the arenas at their final size: no reallocation synchronises the device below
        pose, e = np.ascontiguousarray(cull[0]), np.ascontiguousarray(ex[0])
        c._check(c.lib.viml_fov_update(c.h, 5, abi.ptr(pose), abi.ptr(e), None))
        c.linearize(other, flags)
        got = c.associate(None, match, ex, l2d, cached=True, fov_slot=[5], want_mask=True)
        ref = c.associate(cull, match, ex, l2d, want_mask=True)
        for k in ("match_index", "fov_count", "fov_mask"):
            assert np.array_equal(got[k], ref[k]), k

        b = synth.make_windows(600, seed=343, f32_obs=True)
        host = c.linearize(b, flags, obs_table="f32")
        arrs = b.arrays()
        arrs["pf_obs"] = None
        arrs["feat_obs_f32"], arrs["pf_obs_j_f32"] = b.obs_table(f32=True)
        d_in = {k: c.to_device(np.ascontiguousarray(v)) for k, v in arrs.items() if v is not None}
        d_out = {k: c.device_alloc(v.nbytes) for k, v in host.items()}
        c.linearize_raw(b.struct(d_in), abi.out_struct(d_out), flags | abi.PTRS_DEVICE)
        c.linearize(other, flags)
        c.sync()
        for k, v in host.items():
            back = np.empty_like(v)
            c.d2h(back, d_out[k])
            c.sync()
            if k.startswith(("pf_", "lf_")):
                assert np.array_equal(back, v), k
            else:
                assert pkg.parity.unit_err(k, back, v) < 1e-12, k
        for p in list(d_in.values()) + list(d_out.values()):
            c.device_free(p)
