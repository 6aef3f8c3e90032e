"""Chunked staging of the host-pointer calls that split into independent units.

A host viml_line_associate runs in chunks of poses, a host viml_linearize_batch of 512 windows or more in chunks of windows (four
chunks from 512 units on).  Every chunk's slice of the outputs must equal what the same units give when sent alone: bit for bit,
except the visual H/b blocks, which are summed through atomics (1e-12 per block).  Entries the kernels leave alone keep the caller's
content, and a bad index in a late chunk is refused without launching it."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EXT = (300.0, 300.0, 30.0)


@pytest.mark.parametrize("cached", [False, True], ids=["culled", "cached"])
def test_association_chunks_match_separate_calls(pkg, cfg, cached):
    """600 poses (four chunks) equal the same poses sent as two 300-pose calls (one chunk each)."""
    abi, synth = pkg._abi, pkg.synth
    Pq, L = 600, 64
    lines = synth.make_line_map(20_000, extent=EXT)
    cull, match, ex, l2d = synth.make_assoc_queries(lines, Pq, L=L, n_true=24, extent=EXT)
    n_lines = np.random.default_rng(411).integers(0, L + 1, Pq).astype(np.int32)   # ragged queries
    with pkg.Context(cfg) as c:
        c.set_map(lines)
        slot = None
        if cached:
            for s in range(abi.FOV_SLOTS):
                c.fov_update(s, cull[s], ex[s])
            slot = np.arange(Pq, dtype=np.int32) % abi.FOV_SLOTS
        cull_q = None if cached else cull

        def assoc(lo, hi, cap):
            return c.associate(None if cull_q is None else cull_q[lo:hi], match[lo:hi], ex[lo:hi], l2d[lo:hi], n_lines2d=n_lines[lo:hi],
                               fov_capacity=cap, want_mask=True, cached=cached, fov_slot=None if slot is None else slot[lo:hi])

        cap = int(np.median(assoc(0, Pq, 0)["fov_count"]))   # some lists shorter than the capacity, some cut
        whole, halves = assoc(0, Pq, cap), [assoc(0, 300, cap), assoc(300, Pq, cap)]
    for k, v in whole.items():
        assert np.array_equal(v, np.concatenate([h[k] for h in halves]), equal_nan=True), k
    # the helper pre-fills match_index with -2, err and projected with NaN, fov_index with -1: past each count they must survive
    past = np.arange(L)[None, :] >= n_lines[:, None]
    assert past.any() and (whole["match_index"][past] == -2).all()
    assert np.isnan(whole["err"][past]).all() and np.isnan(whole["projected"][past]).all()
    assert (whole["match_index"][~past] >= -1).all()
    short = np.arange(cap)[None, :] >= whole["fov_count"][:, None]
    assert short.any() and (whole["fov_index"][short] == -1).all()
    assert cap > 0 and (whole["fov_count"] > cap).any()


@pytest.mark.parametrize("obs_table,line_table", [(False, False), (False, True), ("f32", False), ("f32", True)],
                         ids=["pairs-planes", "pairs-line_table", "f32_table-planes", "f32_table-line_table"])
def test_linearize_chunks_match_separate_calls(pkg, cfg, obs_table, line_table):
    """Windows 0-11 (first chunk) and 588-599 (last chunk) of a 600-window batch equal the same windows sent alone, with
    pf_pts_i_z given."""
    abi, synth = pkg._abi, pkg.synth
    b, lmap = synth.with_line_map(synth.make_windows(600, seed=421, f32_obs=True), cfg)
    b.pf_pts_i_z = 1.0 + 0.01 * np.random.default_rng(423).standard_normal(b.NP)
    flags = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    with pkg.Context(cfg) as c:
        c.set_map(lmap)
        big = c.linearize(b, flags, obs_table=obs_table, line_table=line_table)
        for lo, hi in ((0, 12), (588, 600)):
            small = c.linearize(b.slice_windows(lo, hi), flags, obs_table=obs_table, line_table=line_table)
            rows = {"pf_": slice(int(b.pf_window_offset[lo]), int(b.pf_window_offset[hi])),
                    "lf_": slice(int(b.lf_window_offset[lo]), int(b.lf_window_offset[hi]))}
            for k, v in small.items():
                assert not np.isnan(v).any(), k
                if k.startswith(("pf_", "lf_")):
                    assert np.array_equal(big[k][rows[k[:3]]], v), (k, lo)
                else:
                    assert pkg.parity.unit_err(k, big[k][lo:hi], v) < 1e-12, (k, lo)


def test_bad_index_in_a_late_chunk(pkg, cfg):
    """A feature index out of range in window 500 (the fourth chunk of 600 windows) is refused with viml_linearize_batch's code and
    message, and the context computes the next valid call correctly."""
    abi, synth = pkg._abi, pkg.synth
    b = synth.make_windows(600, seed=431)
    flags = abi.OUT_RESIDUAL_JACOBIAN | abi.OUT_HB | abi.OUT_SCHUR | abi.LOSS_CAUCHY
    bad = synth.make_windows(600, seed=431)
    k = int(bad.pf_window_offset[500])
    bad.pf_idx[k] = (bad.pf_idx[k] & 0xffff) | (bad.F << 16)
    with pkg.Context(cfg) as c:
        ref = c.linearize(b, flags)
        with pytest.raises(pkg.VimlError) as chunked:
            c.linearize(bad, flags)
        with pytest.raises(pkg.VimlError) as alone:
            c.linearize(bad.slice_windows(498, 502), flags)   # one copy: checked before any copy
        assert str(chunked.value) == str(alone.value)
        assert str(chunked.value).startswith(f"viml error {abi.VIML_ERR_INVALID}: factor index out of range")
        got = c.linearize(b, flags)
    for k, v in ref.items():
        if k.startswith(("pf_", "lf_")):
            assert np.array_equal(got[k], v), k
        else:
            assert pkg.parity.unit_err(k, got[k], v) < 1e-12, k
