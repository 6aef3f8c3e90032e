"""viml_slide_vi without a GPU: the ctypes mirror of viml_slide_out against sizeof / offsetof of the C struct, and the restatement of
tests/slide_policy.py — its re-anchored depth against an independent numpy computation of the same world point, the init_depth
fall-backs, and the next-frame structure the test chains build."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import marg_vi_policy as mp
import slide_policy as sp
from conftest import ROOT

PROGRAM = r"""
#include <cstddef>
#include <cstdio>
#include "viml.h"
#define F(m) std::printf("\"%s\": %zu,\n", #m, offsetof(viml_slide_out, m))
int main() {
  std::printf("{\n");
  F(poses); F(ex_pose); F(inv_depth); F(extra);
  std::printf("\"sizeof\": %zu\n}\n", sizeof(viml_slide_out));
}
"""


@pytest.fixture(scope="module")
def c_layout(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("slide_out_abi")
    cpp = tmp / "layout.cpp"
    cpp.write_text(PROGRAM)
    exe = tmp / "layout"
    subprocess.check_call(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(cpp)])
    return json.loads(subprocess.check_output([str(exe)]))


def test_slide_out_layout_matches_c(pkg, c_layout):
    cls = pkg._abi.SlideOut
    assert C.sizeof(cls) == c_layout["sizeof"]
    for name, _ in cls._fields_:
        assert getattr(cls, name).offset == c_layout[name], name
    assert sorted(f[0] for f in cls._fields_) == sorted(k for k in c_layout if k != "sizeof")
    assert "viml_slide_vi" in pkg.ABI_SYMBOLS


def _rot_np(p7):
    q = np.asarray(p7[3:7], dtype=np.float64)
    x, y, z, w = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def test_reanchored_depth_is_the_same_world_point(pkg):
    """The restatement's depth against numpy matrices: the world point from the old anchor's ray and depth, its z in the camera of
    the old pose 1."""
    batch = pkg.synth.make_windows(4, seed=3, F=40)
    pts = sp.pts_i_of(batch)
    n = 0
    for w in range(batch.W):
        p0, p1 = batch.pf_window_offset[w], batch.pf_window_offset[w + 1]
        ex = batch.ex_pose[w]
        Ric, tic = _rot_np(ex), ex[:3]
        c0, c1 = sp.camera(batch.poses[w, 0], ex), sp.camera(batch.poses[w, 1], ex)
        for f, k in sp.reanchored(batch.pf_idx[p0:p1]).items():
            got = sp.reanchor(batch.inv_depth[w, f], pts[p0 + k], c0, c1, 5.0)
            R0, R1 = _rot_np(batch.poses[w, 0]), _rot_np(batch.poses[w, 1])
            Xw = R0 @ (Ric @ (pts[p0 + k] / batch.inv_depth[w, f]) + tic) + batch.poses[w, 0, :3]
            zj = (Ric.T @ (R1.T @ (Xw - batch.poses[w, 1, :3]) - tic))[2]
            assert zj > 0
            assert abs(got - 1.0 / zj) <= 1e-12 * abs(1.0 / zj), (w, f)
            n += 1
    assert n >= 10


def _cams():
    ident = np.array([0, 0, 0, 0, 0, 0, 1.0])
    p1 = np.array([0, 0, 3.0, 0, 0, 0, 1.0])   # the new anchor 3 m ahead along the optical axis
    return sp.camera(ident, ident), sp.camera(p1, ident)


def test_behind_the_new_camera_gets_init_depth():
    c0, c1 = _cams()
    assert sp.reanchor(1 / 5.0, (0.0, 0.0, 1.0), c0, c1, 5.0) == 1 / 2.0      # 5 m ahead of c0: 2 m ahead of c1
    assert sp.reanchor(1 / 2.0, (0.0, 0.0, 1.0), c0, c1, 7.0) == 1 / 7.0      # 2 m ahead of c0: behind c1
    assert sp.reanchor(1 / 3.0, (0.0, 0.0, 1.0), c0, c1, 7.0) == 1 / 7.0      # on c1's plane: not > 0


def test_nan_depth_gets_init_depth():
    c0, c1 = _cams()
    assert sp.reanchor(np.nan, (0.1, 0.2, 1.0), c0, c1, 5.0) == 1 / 5.0


def test_slide_moves_the_state_and_only_re_anchored_depths():
    P, F = 5, 4
    rng = np.random.default_rng(0)
    poses = np.concatenate([rng.standard_normal((P, 3)), np.tile([0, 0, 0, 1.0], (P, 1))], axis=1)
    ex = np.array([0.1, 0, 0, 0, 0, 0, 1.0])
    dep = np.array([0.2, 0.25, 0.3, 0.5])
    extra = np.arange(9 * P + 3, dtype=float)
    # feature 0: two anchor-0 factors; 1: one; 2: anchored at 1; 3: none
    pf = np.array([0 | (1 << 8), 0 | (2 << 8), 0 | (1 << 8) | (1 << 16), 1 | (2 << 8) | (2 << 16), 1 | (3 << 8) | (2 << 16)])
    pts = np.tile([0.1, -0.1, 1.0], (len(pf), 1))
    po, eo, do, xo = sp.slide(poses, ex, dep, extra, mp.OLD, pf, pts)
    assert np.array_equal(po[:-1], poses[1:]) and np.array_equal(po[-1], poses[-1]) and np.array_equal(eo, ex)
    assert np.array_equal(xo[:9 * (P - 1)], extra[9:9 * P]) and np.array_equal(xo[9 * P:], extra[9 * P:])
    assert do[0] != dep[0] and np.array_equal(do[1:], dep[1:])
    po, eo, do, xo = sp.slide(poses, ex, dep, extra, mp.SECOND_NEW, pf, pts)
    assert np.array_equal(po[P - 2], poses[P - 1]) and np.array_equal(po[P - 1], poses[P - 1]) and np.array_equal(do, dep)
    assert np.array_equal(xo[9 * (P - 2):9 * (P - 1)], extra[9 * (P - 1):9 * P]) and np.array_equal(xo[9 * (P - 1):], extra[9 * (P - 1):])


def _pf(*ijf):
    return np.array([i | (j << 8) | (f << 16) for i, j, f in ijf], dtype=np.uint32)


def test_next_structure():
    P = 5
    idx = _pf((0, 1, 0), (0, 2, 0), (0, 3, 0), (0, 2, 1), (1, 2, 2), (1, 4, 2), (0, 2, 3), (0, 3, 3))
    obs = np.array([[0.1, 0.2, 1.0 + k, 2.0 + k] for k in range(len(idx))])
    i2, o2 = sp.next_structure(P, mp.OLD, idx, obs)
    # feature 0: pts_i from its observation in frame 1, the frame-1 factor dropped; 1 (one factor) and 3 (no frame-1 observation)
    # dropped; 2 shifted
    assert i2.tolist() == _pf((0, 1, 0), (0, 2, 0), (0, 1, 2), (0, 3, 2)).tolist()
    assert np.array_equal(o2[:2], [[1.0, 2.0, 2.0, 3.0], [1.0, 2.0, 3.0, 4.0]]) and np.array_equal(o2[2:], obs[4:6])
    i3, o3 = sp.next_structure(P, mp.SECOND_NEW, idx, obs)
    # the observations in frame P-2 = 3 dropped, those in frame P-1 = 4 moved to 3
    assert i3.tolist() == _pf((0, 1, 0), (0, 2, 0), (0, 2, 1), (1, 2, 2), (1, 3, 2), (0, 2, 3)).tolist()
    assert np.array_equal(o3, obs[[0, 1, 3, 4, 5, 6]])
