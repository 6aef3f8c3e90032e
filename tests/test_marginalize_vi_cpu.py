"""viml_marginalize_vi without a GPU: the ctypes mirror of viml_prior_out against sizeof / offsetof of the C struct (a small program
that includes include/viml.h, compiled with g++), and the selection, block order and slide of tests/marg_vi_policy.py on
hand-built windows."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import marg_vi_policy as mp
from conftest import ROOT

P = 5
D = 6 * (P + 1)
X = 9 * P

PROGRAM = r"""
#include <cstddef>
#include <cstdio>
#include "viml.h"
#define F(m) std::printf("\"%s\": %zu,\n", #m, offsetof(viml_prior_out, m))
int main() {
  std::printf("{\n");
  F(prior_n_max); F(prior_max_blocks); F(prior_n); F(prior_jacobian); F(prior_residual); F(prior_n_blocks); F(prior_block);
  F(prior_x0);
  std::printf("\"margin\": [%d, %d],\n\"sizeof\": %zu\n}\n", VIML_MARGIN_OLD, VIML_MARGIN_SECOND_NEW, sizeof(viml_prior_out));
}
"""


@pytest.fixture(scope="module")
def c_layout(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("prior_out_abi")
    cpp = tmp / "layout.cpp"
    cpp.write_text(PROGRAM)
    exe = tmp / "layout"
    subprocess.check_call(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(cpp)])
    return json.loads(subprocess.check_output([str(exe)]))


def test_prior_out_layout_matches_c(pkg, c_layout):
    cls = pkg._abi.PriorOut
    assert C.sizeof(cls) == c_layout["sizeof"]
    for name, _ in cls._fields_:
        assert getattr(cls, name).offset == c_layout[name], name
    assert sorted(f[0] for f in cls._fields_) == sorted(k for k in c_layout if k not in ("sizeof", "margin"))
    assert [pkg.MARGIN_OLD, pkg.MARGIN_SECOND_NEW] == c_layout["margin"] == [mp.OLD, mp.SECOND_NEW]
    assert "viml_marginalize_vi" in pkg.ABI_SYMBOLS


def _pf(*ijf):
    return np.array([i | (j << 8) | (f << 16) for i, j, f in ijf], dtype=np.int64)


IMU_POSE = np.array([(p, p + 1) for p in range(P - 1)])
IMU_PRE = np.full((P - 1, 17), 0.1)
PRIOR_NO_POSE0 = [(mp.POSE, p, 7, 6 * (p - 1)) for p in range(1, P)] + [(mp.EX, 0, 7, 6 * (P - 1)), (mp.EXTRA, 9, 9, 6 * P)]
PRIOR_POSE0 = [(mp.POSE, p, 7, 6 * p) for p in range(P)] + [(mp.EX, 0, 7, 6 * P), (mp.EXTRA, 0, 9, 6 * P + 6)]
POINTS = _pf((0, 1, 0), (0, 3, 0), (0, 2, 1), (1, 2, 2), (2, 4, 3))


def _cols(*blocks):
    return [c for kind, idx in blocks for c in (range(6 * idx, 6 * idx + 6) if kind == mp.POSE else range(6 * P, 6 * P + 6)
                                                 if kind == mp.EX else range(D + idx, D + idx + 9))]


def test_old_prior_without_pose0():
    r = mp.plan(P, X, mp.OLD, POINTS, IMU_POSE, IMU_PRE, PRIOR_NO_POSE0)
    assert not r["copy"] and r["prior"]
    assert r["points"].tolist() == [True, True, True, False, False]
    assert r["imu"].tolist() == [True, False, False, False]
    assert r["drop"] == list(range(6)) + list(range(D, D + 9))
    # poses 1..P-1 -> 0..P-2, the extrinsic, speed-bias 1 -> 0
    assert r["keep"] == [[mp.POSE, p - 1, 7, 6 * (p - 1)] for p in range(1, P)] + [[mp.EX, 0, 7, 6 * (P - 1)], [mp.EXTRA, 0, 9, 6 * P]]
    assert r["src"] == [(mp.POSE, p) for p in range(1, P)] + [(mp.EX, 0), (mp.EXTRA, 9)]
    assert r["cols"] == _cols(*[(mp.POSE, p) for p in range(1, P)], (mp.EX, 0), (mp.EXTRA, 9))


def test_old_prior_with_pose0_and_its_speed_bias():
    r = mp.plan(P, X, mp.OLD, POINTS[3:], IMU_POSE, IMU_PRE, PRIOR_POSE0)
    assert not r["points"].any()
    assert r["drop"] == list(range(6)) + list(range(D, D + 9))
    assert r["keep"][-2:] == [[mp.EX, 0, 7, 6 * (P - 1)], [mp.EXTRA, 0, 9, 6 * P]]
    assert [b[1] for b in r["keep"][:-2]] == list(range(P - 1))


def test_old_without_imu_and_anchor0_features():
    """The prior alone, without pose 0: nothing is marginalised (m = 0), every block slides."""
    r = mp.plan(P, X, mp.OLD, POINTS[3:], np.zeros((0, 2)), np.zeros((0, 17)), PRIOR_NO_POSE0)
    assert r["drop"] == [] and len(r["keep"]) == P + 1 and r["keep"][0] == [mp.POSE, 0, 7, 0]
    # no prior either: nothing at all
    r = mp.plan(P, X, mp.OLD, POINTS[3:], np.zeros((0, 2)), np.zeros((0, 17)), np.zeros((0, 4)))
    assert r["drop"] == [] and r["keep"] == [] and not r["prior"]


def test_old_points_and_long_imu_gap():
    """Without a prior: pose 0 and the observing poses and the extrinsic from the points; an IMU factor of sum_dt >= 10 takes no
    part (est.cpp:1916)."""
    pre = IMU_PRE.copy()
    pre[0, 0] = 10.0
    r = mp.plan(P, X, mp.OLD, POINTS, IMU_POSE, pre, np.zeros((0, 4)))
    assert not r["imu"].any()
    assert r["drop"] == list(range(6))
    assert r["keep"] == [[mp.POSE, 0, 7, 0], [mp.POSE, 1, 7, 6], [mp.POSE, 2, 7, 12], [mp.EX, 0, 7, 18]]


def test_second_new_with_pose_p_minus_2():
    blocks = [(mp.POSE, p, 7, 6 * p) for p in range(P)] + [(mp.EX, 0, 7, 6 * P), (mp.EXTRA, 9 * (P - 1), 9, 6 * P + 6)]
    r = mp.plan(P, X, mp.SECOND_NEW, POINTS, IMU_POSE, IMU_PRE, blocks)
    assert not r["copy"] and not r["points"].any() and not r["imu"].any()
    assert r["drop"] == list(range(6 * (P - 2), 6 * (P - 1)))
    assert r["keep"] == ([[mp.POSE, p, 7, 6 * p] for p in range(P - 2)] + [[mp.POSE, P - 2, 7, 6 * (P - 2)], [mp.EX, 0, 7, 6 * (P - 1)],
                         [mp.EXTRA, 9 * (P - 2), 9, 6 * P]])
    assert r["src"][P - 2] == (mp.POSE, P - 1) and r["src"][-1] == (mp.EXTRA, 9 * (P - 1))


def test_second_new_without_pose_p_minus_2_is_a_copy():
    blocks = [(mp.POSE, p, 7, 6 * p) for p in range(P - 2)] + [(mp.EX, 0, 7, 6 * (P - 2))]
    assert mp.plan(P, X, mp.SECOND_NEW, POINTS, IMU_POSE, IMU_PRE, blocks)["copy"]
    assert mp.plan(P, X, mp.SECOND_NEW, POINTS, IMU_POSE, IMU_PRE, np.zeros((0, 4)))["copy"]


def test_slide_state():
    poses = np.arange(P * 7, dtype=float).reshape(P, 7)
    extra = np.arange(X + 2, dtype=float)
    po, eo = mp.slide_state(poses, extra, mp.OLD)
    assert np.array_equal(po[:-1], poses[1:]) and np.array_equal(eo[:9 * (P - 1)], extra[9:9 * P]) and np.array_equal(eo[X:], extra[X:])
    pn, en = mp.slide_state(poses, extra, mp.SECOND_NEW)
    assert np.array_equal(pn[P - 2], poses[P - 1]) and np.array_equal(en[9 * (P - 2):9 * (P - 1)], extra[9 * (P - 1):9 * P])
    assert np.array_equal(pn[:P - 2], poses[:P - 2])
