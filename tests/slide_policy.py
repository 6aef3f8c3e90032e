"""What viml_slide_vi writes for one window (include/viml.h), restated on host arrays with Python floats: IEEE binary64, no fused
multiply-add, sums left to right, so it reproduces the kernel bit for bit.  The pose / speed-bias part is marg_vi_policy.slide_state.
Also the structure of the next frame's problem that the test chains need (next_structure)."""
import math

import numpy as np

import marg_vi_policy as mp


def rot(p7):
    """normalized(q).toRotationMatrix() of a [p, q] block, Eigen's order, as 3 rows of 3 floats."""
    qx, qy, qz, qw = (float(v) for v in p7[3:7])
    n = math.sqrt(qx * qx + qy * qy + qz * qz + qw * qw)
    w, x, y, z = qw / n, qx / n, qy / n, qz / n
    tx, ty, tz = 2.0 * x, 2.0 * y, 2.0 * z
    twx, twy, twz = tx * w, ty * w, tz * w
    txx, txy, txz = tx * x, ty * x, tz * x
    tyy, tyz, tzz = ty * y, tz * y, tz * z
    return [[1.0 - (tyy + tzz), txy - twz, txz + twy],
            [txy + twz, 1.0 - (txx + tzz), tyz - twx],
            [txz - twy, tyz + twx, 1.0 - (txx + tyy)]]


def _dot3(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def camera(pose, ex):
    """(R, P) of a pose's camera: R = R(q) R(q_ex), P = p + R(q) t_ex."""
    Rb, Re = rot(pose), rot(ex)
    t = [float(v) for v in ex[:3]]
    R = [[_dot3(Rb[r], [Re[0][c], Re[1][c], Re[2][c]]) for c in range(3)] for r in range(3)]
    P = [float(pose[r]) + _dot3(Rb[r], t) for r in range(3)]
    return R, P


def reanchor(inv, uv, cam0, cam1, init_depth):
    """removeBackShiftDepth for one feature: the inverse depth, in camera cam1, of the point at depth 1 / inv along uv = (x, y, z) of
    camera cam0; 1 / init_depth when that depth is not > 0 (NaN included)."""
    (R0, P0), (R1, P1) = cam0, cam1
    d = 1.0 / float(inv)
    a = [float(uv[0]) * d, float(uv[1]) * d, float(uv[2]) * d]
    v = [(_dot3(R0[r], a) + P0[r]) - P1[r] for r in range(3)]
    zj = R1[0][2] * v[0] + R1[1][2] * v[1] + R1[2][2] * v[2]
    return 1.0 / zj if zj > 0.0 else 1.0 / float(init_depth)


def reanchored(pf_idx):
    """{feature: index of its first factor} of the features with two or more factors with i == 0 (the ones MARGIN_OLD re-anchors)."""
    first, cnt = {}, {}
    for k, ix in enumerate(np.asarray(pf_idx, dtype=np.int64)):
        if ix & 0xff == 0:
            f = int(ix >> 16)
            cnt[f] = cnt.get(f, 0) + 1
            first.setdefault(f, k)
    return {f: k for f, k in first.items() if cnt[f] >= 2}


def slide(poses, ex_pose, inv_depth, extra, margin, pf_idx, pts_i, init_depth=5.0):
    """One window: (poses, ex_pose, inv_depth, extra) of the next frame.  pf_idx [NP] of the window's point factors, pts_i [NP, 3] their
    (x, y, z) of pts_i."""
    po, xo = mp.slide_state(poses, extra, margin)
    dep = inv_depth.copy()
    if margin == mp.OLD:
        c0, c1 = camera(poses[0], ex_pose), camera(poses[1], ex_pose)
        for f, k in reanchored(pf_idx).items():
            dep[f] = reanchor(inv_depth[f], pts_i[k], c0, c1, init_depth)
    return po, ex_pose.copy(), dep, xo


def pts_i_of(batch):
    """[NP, 3] pts_i of every point factor of a Batch (z = pf_pts_i_z or 1)."""
    z = np.ones(batch.NP) if batch.pf_pts_i_z is None else batch.pf_pts_i_z
    return np.column_stack([batch.pf_obs[:, 0], batch.pf_obs[:, 1], z])


def slide_batch(batch, extra, margin, init_depth=5.0):
    """slide() of every window of a Batch: dict(poses, ex_pose, inv_depth, extra) like Context.slide_vi."""
    res = {"poses": batch.poses.copy(), "ex_pose": batch.ex_pose.copy(), "inv_depth": batch.inv_depth.copy(), "extra": extra.copy()}
    pts = pts_i_of(batch)
    for w in range(batch.W):
        p0, p1 = batch.pf_window_offset[w], batch.pf_window_offset[w + 1]
        out = slide(batch.poses[w], batch.ex_pose[w], batch.inv_depth[w], extra[w], margin[w], batch.pf_idx[p0:p1], pts[p0:p1],
                    init_depth)
        for k, v in zip(("poses", "ex_pose", "inv_depth", "extra"), out):
            res[k][w] = v
    return res


def next_structure(P, margin, pf_idx, pf_obs):
    """The point factors of one window in the next frame, as FeatureManager leaves them after the slide (for test chains; the host
    keeps building the real factor lists).  MARGIN_OLD: a feature anchored at frame 0 is re-anchored at frame 1 — its factor with
    j == 1 becomes the anchor observation (pts_i), the others become (0, j - 1) with that pts_i; it is dropped when it had fewer than
    two factors or none with j == 1.  Every other factor moves to (i - 1, j - 1).  MARGIN_SECOND_NEW (removeFront): the observations
    in frame P-2 are dropped and those in frame P-1 move to P-2.  Returns (pf_idx [n] uint32, pf_obs [n, 4])."""
    pf_idx = np.asarray(pf_idx, dtype=np.int64)
    idx, obs = [], []
    anchor = {}
    if margin == mp.OLD:
        for k, ix in enumerate(pf_idx):
            if ix & 0xff == 0 and (ix >> 8) & 0xff == 1:
                anchor[int(ix >> 16)] = pf_obs[k, 2:4]
    keep = reanchored(pf_idx)
    for k, ix in enumerate(pf_idx):
        i, j, f = int(ix & 0xff), int((ix >> 8) & 0xff), int(ix >> 16)
        if margin == mp.OLD:
            if i == 0:
                if f not in keep or f not in anchor or j == 1:
                    continue
                idx.append(0 | ((j - 1) << 8) | (f << 16)), obs.append(np.concatenate([anchor[f], pf_obs[k, 2:4]]))
            else:
                idx.append((i - 1) | ((j - 1) << 8) | (f << 16)), obs.append(pf_obs[k])
        else:
            if j == P - 2:
                continue
            idx.append(i | ((P - 2 if j == P - 1 else j) << 8) | (f << 16)), obs.append(pf_obs[k])
    return np.array(idx, dtype=np.uint32), np.array(obs, dtype=np.float64).reshape(-1, 4)


def next_structure_batch(batch, margin):
    """next_structure() of every window of a Batch: (pf_window_offset [W+1], pf_idx, pf_obs)."""
    idx, obs, off = [], [], [0]
    for w in range(batch.W):
        p0, p1 = batch.pf_window_offset[w], batch.pf_window_offset[w + 1]
        i, o = next_structure(batch.P, margin[w], batch.pf_idx[p0:p1], batch.pf_obs[p0:p1])
        idx.append(i), obs.append(o), off.append(off[-1] + len(i))
    return np.array(off, dtype=np.int32), np.concatenate(idx).astype(np.uint32), np.concatenate(obs).reshape(-1, 4)
