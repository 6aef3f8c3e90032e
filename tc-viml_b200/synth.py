"""Deterministic synthetic workloads for the hot path (SURVEY.md §8d): EuRoC-shaped sliding windows,
a large prior line map with poses and LSD-style 2D segments.  numpy only; no product or oracle code.

Camera: EuRoC cam0 752x480, fx 461.6 fy 460.3 cx 363.0 cy 248.1; extrinsic and Rbw/Tbw are the values of
benchmark_publisher/config/V1_01_easy/sensor.yaml:9-10,29-32,40-73 (reference tree).
"""
import numpy as np

from ._abi import Batch, make_config

FX, FY, CX, CY, WIDTH, HEIGHT = 461.6, 460.3, 363.0, 248.1, 752, 480
RIC = np.array([[0.0148655429818, -0.999880929698, 0.00414029679422],
                [0.999557249008, 0.0149672133247, 0.025715529948],
                [-0.0257744366974, 0.00375618835797, 0.999660727178]])
TIC = np.array([-0.0216401454975, -0.064676986768, 0.00981073058949])
RBW = np.array([[0.958882, 0.283788, -0.00258614],
                [-0.283713, 0.958774, 0.016038],
                [0.00703105, -0.0146448, 0.999868]])
TBW = np.array([-1.4494, -1.83337, -0.899281])


def euroc_config(**kw):
    return make_config(Rbw=RBW, Tbw=TBW, **kw)


# ---- small rotation helpers (batched) ---------------------------------------------------------------
def rot_from_axis_angle(v):
    """Rodrigues; v [...,3] -> R [...,3,3]."""
    v = np.asarray(v, dtype=np.float64)
    th = np.linalg.norm(v, axis=-1)[..., None, None]
    k = v / np.maximum(np.linalg.norm(v, axis=-1, keepdims=True), 1e-300)
    K = np.zeros(v.shape[:-1] + (3, 3))
    K[..., 0, 1], K[..., 0, 2] = -k[..., 2], k[..., 1]
    K[..., 1, 0], K[..., 1, 2] = k[..., 2], -k[..., 0]
    K[..., 2, 0], K[..., 2, 1] = -k[..., 1], k[..., 0]
    eye = np.broadcast_to(np.eye(3), K.shape)
    return eye + np.sin(th) * K + (1 - np.cos(th)) * (K @ K)


def quat_from_rot(R):
    """R [...,3,3] -> q [...,4] as (x,y,z,w), w >= 0; robust branch on the largest diagonal term."""
    R = np.asarray(R, dtype=np.float64)
    m00, m11, m22 = R[..., 0, 0], R[..., 1, 1], R[..., 2, 2]
    tr = m00 + m11 + m22
    q = np.zeros(R.shape[:-2] + (4,))
    c0 = tr > 0
    c1 = (~c0) & (m00 >= m11) & (m00 >= m22)
    c2 = (~c0) & (~c1) & (m11 >= m22)
    c3 = (~c0) & (~c1) & (~c2)
    with np.errstate(invalid="ignore", divide="ignore"):
        s = np.sqrt(np.maximum(tr + 1.0, 0)) * 2
        q0 = np.stack([(R[..., 2, 1] - R[..., 1, 2]) / s, (R[..., 0, 2] - R[..., 2, 0]) / s,
                       (R[..., 1, 0] - R[..., 0, 1]) / s, 0.25 * s], -1)
        s = np.sqrt(np.maximum(1.0 + m00 - m11 - m22, 0)) * 2
        q1 = np.stack([0.25 * s, (R[..., 0, 1] + R[..., 1, 0]) / s, (R[..., 0, 2] + R[..., 2, 0]) / s,
                       (R[..., 2, 1] - R[..., 1, 2]) / s], -1)
        s = np.sqrt(np.maximum(1.0 + m11 - m00 - m22, 0)) * 2
        q2 = np.stack([(R[..., 0, 1] + R[..., 1, 0]) / s, 0.25 * s, (R[..., 1, 2] + R[..., 2, 1]) / s,
                       (R[..., 0, 2] - R[..., 2, 0]) / s], -1)
        s = np.sqrt(np.maximum(1.0 + m22 - m00 - m11, 0)) * 2
        q3 = np.stack([(R[..., 0, 2] + R[..., 2, 0]) / s, (R[..., 1, 2] + R[..., 2, 1]) / s, 0.25 * s,
                       (R[..., 1, 0] - R[..., 0, 1]) / s], -1)
    for c, qq in ((c0, q0), (c1, q1), (c2, q2), (c3, q3)):
        q[c] = qq[c]
    q *= np.where(q[..., 3:4] < 0, -1.0, 1.0)
    return q / np.linalg.norm(q, axis=-1, keepdims=True)


def pose7(p, R, rng=None, norm_jitter=1e-12):
    """[px,py,pz,qx,qy,qz,qw]; quaternion norm perturbed by ~1e-12 to exercise the un-normalised path
    of ProjectionFactor (projection_factor.cpp:25-31)."""
    q = quat_from_rot(R)
    if rng is not None and norm_jitter:
        q = q * (1.0 + norm_jitter * rng.standard_normal(q.shape[:-1] + (1,)))
    return np.concatenate([p, q], -1)


# ---- sliding windows (cfg 1, 2, 4, 5) ---------------------------------------------------------------
def make_windows(W, seed=0x5EED, P=11, F=150, lines_per_frame=10, start_max=None, min_len=2,
                 all_start_zero=False, noise_px=0.5, z_plane=False, max_len=None, f32_obs=False):
    """W independent EuRoC-shaped windows.

    P poses on a smooth random trajectory, F landmarks 2.5-8 m ahead of their start frame with
    start_frame ~ U{0..P-4}, track length ~ U{2..P-start} (=> ~3.7 factors per feature, ~560 per window
    at P=11, F=150), observations = exact projection + N(0,(noise_px/460)^2), inverse depth = truth *
    (1+N(0,0.05^2)); state = truth + small perturbation.  Line factors: `lines_per_frame` per pose,
    segments 2-8 m ahead, detected line = projection + N(0,1 px), float32-rounded pixel endpoints.
    all_start_zero=True gives the marginalisation stress shape (every landmark starts in frame 0).
    f32_obs=True rounds the point observations to float32, which is what the estimator receives (the tracker publishes
    geometry_msgs::Point32, feature_tracker_node.cpp:159-162; estimator_node.cpp:388-390 widens them).
    """
    rng = np.random.Generator(np.random.PCG64(seed))
    if start_max is None:
        start_max = max(P - 4, 0)  # start_frame < WINDOW_SIZE-2 (estimator.cpp:1740)
    # -- true trajectory (body in VIO world) --
    R0 = rot_from_axis_angle(rng.standard_normal((W, 3)) * 1.0)
    p0 = rng.uniform(-3, 3, (W, 3))
    Rwb = np.empty((W, P, 3, 3))
    pwb = np.empty((W, P, 3))
    Rwb[:, 0], pwb[:, 0] = R0, p0
    for k in range(1, P):
        ax = rng.standard_normal((W, 3))
        ax /= np.linalg.norm(ax, axis=-1, keepdims=True)
        dR = rot_from_axis_angle(ax * rng.uniform(0, np.deg2rad(3.0), (W, 1)))
        Rwb[:, k] = Rwb[:, k - 1] @ dR
        d = rng.standard_normal((W, 3))
        d /= np.linalg.norm(d, axis=-1, keepdims=True)
        pwb[:, k] = pwb[:, k - 1] + d * rng.uniform(0.03, 0.15, (W, 1))
    Rwc = Rwb @ RIC
    pwc = pwb + np.einsum("wpij,j->wpi", Rwb, TIC)
    # -- landmarks --
    if all_start_zero:
        start = np.zeros((W, F), dtype=np.int64)
    else:
        start = rng.integers(0, start_max + 1, (W, F))
    length = rng.integers(min_len, P - start + 1)  # frames observed incl. start
    if max_len is not None:
        length = np.minimum(length, max_len)
    u = rng.uniform(20, WIDTH - 20, (W, F))
    v = rng.uniform(20, HEIGHT - 20, (W, F))
    depth = rng.uniform(2.5, 8.0, (W, F))
    xc = np.stack([(u - CX) / FX * depth, (v - CY) / FY * depth, depth], -1)  # in start camera
    wi = np.arange(W)[:, None]
    Rs, ps = Rwc[wi, start], pwc[wi, start]
    Xw = np.einsum("wfij,wfj->wfi", Rs, xc) + ps
    # all projections [W,F,P,3]
    Xc_all = np.einsum("wpji,wfpj->wfpi", Rwc, Xw[:, :, None, :] - pwc[:, None, :, :])
    nz = noise_px / 460.0
    pts_all = Xc_all[..., :2] / Xc_all[..., 2:3] + nz * rng.standard_normal((W, F, P, 2))
    jj = np.arange(P)[None, None, :]
    mask = (jj > start[..., None]) & (jj < (start + length)[..., None]) & (Xc_all[..., 2] > 0.3)
    w_idx, f_idx, j_idx = np.nonzero(mask)  # window-major, then feature, then j (reference loop order)
    i_idx = start[w_idx, f_idx]
    pts_i = pts_all[w_idx, f_idx, i_idx]
    pts_j = pts_all[w_idx, f_idx, j_idx]
    pf_obs = np.concatenate([pts_i, pts_j], -1)
    if f32_obs:
        pf_obs = pf_obs.astype(np.float32).astype(np.float64)
    pf_idx = (i_idx | (j_idx << 8) | (f_idx << 16)).astype(np.uint32)
    counts = np.bincount(w_idx, minlength=W)
    pf_off = np.zeros(W + 1, dtype=np.int32)
    pf_off[1:] = np.cumsum(counts)
    inv_depth = (1.0 / depth) * (1.0 + 0.05 * rng.standard_normal((W, F)))
    # -- estimated state = truth + perturbation --
    Rest = Rwb @ rot_from_axis_angle(rng.standard_normal((W, P, 3)) * 0.003)
    pest = pwb + 0.01 * rng.standard_normal((W, P, 3))
    poses = pose7(pest, Rest, rng)
    ex = pose7(np.broadcast_to(TIC, (W, 3)) + 1e-3 * rng.standard_normal((W, 3)),
               RIC @ rot_from_axis_angle(rng.standard_normal((W, 3)) * 1e-3), rng)
    # -- line factors --
    NLf = lines_per_frame
    if NLf > 0:
        shape = (W, P, NLf)
        u0, v0 = rng.uniform(10, WIDTH - 10, shape), rng.uniform(10, HEIGHT - 10, shape)
        ang = rng.uniform(0, 2 * np.pi, shape)
        # axis-aligned bias like the EuRoC room maps (SURVEY.md §8d): snap 60 % to 0/90 deg
        snap = rng.uniform(size=shape) < 0.6
        ang = np.where(snap, np.round(ang / (np.pi / 2)) * (np.pi / 2) + 0.02 * rng.standard_normal(shape), ang)
        ln = rng.uniform(100, 300, shape)
        u1 = np.clip(u0 + ln * np.cos(ang), 5, WIDTH - 5)
        v1 = np.clip(v0 + ln * np.sin(ang), 5, HEIGHT - 5)
        d0, d1 = rng.uniform(2, 8, shape), rng.uniform(2, 8, shape)
        if z_plane:
            d1 = d0
        Pc0 = np.stack([(u0 - CX) / FX * d0, (v0 - CY) / FY * d0, d0], -1)
        Pc1 = np.stack([(u1 - CX) / FX * d1, (v1 - CY) / FY * d1, d1], -1)
        Pw0 = np.einsum("wpij,wpnj->wpni", Rwc, Pc0) + pwc[:, :, None, :]
        Pw1 = np.einsum("wpij,wpnj->wpni", Rwc, Pc1) + pwc[:, :, None, :]
        det = np.stack([u0, v0, u1, v1], -1) + rng.standard_normal(shape + (4,))
        det = det.astype(np.float32).astype(np.float64)  # float32 ROS channels (estimator_node.cpp:406-410)
        A = det[..., 3] - det[..., 1]                      # feature_manager.cpp:11-13
        B = det[..., 0] - det[..., 2]
        Cc = det[..., 2] * det[..., 1] - det[..., 0] * det[..., 3]
        lf_frame = np.broadcast_to(np.arange(P)[None, :, None], shape).reshape(-1).astype(np.int32)
        lf_geom = np.stack([Pw0[..., 0], Pw0[..., 1], Pw0[..., 2], Pw1[..., 0], Pw1[..., 1], Pw1[..., 2],
                            A, B, Cc], 0).reshape(9, -1)
        lf_off = (np.arange(W + 1) * (P * NLf)).astype(np.int32)
        lf_seg2d = det.reshape(-1, 4).astype(np.float32)
    else:
        lf_frame, lf_geom, lf_off, lf_seg2d = None, None, None, None
    return Batch(poses, ex, inv_depth, pf_off, pf_idx, pf_obs, lf_off, lf_frame, lf_geom, lf_seg2d=lf_seg2d)


def with_line_map(batch, cfg):
    """(batch2, line_map): the same batch with its line factors tied to a prior map, the way the estimator builds them
    (estimator.cpp:1831-1835: ptr = Rbw * lineWorld.Ptr + Tbw).  line_map [NL][6] holds one map line per factor in the MAP frame;
    batch2.lf_geom[0:6] is fl(Rbw p + Tbw) with the reference's operation order (row dot product left to right, then the
    translation; no fused multiply-add), batch2.lf_map_index = arange(NL).  The nine planes of batch2.lf_geom are then exactly what
    the line table (lf_map_index + lf_seg2d) expands to on the device."""
    R = np.array([cfg.Rbw[k] for k in range(9)]).reshape(3, 3)
    T = np.array([cfg.Tbw[k] for k in range(3)])
    Pw = batch.lf_geom[:6].T
    pm = np.concatenate([(Pw[:, :3] - T) @ R, (Pw[:, 3:] - T) @ R], 1)      # R^T (p - T): any map point near it will do

    def fwd(p):
        return ((R[:, 0] * p[:, 0:1] + R[:, 1] * p[:, 1:2]) + R[:, 2] * p[:, 2:3]) + T

    geom = batch.lf_geom.copy()
    geom[0:3], geom[3:6] = fwd(pm[:, :3]).T, fwd(pm[:, 3:]).T
    s = batch.lf_seg2d.astype(np.float64)
    abc = np.stack([s[:, 3] - s[:, 1], s[:, 0] - s[:, 2], s[:, 2] * s[:, 1] - s[:, 0] * s[:, 3]], 0)   # feature_manager.cpp:11-13
    assert np.array_equal(abc, geom[6:9]), "lf_seg2d does not reproduce the A, B, C planes"
    b2 = Batch(batch.poses, batch.ex_pose, batch.inv_depth, batch.pf_window_offset, batch.pf_idx, batch.pf_obs, batch.lf_window_offset,
               batch.lf_frame, geom, batch.pf_pts_i_z, batch.lf_seg2d, np.arange(batch.NL, dtype=np.int32))
    return b2, pm


# ---- prior line map + association queries (cfg 3) --------------------------------------------------
def make_line_map(n_lines, seed=0x5EED + 3, extent=(2000.0, 2000.0, 30.0)):
    """n_lines segments uniform in extent (metres), length 0.5-8 m, ~70 % axis aligned (dominant z),
    like the shipped room maps (SURVEY.md §8d fixture statistics).  Rows [sx sy sz ex ey ez]."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ext = np.asarray(extent)
    mid = rng.uniform(0, 1, (n_lines, 3)) * ext
    ln = rng.uniform(0.5, 8.0, (n_lines, 1))
    d = rng.standard_normal((n_lines, 3))
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    kind = rng.uniform(size=n_lines)
    axes = np.eye(3)
    d = np.where((kind < 0.46)[:, None], axes[2], d)
    d = np.where(((kind >= 0.46) & (kind < 0.60))[:, None], axes[1], d)
    d = np.where(((kind >= 0.60) & (kind < 0.70))[:, None], axes[0], d)
    s, e = mid - 0.5 * ln * d, mid + 0.5 * ln * d
    s[:, 2] = np.clip(s[:, 2], 0, ext[2])
    e[:, 2] = np.clip(e[:, 2], 0, ext[2])
    return np.ascontiguousarray(np.concatenate([s, e], -1))


def project_map(cfg_R, cfg_T, pose, ex, lines):
    """Plain numpy projection used only to synthesise 2D detections (not a parity path)."""
    q = pose[3:7] / np.linalg.norm(pose[3:7])
    qe = ex[3:7] / np.linalg.norm(ex[3:7])
    Rbi, Ric = _rot_from_quat(q), _rot_from_quat(qe)
    R = Ric.T @ Rbi.T @ cfg_R
    T = Ric.T @ (Rbi.T @ (cfg_T - pose[:3]) - ex[:3])
    ps = lines[:, :3] @ R.T + T
    pe = lines[:, 3:] @ R.T + T
    with np.errstate(divide="ignore", invalid="ignore"):
        uv = np.stack([FX * ps[:, 0] / ps[:, 2] + CX, FY * ps[:, 1] / ps[:, 2] + CY,
                       FX * pe[:, 0] / pe[:, 2] + CX, FY * pe[:, 1] / pe[:, 2] + CY], -1)
    front = (ps[:, 2] > 0) & (pe[:, 2] > 0)
    return uv, front


def _rot_from_quat(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


_QCTX = None


def _pose_queries(c, p):
    """The L 2D segments of pose p (own generator seeded by (seed, p): the result does not depend on how poses are
    distributed over worker processes)."""
    rng = np.random.Generator(np.random.PCG64([int(c["seed"]), int(p)]))
    lines, order, cstart, nxc, nyc, cell, reach, pm = (c[k] for k in ("lines", "order", "cstart", "nxc", "nyc", "cell", "reach", "pm"))
    L, n_true = c["L"], c["n_true"]
    cx0, cy0 = int(pm[p, 0] / cell), int(pm[p, 1] / cell)
    sel = []
    for yy in range(max(cy0 - reach, 0), min(cy0 + reach, nyc - 1) + 1):
        a = cstart[yy * nxc + max(cx0 - reach, 0)]
        b = cstart[yy * nxc + min(cx0 + reach, nxc - 1) + 1]
        sel.append(order[a:b])
    sel = np.concatenate(sel) if sel else np.zeros(0, dtype=np.int64)
    uv, front = project_map(c["Rbw"], c["Tbw"], c["cull"][p], c["ex"][p], lines[sel])
    inside = front & (uv[:, 0] > 1) & (uv[:, 0] < WIDTH - 2) & (uv[:, 1] > 1) & (uv[:, 1] < HEIGHT - 2) & \
        (uv[:, 2] > 1) & (uv[:, 2] < WIDTH - 2) & (uv[:, 3] > 1) & (uv[:, 3] < HEIGHT - 2)
    inside &= np.hypot(uv[:, 2] - uv[:, 0], uv[:, 3] - uv[:, 1]) > 15.0
    vis = np.nonzero(inside)[0]
    k = min(n_true, len(vis))
    out = np.empty((L, 4))
    if k:
        pick = rng.choice(vis, size=k, replace=False)
        seg = uv[pick]
        a0 = rng.uniform(0.0, 0.2, (k, 1))
        a1 = rng.uniform(0.8, 1.0, (k, 1))
        s0, e0 = seg[:, :2], seg[:, 2:]
        out[:k, :2] = s0 + a0 * (e0 - s0)
        out[:k, 2:] = s0 + a1 * (e0 - s0)
        out[:k] += rng.standard_normal((k, 4))
        flip = rng.uniform(size=k) < 0.5
        out[:k][flip] = out[:k][flip][:, [2, 3, 0, 1]]
    nclut = L - k
    u0, v0 = rng.uniform(0, WIDTH, nclut), rng.uniform(0, HEIGHT, nclut)
    ang, ln = rng.uniform(0, 2 * np.pi, nclut), rng.uniform(100, 400, nclut)
    out[k:, 0], out[k:, 1] = u0, v0
    out[k:, 2] = np.clip(u0 + ln * np.cos(ang), 0, WIDTH - 1)
    out[k:, 3] = np.clip(v0 + ln * np.sin(ang), 0, HEIGHT - 1)
    return out[rng.permutation(L)]


def _pose_range(args):
    lo, hi = args
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.stack([_pose_queries(_QCTX, p) for p in range(lo, hi)]) if hi > lo else np.empty((0, _QCTX["L"], 4))


def _queries_for_poses(c, lo, hi):
    """Serial for small query sets; large ones (the cfg-3 bench, 4096 poses) are spread over forked worker processes."""
    global _QCTX
    _QCTX = c
    n = hi - lo
    if n < 512:
        return _pose_range((lo, hi))
    import multiprocessing as mp
    import os
    nw = max(1, min(32, (os.cpu_count() or 1)))
    cuts = [lo + (n * k) // (4 * nw) for k in range(4 * nw + 1)]
    try:
        with mp.get_context("fork").Pool(nw) as pool:
            parts = pool.map(_pose_range, list(zip(cuts[:-1], cuts[1:])))
    except Exception:
        parts = [_pose_range((lo, hi))]
    return np.concatenate(parts, 0)



def make_assoc_queries(lines, n_poses, L=300, n_true=100, seed=0x5EED + 33, altitude=(45.0, 60.0),
                       extent=(2000.0, 2000.0, 30.0), Rbw=RBW, Tbw=TBW, pose_drift=True):
    """n_poses down-looking camera poses on a trajectory over the map, each with L 2D segments:
    n_true = projections of visible map lines + N(0,1 px) endpoint noise and random shortening, the
    rest clutter 100-400 px long (LSD/FLD style), rounded to float32.  Returns (cull_poses, match_poses,
    ex_pose, lines2d) in the viml_assoc_query layout.  The camera looks down (tilt <= 15 deg) so the FoV
    list stays at 10^2-10^3 of the map (there is no occlusion test in UpdateLinesInFoV)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ext = np.asarray(extent)
    # trajectory in the MAP frame: smooth loop
    t = np.linspace(0, 2 * np.pi, n_poses, endpoint=False)
    cxm, cym = ext[0] / 2, ext[1] / 2
    rad = 0.35 * min(ext[0], ext[1])
    pm = np.stack([cxm + rad * np.cos(t) * (1 + 0.2 * np.sin(5 * t)), cym + rad * np.sin(t) * (1 + 0.2 * np.cos(3 * t)),
                   ext[2] + rng.uniform(altitude[0] - ext[2], altitude[1] - ext[2], n_poses)], -1)
    # camera looks along -z of the map (x right, y "down" in image = -map y), small random tilt + yaw
    Rdown = np.array([[1.0, 0, 0], [0, -1.0, 0], [0, 0, -1.0]])
    yaw = rng.uniform(0, 2 * np.pi, n_poses)
    Rz = rot_from_axis_angle(np.stack([np.zeros(n_poses), np.zeros(n_poses), yaw], -1))
    tilt = rot_from_axis_angle(rng.standard_normal((n_poses, 3)) * np.deg2rad(5.0))
    Rmc = Rz @ Rdown @ tilt                      # map <- camera
    # body pose in VIO world: R_vio_c = Rbw Rmc ; body = camera * ric^-1
    Rvc = Rbw @ Rmc
    pvc = pm @ Rbw.T + Tbw
    Rvb = Rvc @ RIC.T
    pvb = pvc - np.einsum("pij,j->pi", Rvb, TIC)
    cull = pose7(pvb, Rvb, rng)
    if pose_drift:  # the match pose is the re-optimised one (estimator.cpp:679-692): small drift
        Rm = Rvb @ rot_from_axis_angle(rng.standard_normal((n_poses, 3)) * 0.002)
        match = pose7(pvb + 0.02 * rng.standard_normal((n_poses, 3)), Rm, rng)
    else:
        match = cull.copy()
    ex = pose7(np.broadcast_to(TIC, (n_poses, 3)).copy(), np.broadcast_to(RIC, (n_poses, 3, 3)).copy(), rng)
    # grid index of line midpoints (map frame) to find visible lines quickly
    cell = 25.0
    mid = 0.5 * (lines[:, :3] + lines[:, 3:])
    gx = np.clip((mid[:, 0] / cell).astype(np.int64), 0, None)
    gy = np.clip((mid[:, 1] / cell).astype(np.int64), 0, None)
    nxc = int(gx.max()) + 1 if len(lines) else 1
    nyc = int(gy.max()) + 1 if len(lines) else 1
    cid = gy * nxc + gx
    order = np.argsort(cid, kind="stable")
    cstart = np.searchsorted(cid[order], np.arange(nxc * nyc + 1))
    reach = int(np.ceil(altitude[1] * np.tan(np.deg2rad(62.0)) / cell)) + 1
    ctxd = dict(lines=lines, order=order, cstart=cstart, nxc=nxc, nyc=nyc, cell=cell, reach=reach, pm=pm, cull=cull, ex=ex,
                Rbw=Rbw, Tbw=Tbw, L=L, n_true=n_true, seed=seed)
    lines2d = _queries_for_poses(ctxd, 0, n_poses)
    lines2d = lines2d.astype(np.float32).astype(np.float64)
    return (np.ascontiguousarray(cull), np.ascontiguousarray(match), np.ascontiguousarray(ex),
            np.ascontiguousarray(lines2d))


# ---- dense-block factors of a window (prior + IMU), SURVEY 8f rank 2 ---------------------------------------------
def make_dense_factors(batch, seed=5):
    """Per window the dense-block factors the reference's problem carries beside the visual ones (estimator.cpp:1717-1733): the
    prior of the last marginalisation — n rows over the kept blocks [pose 1 .. P-1, extrinsic, speed-bias 1], n = their tangent size
    + 1 <= 76 (marginalization_factor.cpp:335-384) — and one IMU block per consecutive pose pair (15 rows over pose i, speed-bias i,
    pose j, speed-bias j: 15 x 30, imu_factor.h:19-181).  Values are synthetic (a strong diagonal keeps the reduced system well
    conditioned: the visual factors alone leave the gauge free).  Extra columns: 9 per pose (speed-bias).  Returns a _abi.Dense."""
    from ._abi import Dense
    rng = np.random.default_rng(seed)
    W, P, D = batch.W, batch.P, batch.D
    X = 9 * P
    fs = []
    for w in range(W):
        cols = np.concatenate([np.arange(6, D), D + 9 + np.arange(9)]) if P > 1 else np.arange(D)
        n = len(cols) + 1
        J = 20.0 * rng.standard_normal((n, len(cols)))
        J[:len(cols)] += np.diag(250.0 + 50.0 * rng.uniform(size=len(cols)))
        fs.append((w, 0.05 * rng.standard_normal(n), J, cols))
        for i in range(P - 1):
            ci = np.concatenate([6 * i + np.arange(6), D + 9 * i + np.arange(9), 6 * (i + 1) + np.arange(6), D + 9 * (i + 1) + np.arange(9)])
            J = 10.0 * rng.standard_normal((15, 30))
            J[:, :15] += np.diag(120.0 + 30.0 * rng.uniform(size=15))
            J[:, 15:] -= np.diag(120.0 + 30.0 * rng.uniform(size=15))
            fs.append((w, 0.1 * rng.standard_normal(15), J, ci))
        # the first pose and speed-bias are tied down by the gauge prior a real window carries through its history
        c0 = np.concatenate([np.arange(6), D + np.arange(9)])
        fs.append((w, 0.01 * rng.standard_normal(15), np.diag(200.0 + 50.0 * rng.uniform(size=15)), c0))
    return Dense(W, X, fs)


# ---- IMU factors and the prior of a window, as inputs of viml_inertial_evaluate / viml_gn_step_vi ------------------------------
def _qmul(a, b):
    """Hamilton product of [..., (x, y, z, w)] quaternions."""
    ax, ay, az, aw = np.moveaxis(a, -1, 0)
    bx, by, bz, bw = np.moveaxis(b, -1, 0)
    return np.stack([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz], -1)


def _qconj(q):
    return np.concatenate([-q[..., :3], q[..., 3:]], -1) / (q * q).sum(-1, keepdims=True)


def _rot(q):
    """toRotationMatrix of an (x, y, z, w) quaternion (no normalisation)."""
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def make_inertial_factors(batch, seed=11, realistic=False, no_imu=(), no_prior=(), extra_pad=0, n_max=None, noise=1e-3):
    """(Inertial, extra_state [W, X]) for a window batch: one IMU factor per consecutive pose pair and one prior per window, the way
    Estimator::optimization adds them (estimator.cpp:1717-1733).

    The extra state holds a speed-bias block [V, Ba, Bg] per pose (offset 9 p), plus `extra_pad` values no factor touches.  The
    pre-integrated deltas are formed from the batch's poses with the chosen velocities and biases (so the residuals are small),
    plus `noise`; linearized_ba / linearized_bg differ from the state's biases so the bias corrections are exercised; the
    pre-integration Jacobian takes its first-order closed forms (dp_dba = -R dt^2 / 2, dq_dbg = -dt I, dv_dba = -R dt, ...) plus
    jitter; sqrt_info = LLT(covariance^-1).matrixL()^T of an SPD covariance.  By default the covariance is scaled like
    make_dense_factors (entries of sqrt_info of order 10^2: the reduced system stays well conditioned); realistic=True takes the
    EuRoC noise densities (acc_n 0.08, gyr_n 0.004, acc_w 4e-5, gyr_w 2e-6: bias rows of the covariance near 1e-11).
    The prior covers [pose 1 .. P-1, extrinsic, speed-bias 1] (n = 6 P + 9, 75 at P = 11) with x0 near the state; windows in
    no_imu / no_prior carry none.  n_max (default n) is the prior stride."""
    from ._abi import BLOCK_EX, BLOCK_EXTRA, BLOCK_POSE, PRIOR_X0_STRIDE, Inertial
    rng = np.random.default_rng(seed)
    W, P = batch.W, batch.P
    X = 9 * P + extra_pad
    G = np.array([0.0, 0.0, 9.81])
    extra = np.zeros((W, X))
    sb = extra[:, :9 * P].reshape(W, P, 9)
    sb[..., 0:3] = 0.5 * rng.standard_normal((W, P, 3))
    sb[..., 3:6] = 0.05 * rng.standard_normal((W, P, 3))
    sb[..., 6:9] = 0.005 * rng.standard_normal((W, P, 3))
    if extra_pad:
        extra[:, 9 * P:] = rng.standard_normal((W, extra_pad))
    pose_list, sb_list, pre, jac, info, off = [], [], [], [], [], [0]
    for w in range(W):
        pairs = [] if w in no_imu else [(p, p + 1) for p in range(P - 1)]
        for (i, j) in pairs:
            dt = rng.uniform(0.05, 0.15)
            xi, xj = batch.poses[w, i], batch.poses[w, j]
            qi, qj = xi[3:7], xj[3:7]
            Ri = _rot(qi)
            RiT = np.linalg.inv(Ri)
            Vi, Bai, Bgi = sb[w, i, 0:3], sb[w, i, 3:6], sb[w, i, 6:9]
            Vj = sb[w, j, 0:3]
            J = np.eye(15) + 0.01 * rng.standard_normal((15, 15))
            J[0:3, 9:12] = -0.5 * RiT * dt * dt + 1e-4 * rng.standard_normal((3, 3))
            J[0:3, 12:15] = 0.01 * dt * rng.standard_normal((3, 3))
            J[3:6, 12:15] = -dt * np.eye(3) + 1e-3 * rng.standard_normal((3, 3))
            J[6:9, 9:12] = -RiT * dt + 1e-3 * rng.standard_normal((3, 3))
            J[6:9, 12:15] = 0.01 * dt * rng.standard_normal((3, 3))
            lin_ba = Bai + 0.02 * rng.standard_normal(3)
            lin_bg = Bgi + 0.002 * rng.standard_normal(3)
            dba, dbg = Bai - lin_ba, Bgi - lin_bg
            dp = RiT @ (0.5 * G * dt * dt + xj[:3] - xi[:3] - Vi * dt) - J[0:3, 9:12] @ dba - J[0:3, 12:15] @ dbg
            dv = RiT @ (G * dt + Vj - Vi) - J[6:9, 9:12] @ dba - J[6:9, 12:15] @ dbg
            corr = np.concatenate([0.5 * (J[3:6, 12:15] @ dbg), [1.0]])
            qij = _qmul(_qconj(qi), qj)
            dq = _qmul(qij, _qconj(corr))
            dq = _qmul(dq, np.concatenate([0.5 * noise * rng.standard_normal(3), [1.0]]))
            dq /= np.linalg.norm(dq)
            dp = dp + noise * rng.standard_normal(3)
            dv = dv + noise * rng.standard_normal(3)
            pre.append(np.concatenate([[dt], dp, dq, dv, lin_ba, lin_bg]))
            jac.append(J)
            if realistic:
                acc_n, gyr_n, acc_w, gyr_w = 0.08, 0.004, 4e-5, 2e-6
                sig2 = np.concatenate([np.full(3, acc_n ** 2 * dt ** 3), np.full(3, gyr_n ** 2 * dt), np.full(3, acc_n ** 2 * dt),
                                       np.full(3, acc_w ** 2 * dt), np.full(3, gyr_w ** 2 * dt)])
            else:
                sig2 = (0.01 * (1.0 + rng.uniform(size=15))) ** 2
            A = rng.standard_normal((15, 15)) * 0.1
            C = np.sqrt(sig2)[:, None] * (np.eye(15) + 0.1 * (A + A.T)) * np.sqrt(sig2)[None, :]
            C = 0.5 * (C + C.T) + np.diag(sig2) * 0.05
            L = np.linalg.cholesky(np.linalg.inv(C))
            info.append(L.T)
            pose_list.append((i, j))
            sb_list.append((9 * i, 9 * j))
        off.append(len(pre))
    n = 6 * (P - 1) + 6 + 9
    nm = n if n_max is None else int(n_max)
    blocks = [(BLOCK_POSE, p, 7, 6 * (p - 1)) for p in range(1, P)] + [(BLOCK_EX, 0, 7, 6 * (P - 1)), (BLOCK_EXTRA, 9, 9, 6 * P)]
    mb = len(blocks)
    prior_n = np.array([0 if w in no_prior else n for w in range(W)], dtype=np.int32)
    pj, pr = np.zeros((W, nm, nm)), np.zeros((W, nm))
    pblk, px0 = np.zeros((W, mb, 4), dtype=np.int32), np.zeros((W, mb, PRIOR_X0_STRIDE))
    for w in range(W):
        J = 20.0 * rng.standard_normal((n, n)) + np.diag(250.0 + 50.0 * rng.uniform(size=n))
        pj[w, :n, :n] = J
        pr[w, :n] = 0.05 * rng.standard_normal(n)
        pblk[w] = np.array(blocks, dtype=np.int32)
        for b, (kind, idx, size, first) in enumerate(blocks):
            x = batch.poses[w, idx] if kind == BLOCK_POSE else batch.ex_pose[w] if kind == BLOCK_EX else extra[w, idx:idx + size]
            x0 = np.array(x, dtype=np.float64).copy()
            if size == 7:
                x0[:3] += 0.01 * rng.standard_normal(3)
                x0[3:7] = _qmul(x0[3:7], np.concatenate([0.005 * rng.standard_normal(3), [1.0]]))
                x0[3:7] /= np.linalg.norm(x0[3:7])
            else:
                x0 = x0 + 0.01 * rng.standard_normal(size)
            px0[w, b, :size] = x0
    NI = len(pre)
    vi = Inertial(W, P, X, G, np.array(off, dtype=np.int32), np.array(pose_list, dtype=np.int32).reshape(NI, 2),
                  np.array(sb_list, dtype=np.int32).reshape(NI, 2), np.array(pre).reshape(NI, 17), np.array(jac).reshape(NI, 15, 15),
                  np.array(info).reshape(NI, 15, 15), prior_n, pj, pr, np.full(W, mb, dtype=np.int32), pblk, px0)
    return vi, extra
