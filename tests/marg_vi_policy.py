"""Which factors and blocks of a window viml_marginalize_vi marginalises, in what order it keeps the rest and how it slides them
(include/viml.h), restated for one window on host arrays."""
import numpy as np

POSE, EX, EXTRA = 0, 1, 2
OLD, SECOND_NEW = 0, 1


def plan(P, X, margin, pf_idx, imu_pose, imu_preint, prior_block):
    """One window.  pf_idx [NP] packed i | j << 8 | feat << 16, imu_pose [NI, 2], imu_preint [NI, 17] (column 0, sum_dt, is read),
    prior_block [nb, 4] rows {kind, index, size, first} (nb = 0: no prior).  Returns a dict:
      copy     True: MARGIN_SECOND_NEW without pose P-2 in the prior, the output is the input prior
      points   bool mask of the point factors that take part, imu: the same for the IMU factors, prior: whether the prior does
      drop     tangent columns of the marginalised blocks (pose 0 then speed-bias 0, or pose P-2), in A's order
      keep     output blocks [kind, index after the slide, size, first column] in output order
      src      per output block the (kind, index) of the state block whose value is its x0
      cols     tangent columns of the kept blocks, in output order (A = [drop | cols])"""
    D = 6 * (P + 1)
    old = margin == OLD
    pf_idx = np.asarray(pf_idx, dtype=np.int64)
    blocks = [tuple(int(t) for t in b) for b in np.asarray(prior_block).reshape(-1, 4)]
    slot = lambda kind, idx: idx if kind == POSE else P if kind == EX else P + 1 + idx // 9
    has = any(k == POSE and i == P - 2 for k, i, _, _ in blocks)
    res = {"copy": not old and not has, "points": np.zeros(len(pf_idx), bool), "imu": np.zeros(len(imu_pose), bool),
           "prior": len(blocks) > 0 and (old or has), "drop": [], "keep": [], "src": [], "cols": []}
    if res["copy"]:
        return res
    touch = set(slot(k, i) for k, i, _, _ in blocks)
    if old:
        res["points"] = (pf_idx & 0xff) == 0
        for ix in pf_idx[res["points"]]:
            touch |= {0, int((ix >> 8) & 0xff), P}
        for k, (i, j) in enumerate(np.asarray(imu_pose).reshape(-1, 2)):
            if i == 0 and imu_preint[k][0] < 10.0:
                res["imu"][k] = True
                touch |= {int(i), int(j), P + 1 + int(i), P + 1 + int(j)}
    dp, ds = (0, P + 1) if old else (P - 2, None)
    if dp in touch:
        res["drop"] += list(range(6 * dp, 6 * dp + 6))
    if ds is not None and ds in touch:
        res["drop"] += list(range(D, D + 9))
    first = 0
    for s in sorted(touch - {dp, ds}):
        q = s if s < P else s - P - 1
        slid = q - 1 if old else (P - 2 if q == P - 1 else q)
        if s < P:
            res["keep"].append([POSE, slid, 7, first]), res["src"].append((POSE, s)), res["cols"].extend(range(6 * s, 6 * s + 6))
        elif s == P:
            res["keep"].append([EX, 0, 7, first]), res["src"].append((EX, 0)), res["cols"].extend(range(6 * P, 6 * P + 6))
        else:
            res["keep"].append([EXTRA, 9 * slid, 9, first]), res["src"].append((EXTRA, 9 * q))
            res["cols"].extend(range(D + 9 * q, D + 9 * q + 9))
        first += 6 if s <= P else 9
    return res


def x0_rows(P, src, pose, ex_pose, extra):
    """prior_x0 rows [len(src), 9] of one window: the kept blocks' values at the state, zeros past a block's size."""
    rows = np.zeros((len(src), 9))
    for b, (kind, idx) in enumerate(src):
        rows[b, :7 if kind != EXTRA else 9] = pose[idx] if kind == POSE else ex_pose if kind == EX else extra[idx:idx + 9]
    return rows


def slide_state(poses, extra, margin):
    """The caller's slide of one window's state after the marginalisation (Estimator::slideWindow): MARGIN_OLD moves pose p and
    speed-bias p to slot p - 1 (the last slot keeps its value), MARGIN_SECOND_NEW moves pose / speed-bias P-1 to P-2."""
    poses, extra = poses.copy(), extra.copy()
    P = poses.shape[0]
    sb = extra[:9 * P].reshape(P, 9)
    if margin == OLD:
        poses[:-1], sb[:-1] = poses[1:].copy(), sb[1:].copy()
    else:
        poses[P - 2], sb[P - 2] = poses[P - 1], sb[P - 1].copy()
    return poses, extra
