"""TEST INFRASTRUCTURE -- statement of record for okp_triangulate_stereo_objects_depth_f64 (stereo objects with depth
association).

stereo_oracle.stereo_objects with one change: candidates are scored by where each view's lift (kp_point, in its own
camera's frame) lands in the other view. It composes the same np_oracle pieces: undistort_point, associate (its cost as
the epipolar gate, its greedy rule on the depth cost) and triangulate_stereo. The depth cost is computed in the kernel's
operation order (scalar float64, no fused multiply-add: the library builds with -fmad=false), so match tables compare
bitwise. Only tests/ import it.
"""
import numpy as np

from oracle import np_oracle
from oracle.stereo_oracle import STEREO_AMBIGUOUS, STEREO_BAD_PAIR

STEREO_NO_DEPTH = 4         # a candidate within max_distance_px had no valid lift in either view


def _greedy(cost, max_cost):
    """np_oracle.associate's greedy one-to-one step on a given cost matrix [nL, nR] -> (match [nL], cost [nL])."""
    nl, nr = cost.shape
    match = np.full(nl, -1, np.int32)
    match_cost = np.zeros(nl)
    free = np.ones((nl, nr), bool)
    for _ in range(min(nl, nr)):
        masked = np.where(free & ~np.isnan(cost), cost, np.inf)        # NaN: not admissible, as in associate
        e = int(np.argmin(masked))                 # first minimum in (left, right) raster order
        i, j = divmod(e, nr)
        if not (masked[i, j] <= max_cost):
            break
        match[i] = j
        match_cost[i] = masked[i, j]
        free[i, :] = False
        free[:, j] = False
    return match, match_cost


def _rigid(T):
    """(R, t) of a 4x4 rigid motion and (R^T, -R^T t) of its inverse, as okp_triangulate_stereo_objects_depth_f64 forms
    them on the host."""
    T = np.asarray(T, dtype=np.float64)
    R, t = T[:3, :3], T[:3, 3]
    t_inv = np.array([-(R[0, r] * t[0] + R[1, r] * t[1] + R[2, r] * t[2]) for r in range(3)])
    return (R, t), (R.T.copy(), t_inv)


def project_lift(X, R, t, cam):
    """q = pi(K (R X + t)) in the undistorted pixels of cam (fx, fy, cx, cy); NaN unless X is finite with z > 0."""
    x, y, z = (np.float64(v) for v in X)
    if not (np.isfinite(x) and np.isfinite(y) and np.isfinite(z) and z > 0.0):
        return np.array([np.nan, np.nan])
    Y = [R[r, 0] * x + R[r, 1] * y + R[r, 2] * z + t[r] for r in range(3)]
    with np.errstate(all='ignore'):
        return np.array([(cam['fx'] * Y[0] + cam['cx'] * Y[2]) / Y[2], (cam['fy'] * Y[1] + cam['cy'] * Y[2]) / Y[2]])


def depth_costs(F, uL, qR, uR, qL, max_distance_px):
    """Depth association costs [nL, nR] of left keypoints (undistorted uL, lifts projected into the right view qR) against
    right keypoints (uR, qL): d = mean of |qR(i) - uR(j)| and |qL(j) - uL(i)|, or the one term whose lift exists; inf
    outside the epipolar gate (np_oracle.associate's cost <= max_distance_px) and where neither lift exists. Returns
    (costs, whether a candidate inside the gate had no lift on either side)."""
    cost = np.full((len(uL), len(uR)), np.inf)
    no_depth = False
    for i in range(len(uL)):
        for j in range(len(uR)):
            if np_oracle.associate(F, uL[i:i + 1], uR[j:j + 1], max_distance_px)[0][0] != 0:
                continue
            has_r, has_l = not np.isnan(qR[i][0]), not np.isnan(qL[j][0])
            if not (has_r or has_l):
                no_depth = True
                continue
            a = b = 0.0
            if has_r:
                dx, dy = qR[i][0] - uR[j][0], qR[i][1] - uR[j][1]
                a = np.sqrt(dx * dx + dy * dy)
            if has_l:
                dx, dy = qL[j][0] - uL[i][0], qL[j][1] - uL[i][1]
                b = np.sqrt(dx * dx + dy * dy)
            cost[i, j] = 0.5 * (a + b) if has_r and has_l else (a if has_r else b)
    return cost, no_depth


def stereo_objects_depth(n_objects, kp_count, kp_xy, kp_point, pairs, keypoint_config, cam_left, cam_right, K_left, K_right,
                         T_RL, F, max_distance_px=2.5, max_depth_px=8.0, optimal_correction=True):
    """Decode tables of N frames (n_objects [N], kp_count [N,O,C], kp_xy [N,O,C,S,2] float32, kp_point [N,O,C,S,3]: each
    frame's lifts in its own camera frame; only valid slots are read), pairs [P,2] (left frame, right frame),
    cam_* = camera_dict -> dict of object_match [P,O], object_cost [P,O] (the depth cost), slot_match [P,O,C,S],
    point [P,O,C,S,3] (left camera frame, NaN where unmatched), flags [P]. A candidate is admissible within
    max_distance_px of the epipolar line and with depth_costs <= max_depth_px; the greedy step runs on depth_costs."""
    lift_r, lift_l = _rigid(T_RL)               # a left lift into the right camera, a right lift into the left camera
    N, O, C, S = kp_xy.shape[:4]
    cfg = [1] + [int(v) for v in keypoint_config]
    P = len(pairs)
    out = {'object_match': np.full((P, O), -1, np.int32), 'object_cost': np.zeros((P, O)),
           'slot_match': np.full((P, O, C, S), -1, np.int32), 'point': np.full((P, O, C, S, 3), np.nan),
           'flags': np.zeros(P, np.uint32)}
    for p, (l, r) in enumerate(np.asarray(pairs).tolist()):
        if not (0 <= l < N and 0 <= r < N):
            out['flags'][p] = STEREO_BAD_PAIR
            continue

        def view(f, cam, rigid, other):
            """1. the frame's valid keypoints, distorted (float32), undistorted and their lifts projected into the other
            view: [object][map] -> [k, 2] each"""
            n = min(max(int(n_objects[f]), 0), O)
            counts = [[min(max(int(kp_count[f, o, c]), 0), cfg[c]) for c in range(C)] for o in range(n)]
            px = [[kp_xy[f, o, c, :k].astype(np.float64) for c, k in enumerate(obj)] for o, obj in enumerate(counts)]
            und = [[np.array([np_oracle.undistort_point(x, y, cam) for x, y in m]).reshape(-1, 2) for m in obj] for obj in px]
            q = [[np.array([project_lift(kp_point[f, o, c, s], *rigid, other) for s in range(k)]).reshape(-1, 2)
                  for c, k in enumerate(obj)] for o, obj in enumerate(counts)]
            return px, und, q
        px_l, und_l, q_l = view(l, cam_left, lift_r, cam_right)
        px_r, und_r, q_r = view(r, cam_right, lift_l, cam_left)
        # 2. objects by their centres
        centres_l = np.array([obj[0][0] for obj in und_l]).reshape(-1, 2)
        centres_r = np.array([obj[0][0] for obj in und_r]).reshape(-1, 2)
        costs, no_depth = depth_costs(F, centres_l, [obj[0][0] for obj in q_l], centres_r, [obj[0][0] for obj in q_r],
                                      max_distance_px)
        if ((costs <= max_depth_px).sum(axis=1) >= 2).any():
            out['flags'][p] = STEREO_AMBIGUOUS
        match, cost = _greedy(costs, max_depth_px)
        out['object_match'][p, :len(match)] = match
        out['object_cost'][p, :len(match)] = cost
        # 3. slots of every matched object pair, type by type (the centre slot with its object)
        left_px, right_px, where = [], [], []
        for i, j in enumerate(match.tolist()):
            if j < 0:
                continue
            for c in range(C):
                if c == 0:
                    slots = [0]
                else:
                    costs, missing = depth_costs(F, und_l[i][c], q_l[i][c], und_r[j][c], q_r[j][c], max_distance_px)
                    no_depth |= missing
                    slots = _greedy(costs, max_depth_px)[0].tolist()
                for s, t in enumerate(slots):
                    if t >= 0:
                        out['slot_match'][p, i, c, s] = t
                        left_px.append(px_l[i][c][s])
                        right_px.append(px_r[j][c][t])
                        where.append((i, c, s))
        # 4. StereoCamera.triangulate of every matched keypoint pair
        if where:
            X = np_oracle.triangulate_stereo(np.array(left_px), np.array(right_px), cam_left, cam_right, K_left, K_right,
                                             T_RL, F, optimal_correction)
            for (i, c, s), x in zip(where, X):
                out['point'][p, i, c, s] = x
        if no_depth:
            out['flags'][p] |= STEREO_NO_DEPTH
    return out
