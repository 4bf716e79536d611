"""TEST INFRASTRUCTURE -- statement of record for okp_triangulate_stereo_objects_f64 (stereo objects).

A composition of np_oracle's undistort_point, associate (AssociationComponent's rule, applied to the centres and then
slot type by type) and triangulate_stereo (StereoCamera.triangulate, camera_utils.py:92-110). Only tests/ import it.
"""
import numpy as np

from oracle import np_oracle

STEREO_AMBIGUOUS = 1        # a left object had two or more right objects within max_distance_px
STEREO_BAD_PAIR = 2         # a frame index of the pair is outside [0, N)


def stereo_objects(n_objects, kp_count, kp_xy, pairs, keypoint_config, cam_left, cam_right, K_left, K_right, T_RL, F,
                   max_distance_px=2.5, optimal_correction=True):
    """Decode tables of N frames (n_objects [N], kp_count [N,O,C], kp_xy [N,O,C,S,2] float32; only valid slots are read),
    pairs [P,2] (left frame, right frame), cam_* = camera_dict -> dict of object_match [P,O], object_cost [P,O],
    slot_match [P,O,C,S], point [P,O,C,S,3] (left camera frame, NaN where unmatched), flags [P]."""
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

        def view(f, cam):
            """1. the frame's valid keypoints, distorted (float32) and undistorted: [object][map] -> [k, 2] each"""
            n = min(max(int(n_objects[f]), 0), O)
            px = [[kp_xy[f, o, c, :min(max(int(kp_count[f, o, c]), 0), cfg[c])].astype(np.float64) for c in range(C)]
                  for o in range(n)]
            und = [[np.array([np_oracle.undistort_point(x, y, cam) for x, y in m]).reshape(-1, 2) for m in obj] for obj in px]
            return px, und
        px_l, und_l = view(l, cam_left)
        px_r, und_r = view(r, cam_right)
        # 2. objects by their centres
        centres_l = np.array([obj[0][0] for obj in und_l]).reshape(-1, 2)
        centres_r = np.array([obj[0][0] for obj in und_r]).reshape(-1, 2)
        within = [sum(np_oracle.associate(F, centres_l[i:i + 1], centres_r[j:j + 1], max_distance_px)[0][0] == 0
                      for j in range(len(centres_r))) for i in range(len(centres_l))]
        if any(w >= 2 for w in within):
            out['flags'][p] = STEREO_AMBIGUOUS
        match, cost = np_oracle.associate(F, centres_l, centres_r, max_distance_px)
        out['object_match'][p, :len(match)] = match
        out['object_cost'][p, :len(match)] = cost
        # 3. slots of every matched object pair, type by type (the centre slot with its object)
        left_px, right_px, where = [], [], []
        for i, j in enumerate(match.tolist()):
            if j < 0:
                continue
            for c in range(C):
                slots = [0] if c == 0 else np_oracle.associate(F, und_l[i][c], und_r[j][c], max_distance_px)[0].tolist()
                for s, t in enumerate(slots):
                    if t >= 0:
                        out['slot_match'][p, i, c, s] = t
                        left_px.append(px_l[i][c][s])
                        right_px.append(px_r[j][c][t])
                        where.append((i, c, s))
        # 4. StereoCamera.triangulate of every matched keypoint pair
        if where:
            X = np_oracle.triangulate_stereo(np.array(left_px), np.array(right_px), cam_left, cam_right, K_left, K_right, T_RL, F,
                                   optimal_correction)
            for (i, c, s), x in zip(where, X):
                out['point'][p, i, c, s] = x
    return out
