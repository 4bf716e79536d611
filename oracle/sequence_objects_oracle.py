"""TEST INFRASTRUCTURE -- statement of record for okp_triangulate_sequence_objects_f64 (SequenceTriangulator.objects): the
decoded objects of a posed sequence, each anchor frame's objects matched into its V - 1 view frames, every anchor slot
triangulated over its track.

A composition of existing pieces, none of them modified: per (anchor, view) pair the stereo rules with the anchor frame as
the left view -- np_oracle.undistort_point, then np_oracle.associate (association 'epipolar', stereo_oracle's rule) or
stereo_depth_oracle's project_lift, depth_costs and _greedy (association 'depth') -- on the pair's F and rigid motion as
SequenceTriangulator.prepare forms them (F [A,V-1,3,3], motion [A,V-1,2,12]: the same doubles the kernel reads); then
c_oracle.triangulate_robust per anchor, as sequence_oracle.sequence_tracks does. PARITY IS UNPINNED for V > 2 (DESIGN.md
section 4), as for the per-peak chain. Only tests/ import it.
"""
import numpy as np

from oracle import c_oracle, np_oracle
from oracle.stereo_depth_oracle import STEREO_NO_DEPTH, _greedy, depth_costs, project_lift
from oracle.stereo_oracle import STEREO_AMBIGUOUS, STEREO_BAD_PAIR


def _epipolar(F, uL, uR, max_distance_px):
    """stereo_oracle's rule: (match, cost, ambiguous) of np_oracle.associate on the undistorted points."""
    ambiguous = any(sum(np_oracle.associate(F, uL[i:i + 1], uR[j:j + 1], max_distance_px)[0][0] == 0 for j in range(len(uR))) >= 2
                    for i in range(len(uL)))
    match, cost = np_oracle.associate(F, uL, uR, max_distance_px)
    return match, cost, ambiguous, False


def _depth(F, uL, qL, uR, qR, max_distance_px, max_depth_px):
    """stereo_depth_oracle's rule: (match, cost, ambiguous, no_depth); qL: the anchor keypoints' lifts in the view frame,
    qR: the view keypoints' lifts in the anchor frame."""
    costs, no_depth = depth_costs(F, uL, qL, uR, qR, max_distance_px)
    match, cost = _greedy(costs, max_depth_px)
    return match, cost, bool(((costs <= max_depth_px).sum(axis=1) >= 2).any()), no_depth


def sequence_objects(n_objects, kp_count, kp_xy, kp_point, keypoint_config, frames, F, motion, poses, camera,
                     association='epipolar', max_distance_px=2.5, max_depth_px=16.0, max_error_px=2.0, max_rounds=None):
    """Decode tables of N frames of one camera (n_objects [N], kp_count [N,O,C], kp_xy [N,O,C,S,2] float32, kp_point
    [N,O,C,S,3] each frame's lifts in its own camera frame; only valid slots are read), frames [A,V] (anchor, views),
    F [A,V-1,3,3], motion [A,V-1,2,12], poses [A,V,4,4] world -> camera, camera: an object with K, D, Kinv, image_size.
    -> dict with the fields of OkpSequenceObjectTables (include/okp.h)."""
    frames = np.asarray(frames)
    N, O, C, S = kp_xy.shape[:4]
    A, V = frames.shape
    cfg = [1] + [int(v) for v in keypoint_config]
    cam = np_oracle.camera_dict(camera)
    out = {'object_match': np.full((A, V - 1, O), -1, np.int32), 'object_cost': np.zeros((A, V - 1, O)),
           'slot_match': np.full((A, V - 1, O, C, S), -1, np.int32), 'flags': np.zeros((A, V - 1), np.uint32),
           'observations': np.zeros((A, O, C, S, V, 2)), 'observed': np.zeros((A, O, C, S, V), np.uint8)}

    def view(f, rigid):
        """1. the frame's valid keypoints, distorted (float32), undistorted and (depth) their lifts projected into the other
        frame (rigid: (R, t) of the motion into it): [object][map] -> [k, 2] each"""
        n = min(max(int(n_objects[f]), 0), O)
        counts = [[min(max(int(kp_count[f, o, c]), 0), cfg[c]) for c in range(C)] for o in range(n)]
        px = [[kp_xy[f, o, c, :k].astype(np.float64) for c, k in enumerate(obj)] for o, obj in enumerate(counts)]
        und = [[np.array([np_oracle.undistort_point(x, y, cam) for x, y in m]).reshape(-1, 2) for m in obj] for obj in px]
        q = None
        if association == 'depth' and rigid is not None:
            q = [[np.array([project_lift(kp_point[f, o, c, s], *rigid, cam) for s in range(k)]).reshape(-1, 2)
                  for c, k in enumerate(obj)] for o, obj in enumerate(counts)]
        return px, und, q

    for a in range(A):
        fl = int(frames[a, 0])
        if 0 <= fl < N:                                       # column 0: the anchor's own keypoints
            px_l = view(fl, None)[0]
            for o, obj in enumerate(px_l):
                for c, m in enumerate(obj):
                    out['observations'][a, o, c, :len(m), 0] = m
                    out['observed'][a, o, c, :len(m), 0] = 1
        for v in range(1, V):
            fr = int(frames[a, v])
            if not (0 <= fl < N and 0 <= fr < N):
                out['flags'][a, v - 1] = STEREO_BAD_PAIR
                continue
            M = motion[a, v - 1]
            rigid = [(M[w, :9].reshape(3, 3), M[w, 9:]) for w in range(2)]
            px_l, und_l, q_l = view(fl, rigid[0])
            px_r, und_r, q_r = view(fr, rigid[1])
            Fp = F[a, v - 1]

            def match(i, j, c):
                if association == 'depth':
                    return _depth(Fp, und_l[i][c], q_l[i][c], und_r[j][c], q_r[j][c], max_distance_px, max_depth_px)
                return _epipolar(Fp, und_l[i][c], und_r[j][c], max_distance_px)
            # 2. objects by their centres
            centres = [np.array([obj[0][0] for obj in und]).reshape(-1, 2) for und in (und_l, und_r)]
            if association == 'depth':
                lifts = [[obj[0][0] for obj in q] for q in (q_l, q_r)]
                objects, cost, ambiguous, no_depth = _depth(Fp, centres[0], lifts[0], centres[1], lifts[1], max_distance_px,
                                                            max_depth_px)
            else:
                objects, cost, ambiguous, no_depth = _epipolar(Fp, centres[0], centres[1], max_distance_px)
            out['object_match'][a, v - 1, :len(objects)] = objects
            out['object_cost'][a, v - 1, :len(objects)] = cost
            # 3. slots of every matched object pair, type by type (the centre slot with its object), and the tracks
            for i, j in enumerate(objects.tolist()):
                if j < 0:
                    continue
                for c in range(C):
                    if c == 0:
                        slots = [0]
                    elif len(und_l[i][c]) == 0 or len(und_r[j][c]) == 0:
                        slots = [-1] * len(und_l[i][c])
                    else:
                        slots, _, _, missing = match(i, j, c)
                        slots = slots.tolist()
                        no_depth |= missing
                    for s, t in enumerate(slots):
                        if t >= 0:
                            out['slot_match'][a, v - 1, i, c, s] = t
                            out['observations'][a, i, c, s, v] = px_r[j][c][t]
                            out['observed'][a, i, c, s, v] = 1
            out['flags'][a, v - 1] = (STEREO_AMBIGUOUS if ambiguous else 0) | (STEREO_NO_DEPTH if no_depth else 0)
    # 4. every anchor's tracks, one robust V-view triangulation per anchor
    rounds = V if max_rounds is None else int(max_rounds)
    Pg = O * C * S
    out['valid'] = out['observed'].copy()
    out['point'] = np.zeros((A, O, C, S, 3))
    out['error'] = np.zeros((A, O, C, S, V))
    out['dropped'] = np.zeros((A, O, C, S), np.int32)
    for a in range(A):
        X, valid, err, dropped = c_oracle.triangulate_robust(out['observations'][a].reshape(Pg, V, 2),
                                                             out['observed'][a].reshape(Pg, V), poses[a], camera, max_error_px,
                                                             rounds)
        err[out['observed'][a].reshape(Pg, V).sum(axis=1) < 2] = np.nan   # no solve: no error
        out['point'][a], out['valid'][a] = X.reshape(O, C, S, 3), valid.reshape(O, C, S, V)
        out['error'][a], out['dropped'][a] = err.reshape(O, C, S, V), dropped.reshape(O, C, S)
    return out
