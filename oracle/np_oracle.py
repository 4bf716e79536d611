"""TEST INFRASTRUCTURE -- NumPy restatement of the reference's heatmap -> 3D keypoint path.

This module is the *checker*, never the product: only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s CPU-baseline legs may import it. Every function cites the reference lines
(relative to /root/reference) it restates. It is pinned against outputs of the unmodified
reference (``oracle/make_goldens.py`` -> ``tests/golden/*.npz``) by ``tests/test_oracle.py``.

Arithmetic contract shared with the C oracle (``okp_oracle.c``) and the CUDA kernels:

* box sum: 25 float32 additions per pixel in raster tap order (dy outer, dx inner), zero
  outside the image -- bitwise what torch's CPU conv2d with a 5x5 ones kernel returns
  (verified in SURVEY.md section 7 and again by make_goldens.py);
* NMS: exact float equality with the 5x5 maximum (-inf outside), all ties kept;
* centroid / confidence: float32, raster order over the border-clipped 5x5 window, products
  and sums rounded separately (no FMA);
* grouping distances, votes, undistortion, unprojection: float64.
"""
import numpy as np

FLAG_PEAK_OVERFLOW = 1      # more peaks on a map than the table holds
FLAG_OBJECT_OVERFLOW = 2    # more centre peaks than max_objects
FLAG_OUTLIER_SKIPPED = 4    # a spoke voted > outlier_distance from every centre (pipeline.py:121-124)
FLAG_CLUSTERED = 8          # > cfg[t] detections with cfg[t] > 1: resolved by clustering (pipeline.py:143-148)
FLAG_VOTE_OVERFLOW = 16     # more votes for one object than max_votes
FLAG_NO_CENTERS = 32        # empty centre map: no objects (pipeline.py:105-106)
FLAG_ARGMAX_RESOLVED = 64   # > cfg[t] detections with cfg[t] == 1: kept the most confident (pipeline.py:139-142)

F32 = np.float32


# ------------------------------------------------------------------------------------------
# A2-A4: box sum, NMS, threshold (perception/pipeline.py:69-73, perception/models.py:55-58)
# ------------------------------------------------------------------------------------------
def box_sum(p, size=5):
    """conv2d(p, ones(size, size), padding=size//2) with sequential float32 accumulation."""
    p = np.asarray(p, dtype=F32)
    H, W = p.shape
    r = size // 2
    padded = np.zeros((H + 2 * r, W + 2 * r), dtype=F32)
    padded[r:r + H, r:r + W] = p
    acc = np.zeros((H, W), dtype=F32)
    for dy in range(size):
        for dx in range(size):
            acc = acc + padded[dy:dy + H, dx:dx + W]        # one float32 rounding per tap
    return acc


def window_max(b, size=5):
    """max_pool2d(b, size, stride 1, padding size//2): padding value is -inf."""
    H, W = b.shape
    r = size // 2
    padded = np.full((H + 2 * r, W + 2 * r), -np.inf, dtype=F32)
    padded[r:r + H, r:r + W] = b
    out = np.full((H, W), -np.inf, dtype=F32)
    for dy in range(size):
        for dx in range(size):
            out = np.maximum(out, padded[dy:dy + H, dx:dx + W])
    return out


def find_peaks(p, threshold=0.5, nms_size=5, use_box_sum=True):
    """Pixels (y, x) in raster order whose (box-summed) value equals the window maximum and
    exceeds the threshold; also returns the score map."""
    score = box_sum(p) if use_box_sum else np.asarray(p, dtype=F32)
    keep = score == window_max(score, nms_size)
    suppressed = score * keep.astype(F32)
    ys, xs = np.nonzero(suppressed > F32(threshold))          # np.nonzero is row-major
    return np.stack([ys, xs], axis=1).astype(np.int32), score


# ------------------------------------------------------------------------------------------
# A5: sub-pixel centroid (perception/pipeline.py:46-62)
# ------------------------------------------------------------------------------------------
def centroid(p, y, x):
    """Probability-weighted mean pixel index over the clipped 5x5 window -> ((x, y), conf)."""
    H, W = p.shape
    sy = F32(0.0)
    sx = F32(0.0)
    s = F32(0.0)
    for i in range(max(y - 2, 0), min(y + 3, H)):
        for j in range(max(x - 2, 0), min(x + 3, W)):
            v = F32(p[i, j])
            sy = F32(sy + F32(v * F32(i)))
            sx = F32(sx + F32(v * F32(j)))
            s = F32(s + v)
    return np.array([F32(sx / s), F32(sy / s)], dtype=F32), s


# ------------------------------------------------------------------------------------------
# A7: equidistant undistortion, float64 (camera_utils.py:75-81 -> cv::fisheye::undistortPoints)
# ------------------------------------------------------------------------------------------
def undistort_point(u, v, cam):
    fx, fy, cx, cy = cam['fx'], cam['fy'], cam['cx'], cam['cy']
    k1, k2, k3, k4 = cam['k']
    px = (u - cx) / fx
    py = (v - cy) / fy
    theta_d = np.sqrt(px * px + py * py)
    theta_d = min(max(-np.pi / 2.0, theta_d), np.pi / 2.0)
    theta = theta_d
    scale = 0.0
    converged = False
    if abs(theta_d) > 1e-8:
        for _ in range(10):
            t2 = theta * theta
            t4 = t2 * t2
            t6 = t4 * t2
            t8 = t6 * t2
            a, b, c, d = k1 * t2, k2 * t4, k3 * t6, k4 * t8
            fix = (theta * (1 + a + b + c + d) - theta_d) / (1 + 3 * a + 5 * b + 7 * c + 9 * d)
            theta = theta - fix
            if abs(fix) < 1e-8:
                converged = True
                break
        scale = np.tan(theta) / theta_d
    else:
        converged = True
    flipped = (theta_d < 0 and theta > 0) or (theta_d > 0 and theta < 0)
    if converged and not flipped:
        return fx * (px * scale) + cx, fy * (py * scale) + cy
    return -1000000.0, -1000000.0


def camera_dict(camera):
    """Pack a camera object (K, D, Kinv, image_size) into the plain dict the oracle uses."""
    size = np.asarray(camera.image_size)
    return {
        'fx': float(camera.K[0, 0]), 'fy': float(camera.K[1, 1]),
        'cx': float(camera.K[0, 2]), 'cy': float(camera.K[1, 2]),
        'k': [float(v) for v in np.asarray(camera.D)[:4]],
        'kinv': np.asarray(camera.Kinv, dtype=np.float64).copy(),
        # pipeline.py:161-162: max_index = image_size.astype(int) - 1, i.e. (H-1, W-1),
        # later applied to (x, y) -- x is clipped with the HEIGHT.
        'clip_x': int(size[0]) - 1, 'clip_y': int(size[1]) - 1,
    }


# ------------------------------------------------------------------------------------------
# A8: DetectionToPoint (pipeline.py:155-171) + PinholeCamera.unproject (camera_utils.py:31-34)
# ------------------------------------------------------------------------------------------
def detection_to_point(xy, depth_map, cam, compat_clip_bug=True):
    """xy float32 (x, y) -> camera-frame point float64 [3]."""
    H, W = depth_map.shape
    ux, uy = undistort_point(float(xy[0]), float(xy[1]), cam)
    ux, uy = F32(ux), F32(uy)                     # OpenCV returns float32 for float32 input
    xi = int(np.rint(ux))
    yi = int(np.rint(uy))
    if compat_clip_bug:
        xi = min(max(xi, 0), cam['clip_x'])
        yi = min(max(yi, 0), cam['clip_y'])
    # the reference would raise IndexError beyond the map; stay inside it
    xi = min(max(xi, 0), W - 1)
    yi = min(max(yi, 0), H - 1)
    z = float(depth_map[yi, xi])
    kinv = cam['kinv']
    hx, hy = float(ux), float(uy)
    ray = np.array([kinv[r, 0] * hx + kinv[r, 1] * hy + kinv[r, 2] for r in range(3)])
    return ray * z


# ------------------------------------------------------------------------------------------
# deterministic replacement for the unseeded KMeans(init='random') of pipeline.py:146-148
# ------------------------------------------------------------------------------------------
def cluster_detections(points, k, iters=16):
    """Lloyd's algorithm from every k-subset of the detections as initial centres; the
    partition with the smallest inertia wins (first subset on ties). For the handful of
    detections this branch ever sees that is the global k-means optimum, which is what the
    reference's 10 random restarts converge to on well separated input. float64 arithmetic,
    centres returned in order of their initial detections. PARITY UNPINNED (nondeterministic
    in the reference)."""
    from itertools import combinations
    pts = np.asarray(points, dtype=np.float64)
    n = pts.shape[0]
    best = None
    for subset in combinations(range(n), k):
        cen = pts[list(subset)].copy()
        assign = None
        for _ in range(iters):
            d = ((pts[:, None, :] - cen[None, :, :]) ** 2).sum(axis=2)
            new_assign = d.argmin(axis=1)
            if assign is not None and (new_assign == assign).all():
                break
            assign = new_assign
            for c in range(k):
                members = pts[assign == c]
                if len(members):
                    cen[c] = members.sum(axis=0) / len(members)
        d = ((pts[:, None, :] - cen[None, :, :]) ** 2).sum(axis=2)
        inertia = d.min(axis=1).sum()
        if best is None or inertia < best[0]:
            best = (inertia, cen.copy())
    return best[1].astype(F32)


# ------------------------------------------------------------------------------------------
# A0/A6: the whole decode for a batch of frames -> fixed-capacity record tables
# ------------------------------------------------------------------------------------------
def decode(heat, depth, centers, keypoint_config, cam, max_peaks=32, max_objects=16,
           max_votes=16, threshold=0.5, outlier_distance=20.0, compat_clip_bug=True,
           with_points=True):
    """heat [N,C,H,W], depth [N,C,H,W], centers [N,T,2,H,W] (float32) -> dict of arrays laid
    out exactly like the device record tables (include/okp.h)."""
    heat = np.asarray(heat, dtype=F32)
    N, C, H, W = heat.shape
    T = C - 1
    cfg = [1] + list(keypoint_config)                       # pipeline.py:36
    assert len(cfg) == C
    S = max(cfg)
    K, O, V = max_peaks, max_objects, max_votes
    out = {
        'peak_count': np.zeros((N, C), np.int32),
        'peak_yx': np.full((N, C, K, 2), -1, np.int32),
        'peak_score': np.zeros((N, C, K), F32),
        'peak_xy': np.zeros((N, C, K, 2), F32),
        'peak_conf': np.zeros((N, C, K), F32),
        'peak_object': np.full((N, C, K), -1, np.int32),
        'peak_vote': np.zeros((N, C, K, 2), np.float64),
        'n_objects': np.zeros((N,), np.int32),
        'flags': np.zeros((N,), np.uint32),
        'kp_assigned': np.zeros((N, O, C), np.int32),
        'kp_count': np.zeros((N, O, C), np.int32),
        'kp_peak': np.full((N, O, C, S), -1, np.int32),
        'kp_xy': np.zeros((N, O, C, S, 2), F32),
        'kp_point': np.zeros((N, O, C, S, 3), np.float64),
        'n_votes': np.zeros((N, O), np.int32),
        'votes': np.zeros((N, O, V, 2), np.float64),
    }
    for n in range(N):
        flags = 0
        # ---- peaks (A2-A5), every map -------------------------------------------------------
        for c in range(C):
            yx, score = find_peaks(heat[n, c], threshold)
            out['peak_count'][n, c] = len(yx)
            if len(yx) > K:
                flags |= FLAG_PEAK_OVERFLOW
            for k, (y, x) in enumerate(yx[:K]):
                xy, conf = centroid(heat[n, c], int(y), int(x))
                out['peak_yx'][n, c, k] = (y, x)
                out['peak_score'][n, c, k] = score[y, x]
                out['peak_xy'][n, c, k] = xy
                out['peak_conf'][n, c, k] = conf
        # ---- objects = centre peaks (pipeline.py:105-114) ------------------------------------
        n_center = min(int(out['peak_count'][n, 0]), K)
        if n_center == 0:
            flags |= FLAG_NO_CENTERS
            out['flags'][n] = flags
            continue
        if n_center > O:
            flags |= FLAG_OBJECT_OVERFLOW
        n_obj = min(n_center, O)
        out['n_objects'][n] = n_obj
        center_xy = out['peak_xy'][n, 0, :n_obj].astype(np.float64)
        members = [[[] for _ in range(C)] for _ in range(n_obj)]
        for o in range(n_obj):
            members[o][0].append(o)
            out['peak_object'][n, 0, o] = o
        # ---- spoke assignment (pipeline.py:115-128) ------------------------------------------
        for t in range(T):
            c = 1 + t
            for k in range(min(int(out['peak_count'][n, c]), K)):
                px, py = out['peak_xy'][n, c, k]
                xi = min(max(int(np.rint(px)), 0), W - 1)              # np.round: half to even
                yi = min(max(int(np.rint(py)), 0), H - 1)
                vote = np.array([xi + 0.5 + float(centers[n, t, 0, yi, xi]),
                                 yi + 0.5 + float(centers[n, t, 1, yi, xi])])
                out['peak_vote'][n, c, k] = vote
                dx = center_xy[:, 0] - vote[0]
                dy = center_xy[:, 1] - vote[1]
                dist = np.sqrt(dx * dx + dy * dy)
                if dist.min() > outlier_distance:
                    flags |= FLAG_OUTLIER_SKIPPED
                    continue
                o = int(dist.argmin())                                  # first minimum
                out['peak_object'][n, c, k] = o
                members[o][c].append(k)
                if out['n_votes'][n, o] < V:
                    out['votes'][n, o, out['n_votes'][n, o]] = vote
                else:
                    flags |= FLAG_VOTE_OVERFLOW
                out['n_votes'][n, o] += 1
        # ---- per (object, type) resolution (pipeline.py:130-152) + 3D (pipeline.py:190-194) --
        for o in range(n_obj):
            for c in range(C):
                idx = members[o][c]
                out['kp_assigned'][n, o, c] = len(idx)
                if len(idx) == 0:
                    continue
                if len(idx) > cfg[c]:
                    if cfg[c] == 1:
                        conf = out['peak_conf'][n, c, idx]
                        idx = [idx[int(conf.argmax())]]                  # first maximum
                        flags |= FLAG_ARGMAX_RESOLVED
                        pts = out['peak_xy'][n, c, idx]
                    else:
                        flags |= FLAG_CLUSTERED
                        pts = cluster_detections(out['peak_xy'][n, c, idx], cfg[c])
                        idx = [-1] * cfg[c]
                else:
                    pts = out['peak_xy'][n, c, idx]
                out['kp_count'][n, o, c] = len(idx)
                for s, (k, xy) in enumerate(zip(idx, pts)):
                    out['kp_peak'][n, o, c, s] = k
                    out['kp_xy'][n, o, c, s] = xy
                    if with_points:
                        out['kp_point'][n, o, c, s] = detection_to_point(
                            xy, depth[n, c], cam, compat_clip_bug)
        out['flags'][n] = flags
    return out


# ------------------------------------------------------------------------------------------
# A11: equidistant projection (camera_utils.py:65-73 -> cv::fisheye::projectPoints)
# ------------------------------------------------------------------------------------------
def project_points(X, T_CW, cam):
    X = np.asarray(X, dtype=np.float64)
    Xc = X @ np.asarray(T_CW)[:3, :3].T + np.asarray(T_CW)[:3, 3]
    a = Xc[:, 0] / Xc[:, 2]
    b = Xc[:, 1] / Xc[:, 2]
    r = np.sqrt(a * a + b * b)
    theta = np.arctan(r)
    t2 = theta * theta
    k1, k2, k3, k4 = cam['k']
    theta_d = theta * (1.0 + k1 * t2 + k2 * t2 ** 2 + k3 * t2 ** 3 + k4 * t2 ** 4)
    with np.errstate(divide='ignore', invalid='ignore'):
        s = np.where(r > 1e-8, theta_d / r, 1.0)
    return np.stack([cam['fx'] * (a * s) + cam['cx'], cam['fy'] * (b * s) + cam['cy']], axis=1)


# ------------------------------------------------------------------------------------------
# A12/A14: DLT triangulation (camera_utils.py:103-108, scripts/label.py:296-305), any V >= 2
# ------------------------------------------------------------------------------------------
def triangulate_dlt(points, valid, projections):
    """points [P,V,2] undistorted pixels, valid [P,V] bool, projections [V,3,4] (or [P,V,3,4])
    -> X [P,3]: right singular vector of the smallest singular value of the stacked
    (x P[2] - P[0], y P[2] - P[1]) rows, dehomogenised. cv2.triangulatePoints at V = 2."""
    points = np.asarray(points, dtype=np.float64)
    Pn, Vn = points.shape[:2]
    projections = np.asarray(projections, dtype=np.float64)
    X = np.full((Pn, 3), np.nan)
    for p in range(Pn):
        rows = []
        for v in range(Vn):
            if not valid[p, v]:
                continue
            M = projections[p, v] if projections.ndim == 4 else projections[v]
            x, y = points[p, v]
            rows.append(x * M[2] - M[0])
            rows.append(y * M[2] - M[1])
        if len(rows) < 4:
            continue
        _, _, vt = np.linalg.svd(np.array(rows))
        h = vt[-1]
        X[p] = h[:3] / h[3]
    return X


# ------------------------------------------------------------------------------------------
# north_star K5 + K6 (no reference code beyond two views): robust V-view triangulation
# ------------------------------------------------------------------------------------------
def triangulate_robust(obs, valid, poses, cam, K, max_error_px=2.0, max_rounds=None):
    """obs [P,V,2] DISTORTED pixels, valid [P,V], poses [V,4,4] world->camera, cam = camera_dict,
    K = 3x3 camera matrix. Per point: DLT over the valid views of the undistorted observations with
    projections K @ poses[v][:3]; reprojection error (distorted pixels) of every view; while the
    worst valid view (first maximum) exceeds max_error_px, more than two views remain and fewer
    than max_rounds were dropped: drop it and solve again. PARITY UNPINNED (absent from the
    reference); reduces to triangulate_dlt when nothing exceeds the gate.
    -> (X [P,3], valid [P,V] uint8, err [P,V], dropped [P])"""
    obs = np.asarray(obs, dtype=np.float64)
    P, V = obs.shape[:2]
    max_rounds = V if max_rounds is None else max_rounds
    mask = np.ones((P, V), bool) if valid is None else np.asarray(valid).astype(bool).copy()
    proj = np.stack([np.asarray(K) @ np.asarray(poses[v])[:3] for v in range(V)])
    und = np.array([[undistort_point(obs[p, v, 0], obs[p, v, 1], cam) for v in range(V)] for p in range(P)])
    X = np.full((P, 3), np.nan)
    err = np.zeros((P, V))
    dropped = np.zeros(P, np.int32)
    for p in range(P):
        while True:
            views = int(mask[p].sum())
            if views < 2:
                X[p] = np.nan
                break
            X[p] = triangulate_dlt(und[p:p + 1], mask[p:p + 1], proj)[0]
            for v in range(V):
                uv = project_points(X[p:p + 1], poses[v], cam)[0]
                err[p, v] = np.hypot(uv[0] - obs[p, v, 0], uv[1] - obs[p, v, 1])
            rank = np.where(np.isnan(err[p]), np.inf, err[p])
            rank = np.where(mask[p], rank, -1.0)
            worst = int(rank.argmax())
            if not (rank[worst] > max_error_px) or views <= 2 or dropped[p] >= max_rounds:
                break
            mask[p, worst] = False
            dropped[p] += 1
    return X, mask.astype(np.uint8), err, dropped


# ------------------------------------------------------------------------------------------
# A13: cv2.correctMatches as camera_utils.py:100-101 calls it -- Hartley-Sturm optimal
# correction (Hartley & Zisserman Alg. 12.1; OpenCV 4.13 modules/calib3d/src/triangulate.cpp,
# a dependency absent from /root/reference, restated from its published algorithm). Pinned
# against cv2 itself by tests/golden/geometry.npz (pairs_corrected_*, pairs_stereo_triangulate).
# ------------------------------------------------------------------------------------------
def correct_matches(F, left, right):
    """left/right [n,2] float64 undistorted pixels with right^T F left = 0 -> corrected pairs."""
    F = np.asarray(F, dtype=np.float64)
    left = np.asarray(left, dtype=np.float64)
    right = np.asarray(right, dtype=np.float64)
    out_l = np.zeros_like(left)
    out_r = np.zeros_like(right)
    for p in range(left.shape[0]):
        x1, y1 = left[p]
        x2, y2 = right[p]
        T1 = np.array([[1, 0, x1], [0, 1, y1], [0, 0, 1.0]])
        T2 = np.array([[1, 0, x2], [0, 1, y2], [0, 0, 1.0]])
        Ft = T2.T @ F @ T1
        U, _, Vt = np.linalg.svd(Ft)
        e1 = Vt[2] / np.hypot(Vt[2, 0], Vt[2, 1])
        e2 = U[:, 2] / np.hypot(U[0, 2], U[1, 2])
        R1 = np.array([[e1[0], e1[1], 0], [-e1[1], e1[0], 0], [0, 0, 1.0]])
        R2 = np.array([[e2[0], e2[1], 0], [-e2[1], e2[0], 0], [0, 0, 1.0]])
        Fp = R2 @ Ft @ R1.T
        f1, f2, a, b, c, d = e1[2], e2[2], Fp[1, 1], Fp[1, 2], Fp[2, 1], Fp[2, 2]
        # g(t) = t((at+b)^2 + f2^2 (ct+d)^2)^2 - (ad-bc)(1+f1^2 t^2)^2 (at+b)(ct+d)
        t = np.polynomial.Polynomial([0.0, 1.0])
        q = (a * t + b) ** 2 + f2 ** 2 * (c * t + d) ** 2
        g = t * q * q - (a * d - b * c) * (1 + f1 ** 2 * t ** 2) ** 2 * (a * t + b) * (c * t + d)
        roots = g.roots()

        def cost(tv):
            return tv * tv / (1 + f1 * f1 * tv * tv) + (c * tv + d) ** 2 / ((a * tv + b) ** 2 + f2 * f2 * (c * tv + d) ** 2)
        with np.errstate(divide='ignore', invalid='ignore'):
            best_s = 1.0 / (f1 * f1) + c * c / (a * a + f2 * f2 * c * c)     # t = infinity
        best_t = None
        for r in roots:
            s = cost(float(np.real(r)))
            if s < best_s:
                best_s, best_t = s, float(np.real(r))
        if best_t is None:
            l1 = np.array([f1, 0.0, f1 * f1])
            l2 = np.array([f2 * c * c, -a * c, f2 * f2 * c * c + a * a])
        else:
            tv = best_t
            l1 = np.array([tv * tv * f1, tv, tv * tv * f1 * f1 + 1])
            l2 = np.array([f2 * (c * tv + d) ** 2, -(a * tv + b) * (c * tv + d),
                           f2 * f2 * (c * tv + d) ** 2 + (a * tv + b) ** 2])
        n1 = T1 @ R1.T @ (l1 / l1[2])
        n2 = T2 @ R2.T @ (l2 / l2[2])
        out_l[p] = n1[:2] / n1[2]
        out_r[p] = n2[:2] / n2[2]
    return out_l, out_r


def triangulate_stereo(left_px, right_px, cam_left, cam_right, K_left, K_right, T_RL, F, optimal_correction=True):
    """StereoCamera.triangulate (camera_utils.py:92-110): float32 cast, undistort (float32 results),
    correctMatches (float32 results), cv2.triangulatePoints, dehomogenise."""
    l32 = np.asarray(left_px).astype(np.float32).astype(np.float64)
    r32 = np.asarray(right_px).astype(np.float32).astype(np.float64)
    uL = np.array([undistort_point(u, v, cam_left) for u, v in l32]).astype(np.float32).astype(np.float64)
    uR = np.array([undistort_point(u, v, cam_right) for u, v in r32]).astype(np.float32).astype(np.float64)
    if optimal_correction:
        uL, uR = correct_matches(F, uL, uR)
        uL = uL.astype(np.float32).astype(np.float64)
        uR = uR.astype(np.float32).astype(np.float64)
    P1 = np.asarray(K_left) @ np.eye(3, 4)
    P2 = np.asarray(K_right) @ np.asarray(T_RL)[:3]
    pts = np.stack([uL, uR], axis=1)
    return triangulate_dlt(pts, np.ones(pts.shape[:2], bool), np.stack([P1, P2]))


# ------------------------------------------------------------------------------------------
# Stereo association -- PARITY UNPINNED: the implementation was removed from the reference, only
# its expectations survive (test/test_pipeline.py:208-261: index of the matching right point, -1 for
# unmatched, one-to-one). Statement of record for okp_stereo_associate_f64.
# ------------------------------------------------------------------------------------------
def associate(F, left, right, max_distance_px=2.5):
    """left [nL,2], right [nR,2] UNDISTORTED pixels -> (match [nL] int32, cost [nL])."""
    F = np.asarray(F, dtype=np.float64)
    left = np.asarray(left, dtype=np.float64).reshape(-1, 2)
    right = np.asarray(right, dtype=np.float64).reshape(-1, 2)
    nl, nr = left.shape[0], right.shape[0]
    cost = np.zeros((nl, nr))
    for i in range(nl):
        x, y = left[i]
        l0 = F[0, 0] * x + F[0, 1] * y + F[0, 2]
        l1 = F[1, 0] * x + F[1, 1] * y + F[1, 2]
        l2 = F[2, 0] * x + F[2, 1] * y + F[2, 2]
        for j in range(nr):
            xp, yp = right[j]
            m0 = F[0, 0] * xp + F[1, 0] * yp + F[2, 0]
            m1 = F[0, 1] * xp + F[1, 1] * yp + F[2, 1]
            r = abs(xp * l0 + yp * l1 + l2)
            cost[i, j] = 0.5 * (r / np.sqrt(l0 * l0 + l1 * l1) + r / np.sqrt(m0 * m0 + m1 * m1))
    match = np.full(nl, -1, np.int32)
    match_cost = np.zeros(nl)
    free = np.ones((nl, nr), bool)
    for _ in range(min(nl, nr)):
        # a NaN cost (a left point at the epipole: l = F x = 0) is never admissible, like any cost above the gate; the
        # step goes on with the other candidates (np.argmin would return the first NaN and end the matching)
        masked = np.where(free & ~np.isnan(cost), cost, np.inf)
        e = int(np.argmin(masked))                 # first minimum in (left, right) raster order
        i, j = divmod(e, nr)
        if not (masked[i, j] <= max_distance_px):
            break
        match[i] = j
        match_cost[i] = masked[i, j]
        free[i, :] = False
        free[:, j] = False
    return match, match_cost


# ------------------------------------------------------------------------------------------
# SURVEY 8(f) rank 3: evaluation bookkeeping, scripts/eval_model.py:137-232 (Results.add /
# Results.print_results), restated on the record tables of include/okp.h
# ------------------------------------------------------------------------------------------
EVAL_EMPTY, EVAL_MATCHED, EVAL_MISSING, EVAL_POINT_NOT_IN_VIEW, EVAL_OBJECT_NOT_IN_VIEW = -1, 0, 1, 2, 3


def _in_frame(px, image_size):
    """PinholeCamera.in_frame (camera_utils.py:36-43): (x, y) against image_size = (H, W) AS GIVEN --
    x is compared with the height, like the clip in pipeline.py:169."""
    return not ((px <= 0.0).any() or (px >= np.asarray(image_size, dtype=np.float64)).any())


def evaluation_match(kp_point, kp_count, n_objects, T_WC, scene_points, cam, image_size, max_coordinate=2.0):
    """Results.add (eval_model.py:141-187) for every frame of a batch.

    kp_point [N,O,C,S,3] camera-frame predictions 'p_C', kp_count [N,O,C], n_objects [N] (the decode
    tables); T_WC [N,4,4] camera->world per frame; scene_points [G,Kp,3] world, row 0 of every object its
    centre (video.py:121-129). Per predicted point: status, matched ground-truth point (camera frame),
    3D error and xy error in metres; per object the ground-truth object it was matched to.
      - object -> ground-truth object: nearest centre in camera-frame XY (:154-155), depth ignored;
      - the object is dropped if that ground-truth centre does not project into the frame (:159-163);
      - a point with every coordinate < max_coordinate (2.0, :171) is matched to the nearest of the
        object's ground-truth points in 3D (:172-173) and dropped if that point is not in view (:176-178);
        any other point counts as missing (:183-185)."""
    N, O, C, S = kp_point.shape[:4]
    status = np.full((N, O, C, S), EVAL_EMPTY, np.int32)
    gt_point = np.zeros((N, O, C, S, 3), np.float64)
    err = np.zeros((N, O, C, S), np.float64)
    err_xy = np.zeros((N, O, C, S), np.float64)
    gt_object = np.full((N, O), -1, np.int32)
    scene_points = np.asarray(scene_points, dtype=np.float64)
    identity = np.eye(4)
    for n in range(N):
        T = np.asarray(T_WC[n], dtype=np.float64)
        T_CW = np.eye(4)
        T_CW[:3, :3] = T[:3, :3].T
        T_CW[:3, 3] = -T_CW[:3, :3] @ T[:3, 3]                      # linalg.py:9-13
        scene_C = (T_CW[:3, :3] @ scene_points[..., None])[..., 0] + T_CW[:3, 3]   # linalg.py:15-20
        centers_C = scene_C[:, 0]
        for o in range(int(n_objects[n])):
            centre = kp_point[n, o, 0, 0]
            d = np.linalg.norm(centers_C[:, :2] - centre[:2], axis=1)
            g = int(d.argmin())
            gt_object[n, o] = g
            object_points = scene_C[g]
            visible = _in_frame(project_points(object_points[0:1], identity, cam)[0], image_size)
            for c in range(C):
                for s in range(int(kp_count[n, o, c])):
                    if not visible:
                        status[n, o, c, s] = EVAL_OBJECT_NOT_IN_VIEW
                        continue
                    point = kp_point[n, o, c, s]
                    if not (point < max_coordinate).all():
                        status[n, o, c, s] = EVAL_MISSING
                        continue
                    k = int(np.linalg.norm(object_points - point, axis=1).argmin())
                    gt = object_points[k]
                    if not _in_frame(project_points(gt[None], identity, cam)[0], image_size):
                        status[n, o, c, s] = EVAL_POINT_NOT_IN_VIEW
                        continue
                    status[n, o, c, s] = EVAL_MATCHED
                    gt_point[n, o, c, s] = gt
                    err[n, o, c, s] = np.linalg.norm(gt - point)
                    err_xy[n, o, c, s] = np.linalg.norm(gt[:2] - point[:2])
    return {'status': status, 'gt_point': gt_point, 'err': err, 'err_xy': err_xy, 'gt_object': gt_object}


def evaluation_summary(status, err, err_xy):
    """Results.print_results (eval_model.py:192-232): the row of the printed table, errors in cm."""
    matched = status == EVAL_MATCHED
    missing = int((status == EVAL_MISSING).sum())
    e = err[matched] * 100.0
    exy = err_xy[matched] * 100.0
    n_points = int(matched.sum()) + missing
    return {
        'mean': float(e.mean()), 'mean_xy': float(exy.mean()), 'std': float(e.std()),
        'small': float((err[matched] < 0.03).sum()) / float(n_points),
        'percentile25': float(np.percentile(e, 25)), 'percentile75': float(np.percentile(e, 75)),
        'missing_percentage': float(missing) / float(n_points) * 100.0, 'points': n_points,
    }


# ------------------------------------------------------------------------------------------
# SURVEY 8(f) rank 4: training / ground-truth targets, perception/datasets/video.py:17-20,44-53,
# 195-213,225-263 (_set_keypoints, the normalisation in _extract_example, _compute_centers, _compute_depth)
# ------------------------------------------------------------------------------------------
def rasterise_targets(keypoints, depths, keypoint_config, size, kernel_size=8, length_scale=2.0, center_radius=4.0):
    """One frame. keypoints [G, Kp, 2] float64 (x, y) in TARGET pixels, Kp = sum([1] + keypoint_config) with the
    object's centre first (video.py:121-129); depths [G, Kp] camera-frame z. -> heat [C,H,W], centers [C-1,2,H,W],
    depth [C,H,W] float32. kernel_size = int(64 / 8), length_scale = 64 / 32, center_radius = 64 / 16 (video.py:17-20)."""
    full = [1] + [int(v) for v in keypoint_config]
    C, (H, W) = len(full), size
    G = keypoints.shape[0]
    heat = np.zeros((C, H, W), np.float32)
    centers = np.zeros((C - 1, 2, H, W), np.float32)
    depth = np.zeros((C, H, W), np.float32)
    jj, ii = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    px = (np.arange(W, dtype=np.float32) + np.float32(0.5))[None, :].astype(np.float64)      # _pixel_indices: float32 (j + 0.5)
    py = (np.arange(H, dtype=np.float32) + np.float32(0.5))[:, None].astype(np.float64)
    for g in range(G):                                            # video.py:197-205
        for i, count in enumerate(full):
            start = sum(full[:i])
            for x, y in keypoints[g, start:start + count]:        # _set_keypoints, video.py:44-53
                ix, iy = int(np.float64(x).astype(np.int32)), int(np.float64(y).astype(np.int32))
                x0, y0 = max(ix - kernel_size, 0), max(iy - kernel_size, 0)
                x1, y1 = min(ix + kernel_size + 1, W), min(iy + kernel_size + 1, H)
                if x1 <= x0 or y1 <= y0:
                    continue
                d2 = (x - jj[y0:y1, x0:x1]) ** 2 + (y - ii[y0:y1, x0:x1]) ** 2
                value = np.exp(-d2 / length_scale ** 2)            # float64 (numba: float64 index, float64 scale)
                heat[i, y0:y1, x0:x1] = (heat[i, y0:y1, x0:x1].astype(np.float64) + value).astype(np.float32)
    for g in range(G):                                            # _compute_centers, video.py:225-242
        cx, cy = keypoints[g, 0]
        k = 1
        for i, count in enumerate(full[1:]):
            for _ in range(count):
                x, y = keypoints[g, k]
                within = np.sqrt((x - px) ** 2 + (y - py) ** 2) < center_radius
                centers[i, 0][within] = (cx - px + 0 * py)[within].astype(np.float32)
                centers[i, 1][within] = (cy - py + 0 * px)[within].astype(np.float32)
                k += 1
    for g in range(G):                                            # _compute_depth, video.py:244-263
        k = 0
        for i, count in enumerate(full):
            for _ in range(count):
                x, y = keypoints[g, k]
                within = np.sqrt((x - px) ** 2 + (y - py) ** 2) < center_radius
                depth[i][within] = np.float32(depths[g, k])
                k += 1
    peak = np.maximum(heat.max(axis=2).max(axis=1), np.float32(0.5))     # video.py:210-211
    heat = np.clip(heat / peak[:, None, None], 0.0, 1.0).astype(np.float32)
    return heat, centers, depth


# ------------------------------------------------------------------------------------------
# K1 parameter modes (SURVEY 8a, last paragraph; BASELINE.json: "3x3 max-pool NMS ... per-type top-k and
# thresholding"): CornerNet's _nms / _topk, perception/corner_net_lite/core/models/py_utils/utils.py:14-38,
# applied per keypoint type
# ------------------------------------------------------------------------------------------
def extract_peak_tables(heat, threshold=0.5, nms_size=5, use_box_sum=True, top_k=0, max_peaks=32):
    """heat [N,C,H,W] -> the peak_* tables of include/okp.h for any (nms_size, box_sum, top_k) combination.
    top_k == 0: every peak in raster order (pipeline.py:73). top_k > 0: the k highest scores of each map,
    score-descending, equal scores in raster order (torch.topk leaves that order unspecified; _topk, utils.py:27-38)."""
    heat = np.asarray(heat, dtype=F32)
    N, C, H, W = heat.shape
    K = max_peaks
    out = {'peak_count': np.zeros((N, C), np.int32), 'peak_yx': np.full((N, C, K, 2), -1, np.int32),
           'peak_score': np.zeros((N, C, K), F32), 'peak_xy': np.zeros((N, C, K, 2), F32),
           'peak_conf': np.zeros((N, C, K), F32)}
    for n in range(N):
        for c in range(C):
            yx, score = find_peaks(heat[n, c], threshold, nms_size, use_box_sum)
            total = len(yx)
            yx = yx[:K]                                          # the table keeps the first K in raster order
            if top_k > 0:
                order = sorted(range(len(yx)), key=lambda i: (-float(score[yx[i, 0], yx[i, 1]]), i))[:top_k]
                yx = yx[order]
                if total <= K:
                    total = len(yx)
            out['peak_count'][n, c] = total
            for k, (y, x) in enumerate(yx):
                xy, conf = centroid(heat[n, c], int(y), int(x))
                out['peak_yx'][n, c, k] = (y, x)
                out['peak_score'][n, c, k] = score[y, x]
                out['peak_xy'][n, c, k] = xy
                out['peak_conf'][n, c, k] = conf
    return out

