"""TEST INFRASTRUCTURE -- generate tests/golden/*.npz by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference, OpenCV and scikit-learn):

    python -m oracle.make_goldens

Every fixture stores the inputs (or, when the seeded generator made them, the recipe and digests
to rebuild them) together with what the reference returned for them, converted to the
fixed-capacity record tables of include/okp.h so tests can compare arrays one to one.
The GPU box has no reference; its tests read these files.
"""
import contextlib
import hashlib
import io
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_import, margins, np_oracle          # noqa: E402
from object_keypoints_b200 import synthetic                  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')
K_PEAKS, O_OBJECTS, V_VOTES = 32, 16, 16

# inputs of the decode fixtures: synthetic.py batches, stored in the fixture as this recipe (JSON)
VALVE_64 = {'generator': 'make_batch',
            'args': {'n_frames': 48, 'keypoint_config': [1, 3], 'size': [64, 64], 'seed': 1001, 'objects': [1, 2]}}
CUPS_64 = {'generator': 'make_batch',
           'args': {'n_frames': 64, 'keypoint_config': [1, 1, 1], 'size': [64, 64], 'seed': 1002, 'objects': [1, 4]}}
VALVE_GRID_180x320 = {'generator': 'make_grid_batch',
                      'args': {'n_frames': 6, 'keypoint_config': [1, 3], 'size': [180, 320], 'seed': 1003}}


def reference_camera(camera_utils, size):
    """The reference's own camera object, built the way eval_model.py:61-69 /
    test_pipeline.py:88-90 do."""
    camera = camera_utils.from_calibration(os.path.join(ref_import.REFERENCE_ROOT, 'config', 'calibration.yaml'))
    if tuple(size) == (64, 64):
        scaled = camera.scale(511.0 / 720.0)
        offset = np.array([(scaled.image_size[1] - 511.0) / 2.0, 0.0])
        return scaled.cut(offset).scale(64.0 / 511.0)
    return camera.scale(size[0] / 720.0)


def reference_tables(ref, camera, heat, depth, centers, cfg, seed=0):
    """Run perception.pipeline.ObjectKeypointPipeline frame by frame -> record tables."""
    N, C, H, W = heat.shape
    S = max([1] + list(cfg))
    K, O, V = K_PEAKS, O_OBJECTS, V_VOTES
    pipe = ref.ObjectKeypointPipeline([H, W], None, {'keypoint_config': list(cfg)})
    pipe.reset(camera)
    captured = []
    inner = pipe.keypoint_extraction._compute_points

    def spy(indices, probabilities):
        captured.append(np.array(indices.numpy(), copy=True).reshape(-1, 2))
        return inner(indices, probabilities)
    pipe.keypoint_extraction._compute_points = spy

    t = {
        'peak_count': np.zeros((N, C), np.int32),
        'peak_yx': np.full((N, C, K, 2), -1, np.int32),
        'peak_score': np.zeros((N, C, K), np.float32),
        'peak_xy': np.zeros((N, C, K, 2), np.float32),
        'peak_conf': np.zeros((N, C, K), np.float32),
        'peak_object': np.full((N, C, K), -1, np.int32),
        'peak_vote': np.zeros((N, C, K, 2), np.float64),
        'n_objects': np.zeros((N,), np.int32),
        'n_skipped': np.zeros((N,), np.int32),
        'kp_assigned': np.zeros((N, O, C), np.int32),
        'kp_count': np.zeros((N, O, C), np.int32),
        'kp_peak': np.full((N, O, C, S), -1, np.int32),
        'kp_xy': np.zeros((N, O, C, S, 2), np.float32),
        'kp_point': np.zeros((N, O, C, S, 3), np.float64),
        'n_votes': np.zeros((N, O), np.int32),
        'votes': np.zeros((N, O, V, 2), np.float64),
    }
    ones = torch.ones((1, 1, 5, 5), dtype=torch.float32)
    for n in range(N):
        captured.clear()
        np.random.seed(seed + n)
        log = io.StringIO()
        with contextlib.redirect_stdout(log):
            objects = pipe(torch.tensor(heat[n:n + 1]), torch.tensor(depth[n:n + 1]),
                           torch.tensor(centers[n:n + 1]))
        t['n_skipped'][n] = log.getvalue().count('skipping point')
        indices = [c.copy() for c in captured]
        points, confidence = pipe.keypoint_extraction(heat[n:n + 1])
        points, confidence = points[0], confidence[0]
        for c in range(C):
            k = len(indices[c])
            assert k <= K, "golden case exceeds the peak table"
            t['peak_count'][n, c] = k
            score = torch.nn.functional.conv2d(torch.tensor(heat[n, c])[None, None], ones, padding=2)[0, 0].numpy()
            for j in range(k):
                y, x = indices[c][j]
                t['peak_yx'][n, c, j] = (y, x)
                t['peak_score'][n, c, j] = score[y, x]
                t['peak_xy'][n, c, j] = points[c][j]
                t['peak_conf'][n, c, j] = float(confidence[c][j])
        t['n_objects'][n] = len(objects)
        assert len(objects) <= O
        # reconstruct the (pre-resolution) assignment from the ordered vote lists
        p_centers = pipe.object_extraction.image_indices + centers[n]
        cursor = [0] * len(objects)
        for o, obj in enumerate(objects):
            t['n_votes'][n, o] = len(obj['p_centers'])
            for v, vote in enumerate(obj['p_centers'][:V]):
                t['votes'][n, o, v] = vote
            t['peak_object'][n, 0, o] = o
        if len(objects):
            for c in range(1, C):
                for j in range(t['peak_count'][n, c]):
                    xy = np.clip(points[c][j].round().astype(np.int32), pipe.object_extraction.min,
                                 pipe.object_extraction.max)
                    vote = p_centers[c - 1, :, xy[1], xy[0]]
                    t['peak_vote'][n, c, j] = vote
                    for o, obj in enumerate(objects):
                        if cursor[o] < len(obj['p_centers']) and (obj['p_centers'][cursor[o]] == vote).all():
                            t['peak_object'][n, c, j] = o
                            t['kp_assigned'][n, o, c] += 1
                            cursor[o] += 1
                            break
            for o, obj in enumerate(objects):
                assert cursor[o] == len(obj['p_centers']), "vote reconstruction failed"
        for o, obj in enumerate(objects):
            for c in range(C):
                kps = np.asarray(obj['keypoints'][c]).reshape(-1, 2)
                t['kp_count'][n, o, c] = len(kps)
                if c == 0:
                    t['kp_assigned'][n, o, 0] = 1
                for s in range(len(kps)):
                    t['kp_xy'][n, o, c, s] = kps[s]
                    t['kp_point'][n, o, c, s] = obj['p_C'][c][s]
                    match = [j for j in range(t['peak_count'][n, c])
                             if (t['peak_xy'][n, c, j] == kps[s].astype(np.float32)).all()]
                    t['kp_peak'][n, o, c, s] = match[0] if match else -1
    return t


def camera_arrays(camera):
    return {'cam_K': np.asarray(camera.K, np.float64), 'cam_D': np.asarray(camera.D, np.float64),
            'cam_image_size': np.asarray(camera.image_size, np.float64)}


def save(name, **arrays):
    path = os.path.join(GOLDEN, name)
    np.savez_compressed(path, **arrays)
    print(f"wrote {name}: {os.path.getsize(path) / 1e6:.2f} MB")


def clean_frames(batch, cfg, cam_dict, wanted):
    keep = []
    for f in range(batch.heat.shape[0]):
        ok, why = margins.frame_is_clean(batch.heat[f], batch.depth[f], batch.centers[f], cfg, cam_dict)
        if ok:
            keep.append(f)
        if len(keep) == wanted:
            break
    assert len(keep) == wanted, f"only {len(keep)} clean frames"
    return np.array(keep)


def generated(recipe):
    """recipe: {'generator': name of a synthetic.py batch function, 'args': its keyword arguments}."""
    return getattr(synthetic, recipe['generator'])(**recipe['args'])


def decode_case(ref, camera_utils, name, recipe, batch, wanted, seed):
    """Stores the generator recipe, the frames kept and the SHA-256 of each input instead of the noise-like maps
    (tests/helpers.py rebuilds and checks them), so that the fixture stays a small file."""
    cfg, size = recipe['args']['keypoint_config'], recipe['args']['size']
    camera = reference_camera(camera_utils, size)
    cam_dict = np_oracle.camera_dict(camera)
    keep = clean_frames(batch, cfg, cam_dict, wanted)
    inputs = {'heat': batch.heat[keep], 'depth': batch.depth[keep], 'centers': batch.centers[keep]}
    tables = reference_tables(ref, camera, inputs['heat'], inputs['depth'], inputs['centers'], cfg, seed)
    digests = {'sha256_' + k: np.array(hashlib.sha256(np.ascontiguousarray(v).tobytes()).hexdigest()) for k, v in inputs.items()}
    save(name, input_recipe=np.array(json.dumps(recipe)), **digests, keypoint_config=np.array(cfg, np.int32),
         source_frames=keep, **camera_arrays(camera), **{'ref_' + k: v for k, v in tables.items()})
    return tables


# ----------------------------------------------------------------------------------------------
def adversarial_frames(size=(64, 64)):
    """Hand-built valve frames that sit ON the knife edges (SURVEY.md section 8d)."""
    H, W = size
    cfg = [1, 3]
    frames = []

    def blank():
        return (np.zeros((3, H, W), np.float32), np.zeros((3, H, W), np.float32),
                np.zeros((2, 2, H, W), np.float32))

    def blob(m, x, y, a=1.0, l=2.0):
        jj = np.arange(W)[None, :]
        ii = np.arange(H)[:, None]
        m += (a * np.exp(-((x - jj) ** 2 + (y - ii) ** 2) / l ** 2)).astype(np.float32)

    # 0: blob centred on a half pixel -> two tied peaks on the centre map
    h, d, c = blank()
    blob(h[0], 30.5, 20.0)
    frames.append(('half_pixel_tie', h, d, c))
    # 1: saturated plateau -> four tied peaks
    h, d, c = blank()
    blob(h[0], 40.5, 30.5, a=3.0, l=3.0)
    np.clip(h, 0, 1, out=h)
    frames.append(('plateau', h, d, c))
    # 2: blobs on the border and in the corner (clipped centroid windows)
    h, d, c = blank()
    blob(h[0], 0.3, 0.2)
    blob(h[1], W - 1.2, 30.0)
    blob(h[2], 20.0, H - 0.6)
    c[0, 0] = -30.0
    c[0, 1] = -30.0
    frames.append(('borders', h, d, c))
    # 3: empty centre map but spokes present -> no objects
    h, d, c = blank()
    blob(h[1], 20.0, 20.0)
    frames.append(('no_centres', h, d, c))
    # 4: one centre, spoke votes land > 20 px away -> skipped
    h, d, c = blank()
    blob(h[0], 12.0, 12.0)
    blob(h[1], 50.0, 50.0)
    blob(h[2], 16.0, 12.0)
    c[1, 0] = 12.0 - 16.5
    c[1, 1] = 12.0 - 12.5
    d[:] = 1.0
    frames.append(('outlier_vote', h, d, c))
    # 5: two detections of a cfg == 1 type for one object -> arg-max confidence wins
    h, d, c = blank()
    blob(h[0], 30.0, 30.0)
    blob(h[1], 24.0, 30.0, a=0.9)
    blob(h[1], 36.0, 30.0, a=0.7)
    jj = np.arange(W)[None, :] + 0.5
    ii = np.arange(H)[:, None] + 0.5
    c[0, 0] = 30.0 - jj
    c[0, 1] = 30.0 - ii
    d[:] = 0.8
    frames.append(('argmax_resolution', h, d, c))
    # 6: everything exactly zero
    h, d, c = blank()
    frames.append(('all_zero', h, d, c))
    # 7: constant map above threshold/25 -> interior plateau of equal sums, all kept
    h, d, c = blank()
    h[0, 20:28, 20:28] = 0.25
    frames.append(('constant_patch', h, d, c))
    names = [f[0] for f in frames]
    heat = np.stack([f[1] for f in frames])
    depth = np.stack([f[2] for f in frames])
    centers = np.stack([f[3] for f in frames])
    return names, cfg, heat, depth, centers


def nan_frames():
    """Valve frames of the clean generator with NaN pixels planted around a blob: torch's max_pool2d propagates NaN, so a
    NaN pixel up to 4 px from a peak (its box sum reaches the peak's 5x5 NMS window) suppresses that peak although the
    peak's own box sum is finite; a NaN pixel far from every blob changes nothing."""
    cfg = [1, 3]
    batch = synthetic.make_batch(6, cfg, (64, 64), seed=1010, objects=(1, 2))
    heat, depth, centers = batch.heat.copy(), batch.depth.copy(), batch.centers.copy()
    names = []
    for f, (offset, where) in enumerate([((4, 0), 'centre'), ((0, 3), 'spoke'), ((1, 1), 'spoke'), ((0, 5), 'centre'),
                                         (None, 'far'), ((-3, -3), 'centre')]):
        scene = batch.scenes[f]
        if where == 'centre':
            x, y = scene.centers[0]
            c = 0
        elif where == 'spoke':
            x, y = scene.spokes[1][0, 0]
            c = 2
        else:
            c, best = 0, None
            for yy in range(4, 60, 4):                     # the pixel farthest from every centre
                for xx in range(4, 60, 4):
                    d = min(np.hypot(xx - cx, yy - cy) for cx, cy in scene.centers)
                    if best is None or d > best[0]:
                        best = (d, xx, yy)
            x, y, offset = best[1], best[2], (0, 0)
            assert best[0] > 9.0
        px, py = int(round(x)) + offset[0], int(round(y)) + offset[1]
        px, py = min(max(px, 0), 63), min(max(py, 0), 63)
        heat[f, c, py, px] = np.nan
        names.append(f"{where}{offset}")
    return names, cfg, heat, depth, centers


def test_pipeline_frames(ref, camera_utils, video):
    """The synthetic-heatmap recipe of test/test_pipeline.py:39-57,97-102 (valve, 180x320)."""
    import cv2
    params = camera_utils.load_calibration_params(os.path.join(ref_import.REFERENCE_ROOT, 'config', 'calibration.yaml'))
    left = camera_utils.FisheyeCamera(params['K'], params['D'], params['image_size'])
    right = camera_utils.FisheyeCamera(params['Kp'], params['Dp'], params['image_size'])
    T_RL = params['T_RL']
    kp = np.array([[0.0, 0.0, 1.0], [0.25, 0.15, 1.0], [-0.25, -0.25, 1.0], [0.25, -0.25, 1.0]])
    keypoints = np.concatenate([kp.mean(axis=0)[None], kp])
    cfg = [1, 3]
    config = [1] + cfg
    video.SceneDataset.kernel = video._compute_kernel(50, 25, 10.0)
    full = np.zeros((2, len(config), 720, 1280))
    pixels = [left.project(keypoints, np.eye(4)), right.project(keypoints, T_RL)]
    for view in range(2):
        current = 0
        for m, count in enumerate(config):
            for _ in range(count):
                video.SceneDataset._add_kernel(full[view, m], pixels[view][current][None])
                current += 1
        full[view] /= full[view].max()
    small = np.zeros((2, len(config), 180, 320), np.float32)
    for view in range(2):
        for m in range(len(config)):
            small[view, m] = cv2.resize(full[view, m], (320, 180))
    scale = 180.0 / 720.0
    depth = np.zeros_like(small)
    depth[0] = 1.0
    depth[1] = 1.0
    centers = np.zeros((2, 2, 2, 180, 320), np.float32)
    jj = np.arange(320)[None, :] + 0.5
    ii = np.arange(180)[:, None] + 0.5
    for view in range(2):
        centre_px = pixels[view][0] * scale
        centers[view, :, 0] = centre_px[0] - jj
        centers[view, :, 1] = centre_px[1] - ii
    truth = np.stack(pixels) * scale
    return cfg, small, depth, centers, truth, keypoints, left, right, T_RL


def geometry_case(camera_utils):
    """Projection / undistortion / two-view triangulation through the reference's camera classes
    (OpenCV), including the golden pixel vectors of test/test_pipeline.py:26-33."""
    import cv2
    rng = np.random.default_rng(7)
    stereo = camera_utils.StereoCamera.from_file(os.path.join(ref_import.REFERENCE_ROOT, 'config', 'calibration.yaml'))
    left, right = stereo.left_camera, stereo.right_camera
    out = {}
    X = np.stack([rng.uniform(-0.6, 0.6, 256), rng.uniform(-0.35, 0.35, 256), rng.uniform(0.4, 2.0, 256)], axis=1)
    T = np.eye(4)
    T[:3, :3] = cv2.Rodrigues(np.array([0.05, -0.1, 0.02]))[0]
    T[:3, 3] = [0.03, -0.02, 0.1]
    out['X'] = X
    out['T_CW'] = T
    out['project_left'] = left.project(X, T)
    out['project_right'] = right.project(X, stereo.T_RL @ T)
    for cam, tag in ((left, 'full'), (left.scale(180 / 720), 'small'),
                     (reference_camera(camera_utils, (64, 64)), 'net')):
        H, W = np.asarray(cam.image_size)
        px = np.stack([rng.uniform(0, W, 512), rng.uniform(0, H, 512)], axis=1)
        out[f'undistort_in_{tag}'] = px
        out[f'undistort_out_{tag}'] = cam.undistort(px)
        out[f'undistort_out32_{tag}'] = cam.undistort(px.astype(np.float32))
        out[f'K_{tag}'] = cam.K
        out[f'D_{tag}'] = cam.D
        out[f'image_size_{tag}'] = np.asarray(cam.image_size, np.float64)
    # golden vectors printed in test/test_pipeline.py:9-12,26-33
    kp = np.array([[0.0, 0.0, 1.1], [0.1, 0.0, 1.0], [-0.1, 0.0, 1.0]])
    keypoints = np.concatenate([kp.mean(axis=0)[None], kp])
    pl = np.array([[641.00771598, 368.16440843], [641.00771598, 368.16440843],
                   [710.73402561, 368.16440843], [571.28140636, 368.16440843]])
    pr = np.array([[600.68550127, 360.58934273], [603.22381954, 360.59871037],
                   [668.67557233, 360.56260433], [530.24191134, 360.61583473]])
    out['golden_keypoints'] = keypoints
    out['golden_left'] = pl
    out['golden_right'] = pr
    out['golden_stereo_triangulate'] = stereo.triangulate(pl, pr)
    # noisy pairs: StereoCamera.triangulate (with correctMatches) and plain DLT (label.py:296-305)
    XL = X[:128]
    pL = left.project(XL, np.eye(4)) + rng.normal(0, 0.3, (128, 2))
    pR = right.project(XL, stereo.T_RL) + rng.normal(0, 0.3, (128, 2))
    out['pairs_X'] = XL
    out['pairs_left'] = pL
    out['pairs_right'] = pR
    out['pairs_stereo_triangulate'] = stereo.triangulate(pL, pR)
    uL = left.undistort(pL)
    uR = right.undistort(pR)
    P1 = left.K @ np.eye(3, 4)
    P2 = right.K @ stereo.T_RL[:3]
    Xh = cv2.triangulatePoints(P1, P2, uL.T, uR.T).T
    out['pairs_plain_dlt'] = Xh[:, :3] / Xh[:, 3:4]
    cl, cr = cv2.correctMatches(stereo.F, uL[None].astype(np.float64), uR[None].astype(np.float64))
    out['pairs_corrected_left'] = cl[0]
    out['pairs_corrected_right'] = cr[0]
    out['pairs_undistorted_left'] = uL
    out['pairs_undistorted_right'] = uR
    out['P1'] = P1
    out['P2'] = P2
    out['F'] = stereo.F
    out['T_RL'] = stereo.T_RL
    out['K_left'] = left.K
    out['D_left'] = left.D
    out['K_right'] = right.K
    out['D_right'] = right.D
    # Hartley-Sturm stress set (cv2.correctMatches): epipoles at infinity (the rig), inside the image
    # (forward motion) and a general pose, 0.5 - 1 px noise; own generator so the arrays above keep
    # their values.
    rng2 = np.random.default_rng(70)
    Kl = left.K
    Fs, ls, rs, cls_, crs = [], [], [], [], []
    poses = [stereo.T_RL]
    T = np.eye(4)
    T[:3, 3] = [0.01, -0.005, -0.25]                      # forward motion: epipole near the image centre
    poses.append(T)
    T = np.eye(4)
    T[:3, :3] = cv2.Rodrigues(np.array([0.2, -0.3, 0.1]))[0]
    T[:3, 3] = [0.2, 0.1, 0.05]
    poses.append(T)
    for T_21, sigma in zip(poses, (0.5, 1.0, 0.7)):
        Fm = camera_utils.fundamental_matrix(T_21, Kl, Kl)
        Xs = np.stack([rng2.uniform(-0.4, 0.4, 96), rng2.uniform(-0.25, 0.25, 96), rng2.uniform(0.6, 2.0, 96)], axis=1)
        x1 = (Kl @ Xs.T).T
        x1 = x1[:, :2] / x1[:, 2:]
        X2 = Xs @ T_21[:3, :3].T + T_21[:3, 3]
        x2 = (Kl @ X2.T).T
        x2 = x2[:, :2] / x2[:, 2:]
        x1 = x1 + rng2.normal(0, sigma, x1.shape)
        x2 = x2 + rng2.normal(0, sigma, x2.shape)
        c1, c2 = cv2.correctMatches(Fm, x1[None], x2[None])
        Fs.append(Fm); ls.append(x1); rs.append(x2); cls_.append(c1[0]); crs.append(c2[0])
    out['hs_F'] = np.stack(Fs)
    out['hs_left'] = np.stack(ls)
    out['hs_right'] = np.stack(rs)
    out['hs_corrected_left'] = np.stack(cls_)
    out['hs_corrected_right'] = np.stack(crs)
    # StereoCamera.triangulate at the reference test's small scale with 0.5 px noise (SURVEY 8a A13:
    # plain DLT is 1.8e-3 relative away from it there)
    small = camera_utils.StereoCamera(left.scale(180 / 720), right.scale(180 / 720), stereo.T_RL)
    Xs = np.stack([rng2.uniform(-0.3, 0.3, 64), rng2.uniform(-0.15, 0.15, 64), rng2.uniform(0.5, 1.5, 64)], axis=1)
    sl = small.left_camera.project(Xs, np.eye(4)) + rng2.normal(0, 0.5, (64, 2))
    sr = small.right_camera.project(Xs, stereo.T_RL) + rng2.normal(0, 0.5, (64, 2))
    out['small_pairs_left'] = sl
    out['small_pairs_right'] = sr
    out['small_pairs_stereo_triangulate'] = small.triangulate(sl, sr)
    return out


def producer_frames(seed, frames=1):
    """Seeded network input the producer fixture and its test both rebuild (not stored: 3 MB per frame)."""
    return np.random.default_rng(seed).normal(0.0, 1.0, (frames, 3, 511, 511)).astype(np.float32)


def producer_case(heatmaps_out=3, seed=21):
    """The UNMODIFIED reference KeypointNet (perception/models.py:60-91; its hourglass comes from
    CornerNet_Squeeze.model().hg) with name-derived weights (producer.deterministic_state_dict), float32 on
    the CPU, deployed forward of scripts/package_model.py:28. KeypointNet opens config files by relative
    path (models.py:71), hence the chdir."""
    from object_keypoints_b200 import producer
    cwd = os.getcwd()
    os.chdir(ref_import.REFERENCE_ROOT)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            from perception.models import KeypointNet
            net = KeypointNet((64, 64), heatmaps_out=heatmaps_out).eval()
    finally:
        os.chdir(cwd)
    weights = producer.deterministic_state_dict(net, seed=seed)
    net.load_state_dict(weights, strict=True)
    frames = torch.from_numpy(producer_frames(seed))
    with torch.no_grad():
        heat, depth, centers = net(frames)
    names = sorted(weights)
    return dict(seed=np.int64(seed), heatmaps_out=np.int64(heatmaps_out),
                heat=torch.sigmoid(heat[-1]).numpy(), depth=depth[-1].numpy(), centers=centers[-1].numpy(),
                parameter_names=np.array(names), parameter_sizes=np.array([weights[n].numel() for n in names], np.int64))


def import_reference_eval_model():
    """scripts/eval_model.py of the UNMODIFIED reference, with stand-ins for the GUI / plotting packages it
    imports at module level (hud, matplotlib); its Results class (:137-232) only needs NumPy."""
    import types
    ref_import.load()
    hud = sys.modules['hud']
    hud.Rect = lambda *a, **k: None
    for name in ['matplotlib', 'matplotlib.cm', 'matplotlib.pyplot']:
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules['matplotlib'].cm = sys.modules['matplotlib.cm']
    sys.modules['matplotlib'].pyplot = sys.modules['matplotlib.pyplot']
    sys.modules['matplotlib.cm'].get_cmap = lambda name: None
    scripts = os.path.join(ref_import.REFERENCE_ROOT, 'scripts')
    if scripts not in sys.path:
        sys.path.insert(0, scripts)
    with contextlib.redirect_stdout(io.StringIO()):
        import eval_model
    return eval_model


def evaluation_case(camera_utils, seed=31, frames=40, cfg=(1, 3)):
    """Results.add / print_results of the unmodified reference (scripts/eval_model.py:137-232) on a synthetic
    scene: G objects in the world, a camera pose per frame, predictions = ground truth + 1 cm noise with
    dropped / reordered / decoy objects, absent keypoints, points beyond 2 m ("missing") and objects or points
    outside the frame. The non-square 180x320 camera pins in_frame's (x, y) vs (H, W) comparison."""
    eval_model = import_reference_eval_model()
    rng = np.random.default_rng(seed)
    camera = reference_camera(camera_utils, (180, 320))
    C, S, O = 1 + len(cfg), max(cfg), O_OBJECTS
    slots = [1] + list(cfg)
    G, Kp = 5, sum(slots)
    scene = np.zeros((G, Kp, 3))
    for g in range(G):
        centre = np.array([rng.uniform(-0.7, 0.15), rng.uniform(-0.4, 0.4), rng.uniform(-0.1, 0.1)])
        scene[g, 1:] = centre + rng.normal(0, 0.08, (Kp - 1, 3))
        scene[g, 0] = scene[g, 1:].mean(axis=0)
    kp_point = np.zeros((frames, O, C, S, 3))
    kp_count = np.zeros((frames, O, C), np.int32)
    n_objects = np.zeros(frames, np.int32)
    T_WC = np.zeros((frames, 4, 4))
    rows = []

    class Row:                                   # stands in for rich.table.Table: keeps what print_results adds
        def __init__(self, *a, **k): pass
        def add_column(self, *a, **k): pass
        def add_row(self, *cells): rows.append(cells)
    eval_model.Table = Row
    results = eval_model.Results()
    results.screen = types_namespace(update=lambda table: None)
    results.set_calibration(camera)
    for n in range(frames):
        from scipy.spatial.transform import Rotation
        R = Rotation.from_euler('xyz', rng.normal(0, [0.15, 0.15, 0.3])).as_matrix()
        T = np.eye(4)
        T[:3, :3] = R
        T[:3, 3] = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), -rng.uniform(0.7, 1.9)])
        T_WC[n] = T
        T_CW = np.linalg.inv(T)
        scene_C = scene @ T_CW[:3, :3].T + T_CW[:3, 3]
        order = [g for g in rng.permutation(G) if rng.uniform() > 0.2]
        objects = []
        for g in order:
            points = scene_C[g] + rng.normal(0, 0.01, (Kp, 3))
            p_C, at = [], 0
            for c, count in enumerate(slots):
                keep = count if c == 0 else int(rng.integers(0, count + 1))
                block = points[at:at + keep].copy()
                at += count
                for row in block:
                    if c > 0 and rng.uniform() < 0.1:
                        row[2] += 2.0                      # beyond the 2 m cut -> "missing"
                p_C.append(block if keep else None)
            objects.append({'p_C': p_C})
        if rng.uniform() < 0.3:                            # a decoy far from every ground-truth object
            objects.append({'p_C': [np.array([[1.5, 1.2, 1.0]])] + [None] * (C - 1)})
        n_objects[n] = len(objects)
        for o, obj in enumerate(objects):
            for c, block in enumerate(obj['p_C']):
                if block is not None:
                    kp_count[n, o, c] = len(block)
                    kp_point[n, o, c, :len(block)] = block
        with contextlib.redirect_stdout(io.StringIO()):
            results.add(T, objects, scene)
    L = Kp
    seq_kind = np.full((frames, O, L), -1, np.int32)
    seq_pred = np.zeros((frames, O, L, 3))
    seq_gt = np.zeros((frames, O, L, 3))
    kept_objects = np.zeros(frames, np.int32)
    for n, (gt_frame, pred_frame) in enumerate(zip(results.gt_keypoints, results.predicted_keypoints)):
        kept_objects[n] = len(gt_frame)
        for o, (gt_points, pred_points) in enumerate(zip(gt_frame, pred_frame)):
            for i, (g, p) in enumerate(zip(gt_points, pred_points)):
                seq_kind[n, o, i] = 1 if p is None else 0
                if p is not None:
                    seq_pred[n, o, i], seq_gt[n, o, i] = p, g
    results.print_results()
    cells = rows[-1]
    summary = np.array([float(c.rstrip('%')) for c in cells], np.float64)
    assert (seq_kind == 1).any() and kept_objects.sum() < n_objects.sum(), "fixture must cover missing points and dropped objects"
    return dict(kp_point=kp_point, kp_count=kp_count, n_objects=n_objects, T_WC=T_WC, scene_points=scene,
                keypoint_config=np.array(cfg, np.int32), ref_seq_kind=seq_kind, ref_seq_pred=seq_pred, ref_seq_gt=seq_gt,
                ref_kept_objects=kept_objects, ref_summary=summary,
                ref_summary_columns=np.array(['mean', 'mean_xy', 'std', 'small', 'percentile25', 'percentile75',
                                              'missing_percentage', 'points']), **camera_arrays(camera))


def targets_case(video, seed=41, frames=6, cfg=(1, 3), size=(64, 64)):
    """Ground-truth targets by the UNMODIFIED reference: video._set_keypoints with the loop and normalisation of
    SceneDataset._extract_example (video.py:195-211) and the bound methods _compute_centers / _compute_depth
    (:225-263) of a bare SceneDataset whose image size equals the target size (scale factor 1). Points near and
    beyond every border, overlapping discs (later keypoints overwrite earlier ones) and crowded maps (sum > 1 ->
    normalisation) are included."""
    rng = np.random.default_rng(seed)
    full = [1] + list(cfg)
    Kp, C, (H, W) = sum(full), len(full), size
    G = 3
    ds = object.__new__(video.SceneDataset)
    ds.keypoint_config, ds.n_keypoints, ds.n_objects, ds.keypoint_maps = full, Kp, G, C
    ds.target_size, ds.image_size = np.array(size), (size[0], size[1])
    ds.target_pixel_indices = video._pixel_indices(*size)
    keypoints = np.zeros((frames, G, Kp, 2))
    depths = rng.uniform(0.4, 1.5, (frames, G, Kp))
    heat = np.zeros((frames, C, H, W), np.float32)
    centers = np.zeros((frames, C - 1, 2, H, W), np.float32)
    depth = np.zeros((frames, C, H, W), np.float32)
    for n in range(frames):
        for g in range(G):
            centre = rng.uniform(-6, 70, 2) if n % 2 else rng.uniform(8, 56, 2)
            keypoints[n, g, 1:] = centre + rng.normal(0, 3.0 if n < 4 else 0.7, (Kp - 1, 2))
            keypoints[n, g, 0] = keypoints[n, g, 1:].mean(axis=0)
        target = np.zeros((C, H, W), np.float32)
        for g in range(G):                                       # video.py:197-205
            for i, count in enumerate(full):
                start = sum(full[:i])
                video._set_keypoints(target[i], keypoints[n, g, start:start + count])
        peak = np.maximum(target.max(axis=2).max(axis=1), 0.5)   # video.py:210-211
        heat[n] = np.clip(target / peak[:, None, None], 0.0, 1.0)
        flat = keypoints[n].reshape(G * Kp, 2)
        centers[n] = ds._compute_centers(flat)
        depth[n] = ds._compute_depth(flat, np.concatenate([np.zeros((G * Kp, 2)), depths[n].reshape(-1, 1)], axis=1))
    assert heat.max() == 1.0 and (centers != 0).any() and (depth != 0).any()
    return dict(keypoints=keypoints, depths=depths, keypoint_config=np.array(cfg, np.int32), size=np.array(size, np.int32),
                ref_heat=heat, ref_centers=centers, ref_depth=depth)


def cornernet_topk_case(seed=51, maps=6, size=(48, 64), k=20, threshold=0.3):
    """CornerNet's own _nms(kernel=3) + _topk(K) (perception/corner_net_lite/core/models/py_utils/utils.py:14-38,
    imported unmodified), applied to one keypoint type at a time. Maps: smooth random fields with distinct values,
    so torch.topk's order is unambiguous, and fewer peaks above `threshold` than table slots."""
    ref_import.load()
    from perception.corner_net_lite.core.models.py_utils import utils as cornernet
    rng = np.random.default_rng(seed)
    H, W = size
    heat = np.zeros((maps, 1, H, W), np.float32)
    yy, xx = np.mgrid[0:H, 0:W]
    for m in range(maps):
        field = rng.uniform(0.0, 0.25, (H, W))
        for _ in range(int(rng.integers(25, 40))):
            cy, cx, a, l = rng.uniform(0, H), rng.uniform(0, W), rng.uniform(0.35, 1.0), rng.uniform(1.0, 2.5)
            field = np.maximum(field, a * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / l ** 2))
        heat[m, 0] = field.astype(np.float32)
    kept = cornernet._nms(torch.from_numpy(heat), kernel=3)
    scores, inds, classes, ys, xs = cornernet._topk(kept, K=k)
    assert len(np.unique(scores.numpy())) == scores.numel(), "scores must be distinct"
    assert (scores.numpy() > threshold).all() and ((kept.numpy() > threshold).sum(axis=(1, 2, 3)) <= 256).all()
    return dict(heat=heat, k=np.int64(k), threshold=np.float32(threshold), ref_scores=scores.numpy(),
                ref_ys=ys.numpy().astype(np.int32), ref_xs=xs.numpy().astype(np.int32),
                ref_suppressed=kept.numpy())


def types_namespace(**kw):
    import types
    return types.SimpleNamespace(**kw)


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    ref, camera_utils, video = ref_import.load()
    if '--only-geometry' in sys.argv:
        save('geometry.npz', **geometry_case(camera_utils))
        return
    if '--only-producer' in sys.argv:
        save('producer_valve.npz', **producer_case())
        return
    if '--only-nan' in sys.argv:
        names, cfg, heat, depth, centers = nan_frames()
        camera = reference_camera(camera_utils, (64, 64))
        tables = reference_tables(ref, camera, heat, depth, centers, cfg, seed=16)
        save('nan_64.npz', heat=heat, depth=depth, centers=centers, names=np.array(names),
             keypoint_config=np.array(cfg, np.int32), **camera_arrays(camera), **{'ref_' + k: v for k, v in tables.items()})
        return
    if '--only-topk' in sys.argv:
        save('cornernet_topk.npz', **cornernet_topk_case())
        return
    if '--only-targets' in sys.argv:
        save('targets_64.npz', **targets_case(video))
        return
    if '--only-evaluation' in sys.argv:
        save('evaluation.npz', **evaluation_case(camera_utils))
        return

    # 1-2: model-resolution clean sets (bit-exact parity)
    valve = generated(VALVE_64)
    decode_case(ref, camera_utils, 'valve_64.npz', VALVE_64, valve, 24, seed=11)
    cups = generated(CUPS_64)
    decode_case(ref, camera_utils, 'cups_64.npz', CUPS_64, cups, 24, seed=12)

    # 3: 180x320, eight valves on a grid (config 3 frames)
    grid = generated(VALVE_GRID_180x320)
    decode_case(ref, camera_utils, 'valve_grid_180x320.npz', VALVE_GRID_180x320, grid, 2, seed=13)

    # 4: knife edges -- compared with set / flag semantics
    names, cfg, heat, depth, centers = adversarial_frames()
    camera = reference_camera(camera_utils, (64, 64))
    tables = reference_tables(ref, camera, heat, depth, centers, cfg, seed=14)
    save('adversarial_64.npz', heat=heat, depth=depth, centers=centers, names=np.array(names),
         keypoint_config=np.array(cfg, np.int32), **camera_arrays(camera),
         **{'ref_' + k: v for k, v in tables.items()})

    # 4b: NaN pixels around peaks (max_pool2d propagates NaN)
    names, cfg, heat, depth, centers = nan_frames()
    tables = reference_tables(ref, camera, heat, depth, centers, cfg, seed=16)
    save('nan_64.npz', heat=heat, depth=depth, centers=centers, names=np.array(names),
         keypoint_config=np.array(cfg, np.int32), **camera_arrays(camera), **{'ref_' + k: v for k, v in tables.items()})

    # 5: the reference's own test recipe (test_pipeline.py)
    cfg, heat, depth, centers, truth, keypoints, left, right, T_RL = test_pipeline_frames(ref, camera_utils, video)
    camera = left.scale(180 / 720)
    tables = reference_tables(ref, camera, heat, depth, centers, cfg, seed=15)
    save('test_pipeline_180x320.npz', heat=heat, depth=depth, centers=centers, truth_pixels=truth,
         keypoints_3d=keypoints, T_RL=T_RL, keypoint_config=np.array(cfg, np.int32),
         **camera_arrays(camera), **{'ref_' + k: v for k, v in tables.items()})

    # 6: full box-sum maps straight from torch's conv2d (bitwise pin of the summation order)
    ones = torch.ones((1, 1, 5, 5), dtype=torch.float32)
    maps = np.concatenate([valve.heat[:2].reshape(-1, 64, 64), cups.heat[:1].reshape(-1, 64, 64)])
    sums = torch.nn.functional.conv2d(torch.tensor(maps)[:, None], ones, padding=2)[:, 0].numpy()
    big = grid.heat[0, :1]
    big_sums = torch.nn.functional.conv2d(torch.tensor(big)[:, None], ones, padding=2)[:, 0].numpy()
    save('boxsum.npz', maps=maps, sums=sums, big=big, big_sums=big_sums)

    # 7: camera geometry and triangulation
    save('geometry.npz', **geometry_case(camera_utils))

    # 9: evaluation bookkeeping (scripts/eval_model.py Results)
    save('evaluation.npz', **evaluation_case(camera_utils))

    # 11: CornerNet's 3x3 NMS + top-k (the K1 parameter modes)
    save('cornernet_topk.npz', **cornernet_topk_case())

    # 10: ground-truth target rasterisation (perception/datasets/video.py)
    save('targets_64.npz', **targets_case(video))

    # 8: the keypoint network (input producer of BASELINE config 5)
    save('producer_valve.npz', **producer_case())


if __name__ == '__main__':
    main()
