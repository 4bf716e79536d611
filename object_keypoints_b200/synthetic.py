"""Synthetic network outputs (heatmaps, depth maps, centre-vector maps) shaped like the
training targets of the reference (``perception/datasets/video.py:17-53,225-263``).

Conventions mirrored from the reference:

* one heatmap per keypoint type plus a leading object-centre map (video.py:75,117-129);
* a keypoint at (x, y) adds ``a * exp(-((x-j)^2 + (y-i)^2) / l^2)`` to pixel (row i, col j),
  l = 2 px at 64x64 (video.py:20,23-25,44-53) -- the blob lives in pixel-INDEX coordinates;
* centre-vector map of spoke type t holds ``centre_xy - (j + 0.5, i + 0.5)`` at the pixels
  whose centre (j + 0.5, i + 0.5) is closer than 4 px to a spoke keypoint (video.py:18,225-242);
* depth map c holds the keypoint's camera-frame z inside the same 4 px disc (video.py:244-263).

Two back ends rasterise the same scene description: NumPy (tests, goldens: defines the exact
float32 values) and torch (bench inputs created directly in HBM).
"""
from dataclasses import dataclass, field

import numpy as np

LENGTH_SCALE = 2.0       # video.py:20 at heatmap_size 64
DISC_RADIUS = 4.0        # video.py:18 center_radius
BLOB_HALF_WINDOW = 8     # video.py:19 kernel_size
NOISE_AMPLITUDE = 0.01


def default_camera(prediction_size=(64, 64)):
    """The camera eval_model.py:61-69 hands to the pipeline: Kalibr cam0 scaled to the
    network input (511 px high), cropped, scaled to the 64x64 prediction; for other
    prediction sizes the full-resolution camera is scaled to the prediction height
    (test_pipeline.py:25,88-90)."""
    import os
    from . import camera_utils
    calibration = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                               'config', 'calibration.yaml')
    camera = camera_utils.from_calibration(calibration)
    if tuple(prediction_size) == (64, 64):
        scaled = camera.scale(511.0 / 720.0)
        offset = np.array([(scaled.image_size[1] - 511.0) / 2.0, 0.0])
        return scaled.cut(offset).scale(64.0 / 511.0)
    return camera.scale(prediction_size[0] / 720.0)


@dataclass
class Scene:
    """Ground truth of one frame. All coordinates are (x, y) in prediction pixels."""
    centers: np.ndarray                 # [n_obj, 2]
    spokes: list                        # per spoke type t: [n_obj, cfg[t], 2]
    amplitude_center: np.ndarray        # [n_obj]
    amplitude_spokes: list              # per type: [n_obj, cfg[t]]
    z_center: np.ndarray                # [n_obj]
    z_spokes: list                      # per type: [n_obj, cfg[t]]


@dataclass
class Batch:
    heat: np.ndarray                    # [N, C, H, W] float32
    depth: np.ndarray                   # [N, C, H, W] float32
    centers: np.ndarray                 # [N, T, 2, H, W] float32
    scenes: list = field(default_factory=list)
    keypoint_config: list = field(default_factory=list)


def _far_enough(candidate, others, min_distance):
    if len(others) == 0:
        return True
    d = np.linalg.norm(np.asarray(others) - candidate[None], axis=1)
    return bool((d >= min_distance).all())


def sample_scene(rng, keypoint_config, size, n_objects, center_separation=22.0,
                 spoke_radius=(5.0, 8.0), peak_separation=6.0, border=4.0, max_tries=2000):
    """Rejection-sample object centres and spoke keypoints (SURVEY.md section 8d, config 2):
    centres >= center_separation apart, spokes spoke_radius from their centre, same-map peaks
    >= peak_separation apart, everything >= border px inside the image."""
    H, W = size
    lo = np.array([border, border])
    hi = np.array([W - 1 - border, H - 1 - border])
    for _ in range(max_tries):
        centers = []
        ok = True
        for _o in range(n_objects):
            for _t in range(200):
                c = rng.uniform(lo + spoke_radius[1], hi - spoke_radius[1])
                if _far_enough(c, centers, center_separation):
                    centers.append(c)
                    break
            else:
                ok = False
                break
        if not ok:
            continue
        centers = np.array(centers).reshape(n_objects, 2)
        spokes = []
        for count in keypoint_config:
            placed = []            # all peaks on this map so far
            per_object = np.zeros((n_objects, count, 2))
            for o in range(n_objects):
                for k in range(count):
                    for _t in range(200):
                        angle = rng.uniform(0.0, 2.0 * np.pi)
                        radius = rng.uniform(*spoke_radius)
                        p = centers[o] + radius * np.array([np.cos(angle), np.sin(angle)])
                        inside = (p >= lo).all() and (p <= hi).all()
                        # a spoke must vote for its own centre: keep it away from other centres
                        own = np.linalg.norm(centers - p[None], axis=1)
                        if inside and own.argmin() == o and _far_enough(p, placed, peak_separation):
                            placed.append(p)
                            per_object[o, k] = p
                            break
                    else:
                        ok = False
                        break
                if not ok:
                    break
            if not ok:
                break
            spokes.append(per_object)
        if not ok:
            continue
        return Scene(
            centers=centers,
            spokes=spokes,
            amplitude_center=rng.uniform(0.6, 1.0, size=n_objects),
            amplitude_spokes=[rng.uniform(0.6, 1.0, size=s.shape[:2]) for s in spokes],
            z_center=rng.uniform(0.4, 1.5, size=n_objects),
            z_spokes=[rng.uniform(0.4, 1.5, size=s.shape[:2]) for s in spokes],
        )
    raise RuntimeError("could not place the requested objects; relax the separations")


def _splat(heatmap, xy, amplitude, length_scale):
    H, W = heatmap.shape
    x, y = float(xy[0]), float(xy[1])
    j0, j1 = max(int(x) - BLOB_HALF_WINDOW, 0), min(int(x) + BLOB_HALF_WINDOW + 1, W)
    i0, i1 = max(int(y) - BLOB_HALF_WINDOW, 0), min(int(y) + BLOB_HALF_WINDOW + 1, H)
    if j1 <= j0 or i1 <= i0:
        return
    jj = np.arange(j0, j1, dtype=np.float64)[None, :]
    ii = np.arange(i0, i1, dtype=np.float64)[:, None]
    blob = amplitude * np.exp(-((x - jj) ** 2 + (y - ii) ** 2) / length_scale ** 2)
    heatmap[i0:i1, j0:j1] += blob.astype(np.float32)


def _disc(H, W, xy, radius=DISC_RADIUS):
    """Boolean mask of pixels whose centre (j+0.5, i+0.5) is within radius of xy, plus the
    window it lives in (to keep rasterisation local)."""
    x, y = float(xy[0]), float(xy[1])
    r = int(np.ceil(radius)) + 1
    j0, j1 = max(int(x) - r, 0), min(int(x) + r + 1, W)
    i0, i1 = max(int(y) - r, 0), min(int(y) + r + 1, H)
    jj = np.arange(j0, j1, dtype=np.float64)[None, :] + 0.5
    ii = np.arange(i0, i1, dtype=np.float64)[:, None] + 0.5
    mask = np.sqrt((x - jj) ** 2 + (y - ii) ** 2) < radius
    return (slice(i0, i1), slice(j0, j1)), mask, jj, ii


def rasterize(scene, keypoint_config, size, rng, vote_noise=0.25, noise=NOISE_AMPLITUDE,
              length_scale=LENGTH_SCALE):
    """Scene -> (heat [C,H,W], depth [C,H,W], centers [T,2,H,W]) float32."""
    H, W = size
    T = len(keypoint_config)
    C = T + 1
    heat = np.zeros((C, H, W), dtype=np.float32)
    depth = np.zeros((C, H, W), dtype=np.float32)
    centers = np.zeros((T, 2, H, W), dtype=np.float32)
    n_objects = scene.centers.shape[0]
    for o in range(n_objects):
        _splat(heat[0], scene.centers[o], scene.amplitude_center[o], length_scale)
        window, mask, _, _ = _disc(H, W, scene.centers[o])
        depth[0][window][mask] = np.float32(scene.z_center[o])
        for t in range(T):
            for k in range(keypoint_config[t]):
                p = scene.spokes[t][o, k]
                _splat(heat[1 + t], p, scene.amplitude_spokes[t][o, k], length_scale)
                window, mask, jj, ii = _disc(H, W, p)
                depth[1 + t][window][mask] = np.float32(scene.z_spokes[t][o, k])
                vx = np.broadcast_to(scene.centers[o, 0] - jj, mask.shape)
                vy = np.broadcast_to(scene.centers[o, 1] - ii, mask.shape)
                jitter = rng.normal(0.0, vote_noise, size=(2,) + mask.shape) if vote_noise > 0 else np.zeros((2,) + mask.shape)
                centers[t, 0][window][mask] = (vx + jitter[0])[mask].astype(np.float32)
                centers[t, 1][window][mask] = (vy + jitter[1])[mask].astype(np.float32)
    if noise > 0:
        heat += rng.uniform(0.0, noise, size=heat.shape).astype(np.float32)
    np.clip(heat, 0.0, 1.0, out=heat)
    return heat, depth, centers


def make_batch(n_frames, keypoint_config, size=(64, 64), seed=0, objects=(1, 4), **layout):
    """N independent frames (SURVEY.md section 8d). Per-frame random substreams come from
    SeedSequence.spawn, so frame f is the same whatever n_frames is."""
    H, W = size
    T = len(keypoint_config)
    heat = np.zeros((n_frames, T + 1, H, W), dtype=np.float32)
    depth = np.zeros_like(heat)
    centers = np.zeros((n_frames, T, 2, H, W), dtype=np.float32)
    scenes = []
    children = np.random.SeedSequence(seed).spawn(n_frames)
    for f in range(n_frames):
        rng = np.random.default_rng(children[f])
        n_objects = int(rng.integers(objects[0], objects[1] + 1))
        scene = sample_scene(rng, keypoint_config, size, n_objects, **layout)
        heat[f], depth[f], centers[f] = rasterize(scene, keypoint_config, size, rng)
        scenes.append(scene)
    return Batch(heat=heat, depth=depth, centers=centers, scenes=scenes,
                 keypoint_config=list(keypoint_config))


def grid_scene(rng, keypoint_config, size, grid=(4, 2), jitter=6.0, spoke_radius=(6.0, 10.0)):
    """Objects on a jittered grid (config 3: eight valves in a 180x320 frame)."""
    H, W = size
    gx, gy = grid
    n_objects = gx * gy
    centers = np.zeros((n_objects, 2))
    for o in range(n_objects):
        cx = (o % gx + 0.5) * W / gx
        cy = (o // gx + 0.5) * H / gy
        centers[o] = (cx + rng.uniform(-jitter, jitter), cy + rng.uniform(-jitter, jitter))
    spokes = []
    for count in keypoint_config:
        per_object = np.zeros((n_objects, count, 2))
        for o in range(n_objects):
            start = rng.uniform(0.0, 2.0 * np.pi)
            for k in range(count):
                angle = start + 2.0 * np.pi * k / max(count, 1) + rng.uniform(-0.3, 0.3)
                radius = rng.uniform(*spoke_radius)
                per_object[o, k] = centers[o] + radius * np.array([np.cos(angle), np.sin(angle)])
        spokes.append(per_object)
    return Scene(
        centers=centers, spokes=spokes,
        amplitude_center=rng.uniform(0.6, 1.0, size=n_objects),
        amplitude_spokes=[rng.uniform(0.6, 1.0, size=s.shape[:2]) for s in spokes],
        z_center=rng.uniform(0.4, 1.5, size=n_objects),
        z_spokes=[rng.uniform(0.4, 1.5, size=s.shape[:2]) for s in spokes],
    )


def make_grid_batch(n_frames, keypoint_config, size=(180, 320), seed=0, grid=(4, 2)):
    H, W = size
    T = len(keypoint_config)
    heat = np.zeros((n_frames, T + 1, H, W), dtype=np.float32)
    depth = np.zeros_like(heat)
    centers = np.zeros((n_frames, T, 2, H, W), dtype=np.float32)
    scenes = []
    children = np.random.SeedSequence(seed).spawn(n_frames)
    for f in range(n_frames):
        rng = np.random.default_rng(children[f])
        scene = grid_scene(rng, keypoint_config, size, grid=grid)
        heat[f], depth[f], centers[f] = rasterize(scene, keypoint_config, size, rng)
        scenes.append(scene)
    return Batch(heat=heat, depth=depth, centers=centers, scenes=scenes,
                 keypoint_config=list(keypoint_config))


# --------------------------------------------------------------------------------------------
# torch back end: the same scene description rasterised directly in device memory, for bench
# inputs that are too large to build with NumPy loops (4096 frames of 180x320).
# --------------------------------------------------------------------------------------------
def torch_grid_batch(n_frames, keypoint_config, size=(180, 320), seed=0, grid=(4, 2),
                     device='cuda', chunk=256):
    """Device-resident (heat, depth, centers) float32 tensors plus the ground-truth object count
    per frame. Every frame is different (per-frame jitter); values follow the same recipe as
    ``rasterize`` but are produced by torch arithmetic, so they are not bit-identical to the
    NumPy back end -- parity tests use NumPy inputs, the bench uses these."""
    import torch
    H, W = size
    T = len(keypoint_config)
    C = T + 1
    gx, gy = grid
    n_obj = gx * gy
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    heat = torch.empty((n_frames, C, H, W), dtype=torch.float32, device=device)
    depth = torch.zeros((n_frames, C, H, W), dtype=torch.float32, device=device)
    centers = torch.zeros((n_frames, T, 2, H, W), dtype=torch.float32, device=device)
    jj = torch.arange(W, device=device, dtype=torch.float32)[None, None, None, :]
    ii = torch.arange(H, device=device, dtype=torch.float32)[None, None, :, None]
    o = torch.arange(n_obj, device=device)
    base_x = ((o % gx).float() + 0.5) * W / gx
    base_y = ((o // gx).float() + 0.5) * H / gy

    def uniform(shape, lo, hi):
        return lo + (hi - lo) * torch.rand(shape, generator=gen, device=device)

    for f0 in range(0, n_frames, chunk):
        n = min(chunk, n_frames - f0)
        cx = base_x[None] + uniform((n, n_obj), -6.0, 6.0)
        cy = base_y[None] + uniform((n, n_obj), -6.0, 6.0)
        maps = [(0, cx, cy, None)]
        for t, count in enumerate(keypoint_config):
            start = uniform((n, n_obj), 0.0, 2.0 * np.pi)
            for k in range(count):
                angle = start + 2.0 * np.pi * k / count + uniform((n, n_obj), -0.3, 0.3)
                radius = uniform((n, n_obj), 6.0, 10.0)
                maps.append((1 + t, cx + radius * torch.cos(angle), cy + radius * torch.sin(angle), t))
        h = uniform((n, C, H, W), 0.0, NOISE_AMPLITUDE)
        for c, px, py, t in maps:
            amp = uniform((n, n_obj), 0.6, 1.0)
            z = uniform((n, n_obj), 0.4, 1.5)
            for ob in range(n_obj):
                x = px[:, ob, None, None, None]
                y = py[:, ob, None, None, None]
                d2 = (x - jj) ** 2 + (y - ii) ** 2
                h[:, c:c + 1] += amp[:, ob, None, None, None] * torch.exp(-d2 / LENGTH_SCALE ** 2)
                disc = ((x - (jj + 0.5)) ** 2 + (y - (ii + 0.5)) ** 2) < DISC_RADIUS ** 2
                dsl = depth[f0:f0 + n, c:c + 1]
                dsl[disc] = z[:, ob, None, None, None].expand_as(disc)[disc]
                if t is not None:
                    vx = (cx[:, ob, None, None, None] - (jj + 0.5)).expand_as(disc)
                    vy = (cy[:, ob, None, None, None] - (ii + 0.5)).expand_as(disc)
                    cxs = centers[f0:f0 + n, t:t + 1, 0]
                    cys = centers[f0:f0 + n, t:t + 1, 1]
                    cxs[disc] = vx[disc]
                    cys[disc] = vy[disc]
        heat[f0:f0 + n] = h.clamp_(0.0, 1.0)
    return heat, depth, centers, n_obj


# --------------------------------------------------------------------------------------------
# Stereo scenes: 3D objects in front of a rig, rasterised in both views (triangulate_stereo_objects).
# --------------------------------------------------------------------------------------------
def stereo_rig(prediction_size=(64, 64)):
    """The config/calibration.yaml rig (cam0 left, cam1 right) with both cameras scaled and cut as default_camera does."""
    import os
    from . import camera_utils
    p = camera_utils.load_calibration_params(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                          'config', 'calibration.yaml'))
    cameras = []
    for K, D in ((p['K'], p['D']), (p['Kp'], p['Dp'])):
        camera = camera_utils.FisheyeCamera(K, D, p['image_size'])
        if tuple(prediction_size) == (64, 64):
            scaled = camera.scale(511.0 / 720.0)
            camera = scaled.cut(np.array([(scaled.image_size[1] - 511.0) / 2.0, 0.0])).scale(64.0 / 511.0)
        else:
            camera = camera.scale(prediction_size[0] / 720.0)
        cameras.append(camera)
    return camera_utils.StereoCamera(cameras[0], cameras[1], p['T_RL'])


@dataclass
class StereoBatch:
    batch: Batch                 # 2P frames: the left view of pair p in row 2p, its right view in row 2p + 1
    points: list                 # per pair: [n_obj, 1 + sum(cfg), 3] left camera frame; centre, then types and slots in order
    right_of_left: list          # per pair: [n_obj], the right view's index of the left view's object i
    pixels: list                 # per pair: ([n_obj, 1 + sum(cfg), 2] left, [...] right) distorted pixels


def _epipolar_distance(F, left, right):
    """Mean of the two point-to-epipolar-line distances, as oracle/np_oracle.associate scores a pair (undistorted px)."""
    lx = F @ np.array([left[0], left[1], 1.0])
    ly = F.T @ np.array([right[0], right[1], 1.0])
    r = abs(right[0] * lx[0] + right[1] * lx[1] + lx[2])
    return 0.5 * (r / np.hypot(lx[0], lx[1]) + r / np.hypot(ly[0], ly[1]))


def stereo_batch(P, keypoint_config, size, stereo, seed, objects=(1, 4), depth_range=(0.5, 1.2), centre_margin=5.0, slot_margin=1.0,
                 center_separation=22.0, spoke_radius=(5.0, 8.0), peak_separation=6.0, border=4.0, max_tries=5000,
                 same_row=False, row_jitter=0.0, depth_scale=0.0):
    """P stereo pairs of one rig. Per pair: objects (a centre and keypoint_config[t] keypoints of every type t) are placed
    in front of the rig: pixels and depths are sampled in the left view under sample_scene's separations, lifted to 3D
    and projected into the right view with FisheyeCamera.project; the right view must keep the centres' separation too.
    Two different objects' centres stay farther than centre_margin from each other's epipolar line (no object is
    ambiguous at max_distance_px < centre_margin), and two different keypoints of one object and type farther than
    slot_margin (the construction's matching is the greedy one on noiseless keypoints). Each view is
    rasterised with `rasterize`, z taken in that view's camera frame; the objects of a view are listed in raster order of
    their centre pixel, the order in which the decode finds them.
    same_row: every object of a pair is moved vertically, with its keypoints, so that its centre lies in the row of the
    first object's centre in the left view, give or take a uniform row_jitter (pixels): parts side by side on a table,
    on one epipolar line of this rig. The centre_margin check is skipped then (slot_margin still applies), the left
    view must keep sample_scene's separations, and every keypoint's depth must be readable where the decode lifts it:
    DetectionToPoint reads the depth map at the undistorted pixel, which near the edges of a wide view lies off the disc
    drawn around the distorted one. depth_scale: each (frame, map) depth map is multiplied by its own factor,
    uniform in [1 - depth_scale, 1 + depth_scale] (a biased depth head); the ground truth is not. Both are off by
    default and then draw nothing, so the batches of other arguments do not change."""
    H, W = size
    cams = (stereo.left_camera, stereo.right_camera)
    T = (np.eye(4), stereo.T_RL)
    n_kp = 1 + sum(keypoint_config)
    heat = np.zeros((2 * P, len(keypoint_config) + 1, H, W), dtype=np.float32)
    depth = np.zeros_like(heat)
    centers = np.zeros((2 * P, len(keypoint_config), 2, H, W), dtype=np.float32)
    scenes, points, right_of_left, pixels = [], [], [], []
    lo, hi = np.array([border, border]), np.array([W - 1 - border, H - 1 - border])

    def inside(px):
        return bool((px >= lo).all() and (px <= hi).all())

    for p, child in enumerate(np.random.SeedSequence(seed).spawn(P)):
        rng = np.random.default_rng(child)
        n_obj = int(rng.integers(objects[0], objects[1] + 1))
        for _ in range(max_tries):
            left = sample_scene(rng, keypoint_config, size, n_obj, center_separation, spoke_radius, peak_separation, border)
            px_l = np.concatenate([left.centers[:, None]] + list(left.spokes), axis=1)        # [n_obj, n_kp, 2]
            if same_row:
                row = px_l[0, 0, 1] + rng.uniform(-row_jitter, row_jitter, size=n_obj)
                px_l[:, :, 1] += (row - px_l[:, 0, 1])[:, None]
                if not (all(inside(v) for v in px_l.reshape(-1, 2)) and
                        _separated(px_l, keypoint_config, center_separation, peak_separation)):
                    continue
            z = rng.uniform(*depth_range, size=n_obj)[:, None] + rng.uniform(-0.03, 0.03, size=(n_obj, n_kp))
            und = cams[0].undistort(px_l.reshape(-1, 2))
            X = (np.concatenate([und, np.ones((und.shape[0], 1))], axis=1) @ cams[0].Kinv.T) * z.reshape(-1, 1)
            views = [c.project(X, t).reshape(n_obj, n_kp, 2) for c, t in zip(cams, T)]
            if not all(inside(v) for v in views[1].reshape(-1, 2)):
                continue
            if not _far_enough_all(views[1][:, 0], center_separation):
                continue
            und_views = [c.undistort(v.reshape(-1, 2)).reshape(n_obj, n_kp, 2) for c, v in zip(cams, views)]
            if not _epipolar_unique(stereo.F, und_views, keypoint_config, -1.0 if same_row else centre_margin, slot_margin):
                continue
            if same_row and not all(_lift_on_disc(u, v) for u, v in zip(und_views, views)):
                continue
            break
        else:
            raise RuntimeError("could not place the requested objects; relax the separations")
        X = X.reshape(n_obj, n_kp, 3)
        orders = [np.lexsort((np.rint(v[:, 0, 0]), np.rint(v[:, 0, 1]))) for v in views]      # raster order of the centres
        for v, (camera_T, order) in enumerate(zip(T, orders)):
            Xc = X[order] @ camera_T[:3, :3].T + camera_T[:3, 3]
            px = views[v][order]
            spokes, zs, k = [], [], 1
            for count in keypoint_config:
                spokes.append(px[:, k:k + count].copy())
                zs.append(Xc[:, k:k + count, 2].copy())
                k += count
            scene = Scene(centers=px[:, 0].copy(), spokes=spokes,
                          amplitude_center=rng.uniform(0.6, 1.0, size=n_obj),
                          amplitude_spokes=[rng.uniform(0.6, 1.0, size=s.shape[:2]) for s in spokes],
                          z_center=Xc[:, 0, 2].copy(), z_spokes=zs)
            heat[2 * p + v], depth[2 * p + v], centers[2 * p + v] = rasterize(scene, keypoint_config, size, rng)
            scenes.append(scene)
        points.append(X[orders[0]])
        rank_right = np.empty(n_obj, np.int64)
        rank_right[orders[1]] = np.arange(n_obj)
        right_of_left.append(rank_right[orders[0]])
        pixels.append((views[0][orders[0]], views[1][orders[1]]))
    if depth_scale:
        scale = np.random.default_rng([seed, 1]).uniform(1.0 - depth_scale, 1.0 + depth_scale, size=depth.shape[:2])
        depth *= scale[:, :, None, None].astype(np.float32)
    batch = Batch(heat=heat, depth=depth, centers=centers, scenes=scenes, keypoint_config=list(keypoint_config))
    return StereoBatch(batch=batch, points=points, right_of_left=right_of_left, pixels=pixels)


def stereo_match_errors(sb, tables, result):
    """A stereo-objects result scored against the construction -> (wrong object matches, wrong slot matches, largest
    relative error of a correctly matched point). tables: the decode tables of sb.batch (n_objects, kp_count, kp_xy;
    NumPy), result: the StereoTables of the interleaved pairs (NumPy). Decoded objects and slots are identified with the
    construction's by their nearest pixel in each view: the decode lists objects in raster order of their peak pixel,
    which for objects in one row need not be the construction's order."""
    cfg = sb.batch.keypoint_config
    wrong_objects = wrong_slots = 0
    worst = 0.0
    groups = np.cumsum([0, 1] + list(cfg))

    def nearest(xy, pixels):
        return int(np.linalg.norm(pixels - xy[None], axis=-1).argmin())
    for p, (perm, X) in enumerate(zip(sb.right_of_left, sb.points)):
        px_l, px_r = sb.pixels[p]
        for i in range(int(tables['n_objects'][2 * p])):
            a = nearest(tables['kp_xy'][2 * p, i, 0, 0], px_l[:, 0])
            j = int(result['object_match'][p, i])
            if j < 0 or nearest(tables['kp_xy'][2 * p + 1, j, 0, 0], px_r[:, 0]) != perm[a]:
                wrong_objects += 1
                continue
            for c in range(len(cfg) + 1):
                k0, k1 = groups[c], groups[c + 1]
                for s in range(int(tables['kp_count'][2 * p, i, c])):
                    k = k0 + nearest(tables['kp_xy'][2 * p, i, c, s], px_l[a, k0:k1])
                    m = int(result['slot_match'][p, i, c, s])
                    if m < 0 or k0 + nearest(tables['kp_xy'][2 * p + 1, j, c, m], px_r[perm[a], k0:k1]) != k:
                        wrong_slots += 1
                        continue
                    error = np.linalg.norm(result['point'][p, i, c, s] - X[a, k]) / np.linalg.norm(X[a, k])
                    worst = max(worst, float(error))
    return wrong_objects, wrong_slots, worst


def _lift_on_disc(undistorted, distorted, radius=DISC_RADIUS - 0.5):
    """The pixel DetectionToPoint reads for every keypoint (the rounded undistorted position) lies inside the keypoint's
    depth disc (drawn around the distorted position, pixel centres at +0.5), with half a pixel to spare."""
    read = np.rint(undistorted.reshape(-1, 2)) + 0.5
    return bool((np.linalg.norm(read - distorted.reshape(-1, 2), axis=1) < radius).all())


def _separated(px, keypoint_config, center_separation, peak_separation):
    """sample_scene's separations on keypoints [n_obj, 1 + sum(cfg), 2]: centres, same-map peaks, and every spoke nearer
    to its own centre than to any other."""
    if not _far_enough_all(px[:, 0], center_separation):
        return False
    k = 1
    for count in keypoint_config:
        spokes = px[:, k:k + count]
        if not _far_enough_all(spokes.reshape(-1, 2), peak_separation):
            return False
        own = np.linalg.norm(spokes[:, :, None] - px[None, None, :, 0], axis=-1).argmin(axis=-1)     # [n_obj, count]
        if not (own == np.arange(len(px))[:, None]).all():
            return False
        k += count
    return True


def _far_enough_all(points, min_distance):
    return all(_far_enough(points[i], points[:i], min_distance) for i in range(len(points)))


def _epipolar_unique(F, und_views, keypoint_config, centre_margin, slot_margin):
    """No centre of one object within centre_margin of the epipolar line of another object's centre, no keypoint of an
    object within slot_margin of the line of another keypoint of the same object and type."""
    left, right = und_views
    n_obj = left.shape[0]
    groups = [[0]]
    k = 1
    for count in keypoint_config:
        groups.append(list(range(k, k + count)))
        k += count
    for i in range(n_obj):
        for j in range(n_obj):
            if i != j and _epipolar_distance(F, left[i, 0], right[j, 0]) <= centre_margin:
                return False
        for g in groups[1:]:
            for a in g:
                for b in g:
                    if a != b and _epipolar_distance(F, left[i, a], right[i, b]) <= slot_margin:
                        return False
    return True
