"""Parity tests proper: the CUDA path (through the C ABI) against (1) fixtures produced by the
unmodified reference, (2) the C oracle on fresh seeded inputs, (3) size-independent properties
at full benchmark sizes. Bit-exact: peak pixels, raster order, box sums, assignments, kept
keypoints, flags. Tolerance: sub-pixel <= 1e-3 px, 3D <= 1e-4 relative (BASELINE.json)."""
import numpy as np
import pytest

from helpers import (load_golden, golden_camera, reference_tables, assert_tables_match, TOL_PIXELS, TOL_METRES_REL)

pytestmark = pytest.mark.gpu
GENERIC_PATH = 128          # OKP_FLAG_GENERIC_PATH

DECODE_FIXTURES = ['valve_64.npz', 'cups_64.npz', 'valve_grid_180x320.npz', 'test_pipeline_180x320.npz',
                   'adversarial_64.npz', 'nan_64.npz']


def gpu_decode(heat, depth, centers, cfg, camera, **options):
    from object_keypoints_b200 import KeypointDecoder
    decoder = KeypointDecoder(cfg, heat.shape[2:], camera=camera, **options)
    return decoder.decode_batch(heat, depth, centers).numpy()


def assert_matches_oracle(got, want):
    """GPU vs C oracle on the same input: integer tables and flags identical; the oracle and the
    kernels share one arithmetic contract, so float32 tables are compared bitwise too; float64
    3D points within 1e-4 relative (CUDA's tan/atan are not the host libm's)."""
    for key in ['peak_count', 'peak_yx', 'peak_object', 'n_objects', 'kp_assigned', 'kp_count', 'kp_peak', 'n_votes']:
        np.testing.assert_array_equal(got[key], want[key], err_msg=key)
    # OKP_FLAG_GENERIC_PATH says which kernels ran, not what the data held: the oracle has no such bit
    np.testing.assert_array_equal(got['flags'] & ~np.uint32(GENERIC_PATH), want['flags'], err_msg='flags')
    for key in ['peak_score', 'peak_xy', 'peak_conf', 'kp_xy']:
        np.testing.assert_array_equal(got[key].view(np.uint32), want[key].view(np.uint32), err_msg=key + " (bitwise)")
    np.testing.assert_array_equal(got['peak_vote'], want['peak_vote'])
    np.testing.assert_array_equal(got['votes'], want['votes'])
    scale = np.maximum(np.linalg.norm(want['kp_point'], axis=-1), 1e-9)
    assert (np.linalg.norm(got['kp_point'] - want['kp_point'], axis=-1) <= TOL_METRES_REL * scale + 1e-12).all()


@pytest.mark.parametrize('name', DECODE_FIXTURES)
def test_cuda_matches_reference_fixture(name):
    g = load_golden(name)
    got = gpu_decode(g['heat'], g['depth'], g['centers'], list(g['keypoint_config']), golden_camera(g))
    assert_tables_match(got, reference_tables(g))


@pytest.mark.parametrize('single_pass', [False, True])
@pytest.mark.parametrize('name', DECODE_FIXTURES)
def test_cuda_matches_oracle_on_fixture_inputs(name, single_pass):
    from oracle import c_oracle
    g = load_golden(name)
    cfg, camera = list(g['keypoint_config']), golden_camera(g)
    got = gpu_decode(g['heat'], g['depth'], g['centers'], cfg, camera, single_pass=single_pass)
    assert_matches_oracle(got, c_oracle.decode(g['heat'], g['depth'], g['centers'], cfg, camera))


@pytest.mark.parametrize('cfg,size,frames,objects', [
    ([1, 3], (64, 64), 96, (1, 2)),          # config 1/4 shape: valve at the model resolution
    ([1, 1, 1], (64, 64), 128, (1, 4)),      # config 2: cups, 64 stereo pairs
    ([1, 3], (180, 320), 12, (1, 6)),        # test_pipeline shape
    ([2], (40, 56), 8, (1, 1)),              # odd sizes, ragged tiles
    ([1, 3], (37, 93), 8, (1, 1)),           # sizes that are not multiples of anything
])
@pytest.mark.parametrize('single_pass', [False, True])
def test_cuda_matches_oracle_on_seeded_batches(cfg, size, frames, objects, single_pass):
    from oracle import c_oracle
    from object_keypoints_b200 import synthetic
    layout = {}
    if size[0] < 64:
        layout = dict(center_separation=18.0, spoke_radius=(4.0, 6.0), peak_separation=5.0, border=3.0)
    batch = synthetic.make_batch(frames, cfg, size, seed=2000 + size[0], objects=objects, **layout)
    camera = synthetic.default_camera((64, 64)) if size == (64, 64) else \
        synthetic.default_camera((180, 320)) if size == (180, 320) else \
        __import__('object_keypoints_b200').camera_utils.FisheyeCamera(
            np.array([[50.0, 0, size[1] / 2], [0, 50.0, size[0] / 2], [0, 0, 1]]), np.array([0.1, 0.01, -0.02, 0.003]), size)
    got = gpu_decode(batch.heat, batch.depth, batch.centers, cfg, camera, single_pass=single_pass)
    assert_matches_oracle(got, c_oracle.decode(batch.heat, batch.depth, batch.centers, cfg, camera))
    assert got['n_objects'].sum() > 0


def test_empty_batch_and_single_map():
    from object_keypoints_b200 import KeypointDecoder, synthetic
    from oracle import c_oracle
    camera = synthetic.default_camera((64, 64))
    decoder = KeypointDecoder([1, 3], (64, 64), camera=camera)
    empty = decoder.decode_batch(np.zeros((0, 3, 64, 64), np.float32), np.zeros((0, 3, 64, 64), np.float32),
                                 np.zeros((0, 2, 2, 64, 64), np.float32)).numpy()
    assert empty['n_objects'].shape == (0,)
    # C = 1: only the centre map, no spokes
    batch = synthetic.make_batch(4, [], (64, 64), seed=9, objects=(1, 3))
    got = gpu_decode(batch.heat, batch.depth, batch.centers, [], camera)
    assert_matches_oracle(got, c_oracle.decode(batch.heat, batch.depth, batch.centers, [], camera))


def test_capacity_overflow_keeps_first_peaks_in_raster_order():
    """Random-init network output (config 5): ~0.5 everywhere, dozens of noise peaks per map. The
    table keeps the first max_peaks in raster order and raises the overflow flags."""
    from oracle import c_oracle, np_oracle
    from object_keypoints_b200 import synthetic
    rng = np.random.default_rng(5)
    heat = (0.5 + 0.002 * rng.standard_normal((3, 3, 64, 64))).astype(np.float32)
    depth = np.ones_like(heat)
    centers = rng.normal(0, 3, (3, 2, 2, 64, 64)).astype(np.float32)
    camera = synthetic.default_camera((64, 64))
    options = dict(max_peaks=16, max_objects=8, max_votes=4)
    got = gpu_decode(heat, depth, centers, [1, 3], camera, **options)
    want = c_oracle.decode(heat, depth, centers, [1, 3], camera, **options)
    assert (want['peak_count'] > 16).all()
    assert (got['flags'] & np_oracle.FLAG_PEAK_OVERFLOW).all() and (got['flags'] & np_oracle.FLAG_OBJECT_OVERFLOW).all()
    assert_matches_oracle(got, want)
    # and with room for everything the clustering branch (cfg > 1 overflow) is exercised identically
    options = dict(max_peaks=128, max_objects=128, max_votes=16)
    got = gpu_decode(heat, depth, centers, [1, 3], camera, **options)
    want = c_oracle.decode(heat, depth, centers, [1, 3], camera, **options)
    assert (got['flags'] & np_oracle.FLAG_CLUSTERED).any()
    for key in ['peak_count', 'peak_yx', 'peak_object', 'n_objects', 'flags', 'kp_assigned', 'kp_count', 'kp_peak']:
        np.testing.assert_array_equal(got[key], want[key], err_msg=key)
    assert np.abs(got['kp_xy'] - want['kp_xy']).max() <= TOL_PIXELS


def test_non_square_clip_rule_and_its_switch():
    """pipeline.py:162,169 clips x with H-1: at 180x320 a keypoint at x = 250 reads depth column 179."""
    from oracle import c_oracle
    from object_keypoints_b200 import synthetic
    H, W = 180, 320
    heat = np.zeros((1, 2, H, W), np.float32)
    jj, ii = np.arange(W)[None, :], np.arange(H)[:, None]
    for c, (x, y) in enumerate([(250.0, 90.0), (256.0, 92.0)]):
        heat[0, c] = np.exp(-((x - jj) ** 2 + (y - ii) ** 2) / 4.0)
    depth = np.tile(np.arange(W, dtype=np.float32)[None, None, None, :] / 100.0 + 0.5, (1, 2, H, 1))
    centers = np.zeros((1, 1, 2, H, W), np.float32)
    centers[0, 0, 0] = 250.0 - (jj + 0.5)
    centers[0, 0, 1] = 90.0 - (ii + 0.5)
    camera = synthetic.default_camera((H, W))
    for bug in (True, False):
        got = gpu_decode(heat, depth, centers, [1], camera, compat_clip_bug=bug)
        want = c_oracle.decode(heat, depth, centers, [1], camera, compat_clip_bug=bug)
        assert_matches_oracle(got, want)
        z = got['kp_point'][0, 0, 0, 0, 2]
        assert abs(z - (1.79 + 0.5 if bug else depth[0, 0, 90, int(round(got['kp_point'][0, 0, 0, 0, 0] / z * camera.K[0, 0] + camera.K[0, 2]))])) < 1e-5


def test_full_size_batch_properties():
    """BASELINE config 4 size (4096 frames) is too big for the oracle in a test: check invariants
    instead -- every frame finds its 8 objects with complete keypoint sets, results do not depend on
    batch composition (decode of a sub-batch is identical), and repeated runs are deterministic."""
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic
    N = 4096
    heat, depth, centers, n_obj = synthetic.torch_grid_batch(N, [1, 3], (64, 128), seed=3, grid=(4, 2), device='cuda')
    camera = synthetic.default_camera((180, 320))
    decoder = KeypointDecoder([1, 3], (64, 128), camera=camera)
    t = decoder.decode_batch(heat, depth, centers)
    full = {k: v.clone() for k, v in t.tensors.items()}
    assert (full['n_objects'] == n_obj).float().mean() > 0.99
    ok = full['n_objects'] == n_obj
    assert (full['kp_count'][ok][:, :n_obj].sum(dim=(1, 2)) == n_obj * 5).float().mean() > 0.95
    # sub-batch independence and determinism
    sub = slice(1000, 1064)
    t2 = KeypointDecoder([1, 3], (64, 128), camera=camera).decode_batch(heat[sub], depth[sub], centers[sub])
    for key in full:
        assert torch.equal(t2[key], full[key][sub]), key
    t3 = decoder.decode_batch(heat, depth, centers)
    for key in full:
        a, b = t3[key], full[key]
        assert torch.equal(a, b) or (a.dtype.is_floating_point and torch.equal(a.isnan(), b.isnan())), key


def test_reference_style_api_returns_reference_structures():
    """ObjectKeypointPipeline(prediction_size, points_3d, keypoint_config).reset(camera)(heat, depth, centers)
    -> list of dicts with 'p_centers', 'keypoints', 'p_C' shaped like pipeline.py:195-199."""
    import torch
    from object_keypoints_b200 import ObjectKeypointPipeline
    g = load_golden('valve_64.npz')
    ref = reference_tables(g)
    pipeline = ObjectKeypointPipeline([64, 64], None, {'keypoint_config': [1, 3]})
    pipeline.reset(golden_camera(g))
    with pytest.raises(AssertionError):
        pipeline(torch.tensor(g['heat'][:2]), torch.tensor(g['depth'][:2]), torch.tensor(g['centers'][:2]))
    for n in range(4):
        objects = pipeline(torch.tensor(g['heat'][n:n + 1]), torch.tensor(g['depth'][n:n + 1]),
                           torch.tensor(g['centers'][n:n + 1]))
        assert len(objects) == ref['n_objects'][n]
        for o, obj in enumerate(objects):
            assert set(obj) == {'p_centers', 'keypoints', 'p_C'}
            assert len(obj['keypoints']) == 3 and len(obj['p_C']) == 3
            assert obj['keypoints'][0].shape == (1, 2) and obj['keypoints'][0].dtype == np.float32
            assert obj['p_C'][0].shape == (1, 3) and obj['p_C'][0].dtype == np.float64
            for c in range(3):
                cnt = ref['kp_count'][n, o, c]
                assert obj['keypoints'][c].shape[0] == cnt
                assert np.abs(obj['keypoints'][c] - ref['kp_xy'][n, o, c, :cnt]).max() <= TOL_PIXELS
                want = ref['kp_point'][n, o, c, :cnt]
                assert np.abs(obj['p_C'][c] - want).max() <= TOL_METRES_REL * np.abs(want).max()
            assert len(obj['p_centers']) == ref['n_votes'][n, o]


def test_component_level_api():
    from object_keypoints_b200 import KeypointExtractionComponent, ObjectExtraction, DetectionToPoint
    from oracle import c_oracle
    g = load_golden('cups_64.npz')
    ref = reference_tables(g)
    cfg = {'keypoint_config': [1, 1, 1]}
    extraction = KeypointExtractionComponent(cfg, [64, 64])
    keypoints, confidence = extraction(g['heat'][:3])
    assert len(keypoints) == 3 and len(keypoints[0]) == 4
    for n in range(3):
        for c in range(4):
            k = ref['peak_count'][n, c]
            assert len(keypoints[n][c]) == k
            for j in range(k):
                assert np.abs(keypoints[n][c][j] - ref['peak_xy'][n, c, j]).max() <= TOL_PIXELS
                assert abs(float(confidence[n][c][j]) - ref['peak_conf'][n, c, j]) <= 1e-5 * ref['peak_conf'][n, c, j]
    grouping = ObjectExtraction(cfg, [64, 64])
    objects = grouping(keypoints[0], confidence[0], g['centers'][0])
    assert len(objects) == ref['n_objects'][0]
    for o, obj in enumerate(objects):
        assert set(obj) >= {'center', 'heatmap_points', 'p_centers'}
        assert np.abs(obj['center'] - ref['kp_xy'][0, o, 0, 0]).max() <= TOL_PIXELS
        for c in range(1, 4):
            cnt = ref['kp_count'][0, o, c]
            assert np.asarray(obj['heatmap_points'][c - 1]).reshape(-1, 2).shape[0] == cnt
    assert ObjectExtraction(cfg, [64, 64])([[], [], [], []], [[], [], [], []], g['centers'][0]) == []
    to_point = DetectionToPoint()
    camera = golden_camera(g)
    to_point.reset(camera)
    assert to_point(np.zeros((0, 2)), g['depth'][0, 0]) is None
    xy = ref['kp_xy'][0, 0, 1, :1]
    got = to_point(xy, g['depth'][0, 1])
    want = c_oracle.detection_to_point(xy, g['depth'][0, 1], camera)
    assert np.abs(got - want).max() <= TOL_METRES_REL * np.abs(want).max()


def assert_peaks_match_oracle(got, want):
    """Peak tables of extract_peaks against the oracle's decode of the same maps: counts and pixels identical, float32
    columns bitwise, and no assignment (extract_peaks groups nothing)."""
    np.testing.assert_array_equal(got['peak_count'], want['peak_count'])
    np.testing.assert_array_equal(got['peak_yx'], want['peak_yx'])
    for key in ['peak_score', 'peak_xy', 'peak_conf']:
        np.testing.assert_array_equal(got[key].view(np.uint32), want[key].view(np.uint32), err_msg=key)
    assert (got['peak_object'] == -1).all()


@pytest.mark.parametrize('H,W,N,C,K', [
    (64, 64, 37, 3, 32),       # maps not a multiple of the maps-per-CTA group
    (3, 4, 5, 2, 8),           # tiny map: every window is clipped
    (1, 8, 3, 1, 8),
    (7, 252, 3, 2, 64),        # widest single TMA box
    (9, 256, 2, 3, 64),        # narrowest two-box row
    (33, 320, 2, 3, 16),       # two boxes, K small: most maps overflow -> overflow path
    (12, 504, 2, 2, 256),      # widest supported row
    (21, 508, 1, 2, 64),       # too wide for the strip kernel -> generic kernel
    (30, 66, 2, 2, 32),        # W % 4 != 0 -> generic kernel
])
def test_peak_extraction_shapes_noise_and_overflow(H, W, N, C, K):
    """Dense random maps (a peak every ~25 pixels, ties included through quantised values): the peak
    tables of the strip kernel / overflow path / generic kernel are bitwise the oracle's."""
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder
    rng = np.random.default_rng(H * 1000 + W)
    heat = rng.uniform(0, 0.2, (N, C, H, W)).astype(np.float32)
    heat[0, 0] = np.round(heat[0, 0] * 8) / 8                    # exact ties
    if N > 1:
        heat[1, C - 1] = 0.001                                    # below threshold everywhere: no peaks
    cfg = [1] * (C - 1)
    decoder = KeypointDecoder(cfg, (H, W), max_peaks=K, max_objects=16)
    got = decoder.extract_peaks(heat).numpy()
    want = c_oracle.decode(heat, np.zeros_like(heat), np.zeros((N, C - 1, 2, H, W), np.float32), cfg, None,
                           max_peaks=K, max_objects=16)
    assert_peaks_match_oracle(got, want)
    if (H, W) == (33, 320):                                       # both the overflow path and the fast path
        assert (want['peak_count'] > K).any() and (want['peak_count'] <= K).any()


def test_candidate_filter_adversarial_inputs_are_bitwise_the_oracle():
    """Inputs chosen against the strip kernel's bounded filter (okp_peaks_strip.cuh): exact ties,
    1-ulp tie breaks, a saturated plateau, random-init-network maps (every pixel above threshold),
    denormal sums, border windows, and maps with negative values (bound void -> exact generic path)."""
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder
    from test_filter_bound import cases
    rng = np.random.default_rng(7)
    for name, p in sorted(cases().items()):
        H, W = p.shape
        if W % 4:
            continue
        threshold = 0.0 if name == 'tiny_values' else 0.5
        negative = p.copy()
        negative[H // 2, W // 2] = -0.25                              # one negative pixel in an otherwise equal map
        mixed = rng.uniform(-0.1, 0.3, p.shape).astype(np.float32)
        heat = np.stack([p, negative, mixed, p[::-1].copy()])[None]    # [1, 4, H, W]
        heat = np.concatenate([heat, heat[:, ::-1]], axis=0)           # 2 frames, maps in a different CTA slot
        cfg = [1, 1, 1]
        K = 128
        decoder = KeypointDecoder(cfg, (H, W), max_peaks=K, max_objects=16, threshold=threshold)
        got = decoder.extract_peaks(heat).numpy()
        want = c_oracle.decode(heat, np.zeros_like(heat), np.zeros((2, 3, 2, H, W), np.float32), cfg, None,
                               max_peaks=K, max_objects=16, threshold=threshold)
        np.testing.assert_array_equal(got['peak_count'], want['peak_count'], err_msg=name)
        np.testing.assert_array_equal(got['peak_yx'], want['peak_yx'], err_msg=name)
        for key in ['peak_score', 'peak_xy', 'peak_conf']:
            np.testing.assert_array_equal(got[key].view(np.uint32), want[key].view(np.uint32), err_msg=f"{name} {key}")


def test_host_batch_in_place_gather_equals_device_decode():
    """decode_host_batch: pinned depth / centre maps are gathered in place over PCIe (okp_host_alias),
    pageable ones are copied; both give the tables of the all-device decode, ragged last chunk included."""
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic
    cfg = [1, 3]
    batch = synthetic.make_batch(37, cfg, (64, 64), seed=11, objects=(1, 3))
    camera = synthetic.default_camera((64, 64))
    decoder = KeypointDecoder(cfg, (64, 64), camera=camera)
    want = decoder.decode_batch(batch.heat, batch.depth, batch.centers).numpy()
    host = [torch.from_numpy(a) for a in (batch.heat, batch.depth, batch.centers)]
    pinned = [t.pin_memory() for t in host]
    assert decoder._host_alias(pinned[1]) is not None, "pinned host memory must be device-accessible on this box"
    assert decoder._host_alias(host[1]) is None
    for inputs, copied_maps in ((pinned, 1), (host, 3)):
        got = decoder.decode_host_batch(*inputs, chunk_frames=16, sparse=False)
        for name in KeypointDecoder.HOST_RESULT_TABLES:
            np.testing.assert_array_equal(got[name].numpy().view(np.uint8), want[name].view(np.uint8), err_msg=name)
        if copied_maps == 1:
            assert decoder.host_bytes_copied == batch.heat.nbytes
        else:
            assert decoder.host_bytes_copied == batch.heat.nbytes + batch.depth.nbytes + batch.centers.nbytes


def _bf16_round(a):
    """float32 array -> (torch bf16 CUDA tensor, the same values as float32 NumPy) -- what a bf16 head emits."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda().to(torch.bfloat16)
    return t, t.float().cpu().numpy()


@pytest.mark.parametrize('cfg,size,frames,objects', [
    ([1, 3], (64, 64), 96, (1, 2)),          # config 5 shape: the network's output resolution
    ([1, 1, 1], (64, 64), 64, (1, 4)),
    ([1, 3], (180, 320), 12, (1, 6)),        # two TMA boxes per row, second box with a 4-element lead
    ([2], (40, 56), 8, (1, 1)),              # W % 8 == 0, single box
    ([1, 3], (36, 92), 6, (1, 1)),           # W % 8 != 0: no bf16 tensor map -> generic kernels
])
def test_bf16_maps_decode_like_the_upcast_float32_maps(cfg, size, frames, objects):
    """okp_decode_bf16 (BASELINE config 5: bf16 head outputs stay on the device): bf16 -> f32 is exact,
    so the tables must be bitwise those of the C oracle run on the up-cast maps."""
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder, synthetic
    layout = {}
    if size[0] < 64:
        layout = dict(center_separation=18.0, spoke_radius=(4.0, 6.0), peak_separation=5.0, border=3.0)
    batch = synthetic.make_batch(frames, cfg, size, seed=3000 + size[1], objects=objects, **layout)
    camera = synthetic.default_camera(size) if size in ((64, 64), (180, 320)) else \
        __import__('object_keypoints_b200').camera_utils.FisheyeCamera(
            np.array([[50.0, 0, size[1] / 2], [0, 50.0, size[0] / 2], [0, 0, 1]]), np.array([0.1, 0.01, -0.02, 0.003]), size)
    (heat, heat32), (depth, depth32), (centers, centers32) = (_bf16_round(a) for a in (batch.heat, batch.depth, batch.centers))
    decoder = KeypointDecoder(cfg, size, camera=camera)
    got = decoder.decode_batch(heat, depth, centers).numpy()
    assert_matches_oracle(got, c_oracle.decode(heat32, depth32, centers32, cfg, camera))
    assert got['n_objects'].sum() > 0
    # mixed: bf16 heatmaps with float32 depth / centre maps (extract and group entries of different types)
    import torch
    got = decoder.decode_batch(heat, torch.from_numpy(batch.depth).cuda(), torch.from_numpy(batch.centers).cuda()).numpy()
    assert_matches_oracle(got, c_oracle.decode(heat32, batch.depth, batch.centers, cfg, camera))


@pytest.mark.parametrize('H,W,N,C,K', [
    (64, 64, 37, 3, 32),
    (3, 8, 5, 2, 8),
    (7, 240, 3, 2, 64),        # widest single bf16 box (4 * 61 + 4 + 4 = 252 -> 256 columns)
    (9, 248, 2, 3, 64),        # narrowest two-box bf16 row
    (33, 320, 2, 3, 16),       # K small: most maps overflow -> overflow path (bf16 generic tiles)
    (12, 488, 2, 2, 256),      # widest bf16 row the strip kernel takes (two boxes of 256 columns)
    (11, 496, 1, 2, 64),       # wider: generic kernel
    (30, 68, 2, 2, 32),        # W % 8 != 0 -> generic kernel
])
def test_bf16_peak_extraction_shapes_noise_and_overflow(H, W, N, C, K):
    """Dense random bf16 maps (bf16 quantisation makes exact ties common): strip kernel, overflow path and
    generic kernel give bitwise the oracle's peak tables on the up-cast maps; also maps with a negative
    value (-0.0 included), which void the bounded filter and take the exact path."""
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder
    rng = np.random.default_rng(H * 1000 + W + 1)
    heat = rng.uniform(0, 0.2, (N, C, H, W)).astype(np.float32)
    heat[0, 0, H // 2, W // 2] = -0.0
    if N > 1:
        heat[1, C - 1] = 0.001
        heat[1, 0, 0, 0] = -0.125
    heat_dev, heat32 = _bf16_round(heat)
    cfg = [1] * (C - 1)
    decoder = KeypointDecoder(cfg, (H, W), max_peaks=K, max_objects=16)
    got = decoder.extract_peaks(heat_dev).numpy()
    want = c_oracle.decode(heat32, np.zeros_like(heat32), np.zeros((N, C - 1, 2, H, W), np.float32), cfg, None,
                           max_peaks=K, max_objects=16)
    np.testing.assert_array_equal(got['peak_count'], want['peak_count'])
    np.testing.assert_array_equal(got['peak_yx'], want['peak_yx'])
    for key in ['peak_score', 'peak_xy', 'peak_conf']:
        np.testing.assert_array_equal(got[key].view(np.uint32), want[key].view(np.uint32), err_msg=key)


def test_record_pack_kernel_equals_the_torch_packing():
    """okp_pack_records_f64 (the dense float64 record of the tables) against sharding.record_tensor, on the tables of a
    real decode."""
    import ctypes
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic, sharding, _lib
    cfg = [1, 3]
    batch = synthetic.make_batch(21, cfg, (64, 64), seed=17, objects=(1, 3))
    decoder = KeypointDecoder(cfg, (64, 64), camera=synthetic.default_camera((64, 64)))
    tables = decoder.decode_batch(batch.heat, batch.depth, batch.centers)
    R = _lib.lib().okp_record_doubles(16, 3, 3)
    assert R == 2 + 16 * 3 + 16 * 3 * 3 * 3
    want = sharding.record_tensor(tables)
    got = torch.zeros((21 + 4, R), dtype=torch.float64, device='cuda')
    destinations = (ctypes.c_void_p * 1)(got.data_ptr())
    rc = _lib.lib().okp_pack_records_f64(ctypes.byref(tables.struct), 21, 16, 3, 3, 4, destinations, 1, None)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(got[4:], want) and not got[:4].any()
    back = sharding.unpack_records(got[4:], tables)
    assert torch.equal(back['kp_point'], tables['kp_point']) and torch.equal(back['n_objects'], tables['n_objects'])


@pytest.mark.parametrize('cfg,size,lean', [([1, 3], (64, 64), False), ([1, 3], (64, 64), True), ([1, 1, 1], (64, 64), False),
                                           ([1, 3], (37, 93), False)])
@pytest.mark.parametrize('single_pass', [False, True])
def test_compact_records_emitted_by_the_decode_kernel(cfg, size, lean, single_pass):
    """okp_decode_emit_*: the record every frame's grouping writes into the sink (the multi-GPU gather's payload) equals
    the torch packing of the tables -- fused kernel (64x64), generic path + stand-alone grouping (37x93), frames that
    take the overflow fix-up, several steps through the slot ring of sharding.RecordExchange (world 1: 'local')."""
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic, sharding
    layout = dict(center_separation=18.0, spoke_radius=(4.0, 6.0), peak_separation=5.0, border=3.0) if size[0] < 64 else {}
    batch = synthetic.make_batch(23, cfg, size, seed=19, objects=(1, 3), **layout)
    heat = batch.heat.copy()
    heat[3, 1] = 0.5                                                   # a map with more than K peaks: overflow fix-up
    heat[5, 0, 10, 10] = -0.25                                         # a negative value: exact path for that map
    heat[7, 0] = 0.0                                                   # no centres
    camera = synthetic.default_camera((64, 64))
    decoder = KeypointDecoder(cfg, size, camera=camera, lean_tables=lean, single_pass=single_pass)
    exchange = sharding.RecordExchange(decoder, 23, world=1, rank=0)
    assert exchange.transport == 'local' and exchange.record_bytes == sharding.compact_layout(16, cfg)['record_bytes']
    tables = decoder.tables(23)
    for step in range(6):
        sink = exchange.begin()
        decoder.decode_batch(heat, batch.depth, batch.centers, tables=tables, records=sink)
        got, done = exchange.end()
        done.synchronize()
        back = sharding.unpack_compact_records(got, 16, cfg)
        for key in ('n_objects', 'kp_count', 'kp_point'):
            want = tables[key]
            if key == 'kp_count':
                want = torch.where(torch.arange(16, device='cuda')[None, :, None] < tables['n_objects'][:, None, None], want, 0)
            if key == 'kp_point':
                slot = torch.arange(want.shape[3], device='cuda')[None, None, None, :] < back['kp_count'][..., None]
                want = torch.where(slot[..., None], want, 0.0)
            assert torch.equal(back[key], want.to(back[key].dtype)), (step, key)
        assert torch.equal(back['flags'], tables['flags'].to(torch.int32))
        if step == 0:
            assert (tables['flags'][3] & 1) and int(tables['n_objects'][7]) == 0
            want_bytes = sharding.pack_compact_records(tables, cfg)
            fresh = torch.equal(got, want_bytes)                      # the buffers start zeroed: byte-identical the first time
            assert fresh, "record bytes differ from the torch packing"


def test_lean_tables_write_only_the_valid_slots():
    """OkpDecodeParams.lean_tables: the valid slots are bitwise those of the default mode; everything else keeps what
    the buffer held (here: the poison written before the call)."""
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic, _abi
    from oracle import c_oracle
    cfg = [1, 3]
    camera = synthetic.default_camera((64, 64))
    for size, frames in (((64, 64), 40), ((180, 320), 6), ((37, 93), 5)):
        layout = dict(center_separation=18.0, spoke_radius=(4.0, 6.0), peak_separation=5.0, border=3.0) if size[0] < 64 else {}
        batch = synthetic.make_batch(frames, cfg, size, seed=23, objects=(1, 3), **layout)
        heat = batch.heat.copy()
        heat[1, 2] = 0.5                                               # overflow map
        heat[2, 0] = 0.0                                               # no centres
        cam = synthetic.default_camera(size) if size != (37, 93) else camera
        want = c_oracle.decode(heat, batch.depth, batch.centers, cfg, cam)
        lean = KeypointDecoder(cfg, size, camera=cam, lean_tables=True)
        tables = lean.tables(frames)
        tables.flat.fill_(0x5A)                                        # poison
        got = lean.decode_batch(heat, batch.depth, batch.centers, tables=tables).numpy()
        assert_matches_oracle(_abi.mask_unspecified(got), want)
        if size == (64, 64):                                           # and the poison is still there where nothing is valid
            assert (got['votes'][2].view(np.uint8) == 0x5A).all() and (got['kp_point'][2].view(np.uint8) == 0x5A).all()
            assert (got['peak_xy'][0, 0, 8:].view(np.uint8) == 0x5A).all()


def test_generic_path_flag_tells_the_caller_the_shape_fell_off_the_tma_kernel():
    from object_keypoints_b200 import KeypointDecoder, synthetic
    camera = synthetic.default_camera((64, 64))
    layout = dict(center_separation=18.0, spoke_radius=(4.0, 6.0), peak_separation=5.0, border=3.0)
    for size, options, generic in (((64, 64), {}, False), ((37, 93), {}, True), ((40, 56), {}, False),
                                   ((64, 64), dict(nms_size=3), True), ((64, 64), dict(box_sum=False), True),
                                   ((64, 64), dict(top_k=4), False)):
        batch = synthetic.make_batch(5, [1, 3], size, seed=29, objects=(1, 2), **(layout if size[0] < 64 else {}))
        decoder = KeypointDecoder([1, 3], size, camera=camera, **options)
        tables = decoder.tables(5)
        tables['flags'].fill_(GENERIC_PATH if not generic else 0)      # a stale bit must not survive, a missing one must appear
        flags = decoder.decode_batch(batch.heat, batch.depth, batch.centers, tables=tables).numpy()['flags']
        assert bool((flags & GENERIC_PATH).all()) == generic and bool((flags & GENERIC_PATH).any()) == generic, (size, options)


def test_nan_maps_follow_torch_max_pool():
    """torch's max_pool2d propagates NaN: no pixel whose 5x5 window holds a NaN box sum is a peak (fixture made with the
    unmodified reference). The stream kernel sees the NaN in its bit test and hands the map to the exact kernels."""
    from oracle import c_oracle
    g = load_golden('nan_64.npz')
    cfg, camera = list(g['keypoint_config']), golden_camera(g)
    got = gpu_decode(g['heat'], g['depth'], g['centers'], cfg, camera)
    ref = reference_tables(g)
    np.testing.assert_array_equal(got['peak_count'], ref['peak_count'])
    np.testing.assert_array_equal(got['peak_yx'], ref['peak_yx'])
    np.testing.assert_array_equal(got['n_objects'], ref['n_objects'])
    assert_matches_oracle(got, c_oracle.decode(g['heat'], g['depth'], g['centers'], cfg, camera))


def test_unaligned_views_and_wrong_host_shapes():
    """A heatmap view whose base is not 16-byte aligned is re-materialised (the C entry refuses it); decode_host_batch
    validates shapes instead of reading out of bounds; every call returns its own result tensors."""
    import ctypes
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic, _lib
    cfg = [1]
    size = (5, 12)                                                     # 2 maps x 60 floats per frame: frame 1 starts at byte 480, frame stride 480
    camera = synthetic.default_camera((64, 64))
    rng = np.random.default_rng(3)
    heat = torch.from_numpy(rng.uniform(0, 0.2, (6, 2, 5, 12)).astype(np.float32)).cuda()
    flat = torch.zeros(heat.numel() + 1, device='cuda')
    flat[1:] = heat.reshape(-1)
    view = flat[1:].reshape(heat.shape)                                # base + 4 bytes
    assert view.data_ptr() % 16 == 4
    decoder = KeypointDecoder(cfg, size, camera=camera)
    a = decoder.extract_peaks(view).numpy()
    b = decoder.extract_peaks(heat).numpy()
    for key in ('peak_count', 'peak_yx', 'peak_score'):
        np.testing.assert_array_equal(a[key], b[key])
    ws = decoder._workspace_for(6)
    rc = _lib.lib().okp_extract_peaks_f32(view.data_ptr(), 6, 2, 5, 12, ctypes.byref(decoder.params),
                                          ctypes.byref(decoder.tables(6).struct), ws.data_ptr(), ws.numel(), None)
    assert rc == -4                                                    # OKP_E_UNSUPPORTED, not a silent slow path
    batch = synthetic.make_batch(9, [1, 3], (64, 64), seed=31, objects=(1, 2))
    dec = KeypointDecoder([1, 3], (64, 64), camera=camera)
    host = [torch.from_numpy(x).pin_memory() for x in (batch.heat, batch.depth, batch.centers)]
    with pytest.raises(ValueError):
        dec.decode_host_batch(host[0], host[1][:, :2], host[2])
    with pytest.raises(ValueError):
        dec.decode_host_batch(host[0], host[1], host[2][:4])
    with pytest.raises(ValueError):
        dec.decode_host_batch(host[0][:, :2], host[1], host[2])
    r1 = dec.decode_host_batch(*host, chunk_frames=4, sparse=False)
    r2 = dec.decode_host_batch(host[0] * 0, host[1], host[2], chunk_frames=4, sparse=False)
    assert r1 is not r2 and int(r1['n_objects'].sum()) > 0 and int(r2['n_objects'].sum()) == 0
    r3 = dec.decode_host_batch(*host, chunk_frames=4, sparse=False, out=r2)
    assert r3 is r2 and torch.equal(r3['kp_point'], r1['kp_point'])
    for chunk in (1, 2, 3, 5):                                         # staging sets are bounded
        dec.decode_host_batch(*host, chunk_frames=chunk, sparse=False)
    assert len([k for k in dec._tables if isinstance(k, tuple)]) <= dec.HOST_STAGING_SETS


def test_sparse_host_transfer_gives_the_tables_of_the_dense_copy():
    """decode_host_batch(sparse='auto'): only the tiles within reach of a value above threshold / 25 cross PCIe
    (okp_host_pack_tiles_f32 + okp_scatter_tiles_f32); tables must be bitwise those of the dense copy -- clean frames,
    the adversarial maps (plateaus, ties, borders, negative values) and dense maps (fallback to the dense copy)."""
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic
    from test_filter_bound import cases
    cfg = [1, 3]
    camera = synthetic.default_camera((64, 64))
    batch = synthetic.make_batch(41, cfg, (64, 64), seed=13, objects=(1, 3))
    heat = batch.heat.copy()
    heat[5] = 0.5                                                        # a dense frame inside a sparse chunk
    heat[7, 1, 30:34, 30:34] = np.nan
    heat[9, 2, 10, 10] = -0.3
    adversarial = [p for p in cases().values() if p.shape == (64, 64)]
    for i, p in enumerate(adversarial[:12]):
        heat[20 + i, i % 3] = p
    decoder = KeypointDecoder(cfg, (64, 64), camera=camera, max_peaks=64)
    decoder.SPARSE_CAPACITY = 1.0                                        # 64x64 blobs mark most 4x16 tiles: pack them anyway
    decoder.SPARSE_MIN_THREADS = 1                                       # whatever the box's core count
    host = [torch.from_numpy(a).pin_memory() for a in (heat, batch.depth, batch.centers)]
    dense = decoder.decode_host_batch(*host, chunk_frames=8, sparse=False)
    dense = {k: v.clone() for k, v in dense.items()}
    dense_bytes = decoder.host_bytes_copied
    for mode, least in (('only', 6), ('auto', 1)):                       # every chunk packed / packed and dense side by side
        sparse = decoder.decode_host_batch(*host, chunk_frames=8, sparse=mode)
        assert decoder.host_chunks_sparse >= least and decoder.host_bytes_copied < dense_bytes
        for name in KeypointDecoder.HOST_RESULT_TABLES:
            np.testing.assert_array_equal(sparse[name].numpy().view(np.uint8), dense[name].numpy().view(np.uint8), err_msg=name)
    decoder.SPARSE_CAPACITY = 0.5
    # all-dense input: every chunk falls back to the plain copy
    full = [torch.from_numpy(np.full_like(heat[:8], 0.4)).pin_memory(), host[1][:8], host[2][:8]]
    decoder.decode_host_batch(*full, chunk_frames=8, sparse='auto')
    assert decoder.host_chunks_sparse == 0 and decoder.host_bytes_copied == full[0].numel() * 4
    # 180x320 (partial tile rows: 180 = 45 x 4, 320 = 20 x 16) and a ragged size, pageable heatmaps
    for size in ((180, 320), (37, 93)):
        b = synthetic.make_batch(6, cfg, size, seed=size[0], objects=(1, 2), **(dict(center_separation=18.0, spoke_radius=(4.0, 6.0), peak_separation=5.0, border=3.0) if size[0] < 64 else {}))
        dec = KeypointDecoder(cfg, size, camera=synthetic.default_camera((180, 320)) if size == (180, 320) else camera)
        inputs = [torch.from_numpy(a) for a in (b.heat, b.depth, b.centers)]
        want = {k: v.clone() for k, v in dec.decode_host_batch(*inputs, chunk_frames=4, sparse=False).items()}
        dec.SPARSE_CAPACITY = 1.0
        got = dec.decode_host_batch(*inputs, chunk_frames=4, sparse='only')
        assert dec.host_chunks_sparse == 2
        for name in KeypointDecoder.HOST_RESULT_TABLES:
            np.testing.assert_array_equal(got[name].numpy().view(np.uint8), want[name].numpy().view(np.uint8), err_msg=name)


@pytest.mark.parametrize('single_pass', [False, True])
@pytest.mark.parametrize('workload,frames', [('config4_180x320', 256), ('config4_64x64', 1024)])
def test_headline_bench_workload_is_bitwise_the_oracle(workload, frames, single_pass):
    """The very frames bench.py times (synthetic.torch_grid_batch with bench.py's seed 1004 and grid) decoded on the GPU
    against the C oracle: bitwise integer and float32 tables, 3D points <= 1e-4 relative. The oracle was checked against the
    unmodified reference on frames of this generator (VERDICT r01); this closes the remaining GPU-vs-oracle comparison."""
    import bench
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder, synthetic
    w = bench.WORKLOADS[workload]
    heat, depth, centers, n_obj = synthetic.torch_grid_batch(frames, w['cfg'], w['size'], seed=1004, grid=w['grid'], device='cuda')
    camera = synthetic.default_camera(w['size'])
    decoder = KeypointDecoder(w['cfg'], w['size'], camera=camera, single_pass=single_pass)
    got = decoder.decode_batch(heat, depth, centers).numpy()
    want = c_oracle.decode(heat.cpu().numpy(), depth.cpu().numpy(), centers.cpu().numpy(), w['cfg'], camera)
    assert_matches_oracle(got, want)
    assert (got['n_objects'] == n_obj).mean() > 0.99
    # bf16 form of the same frames (config 5's element type): bitwise the oracle on the up-cast maps
    import torch
    heat16, depth16, centers16 = (t.to(torch.bfloat16) for t in (heat, depth, centers))
    got16 = decoder.decode_batch(heat16, depth16, centers16).numpy()
    want16 = c_oracle.decode(heat16.float().cpu().numpy(), depth16.float().cpu().numpy(), centers16.float().cpu().numpy(),
                             w['cfg'], camera)
    assert_matches_oracle(got16, want16)


def _tiny_scripted_model(path, heat, depth, centers):
    """A TorchScript module with the deployed model's contract (scripts/package_model.py:22-28): frames [N,3,h,w] ->
    (heat [N,C,H,W], depth, centers [N,C-1,2,H,W]); it replays fixed maps scaled by a function of the frame so that the
    input matters."""
    import torch

    class Replay(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.register_buffer('heat', torch.from_numpy(heat))
            self.register_buffer('depth', torch.from_numpy(depth))
            self.register_buffer('centers', torch.from_numpy(centers))

        def forward(self, frames):
            gain = 1.0 + 0.0 * frames.mean()
            return self.heat * gain, self.depth * gain, self.centers * gain

    torch.jit.script(Replay()).save(path)


def test_inference_component_and_learned_pipeline(tmp_path):
    """A9: InferenceComponent loads a TorchScript file, runs it on the device and leaves the outputs there;
    LearnedKeypointTrackingPipeline(model, cuda, prediction_size, points_3d, keypoint_config)(frame) returns
    (objects, heatmap) like perception/pipeline.py:13-28,202-209."""
    import torch
    from object_keypoints_b200 import InferenceComponent, LearnedKeypointTrackingPipeline, ObjectKeypointPipeline
    g = load_golden('valve_64.npz')
    ref = reference_tables(g)
    path = str(tmp_path / 'model.pt')
    _tiny_scripted_model(path, g['heat'][:1], g['depth'][:1], g['centers'][:1])
    inference = InferenceComponent(path, cuda=True)
    assert inference.name == 'inference'
    outputs = inference(torch.zeros(1, 3, 32, 32))
    assert len(outputs) == 3 and all(o.is_cuda for o in outputs), "outputs stay on the device (no .cpu() round trip)"
    assert outputs[0].shape == (1, 3, 64, 64) and outputs[2].shape == (1, 2, 2, 64, 64)
    pipeline = LearnedKeypointTrackingPipeline(path, True, [64, 64], None, {'keypoint_config': [1, 3]})
    pipeline.reset(golden_camera(g))
    objects, heatmap = pipeline(torch.zeros(1, 3, 32, 32))
    assert torch.equal(heatmap.cpu(), torch.from_numpy(g['heat'][:1]))
    plain = ObjectKeypointPipeline([64, 64], None, {'keypoint_config': [1, 3]})
    plain.reset(golden_camera(g))
    want = plain(torch.from_numpy(g['heat'][:1]), torch.from_numpy(g['depth'][:1]), torch.from_numpy(g['centers'][:1]))
    assert len(objects) == len(want) == ref['n_objects'][0]
    for a, b in zip(objects, want):
        for c in range(3):
            np.testing.assert_array_equal(a['keypoints'][c], b['keypoints'][c])
            np.testing.assert_array_equal(a['p_C'][c], b['p_C'][c])
            cnt = ref['kp_count'][0, objects.index(a), c]
            assert np.abs(a['keypoints'][c] - ref['kp_xy'][0, objects.index(a), c, :cnt]).max(initial=0) <= TOL_PIXELS
