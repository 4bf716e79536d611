"""float16 maps: the okp_*_f16 entries and the Python paths that reach them. Every float16 value, subnormals included, is
exactly a float32 value, so the f16 entries must give the tables of the f32 entries (and of the C oracle) on the
up-cast maps bit for bit. "Up-cast" below is ``t.float()``."""
import ctypes

import numpy as np
import pytest
import torch

from object_keypoints_b200 import _abi, _lib
from test_gpu_decode import assert_matches_oracle, _tiny_scripted_model

gpu = pytest.mark.gpu
GENERIC_PATH = 128          # OKP_FLAG_GENERIC_PATH
SMALL_LAYOUT = dict(center_separation=18.0, spoke_radius=(4.0, 6.0), peak_separation=5.0, border=3.0)


def _camera(size):
    from object_keypoints_b200 import camera_utils, synthetic
    if size in ((64, 64), (180, 320)):
        return synthetic.default_camera(size)
    return camera_utils.FisheyeCamera(np.array([[50.0, 0, size[1] / 2], [0, 50.0, size[0] / 2], [0, 0, 1]]),
                                      np.array([0.1, 0.01, -0.02, 0.003]), size)


def _f16(a):
    """float32 array -> (torch float16 CUDA tensor, its up-cast as float32 NumPy) -- what a half-precision head emits."""
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda().half()
    return t, t.float().cpu().numpy()


def _call_decode(entry, decoder, heat, depth, centers, sink=None):
    """One okp_decode_* / okp_decode_emit_* call on fresh tables -> NumPy tables."""
    from object_keypoints_b200.pipeline import DecodeTables
    N = heat.shape[0]
    tables = DecodeTables(N, decoder.C, decoder.cfg, decoder.params, decoder.device)
    ws = decoder._workspace_for(N)
    cam = ctypes.byref(decoder._camera) if decoder._camera is not None else None
    args = [heat.data_ptr(), depth.data_ptr(), centers.data_ptr(), N, decoder.C, decoder.H, decoder.W, decoder._cfg_array, cam,
            ctypes.byref(decoder.params), ctypes.byref(tables.struct), ws.data_ptr(), ws.numel()]
    if sink is not None:
        args.append(ctypes.byref(sink))
    rc = getattr(_lib.lib(), entry)(*args, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, entry)
    return tables.numpy()


def _assert_same_tables(got, want, context=''):
    """Two decodes with one arithmetic: integer tables and flags equal, float tables bitwise or NaN in the same places.
    OKP_FLAG_GENERIC_PATH says which kernels ran, not what the data held: 16-bit maps with W % 8 != 0 take the generic
    kernels where float32 maps still take the TMA kernel, so that bit is left out."""
    for key in want:
        a, b = got[key], want[key]
        if key == 'flags':
            a, b = a & ~np.uint32(GENERIC_PATH), b & ~np.uint32(GENERIC_PATH)
        if a.dtype.kind == 'f':
            both_nan = np.isnan(a) & np.isnan(b)
            a, b = np.where(both_nan, 0, a), np.where(both_nan, 0, b)
            a = a.view(np.uint32 if a.dtype == np.float32 else np.uint64)
            b = b.view(np.uint32 if b.dtype == np.float32 else np.uint64)
        np.testing.assert_array_equal(a, b, err_msg=f"{context} {key}")


def _all_f16_maps(H, W):
    """Every finite non-negative float16 (0x0000-0x7BFF, subnormals included) at an isolated pixel of a [N, 2, H, W] batch.
    An isolated value v makes a 5x5 plateau of box sums equal to v, i.e. 25 tied peaks: ten values per map on a 12-pixel
    grid keep each map's 250 peaks within max_peaks = 256 and no two plateaus in one 5x5 window."""
    values = np.arange(0x7C00, dtype=np.uint16).view(np.float16)
    spots = [(y, x) for y in range(6, H - 5, 12) for x in range(6, W - 5, 12)][:10]
    assert len(spots) == 10
    maps = (len(values) + 9) // 10
    maps += maps % 2
    heat = np.zeros((maps, H, W), np.float16)
    for i, v in enumerate(values):
        y, x = spots[i % 10]
        heat[i // 10, y, x] = v
    return heat.reshape(maps // 2, 2, H, W)


@gpu
@pytest.mark.parametrize('size', [(64, 64), (64, 60)])     # TMA kernel / W % 8 != 0: generic kernels for 16-bit maps
def test_every_float16_value_decodes_like_its_float32_upcast(size):
    from object_keypoints_b200 import KeypointDecoder
    H, W = size
    heat16 = _all_f16_maps(H, W)
    N = heat16.shape[0]
    rng = np.random.default_rng(16)
    depth16 = rng.uniform(0.5, 3.0, heat16.shape).astype(np.float16)
    centers16 = rng.uniform(-4.0, 4.0, (N, 1, 2, H, W)).astype(np.float16)
    decoder = KeypointDecoder([1], size, camera=_camera(size), threshold=1e-30, max_peaks=256, max_objects=128, max_votes=64)
    maps16 = [torch.from_numpy(a).cuda() for a in (heat16, depth16, centers16)]
    got = _call_decode('okp_decode_f16', decoder, *maps16)
    want = _call_decode('okp_decode_f32', decoder, *(t.float() for t in maps16))
    _assert_same_tables(got, want, str(size))
    assert (got['peak_count'] == 250).sum() == N * 2 - 3                 # all but the first (0x0000) and the last two
    assert (got['peak_count'] <= 256).all() and not (got['flags'] & 1).any()
    if W % 8:
        assert (got['flags'] & GENERIC_PATH).all()
    else:
        assert not (want['flags'] & GENERIC_PATH).any()


@gpu
@pytest.mark.parametrize('size', [(64, 64), (36, 92)])
def test_special_values_decode_like_the_float32_upcast(size):
    """+inf, NaN, negative values and -0.0 in heat, depth and centre maps: both entries hand such maps to the exact kernels
    and group them identically."""
    from object_keypoints_b200 import KeypointDecoder, synthetic
    batch = synthetic.make_batch(12, [1, 3], size, seed=4000 + size[1], objects=(1, 3),
                                 **(SMALL_LAYOUT if size[0] < 64 else {}))
    heat, depth, centers = batch.heat.copy(), batch.depth.copy(), batch.centers.copy()
    H, W = size
    heat[0, 0, H // 2, W // 2] = np.inf
    heat[1, 1, 10:12, 10:12] = np.nan
    heat[2, 2, 5, 7] = -0.25
    heat[3, 0, :, :] = -0.0
    heat[4, 1] = -heat[4, 1]
    heat[5, 0, 0, 0] = -np.inf
    depth[6] = np.nan
    depth[7, :, :, : W // 2] = np.inf
    centers[8, 0, 0] = np.nan
    centers[9] = -0.0
    heat[10] = 70000.0                                              # rounds to float16 +inf
    decoder = KeypointDecoder([1, 3], size, camera=_camera(size))
    maps16 = [_f16(a)[0] for a in (heat, depth, centers)]
    got = _call_decode('okp_decode_f16', decoder, *maps16)
    want = _call_decode('okp_decode_f32', decoder, *(t.float() for t in maps16))
    _assert_same_tables(got, want, str(size))
    assert got['n_objects'].sum() > 0


@gpu
@pytest.mark.parametrize('H,W,N,C,K', [
    (64, 64, 37, 3, 32),
    (3, 8, 5, 2, 8),
    (7, 240, 3, 2, 64),        # widest single 16-bit box (4 * 61 + 4 + 4 = 252 -> 256 columns)
    (9, 248, 2, 3, 64),        # narrowest two-box 16-bit row
    (33, 320, 2, 3, 16),       # K small: most maps overflow -> overflow path (float16 generic tiles)
    (12, 488, 2, 2, 256),      # widest 16-bit row the strip kernel takes (two boxes of 256 columns)
    (11, 496, 1, 2, 64),       # wider: generic kernel
    (30, 68, 2, 2, 32),        # W % 8 != 0 -> generic kernel
])
def test_f16_peak_extraction_shapes_noise_and_overflow(H, W, N, C, K):
    """Dense random float16 maps (quantisation makes exact ties common), -0.0 and negative values: strip kernel, overflow
    path and generic kernel give bitwise the C oracle's peak tables on the up-cast maps."""
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder
    rng = np.random.default_rng(H * 1000 + W + 2)
    heat = rng.uniform(0, 0.2, (N, C, H, W)).astype(np.float32)
    heat[0, 0, H // 2, W // 2] = -0.0
    if N > 1:
        heat[1, C - 1] = 0.001
        heat[1, 0, 0, 0] = -0.125
    heat_dev, heat32 = _f16(heat)
    cfg = [1] * (C - 1)
    decoder = KeypointDecoder(cfg, (H, W), max_peaks=K, max_objects=16)
    got = decoder.extract_peaks(heat_dev).numpy()
    want = c_oracle.decode(heat32, np.zeros_like(heat32), np.zeros((N, C - 1, 2, H, W), np.float32), cfg, None,
                           max_peaks=K, max_objects=16)
    np.testing.assert_array_equal(got['peak_count'], want['peak_count'])
    np.testing.assert_array_equal(got['peak_yx'], want['peak_yx'])
    for key in ['peak_score', 'peak_xy', 'peak_conf']:
        np.testing.assert_array_equal(got[key].view(np.uint32), want[key].view(np.uint32), err_msg=key)
    if (H, W) == (33, 320):
        assert (want['peak_count'] > K).any() and (want['peak_count'] <= K).any()


@gpu
@pytest.mark.parametrize('cfg,size,frames,objects', [
    ([1, 3], (64, 64), 96, (1, 2)),
    ([1, 1, 1], (64, 64), 64, (1, 4)),
    ([1, 3], (180, 320), 12, (1, 6)),        # two TMA boxes per row, second box with a 4-element lead
    ([2], (40, 56), 8, (1, 1)),              # W % 8 == 0, single box
    ([1, 3], (36, 92), 6, (1, 1)),           # W % 8 != 0: no 16-bit tensor map -> generic kernels
])
@pytest.mark.parametrize('single_pass', [False, True])
def test_f16_maps_decode_like_the_oracle_on_the_upcast_maps(cfg, size, frames, objects, single_pass):
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder, synthetic
    batch = synthetic.make_batch(frames, cfg, size, seed=5000 + size[1], objects=objects,
                                 **(SMALL_LAYOUT if size[0] < 64 else {}))
    camera = _camera(size)
    (heat, heat32), (depth, depth32), (centers, centers32) = (_f16(a) for a in (batch.heat, batch.depth, batch.centers))
    decoder = KeypointDecoder(cfg, size, camera=camera, single_pass=single_pass)
    got = decoder.decode_batch(heat, depth, centers).numpy()
    assert_matches_oracle(got, c_oracle.decode(heat32, depth32, centers32, cfg, camera))
    assert got['n_objects'].sum() > 0
    # float16 heatmaps with float32 depth / centre maps: peaks from okp_extract_peaks_f16, grouping from the f32 entry
    got = decoder.decode_batch(heat, torch.from_numpy(batch.depth).cuda(), torch.from_numpy(batch.centers).cuda()).numpy()
    assert_matches_oracle(got, c_oracle.decode(heat32, batch.depth, batch.centers, cfg, camera))
    # float16 heatmaps with bfloat16 depth / centre maps
    depth_bf, centers_bf = (torch.from_numpy(a).cuda().bfloat16() for a in (batch.depth, batch.centers))
    got = decoder.decode_batch(heat, depth_bf, centers_bf).numpy()
    assert_matches_oracle(got, c_oracle.decode(heat32, depth_bf.float().cpu().numpy(), centers_bf.float().cpu().numpy(),
                                               cfg, camera))


@gpu
@pytest.mark.parametrize('single_pass', [False, True])
@pytest.mark.parametrize('workload,frames', [('config4_180x320', 256), ('config4_64x64', 1024)])
def test_headline_bench_frames_in_float16_are_bitwise_the_oracle(workload, frames, single_pass):
    """The frames bench.py times (seed 1004), as a half-precision head would hand them over."""
    import bench
    from oracle import c_oracle
    from object_keypoints_b200 import KeypointDecoder, synthetic
    w = bench.WORKLOADS[workload]
    heat, depth, centers, n_obj = synthetic.torch_grid_batch(frames, w['cfg'], w['size'], seed=1004, grid=w['grid'], device='cuda')
    heat, depth, centers = heat.half(), depth.half(), centers.half()
    camera = synthetic.default_camera(w['size'])
    decoder = KeypointDecoder(w['cfg'], w['size'], camera=camera, single_pass=single_pass)
    got = decoder.decode_batch(heat, depth, centers).numpy()
    want = c_oracle.decode(heat.float().cpu().numpy(), depth.float().cpu().numpy(), centers.float().cpu().numpy(),
                           w['cfg'], camera)
    assert_matches_oracle(got, want)
    assert (got['n_objects'] == n_obj).mean() > 0.99


@gpu
@pytest.mark.parametrize('size', [(64, 64), (40, 56), (37, 92)])
@pytest.mark.parametrize('single_pass', [False, True])
def test_f16_records_are_those_of_the_f32_entry(size, single_pass):
    """okp_decode_emit_f16 writes byte for byte the compact records okp_decode_emit_f32 writes for the up-cast maps. At
    W % 8 != 0 the float16 maps take the generic kernels and the float32 maps the TMA kernel: there the records differ
    only by OKP_FLAG_GENERIC_PATH in the header's flags word."""
    from object_keypoints_b200 import KeypointDecoder, synthetic
    cfg = [1, 3]
    batch = synthetic.make_batch(23, cfg, size, seed=41, objects=(1, 3), **(SMALL_LAYOUT if size[0] < 64 else {}))
    heat = batch.heat.copy()
    heat[3, 1] = 0.5                                                   # overflow fix-up
    heat[5, 0, 10, 10] = -0.25                                         # exact path for that map
    heat[7, 0] = 0.0                                                   # no centres
    decoder = KeypointDecoder(cfg, size, camera=_camera(size), single_pass=single_pass)
    maps16 = [_f16(a)[0] for a in (heat, batch.depth, batch.centers)]
    records = {}
    for entry, maps in (('okp_decode_emit_f16', maps16), ('okp_decode_emit_f32', [t.float() for t in maps16])):
        buffer = torch.zeros((23 + 2, decoder.record_bytes()), dtype=torch.uint8, device='cuda')
        pointers = (ctypes.c_void_p * 1)(buffer.data_ptr())
        sink = _abi.OkpRecordSink(buffers_dev=pointers, n_buffers=1, record_bytes=decoder.record_bytes(), first_row=2)
        tables = _call_decode(entry, decoder, *maps, sink=sink)
        records[entry] = buffer.cpu()
    if size[1] % 8:
        flags16, flags32 = (records[k][2:].view(torch.int32)[:, 1] for k in ('okp_decode_emit_f16', 'okp_decode_emit_f32'))
        assert (flags16 & GENERIC_PATH).all() and not (flags32 & GENERIC_PATH).any()
        flags16 &= ~GENERIC_PATH
    assert torch.equal(records['okp_decode_emit_f16'], records['okp_decode_emit_f32'])
    assert records['okp_decode_emit_f16'][2:].any() and not records['okp_decode_emit_f16'][:2].any()
    assert tables['n_objects'].sum() > 0


def _half_scripted_model(path, heat, depth, centers):
    """_tiny_scripted_model, converted to half precision the way a user exports one (model.half())."""
    _tiny_scripted_model(path, heat, depth, centers)
    torch.jit.load(path).half().save(path)


@gpu
def test_half_precision_model_outputs_reach_the_f16_entries(tmp_path):
    from object_keypoints_b200 import InferenceComponent, LearnedKeypointTrackingPipeline, ObjectKeypointPipeline, synthetic
    from object_keypoints_b200 import pipeline as pipeline_module
    batch = synthetic.make_batch(1, [1, 3], (64, 64), seed=43, objects=(2, 2))
    path = str(tmp_path / 'model_half.pt')
    _half_scripted_model(path, batch.heat, batch.depth, batch.centers)
    outputs = InferenceComponent(path, cuda=True)(torch.zeros(1, 3, 32, 32))
    assert all(o.is_cuda and o.dtype == torch.float16 for o in outputs), "half-precision outputs stay float16 on the device"
    assert all(pipeline_module._as_device_map(o, o.device)[1] == 'f16' for o in outputs)
    camera = synthetic.default_camera((64, 64))
    learned = LearnedKeypointTrackingPipeline(path, True, [64, 64], None, {'keypoint_config': [1, 3]})
    learned.reset(camera)
    calls = []
    real = learned.decoder._lib
    learned.decoder._lib = type('Spy', (), {'__getattr__': lambda self, name: calls.append(name) or getattr(real, name)})()
    objects, heatmap = learned(torch.zeros(1, 3, 32, 32))
    assert heatmap.dtype == torch.float16 and 'okp_decode_emit_f16' in calls
    plain = ObjectKeypointPipeline([64, 64], None, {'keypoint_config': [1, 3]})
    plain.reset(camera)
    want = plain(*(o.float() for o in outputs))
    assert len(objects) == len(want) > 0
    for a, b in zip(objects, want):
        for c in range(3):
            np.testing.assert_array_equal(a['keypoints'][c], b['keypoints'][c])
            np.testing.assert_array_equal(a['p_C'][c], b['p_C'][c])
        np.testing.assert_array_equal(np.array(a['p_centers']), np.array(b['p_centers']))


@gpu
def test_float16_producer_decodes_through_the_overflow_path():
    """A random-init network in float16 at a test batch: ~100 noise peaks per map against max_peaks 32, so every map takes
    the overflow fix-up; the f16 tables are those of the f32 entry on the up-cast maps."""
    from object_keypoints_b200 import KeypointDecoder, producer, synthetic
    cfg = [1, 3]
    net = producer.build_producer(cfg, device='cuda', dtype=torch.float16, seed=0)
    frames = torch.randn(4, 3, 511, 511, device='cuda', dtype=torch.float16,
                         generator=torch.Generator('cuda').manual_seed(6)).contiguous(memory_format=torch.channels_last)
    with torch.no_grad():
        heat, depth, centers = net(frames)
    assert heat.dtype == torch.float16 and heat.is_contiguous() and heat.shape == (4, 3, 64, 64)
    decoder = KeypointDecoder(cfg, (64, 64), camera=synthetic.default_camera((64, 64)), max_peaks=32, max_objects=32,
                              max_votes=16)
    got = decoder.decode_batch(heat, depth, centers).numpy()
    want = decoder.decode_batch(heat.float(), depth.float(), centers.float()).numpy()
    assert (got['flags'] & 1).all(), "every frame overflows max_peaks"
    _assert_same_tables(got, want)


@gpu
@pytest.mark.parametrize('dtype', [torch.float16, torch.bfloat16])
def test_host_batch_of_16bit_maps_equals_the_device_decode(dtype):
    """decode_host_batch on 16-bit CPU maps, pinned (depth / centres gathered in place) and pageable (copied), with a chunk
    size that does not divide N: the tables of decode_batch on the same maps on the device, half the float32 bytes."""
    from object_keypoints_b200 import KeypointDecoder, synthetic
    cfg = [1, 3]
    batch = synthetic.make_batch(37, cfg, (64, 64), seed=47, objects=(1, 3))
    decoder = KeypointDecoder(cfg, (64, 64), camera=synthetic.default_camera((64, 64)))
    host32 = [torch.from_numpy(a) for a in (batch.heat, batch.depth, batch.centers)]
    host = [t.to(dtype) for t in host32]
    want = decoder.decode_batch(*(t.cuda() for t in host)).numpy()
    for pinned in (True, False):
        inputs = [t.pin_memory() for t in host] if pinned else host
        assert (decoder._host_alias(inputs[1]) is not None) == pinned
        got = decoder.decode_host_batch(*inputs, chunk_frames=16, sparse='auto')
        for name in KeypointDecoder.HOST_RESULT_TABLES:
            np.testing.assert_array_equal(got[name].numpy().view(np.uint8), want[name].view(np.uint8), err_msg=f"{pinned} {name}")
        copied16 = decoder.host_bytes_copied
        assert decoder.host_chunks_sparse == 0
        decoder.decode_host_batch(*([t.pin_memory() for t in host32] if pinned else host32), chunk_frames=16, sparse=False)
        assert 2 * copied16 == decoder.host_bytes_copied
        assert copied16 == sum(t.nbytes for t in (host[:1] if pinned else host))
    with pytest.raises(ValueError, match='dtype'):
        decoder.decode_host_batch(host[0], host32[1], host[2])
    with pytest.raises(ValueError, match='dtype'):
        decoder.decode_host_batch(host[0], host[1], host[2].to(torch.float16 if dtype == torch.bfloat16 else torch.bfloat16))


def test_f16_entries_validate_their_arguments_on_the_host():
    """As okp_*_f32 do: NULL maps, bad shapes and bad parameters are rejected before anything touches a device."""
    if _lib.needs_build():
        _lib.build()
    lib = _lib.lib()
    prm, tables = _abi.make_params(), _abi.OkpDecodeTables()
    cfg = (ctypes.c_int32 * 2)(1, 3)
    bad_mode, bad_capacity = _abi.make_params(), _abi.make_params()
    bad_mode.nms_size = 7
    bad_capacity.top_k = 64                                           # more than max_peaks

    def extract(N, C, p):
        return lib.okp_extract_peaks_f16(None, N, C, 64, 64, ctypes.byref(p), ctypes.byref(tables), None, 0, None)

    def decode(N, C, p):
        return lib.okp_decode_f16(None, None, None, N, C, 64, 64, cfg, None, ctypes.byref(p), ctypes.byref(tables), None, 0, None)

    def decode_emit(N, C, p):
        return lib.okp_decode_emit_f16(None, None, None, N, C, 64, 64, cfg, None, ctypes.byref(p), ctypes.byref(tables),
                                       None, 0, None, None)

    def group(N, C, p):
        return lib.okp_group_objects_f16(None, None, N, C, 64, 64, cfg, None, ctypes.byref(p), ctypes.byref(tables), None)

    def group_emit(N, C, p):
        return lib.okp_group_objects_emit_f16(None, None, N, C, 64, 64, cfg, None, ctypes.byref(p), ctypes.byref(tables),
                                              None, None)

    for call in (extract, decode, decode_emit, group, group_emit):
        assert call(1, 3, prm) == -1, call.__name__                  # OKP_E_NULL
        assert call(1, 0, prm) == -2, call.__name__                  # OKP_E_SHAPE
        assert call(1, 99, prm) == -2, call.__name__
        assert call(0, 3, prm) == 0, call.__name__                   # nothing to do
        assert call(1, 3, bad_mode) == -4, call.__name__             # OKP_E_UNSUPPORTED
        assert call(1, 3, bad_capacity) == -3, call.__name__         # OKP_E_CAPACITY
