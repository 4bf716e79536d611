"""Parity at multi-wave sizes: batches large enough that every work loop of the peak path runs several times per CTA,
compared with the C oracle (oracle/okp_oracle.c) by the rules of test_gpu_decode.py.

- okp_peaks_stream_kernel (csrc/okp_peaks_stream.cuh): resident CTAs claim groups of M maps from a counter; groups
  alternate between two candidate buffers, an 8-entry ring passes the claimed ids on, and the epilogue warps clear the
  per-group counters for the next group. Only a CTA's second and later groups go through the buffer alternation, the
  ring wrap, the parity flips and those resets.
- okp_peaks_overflow_kernel (csrc/okp_peaks.cuh): each of at most 592 CTAs redoes the overflowing maps of its slice of
  ceil(maps / 592) maps one after the other, on the same tile lists, in steps of 256 maps.
- okp_peaks_generic_kernel: maps x tiles work items over min(work, 148 x 8) CTAs.

test_cases_are_multi_wave (CPU; nvcc) derives from the planner how many groups, slices or work items each CTA gets,
so a planner change that makes a case single-wave fails there. The GPU tests plant adversarial maps at seeded places
in clean batches -- whole adversarial groups, maps in the ragged last group, maps beside clean ones -- and check that
the oracle's tables show every planted situation, so that the comparison cannot quietly become a clean-only run."""
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMS = 148                          # B200; the device's own count where one is visible
REGISTERS = 96                     # __maxnreg__ of okp_peaks_stream_kernel
OVERFLOW_CTAS = 592                # OKP_OVERFLOW_CTAS
GENERIC_CTAS = 148 * 8             # plan_peaks: kSmCount * 8
ESIZE = {'f32': 4, 'bf16': 2, 'f16': 2}

# Stream-kernel cases. M: maps per group of each form's plan ('split' / 'peaks': the peak kernel alone, 'fused':
# single_pass), pinned by test_cases_are_multi_wave. waves: least groups per resident CTA. Frame counts leave the
# last group ragged wherever the plan allows it (M does not divide C, F > 1).
STREAM = {
    'small_maps_64x64': dict(size=(64, 64), cfg=[1, 3], K=32, frames=4099, dtypes=('f32', 'bf16', 'f16'),
                             forms=('split', 'fused'), M={'split': 13, 'fused': 12}, waves=3, grid=(2, 1)),
    'bench_180x320': dict(size=(180, 320), cfg=[1, 3], K=32, frames=600, dtypes=('f32', 'bf16'),
                          forms=('split', 'fused'), M={'split': 3, 'fused': 3}, waves=2, grid=(4, 2)),
    'bench_180x320_peaks': dict(size=(180, 320), cfg=[1, 3], K=32, frames=1200, dtypes=('f32', 'bf16'),
                                forms=('peaks',), M={'peaks': 3}, waves=3, grid=(4, 2)),
    'two_maps_180x320': dict(size=(180, 320), cfg=[1], K=32, frames=900, dtypes=('f32',), forms=('fused',),
                             M={'fused': 2}, waves=3, grid=(4, 2)),
    'short_20x320': dict(size=(20, 320), cfg=[1, 1], K=32, frames=3001, dtypes=('f32',), forms=('split',),
                         M={'split': 2}, waves=3, grid=(4, 1)),
    'widest_12x496': dict(size=(12, 496), cfg=[1], K=64, frames=2000, dtypes=('f32',), forms=('split',),
                          M={'split': 1}, waves=3, grid=(4, 1)),
    'tiny_5x64': dict(size=(5, 64), cfg=[1, 1, 1], K=32, frames=40000, dtypes=('f32',), forms=('split', 'fused'),
                      M={'split': 13, 'fused': 12}, waves=3, grid=(2, 1)),
}

# Overflow fix-up cases: every map (random-init network), maps on slice edges, and K = 1 (any second peak overflows).
OVERFLOW = {
    'random_init_64x64': dict(size=(64, 64), cfg=[1, 3], K=32, frames=256, dtypes=('f32', 'bf16', 'f16')),
    'slice_edges_64x64': dict(size=(64, 64), cfg=[1, 3], K=32, frames=2000, dtypes=('f32',)),
    'k1_5x64': dict(size=(5, 64), cfg=[1, 1, 1], K=1, frames=40000, dtypes=('f32',)),
}

# Generic tile-kernel cases: shapes the stream kernel does not take, and a peak mode it does not implement.
GENERIC = {
    'odd_37x93': dict(size=(37, 93), cfg=[1, 3], K=32, frames=600, modes={}),
    'bench_plus_2_180x322': dict(size=(180, 322), cfg=[1, 3], K=32, frames=40, modes={}),
    'modes_64x64': dict(size=(64, 64), cfg=[1, 3], K=32, frames=1600, modes=dict(nms_size=3, box_sum=False, top_k=5)),
}


def slice_maps(maps):
    """Maps per CTA of the overflow fix-up (overflow_maps_per_cta, okp_api.cu)."""
    grid = min(maps, OVERFLOW_CTAS)
    return -(-maps // grid)


def generic_tiles(H, W):
    """Tiles per map of the generic kernel (plan_peaks, okp_api.cu)."""
    TW = -(-W // 8) * 8 if W <= 64 else 64
    TH = H if H <= 64 else 32
    return -(-W // TW) * -(-H // TH)


# ------------------------------------------------------------------------------------------------ CPU: the plans ---
@pytest.fixture(scope='module')
def print_plan(tmp_path_factory):
    if shutil.which('nvcc') is None:
        pytest.skip("nvcc not on PATH")
    out = str(tmp_path_factory.mktemp('plans') / 'print_plan')
    run = subprocess.run(['nvcc', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', out,
                          os.path.join(ROOT, 'tools', 'print_plan.cu')], capture_output=True, text=True)
    assert run.returncode == 0, run.stderr[-2000:]
    return out


def plan(print_plan, H, W, esize, maps, C, K, fused):
    """okp_stream_plan's figures for one shape (print_plan shape), or None where the stream kernel does not take it."""
    text = subprocess.run([print_plan, 'shape', str(H), str(W), str(esize), str(maps), str(C), str(K), str(int(fused))],
                          capture_output=True, text=True, timeout=60, check=True).stdout.splitlines()
    head, row = text[0].split(':')[1].split(), text[1].split(':')[1].split()
    return None if row == ['-'] else dict(zip(head, (int(v) for v in row)))


def sm_count():
    try:
        import torch
        if torch.cuda.is_available():
            return torch.cuda.get_device_properties(0).multi_processor_count
    except ImportError:
        pass
    return SMS


def resident_ctas(p):
    """Upper bound of the stream kernel's CTAs resident at once: 96 registers per thread (whole warps) within 65 536
    registers, smem + 1 KB within 228 KB, per SM."""
    by_registers = 65536 // (REGISTERS * (-(-p['total'] // 32) * 32))
    by_smem = 228 * 1024 // (p['smem'] + 1024)
    return min(by_registers, by_smem) * sm_count()


def test_cases_are_multi_wave(print_plan):
    for name, case in STREAM.items():
        (H, W), C, K, N = case['size'], 1 + len(case['cfg']), case['K'], case['frames']
        for dtype in case['dtypes']:
            for form in case['forms']:
                p = plan(print_plan, H, W, ESIZE[dtype], N * C, C, K, form == 'fused')
                what = (name, dtype, form, p)
                assert p is not None and p['M'] == case['M'][form], what
                ctas = resident_ctas(p)
                assert p['groups'] >= case['waves'] * ctas, (what, ctas)
                if form == 'fused':
                    assert p['F'] == p['M'] // C and (N % p['F'] or p['F'] == 1), what
                else:
                    assert N * C % p['M'] or C % p['M'] == 0, what
                print(f"{name} {dtype} {form}: M {p['M']}, {p['groups']} groups over <= {ctas} CTAs "
                      f"({p['groups'] / ctas:.1f} per CTA)")
    per_slice = []
    for name, case in OVERFLOW.items():
        (H, W), C, K = case['size'], 1 + len(case['cfg']), case['K']
        maps = case['frames'] * C
        for dtype in case['dtypes']:
            assert plan(print_plan, H, W, ESIZE[dtype], maps, C, K, False) is not None, (name, dtype)
        per_slice.append(slice_maps(maps))
        assert per_slice[-1] >= 2, (name, per_slice[-1])
        print(f"{name}: {maps} maps, {per_slice[-1]} per overflow CTA")
    assert max(per_slice) > 256                       # okp_peaks_overflow_kernel's `base += THREADS` loop
    for name, case in GENERIC.items():
        (H, W), C, K = case['size'], 1 + len(case['cfg']), case['K']
        maps = case['frames'] * C
        if not case['modes']:
            assert plan(print_plan, H, W, 4, maps, C, K, False) is None, name
        work = maps * generic_tiles(H, W)
        assert work > 3 * GENERIC_CTAS, (name, work)
        print(f"{name}: {work} work items over {GENERIC_CTAS} CTAs ({work / GENERIC_CTAS:.1f} per CTA)")


# --------------------------------------------------------------------------------------------- GPU: the batches ---
def _camera(size):
    from test_gpu_f16 import _camera as camera
    return camera(size)


def _isolated(flat, m, y, x):
    """A lone 0.9 in a cleared 13 x 13 patch: a 5 x 5 plateau of box sums 0.9, i.e. 25 tied peaks whose 336 tie
    neighbours exceed the 64 items a group keeps per map (okp_stream_epilogue: the `redo` route)."""
    H, W = flat.shape[1:]
    flat[m, max(y - 6, 0):y + 7, max(x - 6, 0):x + 7] = 0.0
    flat[m, y, x] = 0.9


def _spots(H, W, rng, count):
    """count columns 13 apart (no window holds two plateaus) on the middle row."""
    x0 = int(rng.integers(6, W - 6 - 13 * (count - 1)))
    return [(H // 2, x0 + 13 * i) for i in range(count)]


def plant(flat, C, K, Ms, rng, decode):
    """Adversarial maps at seeded places of a [maps, H, W] float32 device batch; returns {situation: [map, ...]}.
    Ms: maps per group of the forms that run (a whole group of each is adversarial)."""
    import torch
    maps, H, W = flat.shape
    dev = flat.device
    used = set()
    out = {k: [] for k in ('overflow', 'ties', 'candidates', 'negative', 'zero_sign', 'nan', 'zero', 'border', 'no_centres')}

    def free(lo=0, hi=maps, frame_free=False):
        while True:
            m = int(rng.integers(lo, hi))
            if frame_free:
                m -= m % C
                if any(f in used for f in range(m, m + C)):
                    continue
            if m not in used:
                return m

    def overflow(m):
        if H >= 12:                                   # a random-init network's map: dozens of noise peaks
            noise = 0.5 + 0.002 * rng.standard_normal((H, W))
            flat[m] = torch.from_numpy(noise.astype(np.float32)).to(dev)
        else:                                         # a few rows hold too few noise peaks: plateaus of 25 peaks
            flat[m] = 0.0
            for y, x in _spots(H, W, rng, K // 25 + 1):
                _isolated(flat, m, y, x)
        out['overflow'].append(m)
        used.add(m)

    def ties(m):                                      # alone in its map: 25 peaks, within K
        y, x = _spots(H, W, rng, 1)[0]
        flat[m] = 0.0
        _isolated(flat, m, y, x)
        out['ties'].append((m, y, x))
        used.add(m)

    groups = [-(-maps // M) for M in Ms]
    for M, count in zip(Ms, groups):
        # whole groups of each kind, past the first wave (ids >= the resident CTAs are a CTA's second group or later)
        for kind in (overflow, ties):
            g = int(rng.integers(count // 2, count - 1))
            for m in range(g * M, min((g + 1) * M, maps)):
                if m not in used:
                    kind(m)
        last = (count - 1) * M                        # the ragged last group: overflow first, ties last
        if last not in used:
            overflow(last)
        if maps - 1 not in used:
            ties(maps - 1)
    for _ in range(4):                                # beside clean maps
        overflow(free(maps // 3))
        ties(free(maps // 3))
    if (H - 6) * (W - 6) > 2 * K:                     # a saturated plateau: more than 2K tied candidates
        for _ in range(2):
            m = free(maps // 3)
            flat[m, 1:H - 1, 1:W - 1] = 1.0
            out['candidates'].append(m)
            used.add(m)
    yy = torch.arange(H, device=dev, dtype=torch.float32)[:, None]
    xx = torch.arange(W, device=dev, dtype=torch.float32)[None, :]
    for kind, value in (('negative', -0.25), ('zero_sign', -0.0), ('nan', float('nan'))):
        for _ in range(2):                            # the value half a map away from a blob that stays a peak
            m = free(maps // 3)
            y, x = int(rng.integers(H)), int(rng.integers(W))
            flat[m] = torch.maximum(flat[m], torch.exp(-((yy - H // 2) ** 2 + (xx - (x + W // 2) % W) ** 2) / 4.0))
            flat[m, y, x] = value
            out[kind].append(m)
            used.add(m)
    m = free(maps // 3)
    flat[m] = 0.0
    out['zero'].append(m)
    used.add(m)
    for _ in range(2):                                # blobs on the last row and the last column
        m = free(maps // 3)
        for y, x in ((H - 1, W - 1), (H - 1, W // 3), (H // 2, W - 1)):
            flat[m] = torch.maximum(flat[m], torch.exp(-((yy - y) ** 2 + (xx - x) ** 2) / 4.0))
        out['border'].append(m)
        used.add(m)
    if decode:
        for _ in range(2):                            # frames without centres: nothing to group
            m = free(maps // 3, frame_free=True)
            flat[m] = 0.0
            out['no_centres'].append(m)
            used.update(range(m, m + C))
    return out


def assert_planted(want, planted, size, C, K, n_obj, decode, full_objects):
    """The oracle's tables show every planted situation, and the clean frames decode as clean frames."""
    count = want['peak_count'].reshape(-1)
    yx = want['peak_yx'].reshape(count.size, K, 2)
    assert (count[planted['overflow']] > K).all()
    assert (count[planted['candidates']] > 2 * K).all()
    for m, y, x in planted['ties']:
        plateau = {(y + dy, x + dx) for dy in range(-2, 3) for dx in range(-2, 3)}
        assert count[m] == 25 and {tuple(p) for p in yx[m, :25]} == plateau, (m, count[m])
    for kind in ('negative', 'zero_sign', 'nan', 'border'):
        assert (count[planted[kind]] > 0).all(), kind
    assert (count[planted['zero']] == 0).all()
    H, W = size
    for m in planted['border']:
        rows, cols = yx[m, :min(count[m], K), 0], yx[m, :min(count[m], K), 1]
        assert (rows >= H - 3).any() and (cols >= W - 3).any(), m
    planted_frames = {(m if k != 'ties' else m[0]) // C for k, v in planted.items() for m in v}
    clean = np.array([n for n in range(count.size // C) if n not in planted_frames])
    found = (want['peak_count'][clean] > 0).all(axis=1) if full_objects else want['peak_count'][clean].sum(axis=1) > 0
    assert found.mean() > 0.9
    if decode:
        for m in planted['no_centres']:
            n = m // C
            assert want['n_objects'][n] == 0
            assert (want['peak_count'][n, 1:] > 0).all() or not full_objects
        if full_objects:
            assert (want['n_objects'][clean] == n_obj).mean() > 0.99
        else:
            assert (want['n_objects'][clean] > 0).mean() > 0.5


class _Batch:
    """One case's planted float32 batch on the device and its oracle tables per element type; one case at a time."""
    key = None
    value = None


def _stream_batch(name):
    import torch
    from object_keypoints_b200 import synthetic
    if _Batch.key == name:
        return _Batch.value
    _Batch.key, _Batch.value = None, None
    case = STREAM[name]
    (H, W), cfg, K, N = case['size'], case['cfg'], case['K'], case['frames']
    C = 1 + len(cfg)
    heat, depth, centers, n_obj = synthetic.torch_grid_batch(N, cfg, (H, W), seed=7000 + H, grid=case['grid'], device='cuda')
    rng = np.random.default_rng(H * 1000 + W + C)
    decode = case['forms'] != ('peaks',)
    planted = plant(heat.view(-1, H, W), C, K, sorted(set(case['M'].values())), rng, decode)
    _Batch.key, _Batch.value = name, dict(heat=heat, depth=depth, centers=centers, n_obj=n_obj, planted=planted, want={})
    return _Batch.value


def _cast(t, dtype):
    """(device tensor of the element type, its up-cast as float32 NumPy): the oracle decodes the up-cast maps."""
    import torch
    if dtype == 'f32':
        return t, t.cpu().numpy()
    low = t.to(torch.bfloat16 if dtype == 'bf16' else torch.float16)
    return low, low.float().cpu().numpy()


def _oracle(b, dtype, cfg, camera, decode, K, **options):
    from oracle import c_oracle
    if dtype not in b['want']:
        heat, heat32 = _cast(b['heat'], dtype)
        N, C, H, W = heat.shape
        if decode:
            (depth, depth32), (centers, centers32) = _cast(b['depth'], dtype), _cast(b['centers'], dtype)
            want = c_oracle.decode(heat32, depth32, centers32, cfg, camera, max_peaks=K, **options)
        else:
            depth = centers = None
            want = c_oracle.decode(heat32, np.zeros_like(heat32), np.zeros((N, C - 1, 2, H, W), np.float32), cfg, None,
                                   max_peaks=K, **options)
        b['want'][dtype] = (heat, depth, centers, want)
    return b['want'][dtype]


STREAM_RUNS = [(name, dtype, form) for name, case in STREAM.items() for dtype in case['dtypes'] for form in case['forms']]


@pytest.mark.gpu
@pytest.mark.parametrize('name,dtype,form', STREAM_RUNS)
def test_stream_kernel_multi_wave_is_bitwise_the_oracle(name, dtype, form):
    from object_keypoints_b200 import KeypointDecoder, _abi
    from test_gpu_decode import assert_matches_oracle, assert_peaks_match_oracle
    case = STREAM[name]
    size, cfg, K = case['size'], case['cfg'], case['K']
    C = 1 + len(cfg)
    camera = _camera(size)
    b = _stream_batch(name)
    decode = form != 'peaks'
    heat, depth, centers, want = _oracle(b, dtype, cfg, camera, decode, K)
    assert_planted(want, b['planted'], size, C, K, b['n_obj'], decode, full_objects=size[0] >= 64)
    if not decode:
        assert_peaks_match_oracle(KeypointDecoder(cfg, size, max_peaks=K).extract_peaks(heat).numpy(), want)
        return
    decoder = KeypointDecoder(cfg, size, camera=camera, max_peaks=K, single_pass=form == 'fused')
    assert_matches_oracle(decoder.decode_batch(heat, depth, centers).numpy(), want)
    if (name, dtype, form) == ('small_maps_64x64', 'f32', 'split'):
        lean = KeypointDecoder(cfg, size, camera=camera, max_peaks=K, lean_tables=True)
        tables = lean.tables(heat.shape[0])
        tables.flat.fill_(0x5A)
        assert_matches_oracle(_abi.mask_unspecified(lean.decode_batch(heat, depth, centers, tables=tables).numpy()), want)


OVERFLOW_RUNS = [(name, dtype, form) for name, case in OVERFLOW.items() for dtype in case['dtypes']
                 for form in (('split', 'fused') if dtype == 'f32' and name != 'k1_5x64' else ('split',))]


@pytest.mark.gpu
@pytest.mark.parametrize('name,dtype,form', OVERFLOW_RUNS)
def test_overflow_fixup_multi_slice_is_bitwise_the_oracle(name, dtype, form):
    import torch
    from object_keypoints_b200 import KeypointDecoder, synthetic
    from test_gpu_decode import assert_matches_oracle
    case = OVERFLOW[name]
    size, cfg, K, N = case['size'], case['cfg'], case['K'], case['frames']
    (H, W), C = size, 1 + len(cfg)
    heat, depth, centers, _ = synthetic.torch_grid_batch(N, cfg, size, seed=8000 + H, grid=(2, 1), device='cuda')
    flat = heat.view(-1, H, W)
    maps, per = flat.shape[0], slice_maps(flat.shape[0])
    rng = np.random.default_rng(N + H)
    if name == 'random_init_64x64':                   # BASELINE config 5: an untrained network, every map overflows
        picks = list(range(maps))
    elif name == 'slice_edges_64x64':                 # both sides of slice boundaries, a whole slice, the last partial one
        picks = sorted({m for k in (1, 2, 97, 300, 544) for m in (k * per - 1, k * per)} |
                       set(range(200 * per, 201 * per)) | set(range((maps - 1) // per * per, maps)))
    else:                                             # K = 1: the clean maps themselves overflow
        picks = []
    for m in picks:
        flat[m] = torch.from_numpy((0.5 + 0.002 * rng.standard_normal((H, W))).astype(np.float32)).cuda()
    camera = _camera(size)
    heat, heat32 = _cast(heat, dtype)
    (depth, depth32), (centers, centers32) = _cast(depth, dtype), _cast(centers, dtype)
    from oracle import c_oracle
    want = c_oracle.decode(heat32, depth32, centers32, cfg, camera, max_peaks=K)
    count = want['peak_count'].reshape(-1)
    assert (count[picks] > K).all()
    if name == 'k1_5x64':                             # overflowing maps past the first 256 of their slice
        over = np.flatnonzero(count > K)
        assert (over % per >= 256).sum() > 100 and (count <= K).any()
    decoder = KeypointDecoder(cfg, size, camera=camera, max_peaks=K, single_pass=form == 'fused')
    assert_matches_oracle(decoder.decode_batch(heat, depth, centers).numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize('name', list(GENERIC))
def test_generic_kernel_multi_wave_is_bitwise_the_oracle(name):
    from object_keypoints_b200 import KeypointDecoder, synthetic
    from oracle import c_oracle, np_oracle
    from test_gpu_decode import assert_matches_oracle, assert_peaks_match_oracle
    case = GENERIC[name]
    size, cfg, K, N, modes = case['size'], case['cfg'], case['K'], case['frames'], case['modes']
    (H, W), C = size, 1 + len(cfg)
    heat, depth, centers, n_obj = synthetic.torch_grid_batch(N, cfg, size, seed=9000 + W, grid=(2, 1), device='cuda')
    planted = plant(heat.view(-1, H, W), C, K, [1], np.random.default_rng(W), decode=not modes)
    camera = _camera(size)
    heat32 = heat.cpu().numpy()
    if modes:                                         # 3x3 NMS on the map values, top 5 of each map by score
        want = np_oracle.extract_peak_tables(heat32, threshold=0.5, nms_size=modes['nms_size'], use_box_sum=modes['box_sum'],
                                             top_k=modes['top_k'], max_peaks=K)
        count = want['peak_count'].reshape(-1)
        assert (count[planted['overflow']] > K).all() and (count[planted['candidates']] > K).all()
        assert (count == modes['top_k']).sum() > count.size // 4
        assert_peaks_match_oracle(KeypointDecoder(cfg, size, max_peaks=K, **modes).extract_peaks(heat).numpy(), want)
        return
    want = c_oracle.decode(heat32, depth.cpu().numpy(), centers.cpu().numpy(), cfg, camera, max_peaks=K)
    assert_planted(want, planted, size, C, K, n_obj, True, full_objects=H >= 64)
    got = KeypointDecoder(cfg, size, camera=camera, max_peaks=K).decode_batch(heat, depth, centers).numpy()
    assert (got['flags'] & 128).all()                 # OKP_FLAG_GENERIC_PATH
    assert_matches_oracle(got, want)
