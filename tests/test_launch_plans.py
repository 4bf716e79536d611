"""Launch plans of the peak kernel (host code of csrc/okp_peaks_stream.cuh, compiled with nvcc; no GPU needed): the shapes the
bench runs must keep TWO CTAs per SM -- at most 320 threads at 96 registers and at most ~113 KB of shared memory per CTA. Round 2
found the 64x64 bfloat16 plan at 352 threads, i.e. one CTA per SM and 719 us instead of 448 us; this pins the fix.

The goldens pin the plans and the workspace sizes of a grid of shapes on both sides of every eligibility edge of the
planner (row width, alignment, map count, frames per group, table capacity): a change to the planner that moves any of
them shows up here, row by row."""
import ctypes
import gzip
import os
import re
import shutil
import subprocess

import pytest

from object_keypoints_b200 import _abi, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')

# the grid of tools/print_plan.cu's `table` mode
HS = (1, 2, 5, 64, 65, 180, 720)
WS = (4, 6, 8, 12, 60, 64, 68, 252, 256, 260, 320, 496, 500, 504)
MAPS = (1, 3, 7, 12288, 98304)
CS = (1, 3, 4)
KS = (1, 32, 256)


@pytest.fixture(scope='module')
def print_plan(tmp_path_factory):
    if shutil.which('nvcc') is None:
        pytest.skip("nvcc not on PATH")
    out = str(tmp_path_factory.mktemp('plans') / 'print_plan')
    run = subprocess.run(['nvcc', '-std=c++17', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', out,
                          os.path.join(ROOT, 'tools', 'print_plan.cu')], capture_output=True, text=True)
    assert run.returncode == 0, run.stderr[-2000:]
    return out


@pytest.fixture(scope='module')
def plans(print_plan):
    text = subprocess.run([print_plan], capture_output=True, text=True, timeout=60).stdout
    rows = []
    for line in text.splitlines():
        m = re.match(r'\s*(\d+)x\s*(\d+) esize (\d) fused (\d): M\s*(\d+) strips\s*(\d+) compute threads\s*(\d+) EW (\d) total threads\s*(\d+) '
                     r'smem\s*(\d+) NS (\d) nb (\d+) groups (\d+) F (\d+)', line)
        if m:
            keys = ('H', 'W', 'esize', 'fused', 'M', 'strips', 'compute', 'EW', 'threads', 'smem', 'NS', 'nb', 'groups', 'F')
            rows.append(dict(zip(keys, (int(v) for v in m.groups()))))
    assert rows, text
    return rows


def test_bench_shapes_keep_two_ctas_per_sm(plans):
    seen = set()
    for p in plans:
        if (p['H'], p['W']) not in ((180, 320), (64, 64)):
            continue
        seen.add((p['H'], p['W'], p['esize'], p['fused']))
        assert p['threads'] <= 320, p                      # 2 x 320 threads x 96 registers = 61440 of the SM's 65536
        assert p['smem'] <= 113 * 1024, p                  # 2 x (smem + 1 KB reserved) within 227 KB
        assert p['compute'] == p['M'] * p['strips'] and p['threads'] == (p['compute'] + 31) // 32 * 32 + 32 + 32 * p['EW'], p
    assert len(seen) == 8


def test_small_maps_take_the_small_map_plan(plans):
    for p in plans:
        if (p['H'], p['W']) == (64, 64):
            assert p['NS'] == 3 and p['compute'] <= 224 and p['EW'] == 2, p
        if (p['H'], p['W']) == (180, 320):
            assert p['NS'] == 4 and p['M'] == 3 and p['EW'] == 1, p
        if p['fused']:
            assert p['F'] >= 1 and p['M'] % 3 == 0, p      # a fused group is a whole number of frames (C = 3 in print_plan.cu)


def golden_lines(name):
    with gzip.open(os.path.join(GOLDEN, name), 'rt') as handle:
        return handle.read().splitlines()


def assert_same_rows(got, want):
    assert len(got) == len(want), (len(got), len(want))
    differ = [(w, g) for w, g in zip(want, got) if w != g]
    assert not differ, f"{len(differ)} rows differ, first ones (golden, now): {differ[:5]}"


def test_stream_plans_match_the_golden(print_plan):
    """Eligibility and every plan figure of okp_stream_plan, peaks only and fused, over the grid."""
    got = subprocess.run([print_plan, 'table'], capture_output=True, text=True, timeout=60).stdout.splitlines()
    assert_same_rows(got, golden_lines('launch_plans.txt.gz'))


def workspace_rows(lib):
    yield 'H W N C K nms_size box_sum: bytes'
    for H in HS:
        for W in WS:
            for maps in MAPS:
                for C in CS:
                    for K in KS:
                        N = -(-maps // C)                    # frames of C maps: at least `maps` maps
                        # the reference mode (the stream kernel where the shape allows it) and two that take the generic path
                        for nms, box in ((5, 1), (3, 1), (5, 0)):
                            prm = _abi.make_params(max_peaks=K, nms_size=nms, box_sum=bool(box))
                            yield f'{H} {W} {N} {C} {K} {nms} {box}: {lib.okp_decode_workspace_bytes(N, C, H, W, ctypes.byref(prm))}'


def test_workspace_bytes_match_the_golden():
    if _lib.needs_build():
        _lib.build()
    assert_same_rows(list(workspace_rows(_lib.lib())), golden_lines('workspace_bytes.txt.gz'))
