"""The stereo, sequence and association kernels at the largest shapes their entries accept, against their oracles.

The decode's object tables reach O = max_objects = 64 objects of P = 1 + sum(keypoint_config) = 64 keypoints, and the
track solve V = 64 views. At those sizes the kernels run code that small scenes never reach: bits 32..63 of the greedy
step's used masks (okp_greedy_match) and of the robust solve's view mask, lane loops in which a lane owns two objects
or two matches, the opt-in to more than 48 KB of dynamic shared memory, and track grids of several x-blocks per group.

The inputs are fabricated decode tables: 3D objects projected into each view (camera.project), each view's own lift in
kp_point. Every keypoint that competes with another one -- the centres of a frame's objects, the slots of one type of
one object -- lies on its own image row, ROW_PX apart, and the epipolar gate is GATE_PX: only the true partner is within
reach unless a case plants a duplicate, which makes an exact tie. Each case plants the situations of the list in
_stereo_tables / _sequence_tables / _association_inputs / _robust_inputs, and a CPU test checks that the oracle's
output shows every one of them, so that the GPU comparison cannot quietly lose one. The oracle of each case is computed
once per module (the stereo oracle triangulates every matched keypoint with the Hartley-Sturm correction, which is the
bulk of this file's run time).

Comparison rules are those of the per-entry test files: stereo tables bit-equal but for object_cost (rtol 1e-9) and
the points (TOL_METRES_REL, NaN in the same places); sequence matches, tracks, masks and drop counts bit-equal; robust
DLT masks and drop counts bit-equal, X within 1e-7 relative, err only where the solve defines it."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import TOL_METRES_REL
from object_keypoints_b200 import _abi, _lib

gpu = pytest.mark.gpu
ROW_PX = 2.0                       # undistorted rows of competing keypoints are this far apart ...
GATE_PX = 0.5                      # ... so that only the true partner is within this epipolar distance
SMEM_OPT_IN = 48 * 1024
SMEM_MAX = 227 * 1024              # sm_100's per-block opt-in shared memory

# (max_objects, keypoint_config): P = 1 + sum(keypoint_config)
SHAPE_64x64 = (64, (8,) * 7 + (7,))
SHAPE_64x32 = (64, (8, 8, 8, 7))
SHAPE_33x32 = (33, (8, 8, 8, 7))
SHAPE_32x64 = (32, (8,) * 7 + (7,))
STEREO = {
    'epipolar_64x64': ('epipolar', SHAPE_64x64),        # the largest shape the entry accepts
    'epipolar_64x32': ('epipolar', SHAPE_64x32),
    'epipolar_33x32': ('epipolar', SHAPE_33x32),        # one object past a warp's width
    'depth_64x32': ('depth', SHAPE_64x32),              # the largest shapes within 227 KB
    'depth_32x64': ('depth', SHAPE_32x64),
}
# (association, shape, views, max_rounds); None: SequenceTriangulator's default (V)
SEQUENCE = {
    'epipolar_64x32_v8': ('epipolar', SHAPE_64x32, 8, None),
    'depth_64x32_v8': ('depth', SHAPE_64x32, 8, None),
    'epipolar_32x64_v8': ('epipolar', SHAPE_32x64, 8, None),
    'depth_32x64_v8': ('depth', SHAPE_32x64, 8, None),
    'epipolar_4x5_v64': ('epipolar', (4, (3,)), 64, None),
    'epipolar_4x5_v64_no_drops': ('epipolar', (4, (3,)), 64, 0),
    'depth_4x5_v64': ('depth', (4, (3,)), 64, None),
    'depth_4x5_v64_no_drops': ('depth', (4, (3,)), 64, 0),
}
# stereo pairs of the fabricated batch: full, ties and leftovers, an empty left frame, a right frame outside the batch
STEREO_PAIRS = [[0, 1], [2, 3], [4, 1], [0, 5]]
NAN_F = np.array([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 0.0]])   # forward translation, K = I: epipole at (0, 0)
NAN_LEFT, NAN_RIGHT = np.array([[0.0, 0.0], [3.0, 4.0]]), np.array([[6.0, 8.0], [1.0, 1.0]])
_CACHE = {}


def _cached(key, make):
    if key not in _CACHE:
        _CACHE[key] = make()
    return _CACHE[key]


def _full(cfg):
    return [1] + [int(v) for v in cfg]


def _smem(O, C, P):
    """okp_stereo_smem_bytes, okp_stereo_depth_smem_bytes and okp_sequence_smem_bytes (okp_stereo.cuh, okp_sequence.cuh)."""
    stereo = 8 * (4 * O * P + O * O + 64) + 4 * O * P + O * P + O + 2 * O * C
    return {'epipolar': stereo, 'depth': stereo + 8 * 4 * O * P,
            'sequence': 8 * (8 * O * P + O * O + 64) + O * P + O + 2 * O * C}


def _objects(rng, O, cfg, K):
    """[O, P, 3] points in the first camera's frame: keypoint s of type c of object o on undistorted row
    16 + ROW_PX ((o + 8 c + s) mod 64) -- distinct for the centres of all objects and for the slots of one type of one
    object -- at a depth of 0.8 .. 1.6 m."""
    full = _full(cfg)
    Kinv = np.linalg.inv(K)
    X = np.zeros((O, sum(full), 3))
    for o in range(O):
        z = rng.uniform(0.8, 1.6)
        k = 0
        for c, count in enumerate(full):
            for s in range(count):
                row = 16.0 + ROW_PX * ((o + 8 * c + s) % 64)
                X[o, k] = (z + rng.uniform(-0.05, 0.05)) * (Kinv @ np.array([rng.uniform(80.0, 240.0), row, 1.0]))
                k += 1
    return X


def _empty_tables(N, O, cfg):
    full = _full(cfg)
    C, S = len(full), max(full)
    return {'n_objects': np.zeros(N, np.int32), 'kp_count': np.zeros((N, O, C), np.int32),
            'kp_xy': np.zeros((N, O, C, S, 2), np.float32), 'kp_point': np.zeros((N, O, C, S, 3))}


def _fill(t, f, ids, X, T, camera, cfg, rng, last=()):
    """Frame f: the objects X[ids] in this order (n_objects = len(ids), kp_count[:, 0] = 1), seen from T (first camera's
    frame -> this camera), their keypoints of every type in a random slot order. last: (object, type, keypoint) triples
    whose keypoint takes the type's last slot. Slots past a type's count hold a copy of its first keypoint, which only a
    kernel that reads past kp_count would match. -> order[o][c]: the object's keypoint of type c in each slot."""
    full = _full(cfg)
    off = np.cumsum([0] + full[:-1])
    t['n_objects'][f] = len(ids)
    orders = []
    for o, w in enumerate(ids):
        px = camera.project(X[w], T)
        lift = X[w] @ T[:3, :3].T + T[:3, 3]
        per_type = []
        for c, count in enumerate(full):
            order = rng.permutation(count)
            for lw, lc, q in last:
                if (lw, lc) == (w, c):
                    order = np.concatenate([order[order != q], [q]])
            k = off[c] + order
            t['kp_count'][f, o, c] = count
            t['kp_xy'][f, o, c, :count], t['kp_point'][f, o, c, :count] = px[k], lift[k]
            t['kp_xy'][f, o, c, count:], t['kp_point'][f, o, c, count:] = px[k[0]], lift[k[0]]
            per_type.append(order)
        orders.append(per_type)
    return orders


def _slot_of(orders, o, c, q):
    return int(np.nonzero(orders[o][c] == q)[0][0])


# ---------------------------------------------------------------------------------------------------------------------
# Stereo objects
# ---------------------------------------------------------------------------------------------------------------------
def _rig():
    from object_keypoints_b200 import synthetic
    return _cached('rig', lambda: synthetic.stereo_rig((180, 320)))


def _stereo_tables(O, cfg):
    """Five frames of the rig (left, right, left, right, empty left) for STEREO_PAIRS. Planted:
    pair 0: every object on both sides, in two different orders (all O matched: 64 greedy rounds at O = 64), so left and
        right object O - 1 are both matched; n_objects above O on both sides and kp_count above cfg[c] on objects 0..3;
        every type of 8 slots matches all 8; nothing flagged;
    pair 1: left object O - 1 has no partner (index >= 32 where O > 32), left object O - 2 is a copy of left object 3
        (a tie on the smaller left index), the right frame holds a copy of left object 7's partner (a tie on the smaller
        right index; STEREO_AMBIGUOUS) and an object without a left partner; the centres of left object 11 and its
        partner have no lift (STEREO_NO_DEPTH in depth mode);
    pair 2: a left frame without objects; pair 3: a right frame index outside the batch (STEREO_BAD_PAIR)."""
    def make():
        stereo = _rig()
        rng = np.random.default_rng(1000 + O + len(cfg))
        X = _objects(rng, O, cfg, stereo.left_camera.K)
        t = _empty_tables(5, O, cfg)
        eye, T_RL = np.eye(4), stereo.T_RL
        ids = {0: rng.permutation(O), 1: rng.permutation(O), 2: rng.permutation(O)}
        ids[2][O - 2] = ids[2][3]
        gone = ids[2][O - 1]
        right = [w for w in rng.permutation(O) if w != gone]
        right.insert(int(rng.integers(0, len(right))), ids[2][7])
        ids[3] = np.array(right)
        orders = {f: _fill(t, f, ids[f], X, T, camera, cfg, rng)
                  for f, T, camera in ((0, eye, stereo.left_camera), (1, T_RL, stereo.right_camera),
                                       (2, eye, stereo.left_camera), (3, T_RL, stereo.right_camera))}
        t['n_objects'][0], t['n_objects'][1] = O + 6, O + 1
        t['kp_count'][0:2, :4, 1:] += 3
        lifted = ids[2][11]
        t['kp_point'][2, 11, 0, 0] = 0.0
        t['kp_point'][3, int(np.nonzero(ids[3] == lifted)[0][0]), 0, 0] = 0.0
        return {'t': t, 'X': X, 'ids': ids, 'orders': orders}
    return _cached(('stereo_tables', O, cfg), make)


def _stereo_oracle(name):
    def make():
        from oracle import np_oracle, stereo_depth_oracle, stereo_oracle
        association, (O, cfg) = STEREO[name]
        stereo, t = _rig(), _stereo_tables(O, cfg)['t']
        cameras = (np_oracle.camera_dict(stereo.left_camera), np_oracle.camera_dict(stereo.right_camera),
                   stereo.left_camera.K, stereo.right_camera.K, stereo.T_RL, stereo.F)
        pairs = np.array(STEREO_PAIRS)
        if association == 'epipolar':
            return stereo_oracle.stereo_objects(t['n_objects'], t['kp_count'], t['kp_xy'], pairs, cfg, *cameras,
                                                max_distance_px=GATE_PX)
        return stereo_depth_oracle.stereo_objects_depth(t['n_objects'], t['kp_count'], t['kp_xy'], t['kp_point'], pairs, cfg,
                                                        *cameras, max_distance_px=GATE_PX)
    return _cached(('stereo_oracle', name), make)


def _epipolar_costs(F, uL, uR):
    """np_oracle.associate's cost matrix, vectorised: [nL, nR]."""
    l = np.concatenate([uL, np.ones((len(uL), 1))], 1) @ F.T
    m = np.concatenate([uR, np.ones((len(uR), 1))], 1) @ F
    r = np.abs(np.concatenate([uR, np.ones((len(uR), 1))], 1) @ l.T).T
    return 0.5 * (r / np.hypot(l[:, 0], l[:, 1])[:, None] + r / np.hypot(m[:, 0], m[:, 1])[None, :])


@pytest.mark.parametrize('O,cfg', [SHAPE_64x64, SHAPE_64x32, SHAPE_33x32, SHAPE_32x64])
def test_stereo_construction_keeps_candidates_apart(O, cfg):
    """Pair 0: the true partners' epipolar costs are rounding noise and every other candidate, centres and the slots of
    each type, is more than twice the gate away -- only the planted duplicates make ties."""
    from oracle import np_oracle
    stereo, scene = _rig(), _stereo_tables(O, cfg)
    t, ids, orders = scene['t'], scene['ids'], scene['orders']
    cams = [np_oracle.camera_dict(c) for c in (stereo.left_camera, stereo.right_camera)]
    und = [np.array([[np_oracle.undistort_point(float(x), float(y), cams[v]) for x, y in t['kp_xy'][v, o, 0, :1]]
                     for o in range(O)]).reshape(O, 2) for v in (0, 1)]
    partner = np.array([int(np.nonzero(ids[1] == w)[0][0]) for w in ids[0]])
    cost = _epipolar_costs(stereo.F, und[0], und[1])
    truth = np.zeros_like(cost, bool)
    truth[np.arange(O), partner] = True
    worst, nearest = cost[truth].max(), cost[~truth].min()
    for o in range(0, O, 7):
        j = partner[o]
        for c, count in enumerate(_full(cfg)[1:], 1):
            ul = np.array([np_oracle.undistort_point(float(x), float(y), cams[0]) for x, y in t['kp_xy'][0, o, c, :count]])
            ur = np.array([np_oracle.undistort_point(float(x), float(y), cams[1]) for x, y in t['kp_xy'][1, j, c, :count]])
            slots = _epipolar_costs(stereo.F, ul, ur)
            match = orders[0][o][c][:, None] == orders[1][j][c][None, :]
            worst, nearest = max(worst, slots[match].max()), min(nearest, slots[~match].min())
    assert worst < 1e-3 and nearest > 2 * GATE_PX, (worst, nearest)


@pytest.mark.parametrize('name', list(STEREO))
def test_stereo_oracle_shows_every_planted_situation(name):
    association, (O, cfg) = STEREO[name]
    scene, want = _stereo_tables(O, cfg), _stereo_oracle(name)
    ids, orders = scene['ids'], scene['orders']
    match = want['object_match']
    # pair 0: all O matched both ways, n_objects and kp_count clamped, types of 8 slots fully matched, nothing flagged
    assert (match[0] >= 0).all() and sorted(match[0]) == list(range(O))
    assert scene['t']['n_objects'][0] > O and scene['t']['n_objects'][1] > O and (scene['t']['kp_count'][0, 0, 1:] > cfg).all()
    for c, count in enumerate(cfg, 1):
        assert ((want['slot_match'][0, :, c] >= 0).sum(axis=1) == count).all()
        if count == 8:
            assert (want['slot_match'][0, :, c, :8] >= 0).all()
    assert want['flags'][0] == 0
    # pair 1: the unmatched left objects (one at index >= 32 where O > 32), the ties, the flags
    assert match[1, O - 1] == -1 and match[1, O - 2] == -1 and (O <= 32 or O - 1 >= 32)
    partner = {w: [int(j) for j in np.nonzero(ids[3] == w)[0]] for w in ids[2]}
    assert match[1, 3] == partner[ids[2][3]][0]                   # left 3 and its copy O - 2: the smaller left index
    assert len(partner[ids[2][7]]) == 2 and match[1, 7] == min(partner[ids[2][7]])   # the smaller right index
    assert want['flags'][1] & _abi.STEREO_AMBIGUOUS
    if association == 'depth':
        assert want['flags'][1] & _abi.STEREO_NO_DEPTH and match[1, 11] == -1
        assert (want['flags'][[0, 2]] & _abi.STEREO_NO_DEPTH == 0).all()
    else:
        assert match[1, 11] == partner[ids[2][11]][0]
    assert (match[2] == -1).all() and want['flags'][2] == 0
    assert (match[3] == -1).all() and want['flags'][3] == _abi.STEREO_BAD_PAIR
    # the pairs' matches are the construction's
    for i, w in enumerate(ids[0]):
        j = int(np.nonzero(ids[1] == w)[0][0])
        assert match[0, i] == j
        for c, count in enumerate(cfg, 1):
            q = orders[0][i][c]
            np.testing.assert_array_equal(want['slot_match'][0, i, c, :count],
                                          [_slot_of(orders[1], j, c, k) for k in q])


@pytest.mark.parametrize('O,cfg', [SHAPE_64x32, SHAPE_32x64])
def test_depth_oracle_recovers_the_construction(O, cfg):
    """Noiseless tables: pair 0's matches are the construction's permutation and its points are the construction's."""
    name = next(k for k, (a, shape) in STEREO.items() if a == 'depth' and shape == (O, cfg))
    scene, want = _stereo_tables(O, cfg), _stereo_oracle(name)
    off = np.cumsum([0] + _full(cfg)[:-1])
    for i, w in enumerate(scene['ids'][0]):
        assert scene['ids'][1][want['object_match'][0, i]] == w
        for c, count in enumerate(_full(cfg)):
            q = scene['orders'][0][i][c]
            X = scene['X'][w, off[c] + q]
            got = want['point'][0, i, c, :count]
            assert (np.linalg.norm(got - X, axis=1) / np.linalg.norm(X, axis=1)).max() < 1e-4


def test_largest_cases_opt_in_to_more_than_48_kb():
    """Every case at a largest shape needs the dynamic shared-memory opt-in above 48 KB and fits 227 KB; the 33-object
    case and the 64-view one (O = 4) stay below 48 KB."""
    for association, shape in STEREO.values():
        O, cfg = shape
        need = _smem(O, len(cfg) + 1, sum(_full(cfg)))[association]
        assert need <= SMEM_MAX and (need > SMEM_OPT_IN) == (shape != SHAPE_33x32), (association, shape, need)
    assert _smem(64, 9, 64)['epipolar'] == 186048
    for association, (O, cfg), V, _ in SEQUENCE.values():
        need = _smem(O, len(cfg) + 1, sum(_full(cfg)))['sequence']
        assert need <= SMEM_MAX and (need > SMEM_OPT_IN) == (O > 4), (association, O, cfg, need)


def _stereo_run(name):
    """The case on the device through the C entry (the pairs unchecked, a frame index outside the batch included), every
    output prefilled with 7 so that an entry the kernel leaves unwritten shows."""
    from object_keypoints_b200 import DecodeTables, StereoTables
    association, (O, cfg) = STEREO[name]
    stereo, t = _rig(), _stereo_tables(O, cfg)['t']
    tables = DecodeTables(len(t['n_objects']), len(cfg) + 1, list(cfg), _abi.make_params(max_objects=O, compat_clip_bug=False),
                          'cuda')
    for key, value in t.items():
        tables[key].copy_(torch.from_numpy(value))
    pairs = torch.tensor(STEREO_PAIRS, dtype=torch.int32, device='cuda')
    out = StereoTables(len(STEREO_PAIRS), O, tables.C, max(cfg), 'cuda')
    for tensor in out.tensors.values():
        tensor.fill_(7)
    d = ctypes.POINTER(ctypes.c_double)
    F, P_L, P_R = (np.ascontiguousarray(m, dtype=np.float64) for m in (stereo.F, *stereo.projection_matrices()))
    head = (ctypes.byref(tables.struct), tables.N, tables.C, (ctypes.c_int32 * len(cfg))(*cfg), ctypes.byref(tables.params),
            pairs.data_ptr(), len(STEREO_PAIRS), ctypes.byref(_abi.pack_camera(stereo.left_camera)),
            ctypes.byref(_abi.pack_camera(stereo.right_camera)), F.ctypes.data_as(d), P_L.ctypes.data_as(d), P_R.ctypes.data_as(d))
    if association == 'depth':
        T_RL = np.ascontiguousarray(stereo.T_RL, dtype=np.float64).reshape(16)
        rc = _lib.lib().okp_triangulate_stereo_objects_depth_f64(*head, T_RL.ctypes.data_as(d), GATE_PX, 8.0, 1,
                                                                 ctypes.byref(out.struct), None)
    else:
        rc = _lib.lib().okp_triangulate_stereo_objects_f64(*head, GATE_PX, 1, ctypes.byref(out.struct), None)
    _lib.check(rc, name)
    return out.numpy()


def _relative(got, want):
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want[..., 0])
    if not ok.any():
        return 0.0
    return float((np.linalg.norm(got[ok] - want[ok], axis=-1) / np.linalg.norm(want[ok], axis=-1)).max())


@gpu
@pytest.mark.parametrize('name', list(STEREO))
def test_stereo_objects_are_the_oracle_at_the_largest_shapes(name):
    got, want = _stereo_run(name), _stereo_oracle(name)
    for key in ('object_match', 'slot_match', 'flags'):
        np.testing.assert_array_equal(got[key], want[key], err_msg=f"{name} {key}")
    np.testing.assert_allclose(got['object_cost'], want['object_cost'], rtol=1e-9, atol=1e-12, err_msg=name)
    deviation = _relative(got['point'], want['point'])
    assert deviation <= TOL_METRES_REL, (name, deviation)


# ---------------------------------------------------------------------------------------------------------------------
# Sequence objects
# ---------------------------------------------------------------------------------------------------------------------
def _sequence_tables(O, cfg, V):
    """N = 2 V frames of one camera moving along its x axis (two anchors, frames[a, v] = a + 2 v): undistorted rows are the
    same in every frame, so the construction's rows keep the candidates apart under every pair's F. Planted (anchor 0
    unless said otherwise; wherever the shape has the objects or slots):
      view 1 lacks the anchor's object O - 1 (index >= 32 where O > 32); view 2 has every object (all O matched);
      view 3 has n_objects above O and kp_count above cfg[c]; anchor 1's view 1 holds a copy of its object 7 mod O
      (an exact tie on the smaller index; STEREO_AMBIGUOUS); anchor 1's view 2 has no objects; anchor 1's last view is a
      frame outside the batch (STEREO_BAD_PAIR);
      the anchor's centre of object 5 mod O has no lift, nor has its partner in view 4 (STEREO_NO_DEPTH there only);
      keypoint 0 of type 1 of the anchor's object 0 is 0.06 m off along x in view 5 (V = 8) or 40 (V = 64): same row,
      matched, then dropped by the robust solve (a view index > 31 at V = 64);
      keypoint cfg[0] - 1 of type 1 of the anchor's object 1 is missing in views 1 .. V - 2: its track has two views,
      0 and V - 1 (63 at V = 64).
    -> dict of the tables, the construction, T_CW [N, 4, 4] and the frames of the objects call (frames_i32)."""
    def make():
        from object_keypoints_b200 import sequence, synthetic
        camera = synthetic.default_camera((180, 320))
        rng = np.random.default_rng(2000 + O + V)
        N = 2 * V
        X = _objects(rng, O, cfg, camera.K)
        T_CW = np.tile(np.eye(4), (N, 1, 1))
        T_CW[:, 0, 3] = -0.15 * np.arange(N) / (N - 1)
        frames = sequence.view_schedule(N, V)
        t = _empty_tables(N, O, cfg)
        ids = {f: rng.permutation(O) for f in range(N)}
        a0 = ids[frames[0, 0]]
        ids[frames[0, 1]] = np.array([w for w in ids[frames[0, 1]] if w != a0[O - 1]])
        twin = ids[frames[1, 0]][7 % O]
        view = [w for w in ids[frames[1, 1]] if w != ids[frames[1, 0]][(7 % O) - 1]]
        view.insert(int(rng.integers(0, len(view))), twin)
        ids[frames[1, 1]] = np.array(view)
        ids[frames[1, 2]] = np.zeros(0, int)
        outlier_view = 5 if V == 8 else 40
        short = (a0[1], 1, cfg[0] - 1)
        orders = {}
        for f in range(N):
            in_short = f in frames[0, 1:V - 1]
            orders[f] = _fill(t, f, ids[f], X, T_CW[f], camera, cfg, rng, last=[short] if in_short else ())
            if in_short:
                t['kp_count'][f, int(np.nonzero(ids[f] == short[0])[0][0]), 1] -= 1
        f = frames[0, outlier_view]
        o = int(np.nonzero(ids[f] == a0[0])[0][0])
        s = _slot_of(orders[f], o, 1, 0)
        t['kp_xy'][f, o, 1, s] = camera.project(X[a0[0], 1:2] + np.array([0.06, 0.0, 0.0]), T_CW[f])[0]
        t['n_objects'][frames[0, 3]] = O + 2
        t['kp_count'][frames[0, 3], :2, 1:] += 3
        w = a0[5 % O]
        for f in (frames[0, 0], frames[0, 4]):
            t['kp_point'][f, int(np.nonzero(ids[f] == w)[0][0]), 0, 0] = 0.0
        frames_i32 = frames.astype(np.int32)
        frames_i32[1, V - 1] = N
        return {'t': t, 'X': X, 'ids': ids, 'orders': orders, 'T_CW': T_CW, 'camera': camera, 'frames': frames_i32,
                'outlier_view': outlier_view, 'short': short}
    return _cached(('sequence_tables', O, cfg, V), make)


def _sequence_prepared(O, cfg, V, device):
    from object_keypoints_b200 import sequence
    scene = _sequence_tables(O, cfg, V)
    chain = sequence.SequenceTriangulator.__new__(sequence.SequenceTriangulator)
    chain.camera, chain.views, chain.device = scene['camera'], V, torch.device(device)
    prepared = chain.prepare(scene['T_CW'])
    prepared['frames_i32'] = torch.from_numpy(scene['frames']).to(device)
    return prepared


def _sequence_oracle(name):
    def make():
        from oracle import sequence_objects_oracle
        association, (O, cfg), V, rounds = SEQUENCE[name]
        scene = _sequence_tables(O, cfg, V)
        prepared = {k: (v.numpy() if torch.is_tensor(v) else v) for k, v in _sequence_prepared(O, cfg, V, 'cpu').items()}
        t = scene['t']
        return sequence_objects_oracle.sequence_objects(t['n_objects'], t['kp_count'], t['kp_xy'], t['kp_point'], cfg,
                                                        scene['frames'], prepared['F'], prepared['motion'], prepared['poses'],
                                                        scene['camera'], association=association, max_distance_px=GATE_PX,
                                                        max_rounds=rounds)
    return _cached(('sequence_oracle', name), make)


@pytest.mark.parametrize('name', list(SEQUENCE))
def test_sequence_oracle_shows_every_planted_situation(name):
    association, (O, cfg), V, rounds = SEQUENCE[name]
    scene, want = _sequence_tables(O, cfg, V), _sequence_oracle(name)
    ids, orders, frames, t = scene['ids'], scene['orders'], scene['frames'], scene['t']
    a0 = ids[frames[0, 0]]
    match, flags = want['object_match'], want['flags']
    assert match[0, 0, O - 1] == -1 and (O <= 32 or O - 1 >= 32)                    # view 1 lacks object O - 1
    assert (match[0, 1] >= 0).all()                                                # view 2: all O matched
    if O == 64:
        assert match[0, 1, 63] >= 0 and (match[0, 1] == 63).any()
    for c, count in enumerate(cfg, 1):
        if count == 8:
            assert ((want['slot_match'][0, 1, 2:, c] >= 0).sum(axis=-1) == 8).all()
    assert t['n_objects'][frames[0, 3]] > O and (t['kp_count'][frames[0, 3], 0, 1:] > cfg).all()
    assert (match[0, 2, :O] >= 0).sum() == O                                       # view 3: clamped, all matched
    twin = ids[frames[1, 0]][7 % O]
    at = np.nonzero(ids[frames[1, 1]] == twin)[0]
    assert len(at) == 2 and match[1, 0, 7 % O] == at.min() and flags[1, 0] & _abi.STEREO_AMBIGUOUS
    assert not (flags[0, :] & _abi.STEREO_AMBIGUOUS).any()
    assert (match[1, 1] == -1).all() and flags[1, 1] == 0                           # anchor 1's empty view 2
    assert flags[1, V - 2] == _abi.STEREO_BAD_PAIR and (match[1, V - 2] == -1).all()
    if association == 'depth':
        no_depth = (flags[0] & _abi.STEREO_NO_DEPTH) != 0
        assert no_depth[3] and no_depth.sum() == 1 and match[0, 3, 5 % O] == -1
    # the outlier: matched, then dropped by the robust solve unless max_rounds is 0
    v_out = scene['outlier_view']
    s = _slot_of(orders[frames[0, 0]], 0, 1, 0)
    assert want['observed'][0, 0, 1, s, v_out] == 1
    if rounds == 0:
        assert want['valid'][0, 0, 1, s, v_out] == 1 and (want['dropped'] == 0).all()
    else:
        assert want['valid'][0, 0, 1, s, v_out] == 0 and want['dropped'][0, 0, 1, s] >= 1
        assert V < 64 or v_out > 31
    # the two-view track ending in view V - 1
    w, c, q = scene['short']
    o = int(np.nonzero(a0 == w)[0][0])
    s = _slot_of(orders[frames[0, 0]], o, c, q)
    np.testing.assert_array_equal(np.nonzero(want['observed'][0, o, c, s])[0], [0, V - 1])
    assert np.isfinite(want['point'][0, o, c, s]).all()


@gpu
@pytest.mark.parametrize('name', list(SEQUENCE))
def test_sequence_objects_are_the_oracle_at_the_largest_shapes(name):
    from object_keypoints_b200 import DecodeTables, sequence
    association, (O, cfg), V, rounds = SEQUENCE[name]
    scene, want = _sequence_tables(O, cfg, V), _sequence_oracle(name)
    t = scene['t']
    tables = DecodeTables(len(t['n_objects']), len(cfg) + 1, list(cfg), _abi.make_params(max_objects=O, compat_clip_bug=False),
                          'cuda')
    for key, value in t.items():
        tables[key].copy_(torch.from_numpy(value))
    chain = sequence.SequenceTriangulator(scene['camera'], views=V, max_distance_px=GATE_PX, max_rounds=rounds)
    got = chain.objects(tables, _sequence_prepared(O, cfg, V, 'cuda'), association=association).numpy()
    for key in ('object_match', 'slot_match', 'flags', 'observations', 'observed', 'valid', 'dropped'):
        np.testing.assert_array_equal(got[key], want[key], err_msg=f"{name} {key}")
    np.testing.assert_allclose(got['object_cost'], want['object_cost'], rtol=1e-9, atol=1e-12, err_msg=name)
    deviation = _relative(got['point'], want['point'])
    assert deviation <= TOL_METRES_REL, (name, deviation)
    assert np.array_equal(np.isnan(got['error']), np.isnan(want['error'])), name
    solved = ~np.isnan(want['error'])
    assert np.abs(got['error'][solved] - want['error'][solved]).max(initial=0.0) < 1e-6, name


# ---------------------------------------------------------------------------------------------------------------------
# Association
# ---------------------------------------------------------------------------------------------------------------------
ASSOCIATION_COUNTS = [(64, 64), (0, 64), (1, 64), (63, 64), (70, 99), (64, 64), (64, 63)]


def _association_inputs():
    """B = 7 pairs of 64 x 64 undistorted points of the rig (left point i on row 16 + ROW_PX i, the right points their
    partners in a random order) with the counts of ASSOCIATION_COUNTS: all 64 matched (left and right 63 among them),
    none, one, 63, counts above 64 (clamped), then pair 5, whose right partner of left 40 is replaced by a copy of left
    10's (a tie on the smaller right index; left 40 unmatched), and pair 6, whose left 50 is a copy of left 20 (a tie on
    the smaller left index)."""
    def make():
        stereo = _rig()
        rng = np.random.default_rng(77)
        B, M = len(ASSOCIATION_COUNTS), 64
        R_, t_ = stereo.T_RL[:3, :3], stereo.T_RL[:3, 3]
        L, R, perms = np.zeros((B, M, 2)), np.zeros((B, M, 2)), []
        for b in range(B):
            X = _objects(rng, M, (), stereo.left_camera.K)[:, 0]
            L[b] = X[:, :2] / X[:, 2:] * np.diag(stereo.left_camera.K)[:2] + stereo.left_camera.K[:2, 2]
            Y = X @ R_.T + t_
            perm = rng.permutation(M)
            R[b, perm] = Y[:, :2] / Y[:, 2:] * np.diag(stereo.right_camera.K)[:2] + stereo.right_camera.K[:2, 2]
            perms.append(perm)
        R[5, perms[5][40]] = R[5, perms[5][10]]
        L[6, 50] = L[6, 20]
        n = np.array(ASSOCIATION_COUNTS, np.int32)
        return {'F': stereo.F, 'left': L, 'right': R, 'n_left': n[:, 0].copy(), 'n_right': n[:, 1].copy(), 'perms': perms}
    return _cached('association', make)


def _association_oracle():
    def make():
        from oracle import np_oracle
        a = _association_inputs()
        match, cost = np.full((len(a['n_left']), 64), -1, np.int32), np.zeros((len(a['n_left']), 64))
        for b in range(len(a['n_left'])):
            nl, nr = min(int(a['n_left'][b]), 64), min(int(a['n_right'][b]), 64)
            match[b, :nl], cost[b, :nl] = np_oracle.associate(a['F'], a['left'][b, :nl], a['right'][b, :nr], GATE_PX)
        return match, cost
    return _cached('association_oracle', make)


def test_association_oracle_shows_every_planted_situation():
    a = _association_inputs()
    match, _ = _association_oracle()
    perms = a['perms']
    np.testing.assert_array_equal(match[0], perms[0])
    assert match[0, 63] >= 0 and (match[0] == 63).any()
    assert (match[1] == -1).all() and match[2, 0] == perms[2][0] and (match[2, 1:] == -1).all()
    np.testing.assert_array_equal(match[3, :63], perms[3][:63])
    assert match[3, 63] == -1
    np.testing.assert_array_equal(match[4], perms[4])                                 # 70 x 99, clamped to 64 x 64
    assert match[5, 40] == -1 and match[5, 10] == min(perms[5][10], perms[5][40])
    assert match[6, 20] == perms[6][20] and match[6, 50] == -1
    missing = int(np.nonzero(perms[6] == 63)[0][0])                                 # pair 6: right point 63 left out
    assert match[6, missing] == -1 or missing == 50


def test_associate_oracle_skips_a_nan_cost():
    """A left point at the left epipole: l = F x = 0, so its costs are 0 / 0. They are not admissible, like costs above
    the gate, and the other candidates are still matched: left 1 -> right 0 at cost 0 (the kernel's rule)."""
    from oracle import np_oracle, stereo_depth_oracle
    with np.errstate(invalid='ignore'):
        match, cost = np_oracle.associate(NAN_F, NAN_LEFT, NAN_RIGHT, 2.5)
    np.testing.assert_array_equal(match, [-1, 0])
    np.testing.assert_array_equal(cost, [0.0, 0.0])
    match, cost = stereo_depth_oracle._greedy(np.array([[np.nan, np.nan], [0.0, 0.5 * (0.2 + 1 / np.sqrt(2))]]), 2.5)
    np.testing.assert_array_equal(match, [-1, 0])
    match, _ = stereo_depth_oracle._greedy(np.array([[np.nan, 1.0], [0.5, np.nan]]), 2.5)
    np.testing.assert_array_equal(match, [1, 0])


def _assert_association(got_match, got_cost, want_match, want_cost, what):
    np.testing.assert_array_equal(got_match, want_match, err_msg=what)
    np.testing.assert_allclose(got_cost, want_cost, rtol=1e-9, atol=1e-12, err_msg=what)


def _associate_call(entry, F, left, right, n_left, n_right, max_distance):
    """One call of okp_stereo_associate_f64 (F: [3, 3]) or okp_associate_pairs_f64 (F: [B, 3, 3] on the device) with the
    outputs prefilled with 7."""
    B, ML, MR = left.shape[0], left.shape[1], right.shape[1]
    dev = lambda a, dtype: torch.from_numpy(np.ascontiguousarray(a)).to('cuda', dtype)          # noqa: E731
    L, R = dev(left, torch.float64), dev(right, torch.float64)
    nl, nr = dev(n_left, torch.int32), dev(n_right, torch.int32)
    match = torch.full((B, ML), 7, dtype=torch.int32, device='cuda')
    cost = torch.full((B, ML), 7.0, dtype=torch.float64, device='cuda')
    if entry == 'one_f':
        Fm = np.ascontiguousarray(F, dtype=np.float64).reshape(9)
        rc = _lib.lib().okp_stereo_associate_f64(Fm.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), L.data_ptr(), nl.data_ptr(),
                                                 R.data_ptr(), nr.data_ptr(), B, ML, MR, max_distance, match.data_ptr(),
                                                 cost.data_ptr(), None)
    else:
        Fd = dev(F, torch.float64)
        rc = _lib.lib().okp_associate_pairs_f64(Fd.data_ptr(), L.data_ptr(), nl.data_ptr(), R.data_ptr(), nr.data_ptr(), B, ML,
                                                MR, max_distance, match.data_ptr(), cost.data_ptr(), None)
    _lib.check(rc, entry)
    return match.cpu().numpy(), cost.cpu().numpy()


@gpu
@pytest.mark.parametrize('entry', ['one_f', 'per_pair'])
def test_association_is_the_oracle_at_64_x_64(entry):
    a = _association_inputs()
    want_match, want_cost = _association_oracle()
    B = len(a['n_left'])
    F = a['F'] if entry == 'one_f' else np.broadcast_to(a['F'], (B, 3, 3))
    got = _associate_call(entry, F, a['left'], a['right'], a['n_left'], a['n_right'], GATE_PX)
    _assert_association(*got, want_match, want_cost, entry)


@gpu
@pytest.mark.parametrize('entry', ['one_f', 'per_pair'])
def test_association_skips_a_nan_cost(entry):
    """The NaN reproduction as its own call and, per pair, beside a full 64 x 64 pair of the rig."""
    from oracle import np_oracle
    a = _association_inputs()
    left, right = np.zeros((2, 64, 2)), np.zeros((2, 64, 2))
    left[0], right[0] = a['left'][0], a['right'][0]
    left[1, :2], right[1, :2] = NAN_LEFT, NAN_RIGHT
    n_left, n_right = np.array([64, 2], np.int32), np.array([64, 2], np.int32)
    want_match, want_cost = np.full((2, 64), -1, np.int32), np.zeros((2, 64))
    want_match[0], want_cost[0] = np_oracle.associate(a['F'], left[0], right[0], 2.5)
    with np.errstate(invalid='ignore'):
        want_match[1, :2], want_cost[1, :2] = np_oracle.associate(NAN_F, NAN_LEFT, NAN_RIGHT, 2.5)
    assert want_match[1, :2].tolist() == [-1, 0] and (want_match[0] >= 0).all()
    if entry == 'one_f':
        got = _associate_call(entry, NAN_F, left[1:], right[1:], n_left[1:], n_right[1:], 2.5)
        _assert_association(*got, want_match[1:], want_cost[1:], entry)
    else:
        got = _associate_call(entry, np.stack([a['F'], NAN_F]), left, right, n_left, n_right, 2.5)
        _assert_association(*got, want_match, want_cost, entry)


# ---------------------------------------------------------------------------------------------------------------------
# Robust V-view DLT and the tracks entry
# ---------------------------------------------------------------------------------------------------------------------
V_MAX = 64
TRACK_GROUPS = {'pg20': (3, 20), 'pg200': (3, 200)}


def _robust_camera():
    from object_keypoints_b200 import synthetic
    return _cached('robust_camera', lambda: synthetic.default_camera((180, 320)).scale(4.0))


def _robust_inputs(P, seed):
    """P points seen from 64 poses (0.3 px noise) with gross outliers (+-20 px) in 20 % of the views >= 32. Planted:
    point 0 has a NaN observation in view 63, a valid view: X and every error are NaN, so views are dropped in index
    order until two remain (62 and 63) and X stays NaN; point 4 has one in view 40: views 0 .. 40 are dropped, then the
    solve is finite; point 1 has two valid views, 7 and 63; point 2 only view 63 (no solve, err unwritten); point 3 an
    outlier in view 63 only; every other point all 64 views valid. -> obs [P, V, 2], valid [P, V] uint8, poses [V, 4, 4]."""
    from scipy.spatial.transform import Rotation
    camera = _robust_camera()
    rng = np.random.default_rng(seed)
    X = np.stack([rng.uniform(-0.3, 0.3, P), rng.uniform(-0.2, 0.2, P), rng.uniform(-0.05, 0.05, P)], axis=1)
    poses = np.zeros((V_MAX, 4, 4))
    for v in range(V_MAX):
        R = Rotation.from_rotvec(rng.normal(0, 0.25, 3)).as_matrix()
        poses[v] = np.eye(4)
        poses[v, :3, :3] = R
        poses[v, :3, 3] = -R @ np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3), -rng.uniform(0.6, 1.0)])
    obs = np.stack([camera.project(X, poses[v]) for v in range(V_MAX)], axis=1) + rng.normal(0, 0.3, (P, V_MAX, 2))
    outliers = np.zeros((P, V_MAX), bool)
    outliers[:, 32:] = rng.uniform(size=(P, V_MAX - 32)) < 0.2
    outliers[:5] = False
    outliers[3, 63] = True
    obs[outliers] += rng.choice([-20.0, 20.0], (int(outliers.sum()), 2))
    valid = np.ones((P, V_MAX), np.uint8)
    obs[0, 63] = np.nan
    obs[4, 40] = np.nan
    valid[1] = 0
    valid[1, [7, 63]] = 1
    valid[2] = 0
    valid[2, 63] = 1
    return obs, valid, poses


def _robust_oracle(obs, valid, poses, rounds=V_MAX):
    from oracle import c_oracle
    X, mask, err, dropped = c_oracle.triangulate_robust(obs, valid, poses, _robust_camera(), 2.0, rounds)
    err[valid.sum(axis=1) < 2] = np.nan                          # no solve: no error
    return X, mask, err, dropped


def _assert_robust(got, want, solved, what):
    """solved: the points that start with two or more valid views (the others' err is left unwritten)."""
    X, mask, err, dropped = got
    np.testing.assert_array_equal(mask, want[1], err_msg=what)
    np.testing.assert_array_equal(dropped, want[3], err_msg=what)
    assert np.array_equal(np.isnan(X), np.isnan(want[0])), what
    ok = ~np.isnan(want[0][:, 0])
    assert (np.linalg.norm(X[ok] - want[0][ok], axis=1) <= 1e-7 * np.linalg.norm(want[0][ok], axis=1) + 1e-10).all(), what
    np.testing.assert_allclose(err[solved], want[2][solved], rtol=0, atol=1e-6, err_msg=what)


def test_robust_oracle_shows_every_planted_situation():
    obs, valid, poses = _robust_inputs(40, 64)
    X, mask, err, dropped = _cached('robust_oracle', lambda: _robust_oracle(obs, valid, poses))
    assert np.isnan(X[0]).all() and mask[0].sum() == 2 and dropped[0] == V_MAX - 2 and np.isnan(err[0]).all()
    np.testing.assert_array_equal(np.nonzero(mask[0])[0], [62, 63])                  # dropped in index order
    np.testing.assert_array_equal(np.nonzero(mask[1])[0], [7, 63])
    assert np.isfinite(X[1]).all()
    assert np.isnan(X[2]).all() and mask[2].sum() == 1
    assert mask[3, 63] == 0 and dropped[3] == 1
    assert dropped[4] >= 41 and (mask[4, :41] == 0).all() and np.isfinite(X[4]).all()
    assert (~mask[5:].astype(bool) & valid[5:].astype(bool))[:, 32:].any()              # outliers >= 32 dropped
    assert np.isfinite(X[3:]).all() and (dropped[5:] >= 1).any()


@gpu
def test_triangulate_multiview_is_the_oracle_at_64_views():
    from object_keypoints_b200 import triangulate_multiview
    obs, valid, poses = _robust_inputs(40, 64)
    want = _cached('robust_oracle', lambda: _robust_oracle(obs, valid, poses))
    got = triangulate_multiview(obs, valid, poses, _robust_camera(), max_error_px=2.0, return_dropped=True)
    _assert_robust([g.cpu().numpy() for g in got], want, valid.sum(axis=1) >= 2, 'triangulate_multiview')


def _tracks_inputs(name):
    def make():
        G, Pg = TRACK_GROUPS[name]
        parts = [_robust_inputs(Pg, 300 + 10 * g + Pg) for g in range(G)]
        obs, valid, poses = (np.stack([p[i] for p in parts]) for i in range(3))
        return obs, valid, poses
    return _cached(('tracks_inputs', name), make)


def _tracks_oracle(name):
    def make():
        obs, valid, poses = _tracks_inputs(name)
        groups = [_robust_oracle(obs[g], valid[g], poses[g]) for g in range(len(obs))]
        return [np.stack([r[i] for r in groups]) for i in range(4)]
    return _cached(('tracks_oracle', name), make)


@pytest.mark.parametrize('name', list(TRACK_GROUPS))
def test_tracks_oracle_shows_every_planted_situation(name):
    X, mask, _, dropped = _tracks_oracle(name)
    G, Pg = TRACK_GROUPS[name]
    assert G >= 3 and (Pg < 32 or Pg > 128)
    assert np.isnan(X[:, 0]).all() and (dropped[:, 0] == V_MAX - 2).all() and (dropped[:, 4] >= 41).all()
    assert (mask[:, 1, 63] == 1).all() and (mask[:, 1].sum(axis=1) == 2).all()
    assert (mask[:, 3, 63] == 0).all()


@gpu
@pytest.mark.parametrize('name', list(TRACK_GROUPS))
def test_tracks_entry_is_the_oracle_at_64_views(name):
    obs, valid, poses = _tracks_inputs(name)
    want = _tracks_oracle(name)
    G, Pg = TRACK_GROUPS[name]
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()          # noqa: E731
    o, v, p = dev(obs), dev(valid), dev(poses)
    X = torch.full((G, Pg, 3), 7.0, dtype=torch.float64, device='cuda')
    err = torch.full((G, Pg, V_MAX), 7.0, dtype=torch.float64, device='cuda')
    dropped = torch.full((G, Pg), 7, dtype=torch.int32, device='cuda')
    rc = _lib.lib().okp_triangulate_tracks_f64(o.data_ptr(), v.data_ptr(), p.data_ptr(), ctypes.byref(_abi.pack_camera(_robust_camera())),
                                               G, Pg, V_MAX, 2.0, V_MAX, X.data_ptr(), err.data_ptr(), dropped.data_ptr(), None)
    _lib.check(rc, 'okp_triangulate_tracks_f64')
    got = [t.cpu().numpy() for t in (X, v, err, dropped)]
    flat = lambda a: a.reshape((G * Pg,) + a.shape[2:])          # noqa: E731
    _assert_robust([flat(g) for g in got], [flat(w) for w in want], flat(valid).sum(axis=1) >= 2, name)
