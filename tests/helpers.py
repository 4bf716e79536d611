"""Shared helpers for the parity tests: golden fixtures and table comparison."""
import hashlib
import json
import os
import types

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
INPUTS = ('heat', 'depth', 'centers')

# tolerances stated by BASELINE.json's north_star
TOL_PIXELS = 1e-3          # 2D sub-pixel positions, px
TOL_METRES_REL = 1e-4      # 3D points, relative


def sha256(array):
    return hashlib.sha256(np.ascontiguousarray(array).tobytes()).hexdigest()


def load_golden(name):
    data = np.load(os.path.join(GOLDEN, name), allow_pickle=False)
    g = {k: data[k] for k in data.files}
    if 'input_recipe' in g:
        g.update(rebuild_inputs(g))
    return g


def rebuild_inputs(g):
    """Fixtures whose inputs came from the seeded generator store the generator call (input_recipe, JSON), the frames
    kept (source_frames) and the SHA-256 of each input array instead of the maps themselves: the maps are noise-like
    and would not fit a small file. They are rebuilt here and must hash to the stored digests, so the reference
    tables are always compared on exactly the inputs the reference saw."""
    from object_keypoints_b200 import synthetic
    recipe = json.loads(str(g['input_recipe']))
    batch = getattr(synthetic, recipe['generator'])(**recipe['args'])
    inputs = {k: getattr(batch, k)[g['source_frames']] for k in INPUTS}
    for k in INPUTS:
        assert sha256(inputs[k]) == str(g['sha256_' + k]), \
            f"synthetic.{recipe['generator']}{recipe['args']} no longer reproduces the fixture's {k}"
    return inputs


def golden_camera(g, prefix='cam_'):
    """Rebuild a camera object from the K/D/image_size stored in a fixture."""
    from object_keypoints_b200 import camera_utils
    return camera_utils.FisheyeCamera(g[prefix + 'K'], g[prefix + 'D'], g[prefix + 'image_size'])


def reference_tables(g):
    return {k[4:]: v for k, v in g.items() if k.startswith('ref_')}


def assert_tables_match(got, ref, exact_assignment=True, check_points=True, frames=None):
    """got: tables from the oracle or the CUDA path; ref: tables from the reference.

    Bit-exact: peak pixel indices, raster order, object count, assignments, kept keypoints.
    Tolerance: sub-pixel positions <= 1e-3 px, 3D points <= 1e-4 relative."""
    N, C, K = ref['peak_count'].shape[0], ref['peak_count'].shape[1], ref['peak_yx'].shape[2]
    frames = range(N) if frames is None else frames
    for n in frames:
        np.testing.assert_array_equal(got['peak_count'][n], ref['peak_count'][n], err_msg=f"frame {n} peak counts")
        for c in range(C):
            k = int(ref['peak_count'][n, c])
            np.testing.assert_array_equal(got['peak_yx'][n, c, :k], ref['peak_yx'][n, c, :k],
                                          err_msg=f"frame {n} map {c} peak pixels")
            np.testing.assert_array_equal(got['peak_score'][n, c, :k], ref['peak_score'][n, c, :k],
                                          err_msg=f"frame {n} map {c} box sums (bitwise)")
            assert np.abs(got['peak_xy'][n, c, :k] - ref['peak_xy'][n, c, :k]).max(initial=0) <= TOL_PIXELS
            np.testing.assert_allclose(got['peak_conf'][n, c, :k], ref['peak_conf'][n, c, :k], rtol=1e-5)
        assert got['n_objects'][n] == ref['n_objects'][n], f"frame {n} object count"
        if exact_assignment:
            for c in range(C):
                k = int(ref['peak_count'][n, c])
                np.testing.assert_array_equal(got['peak_object'][n, c, :k], ref['peak_object'][n, c, :k],
                                              err_msg=f"frame {n} map {c} assignment")
                if c > 0 and ref['n_objects'][n] > 0:
                    np.testing.assert_allclose(got['peak_vote'][n, c, :k], ref['peak_vote'][n, c, :k], rtol=0, atol=1e-9)
        O = int(ref['n_objects'][n])
        np.testing.assert_array_equal(got['kp_count'][n, :O], ref['kp_count'][n, :O], err_msg=f"frame {n} kept keypoints")
        if exact_assignment:
            np.testing.assert_array_equal(got['kp_assigned'][n, :O], ref['kp_assigned'][n, :O])
            np.testing.assert_array_equal(got['kp_peak'][n, :O], ref['kp_peak'][n, :O], err_msg=f"frame {n} kept peak ids")
            np.testing.assert_array_equal(got['n_votes'][n, :O], ref['n_votes'][n, :O])
            V = ref['votes'].shape[2]
            for o in range(O):
                v = min(int(ref['n_votes'][n, o]), V)
                np.testing.assert_allclose(got['votes'][n, o, :v], ref['votes'][n, o, :v], rtol=0, atol=1e-9)
        for o in range(O):
            for c in range(C):
                for s in range(int(ref['kp_count'][n, o, c])):
                    assert np.abs(got['kp_xy'][n, o, c, s] - ref['kp_xy'][n, o, c, s]).max() <= TOL_PIXELS
                    if check_points:
                        want = ref['kp_point'][n, o, c, s]
                        have = got['kp_point'][n, o, c, s]
                        scale = max(np.linalg.norm(want), 1e-12)
                        assert np.linalg.norm(have - want) <= TOL_METRES_REL * scale + 1e-12, \
                            f"frame {n} object {o} map {c} slot {s}: {have} vs {want}"
