"""Loader for libokp.so (the CUDA library behind include/okp.h).

There is deliberately no fallback: if the shared library is missing or a call fails, the
error is raised -- nothing in this package computes the hot path on the CPU.
"""
import ctypes
import os

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIBRARY_PATH = os.path.join(_HERE, 'libokp.so')
_LIB = None

EXPORTS = [
    'okp_version', 'okp_strerror', 'okp_decode_workspace_bytes', 'okp_extract_peaks_f32',
    'okp_group_objects_f32', 'okp_decode_f32', 'okp_fisheye_undistort_f64', 'okp_fisheye_project_f64',
    'okp_detection_to_point_f32', 'okp_triangulate_f64', 'okp_reprojection_filter_f64',
    'okp_triangulate_robust_f64', 'okp_host_alias', 'okp_correct_matches_f64', 'okp_stereo_associate_f64',
    'okp_extract_peaks_bf16', 'okp_group_objects_bf16', 'okp_decode_bf16',
    'okp_eval_match_f64', 'okp_eval_summary_f64', 'okp_record_doubles', 'okp_pack_records_f64',
    'okp_rasterise_targets_f32', 'okp_host_pack_scratch_bytes', 'okp_host_pack_tiles_f32', 'okp_scatter_tiles_f32',
    'okp_record_bytes', 'okp_decode_emit_f32', 'okp_decode_emit_bf16', 'okp_triangulate_tracks_f64', 'okp_associate_pairs_f64',
    'okp_group_objects_emit_f32', 'okp_group_objects_emit_bf16', 'okp_extract_peaks_events_f32',
    'okp_extract_peaks_f16', 'okp_group_objects_f16', 'okp_decode_f16', 'okp_decode_emit_f16', 'okp_group_objects_emit_f16',
    'okp_decode_cameras_f32', 'okp_decode_cameras_bf16', 'okp_decode_cameras_f16',
    'okp_group_objects_cameras_f32', 'okp_group_objects_cameras_bf16', 'okp_group_objects_cameras_f16',
    'okp_triangulate_stereo_objects_f64', 'okp_triangulate_stereo_objects_depth_f64', 'okp_triangulate_sequence_objects_f64',
]


class OkpError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        super().__init__(f"{where}: {_abi.ERRORS.get(code, code)} ({strerror(code)})")


def build(verbose=False):
    """Compile csrc/okp_api.cu for sm_100a into libokp.so (nvcc cross-compiles without a GPU)."""
    import subprocess
    src = os.path.join(_HERE, 'csrc', 'okp_api.cu')
    # the host side of the sparse transfer is plain C++ (OpenMP; its AVX2 loop is a run-time-dispatched target function,
    # so no -mavx2 here and the file also builds on aarch64 hosts): g++ compiles it, nvcc links it in
    host_src = os.path.join(_HERE, 'csrc', 'okp_host_pack.cpp')
    host_obj = os.path.join(_HERE, 'csrc', 'okp_host_pack.o')
    host = subprocess.run(['g++', '-O3', '-fopenmp', '-fPIC', '-std=c++17', '-c', host_src, '-o', host_obj],
                          capture_output=True, text=True)
    if host.returncode != 0:
        raise RuntimeError("g++ failed:\n" + host.stdout + host.stderr)
    cmd = ['nvcc', '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-fmad=false',
           '-std=c++17', '-Xcompiler', '-fPIC', '-shared', '-cudart', 'static', '-o', LIBRARY_PATH, src, host_obj, '-lgomp']
    if verbose:
        cmd.insert(1, '-Xptxas')
        cmd.insert(2, '-v')
    result = subprocess.run(cmd, capture_output=True, text=True)
    if result.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + result.stdout + result.stderr)
    with open(STAMP_PATH, 'w') as handle:
        handle.write(_source_digest() + '\n')
    return result.stdout + result.stderr


STAMP_PATH = LIBRARY_PATH + '.stamp'


def _source_digest():
    """sha256 over the contents of everything libokp.so is built from (robust against mtime changes when the tree is
    copied to another box)."""
    import hashlib
    digest = hashlib.sha256()
    csrc = os.path.join(_HERE, 'csrc')
    names = sorted(f for f in os.listdir(csrc) if f.endswith(('.cu', '.cuh', '.cpp', '.h')))
    for path in [os.path.join(csrc, f) for f in names] + [os.path.join(os.path.dirname(_HERE), 'include', 'okp.h')]:
        with open(path, 'rb') as handle:
            digest.update(handle.read())
    return digest.hexdigest()


def needs_build():
    """True when libokp.so is missing or was built from other sources than the ones in the tree."""
    if not os.path.exists(LIBRARY_PATH) or not os.path.exists(STAMP_PATH):
        return True
    with open(STAMP_PATH) as handle:
        return handle.read().strip() != _source_digest()


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIBRARY_PATH):
        raise ImportError(f"{LIBRARY_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback for the decode path)")
    if needs_build():
        import warnings
        warnings.warn(f"{LIBRARY_PATH} is older than its sources (csrc/, include/okp.h): rebuild it with "
                      "`python -c 'import __graft_entry__ as g; g.build()'`", RuntimeWarning, stacklevel=2)
    L = ctypes.CDLL(LIBRARY_PATH)
    vp, i32, sz, dbl = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t, ctypes.c_double
    P = ctypes.POINTER
    L.okp_version.restype = i32
    L.okp_version.argtypes = []
    L.okp_strerror.restype = ctypes.c_char_p
    L.okp_strerror.argtypes = [i32]
    L.okp_decode_workspace_bytes.restype = sz
    L.okp_decode_workspace_bytes.argtypes = [i32, i32, i32, i32, P(_abi.OkpDecodeParams)]
    L.okp_extract_peaks_f32.restype = i32
    L.okp_extract_peaks_f32.argtypes = [vp, i32, i32, i32, i32, P(_abi.OkpDecodeParams), P(_abi.OkpDecodeTables),
                                        vp, sz, vp]
    L.okp_extract_peaks_events_f32.restype = i32
    L.okp_extract_peaks_events_f32.argtypes = L.okp_extract_peaks_f32.argtypes[:-1] + [vp, vp, vp]
    L.okp_group_objects_f32.restype = i32
    L.okp_group_objects_f32.argtypes = [vp, vp, i32, i32, i32, i32, P(ctypes.c_int32), P(_abi.OkpCamera),
                                        P(_abi.OkpDecodeParams), P(_abi.OkpDecodeTables), vp]
    L.okp_decode_f32.restype = i32
    L.okp_decode_f32.argtypes = [vp, vp, vp, i32, i32, i32, i32, P(ctypes.c_int32), P(_abi.OkpCamera),
                                 P(_abi.OkpDecodeParams), P(_abi.OkpDecodeTables), vp, sz, vp]
    for suffix in ('f32', 'bf16', 'f16'):
        extract, group, decode = (getattr(L, f'okp_{stem}_{suffix}') for stem in ('extract_peaks', 'group_objects', 'decode'))
        extract.restype = group.restype = decode.restype = i32
        extract.argtypes = L.okp_extract_peaks_f32.argtypes
        group.argtypes = L.okp_group_objects_f32.argtypes
        decode.argtypes = L.okp_decode_f32.argtypes
    L.okp_record_bytes.restype = i32
    L.okp_record_bytes.argtypes = [i32, i32, P(ctypes.c_int32)]
    for suffix in ('f32', 'bf16', 'f16'):
        emit = getattr(L, f'okp_decode_emit_{suffix}')
        emit.restype = i32
        emit.argtypes = L.okp_decode_f32.argtypes[:-1] + [P(_abi.OkpRecordSink), vp]
        group_emit = getattr(L, f'okp_group_objects_emit_{suffix}')
        group_emit.restype = i32
        group_emit.argtypes = L.okp_group_objects_f32.argtypes[:-1] + [P(_abi.OkpRecordSink), vp]
        # the _cameras forms: the emit entries with a DEVICE camera table [N] in place of the host camera
        cameras = getattr(L, f'okp_decode_cameras_{suffix}')
        cameras.restype = i32
        cameras.argtypes = emit.argtypes[:8] + [vp] + emit.argtypes[9:]
        group_cameras = getattr(L, f'okp_group_objects_cameras_{suffix}')
        group_cameras.restype = i32
        group_cameras.argtypes = group_emit.argtypes[:7] + [vp] + group_emit.argtypes[8:]
    L.okp_host_alias.restype = i32
    L.okp_host_alias.argtypes = [vp, P(vp)]
    L.okp_fisheye_undistort_f64.restype = i32
    L.okp_fisheye_undistort_f64.argtypes = [vp, i32, P(_abi.OkpCamera), i32, vp, vp]
    L.okp_fisheye_project_f64.restype = i32
    L.okp_fisheye_project_f64.argtypes = [vp, i32, P(dbl), P(_abi.OkpCamera), vp, vp]
    L.okp_detection_to_point_f32.restype = i32
    L.okp_detection_to_point_f32.argtypes = [vp, i32, vp, i32, i32, P(_abi.OkpCamera), P(_abi.OkpDecodeParams), vp, vp]
    L.okp_triangulate_f64.restype = i32
    L.okp_triangulate_f64.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp]
    L.okp_reprojection_filter_f64.restype = i32
    L.okp_reprojection_filter_f64.argtypes = [vp, vp, vp, vp, P(_abi.OkpCamera), i32, i32, dbl, vp, vp]
    L.okp_triangulate_robust_f64.restype = i32
    L.okp_triangulate_robust_f64.argtypes = [vp, vp, vp, P(_abi.OkpCamera), i32, i32, dbl, i32, vp, vp, vp, vp]
    L.okp_triangulate_tracks_f64.restype = i32
    L.okp_triangulate_tracks_f64.argtypes = [vp, vp, vp, P(_abi.OkpCamera), i32, i32, i32, dbl, i32, vp, vp, vp, vp]
    L.okp_associate_pairs_f64.restype = i32
    L.okp_associate_pairs_f64.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, dbl, vp, vp, vp]
    L.okp_correct_matches_f64.restype = i32
    L.okp_correct_matches_f64.argtypes = [P(dbl), vp, vp, i32, i32, vp, vp, vp]
    L.okp_stereo_associate_f64.restype = i32
    L.okp_stereo_associate_f64.argtypes = [P(dbl), vp, vp, vp, vp, i32, i32, i32, dbl, vp, vp, vp]
    L.okp_triangulate_stereo_objects_f64.restype = i32
    L.okp_triangulate_stereo_objects_f64.argtypes = [P(_abi.OkpDecodeTables), i32, i32, P(ctypes.c_int32),
                                                     P(_abi.OkpDecodeParams), vp, i32, P(_abi.OkpCamera), P(_abi.OkpCamera),
                                                     P(dbl), P(dbl), P(dbl), dbl, i32, P(_abi.OkpStereoTables), vp]
    L.okp_triangulate_stereo_objects_depth_f64.restype = i32
    L.okp_triangulate_stereo_objects_depth_f64.argtypes = [P(_abi.OkpDecodeTables), i32, i32, P(ctypes.c_int32),
                                                           P(_abi.OkpDecodeParams), vp, i32, P(_abi.OkpCamera),
                                                           P(_abi.OkpCamera), P(dbl), P(dbl), P(dbl), P(dbl), dbl, dbl, i32,
                                                           P(_abi.OkpStereoTables), vp]
    L.okp_triangulate_sequence_objects_f64.restype = i32
    L.okp_triangulate_sequence_objects_f64.argtypes = [P(_abi.OkpDecodeTables), i32, i32, P(ctypes.c_int32),
                                                       P(_abi.OkpDecodeParams), vp, i32, i32, vp, vp, vp, P(_abi.OkpCamera),
                                                       i32, dbl, dbl, dbl, i32, P(_abi.OkpSequenceObjectTables), vp]
    L.okp_eval_match_f64.restype = i32
    L.okp_eval_match_f64.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, P(_abi.OkpCamera), dbl, dbl, dbl, dbl,
                                     vp, vp, vp, vp, vp, vp, vp]
    L.okp_eval_summary_f64.restype = i32
    L.okp_eval_summary_f64.argtypes = [vp, i32, vp, vp]
    L.okp_record_doubles.restype = i32
    L.okp_record_doubles.argtypes = [i32, i32, i32]
    L.okp_pack_records_f64.restype = i32
    L.okp_pack_records_f64.argtypes = [P(_abi.OkpDecodeTables), i32, i32, i32, i32, ctypes.c_longlong, P(vp), i32, vp]
    L.okp_rasterise_targets_f32.restype = i32
    L.okp_rasterise_targets_f32.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, P(ctypes.c_int32), i32, dbl, dbl,
                                            vp, vp, vp, vp]
    L.okp_host_pack_scratch_bytes.restype = sz
    L.okp_host_pack_scratch_bytes.argtypes = [i32, i32, i32]
    L.okp_host_pack_tiles_f32.restype = i32
    L.okp_host_pack_tiles_f32.argtypes = [vp, i32, i32, i32, ctypes.c_float, vp, vp, vp, vp, ctypes.c_longlong,
                                          P(ctypes.c_longlong), i32]
    L.okp_scatter_tiles_f32.restype = i32
    L.okp_scatter_tiles_f32.argtypes = [vp, vp, ctypes.c_longlong, i32, i32, i32, vp, vp]
    _LIB = L
    return L


def strerror(code):
    try:
        return lib().okp_strerror(int(code)).decode()
    except Exception:
        return "?"


def check(code, where):
    if code != 0:
        raise OkpError(code, where)
