"""Drop-in for the reference's ``perception/pipeline.py`` on a B200.

Same class names, constructor / ``reset`` / ``__call__`` signatures and return structures as
the reference (file:line cited per class); the arithmetic runs in libokp.so (CUDA, sm_100a)
through the C ABI of include/okp.h. PyTorch only owns device memory and streams.

Two levels:

* ``KeypointDecoder`` -- the batched device API (no batch-1 limit, tensors stay in HBM,
  fixed-capacity record tables come back as tensors);
* ``KeypointExtractionComponent``, ``ObjectExtraction``, ``DetectionToPoint``,
  ``ObjectKeypointPipeline``, ``LearnedKeypointTrackingPipeline`` -- the reference's
  interface, converting the tables to the reference's nested lists / dicts.
"""
import ctypes
import time

import numpy as np
import torch

from . import _abi, _lib

_TORCH_DTYPES = {np.dtype(np.int32): torch.int32, np.dtype(np.uint32): torch.int32,
                 np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64, np.dtype(np.uint8): torch.uint8}


def _device(device=None):
    if not torch.cuda.is_available():
        raise RuntimeError("object_keypoints_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
    if device is None:
        return torch.device('cuda', torch.cuda.current_device())
    return torch.device(device)


def _stream_handle(stream=None):
    stream = torch.cuda.current_stream() if stream is None else stream
    return ctypes.c_void_p(stream.cuda_stream)


def _host_threads():
    """Threads for the host pass of the sparse transfer: this process's share of the cores (the affinity mask divided
    by the ranks torchrun started on this node), whatever OMP_NUM_THREADS says (torchrun sets it to 1)."""
    import os
    cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    return max(1, cores // max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1'))))


def _local_world():
    import os
    return max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))


def _as_device_f32(x, device):
    """NumPy array / CPU tensor / CUDA tensor -> contiguous float32 CUDA tensor."""
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(np.ascontiguousarray(x))
    if x.dtype != torch.float32:
        x = x.float()
    if x.device != device:
        x = x.to(device, non_blocking=True)
    return _aligned(x.contiguous())


def _aligned(x):
    """The TMA kernel needs a 16-byte aligned base (okp.h: OKP_E_UNSUPPORTED otherwise): a view that starts in the
    middle of an allocation (``batch[1:]`` of a map with an odd element count) is re-materialised."""
    return x.clone() if x.data_ptr() % 16 else x


# element type of a map -> suffix of the okp_* entries that read it in place
_MAP_KINDS = {torch.float32: 'f32', torch.bfloat16: 'bf16', torch.float16: 'f16'}


def _as_device_map(x, device):
    """Like _as_device_f32, but a bfloat16 or float16 tensor (the output of a bf16 or half-precision network head)
    keeps its type: the okp_*_bf16 / okp_*_f16 entries read it in place, on the device or after a copy of the 16-bit
    bytes from the host. -> (tensor, 'f32' | 'bf16' | 'f16')."""
    if isinstance(x, torch.Tensor) and x.dtype in (torch.bfloat16, torch.float16):
        if x.device != device:
            x = x.to(device, non_blocking=True)
        return _aligned(x.contiguous()), _MAP_KINDS[x.dtype]
    return _as_device_f32(x, device), 'f32'


class _TableSet:
    """Tables as torch tensors on one device, all views into ONE allocation (each starting on a 256-byte boundary), so
    that the synchronising host copy of a call is a single transfer. shapes: (name, numpy dtype, shape) in the field
    order of `struct_type`, the matching ctypes struct of device pointers (include/okp.h)."""
    ALIGN = 256

    def __init__(self, shapes, struct_type, device):
        self._layout = []
        offset = 0
        for name, dtype, shape in shapes:
            nbytes = int(np.prod(shape, dtype=np.int64)) * np.dtype(dtype).itemsize
            self._layout.append((name, np.dtype(dtype), tuple(shape), offset, nbytes))
            offset += (nbytes + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        self.flat = torch.zeros(max(offset, self.ALIGN), dtype=torch.uint8, device=device)
        self.tensors = {}
        for name, dtype, shape, start, nbytes in self._layout:
            self.tensors[name] = self.flat[start:start + nbytes].view(_TORCH_DTYPES[dtype]).reshape(shape)
        self.struct = struct_type(**{k: v.data_ptr() for k, v in self.tensors.items()})

    def __getitem__(self, name):
        return self.tensors[name]

    def numpy(self):
        """Synchronising copy of every table to host NumPy arrays (flags as uint32): one device-to-host transfer."""
        host = self.flat.cpu().numpy()
        return {name: host[start:start + nbytes].view(np.uint32 if name == 'flags' else dtype).reshape(shape)
                for name, dtype, shape, start, nbytes in self._layout}


class DecodeTables(_TableSet):
    """The OkpDecodeTables record as torch tensors on one device (layout: include/okp.h), in one allocation: the
    synchronising host copy of a decode -- what the reference-style per-frame ``__call__`` does after every frame -- is a
    single transfer. keypoint_config and params are kept for the calls that read the tables (triangulate_stereo_objects)."""

    def __init__(self, N, C, keypoint_config, params, device):
        self.N, self.C = N, C
        self.keypoint_config, self.params = list(keypoint_config), params
        super().__init__(_abi.table_shapes(N, C, keypoint_config, params), _abi.OkpDecodeTables, device)


class StereoTables(_TableSet):
    """The OkpStereoTables record of triangulate_stereo_objects as torch tensors on one device, in one allocation:
    object_match [P,O], object_cost [P,O], slot_match [P,O,C,S], point [P,O,C,S,3] (left camera frame, NaN where
    slot_match is -1), flags [P] (_abi.STEREO_*)."""

    def __init__(self, P, O, C, S, device):
        self.P = P
        super().__init__([(name, dtype, shape(P, O, C, S)) for name, dtype, shape in _abi.STEREO_LAYOUT],
                         _abi.OkpStereoTables, device)


class SequenceObjectTables(_TableSet):
    """The OkpSequenceObjectTables record of SequenceTriangulator.objects as torch tensors on one device, in one
    allocation: per (anchor, view) pair object_match / object_cost [A,V-1,O], slot_match [A,V-1,O,C,S], flags [A,V-1]
    (_abi.STEREO_*); per anchor slot a track of V views, observations [A,O,C,S,V,2] (distorted pixels; view 0 is the
    anchor's own keypoint), observed / valid [A,O,C,S,V] (before / after the reprojection filter), error [A,O,C,S,V],
    dropped [A,O,C,S], and point [A,O,C,S,3] in the world frame (NaN where fewer than two views are valid)."""

    def __init__(self, A, V, O, C, S, device):
        self.A, self.V = A, V
        super().__init__([(name, dtype, shape(A, V, O, C, S)) for name, dtype, shape in _abi.SEQUENCE_LAYOUT],
                         _abi.OkpSequenceObjectTables, device)


class CameraTable:
    """One camera per frame on the device (KeypointDecoder.camera_table): ``rows`` is a [N, 144] uint8 CUDA tensor of
    OkpCamera records (include/okp.h), row n the camera frame n of a batch is lifted with. Built once per batch layout
    and passed as ``cameras=`` to every decode of that layout, so no call uploads cameras."""
    RECORD_BYTES = ctypes.sizeof(_abi.OkpCamera)

    def __init__(self, rows):
        if rows.dtype != torch.uint8 or rows.dim() != 2 or rows.shape[1] != self.RECORD_BYTES or not rows.is_cuda:
            raise ValueError(f"rows must be a [N, {self.RECORD_BYTES}] uint8 CUDA tensor")
        if rows.data_ptr() % 16 or not rows.is_contiguous():
            raise ValueError("rows must be contiguous and 16-byte aligned")
        self.rows = rows
        self.N = int(rows.shape[0])

    def data_ptr(self):
        return self.rows.data_ptr()

    def frames(self, start, stop):
        """The rows of frames [start, stop): a view, i.e. a pointer offset into the same table."""
        return CameraTable(self.rows[start:stop])

    def check(self, N, device):
        """The table must describe this batch and live on the decoder's device: the kernel reads it by raw pointer."""
        if self.N != N:
            raise ValueError(f"the camera table has {self.N} rows, the batch {N} frames")
        if device.index is None:                             # 'cuda' = the current device
            device = torch.device(device.type, torch.cuda.current_device())
        if self.rows.device != device:
            raise ValueError(f"the camera table is on {self.rows.device}, the decoder on {device}")
        return self


class KeypointDecoder:
    """Batched heatmap -> grouped 2D keypoints -> 3D points on the GPU.

    keypoint_config: the parsed JSON dict {'keypoint_config': [...]} or the bare list.
    prediction_size: (H, W) of the network output.
    """

    def __init__(self, keypoint_config, prediction_size, camera=None, device=None, max_peaks=32, max_objects=16,
                 max_votes=16, threshold=0.5, outlier_distance=20.0, compat_clip_bug=True, nms_size=5, box_sum=True,
                 top_k=0, lean_tables=False, single_pass=False):
        self.cfg = _abi.check_keypoint_config(keypoint_config)
        self.C = 1 + len(self.cfg)
        self.H, self.W = int(prediction_size[0]), int(prediction_size[1])
        self.params = _abi.make_params(threshold=threshold, outlier_distance=outlier_distance, max_peaks=max_peaks,
                                       max_objects=max_objects, max_votes=max_votes, compat_clip_bug=compat_clip_bug,
                                       nms_size=nms_size, box_sum=box_sum, top_k=top_k, lean_tables=lean_tables,
                                       single_pass=single_pass)
        self.device = _device(device)
        self._cfg_array = (ctypes.c_int32 * max(len(self.cfg), 1))(*self.cfg)
        self._camera = None
        self._tables = {}
        self._workspace = None
        self._lib = _lib.lib()
        if camera is not None:
            self.reset(camera)

    def reset(self, camera):
        """camera: object exposing K, D, Kinv, image_size (camera_utils.FisheyeCamera or the
        reference's own class), as DetectionToPoint.reset receives it (pipeline.py:159-162)."""
        self._camera = _abi.pack_camera(camera)

    def camera_table(self, cameras, camera_index):
        """Per-frame cameras for ``decode_batch`` / ``group_objects`` / ``decode_host_batch(cameras=...)``: a short
        sequence of camera objects (as ``reset`` takes them) and camera_index [N], the index into ``cameras`` of every
        frame -> CameraTable on this decoder's device. E.g. a stereo batch with the left views in even and the right views
        in odd rows: ``camera_table((stereo.left_camera, stereo.right_camera), np.arange(N) % 2)``. The indices are
        checked here (_abi.pack_camera_table); build the table once per batch layout and reuse it."""
        packed = _abi.pack_camera_table(cameras, camera_index)
        host = np.frombuffer(bytes(packed), dtype=np.uint8).reshape(len(packed), CameraTable.RECORD_BYTES)
        return CameraTable(_aligned(torch.from_numpy(host.copy()).to(self.device)))

    def tables(self, N):
        if N not in self._tables:
            self._tables[N] = DecodeTables(N, self.C, self.cfg, self.params, self.device)
        return self._tables[N]

    def _workspace_for(self, N):
        need = self._lib.okp_decode_workspace_bytes(N, self.C, self.H, self.W, ctypes.byref(self.params))
        if need == 0:
            raise ValueError("unsupported shape or parameters")
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._workspace

    def _check(self, heat):
        if heat.dim() != 4 or heat.shape[1] != self.C or heat.shape[2] != self.H or heat.shape[3] != self.W:
            raise ValueError(f"heatmap must be [N,{self.C},{self.H},{self.W}], got {tuple(heat.shape)}")

    def extract_peaks(self, heat, tables=None, stream=None):
        """K1 only: fills the peak_* tables. Asynchronous on the current (or given) stream."""
        heat, kind = _as_device_map(heat, self.device)
        self._check(heat)
        N = heat.shape[0]
        tables = self.tables(N) if tables is None else tables
        ws = self._workspace_for(N)
        entry = getattr(self._lib, f'okp_extract_peaks_{kind}')
        rc = entry(heat.data_ptr(), N, self.C, self.H, self.W, ctypes.byref(self.params),
                   ctypes.byref(tables.struct), ws.data_ptr(), ws.numel(), _stream_handle(stream))
        _lib.check(rc, f'okp_extract_peaks_{kind}')
        return tables

    def record_bytes(self):
        """Bytes of one compact per-frame record (okp_decode_emit_*, include/okp.h)."""
        return int(self._lib.okp_record_bytes(self.params.max_objects, self.C, self._cfg_array))

    def decode_batch(self, heat, depth, centers, tables=None, stream=None, records=None, peaks_done=None, cameras=None):
        """heat [N,C,H,W], depth [N,C,H,W], centers [N,C-1,2,H,W] (float32, bfloat16 or float16; CUDA tensors
        are used in place, host arrays are copied, 16-bit tensors keep their type) -> DecodeTables on the device. No
        synchronisation. Heatmaps of one type with depth / centre maps of another take two C calls (peaks, then
        grouping); depth and centre maps of different types are both up-cast to float32.
        records: an ``_abi.OkpRecordSink`` (sharding.RecordExchange.begin()): the kernel also writes every frame's
        compact record into the sink's buffers while it decodes (the multi-GPU gather).
        peaks_done: a ``torch.cuda.Event`` recorded between the peak kernel (+ its overflow fix-up) and the grouping
        kernel -- the two halves are then enqueued by two C calls instead of one. A PAIR of timing events instead is
        recorded by the library right before and right after the peak kernel itself (okp_extract_peaks_events_f32:
        bench.py's roofline figure is the time between them).
        cameras: a CameraTable with N rows (camera_table): frame n is lifted with its own camera instead of ``reset``'s
        (okp_decode_cameras_* / okp_group_objects_cameras_*; not with ``single_pass``)."""
        heat, heat_kind = _as_device_map(heat, self.device)
        self._check(heat)
        depth, depth_kind = _as_device_map(depth, self.device)
        centers, centers_kind = _as_device_map(centers, self.device)
        if depth_kind != centers_kind:                       # the grouping entry takes one element type
            depth, centers, depth_kind = depth.float(), centers.float(), 'f32'
        N = heat.shape[0]
        if tuple(depth.shape) != tuple(heat.shape):
            raise ValueError("depth must have the heatmap's shape")
        if tuple(centers.shape) != (N, self.C - 1, 2, self.H, self.W):
            raise ValueError(f"centers must be [N,{self.C - 1},2,{self.H},{self.W}], got {tuple(centers.shape)}")
        tables = self.tables(N) if tables is None else tables
        ws = self._workspace_for(N)
        # the _cameras entries take the DEVICE table where the _emit entries take the host camera
        form, cam = ('cameras', ctypes.c_void_p(cameras.check(N, self.device).data_ptr())) if cameras is not None else \
            ('emit', ctypes.byref(self._camera) if self._camera is not None else None)
        if heat_kind == depth_kind and peaks_done is None:
            rc = getattr(self._lib, f'okp_decode_{form}_{heat_kind}')(
                heat.data_ptr(), depth.data_ptr(), centers.data_ptr(), N, self.C, self.H, self.W, self._cfg_array, cam,
                ctypes.byref(self.params), ctypes.byref(tables.struct), ws.data_ptr(), ws.numel(),
                ctypes.byref(records) if records is not None else None, _stream_handle(stream))
            _lib.check(rc, f'okp_decode_{form}_{heat_kind}')
        else:                                                # e.g. 16-bit heatmaps with float32 depth / centre maps
            pair = peaks_done if isinstance(peaks_done, (tuple, list)) else None
            if pair is not None and heat_kind == 'f32':
                for event in pair:
                    if not event.cuda_event:                 # torch creates the CUDA event at its first record
                        event.record(torch.cuda.current_stream(self.device) if stream is None else stream)
                rc = self._lib.okp_extract_peaks_events_f32(
                    heat.data_ptr(), N, self.C, self.H, self.W, ctypes.byref(self.params), ctypes.byref(tables.struct),
                    ws.data_ptr(), ws.numel(), ctypes.c_void_p(pair[0].cuda_event), ctypes.c_void_p(pair[1].cuda_event),
                    _stream_handle(stream))
                _lib.check(rc, 'okp_extract_peaks_events_f32')
            else:
                rc = getattr(self._lib, f'okp_extract_peaks_{heat_kind}')(
                    heat.data_ptr(), N, self.C, self.H, self.W, ctypes.byref(self.params), ctypes.byref(tables.struct),
                    ws.data_ptr(), ws.numel(), _stream_handle(stream))
                _lib.check(rc, f'okp_extract_peaks_{heat_kind}')
                for event in (pair if pair is not None else [peaks_done] if peaks_done is not None else []):
                    event.record(torch.cuda.current_stream(self.device) if stream is None else stream)
            rc = getattr(self._lib, f'okp_group_objects_{form}_{depth_kind}')(
                depth.data_ptr(), centers.data_ptr(), N, self.C, self.H, self.W, self._cfg_array, cam,
                ctypes.byref(self.params), ctypes.byref(tables.struct),
                ctypes.byref(records) if records is not None else None, _stream_handle(stream))
            _lib.check(rc, f'okp_group_objects_{form}_{depth_kind}')
        return tables

    HOST_RESULT_TABLES = ('n_objects', 'flags', 'kp_count', 'kp_xy', 'kp_point')

    def _host_alias(self, tensor):
        """Device-side address of a pinned CPU tensor (okp_host_alias), or None if it has to be copied."""
        if (tensor.device.type != 'cpu' or tensor.dtype not in _MAP_KINDS or not tensor.is_contiguous() or
                not tensor.is_pinned()):
            return None
        alias = ctypes.c_void_p()
        if self._lib.okp_host_alias(ctypes.c_void_p(tensor.data_ptr()), ctypes.byref(alias)) != 0 or not alias.value:
            return None
        return alias.value

    SPARSE_CAPACITY = 0.5          # fall back to the dense copy when more than this share of a chunk's tiles is marked
    SPARSE_MAX_LOCAL_WORLD = int(__import__('os').environ.get('OKP_SPARSE_MAX_LOCAL_WORLD', '4'))   # see _sparse_ok
    SPARSE_MIN_THREADS = 2         # sparse='auto' runs the host pass from this many host threads per rank on: the scheduler
                                   # below hands it a chunk only when it will finish before the copy engine could have moved
                                   # the remaining chunks densely, so a slow pass (few threads) just takes fewer chunks

    def _sparse_ok(self, heat, sparse):
        """The sparse transfer holds for the reference's configuration only (csrc/okp_sparse.cuh)."""
        if sparse in (False, 'off', None):
            return False
        # The pass trades PCIe bytes for host-DRAM bytes: it reads every heatmap byte once with the CPU and sends ~19 % of
        # them, i.e. 1.19x the dense copy's host-memory traffic for 0.19x of its PCIe traffic. It pays while the rank's
        # PCIe link is the limit (1-2 ranks per host: 121 k against 79 k frames/s on one GPU, 198 k against 156 k on two) and
        # costs when the ranks of a host together saturate its memory first (8 ranks on a 32-core host: 246 k against 262 k
        # frames/s, gpurun_out/r2j) -- so 'auto' also looks at how many ranks share the host.
        if sparse == 'auto' and (_host_threads() < self.SPARSE_MIN_THREADS or _local_world() > self.SPARSE_MAX_LOCAL_WORLD):
            return False
        return (self.params.nms_size == 5 and self.params.box_sum == 1 and self.params.threshold > 0.0 and
                heat.device.type == 'cpu' and heat.dtype == torch.float32 and heat.is_contiguous())

    HOST_STAGING_SETS = 2          # staging sets (device chunk buffers + pinned packing buffers) kept, least recently used out

    def _check_host_inputs(self, heat, depth, centers):
        """Shapes / dtypes of decode_host_batch's inputs: the host pass and the in-place gathers work on raw pointers, so a
        wrong shape or element type would be an out-of-bounds read, not an exception. All three maps share one dtype:
        float32, bfloat16 or float16."""
        for name, tensor in (('heat', heat), ('depth', depth), ('centers', centers)):
            if not isinstance(tensor, torch.Tensor) or tensor.device.type != 'cpu' or tensor.dtype not in _MAP_KINDS:
                raise ValueError(f"{name} must be a float32, bfloat16 or float16 CPU tensor")
        if not heat.dtype == depth.dtype == centers.dtype:
            raise ValueError(f"heat, depth and centers must share one dtype, got {heat.dtype}, {depth.dtype} and "
                             f"{centers.dtype}")
        self._check(heat)
        N = int(heat.shape[0])
        if tuple(depth.shape) != tuple(heat.shape):
            raise ValueError(f"depth must have the heatmap's shape {tuple(heat.shape)}, got {tuple(depth.shape)}")
        if tuple(centers.shape) != (N, self.C - 1, 2, self.H, self.W):
            raise ValueError(f"centers must be [{N},{self.C - 1},2,{self.H},{self.W}], got {tuple(centers.shape)}")

    def host_result(self, N, like=None):
        """Pinned CPU tensors for decode_host_batch's result (pass them back as ``out=`` to reuse them)."""
        like = like if like is not None else DecodeTables(1, self.C, self.cfg, self.params, self.device)
        return {name: torch.empty((N,) + tuple(like[name].shape[1:]), dtype=like[name].dtype).pin_memory()
                for name in self.HOST_RESULT_TABLES}

    def decode_host_batch(self, heat, depth, centers, chunk_frames=128, sparse='auto', out=None, cameras=None):
        """End-to-end form for HOST inputs, the shape the reference's caller has (CPU tensors out of
        InferenceComponent, pipeline.py:24-28). The batch is cut into chunks that are pipelined: while chunk i is
        decoded, chunk i+1 crosses PCIe and chunk i+2 is prepared on the host. The three maps are float32, bfloat16
        or float16 CPU tensors of one dtype; 16-bit maps cross the bus as they are (half the bytes of float32) and are
        decoded by the okp_*_bf16 / okp_*_f16 entries.

        Heatmaps: with ``sparse='auto'`` a host pass (okp_host_pack_tiles_f32, OpenMP + AVX2, in a worker thread)
        marks the 4x16-pixel tiles within reach of a value above threshold / 25 and only those cross the bus; the
        device scatters them into a zeroed map (okp_scatter_tiles_f32). Everything farther than 4 px from such a
        value cannot change any table (csrc/okp_sparse.cuh), so the result is bit-identical to the dense copy.
        The host pass is bound by host memory bandwidth and the dense copy by PCIe, so both run side by side: chunks
        are handed to the host pass one after the other, and whenever the copy engine has fewer than two dense
        chunks queued the next chunk goes over the bus as it is. A chunk with more than half of its tiles marked
        (dense maps) is copied densely too; ``sparse=False`` disables the host pass, ``sparse='only'`` the side-by-side
        dense copies. Depth and centre maps are only gathered from (3 values per spoke peak): when they live in
        pinned host memory the kernels read them in place over PCIe; pageable tensors are copied like dense
        heatmaps. The host pass is float32-only: 16-bit heatmaps always take the dense copy. The object tables of
        every chunk are copied back into pinned host tensors.
        Returns a dict of CPU tensors (synchronised): freshly allocated for every call, or ``out`` (a dict from an earlier
        call or from ``host_result``) filled in place. cameras: a CameraTable with N rows, as in ``decode_batch``; each
        chunk reads its own rows of it, wherever the chunk boundaries fall."""
        self._check_host_inputs(heat, depth, centers)
        if cameras is not None:
            cameras.check(int(heat.shape[0]), self.device)
        heat, depth, centers = heat.contiguous(), depth.contiguous(), centers.contiguous()
        N = int(heat.shape[0])
        chunk = max(1, min(chunk_frames, N))
        depth_alias = self._host_alias(depth)
        centers_alias = self._host_alias(centers)
        in_place = depth_alias is not None and centers_alias is not None
        use_sparse = self._sparse_ok(heat, sparse)
        dtype, kind = heat.dtype, _MAP_KINDS[heat.dtype]
        key = ('host', chunk, in_place, use_sparse, dtype)
        tiles_per_map = ((self.H + 3) // 4) * ((self.W + 15) // 16)
        capacity = max(1, int(self.SPARSE_CAPACITY * chunk * self.C * tiles_per_map))
        if key not in self._tables:
            staging = []
            for slot_index in range(5 if use_sparse else 2):       # sparse: three packing slots, two dense-copy slots
                slot = {
                    'heat': torch.empty((chunk, self.C, self.H, self.W), dtype=dtype, device=self.device),
                    'tables': DecodeTables(chunk, self.C, self.cfg, self.params, self.device),
                    'ready': torch.cuda.Event(), 'done': torch.cuda.Event(), 'copied': torch.cuda.Event(),
                }
                if not in_place:
                    slot['depth'] = torch.empty((chunk, self.C, self.H, self.W), dtype=dtype, device=self.device)
                    slot['centers'] = torch.empty((chunk, self.C - 1, 2, self.H, self.W), dtype=dtype, device=self.device)
                if use_sparse and slot_index < 3:
                    maps = chunk * self.C
                    slot['packed_host'] = torch.empty((capacity, 64), dtype=torch.float32).pin_memory()
                    slot['ids_host'] = torch.empty(capacity, dtype=torch.int32).pin_memory()
                    slot['packed'] = torch.empty((capacity, 64), dtype=torch.float32, device=self.device)
                    slot['ids'] = torch.empty(capacity, dtype=torch.int32, device=self.device)
                    slot['scratch'] = np.zeros(self._lib.okp_host_pack_scratch_bytes(maps, self.H, self.W), np.uint8)
                    slot['offsets'] = np.zeros(maps + 1, np.int64)
                staging.append(slot)
            held = [k for k in self._tables if isinstance(k, tuple) and k[0] == 'host']
            while len(held) >= self.HOST_STAGING_SETS:            # bounded: callers with varying chunk sizes do not pile up HBM
                del self._tables[held.pop(0)]
            self._tables[key] = (staging, torch.cuda.Stream(device=self.device))
        else:
            self._tables[key] = self._tables.pop(key)              # most recently used last
        staging, copy_stream = self._tables[key]
        if out is None:
            result = self.host_result(N, staging[0]['tables'])
        else:
            result = out
            for name in self.HOST_RESULT_TABLES:
                if name not in result or result[name].shape[0] != N or not result[name].is_pinned():
                    raise ValueError(f"out['{name}'] must be a pinned CPU tensor with {N} rows (see host_result)")
        compute = torch.cuda.current_stream()
        self._workspace_for(chunk)
        depth_frame = self.C * self.H * self.W * heat.element_size()            # bytes of one frame's heat or depth maps
        centers_frame = (self.C - 1) * 2 * self.H * self.W * heat.element_size()
        cam = ctypes.byref(self._camera) if self._camera is not None else None
        self.host_bytes_copied = 0
        self.host_chunks_sparse = 0
        self.host_pack_threads = _host_threads() if use_sparse else 0
        marked_tiles = [0, 0]                              # tiles marked / tiles looked at by the host pass
        starts = list(range(0, N, chunk))

        def pack(index, slot):
            """Host pass for chunk `index` into the slot's pinned staging; returns the number of marked tiles."""
            slot['copied'].synchronize()                  # the slot's previous transfer has left the pinned buffers
            began = time.perf_counter()
            f0 = starts[index]
            n = min(f0 + chunk, N) - f0
            count = ctypes.c_longlong()
            rc = self._lib.okp_host_pack_tiles_f32(
                ctypes.c_void_p(heat.data_ptr() + f0 * depth_frame), n * self.C, self.H, self.W,
                ctypes.c_float(self.params.threshold), ctypes.c_void_p(slot['scratch'].ctypes.data),
                ctypes.c_void_p(slot['offsets'].ctypes.data), ctypes.c_void_p(slot['ids_host'].data_ptr()),
                ctypes.c_void_p(slot['packed_host'].data_ptr()), capacity, ctypes.byref(count), _host_threads())
            _lib.check(rc, 'okp_host_pack_tiles_f32')
            self._pack_seconds = time.perf_counter() - began
            marked_tiles[0] += int(count.value)
            marked_tiles[1] += n * self.C * tiles_per_map
            return int(count.value)

        def enqueue(index, slot, n_tiles):
            """Transfer (sparse if n_tiles fits, else dense) + decode + read-back of chunk `index`, all asynchronous."""
            f0 = starts[index]
            f1 = min(f0 + chunk, N)
            n = f1 - f0
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(slot['done'])              # the slot's previous decode + read-back finished
                if n_tiles is not None and n_tiles <= capacity:
                    slot['packed'][:n_tiles].copy_(slot['packed_host'][:n_tiles], non_blocking=True)
                    slot['ids'][:n_tiles].copy_(slot['ids_host'][:n_tiles], non_blocking=True)
                    slot['copied'].record(copy_stream)
                    slot['heat'][:n].zero_()
                    rc = self._lib.okp_scatter_tiles_f32(slot['packed'].data_ptr(), slot['ids'].data_ptr(), n_tiles,
                                                         n * self.C, self.H, self.W, slot['heat'].data_ptr(),
                                                         ctypes.c_void_p(copy_stream.cuda_stream))
                    _lib.check(rc, 'okp_scatter_tiles_f32')
                    self.host_bytes_copied += n_tiles * (64 * 4 + 4)
                    self.host_chunks_sparse += 1
                else:
                    slot['heat'][:n].copy_(heat[f0:f1], non_blocking=True)
                    slot['copied'].record(copy_stream)
                    self.host_bytes_copied += n * depth_frame
                if not in_place:
                    slot['depth'][:n].copy_(depth[f0:f1], non_blocking=True)
                    slot['centers'][:n].copy_(centers[f0:f1], non_blocking=True)
                    self.host_bytes_copied += n * (depth_frame + centers_frame)
                slot['ready'].record(copy_stream)
            compute.wait_event(slot['ready'])
            tables = slot['tables'] if n == chunk else self.tables(n)
            chunk_cameras = cameras.frames(f0, f1) if cameras is not None else None
            if in_place and chunk_cameras is not None:
                ws = self._workspace_for(n)
                rc = getattr(self._lib, f'okp_decode_cameras_{kind}')(
                    slot['heat'].data_ptr(), depth_alias + f0 * depth_frame, centers_alias + f0 * centers_frame, n, self.C,
                    self.H, self.W, self._cfg_array, ctypes.c_void_p(chunk_cameras.data_ptr()), ctypes.byref(self.params),
                    ctypes.byref(tables.struct), ws.data_ptr(), ws.numel(), None, _stream_handle(compute))
                _lib.check(rc, f'okp_decode_cameras_{kind}')
            elif in_place:
                ws = self._workspace_for(n)
                rc = getattr(self._lib, f'okp_decode_{kind}')(
                    slot['heat'].data_ptr(), depth_alias + f0 * depth_frame, centers_alias + f0 * centers_frame, n, self.C,
                    self.H, self.W, self._cfg_array, cam, ctypes.byref(self.params), ctypes.byref(tables.struct),
                    ws.data_ptr(), ws.numel(), _stream_handle(compute))
                _lib.check(rc, f'okp_decode_{kind}')
            else:
                self.decode_batch(slot['heat'][:n], slot['depth'][:n], slot['centers'][:n], tables=tables,
                                  cameras=chunk_cameras)
            for name in self.HOST_RESULT_TABLES:
                result[name][f0:f1].copy_(tables[name][:n], non_blocking=True)
            slot['done'].record(compute)

        # Chunks are independent (each writes its own rows of the result), so they are handed out to two producers
        # that run side by side: the host pass (CPU-bound; its chunks need a sixth of the PCIe time) and, with
        # sparse='auto', the plain dense copy (PCIe-bound; needs no CPU) whenever the copy engine has less than two
        # dense chunks queued. Host memory bandwidth and the PCIe link are both kept busy.
        claimed = 0
        dense_seconds = chunk * depth_frame / 50e9              # a dense chunk on a Gen5 x16 link
        self._pack_seconds = getattr(self, '_pack_seconds', 0.0)   # the last pass's duration (previous call included)
        sparse_slots = staging[:3] if use_sparse else []
        dense_slots = staging[3:] if use_sparse else staging
        packing = None                                            # (future, chunk index, slot)
        packed_chunks = dense_chunks = 0
        dense_events = []
        if use_sparse:
            if getattr(self, '_pack_executor', None) is None:      # one long-lived worker: its OpenMP team is reused
                from concurrent.futures import ThreadPoolExecutor
                self._pack_executor = ThreadPoolExecutor(max_workers=1, thread_name_prefix='okp-pack')
            packing = (self._pack_executor.submit(pack, 0, sparse_slots[0]), 0, sparse_slots[0])
            claimed = 1
        try:
            while claimed < len(starts) or packing is not None:
                progressed = False
                if packing is not None and packing[0].done():
                    future, index, slot = packing
                    n_tiles = future.result()
                    packed_chunks += 1
                    packing = None
                    # the pass takes another chunk only if it will be done before the copy engine could have moved all
                    # the remaining chunks densely (few host threads per rank, the last chunks of a batch)
                    remaining = len(starts) - claimed
                    if remaining > 0 and (sparse == 'only' or self._pack_seconds <= remaining * dense_seconds):
                        nxt = sparse_slots[packed_chunks % len(sparse_slots)]
                        packing = (self._pack_executor.submit(pack, claimed, nxt), claimed, nxt)
                        claimed += 1
                    enqueue(index, slot, n_tiles)
                    progressed = True
                elif claimed < len(starts) and dense_slots:
                    dense_events = [e for e in dense_events if not e.query()]
                    if not use_sparse or (sparse != 'only' and len(dense_events) < 2):
                        slot = dense_slots[dense_chunks % len(dense_slots)]
                        dense_chunks += 1
                        enqueue(claimed, slot, None)
                        claimed += 1
                        if use_sparse:
                            dense_events.append(slot['ready'])
                        progressed = True
                if not progressed:
                    time.sleep(5e-5)
        finally:
            if packing is not None:                                # an exception above: do not leave a pass running
                packing[0].cancel() or packing[0].exception()
        compute.synchronize()
        self.host_marked_fraction = marked_tiles[0] / marked_tiles[1] if marked_tiles[1] else None
        return result

    def group_objects(self, depth, centers, tables, stream=None, cameras=None):
        """K3 + K4 on peak tables that are already filled (ObjectExtraction + DetectionToPoint). cameras: a CameraTable
        with tables.N rows, as in ``decode_batch`` (needs depth)."""
        N = tables.N
        centers, kind = _as_device_map(centers, self.device)
        if cameras is not None:
            if depth is None:
                raise ValueError("the 3D lift with per-frame cameras needs the depth maps")
            cameras.check(N, self.device)
            depth, depth_kind = _as_device_map(depth, self.device)
            if depth_kind != kind:
                depth, centers, kind = depth.float(), centers.float(), 'f32'
            rc = getattr(self._lib, f'okp_group_objects_cameras_{kind}')(
                depth.data_ptr(), centers.data_ptr(), N, self.C, self.H, self.W, self._cfg_array,
                ctypes.c_void_p(cameras.data_ptr()), ctypes.byref(self.params), ctypes.byref(tables.struct), None,
                _stream_handle(stream))
            _lib.check(rc, f'okp_group_objects_cameras_{kind}')
            return tables
        depth_ptr = None
        cam = None
        if depth is not None and self._camera is not None:
            depth, depth_kind = _as_device_map(depth, self.device)
            if depth_kind != kind:
                depth, centers, kind = depth.float(), centers.float(), 'f32'
            depth_ptr = depth.data_ptr()
            cam = ctypes.byref(self._camera)
        rc = getattr(self._lib, f'okp_group_objects_{kind}')(
            depth_ptr, centers.data_ptr(), N, self.C, self.H, self.W, self._cfg_array, cam, ctypes.byref(self.params),
            ctypes.byref(tables.struct), _stream_handle(stream))
        _lib.check(rc, f'okp_group_objects_{kind}')
        return tables


# ------------------------------------------------------------------------------------------------
# conversion of record tables to the reference's Python structures
# ------------------------------------------------------------------------------------------------
def tables_to_keypoints(t, n):
    """-> (keypoints[C][k] of (2,) float32 (x, y), confidence[C][k]) like
    KeypointExtractionComponent._extract_keypoints (pipeline.py:64-79)."""
    C, K = t['peak_count'].shape[1], t['peak_xy'].shape[2]
    points, confidence = [], []
    for c in range(C):
        k = min(int(t['peak_count'][n, c]), K)
        points.append([t['peak_xy'][n, c, j].copy() for j in range(k)])
        confidence.append([t['peak_conf'][n, c, j] for j in range(k)])
    return points, confidence


def tables_to_objects(t, n, with_points=True):
    """-> list of dicts with the keys ObjectKeypointPipeline.__call__ returns (pipeline.py:195-199)."""
    C = t['kp_count'].shape[2]
    V = t['votes'].shape[2]
    objects = []
    for o in range(int(t['n_objects'][n])):
        keypoints, points = [], []
        for c in range(C):
            cnt = int(t['kp_count'][n, o, c])
            if cnt == 0:
                keypoints.append(np.array([]))                 # pipeline.py:152
                points.append(None)                            # pipeline.py:165-166
            else:
                keypoints.append(t['kp_xy'][n, o, c, :cnt].copy())
                points.append(t['kp_point'][n, o, c, :cnt].copy())
        votes = [t['votes'][n, o, v].copy() for v in range(min(int(t['n_votes'][n, o]), V))]
        obj = {'p_centers': votes, 'keypoints': keypoints}
        if with_points:
            obj['p_C'] = points
        objects.append(obj)
    return objects


# ------------------------------------------------------------------------------------------------
# the reference's interface
# ------------------------------------------------------------------------------------------------
class InferenceComponent:
    """TorchScript model runner (pipeline.py:13-28). Unlike the reference it leaves the three
    outputs on the device: the decode kernels read them in place."""
    name = "inference"

    def __init__(self, model, cuda=True):
        self.cuda = cuda
        self.model = torch.jit.load(model) if isinstance(model, (str, bytes)) else model
        self.model = self.model.cuda() if cuda else self.model.cpu().float()

    def __call__(self, frames):
        if self.cuda:
            frames = frames.cuda(non_blocking=True)
        with torch.no_grad():
            heatmaps, depth, centers = self.model(frames)
        return heatmaps, depth, centers


class KeypointExtractionComponent:
    """pipeline.py:30-91. ``__call__(frames[N,C,H,W])`` -> ``(keypoints, confidence)`` nested
    lists [N][C][k]; keypoints are (2,) float32 (x, y)."""
    name = "keypoints"
    PROBABILITY_CUTOFF = 0.1

    def __init__(self, keypoint_config, prediction_size, bandwidth=1.0, **decoder_options):
        self.keypoint_config = [1] + _abi.check_keypoint_config(keypoint_config)
        self.n_keypoints = sum(self.keypoint_config)
        self.decoder = KeypointDecoder(keypoint_config, prediction_size, **decoder_options)

    def __call__(self, frames):
        tables = self.decoder.extract_peaks(frames).numpy()
        keypoints, confidence = [], []
        for n in range(tables['peak_count'].shape[0]):
            kp, conf = tables_to_keypoints(tables, n)
            keypoints.append(kp)
            confidence.append(conf)
        return keypoints, confidence


class ObjectExtraction:
    """pipeline.py:93-153. ``__call__(keypoints[C][k], confidence[C][k], centers[T,2,H,W])`` for one
    frame -> list of dicts with 'center', 'heatmap_points', 'p_centers', 'confidence'."""

    def __init__(self, keypoint_config, prediction_size, **decoder_options):
        self.keypoint_config = _abi.check_keypoint_config(keypoint_config)
        self.prediction_size = prediction_size
        self.decoder = KeypointDecoder(keypoint_config, prediction_size, **decoder_options)

    def __call__(self, keypoints, confidence, centers):
        if len(keypoints[0]) == 0:
            return []
        d = self.decoder
        K = d.params.max_peaks
        tables = DecodeTables(1, d.C, d.cfg, d.params, d.device)
        count = np.zeros((1, d.C), np.int32)
        xy = np.zeros((1, d.C, K, 2), np.float32)
        conf = np.zeros((1, d.C, K), np.float32)
        for c in range(d.C):
            count[0, c] = len(keypoints[c])
            for j in range(min(len(keypoints[c]), K)):
                xy[0, c, j] = np.asarray(keypoints[c][j], dtype=np.float32)
                conf[0, c, j] = float(confidence[c][j])
        tables['peak_count'].copy_(torch.from_numpy(count))
        tables['peak_xy'].copy_(torch.from_numpy(xy))
        tables['peak_conf'].copy_(torch.from_numpy(conf))
        tables['peak_object'].fill_(-1)
        centers = np.asarray(centers, dtype=np.float32)[None]
        t = d.group_objects(None, centers, tables).numpy()
        objects = []
        for o in range(int(t['n_objects'][0])):
            obj = {'center': t['kp_xy'][0, o, 0, 0].copy(), 'heatmap_points': [], 'confidence': [],
                   'p_centers': [t['votes'][0, o, v].copy() for v in range(min(int(t['n_votes'][0, o]), t['votes'].shape[2]))]}
            for c in range(1, d.C):
                cnt = int(t['kp_count'][0, o, c])
                obj['heatmap_points'].append(t['kp_xy'][0, o, c, :cnt].copy() if cnt else np.array([]))
                members = [j for j in range(min(int(t['peak_count'][0, c]), K)) if t['peak_object'][0, c, j] == o]
                obj['confidence'].append([t['peak_conf'][0, c, j] for j in members])
            objects.append(obj)
        return objects


class DetectionToPoint:
    """pipeline.py:155-171. ``reset(camera)``, ``__call__(xy[n,2], depth_map[H,W])`` -> [n,3]
    float64 camera-frame points (None for empty input)."""

    def __init__(self, compat_clip_bug=True, device=None):
        self.params = _abi.make_params(compat_clip_bug=compat_clip_bug)
        self.device = None if device is None else torch.device(device)
        self.camera = None
        self._packed = None

    def reset(self, camera):
        self.camera = camera
        self._packed = _abi.pack_camera(camera)

    def __call__(self, xy, p_depth):
        xy = np.asarray(xy)
        if xy.shape[0] == 0:
            return None
        device = _device(self.device)
        xy_dev = _as_device_f32(xy.astype(np.float32), device)
        depth_dev = _as_device_f32(p_depth, device)
        out = torch.empty((xy_dev.shape[0], 3), dtype=torch.float64, device=device)
        rc = _lib.lib().okp_detection_to_point_f32(xy_dev.data_ptr(), xy_dev.shape[0], depth_dev.data_ptr(),
                                                   depth_dev.shape[0], depth_dev.shape[1], ctypes.byref(self._packed),
                                                   ctypes.byref(self.params), out.data_ptr(), _stream_handle())
        _lib.check(rc, 'okp_detection_to_point_f32')
        return out.cpu().numpy()


class ObjectKeypointPipeline:
    """pipeline.py:173-200. ``ObjectKeypointPipeline(prediction_size, points_3d, keypoint_config)``,
    ``reset(camera)``, ``__call__(heatmap[1,C,H,W], p_depth[1,C,H,W], p_centers[1,C-1,2,H,W])`` ->
    list of {'p_centers', 'keypoints', 'p_C'} per object. ``decode_batch`` is the batched form."""

    def __init__(self, prediction_size, points_3d, keypoint_config, **decoder_options):
        self.decoder = KeypointDecoder(keypoint_config, prediction_size, **decoder_options)
        self.points_3d = points_3d                     # unused by the reference as well (pipeline.py:174)

    def reset(self, camera):
        self.decoder.reset(camera)

    def decode_batch(self, heatmap, p_depth, p_centers, stream=None, cameras=None):
        """Any batch size, device tables out (no host round trip). cameras: a ``self.decoder.camera_table(...)`` with one
        camera per frame, in place of ``reset``'s."""
        return self.decoder.decode_batch(heatmap, p_depth, p_centers, stream=stream, cameras=cameras)

    def __call__(self, heatmap, p_depth, p_centers):
        assert heatmap.shape[0] == 1, "One at the time, please."
        if self.decoder._camera is None:
            raise RuntimeError("call reset(camera) first")
        tables = self.decoder.decode_batch(heatmap, p_depth, p_centers).numpy()
        return tables_to_objects(tables, 0)


class LearnedKeypointTrackingPipeline(ObjectKeypointPipeline):
    """pipeline.py:202-209: model + decode; returns (objects, heatmap)."""

    def __init__(self, model, cuda=True, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.inference = InferenceComponent(model, cuda)

    def __call__(self, frame):
        heatmap, depth, centers = self.inference(frame)
        return super().__call__(heatmap, depth, centers), heatmap
